// Host build of csrc/tinyram_witness.h (the row logic of trp_dev_tinyram_witness) so that tests/test_tinyram_witness_cpu.py
// holds it against tinyram.build on the CPU, fed the packed inputs the device gets.  Not part of the product.
#include <string.h>

#include "../tiny-ram-halo2_b200/csrc/tinyram_witness.h"

struct HostSink {
  uint64_t* out;   // (n_cols, rows, 4) canonical limbs
  size_t rows;
  void put(uint32_t col, size_t row, const trw::U256& v) { memcpy(out + ((size_t)col * rows + row) * 4, v.w, 32); }
};

extern "C" {
// Writes the rows of a zeroed `out` (a_flag holds (tc + flag_next) mod p, before the inversion) and returns the error key of the
// first failure (trw::err_key), or 0.
uint64_t trw_host_run(unsigned W, unsigned R, int flags, const uint64_t* steps, size_t n_steps, const uint64_t* ins,
                      const uint32_t* prog, size_t prog_len, const uint32_t* colmap, uint64_t* out, size_t rows) {
  trw::Shape sh{W, R, n_steps, flags & 1};
  HostSink sink{out, rows};
  uint64_t err = 0;
  for (size_t i = 0; i < n_steps; ++i) {
    const uint64_t e = trw::exe_row(sh, steps, ins, colmap, i, sink);
    if (e && (!err || e < err)) err = e;
  }
  if (flags & 2)
    for (size_t r = 0; r < ((size_t)1 << (W / 2)); ++r) trw::prog_row(R, ins, prog, prog_len, colmap, r, sink);
  return err;
}
}
