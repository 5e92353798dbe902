// The TinyRAM witness block on the device (include/tr_prover.h, trp_dev_tinyram_witness): tinyram.TinyRamCircuit.synthesize +
// program_instance + HostWitness.upload for one trace, from the packed steps and two small tables instead of ~190 MB of host
// columns.  The per-row logic is tinyram_witness.h (one thread per step); values are written in Montgomery form (fe_to_mont) into
// a zeroed block, and a_flag is inverted in place by the library's batch inversion (products.cu).
#include "common.cuh"
#include "tinyram_witness.h"

using namespace ff;

namespace {

struct Locked {
  std::lock_guard<std::mutex> g;
  explicit Locked(trp_ctx* c) : g(c->mu) { cudaSetDevice(c->device); }
};

struct DevSink {
  uint64_t* out;
  size_t n;
  __device__ __forceinline__ void put(uint32_t col, size_t row, const trw::U256& v) {
    Fe<FpParams> a;
#pragma unroll
    for (int k = 0; k < 4; ++k) { a.v[2 * k] = (uint32_t)v.w[k]; a.v[2 * k + 1] = (uint32_t)(v.w[k] >> 32); }
    fe_store(out + ((size_t)col * n + row) * 4, fe_to_mont(a));
  }
};

__global__ void __launch_bounds__(128) tinyram_exe_rows_kernel(trw::Shape sh, const uint64_t* steps, const uint64_t* ins,
                                                               const uint32_t* cm, uint64_t* out, size_t n, unsigned long long* err) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= sh.ne) return;
  DevSink sink{out, n};
  const uint64_t e = trw::exe_row(sh, steps, ins, cm, i, sink);
  if (e) atomicMin(err, (unsigned long long)e);
}

__global__ void __launch_bounds__(128) tinyram_prog_rows_kernel(unsigned R, const uint64_t* ins, const uint32_t* prog, size_t prog_len,
                                                                const uint32_t* cm, size_t table_len, uint64_t* out, size_t n) {
  const size_t r = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= table_len) return;
  DevSink sink{out, n};
  trw::prog_row(R, ins, prog, prog_len, cm, r, sink);
}

}  // namespace

extern "C" int trp_dev_tinyram_witness(trp_ctx* ctx, unsigned word_bits, unsigned reg_count, int flags, const uint64_t* steps,
                                       size_t n_steps, const uint64_t* ins, size_t n_ins, const uint32_t* prog, size_t prog_len,
                                       const uint32_t* colmap, size_t colmap_len, uint64_t* d_out, size_t n_cols, size_t n,
                                       uint64_t* err_row, int* err_code) {
  if (!ctx) return TRP_E_INVALID;
  Locked l(ctx);
  const unsigned W = word_bits, R = reg_count;
  if (ctx->curve != TRP_CURVE_VESTA) TRP_FAIL(ctx, TRP_E_INVALID, "the TinyRAM circuit is over Fp, the scalar field of a Vesta ctx");
  if (W % 8 || W < 8 || W > 32 || R == 0 || R > 64) TRP_FAIL(ctx, TRP_E_INVALID, "machine shape W = %u, R = %u", W, R);
  const size_t table_len = (size_t)1 << (W / 2);
  const bool with_prog = (flags & 2) != 0;
  if (!d_out || !err_row || !err_code || (n_steps && !steps) || !ins || !colmap || (with_prog && (!prog || !prog_len)))
    TRP_FAIL(ctx, TRP_E_INVALID, "NULL buffer");
  if (table_len > n || n_steps > table_len - 1) TRP_FAIL(ctx, TRP_E_INVALID, "%zu steps, TABLE_LEN %zu, %zu rows", n_steps, table_len, n);
  // the tables index each other and the block: check every index before anything is launched
  const unsigned IS = trw::ins_stride(R), SS = trw::step_stride(R);
  if (colmap_len <= trw::cm_n_int(R) || colmap_len != trw::cm_n_int(R) + 1 + (size_t)colmap[trw::cm_n_int(R)])
    TRP_FAIL(ctx, TRP_E_INVALID, "column map of %zu entries", colmap_len);
  for (size_t k = 0; k < colmap_len; ++k) {
    if (k == trw::cm_n_int(R)) continue;
    const bool prog_part = k >= trw::cm_prog(R) && k < trw::cm_n_int(R);
    if (colmap[k] >= n_cols && !(colmap[k] == trw::NONE && prog_part && !with_prog))
      TRP_FAIL(ctx, TRP_E_INVALID, "column map entry %zu = %u, block of %zu columns", k, colmap[k], n_cols);
  }
  for (size_t k = 0; k < n_ins; ++k) {
    const uint64_t* d = ins + k * IS;
    bool ok = d[trw::I_RI] < R && d[trw::I_RJ] < R && (!d[trw::I_A_IS_REG] || d[trw::I_A_VAL] < R);
    for (int s = 0; s < 4; ++s) ok = ok && d[trw::I_SEL_KIND + s] <= trw::S_NONDET && d[trw::I_SEL_REG + s] < R;
    if (!ok) TRP_FAIL(ctx, TRP_E_INVALID, "instruction %zu names a register >= %u or an unknown selection", k, R);
  }
  for (size_t i = 0; i < n_steps; ++i)
    if (steps[i * SS + 3] >= n_ins) TRP_FAIL(ctx, TRP_E_INVALID, "step %zu: instruction index %llu of %zu", i, (unsigned long long)steps[i * SS + 3], n_ins);
  for (size_t r = 0; with_prog && r < prog_len; ++r)
    if (prog[r] >= n_ins) TRP_FAIL(ctx, TRP_E_INVALID, "program line %zu: instruction index %u of %zu", r, prog[r], n_ins);

  const size_t b_steps = ws_align((n_steps ? n_steps : 1) * SS * 8), b_ins = ws_align(n_ins * IS * 8);
  const size_t b_prog = ws_align((prog_len ? prog_len : 1) * 4), b_cm = ws_align(colmap_len * 4);
  TRP_TRY(trp_ws_reserve(ctx, b_steps + b_ins + b_prog + b_cm + 256));
  char* p = (char*)ctx->ws;
  uint64_t* d_steps = (uint64_t*)p; p += b_steps;
  uint64_t* d_ins = (uint64_t*)p; p += b_ins;
  uint32_t* d_prog = (uint32_t*)p; p += b_prog;
  uint32_t* d_cm = (uint32_t*)p; p += b_cm;
  unsigned long long* d_err = (unsigned long long*)p;
  if (n_steps) TRP_CUDA(ctx, cudaMemcpyAsync(d_steps, steps, n_steps * SS * 8, cudaMemcpyHostToDevice, ctx->stream));
  TRP_CUDA(ctx, cudaMemcpyAsync(d_ins, ins, n_ins * IS * 8, cudaMemcpyHostToDevice, ctx->stream));
  if (with_prog) TRP_CUDA(ctx, cudaMemcpyAsync(d_prog, prog, prog_len * 4, cudaMemcpyHostToDevice, ctx->stream));
  TRP_CUDA(ctx, cudaMemcpyAsync(d_cm, colmap, colmap_len * 4, cudaMemcpyHostToDevice, ctx->stream));
  TRP_CUDA(ctx, cudaMemsetAsync(d_err, 0xff, 8, ctx->stream));
  TRP_CUDA(ctx, cudaMemsetAsync(d_out, 0, n_cols * n * 32, ctx->stream));

  trw::Shape sh{W, R, n_steps, flags & 1};
  if (n_steps) {
    tinyram_exe_rows_kernel<<<(unsigned)((n_steps + 127) / 128), 128, 0, ctx->stream>>>(sh, d_steps, d_ins, d_cm, d_out, n, d_err);
    TRP_LAUNCHED(ctx);
  }
  if (with_prog) {
    tinyram_prog_rows_kernel<<<(unsigned)((table_len + 127) / 128), 128, 0, ctx->stream>>>(R, d_ins, d_prog, prog_len, d_cm, table_len, d_out, n);
    TRP_LAUNCHED(ctx);
  }
  // a_flag = 1 / (tc + flag_next), 0 where that is 0 (flag2.rs:62-74)
  TRP_TRY(trp_batch_invert_impl(ctx, 0, d_out + (size_t)colmap[trw::C_A_FLAG] * n * 4, nullptr,
                                d_out + (size_t)colmap[trw::C_A_FLAG] * n * 4, n_steps));
  unsigned long long key = 0;
  TRP_CUDA(ctx, cudaMemcpyAsync(&key, d_err, 8, cudaMemcpyDeviceToHost, ctx->stream));
  TRP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  if (key == ~0ull) { *err_code = 0; *err_row = 0; }
  else { *err_code = (int)(key & 0xff); *err_row = (key >> 8) & 0xffffffffull; }
  return TRP_OK;
}
