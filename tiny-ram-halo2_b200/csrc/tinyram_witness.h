// Row logic of the TinyRAM witness (tinyram.TinyRamCircuit.synthesize) as host/device functions: one execution-table row per
// call, written through a sink in the order synthesize writes it (the last write to a cell wins), so that tinyram_witness.cu
// runs it one thread per step and tests/tinyram_witness_host_shim.cpp runs the same code on the CPU.
//
// Inputs (packed by tinyram._witness_inputs; the formats are documented with trp_dev_tinyram_witness in include/tr_prover.h):
//   steps    n_steps rows of step_stride(R) u64: pc, flag, v_addr (None -> 0), instruction index, regs[R]
//   ins      one row of ins_stride(R) u64 per distinct instruction: the decode words below, then the program-line values (ProgramLine
//            .row_values in to_vec order), then the Out row (OUT_NAMES order)
//   colmap   block column of every role below, then regs[R], out[13], the exe line[L], the program table line[L], the instance
//            line[L] (NONE without a program table), then the count and the list of the intermediate columns
// Values are canonical field elements (U256, < p); the sink converts them (the device sink to Montgomery form).
#pragma once
#include <stddef.h>
#include <stdint.h>

#include "ff.cuh"

namespace trw {

constexpr uint32_t NONE = 0xffffffffu;

// SelectionA..D kinds (tinyram.selections)
enum Sel : uint32_t { S_UNSET, S_ZERO, S_REG, S_REGN, S_A, S_PC, S_PCN, S_PCPLUSONE, S_VADDR, S_MAXWORD, S_ONE, S_NONDET };
// instruction decode words
enum InsWord : uint32_t { I_OPCODE, I_RI, I_RJ, I_A_IS_REG, I_A_VAL, I_SEL_KIND, I_SEL_REG = I_SEL_KIND + 4, I_DECODE = 16 };
// opcodes (trace.OPCODES) the row logic branches on
enum Opc : uint32_t { OP_AND = 0, OP_OR = 1, OP_XOR = 2, OP_MULL = 6, OP_UMULH = 7, OP_SMULH = 8, OP_UDIV = 9, OP_UMOD = 10, OP_SHL = 11,
                      OP_SHR = 12, OP_CMPE = 13, OP_CMPA = 14, OP_CMPAE = 15, OP_CMPG = 16, OP_CMPGE = 17, OP_MOV = 18 };
// column roles; an even-bits config takes three (word, even, odd), a signed config eight (its word's three, msb, word_sigma, check_sign's three)
enum Role : uint32_t {
  C_PC, C_FLAG, C_VALUE, C_S_TRACE, C_A_FLAG,
  C_TV = 5,            // tv_a, tv_b, tv_c, tv_d
  C_R_DEC = 17, C_A_DEC = 20, C_LOGIC_B = 23, C_EVEN_SUM = 26, C_ODD_SUM = 29,
  C_SIGNED = 32,       // signed_a, signed_b, signed_c
  C_A_SHIFT = 56, C_A_POWER, C_LSB_B, C_B_FLAG,
  C_ROLES
};
enum SignedPart : uint32_t { SG_WORD = 0, SG_MSB = 3, SG_SIGMA = 4, SG_CHECK = 5, SG_LEN = 8 };
// errors, with the exception synthesize raises: 1 RuntimeError "Unhandled non-deterministic advice", 2 AssertionError (a next-register
// check of Shl / Shr, SMulh's sign check), 3 IndexError (a step after the last one), 4 OverflowError (shift >= 64),
// 5 AssertionError "assertion failed: cs >= 0" (kept although no word reaches it: bit W - 1 is an odd bit, so msb = 1 puts
// 2^(W-2) into the odd half).  synthesize's "tb does not fit u64" cannot happen here: tb is masked to 32 bits.
enum Err : uint32_t { E_NONDET = 1, E_ASSERT = 2, E_INDEX = 3, E_SHIFT = 4, E_CS = 5 };
constexpr unsigned N_OUT = 13;

FF_HD unsigned line_len(unsigned R) { return 9 * R + 22; }
FF_HD unsigned ins_stride(unsigned R) { return I_DECODE + line_len(R) + N_OUT; }
FF_HD unsigned step_stride(unsigned R) { return 4 + R; }
FF_HD unsigned cm_regs() { return C_ROLES; }
FF_HD unsigned cm_out(unsigned R) { return C_ROLES + R; }
FF_HD unsigned cm_line(unsigned R) { return cm_out(R) + N_OUT; }
FF_HD unsigned cm_prog(unsigned R) { return cm_line(R) + line_len(R); }
FF_HD unsigned cm_inst(unsigned R) { return cm_prog(R) + line_len(R); }
FF_HD unsigned cm_n_int(unsigned R) { return cm_inst(R) + line_len(R); }

// Errors order as synthesize raises them: every row's temporary variables are computed before any gadget is assigned, so a
// phase-1 error of any row comes before a phase-2 error; within a phase the lowest row wins.  0 = no error.
FF_HD uint64_t err_key(unsigned phase, size_t row, uint32_t code) { return ((uint64_t)phase << 40) | ((uint64_t)row << 8) | code; }

struct U256 { uint64_t w[4]; };
FF_HD U256 u256(uint64_t x) { U256 r = {{x, 0, 0, 0}}; return r; }
FF_HD bool u256_is_zero(const U256& a) { return !(a.w[0] | a.w[1] | a.w[2] | a.w[3]); }

constexpr uint64_t P0 = 0x992d30ed00000001ull, P1 = 0x224698fc094cf91bull, P3 = 0x4000000000000000ull;   // Fp, u64 limbs (limb 2 = 0)

// p - x for 0 < x < 2^128
FF_HD U256 p_minus(unsigned __int128 x) {
  const uint64_t lo = (uint64_t)x, hi = (uint64_t)(x >> 64);
  U256 r;
  r.w[0] = P0 - lo;
  uint64_t b = P0 < lo;
  uint64_t t = P1 - hi;
  uint64_t b2 = (P1 < hi) | (t < b);
  r.w[1] = t - b;
  r.w[2] = 0 - b2;
  r.w[3] = P3 - b2;
  return r;
}
// x mod p for |x| < 2^127
FF_HD U256 from_i128(__int128 x) {
  if (x >= 0) { U256 r = {{(uint64_t)x, (uint64_t)((unsigned __int128)x >> 64), 0, 0}}; return r; }
  return x == 0 ? u256(0) : p_minus((unsigned __int128)(-x));
}
// (a + d) mod p, a < p, d in {0, 1}
FF_HD U256 add_small(const U256& a, uint64_t d) {
  if (!d) return a;
  if (a.w[0] == P0 - 1 && a.w[1] == P1 && a.w[2] == 0 && a.w[3] == P3) return u256(0);
  U256 r = a;
  for (int k = 0; k < 4; ++k) { r.w[k] += 1; if (r.w[k]) break; }
  return r;
}
// (a - s) mod p, a < p, s < 2^64
FF_HD U256 sub_small(const U256& a, uint64_t s) {
  if (!(a.w[1] | a.w[2] | a.w[3]) && a.w[0] < s) return p_minus(s - a.w[0]);
  U256 r = a;
  uint64_t b = s;
  for (int k = 0; k < 4 && b; ++k) { uint64_t t = r.w[k]; r.w[k] = t - b; b = t < b; }
  return r;
}
// tinyram.decompose: the even bits of the 256-bit representation; the odd bits of its lower 128 bits shifted right by one
FF_HD void decompose(const U256& w, U256& e, U256& o) {
  const uint64_t EV = 0x5555555555555555ull, OD = 0xAAAAAAAAAAAAAAAAull;
  for (int k = 0; k < 4; ++k) e.w[k] = w.w[k] & EV;
  o = u256(0);
  o.w[0] = (w.w[0] & OD) >> 1;          // bit 0 of (w.w[1] & OD) is 0, so nothing crosses the limb boundary
  o.w[1] = (w.w[1] & OD) >> 1;
}

struct Shape {
  unsigned W, R;
  size_t ne;                 // steps in the trace
  int reg_operand_value;     // synthesize's reg_operand_value
};

template <class Sink>
struct Row {
  const Shape& sh;
  const uint32_t* cm;
  size_t i;
  Sink& out;
  FF_HD void put(uint32_t role_col, const U256& v) { out.put(role_col, i, v); }
  FF_HD void put64(uint32_t col, uint64_t v) { out.put(col, i, u256(v)); }
  FF_HD void decomp(unsigned role, const U256& w, U256* ev = nullptr, U256* od = nullptr) {   // _assign_decompose
    U256 e, o;
    decompose(w, e, o);
    put(cm[role + 1], e); put(cm[role + 2], o);
    if (ev) *ev = e;
    if (od) *od = o;
  }
  // _assign_signed; words here are below 2^128 (tv & (2^128 - 1))
  FF_HD bool signed_(unsigned role, unsigned __int128 word) {
    const unsigned W = sh.W;
    const uint64_t msb = (uint64_t)(word >> (W - 1)) & 1;
    put64(cm[role + SG_MSB], msb);
    const unsigned __int128 top = (unsigned __int128)1 << W;
    const unsigned __int128 sigma = !msb ? word : word >= top ? word - top : top - word;
    U256 s = {{(uint64_t)sigma, (uint64_t)(sigma >> 64), 0, 0}};
    put(cm[role + SG_MSB + 1], s);
    U256 w = {{(uint64_t)word, (uint64_t)(word >> 64), 0, 0}}, o;
    decomp(role + SG_WORD, w, nullptr, &o);
    const __int128 cs = (__int128)(((unsigned __int128)o.w[1] << 64) | o.w[0]) + (msb ? -1 : 1) * ((__int128)1 << (W - 2));
    if (cs < 0) return false;
    const U256 c = from_i128(cs);
    decomp(role + SG_CHECK, c);
    put(cm[role + SG_CHECK], c);
    return true;
  }
};

FF_HD unsigned __int128 low128(const U256& a) { return ((unsigned __int128)a.w[1] << 64) | a.w[0]; }

// One execution-table row: the static cells of the row's instruction, pc / registers / flag, the four temporary variables and their
// halves, the input of a_flag ((tc + flag_next) mod p: the caller inverts the column), the gadget of the instruction and `value`.
// Static cells that are 0 are not written (the caller's block starts zeroed).  Returns err_key(...) of the row's error, or 0.
template <class Sink>
FF_HD uint64_t exe_row(const Shape& sh, const uint64_t* steps, const uint64_t* ins_tab, const uint32_t* cm, size_t i, Sink& out) {
  const unsigned W = sh.W, R = sh.R, L = line_len(R);
  const uint64_t* st = steps + i * step_stride(R);
  const uint64_t* nx = i + 1 < sh.ne ? st + step_stride(R) : nullptr;
  const uint64_t pc = st[0], flag = st[1], v_addr = st[2], *regs = st + 4;
  const uint64_t* ins = ins_tab + st[3] * ins_stride(R);
  const uint32_t opc = (uint32_t)ins[I_OPCODE], ri = (uint32_t)ins[I_RI], rj = (uint32_t)ins[I_RJ];
  const bool a_reg = ins[I_A_IS_REG] != 0;
  const uint64_t a_val = ins[I_A_VAL];
  const uint64_t wmask = (1ull << W) - 1, mask32 = 0xffffffffull;
  Row<Sink> rw{sh, cm, i, out};

  // phase 1: _temp_var_vals (synthesize computes these for every row before it assigns any gadget)
  const uint64_t get = a_reg ? regs[a_val] : a_val;                                     // ImmediateOrRegName::get
  const uint64_t a_of = a_reg ? (sh.reg_operand_value ? regs[a_val] : a_val) : a_val;
  U256 t[4];
  for (int s = 0; s < 4; ++s) {
    const uint32_t kind = (uint32_t)ins[I_SEL_KIND + s], reg = (uint32_t)ins[I_SEL_REG + s];
    uint64_t v = 0;
    switch (kind) {
      case S_UNSET: case S_ZERO: break;
      case S_REG: v = regs[reg]; break;
      case S_REGN: if (!nx) return err_key(1, i, E_INDEX); v = nx[4 + reg]; break;
      case S_A: v = a_of; break;
      case S_PC: v = pc; break;
      case S_PCN: if (!nx) return err_key(1, i, E_INDEX); v = nx[0]; break;
      case S_PCPLUSONE: v = pc + 1; break;
      case S_VADDR: v = v_addr; break;
      case S_MAXWORD: v = wmask; break;
      case S_ONE: v = 1; break;
      default:                                            // the non-deterministic advice
        if (s == 0) {
          if (opc != OP_UDIV) return err_key(1, i, E_NONDET);
          v = get == 0 ? 0 : regs[rj] % get;
        } else if (s == 1) {
          if (opc == OP_UMOD) {
            v = get == 0 ? 0 : regs[rj] / get;
          } else if (opc == OP_CMPA || opc == OP_CMPG || opc == OP_CMPAE || opc == OP_CMPGE) {
            const int64_t x = (int64_t)regs[ri], c = (int64_t)a_of, top = (int64_t)1 << W;
            const bool strict = opc == OP_CMPA || opc == OP_CMPG;
            v = (uint64_t)(strict ? (x > c ? top - (x - c) : c - x) : (x >= c ? top - 1 - (x - c) : c - x - 1));
          } else {
            return err_key(1, i, E_NONDET);
          }
        } else if (s == 2) {
          if (opc == OP_MULL) v = ((regs[rj] * get) >> W) & wmask;
          else if (opc == OP_CMPE) v = regs[ri] ^ get;
          else if (opc == OP_SHL) {                       // shift::non_det_c: ((b << a) - d) / 2^W, d = the low W bits of b << a
            const uint64_t b = regs[rj];
            const uint64_t d = get >= W ? 0 : (b << get) & wmask;
            if (!nx) return err_key(1, i, E_INDEX);
            if (d != nx[4 + ri]) return err_key(1, i, E_ASSERT);
            t[2] = u256(0);                               // a shift >= 64 fails in phase 2 (OverflowError): tc is never used then
            if (get < 64) {
              const unsigned __int128 q = ((unsigned __int128)b << get) >> W;
              t[2] = U256{{(uint64_t)q, (uint64_t)(q >> 64), 0, 0}};
            }
            continue;
          } else return err_key(1, i, E_NONDET);
        } else {
          if (opc == OP_UMULH) v = (regs[rj] * get) & wmask;
          else if (opc == OP_SMULH) {                     // trace.smulh_eval: the lower word, and its sign check
            const int64_t top = (int64_t)1 << W;
            const int64_t x = (int64_t)get, y = (int64_t)regs[rj];
            const __int128 f = (__int128)((x >> (W - 1)) & 1 ? x - top : x) * ((y >> (W - 1)) & 1 ? y - top : y);
            const uint64_t upper = (uint64_t)(f >> W) & wmask;
            if ((f < 0) != (((upper >> (W - 1)) & 1) != 0)) return err_key(1, i, E_ASSERT);
            v = (uint64_t)f & wmask;
          } else if (opc == OP_SHR) {                     // shift::non_det_d: (2^a * b - 2^W * (b >> a)) mod p
            const uint64_t b = regs[rj];
            const uint64_t c = get >= 64 ? 0 : b >> get;
            if (!nx) return err_key(1, i, E_INDEX);
            if (c != nx[4 + ri]) return err_key(1, i, E_ASSERT);
            t[3] = get < 64 ? from_i128((__int128)((unsigned __int128)b << get) - (__int128)((unsigned __int128)c << W)) : u256(0);
            continue;
          } else return err_key(1, i, E_NONDET);
        }
    }
    t[s] = u256(s < 2 ? v & mask32 : v);                  // ta, tb masked to 32 bits; tc, td (< 2^64 here) reduced mod p
  }
  const uint64_t ta = t[0].w[0], tb = t[1].w[0];
  const U256 tc = t[2];

  // static cells of the instruction: intermediate fill, program line, Out row
  const uint32_t n_int = cm[cm_n_int(R)];
  for (uint32_t k = 0; k < n_int; ++k) rw.put64(cm[cm_n_int(R) + 1 + k], ~0ull);
  for (unsigned k = 0; k < L; ++k)
    if (ins[I_DECODE + k]) rw.put64(cm[cm_line(R) + k], ins[I_DECODE + k]);
  for (unsigned k = 0; k < N_OUT; ++k)
    if (ins[I_DECODE + L + k]) rw.put64(cm[cm_out(R) + k], ins[I_DECODE + L + k]);
  // machine state
  rw.put64(cm[C_S_TRACE], 1);
  rw.put64(cm[C_PC], pc);
  for (unsigned r = 0; r < R; ++r) rw.put64(cm[cm_regs() + r], regs[r]);
  rw.put64(cm[C_FLAG], flag);
  // temporary variables and their even / odd halves
  for (int s = 0; s < 4; ++s) {
    rw.put(cm[C_TV + 3 * s], t[s]);
    rw.decomp(C_TV + 3 * s, t[s]);
  }
  rw.put(cm[C_A_FLAG], add_small(tc, nx ? nx[1] : 0));

  // phase 2: the gadget of the instruction
  switch (opc) {
    case OP_AND: case OP_OR: case OP_XOR: case OP_CMPE: case OP_MOV: {      // _assign_logic
      U256 le, lo, re, ro;
      rw.decomp(C_A_DEC, u256(ta), &le, &lo);
      rw.decomp(C_LOGIC_B, u256(tb), &re, &ro);
      const U256 es = u256(le.w[0] + re.w[0]), os = u256(lo.w[0] + ro.w[0]);
      rw.put(cm[C_EVEN_SUM], es); rw.decomp(C_EVEN_SUM, es);
      rw.put(cm[C_ODD_SUM], os); rw.decomp(C_ODD_SUM, os);
      rw.put64(cm[C_TV + 6], opc == OP_AND ? (ta & tb) : opc == OP_OR ? (ta | tb) : (ta ^ tb));
      break;
    }
    case OP_CMPG: case OP_CMPGE:
      if (!rw.signed_(C_SIGNED, ta)) return err_key(2, i, E_CS);
      if (!rw.signed_(C_SIGNED + 2 * SG_LEN, low128(tc))) return err_key(2, i, E_CS);
      rw.decomp(C_SIGNED + 2 * SG_LEN + SG_WORD, tc);
      break;
    case OP_SMULH:
      if (!rw.signed_(C_SIGNED, ta)) return err_key(2, i, E_CS);
      if (!rw.signed_(C_SIGNED + SG_LEN, tb)) return err_key(2, i, E_CS);
      rw.decomp(C_SIGNED + SG_LEN + SG_WORD, u256(tb));
      if (!rw.signed_(C_SIGNED + 2 * SG_LEN, low128(tc))) return err_key(2, i, E_CS);
      rw.decomp(C_SIGNED + 2 * SG_LEN + SG_WORD, tc);
      break;
    case OP_UMOD: case OP_UDIV: {                                                 // flag3
      const U256 r = u256_is_zero(tc) ? u256(0) : sub_small(tc, ta + 1);
      rw.put(cm[C_R_DEC], r);
      rw.decomp(C_R_DEC, r);
      break;
    }
    case OP_SHL: case OP_SHR: {                                                   // _assign_shift, then flag4
      const uint64_t bits = get;
      rw.put64(cm[C_A_SHIFT], W < bits);
      if (bits >= 64) return err_key(2, i, E_SHIFT);
      rw.put64(cm[C_A_POWER], bits == W ? 0 : 1ull << bits);
      const U256 r = u256(bits > W ? 0 : W - bits);
      rw.put(cm[C_R_DEC], r);
      rw.decomp(C_R_DEC, r);
      rw.put64(cm[C_LSB_B], tb & 1);
      rw.put64(cm[C_B_FLAG], opc == OP_SHL);
      if (!rw.signed_(C_SIGNED + SG_LEN, tb)) return err_key(2, i, E_CS);
      break;
    }
    default: break;
  }
  rw.put64(cm[C_VALUE], v_addr);
  return 0;
}

// One row r < TABLE_LEN of the program table and of the instance columns: the line of prog[min(r, prog_len - 1)] (program_instance
// pads with the terminal Answer).  Zeros are not written.
template <class Sink>
FF_HD void prog_row(unsigned R, const uint64_t* ins_tab, const uint32_t* prog, size_t prog_len, const uint32_t* cm, size_t r, Sink& out) {
  const unsigned L = line_len(R);
  const uint64_t* ins = ins_tab + (size_t)prog[r < prog_len ? r : prog_len - 1] * ins_stride(R) + I_DECODE;
  for (unsigned k = 0; k < L; ++k) {
    if (!ins[k]) continue;
    out.put(cm[cm_prog(R) + k], r, u256(ins[k]));
    out.put(cm[cm_inst(R) + k], r, u256(ins[k]));
  }
}

}  // namespace trw
