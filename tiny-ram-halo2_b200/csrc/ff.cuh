// K1: 255-bit Pasta prime-field arithmetic for sm_100a, 8 x 32-bit limbs, Montgomery form (R = 2^256).
//
// Replaces pasta_curves::fields::{Fp,Fq} (pasta_curves 0.4.1, Cargo.lock:847-849; the circuit field is chosen
// at /root/reference/src/test_utils.rs:2).  Memory format is identical to the Rust side: uint64_t[4]
// little-endian limbs holding a*R mod p, value < p.
//
// Multiplication is word-serial CIOS over 32-bit limbs written as mad.lo.cc/madc.hi.cc chains that ptxas
// fuses into IMAD.WIDE.U32(.X).  Products a_j*b_i with even j accumulate in E (limb positions 0..7), odd j
// in O (positions 1..8); the two are merged once at the end.  Both Pasta moduli have 32-bit limbs
//     [1, p1, p2, p3, 0, 0, 0, 0x40000000]   and   -p^-1 mod 2^32 = 0xffffffff,
// so a reduction round is m = -T0, three wide MACs (p1,p2,p3), one carry ripple to the top and one funnel
// shift for the 2^254 term (see redc_row): 88 wide MACs per product instead of 128.
//
// Every asm block below has a plain-C twin (used when compiled for the host) so the carry logic is
// unit-tested on the CPU build box (tests/test_ff_host.py) before going to the GPU.
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define FF_HD __host__ __device__ __forceinline__
#define FF_D __device__ __forceinline__
#else
#define FF_HD inline
#define FF_D inline
#endif

namespace ff {

struct FpParams {   // Pallas base field / Vesta scalar field
  static constexpr uint32_t P1 = 0x992d30edu, P2 = 0x094cf91bu, P3 = 0x224698fcu;
  static FF_HD constexpr uint32_t p(int i) { return i == 0 ? 0x00000001u : i == 1 ? 0x992d30edu : i == 2 ? 0x094cf91bu : i == 3 ? 0x224698fcu : i == 4 ? 0x00000000u : i == 5 ? 0x00000000u : i == 6 ? 0x00000000u : 0x40000000u; }
  static FF_HD constexpr uint32_t one(int i) { return i == 0 ? 0xfffffffdu : i == 1 ? 0x34786d38u : i == 2 ? 0xe41914adu : i == 3 ? 0x992c350bu : i == 4 ? 0xffffffffu : i == 5 ? 0xffffffffu : i == 6 ? 0xffffffffu : 0x3fffffffu; }
  static FF_HD constexpr uint32_t r2(int i) { return i == 0 ? 0x0000000fu : i == 1 ? 0x8c78ecb3u : i == 2 ? 0x8b0de0e7u : i == 3 ? 0xd7d30dbdu : i == 4 ? 0xc3c95d18u : i == 5 ? 0x7797a99bu : i == 6 ? 0x7b9cb714u : 0x096d41afu; }
};
struct FqParams {   // Vesta base field / Pallas scalar field
  static constexpr uint32_t P1 = 0x8c46eb21u, P2 = 0x0994a8ddu, P3 = 0x224698fcu;
  static FF_HD constexpr uint32_t p(int i) { return i == 0 ? 0x00000001u : i == 1 ? 0x8c46eb21u : i == 2 ? 0x0994a8ddu : i == 3 ? 0x224698fcu : i == 4 ? 0x00000000u : i == 5 ? 0x00000000u : i == 6 ? 0x00000000u : 0x40000000u; }
  static FF_HD constexpr uint32_t one(int i) { return i == 0 ? 0xfffffffdu : i == 1 ? 0x5b2b3e9cu : i == 2 ? 0xe3420567u : i == 3 ? 0x992c350bu : i == 4 ? 0xffffffffu : i == 5 ? 0xffffffffu : i == 6 ? 0xffffffffu : 0x3fffffffu; }
  static FF_HD constexpr uint32_t r2(int i) { return i == 0 ? 0x0000000fu : i == 1 ? 0xfc9678ffu : i == 2 ? 0x891a16e3u : i == 3 ? 0x67bb433du : i == 4 ? 0x04ccf590u : i == 5 ? 0x7fae2310u : i == 6 ? 0x7ccfdaa9u : 0x096d41afu; }
};

template <class PR>
struct Fe {
  uint32_t v[8];
};

// ------------------------------------------------------------------------------------------------
// carry-chain building blocks (asm on device, C twin on host)
// ------------------------------------------------------------------------------------------------

// r = a + b over 8 limbs, returns carry out
FF_HD uint32_t add8(uint32_t* r, const uint32_t* a, const uint32_t* b) {
  uint32_t c;
#ifdef __CUDA_ARCH__
  asm("add.cc.u32 %0, %9, %17;\n\t"
      "addc.cc.u32 %1, %10, %18;\n\t"
      "addc.cc.u32 %2, %11, %19;\n\t"
      "addc.cc.u32 %3, %12, %20;\n\t"
      "addc.cc.u32 %4, %13, %21;\n\t"
      "addc.cc.u32 %5, %14, %22;\n\t"
      "addc.cc.u32 %6, %15, %23;\n\t"
      "addc.cc.u32 %7, %16, %24;\n\t"
      "addc.u32 %8, 0, 0;"
      : "=&r"(r[0]), "=&r"(r[1]), "=&r"(r[2]), "=&r"(r[3]), "=&r"(r[4]), "=&r"(r[5]), "=&r"(r[6]), "=&r"(r[7]), "=&r"(c)
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(a[4]), "r"(a[5]), "r"(a[6]), "r"(a[7]),
        "r"(b[0]), "r"(b[1]), "r"(b[2]), "r"(b[3]), "r"(b[4]), "r"(b[5]), "r"(b[6]), "r"(b[7]));
#else
  uint64_t t = 0;
  for (int i = 0; i < 8; ++i) { t += (uint64_t)a[i] + b[i]; r[i] = (uint32_t)t; t >>= 32; }
  c = (uint32_t)t;
#endif
  return c;
}

// r = a - b over 8 limbs, returns borrow (1 if a < b)
FF_HD uint32_t sub8(uint32_t* r, const uint32_t* a, const uint32_t* b) {
  uint32_t bw;
#ifdef __CUDA_ARCH__
  asm("sub.cc.u32 %0, %9, %17;\n\t"
      "subc.cc.u32 %1, %10, %18;\n\t"
      "subc.cc.u32 %2, %11, %19;\n\t"
      "subc.cc.u32 %3, %12, %20;\n\t"
      "subc.cc.u32 %4, %13, %21;\n\t"
      "subc.cc.u32 %5, %14, %22;\n\t"
      "subc.cc.u32 %6, %15, %23;\n\t"
      "subc.cc.u32 %7, %16, %24;\n\t"
      "subc.u32 %8, 0, 0;"
      : "=&r"(r[0]), "=&r"(r[1]), "=&r"(r[2]), "=&r"(r[3]), "=&r"(r[4]), "=&r"(r[5]), "=&r"(r[6]), "=&r"(r[7]), "=&r"(bw)
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(a[4]), "r"(a[5]), "r"(a[6]), "r"(a[7]),
        "r"(b[0]), "r"(b[1]), "r"(b[2]), "r"(b[3]), "r"(b[4]), "r"(b[5]), "r"(b[6]), "r"(b[7]));
  bw &= 1u;   // subc.u32 0-0-borrow = 0xffffffff when borrow
#else
  int64_t t = 0;
  for (int i = 0; i < 8; ++i) { t += (int64_t)a[i] - (int64_t)b[i]; r[i] = (uint32_t)t; t >>= 32; }
  bw = (uint32_t)(t & 1);
#endif
  return bw;
}

// Row i > 0 of the CIOS product: shift the running value right by one limb and add a * bi.
//   value = E (positions 0..7; E[0] is known to be 0 and ignored) + O * 2^32 (positions 1..8)
//   En = O + E[1] + a_even * bi ;  On = (E >> 2 limbs) + a_odd * bi   (new value = En + On * 2^32)
FF_HD void mul_row(uint32_t* En, uint32_t* On, const uint32_t* E, const uint32_t* O, const uint32_t* a, uint32_t bi) {
#ifdef __CUDA_ARCH__
  asm("add.cc.u32      %0, %16, %25;\n\t"        // En0 = O0 + E1
      "madc.lo.cc.u32  %8, %33, %40, %26;\n\t"   // On0 = a1*bi + E2 + c
      "madc.hi.cc.u32  %9, %33, %40, %27;\n\t"
      "madc.lo.cc.u32 %10, %35, %40, %28;\n\t"   // a3
      "madc.hi.cc.u32 %11, %35, %40, %29;\n\t"
      "madc.lo.cc.u32 %12, %37, %40, %30;\n\t"   // a5
      "madc.hi.cc.u32 %13, %37, %40, %31;\n\t"
      "madc.lo.cc.u32 %14, %39, %40, 0;\n\t"     // a7
      "madc.hi.u32    %15, %39, %40, 0;\n\t"
      "mad.lo.cc.u32   %0, %32, %40, %0;\n\t"    // En0 += a0*bi
      "madc.hi.cc.u32  %1, %32, %40, %17;\n\t"
      "madc.lo.cc.u32  %2, %34, %40, %18;\n\t"   // a2
      "madc.hi.cc.u32  %3, %34, %40, %19;\n\t"
      "madc.lo.cc.u32  %4, %36, %40, %20;\n\t"   // a4
      "madc.hi.cc.u32  %5, %36, %40, %21;\n\t"
      "madc.lo.cc.u32  %6, %38, %40, %22;\n\t"   // a6
      "madc.hi.cc.u32  %7, %38, %40, %23;\n\t"
      "addc.u32       %15, %15, 0;"
      : "=&r"(En[0]), "=&r"(En[1]), "=&r"(En[2]), "=&r"(En[3]), "=&r"(En[4]), "=&r"(En[5]), "=&r"(En[6]), "=&r"(En[7]),
        "=&r"(On[0]), "=&r"(On[1]), "=&r"(On[2]), "=&r"(On[3]), "=&r"(On[4]), "=&r"(On[5]), "=&r"(On[6]), "=&r"(On[7])
      : "r"(O[0]), "r"(O[1]), "r"(O[2]), "r"(O[3]), "r"(O[4]), "r"(O[5]), "r"(O[6]), "r"(O[7]),   // 16..23
        "r"(E[0]), "r"(E[1]), "r"(E[2]), "r"(E[3]), "r"(E[4]), "r"(E[5]), "r"(E[6]), "r"(E[7]),   // 24..31
        "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(a[4]), "r"(a[5]), "r"(a[6]), "r"(a[7]),   // 32..39
        "r"(bi));                                                                                   // 40
#else
  uint64_t t; uint32_t c;
  t = (uint64_t)O[0] + E[1]; En[0] = (uint32_t)t; c = (uint32_t)(t >> 32);
  // odd chain
  uint64_t carry = c;
  for (int j = 0; j < 4; ++j) {
    uint64_t prod = (uint64_t)a[2 * j + 1] * bi;
    uint32_t addlo = j < 3 ? E[2 * j + 2] : 0, addhi = j < 3 ? E[2 * j + 3] : 0;
    t = (uint64_t)(uint32_t)prod + addlo + carry; On[2 * j] = (uint32_t)t; carry = t >> 32;
    t = (prod >> 32) + addhi + carry; On[2 * j + 1] = (uint32_t)t; carry = t >> 32;
  }
  // even chain
  carry = 0;
  for (int j = 0; j < 4; ++j) {
    uint64_t prod = (uint64_t)a[2 * j] * bi;
    uint32_t addlo = j == 0 ? En[0] : O[2 * j], addhi = O[2 * j + 1];
    t = (uint64_t)(uint32_t)prod + addlo + carry; En[2 * j] = (uint32_t)t; carry = t >> 32;
    t = (prod >> 32) + addhi + carry; En[2 * j + 1] = (uint32_t)t; carry = t >> 32;
  }
  On[7] += (uint32_t)carry;
#endif
}

// One Montgomery reduction round on (E, O): adds m*p with m = -E[0] so that position 0 becomes zero.
// E[0] is left stale (callers ignore it).  `mprev` is the previous round's m (0 before round 0) and is
// replaced by this round's.
//
// p = 1 + P1*2^32 + P2*2^64 + P3*2^96 + 2^254, so m*p touches positions 0..4 and 7..8 only.  Positions
// are 32-bit limbs of the running value; E[k] sits at position k, O[k] at position k+1.
//   * m*P2 (positions 2,3) goes into E; its carry is taken one limb further (E4, position 4) and caught
//     in cE.  m*P1 (1,2) and m*P3 (3,4) go into O in one chain that starts from the carry of E0 + m
//     (E0 + m is 0 or 2^32) and adds cE at position 5.  That O chain is the only ripple to the top; it
//     passes the zero limbs 5..6 of p once per round instead of once per chain.  (Each product lands on
//     an even-aligned register pair, E2:E3, O0:O1, O2:O3, which ptxas fuses into one IMAD.WIDE.)
//   * m*2^254 is m<<30 at position 7 and m>>2 at position 8.  Position 8 of this round is position 7 of
//     the next, where the next round's m<<30 lands too, so the two share a word:
//         w = (mprev >> 2) | (m << 30)   (one funnel shift; the bit ranges are disjoint, no carry)
//     added at position 7 by the same O chain.  Deferring mprev>>2 by one round is safe because position
//     8 of round i is absolute limb i+8 >= 8: no later m reads it.  The last round's m>>2 is added by
//     merge_eo.
// Bounds: with a, b < p every CIOS round keeps the shifted value U < 2p (U' = (U + a*bi + m*p)/2^32 <
// (2p + 2*(2^32-1)*p)/2^32 < 2p), so before the shift the value is < 2p*2^32 < 2^288 and fits positions
// 0..8.  The deferred m>>2 only makes the represented value smaller.  Every carry is either consumed in
// a chain or caught (cE), none is dropped except the last one out of position 8 (O7), which is zero
// because the value represented by E, O and cE is < 2^288 and every limb is non-negative.
template <class PR>
FF_HD void redc_row(uint32_t* E, uint32_t* O, uint32_t& mprev) {
  uint32_t m = 0u - E[0];
#ifdef __CUDA_ARCH__
  uint32_t w = __funnelshift_r(mprev, m, 2);
  uint32_t cE, junk;
  asm("mad.lo.cc.u32   %0, %14, %16, %0;\n\t"    // E2 += m*p2 (positions 2, 3)
      "madc.hi.cc.u32  %1, %14, %16, %1;\n\t"
      "addc.cc.u32     %2, %2, 0;\n\t"           // E4 (position 4)
      "addc.u32       %11, 0, 0;\n\t"            // cE: carry into position 5
      "add.cc.u32     %12, %13, %14;\n\t"        // E0 + m -> carry = (E0 != 0)
      "madc.lo.cc.u32  %3, %14, %15, %3;\n\t"    // O0 += m*p1 (positions 1, 2)
      "madc.hi.cc.u32  %4, %14, %15, %4;\n\t"
      "madc.lo.cc.u32  %5, %14, %17, %5;\n\t"    // O2 += m*p3 (positions 3, 4)
      "madc.hi.cc.u32  %6, %14, %17, %6;\n\t"
      "addc.cc.u32     %7, %7, %11;\n\t"         // O4 += cE (position 5)
      "addc.cc.u32     %8, %8, 0;\n\t"
      "addc.cc.u32     %9, %9, %18;\n\t"         // O6 += w (position 7)
      "addc.u32       %10, %10, 0;"              // O7 (position 8)
      : "+r"(E[2]), "+r"(E[3]), "+r"(E[4]),                                                          // 0..2
        "+r"(O[0]), "+r"(O[1]), "+r"(O[2]), "+r"(O[3]), "+r"(O[4]), "+r"(O[5]), "+r"(O[6]), "+r"(O[7]),  // 3..10
        "=&r"(cE), "=&r"(junk)                                                                       // 11, 12
      : "r"(E[0]), "r"(m), "r"(PR::P1), "r"(PR::P2), "r"(PR::P3), "r"(w));                         // 13..18
#else
  uint32_t w = (mprev >> 2) | (m << 30);
  uint64_t t, carry;
  // E: m*p2 at positions 2, 3, one more limb, carry caught in cE
  uint64_t prod = (uint64_t)m * PR::P2;
  t = (uint64_t)(uint32_t)prod + E[2]; E[2] = (uint32_t)t; carry = t >> 32;
  t = (prod >> 32) + E[3] + carry; E[3] = (uint32_t)t; carry = t >> 32;
  t = (uint64_t)E[4] + carry; E[4] = (uint32_t)t; carry = t >> 32;
  uint32_t cE = (uint32_t)carry;
  // O: m at position 0, m*p1, m*p3, cE, w, up to position 8
  t = (uint64_t)E[0] + m; carry = t >> 32;
  prod = (uint64_t)m * PR::P1;
  t = (uint64_t)(uint32_t)prod + O[0] + carry; O[0] = (uint32_t)t; carry = t >> 32;
  t = (prod >> 32) + O[1] + carry; O[1] = (uint32_t)t; carry = t >> 32;
  prod = (uint64_t)m * PR::P3;
  t = (uint64_t)(uint32_t)prod + O[2] + carry; O[2] = (uint32_t)t; carry = t >> 32;
  t = (prod >> 32) + O[3] + carry; O[3] = (uint32_t)t; carry = t >> 32;
  t = (uint64_t)O[4] + cE + carry; O[4] = (uint32_t)t; carry = t >> 32;
  t = (uint64_t)O[5] + carry; O[5] = (uint32_t)t; carry = t >> 32;
  t = (uint64_t)O[6] + w + carry; O[6] = (uint32_t)t; carry = t >> 32;
  O[7] += (uint32_t)carry;
#endif
  mprev = m;
}

// r = O + (E >> one limb) + top * 2^224, 8 limbs (the value is < 2p < 2^256, so no carry out).  `top` is the
// last reduction round's m >> 2 (see redc_row).
FF_HD void merge_eo(uint32_t* r, const uint32_t* E, const uint32_t* O, uint32_t top) {
#ifdef __CUDA_ARCH__
  asm("add.cc.u32  %0, %8, %16;\n\t"
      "addc.cc.u32 %1, %9, %17;\n\t"
      "addc.cc.u32 %2, %10, %18;\n\t"
      "addc.cc.u32 %3, %11, %19;\n\t"
      "addc.cc.u32 %4, %12, %20;\n\t"
      "addc.cc.u32 %5, %13, %21;\n\t"
      "addc.cc.u32 %6, %14, %22;\n\t"
      "addc.u32    %7, %15, %23;"
      : "=&r"(r[0]), "=&r"(r[1]), "=&r"(r[2]), "=&r"(r[3]), "=&r"(r[4]), "=&r"(r[5]), "=&r"(r[6]), "=&r"(r[7])
      : "r"(O[0]), "r"(O[1]), "r"(O[2]), "r"(O[3]), "r"(O[4]), "r"(O[5]), "r"(O[6]), "r"(O[7]),
        "r"(E[1]), "r"(E[2]), "r"(E[3]), "r"(E[4]), "r"(E[5]), "r"(E[6]), "r"(E[7]), "r"(top));
#else
  uint64_t t = 0;
  for (int i = 0; i < 8; ++i) { t += (uint64_t)O[i] + (i < 7 ? E[i + 1] : top); r[i] = (uint32_t)t; t >>= 32; }
#endif
}

// ------------------------------------------------------------------------------------------------
// field operations
// ------------------------------------------------------------------------------------------------
template <class PR> FF_HD Fe<PR> fe_zero() { Fe<PR> r; for (int i = 0; i < 8; ++i) r.v[i] = 0; return r; }
template <class PR> FF_HD Fe<PR> fe_one() { Fe<PR> r; for (int i = 0; i < 8; ++i) r.v[i] = PR::one(i); return r; }
template <class PR> FF_HD bool fe_is_zero(const Fe<PR>& a) {
  return (a.v[0] | a.v[1] | a.v[2] | a.v[3] | a.v[4] | a.v[5] | a.v[6] | a.v[7]) == 0;
}
template <class PR> FF_HD bool fe_eq(const Fe<PR>& a, const Fe<PR>& b) {
  uint32_t d = 0;
  for (int i = 0; i < 8; ++i) d |= a.v[i] ^ b.v[i];
  return d == 0;
}

// if x >= p then x - p else x   (x < 2p)
template <class PR> FF_HD void fe_final_sub(Fe<PR>& x) {
  uint32_t t[8], p[8];
  for (int i = 0; i < 8; ++i) p[i] = PR::p(i);
  uint32_t bw = sub8(t, x.v, p);
  for (int i = 0; i < 8; ++i) x.v[i] = bw ? x.v[i] : t[i];
}

template <class PR> FF_HD Fe<PR> fe_add(const Fe<PR>& a, const Fe<PR>& b) {
  Fe<PR> r;
  add8(r.v, a.v, b.v);          // a + b < 2p < 2^256
  fe_final_sub(r);
  return r;
}
template <class PR> FF_HD Fe<PR> fe_sub(const Fe<PR>& a, const Fe<PR>& b) {
  Fe<PR> r;
  uint32_t bw = sub8(r.v, a.v, b.v);
  uint32_t p[8];
  for (int i = 0; i < 8; ++i) p[i] = bw ? PR::p(i) : 0u;
  add8(r.v, r.v, p);
  return r;
}
template <class PR> FF_HD Fe<PR> fe_neg(const Fe<PR>& a) { return fe_sub(fe_zero<PR>(), a); }
template <class PR> FF_HD Fe<PR> fe_dbl(const Fe<PR>& a) { return fe_add(a, a); }

template <class PR> FF_HD Fe<PR> fe_mul(const Fe<PR>& a, const Fe<PR>& b) {
  uint32_t E[8], O[8], E2[8], O2[8];
  // row 0: plain wide products
  for (int j = 0; j < 4; ++j) {
    uint64_t pe = (uint64_t)a.v[2 * j] * b.v[0];
    uint64_t po = (uint64_t)a.v[2 * j + 1] * b.v[0];
    E[2 * j] = (uint32_t)pe; E[2 * j + 1] = (uint32_t)(pe >> 32);
    O[2 * j] = (uint32_t)po; O[2 * j + 1] = (uint32_t)(po >> 32);
  }
  uint32_t m = 0;
  redc_row<PR>(E, O, m);
#pragma unroll
  for (int i = 1; i < 8; i += 2) {
    mul_row(E2, O2, E, O, a.v, b.v[i]);
    redc_row<PR>(E2, O2, m);
    if (i + 1 < 8) {
      mul_row(E, O, E2, O2, a.v, b.v[i + 1]);
      redc_row<PR>(E, O, m);
    }
  }
  Fe<PR> r;
  merge_eo(r.v, E2, O2, m >> 2);
  fe_final_sub(r);
  return r;
}
template <class PR> FF_HD Fe<PR> fe_sqr(const Fe<PR>& a) { return fe_mul(a, a); }

// Montgomery -> canonical (multiply by 1) and back
template <class PR> FF_HD Fe<PR> fe_from_mont(const Fe<PR>& a) {
  Fe<PR> one = fe_zero<PR>(); one.v[0] = 1;
  return fe_mul(a, one);
}
template <class PR> FF_HD Fe<PR> fe_to_mont(const Fe<PR>& a) {
  Fe<PR> r2; for (int i = 0; i < 8; ++i) r2.v[i] = PR::r2(i);
  return fe_mul(a, r2);
}

// a^e, e given as 8 x u32 limbs (not constant time; exponents are public)
template <class PR> FF_HD Fe<PR> fe_pow(const Fe<PR>& a, const uint32_t* e, int nlimbs) {
  Fe<PR> acc = fe_one<PR>();
  bool started = false;
  for (int i = nlimbs - 1; i >= 0; --i)
    for (int b = 31; b >= 0; --b) {
      if (started) acc = fe_sqr(acc);
      if ((e[i] >> b) & 1) { acc = started ? fe_mul(acc, a) : a; started = true; }
    }
  return acc;
}
// a^(p-2); 0 -> 0 (ff::Field::invert returns None for 0; callers treat 0 specially)
template <class PR> FF_HD Fe<PR> fe_inv(const Fe<PR>& a) {
  uint32_t e[8];
  for (int i = 0; i < 8; ++i) e[i] = PR::p(i);
  e[0] = 0xffffffffu; e[1] -= 1;   // p - 2: limb0 = 1 - 2 wraps, borrow from limb1 (P1 != 0 for both fields)
  return fe_pow(a, e, 8);
}

#if defined(__CUDACC__)
// 32-byte global/shared load & store as two 128-bit accesses
template <class PR> FF_D Fe<PR> fe_load(const void* p) {
  const uint4* q = reinterpret_cast<const uint4*>(p);
  uint4 lo = q[0], hi = q[1];
  Fe<PR> r;
  r.v[0] = lo.x; r.v[1] = lo.y; r.v[2] = lo.z; r.v[3] = lo.w;
  r.v[4] = hi.x; r.v[5] = hi.y; r.v[6] = hi.z; r.v[7] = hi.w;
  return r;
}
template <class PR> FF_D Fe<PR> fe_load_ro(const void* p) {   // read-only path
  const uint4* q = reinterpret_cast<const uint4*>(p);
  uint4 lo = __ldg(q), hi = __ldg(q + 1);
  Fe<PR> r;
  r.v[0] = lo.x; r.v[1] = lo.y; r.v[2] = lo.z; r.v[3] = lo.w;
  r.v[4] = hi.x; r.v[5] = hi.y; r.v[6] = hi.z; r.v[7] = hi.w;
  return r;
}
template <class PR> FF_D void fe_store(void* p, const Fe<PR>& a) {
  uint4* q = reinterpret_cast<uint4*>(p);
  q[0] = make_uint4(a.v[0], a.v[1], a.v[2], a.v[3]);
  q[1] = make_uint4(a.v[4], a.v[5], a.v[6], a.v[7]);
}
#endif

}  // namespace ff
