// K4/K5: batched radix-2 NTT over the Pasta fields, natural order in and out.
//
// Replaces halo2_proofs::arithmetic::best_fft (field instance) and the transforms of
// halo2_proofs::poly::EvaluationDomain (lagrange_to_coeff / coeff_to_extended / extended_to_coeff), reached
// from the reference through keygen_pk and create_proof (/root/reference/src/test_utils.rs:25,41).
//
// best_fft = bit-reversal permutation followed by log_n radix-2 DIT stages, stage t pairing elements 2^t apart
// with twiddle omega^((pos mod 2^t) * 2^(log_n-t-1)).  Here the stages are grouped into passes of s <= 10
// consecutive stages.  A pass touches index bits [lo, lo+s): one CTA stages 2^c independent tiles of 2^s
// elements in shared memory (2^c adjacent columns of the strided view, so global accesses are 2^c*32 B
// contiguous), runs the s stages there and writes back.  The bit reversal is folded into the first pass's
// loads; coset / vanishing-divisor pre-scaling into the first pass's loads; the 1/n (x zeta^-i) post-scaling
// and truncation into the last pass's stores; zero padding is never materialised.
//
// HBM traffic per transform: (#passes) x (read + write) of the vector, #passes = ceil(log_n / 10).
#include "common.cuh"

#include <cuda.h>          // CUtensorMap (types only: the encoder is fetched through cudaGetDriverEntryPoint, no -lcuda)
#include <cstdlib>
#include <type_traits>

using namespace ff;

namespace {

constexpr unsigned S_MAX = 10;         // stages per pass
constexpr unsigned TILE_LOG_MAX = 11;  // elements per CTA (2 KiB .. 64 KiB of shared memory)
constexpr unsigned C_MAX = 2;          // up to 4 adjacent columns (128 B contiguous)
constexpr unsigned NTT_THREADS = 256;

struct NttPass {
  const uint4* src;
  uint4* dst;
  const uint4* tw;
  unsigned L, lo, s, c;
  int first, last;
  size_t src_stride, dst_stride;   // elements between consecutive columns of the batch
  unsigned n_src, n_dst;
  const uint4* pre; unsigned pre_period;
  const uint4* post; unsigned post_period;
  const uint4* const* src_tab;     // first pass only, or NULL: column y of the batch is read from src_tab[y] (src unused)
};

template <class PR>
__device__ __forceinline__ Fe<PR> lds_fe(const uint4* p0, const uint4* p1, unsigned idx) {
  uint4 lo = p0[idx], hi = p1[idx];
  Fe<PR> r;
  r.v[0] = lo.x; r.v[1] = lo.y; r.v[2] = lo.z; r.v[3] = lo.w;
  r.v[4] = hi.x; r.v[5] = hi.y; r.v[6] = hi.z; r.v[7] = hi.w;
  return r;
}
template <class PR>
__device__ __forceinline__ void sts_fe(uint4* p0, uint4* p1, unsigned idx, const Fe<PR>& a) {
  p0[idx] = make_uint4(a.v[0], a.v[1], a.v[2], a.v[3]);
  p1[idx] = make_uint4(a.v[4], a.v[5], a.v[6], a.v[7]);
}

template <class PR>
__global__ void __launch_bounds__(NTT_THREADS) ntt_pass_kernel(NttPass p) {
  extern __shared__ uint4 smem[];
  const unsigned s = p.s, c = p.c, L = p.L, lo = p.lo;
  const unsigned nelem = 1u << (s + c);
  uint4* plane0 = smem;
  uint4* plane1 = smem + nelem;
  const unsigned g = blockIdx.x;
  const uint4* src = p.src_tab ? p.src_tab[blockIdx.y] : p.src + 2 * (size_t)blockIdx.y * p.src_stride;
  uint4* dst = p.dst + 2 * (size_t)blockIdx.y * p.dst_stride;
  const unsigned smask = (1u << s) - 1, cmask = (1u << c) - 1;

  // position of local element (t, i) in the (bit-reversed-input) stage array
  unsigned low_base = 0, hi = 0;
  if (!p.first) { low_base = (g & ((1u << (lo - c)) - 1)) << c; hi = g >> (lo - c); }
  auto pos_of = [&](unsigned t, unsigned i) -> unsigned {
    if (p.first) return (t << (L - c)) | (g << s) | i;          // c == 0 => t == 0
    return (hi << (lo + s)) | (i << lo) | low_base | t;
  };

  // ---- load -----------------------------------------------------------------------------------------
  for (unsigned e = threadIdx.x; e < nelem; e += blockDim.x) {
    unsigned t = e & cmask, i = e >> c;
    unsigned sidx;
    if (p.first) {
      t = c ? (__brev(t) >> (32 - c)) : 0;
      sidx = L ? (__brev(pos_of(t, i)) >> (32 - L)) : 0;
    } else {
      sidx = pos_of(t, i);
    }
    Fe<PR> v;
    if (sidx < p.n_src) {
      v = fe_load<PR>(src + 2 * (size_t)sidx);
      if (p.pre) {
        unsigned r = sidx % p.pre_period;
        v = fe_mul(v, fe_load_ro<PR>(p.pre + 2 * r));
      }
    } else {
      v = fe_zero<PR>();
    }
    sts_fe(plane0, plane1, (t << s) | i, v);
  }
  __syncthreads();

  // ---- s radix-2 stages in shared memory ---------------------------------------------------------------
  const unsigned half = nelem >> 1;
  for (unsigned q = 0; q < s; ++q) {
    const unsigned tt = lo + q;
    for (unsigned b = threadIdx.x; b < half; b += blockDim.x) {
      unsigned t = b >> (s - 1), j = b & ((1u << (s - 1)) - 1);
      unsigned jl = j & ((1u << q) - 1);
      unsigned i0 = ((j >> q) << (q + 1)) | jl, i1 = i0 | (1u << q);
      Fe<PR> x = lds_fe<PR>(plane0, plane1, (t << s) | i0);
      Fe<PR> y = lds_fe<PR>(plane0, plane1, (t << s) | i1);
      if (tt > 0) {
        unsigned low = p.first ? 0u : (low_base | t);
        unsigned expo = ((jl << lo) | low) << (L - tt - 1);
        y = fe_mul(y, fe_load_ro<PR>(p.tw + 2 * (size_t)expo));
      }
      sts_fe(plane0, plane1, (t << s) | i0, fe_add(x, y));
      sts_fe(plane0, plane1, (t << s) | i1, fe_sub(x, y));
    }
    __syncthreads();
  }

  // ---- store ----------------------------------------------------------------------------------------
  for (unsigned e = threadIdx.x; e < nelem; e += blockDim.x) {
    unsigned t, i;
    if (p.first) { i = e & smask; t = e >> s; } else { t = e & cmask; i = e >> c; }
    unsigned pos = pos_of(t, i);
    if (p.last && pos >= p.n_dst) continue;
    Fe<PR> v = lds_fe<PR>(plane0, plane1, (t << s) | i);
    if (p.last && p.post) {
      unsigned r = pos % p.post_period;
      v = fe_mul(v, fe_load_ro<PR>(p.post + 2 * r));
    }
    fe_store(dst + 2 * (size_t)pos, v);
  }
}

// ---- register-blocked pass ---------------------------------------------------------------------------------------------
// Same pass geometry as ntt_pass_kernel, but the s stages run in groups of r <= R consecutive stages held in REGISTERS:
// a thread owns the 2^r elements that differ only in index bits [q0, q0+r), runs the r stages on them (2^(r-1) independent
// butterflies per stage: instruction-level parallelism for the multiplier) and touches shared memory and the CTA barrier
// once per group instead of once per stage.  The first group reads global memory directly (bit reversal, zero padding and
// pre-scaling folded in), the last group writes it directly (post-scaling, truncation).  Shared memory is XOR-swizzled so
// that the 128-bit accesses of every group are bank-conflict free (a quarter warp covers eight distinct 16-byte bank
// groups): slot = idx ^ (((idx >> 3) ^ (tile << (3 - c))) & 7).
template <class PR, int R>
__global__ void __launch_bounds__(NTT_THREADS, R >= 3 ? 2 : 3) ntt_pass_reg_kernel(NttPass p) {
  extern __shared__ uint4 smem[];
  const unsigned s = p.s, c = p.c, L = p.L, lo = p.lo;
  const unsigned nelem = 1u << (s + c);
  uint4* plane0 = smem;
  uint4* plane1 = smem + nelem;
  const unsigned g = blockIdx.x;
  const uint4* src = p.src_tab ? p.src_tab[blockIdx.y] : p.src + 2 * (size_t)blockIdx.y * p.src_stride;
  uint4* dst = p.dst + 2 * (size_t)blockIdx.y * p.dst_stride;
  const unsigned cmask = (1u << c) - 1;
  unsigned low_base = 0, hi = 0;
  if (!p.first) { low_base = (g & ((1u << (lo - c)) - 1)) << c; hi = g >> (lo - c); }
  auto pos_of = [&](unsigned t, unsigned i) -> unsigned {
    if (p.first) return (t << (L - c)) | (g << s) | i;
    return (hi << (lo + s)) | (i << lo) | low_base | t;
  };
  auto slot = [&](unsigned t, unsigned i) -> unsigned {
    unsigned idx = (t << s) | i;
    return idx ^ (((idx >> 3) ^ (t << (3 - c))) & 7u);
  };
  const unsigned ngroups = (s + R - 1) / R;
  unsigned q0 = 0;
  for (unsigned gi = 0; gi < ngroups; ++gi) {
    const unsigned r = s / ngroups + (gi < s % ngroups ? 1u : 0u);
    const bool gfirst = gi == 0, glast = gi + 1 == ngroups;
    const unsigned units = nelem >> r, tile_units_log = s - r;
    auto body = [&](auto rtag) {
      constexpr int RR = decltype(rtag)::value;
      constexpr int E = 1 << RR;
      for (unsigned u = threadIdx.x; u < units; u += blockDim.x) {
        unsigned t, j;
        if (glast && p.first) { j = u & ((1u << tile_units_log) - 1); t = u >> tile_units_log; }   // contiguous stores along i
        else { t = u & cmask; j = u >> c; }                                                        // adjacent tiles are adjacent in memory
        if (gfirst && p.first && c) t = __brev(t) >> (32 - c);
        const unsigned j_low = j & ((1u << q0) - 1), j_high = j >> q0;
        const unsigned i_base = (j_high << (q0 + RR)) | j_low;
        Fe<PR> x[E];
#pragma unroll
        for (int e = 0; e < E; ++e) {
          const unsigned i = i_base | ((unsigned)e << q0);
          if (gfirst) {
            unsigned sidx = p.first ? (L ? (__brev(pos_of(t, i)) >> (32 - L)) : 0u) : pos_of(t, i);
            if (sidx < p.n_src) {
              x[e] = fe_load<PR>(src + 2 * (size_t)sidx);
              if (p.pre) x[e] = fe_mul(x[e], fe_load_ro<PR>(p.pre + 2 * (sidx % p.pre_period)));
            } else {
              x[e] = fe_zero<PR>();
            }
          } else {
            x[e] = lds_fe<PR>(plane0, plane1, slot(t, i));
          }
        }
        const unsigned low = p.first ? 0u : (low_base | t);
#pragma unroll
        for (int a = 0; a < RR; ++a) {
          const unsigned tt = lo + q0 + a;
#pragma unroll
          for (int b = 0; b < E / 2; ++b) {
            const int el = b & ((1 << a) - 1);                 // bits of e below a
            const int e0 = ((b >> a) << (a + 1)) | el, e1 = e0 | (1 << a);
            Fe<PR> y = x[e1];
            // first group of the first pass: lo = q0 = 0 and low = j_low = 0, so the exponent is el << (L - tt - 1) and the
            // butterflies with el == 0 (known at compile time) multiply by omega^0 = 1: skipped, bit-identical
            if (tt > 0 && !(el == 0 && gfirst && p.first)) {
              const unsigned jl = j_low | ((unsigned)el << q0);
              const unsigned expo = ((jl << lo) | low) << (L - tt - 1);
              y = fe_mul(y, fe_load_ro<PR>(p.tw + 2 * (size_t)expo));
            }
            x[e1] = fe_sub(x[e0], y);
            x[e0] = fe_add(x[e0], y);
          }
        }
#pragma unroll
        for (int e = 0; e < E; ++e) {
          const unsigned i = i_base | ((unsigned)e << q0);
          if (glast) {
            unsigned pos = pos_of(t, i);
            if (p.last && pos >= p.n_dst) continue;
            Fe<PR> v = x[e];
            if (p.last && p.post) v = fe_mul(v, fe_load_ro<PR>(p.post + 2 * (pos % p.post_period)));
            fe_store(dst + 2 * (size_t)pos, v);
          } else {
            sts_fe(plane0, plane1, slot(t, i), x[e]);
          }
        }
      }
    };
    if (r == 1) body(std::integral_constant<int, 1>());
    else if (r == 2) body(std::integral_constant<int, 2>());
    else if constexpr (R >= 3) body(std::integral_constant<int, 3>());
    if (!glast) __syncthreads();
    q0 += r;
  }
}

// ---- specialised register-blocked pass ---------------------------------------------------------------------------------
// ntt_pass_reg_kernel<PR, 2> with everything the host knows at launch made a template parameter: the stage count S, the tile
// width C, first / last pass, the scalings and the gathered source.  The radix-4 groups, their stage offsets and the unit
// counts are then constants; the per-element bit reversal, swizzle and output position become one per-unit base combined
// with a compile-time offset per element, and no scaling needs a division:
//   SCALE_ONE    one scalar (period 1), loaded once per thread;
//   SCALE_TABLE  a table whose period is at least the index range (the index is its own table index).
// Any other period runs the generic kernel.
enum : int { SCALE_NONE = 0, SCALE_ONE = 1, SCALE_TABLE = 2, SCALE_GENERAL = 3 };

constexpr unsigned rev_bits(unsigned x, unsigned n) {
  unsigned r = 0;
  for (unsigned b = 0; b < n; ++b) r |= ((x >> b) & 1u) << (n - 1 - b);
  return r;
}

template <class F, unsigned... G>
__device__ __forceinline__ void static_for(F&& f, std::integer_sequence<unsigned, G...>) { (f(std::integral_constant<unsigned, G>()), ...); }

template <class PR, unsigned S, unsigned C, bool FIRST, bool LAST, int PRE, int POST, bool GATHER>
__global__ void __launch_bounds__(NTT_THREADS, 3) ntt_pass_spec_kernel(NttPass p) {
  extern __shared__ uint4 smem[];
  constexpr unsigned NELEM = 1u << (S + C), CMASK = (1u << C) - 1;
  constexpr unsigned NG = (S + 1) / 2;                          // radix-4 groups, a radix-2 one first when S is odd
  uint4* plane0 = smem;
  uint4* plane1 = smem + NELEM;
  const unsigned L = p.L, lo = FIRST ? 0u : p.lo;
  const unsigned g = blockIdx.x;
  const uint4* src = GATHER ? p.src_tab[blockIdx.y] : p.src + 2 * (size_t)blockIdx.y * p.src_stride;
  uint4* dst = p.dst + 2 * (size_t)blockIdx.y * p.dst_stride;
  unsigned low_base = 0, hi = 0;
  if (!FIRST) { low_base = (g & ((1u << (lo - C)) - 1)) << C; hi = g >> (lo - C); }
  Fe<PR> pre_one, post_one;
  if constexpr (FIRST && PRE == SCALE_ONE) pre_one = fe_load_ro<PR>(p.pre);
  if constexpr (LAST && POST == SCALE_ONE) post_one = fe_load_ro<PR>(p.post);
  // the swizzle is XOR-linear in the index: slot(t, i_base | e << q0) = slot(t, i_base) ^ swz(e << q0)
  auto slot = [&](unsigned t, unsigned i) -> unsigned {
    const unsigned idx = (t << S) | i;
    return idx ^ (((idx >> 3) ^ (t << (3 - C))) & 7u);
  };
  static_for([&](auto gtag) {
    constexpr unsigned GI = decltype(gtag)::value;
    constexpr unsigned RR = (S & 1) && GI == 0 ? 1 : 2;
    constexpr unsigned Q0 = GI == 0 ? 0 : 2 * GI - (S & 1);
    constexpr unsigned E = 1u << RR;
    constexpr bool GFIRST = GI == 0, GLAST = GI + 1 == NG;
    constexpr unsigned UNITS = NELEM >> RR, TILE_UNITS_LOG = S - RR;
#pragma unroll 1
    for (unsigned u = threadIdx.x; u < UNITS; u += NTT_THREADS) {
      unsigned t, j;
      if (GLAST && FIRST) { j = u & ((1u << TILE_UNITS_LOG) - 1); t = u >> TILE_UNITS_LOG; }   // contiguous stores along i
      else { t = u & CMASK; j = u >> C; }                                                        // adjacent tiles adjacent in memory
      if (GFIRST && FIRST && C) t = __brev(t) >> (32 - C);
      const unsigned j_low = j & ((1u << Q0) - 1), j_high = j >> Q0;
      const unsigned i_base = (j_high << (Q0 + RR)) | j_low;
      Fe<PR> x[E];
      if constexpr (GFIRST) {
        // source index of element e: the bit reversal (first pass) maps index bit Q0 + k to bit L - 1 - Q0 - k
        unsigned sbase, sshift;
        if constexpr (FIRST) {
          sbase = L ? __brev((t << (L - C)) | (g << S) | i_base) >> (32 - L) : 0u;
          sshift = L - Q0 - RR;
        } else {
          sbase = (hi << (lo + S)) | (i_base << lo) | low_base | t;
          sshift = lo + Q0;
        }
#pragma unroll
        for (unsigned e = 0; e < E; ++e) {
          const unsigned sidx = sbase | ((FIRST ? rev_bits(e, RR) : e) << sshift);
          if (sidx < p.n_src) {
            x[e] = fe_load<PR>(src + 2 * (size_t)sidx);
            if constexpr (PRE == SCALE_ONE) x[e] = fe_mul(x[e], pre_one);
            else if constexpr (PRE == SCALE_TABLE) x[e] = fe_mul(x[e], fe_load_ro<PR>(p.pre + 2 * (size_t)sidx));
          } else {
            x[e] = fe_zero<PR>();
          }
        }
      } else {
        const unsigned sl = slot(t, i_base);
#pragma unroll
        for (unsigned e = 0; e < E; ++e) {
          const unsigned d = e << Q0;
          x[e] = lds_fe<PR>(plane0, plane1, sl ^ (d ^ ((d >> 3) & 7u)));
        }
      }
      const unsigned low = FIRST ? 0u : (low_base | t);
#pragma unroll
      for (unsigned a = 0; a < RR; ++a) {
        const unsigned tt = lo + Q0 + a;
#pragma unroll
        for (unsigned b = 0; b < E / 2; ++b) {
          const unsigned el = b & ((1u << a) - 1);
          const unsigned e0 = ((b >> a) << (a + 1)) | el, e1 = e0 | (1u << a);
          Fe<PR> y = x[e1];
          // first group of the first pass: the butterflies with el == 0 multiply by omega^0 = 1 (skipped, bit-identical)
          if (!(FIRST && GFIRST && el == 0) && tt > 0) {
            const unsigned expo = (((j_low | (el << Q0)) << lo) | low) << (L - tt - 1);
            y = fe_mul(y, fe_load_ro<PR>(p.tw + 2 * (size_t)expo));
          }
          x[e1] = fe_sub(x[e0], y);
          x[e0] = fe_add(x[e0], y);
        }
      }
      if constexpr (GLAST) {
        const unsigned pbase = FIRST ? ((t << (L - C)) | (g << S) | i_base) : ((hi << (lo + S)) | (i_base << lo) | low_base | t);
        const unsigned pshift = FIRST ? Q0 : lo + Q0;
#pragma unroll
        for (unsigned e = 0; e < E; ++e) {
          const unsigned pos = pbase | (e << pshift);
          if (LAST && pos >= p.n_dst) continue;
          Fe<PR> v = x[e];
          if constexpr (LAST && POST == SCALE_ONE) v = fe_mul(v, post_one);
          else if constexpr (LAST && POST == SCALE_TABLE) v = fe_mul(v, fe_load_ro<PR>(p.post + 2 * (size_t)pos));
          fe_store(dst + 2 * (size_t)pos, v);
        }
      } else {
        const unsigned sl = slot(t, i_base);
#pragma unroll
        for (unsigned e = 0; e < E; ++e) {
          const unsigned d = e << Q0;
          sts_fe(plane0, plane1, sl ^ (d ^ ((d >> 3) & 7u)), x[e]);
        }
      }
    }
    if constexpr (!GLAST) __syncthreads();
  }, std::make_integer_sequence<unsigned, NG>());
}

using PassKernel = void (*)(NttPass);

// The specialised instance for a pass of a two-pass plan, or NULL (middle passes, single-pass transforms, general periods,
// a zero-padded first pass or a truncated last pass: coeff_to_extended pads and extended_to_coeff truncates, both with a
// period-3 scaling that the generic kernel runs anyway).  A gathered source is always scaled by a table of n coset powers.
template <class PR, unsigned S, unsigned C>
PassKernel spec_pass_kernel(const NttPass& p, int pre, int post) {
  if (p.s != S || p.c != C || p.first == p.last) return nullptr;
  const unsigned N = 1u << p.L;
  if (p.first) {
    if (p.n_src < N) return nullptr;
    if (p.src_tab) {
      if (pre == SCALE_TABLE) return ntt_pass_spec_kernel<PR, S, C, true, false, SCALE_TABLE, SCALE_NONE, true>;
    } else {
      if (pre == SCALE_NONE) return ntt_pass_spec_kernel<PR, S, C, true, false, SCALE_NONE, SCALE_NONE, false>;
      if (pre == SCALE_ONE) return ntt_pass_spec_kernel<PR, S, C, true, false, SCALE_ONE, SCALE_NONE, false>;
      if (pre == SCALE_TABLE) return ntt_pass_spec_kernel<PR, S, C, true, false, SCALE_TABLE, SCALE_NONE, false>;
    }
    return nullptr;
  }
  if (p.n_dst < N) return nullptr;
  if (post == SCALE_NONE) return ntt_pass_spec_kernel<PR, S, C, false, true, SCALE_NONE, SCALE_NONE, false>;
  if (post == SCALE_ONE) return ntt_pass_spec_kernel<PR, S, C, false, true, SCALE_NONE, SCALE_ONE, false>;
  if (post == SCALE_TABLE) return ntt_pass_spec_kernel<PR, S, C, false, true, SCALE_NONE, SCALE_TABLE, false>;
  return nullptr;
}

// how a scaling with this table and period reaches indices below `range`
int scale_kind(const void* tab, unsigned period, unsigned range) {
  if (!tab) return SCALE_NONE;
  if (period <= 1) return SCALE_ONE;
  return period >= range ? SCALE_TABLE : SCALE_GENERAL;
}

// ---- TMA-staged pass (sm_100a: cp.async.bulk.tensor + mbarrier) ------------------------------------------------------------------
// Same pass geometry and the same register-blocked butterflies as ntt_pass_reg_kernel, but the tile reaches shared memory
// through the TMA unit instead of through registers: the 2^(s+c) elements of a tile are 2^s runs of 2^c adjacent elements
// (2^c * 32 B contiguous), i.e. ONE 2-D box of the vector viewed as rows of 2^lo elements (later passes) or rows of
// 2^(L-s) elements (first pass: the bit reversal turns the tile's index i into the row index bitrev_s(i), so the bit-reversed
// gather is just a box whose rows are read in a different order).  One elected thread arms an mbarrier with the tile's byte
// count and issues the bulk tensor copies (<= 256 rows per box); the CTA waits on the barrier and then runs every stage group
// in place on that buffer (element (t, i) lives where the box put it; a thread rewrites only the slots it read), so no
// global load instruction, no address arithmetic per element and no bit-reversal arithmetic on the load path remain.
// Out-of-range rows of a zero-padded input (n_src < 2^L) come back as zeros from the TMA unit itself.
struct NttTma {
  CUtensorMap map;        // rank 3: { 8 x u32 per element x row length, rows, batch columns }
  unsigned rows_per_box;  // <= 256
};

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

template <class PR, int R>
__global__ void __launch_bounds__(NTT_THREADS, R >= 3 ? 2 : 3) ntt_pass_tma_kernel(NttPass p, const __grid_constant__ NttTma tma) {
  extern __shared__ __align__(128) uint4 smem[];
  const unsigned s = p.s, c = p.c, L = p.L, lo = p.lo;
  const unsigned nelem = 1u << (s + c);
  uint4* tile = smem;                                      // AoS: element e at tile[2 e], tile[2 e + 1]
  uint64_t* bar = reinterpret_cast<uint64_t*>(smem + 2 * nelem);
  const unsigned g = blockIdx.x;
  uint4* dst = p.dst + 2 * (size_t)blockIdx.y * p.dst_stride;
  const unsigned cmask = (1u << c) - 1;
  unsigned low_base = 0, hi = 0;
  if (!p.first) { low_base = (g & ((1u << (lo - c)) - 1)) << c; hi = g >> (lo - c); }
  auto pos_of = [&](unsigned t, unsigned i) -> unsigned {
    if (p.first) return (t << (L - c)) | (g << s) | i;
    return (hi << (lo + s)) | (i << lo) | low_base | t;
  };
  // where the box put element (t, i): row-major [row][run of 2^c]; the first pass reads rows (and the run) bit-reversed
  auto slot = [&](unsigned t, unsigned i) -> unsigned {
    if (p.first) return ((s ? (__brev(i) >> (32 - s)) : 0u) << c) | (c ? (__brev(t) >> (32 - c)) : 0u);
    return (i << c) | t;
  };

  // ---- tile load: one thread, TMA ------------------------------------------------------------------------------------------
  if (threadIdx.x == 0) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(bar)));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(nelem * 32u) : "memory");
    const unsigned rows = 1u << s;
    // first pass: inner coordinate = bitrev_{L-s-c}(g) runs in, rows 0 .. 2^s; later passes: inner = low_base, rows from hi * 2^s
    const unsigned x0 = (p.first ? ((L - s - c) ? (__brev(g) >> (32 - (L - s - c))) : 0u) << c : low_base) * 8u;
    const unsigned r0 = p.first ? 0u : hi << s;
    for (unsigned r = 0; r < rows; r += tma.rows_per_box) {
      asm volatile(
          "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];"
          ::"r"(smem_u32(tile + 2 * ((size_t)r << c))), "l"(&tma.map), "r"(x0), "r"(r0 + r), "r"((unsigned)blockIdx.y), "r"(smem_u32(bar))
          : "memory");
    }
  }
  {
    uint32_t done = 0;
    while (!done) {
      asm volatile("{ .reg .pred q; mbarrier.try_wait.parity.shared::cta.b64 q, [%1], 0; selp.u32 %0, 1, 0, q; }"
                   : "=r"(done) : "r"(smem_u32(bar)) : "memory");
    }
  }

  // ---- the stage groups, in place ---------------------------------------------------------------------------------------------
  const unsigned ngroups = (s + R - 1) / R;
  unsigned q0 = 0;
  for (unsigned gi = 0; gi < ngroups; ++gi) {
    const unsigned r = s / ngroups + (gi < s % ngroups ? 1u : 0u);
    const bool gfirst = gi == 0, glast = gi + 1 == ngroups;
    const unsigned units = nelem >> r, tile_units_log = s - r;
    auto body = [&](auto rtag) {
      constexpr int RR = decltype(rtag)::value;
      constexpr int E = 1 << RR;
      for (unsigned u = threadIdx.x; u < units; u += blockDim.x) {
        unsigned t, j;
        if (glast && p.first) { j = u & ((1u << tile_units_log) - 1); t = u >> tile_units_log; }   // contiguous stores along i
        else { t = u & cmask; j = u >> c; }
        const unsigned j_low = j & ((1u << q0) - 1), j_high = j >> q0;
        const unsigned i_base = (j_high << (q0 + RR)) | j_low;
        Fe<PR> x[E];
#pragma unroll
        for (int e = 0; e < E; ++e) {
          const unsigned i = i_base | ((unsigned)e << q0);
          const unsigned sl = slot(t, i);
          x[e] = lds_fe<PR>(tile, tile + 1, 2 * sl);
          if (gfirst && p.pre) {
            const unsigned sidx = p.first ? (L ? (__brev(pos_of(t, i)) >> (32 - L)) : 0u) : pos_of(t, i);
            if (sidx < p.n_src) x[e] = fe_mul(x[e], fe_load_ro<PR>(p.pre + 2 * (sidx % p.pre_period)));
          }
        }
        const unsigned low = p.first ? 0u : (low_base | t);
#pragma unroll
        for (int a = 0; a < RR; ++a) {
          const unsigned tt = lo + q0 + a;
#pragma unroll
          for (int b = 0; b < E / 2; ++b) {
            const int el = b & ((1 << a) - 1);
            const int e0 = ((b >> a) << (a + 1)) | el, e1 = e0 | (1 << a);
            Fe<PR> y = x[e1];
            if (tt > 0 && !(el == 0 && gfirst && p.first)) {
              const unsigned jl = j_low | ((unsigned)el << q0);
              const unsigned expo = ((jl << lo) | low) << (L - tt - 1);
              y = fe_mul(y, fe_load_ro<PR>(p.tw + 2 * (size_t)expo));
            }
            x[e1] = fe_sub(x[e0], y);
            x[e0] = fe_add(x[e0], y);
          }
        }
#pragma unroll
        for (int e = 0; e < E; ++e) {
          const unsigned i = i_base | ((unsigned)e << q0);
          if (glast) {
            unsigned pos = pos_of(t, i);
            if (p.last && pos >= p.n_dst) continue;
            Fe<PR> v = x[e];
            if (p.last && p.post) v = fe_mul(v, fe_load_ro<PR>(p.post + 2 * (pos % p.post_period)));
            fe_store(dst + 2 * (size_t)pos, v);
          } else {
            const unsigned sl = slot(t, i);
            sts_fe(tile, tile + 1, 2 * sl, x[e]);
          }
        }
      }
    };
    if (r == 1) body(std::integral_constant<int, 1>());
    else if (r == 2) body(std::integral_constant<int, 2>());
    else if constexpr (R >= 3) body(std::integral_constant<int, 3>());
    if (!glast) __syncthreads();
    q0 += r;
  }
}

// tab[i] = omega^i, i < count
template <class PR>
__global__ void gen_twiddles_kernel(uint4* tab, Fe<PR> omega, unsigned count, unsigned chunk) {
  size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  size_t start = t * chunk;
  if (start >= count) return;
  uint32_t e[1] = {(uint32_t)start};
  Fe<PR> w = fe_pow(omega, e, 1);
  for (unsigned k = 0; k < chunk && start + k < count; ++k) {
    fe_store(tab + 2 * (start + k), w);
    w = fe_mul(w, omega);
  }
}

template <class PR>
__global__ void copy_columns_kernel(const uint4* src, uint4* dst, size_t n, size_t src_stride, size_t dst_stride) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= 2 * n) return;
  dst[2 * (size_t)blockIdx.y * dst_stride + i] = src[2 * (size_t)blockIdx.y * src_stride + i];
}

// cuTensorMapEncodeTiled through the runtime (no link against libcuda)
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                  const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn tensor_map_encoder() {
  static EncodeTiledFn fn = [] {
    void* f = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &f, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess) f = nullptr;
    return (EncodeTiledFn)f;
  }();
  return fn;
}

// The pass's source as a rank-3 tensor of u32: { 8 * row_len, rows, batch }, box { 8 * 2^c, rows_per_box, 1 }
bool encode_pass_map(NttTma& out, const void* src, size_t row_len, size_t rows, size_t batch, size_t batch_stride, unsigned c, unsigned rows_per_box) {
  EncodeTiledFn enc = tensor_map_encoder();
  if (!enc) return false;
  cuuint64_t dims[3] = {8 * (cuuint64_t)row_len, (cuuint64_t)rows, (cuuint64_t)batch};
  cuuint64_t strides[2] = {(cuuint64_t)row_len * 32, (cuuint64_t)batch_stride * 32};       // bytes, dims 1 and 2
  cuuint32_t box[3] = {8u << c, rows_per_box, 1};
  cuuint32_t estr[3] = {1, 1, 1};
  if (batch == 1) strides[1] = strides[0] * rows;                                        // unused, but must be a multiple of 16
  out.rows_per_box = rows_per_box;
  return enc(&out.map, CU_TENSOR_MAP_DATA_TYPE_UINT32, 3, const_cast<void*>(src), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
             CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

struct PassPlan { unsigned lo, s, c; };

std::vector<PassPlan> plan_passes(unsigned L) {
  std::vector<PassPlan> out;
  if (L == 0) return out;
  unsigned P = (L + S_MAX - 1) / S_MAX;
  unsigned lo = 0;
  for (unsigned i = 0; i < P; ++i) {
    unsigned s = (L - lo + (P - i) - 1) / (P - i);
    unsigned c = 0;
    if (P > 1) {
      c = TILE_LOG_MAX - s < C_MAX ? TILE_LOG_MAX - s : C_MAX;
      if (i == 0) { if (L - s < c) c = L - s; }
      else if (lo < c) c = lo;
    }
    out.push_back({lo, s, c});
    lo += s;
  }
  return out;
}

template <class PR>
int get_twiddles(trp_ctx* ctx, unsigned log_n, const uint64_t omega[4], const uint4** out) {
  for (auto& t : ctx->twiddles)
    if (t.log_n == log_n && t.omega[0] == omega[0] && t.omega[1] == omega[1] && t.omega[2] == omega[2] && t.omega[3] == omega[3]) {
      *out = (const uint4*)t.d_tab;
      return TRP_OK;
    }
  unsigned count = log_n ? (1u << (log_n - 1)) : 1;
  void* d = nullptr;
  TRP_CUDA(ctx, cudaMalloc(&d, (size_t)count * 32));
  Fe<PR> w;
  for (int i = 0; i < 4; ++i) { w.v[2 * i] = (uint32_t)omega[i]; w.v[2 * i + 1] = (uint32_t)(omega[i] >> 32); }
  unsigned chunk = 64;
  unsigned threads = (count + chunk - 1) / chunk;
  gen_twiddles_kernel<PR><<<(threads + 127) / 128, 128, 0, ctx->stream>>>((uint4*)d, w, count, chunk);
  TRP_LAUNCHED(ctx);
  TwiddleTable tt;
  tt.log_n = log_n; tt.d_tab = d;
  for (int i = 0; i < 4; ++i) tt.omega[i] = omega[i];
  ctx->twiddles.push_back(tt);
  *out = (const uint4*)d;
  return TRP_OK;
}

template <class PR>
int ntt_run(trp_ctx* ctx, const void* d_src, void* d_dst, size_t batch, unsigned L, const uint64_t omega[4],
            size_t src_stride, size_t dst_stride, unsigned n_src, const void* d_pre, unsigned pre_period,
            const void* d_post, unsigned post_period, unsigned n_dst, void* d_tmp, const void* const* d_src_tab) {
  if (batch == 0) return TRP_OK;
  if (L > 30) TRP_FAIL(ctx, TRP_E_INVALID, "log_n = %u is out of range (max 30)", L);
  if (batch > 65535) TRP_FAIL(ctx, TRP_E_INVALID, "batch = %zu exceeds 65535 columns per call", batch);
  const uint4* tw = nullptr;
  TRP_TRY(get_twiddles<PR>(ctx, L, omega, &tw));
  auto plan = plan_passes(L);
  if (plan.empty()) {   // n = 1: identity transform, only the scalings apply; handle as a one-element "pass"
    plan.push_back({0, 0, 0});
  }
  // buffers: a single pass runs src -> dst; otherwise src -> mid -> ... -> mid -> dst, where mid is the scratch
  // buffer when one is given (stride N) and dst itself otherwise (dst must then hold 2^L elements per column)
  void* d_mid = d_tmp ? d_tmp : d_dst;
  if (plan.size() > 1 && d_mid == d_src) TRP_FAIL(ctx, TRP_E_INVALID, "in-place multi-pass NTT needs scratch");
  const size_t N = (size_t)1 << L;
  const size_t mid_stride = d_tmp ? N : dst_stride;
  for (size_t i = 0; i < plan.size(); ++i) {
    NttPass p;
    p.tw = tw; p.L = L; p.lo = plan[i].lo; p.s = plan[i].s; p.c = plan[i].c;
    p.first = (i == 0); p.last = (i + 1 == plan.size());
    p.n_src = p.first ? n_src : (unsigned)N;
    p.n_dst = n_dst;
    p.pre = p.first ? (const uint4*)d_pre : nullptr; p.pre_period = pre_period ? pre_period : 1;
    p.post = (const uint4*)d_post; p.post_period = post_period ? post_period : 1;
    const void* in = p.first ? d_src : d_mid;
    void* out = p.last ? d_dst : d_mid;
    size_t in_stride = p.first ? src_stride : mid_stride;
    size_t out_stride = p.last ? dst_stride : mid_stride;
    p.src = (const uint4*)in; p.dst = (uint4*)out; p.src_stride = in_stride; p.dst_stride = out_stride;
    p.src_tab = p.first ? (const uint4* const*)d_src_tab : nullptr;
    // register-blocked kernel, radix-4 groups by default (measured on B200 at 8 x 2^20: radix 4 1.53 ms, radix 8 1.61 ms --
    // 117 registers cost a CTA per SM --, one stage per barrier 1.58 ms); TRP_NTT_RADIX=8 / 2 select the other two
    static const int radix_log = [] { const char* e = getenv("TRP_NTT_RADIX"); int v = e ? atoi(e) : 4; return v == 2 ? 1 : v == 8 ? 3 : 2; }();
    // TMA-staged tile loads (TRP_NTT_TMA=1; profiles/ncu_ntt_r02.md has the A/B)
    static const bool use_tma = [] { const char* e = getenv("TRP_NTT_TMA"); return e && atoi(e) == 1; }();
    if (radix_log == 2 && !use_tma) {
      // the shapes a proof runs have a specialised instance: both passes of a size-2^20 transform, the first pass of a
      // size-2^19 one (its second pass, s = 9 and c = 2, runs the generic kernel)
      const int pre_kind = p.first ? scale_kind(p.pre, p.pre_period, p.n_src < N ? p.n_src : (unsigned)N) : SCALE_NONE;
      const int post_kind = p.last ? scale_kind(p.post, p.post_period, p.n_dst < N ? p.n_dst : (unsigned)N) : SCALE_NONE;
      if (PassKernel k = spec_pass_kernel<PR, 10, 1>(p, pre_kind, post_kind)) {
        const size_t sm = (size_t)32 << (p.s + p.c);
        ProfScope ps(ctx, PROF_NTT_PASS, (double)batch * (double)(N >> 1) * (double)p.s);
        if (sm > 48 * 1024) TRP_CUDA(ctx, cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm));
        k<<<dim3((unsigned)(N >> (p.s + p.c)), (unsigned)batch), NTT_THREADS, sm, ctx->stream>>>(p);
        TRP_LAUNCHED(ctx);
        continue;
      }
    }
    unsigned nelem = 1u << (p.s + p.c);
    unsigned threads = nelem / 2 < NTT_THREADS ? nelem / 2 : NTT_THREADS;
    if (threads < 32) threads = 32;
    dim3 grid((unsigned)(N >> (p.s + p.c)), (unsigned)batch);
    size_t smem = (size_t)nelem * 32;
    // generic register-blocked kernel for every other shape
    ProfScope ps(ctx, PROF_NTT_PASS, (double)batch * (double)(N >> 1) * (double)p.s);      // work = radix-2 butterflies of this pass
    if (p.s == 0 || radix_log == 1) {
      if (smem > 48 * 1024)
        TRP_CUDA(ctx, cudaFuncSetAttribute(ntt_pass_kernel<PR>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(32u << TILE_LOG_MAX)));
      ntt_pass_kernel<PR><<<grid, threads, smem, ctx->stream>>>(p);
    } else if (radix_log == 2) {
      unsigned th = nelem / 4 < NTT_THREADS ? nelem / 4 : NTT_THREADS;
      if (th < 32) th = 32;
      // TMA-staged tile loads (TRP_NTT_TMA=1; profiles/ncu_ntt_r02.md has the A/B): needs whole rows, so a zero-padded first
      // pass qualifies only when the padding starts on a row boundary
      const size_t row_len = p.first ? (N >> p.s) : ((size_t)1 << p.lo);
      const size_t rows = p.first ? (p.n_src / row_len) : (N >> p.lo);
      if (use_tma && !p.src_tab && p.s >= 2 && (!p.first || (p.n_src % row_len == 0 && rows >= 1)) && ((uintptr_t)in % 16 == 0)) {
        NttTma tma;
        const unsigned rpb = (1u << p.s) < 256u ? (1u << p.s) : 256u;
        if (encode_pass_map(tma, in, row_len, rows, batch, in_stride, p.c, rpb)) {
          const size_t smem_tma = smem + 16;
          if (smem_tma > 48 * 1024)
            TRP_CUDA(ctx, cudaFuncSetAttribute(ntt_pass_tma_kernel<PR, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)((32u << TILE_LOG_MAX) + 16)));
          ntt_pass_tma_kernel<PR, 2><<<grid, th, smem_tma, ctx->stream>>>(p, tma);
          TRP_LAUNCHED(ctx);
          continue;
        }
      }
      if (smem > 48 * 1024)
        TRP_CUDA(ctx, cudaFuncSetAttribute(ntt_pass_reg_kernel<PR, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(32u << TILE_LOG_MAX)));
      ntt_pass_reg_kernel<PR, 2><<<grid, th, smem, ctx->stream>>>(p);
    } else {
      unsigned th = nelem / 8 < NTT_THREADS ? nelem / 8 : NTT_THREADS;
      if (th < 32) th = 32;
      if (smem > 48 * 1024)
        TRP_CUDA(ctx, cudaFuncSetAttribute(ntt_pass_reg_kernel<PR, 3>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(32u << TILE_LOG_MAX)));
      ntt_pass_reg_kernel<PR, 3><<<grid, th, smem, ctx->stream>>>(p);
    }
    TRP_LAUNCHED(ctx);
  }
  return TRP_OK;
}

}  // namespace

// tab[i] = g^i for i < 2^(log_n-1), cached per (log_n, g) in the ctx (the NTT twiddle tables are the g = omega case)
int trp_get_powers(trp_ctx* ctx, int field, unsigned log_n, const uint64_t g[4], const void** out) {
  const uint4* t = nullptr;
  int rc = field == 0 ? get_twiddles<FpParams>(ctx, log_n, g, &t) : get_twiddles<FqParams>(ctx, log_n, g, &t);
  *out = t;
  return rc;
}

size_t trp_ntt_passes(unsigned log_n) { return log_n == 0 ? 1 : (log_n + S_MAX - 1) / S_MAX; }

int trp_ntt_impl(trp_ctx* ctx, int field, const void* d_src, void* d_dst, size_t batch, unsigned log_n,
                 const uint64_t omega[4], size_t src_stride, size_t dst_stride, unsigned n_src, const void* d_pre,
                 unsigned pre_period, const void* d_post, unsigned post_period, unsigned n_dst, void* d_tmp,
                 const void* const* d_src_tab) {
  if (field == 0)
    return ntt_run<FpParams>(ctx, d_src, d_dst, batch, log_n, omega, src_stride, dst_stride, n_src, d_pre, pre_period,
                             d_post, post_period, n_dst, d_tmp, d_src_tab);
  return ntt_run<FqParams>(ctx, d_src, d_dst, batch, log_n, omega, src_stride, dst_stride, n_src, d_pre, pre_period,
                           d_post, post_period, n_dst, d_tmp, d_src_tab);
}

// ---- elementwise glue kernels (K7) ------------------------------------------------------------------------
namespace {
template <class PR>
__global__ void field_op_kernel(int op, const uint4* a, const uint4* b, uint4* out, size_t n) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const bool bcast = op >= 16;          // op | 16: b is ONE element applied to every a[i]
  op &= 15;
  Fe<PR> x = fe_load<PR>(a + 2 * i), y = b ? fe_load<PR>(b + (bcast ? 0 : 2 * i)) : fe_zero<PR>(), r;
  switch (op) {
    case 0: r = fe_add(x, y); break;
    case 1: r = fe_sub(x, y); break;
    case 2: r = fe_mul(x, y); break;
    case 3: r = fe_inv(x); break;
    default: r = fe_sqr(x);
  }
  fe_store(out + 2 * i, r);
}
}  // namespace

int trp_field_op_impl(trp_ctx* ctx, int field, int op, const void* d_a, const void* d_b, void* d_out, size_t n) {
  if (n == 0) return TRP_OK;
  unsigned blocks = (unsigned)((n + 127) / 128);
  if (field == 0) field_op_kernel<FpParams><<<blocks, 128, 0, ctx->stream>>>(op, (const uint4*)d_a, (const uint4*)d_b, (uint4*)d_out, n);
  else field_op_kernel<FqParams><<<blocks, 128, 0, ctx->stream>>>(op, (const uint4*)d_a, (const uint4*)d_b, (uint4*)d_out, n);
  TRP_LAUNCHED(ctx);
  return TRP_OK;
}
