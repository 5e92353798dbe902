// Shared host-side plumbing for the C ABI: context, error reporting, workspace arena, launch accounting.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/tr_prover.h"
#include "ff.cuh"

struct TwiddleTable {
  unsigned log_n;        // table holds omega^i for i < 2^(log_n-1)
  uint64_t omega[4];
  void* d_tab;
};

// optional per-phase device timing (CUDA events on the ctx stream); used by bench.py for the live roofline number
enum ProfPhase { PROF_MSM_SORT = 0, PROF_MSM_ACCUM_L1, PROF_MSM_LEVELS, PROF_MSM_REDUCE, PROF_NTT_PASS, PROF_QUOTIENT, PROF_PRODUCTS, PROF_LOOKUP_SORT, PROF_NPHASES };
struct ProfSpan { int phase; cudaEvent_t e0, e1; double work; };

struct trp_ctx {
  bool prof_on = false;
  std::vector<ProfSpan> prof_spans;
  std::vector<cudaEvent_t> prof_pool;
  double prof_ms[PROF_NPHASES] = {};
  uint64_t prof_count[PROF_NPHASES] = {};
  double prof_work[PROF_NPHASES] = {};    // algorithmic units of the timed spans (ntt: butterflies; msm level 1: sorted entries' upper bound; quotient: rows)
  int device = 0;
  int curve = 0;
  cudaStream_t own_stream = nullptr;
  cudaStream_t stream = nullptr;
  // host->device staging runs on its own stream so that uploads overlap the kernels of the previous chunk
  cudaStream_t copy_stream = nullptr;
  cudaEvent_t copy_ev[3] = {nullptr, nullptr, nullptr};
  std::string err;
  std::mutex mu;
  uint64_t launches = 0;
  int sm_count = 148;
  // scratch arena (grown on demand, never shrunk)
  void* ws = nullptr;
  size_t ws_bytes = 0;
  // small pinned staging buffer for results
  void* pinned = nullptr;
  size_t pinned_bytes = 0;
  std::vector<TwiddleTable> twiddles;
  // quotient.cu: the caller's last few quotient programs and their lowered forms (qlower.h), most recent first; a prover runs
  // one program per constraint degree on each coset it needs, the same programs proof after proof
  struct QProgram {
    std::vector<uint32_t> src, low;
    unsigned src_regs = 0, low_regs = 0;
    size_t src_consts = 0;
  };
  std::vector<QProgram> q_progs;
  std::vector<uint32_t> q_staged;
};

struct trp_bases {
  trp_ctx* ctx;
  size_t n;
  void* d_xy;   // n x 64 B affine
};

struct trp_domain {
  trp_ctx* ctx;
  int field;
  unsigned k, j, ext_k;
  uint64_t omega[4], omega_inv[4], ext_omega[4], ext_omega_inv[4], g_coset[4], g_coset_inv[4];
  // device tables (Montgomery field elements)
  void* d_tabs;        // one allocation holding the tables below
  void* d_zeta_in;     // [1, zeta, zeta^2]
  void* d_l2c_post;    // [2^-k]
  void* d_e2c_post;    // 2^-ext_k * [1, zeta^-1, zeta^-2]
  void* d_tinv;        // 1 / (X^n - 1) on the coset, period 2^(ext_k - k)
  unsigned t_period;
  uint64_t coset_gen[64][4];   // zeta * ext_omega^j, j < 2^(ext_k - k) (generator of the j-th size-n coset)
};

#define TRP_FAIL(ctx, code, ...)                              \
  do {                                                        \
    char _buf[512];                                           \
    snprintf(_buf, sizeof(_buf), __VA_ARGS__);                \
    (ctx)->err = _buf;                                        \
    return (code);                                            \
  } while (0)

#define TRP_CUDA(ctx, expr)                                                                          \
  do {                                                                                               \
    cudaError_t _e = (expr);                                                                         \
    if (_e != cudaSuccess) {                                                                         \
      int _code = (_e == cudaErrorMemoryAllocation) ? TRP_E_OOM : TRP_E_CUDA;                        \
      TRP_FAIL(ctx, _code, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
    }                                                                                                \
  } while (0)

#define TRP_TRY(expr)            \
  do {                           \
    int _rc = (expr);            \
    if (_rc != TRP_OK) return _rc; \
  } while (0)

// check the launch that was just issued
#define TRP_LAUNCHED(ctx)                      \
  do {                                         \
    (ctx)->launches++;                         \
    TRP_CUDA(ctx, cudaGetLastError());         \
  } while (0)

struct ProfScope {
  trp_ctx* ctx; int idx;
  ProfScope(trp_ctx* c, int phase, double work = 0) : ctx(c), idx(-1) {
    if (!c->prof_on) return;
    ProfSpan s; s.phase = phase; s.work = work;
    for (cudaEvent_t* e : {&s.e0, &s.e1}) {
      if (!c->prof_pool.empty()) { *e = c->prof_pool.back(); c->prof_pool.pop_back(); }
      else cudaEventCreate(e);
    }
    cudaEventRecord(s.e0, c->stream);
    c->prof_spans.push_back(s);
    idx = (int)c->prof_spans.size() - 1;
  }
  ~ProfScope() { if (idx >= 0) cudaEventRecord(ctx->prof_spans[idx].e1, ctx->stream); }
};
// fold finished spans into the per-phase totals (synchronises the stream)
inline void trp_prof_collect(trp_ctx* ctx) {
  if (ctx->prof_spans.empty()) return;
  cudaStreamSynchronize(ctx->stream);
  for (auto& s : ctx->prof_spans) {
    float ms = 0;
    if (cudaEventElapsedTime(&ms, s.e0, s.e1) == cudaSuccess) { ctx->prof_ms[s.phase] += ms; ctx->prof_count[s.phase]++; ctx->prof_work[s.phase] += s.work; }
    ctx->prof_pool.push_back(s.e0); ctx->prof_pool.push_back(s.e1);
  }
  ctx->prof_spans.clear();
}

// grow-only scratch arena
inline int trp_ws_reserve(trp_ctx* ctx, size_t bytes) {
  if (bytes <= ctx->ws_bytes) return TRP_OK;
  if (ctx->ws) {
    TRP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    TRP_CUDA(ctx, cudaFree(ctx->ws));
    ctx->ws = nullptr; ctx->ws_bytes = 0;
  }
  size_t want = bytes + (bytes >> 3);
  cudaError_t e = cudaMalloc(&ctx->ws, want);
  if (e != cudaSuccess) { want = bytes; e = cudaMalloc(&ctx->ws, want); }
  if (e != cudaSuccess) { cudaGetLastError(); TRP_FAIL(ctx, TRP_E_OOM, "workspace allocation of %zu bytes failed: %s", want, cudaGetErrorString(e)); }
  ctx->ws_bytes = want;
  return TRP_OK;
}

// bump allocator over the arena (256-byte aligned)
struct WsCursor {
  char* base; size_t off; size_t cap;
  template <class T> T* take(size_t count) {
    size_t bytes = (count * sizeof(T) + 255) & ~(size_t)255;
    T* p = reinterpret_cast<T*>(base + off);
    off += bytes;
    return p;
  }
};
inline size_t ws_align(size_t b) { return (b + 255) & ~(size_t)255; }

// entry points implemented per translation unit
int trp_ntt_impl(trp_ctx* ctx, int field, const void* d_src, void* d_dst, size_t batch, unsigned log_n,
                 const uint64_t omega[4], size_t src_stride, size_t dst_stride, unsigned n_src,
                 const void* d_pre, unsigned pre_period, const void* d_post, unsigned post_period, unsigned n_dst,
                 void* d_tmp /* batch*2^log_n elements, needed iff src==dst and passes>1 */,
                 const void* const* d_src_tab = nullptr /* DEVICE table of batch column addresses read instead of d_src */);
size_t trp_ntt_passes(unsigned log_n);
int trp_get_powers(trp_ctx* ctx, int field, unsigned log_n, const uint64_t g[4], const void** out);
int trp_msm_impl(trp_ctx* ctx, const trp_bases* bases, const void* d_scalars, size_t n, size_t m, void* d_out_jac,
                 void* ws, size_t ws_bytes);
size_t trp_msm_ws_bytes(const trp_bases* bases, size_t n, size_t m);
int trp_points_sum_impl(trp_ctx* ctx, const void* d_jac, size_t g, void* d_out);
int trp_points_progression_impl(trp_ctx* ctx, const uint64_t* p0, const uint64_t* d, size_t n, void* d_out);
size_t trp_points_prefix_ws_bytes(size_t n);
int trp_points_prefix_sum_impl(trp_ctx* ctx, const void* d_in, size_t n, void* d_out, void* ws);
int trp_bases_create(trp_ctx* ctx, const void* src, bool src_on_device, size_t n, int flags, trp_bases** out);
void trp_bases_destroy(trp_bases* b);
int trp_bases_info(const trp_bases* b, unsigned* c, unsigned* W, unsigned* precomp);
int trp_field_op_impl(trp_ctx* ctx, int field, int op, const void* d_a, const void* d_b, void* d_out, size_t n);
int trp_microbench_impl(trp_ctx* ctx, int kind, int iters, double* out_gops);
// products.cu (row f1): out = mul / a with zeros kept; z[0] = init, z[i] = z[i-1] * v[i-1]; fused permutation / lookup Z columns
int trp_batch_invert_impl(trp_ctx* ctx, int field, const void* d_a, const void* d_mul, void* d_out, size_t n);
size_t trp_grand_product_ws_bytes(size_t n_out);
int trp_grand_product_impl(trp_ctx* ctx, int field, const void* d_v, size_t n_in, const void* d_init, void* d_z, size_t n_out, void* d_tiles);
size_t trp_product_ws_bytes(size_t n);
int trp_permutation_product_impl(trp_domain* d, const uint64_t* const* d_values, const uint64_t* const* d_sigmas, size_t m,
                                 const uint64_t* consts_host, const void* d_last_z, void* d_z, void* ws);
int trp_lookup_product_impl(trp_domain* d, const void* d_a, const void* d_s, const void* d_ap, const void* d_sp,
                            const uint64_t* consts_host, void* d_z, size_t n_out, void* ws);
int trp_suffix_sum_impl(trp_ctx* ctx, int field, void* d_a, size_t n, void* d_tiles);
// ipa.cu (row f2): evaluations, inner products, Kate division, IPA round folding; msm.cu: MSM over caller-owned bases
size_t trp_reduce_ws_bytes(trp_ctx* ctx, size_t n, size_t m);
int trp_lincomb_impl(trp_ctx* ctx, int field, const void* const* d_ptrs, const void* d_scal, size_t m, size_t n, void* d_out);
int trp_eval_polys_impl(trp_ctx* ctx, int field, const void* d_polys, size_t stride, const void* const* d_ptrs, size_t n, size_t m,
                        const uint64_t x[4], void* d_out, void* ws);
int trp_inner_products_impl(trp_ctx* ctx, int field, const void* d_a, size_t a_stride, const void* d_b, size_t b_stride, size_t n, size_t m,
                            void* d_out, void* ws);
int trp_fold_impl(trp_ctx* ctx, int field, void* d_a, size_t half, const uint64_t u[4]);
int trp_ipa_round_scalars_impl(trp_ctx* ctx, int field, const void* d_p, const void* d_s, unsigned cur_log, size_t lo, size_t count,
                                size_t col_stride, void* d_out);
int trp_ipa_s_double_impl(trp_ctx* ctx, int field, const void* d_s, size_t m, const uint64_t u[4], void* d_out);
int trp_powers_impl(trp_ctx* ctx, int field, const uint64_t x[4], size_t n, void* d_out);
size_t trp_kate_ws_bytes(size_t n);
int trp_kate_division_impl(trp_ctx* ctx, int field, const void* d_coeffs, size_t n, const uint64_t b[4], const uint64_t b_inv[4],
                           int b_is_zero, void* d_q, void* ws);
size_t trp_collapse_ws_bytes(size_t half);
int trp_generator_collapse_impl(trp_ctx* ctx, void* d_g, size_t half, const uint64_t u_canonical[4], void* ws);
size_t trp_msm_var_ws_bytes(size_t n, size_t m);
int trp_msm_var_impl(trp_ctx* ctx, const void* d_bases, const void* d_scalars, size_t n, size_t m, void* d_out_jac, void* ws, size_t ws_bytes);
// lookup.cu (row f1): permute_expression_pair
size_t trp_permute_pair_ws_bytes(size_t rows);
int trp_permute_pair_impl(trp_ctx* ctx, int field, const void* d_input, const void* d_table, size_t rows, void* d_perm_input,
                          void* d_perm_table, void* ws, int* all_found);

// field ids used internally: 0 = Fp, 1 = Fq
inline int scalar_field_of(int curve) { return curve == TRP_CURVE_PALLAS ? 1 : 0; }
inline int base_field_of(int curve) { return curve == TRP_CURVE_PALLAS ? 0 : 1; }
