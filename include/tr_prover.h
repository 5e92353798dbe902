/* tr_prover.h -- C ABI of the B200 (sm_100a) backend for the data-parallel core of the halo2/IPA prover
 * that proves the TinyRAM circuit of Orbis-Tertius/tiny-ram-halo2.
 *
 * The reference crate has no FFI of its own: it reaches the prover through halo2_proofs' free functions and
 * EvaluationDomain methods (un-vendored dependency halo2_proofs 0.2.0 @ a95945254dcc, /root/reference/Cargo.lock:619-621),
 * called from /root/reference/src/test_utils.rs:21-49 (Params::new, keygen_vk/pk, create_proof).  Each entry point
 * below names the halo2_proofs routine it stands in for; INTEGRATION.md shows the Rust-side binding.
 *
 * Conventions
 *   status      0 = ok, < 0 = error (TRP_E_*); message via trp_last_error(ctx).  Never aborts, never throws.
 *   field elem  uint64_t[4], little-endian limbs, MONTGOMERY form (exactly what pasta_curves' Fp/Fq hold in
 *               memory), value < modulus.
 *   affine pt   { uint64_t x[4]; uint64_t y[4]; } Montgomery; the identity is encoded as x = y = 0.
 *   jacobian pt { x[4], y[4], z[4] } Montgomery; identity <=> z = 0.  Results are returned NORMALISED
 *               (z = 1 in Montgomery form, or x = y = z = 0): a valid Jacobian representative whose affine
 *               form / 32-byte encoding is the unique group element the CPU prover computes.
 *   curve       0 = Pallas (coordinates Fp, scalars Fq), 1 = Vesta (coordinates Fq, scalars Fp).  The
 *               reference proves over Fp and commits on Vesta (src/test_utils.rs:2,12,21,40) => curve = 1.
 *               NTT / domain entry points work over the curve's SCALAR field.
 *   ownership   caller owns all host buffers; the library owns device memory behind handles.
 *   threading   a ctx is bound to one device and one stream; calls on one ctx are serialised internally;
 *               distinct ctxs are independent.
 *   host/dev    trp_*      take HOST pointers (copies inside the call, synchronous);
 *               trp_dev_*  take DEVICE pointers, enqueue on the ctx stream and return without synchronising
 *               (results are valid after trp_ctx_sync or stream synchronisation).
 */
#ifndef TR_PROVER_H
#define TR_PROVER_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TRP_OK 0
#define TRP_E_INVALID (-1)   /* bad argument / size mismatch (halo2 would panic on assert_eq!) */
#define TRP_E_CUDA (-2)      /* CUDA runtime error */
#define TRP_E_OOM (-3)       /* device allocation failed */
#define TRP_E_NODEVICE (-4)  /* no usable CUDA device: there is no CPU fallback */

#define TRP_CURVE_PALLAS 0
#define TRP_CURVE_VESTA 1

typedef struct trp_ctx trp_ctx;
typedef struct trp_bases trp_bases;
typedef struct trp_domain trp_domain;

/* ---- context ------------------------------------------------------------------------------------------ */
int trp_ctx_create(trp_ctx** out, int device, int curve);
void trp_ctx_destroy(trp_ctx* ctx);
const char* trp_last_error(const trp_ctx* ctx);
/* Use an externally owned CUDA stream (cudaStream_t passed as void*); NULL restores the ctx's own stream. */
int trp_ctx_set_stream(trp_ctx* ctx, void* cuda_stream);
int trp_ctx_sync(trp_ctx* ctx);
/* number of kernels this ctx has launched so far (bench.py's gpu_launches) */
uint64_t trp_ctx_launch_count(const trp_ctx* ctx);
const char* trp_version(void);
/* Per-phase device timing with CUDA events on the ctx stream (off by default; a few microseconds per span).
 * phase: 0 msm hist+scan+scatter, 1 msm bucket accumulation level 1 (the dominant kernel), 2 msm upper
 * reduction levels, 3 msm bucket reduce + final, 4 ntt pass kernels, 5 quotient VM kernel, 6 batch inversion / grand product /
 * lookup permutation kernels, 7 lookup radix sort.
 * trp_prof_get synchronises the stream. */
int trp_prof_enable(trp_ctx* ctx, int on);
int trp_prof_reset(trp_ctx* ctx);
int trp_prof_get(trp_ctx* ctx, int phase, double* total_ms, uint64_t* count);
/* algorithmic work of the spans timed so far: phase 4 = radix-2 butterflies (columns x N/2 x stages of every pass launched),
 * phase 1 = bucket additions if no digit were zero (n x windows x columns), phase 5 = rows evaluated by the quotient program */
int trp_prof_get_work(trp_ctx* ctx, int phase, double* work);

/* ---- MSM: halo2_proofs::arithmetic::best_multiexp(coeffs, bases) -> C::Curve ---------------------------
 * and poly::commitment::Params::{commit, commit_lagrange} which append blind * w and call it.
 * Bases (Params.g / Params.g_lagrange ++ [w]) are uploaded once and reused by hundreds of MSMs.            */
int trp_bases_load(trp_ctx* ctx, const uint64_t* affine_xy /* n x 8 */, size_t n, trp_bases** out);
int trp_dev_bases_load(trp_ctx* ctx, const uint64_t* d_affine_xy, size_t n, trp_bases** out);
/* flags: bit 0 = keep one bucket set per window (no precomputed table), bit 1 = force the precomputed
 * table of 2^(c*w) * P_i multiples (default: precompute when the table fits the memory budget), bits 8..15 = window width c
 * (0 = the library's choice for n).  The same bases may be loaded more than once with different widths: a prover whose columns
 * are mostly zero (TinyRAM advice: 2^16 assigned rows of 2^20) wants a narrow table for those and a wide one for dense columns. */
int trp_bases_load_ex(trp_ctx* ctx, const uint64_t* affine_xy, size_t n, int flags, trp_bases** out);
int trp_dev_bases_load_ex(trp_ctx* ctx, const uint64_t* d_affine_xy, size_t n, int flags, trp_bases** out);
size_t trp_bases_len(const trp_bases* b);
/* out = { window bits c, number of windows, 1 if the multiples were precomputed } */
int trp_bases_describe(const trp_bases* b, unsigned out[3]);
void trp_bases_free(trp_bases* b);
/* sum_i scalars[i] * bases[i], i < n <= len(bases) (a prefix of the loaded bases).  n = 0 gives the identity. */
int trp_msm(trp_ctx* ctx, const trp_bases* bases, const uint64_t* scalars /* n x 4 */, size_t n,
            uint64_t out_jacobian[12]);
/* m independent MSMs over the same bases; scalars is m contiguous columns of n. */
int trp_msm_batch(trp_ctx* ctx, const trp_bases* bases, const uint64_t* scalars /* m x n x 4 */, size_t n,
                  size_t m, uint64_t* out_jacobian /* m x 12 */);
int trp_dev_msm_batch(trp_ctx* ctx, const trp_bases* bases, const uint64_t* d_scalars, size_t n, size_t m,
                      uint64_t* d_out_jacobian /* m x 12, device */);

/* Sum of g group elements (Jacobian in, normalised Jacobian out).  Combines the per-GPU partial sums when one MSM's point
 * range is split across devices -- the same final step best_multiexp performs over its per-thread partial results. */
int trp_points_sum(trp_ctx* ctx, const uint64_t* jacobian /* g x 12 */, size_t g, uint64_t out_jacobian[12]);
int trp_dev_points_sum(trp_ctx* ctx, const uint64_t* d_jacobian, size_t g, uint64_t* d_out_jacobian);

/* Synthetic input generator for benchmarks and large tests: d_out[i] = P0 + i*D as affine points in DEVICE
 * memory (SURVEY.md 8(d) config 2: an arithmetic progression of random multiples of the generator). */
int trp_dev_points_progression(trp_ctx* ctx, const uint64_t p0[8], const uint64_t d[8], size_t n, uint64_t* d_out);

/* Inclusive prefix sums of n affine points in DEVICE memory: d_out[j] = d_in[0] + ... + d_in[j] (affine; may alias d_in).
 * Summation by parts turns a commitment into one over these sums: sum_i z_i G_i = sum_j (z_j - z_{j+1}) Q_j (z_n = 0), and the
 * difference column is SPARSE whenever z rarely changes from row to row -- halo2's grand-product columns (permutation::Argument::
 * commit, lookup::Permuted::commit_product) stay constant over the rows a circuit does not use.  Same group element, so
 * Params::commit_lagrange's result is unchanged; the prover builds Q once per parameter set and commits such columns through
 * its sparse path. */
int trp_dev_points_prefix_sum(trp_ctx* ctx, const uint64_t* d_in, size_t n, uint64_t* d_out);

/* ---- NTT: halo2_proofs::arithmetic::best_fft(a, omega, log_n) (field instance) -------------------------
 * In place, natural order in and out: a[k] <- sum_j a[j] * omega^(j k); batch contiguous vectors of 2^log_n. */
int trp_ntt(trp_ctx* ctx, uint64_t* a, size_t batch, unsigned log_n, const uint64_t omega[4]);
int trp_dev_ntt(trp_ctx* ctx, uint64_t* d_a, size_t batch, unsigned log_n, const uint64_t omega[4]);

/* ---- EvaluationDomain: halo2_proofs::poly::EvaluationDomain::new(j, k) and its transforms ---------------- */
int trp_domain_create(trp_ctx* ctx, unsigned k, unsigned j, trp_domain** out);
void trp_domain_free(trp_domain* d);
unsigned trp_domain_extended_k(const trp_domain* d);
/* omega, extended_omega, g_coset (zeta), g_coset_inv as Montgomery limbs: out[4][4] */
int trp_domain_constants(const trp_domain* d, uint64_t out[16]);
/* lagrange_to_coeff: iNTT with omega^-1 then * 2^-k; batch columns of n = 2^k, in place */
int trp_lagrange_to_coeff(trp_domain* d, uint64_t* cols, size_t batch);
int trp_dev_lagrange_to_coeff(trp_domain* d, uint64_t* d_cols, size_t batch);
/* coeff_to_lagrange: plain NTT with omega (EvaluationDomain::coeff_to_lagrange is not in 0.2.0; used by tests) */
int trp_coeff_to_lagrange(trp_domain* d, uint64_t* cols, size_t batch);
/* coeff_to_extended: a[i] *= zeta^(i mod 3), zero-pad to 2^extended_k, NTT with extended_omega */
int trp_coeff_to_extended(trp_domain* d, const uint64_t* coeff /* batch x n */, uint64_t* ext /* batch x 2^ext_k */,
                          size_t batch);
int trp_dev_coeff_to_extended(trp_domain* d, const uint64_t* d_coeff, uint64_t* d_ext, size_t batch);
/* extended_to_coeff (optionally preceded by divide_by_vanishing_poly): ext is consumed (overwritten);
 * out_coeff receives n * (j - 1) coefficients. */
int trp_extended_to_coeff(trp_domain* d, uint64_t* ext /* 2^ext_k */, uint64_t* out_coeff /* n*(j-1) */,
                          int divide_by_vanishing);
int trp_dev_extended_to_coeff(trp_domain* d, uint64_t* d_ext, uint64_t* d_out_coeff, int divide_by_vanishing);

/* ---- quotient evaluation: halo2_proofs::poly::Evaluator::evaluate(&ast, domain) (poly/evaluator.rs) as driven by
 * plonk::vanishing::Argument::construct in create_proof: h_ext[r] = sum_j y^j expr_j(row r) over the extended domain.
 * The caller lowers its poly::Ast into a straight-line program over n_regs virtual registers (field elements);
 * an instruction is 4 x uint32 { op, dst, a, b }:
 *    0 LOAD   dst = cols[a][(row + (int32)b * step) mod rows]      (Ast::Poly(leaf).with_rotation(b), |b| <= 32767)
 *    1 CONST  dst = consts[a]                                       (Ast::ConstantTerm)
 *    2 ADD  3 SUB  4 MUL   dst = r[a] op r[b]                       (Ast::Add / Ast::Mul)
 *    5 NEG  6 SQR  7 DBL   dst = op r[a]
 *    8 COSETX dst = zeta * extended_omega^row                       (Ast::LinearTerm(1): the value of X at this row)
 *    9 STORE  out[row] = r[a]
 *   10 MULC 11 ADDC 12 SUBC  dst = r[a] op consts[b]                (Ast::Scale and friends)
 * coset = -1: rows = the whole extended domain; columns hold 2^extended_k values, step = 2^(extended_k - k).
 * coset = j >= 0: rows = the j-th size-n coset (zeta * extended_omega^j * <omega>); columns hold the n values
 *   produced by trp_dev_coeff_to_coset(.., j), step = 1, and results go to d_out[row * 2^(extended_k-k) + j], so
 *   2^(extended_k-k) calls fill h_ext without materialising any extended column.
 * Malformed programs are rejected with TRP_E_INVALID before anything is launched.  The format above is the ABI and may be as naive
 * as a post-order walk of the Ast emits it: the library rewrites the program before launch (csrc/qlower.h, cached per ctx: leaf loads
 * folded into their consumer, x + (-y) -> x - y, the value of X computed once, results forwarded through an accumulator) and
 * stores exactly the values the program above defines. */
int trp_dev_quotient_eval(trp_domain* d, const uint32_t* program /* host */, size_t n_instr, unsigned n_regs,
                          const uint64_t* consts /* host, n_consts x 4 */, size_t n_consts,
                          const uint64_t* const* d_cols /* host array of n_cols DEVICE pointers */, size_t n_cols,
                          int coset, uint64_t* d_out /* device, 2^extended_k x 4 */);
/* The same over a SLICE of a coset's rows (SURVEY.md 8(e) item 3 refined: a coset's rows are split between the GPUs so that j - 1
 * cosets load any number of devices evenly): the columns hold rows [row0 - halo_before, row0 + nrows + halo_after) of coset j
 * (cyclic neighbours included by the caller), rotations must stay within the halo, d_out receives the nrows results contiguously. */
int trp_dev_quotient_eval_rows(trp_domain* d, const uint32_t* program, size_t n_instr, unsigned n_regs, const uint64_t* consts,
                               size_t n_consts, const uint64_t* const* d_cols, size_t n_cols, unsigned coset, size_t row0, size_t nrows,
                               unsigned halo_before, unsigned halo_after, uint64_t* d_out /* device, nrows x 4 */);
int trp_quotient_eval(trp_domain* d, const uint32_t* program, size_t n_instr, unsigned n_regs, const uint64_t* consts,
                      size_t n_consts, const uint64_t* const* cols /* n_cols HOST pointers, 2^extended_k x 4 each */,
                      size_t n_cols, uint64_t* out_ext /* host, 2^extended_k x 4 */);
/* out[i] = p(zeta * extended_omega^(j + i * 2^(extended_k-k))) for coefficient-form columns p (n each): row j, j + 2^(..),
 * ... of coeff_to_extended, computed with ONE size-n NTT per column. */
int trp_dev_coeff_to_coset(trp_domain* d, const uint64_t* d_coeff, uint64_t* d_out, size_t batch, unsigned coset);
/* The same for columns anywhere in device memory: d_src_tab is a DEVICE array of batch column addresses, column i's values go
 * to d_out[i * n ..] (which must not overlap a source).  Expands a subset of a prover's columns with no staging copy. */
int trp_dev_coeff_to_coset_gather(trp_domain* d, const uint64_t* const* d_src_tab, uint64_t* d_out, size_t batch, unsigned coset);
/* OR into trp_dev_quotient_eval's coset index: write the coset's n results contiguously at d_out[row] instead of
 * interleaving them into the extended vector (input layout of trp_dev_cosets_to_coeff). */
#define TRP_Q_CONTIGUOUS 0x10000
/* Coefficients of a polynomial of degree < n * ncos from its values on the first ncos cosets (d_vals: ncos x n, coset i
 * at d_vals[i * n ..]; consumed).  With divide_by_vanishing the values are first divided by X^n - 1.  Equals
 * extended_to_coeff(divide_by_vanishing_poly(h_ext)) while only ncos = j - 1 of the 2^(extended_k - k) cosets are ever
 * evaluated: the quotient h(X) is unique, so commitments and proof bytes are unchanged. */
int trp_dev_cosets_to_coeff(trp_domain* d, uint64_t* d_vals, unsigned ncos, uint64_t* d_out_coeff, int divide_by_vanishing);
/* The same for h = sum_p h_p given part by part, deg h_p < n * ncos[p] <= n * ncos_out: part p brings its values on the first
 * ncos[p] cosets (d_vals: the parts' rows back to back, sum_p ncos[p] x n; consumed), the ncos_out x n coefficients of h are
 * written to d_out_coeff.  A quotient numerator split by constraint degree is evaluated only on the cosets each part needs;
 * h is unique, so the result equals trp_dev_cosets_to_coeff of the whole numerator on ncos_out cosets.  1 <= n_parts <= 64. */
int trp_dev_cosets_to_coeff_parts(trp_domain* d, uint64_t* d_vals, const unsigned* ncos /* host, n_parts */, unsigned n_parts,
                                  unsigned ncos_out, uint64_t* d_out_coeff, int divide_by_vanishing);

/* ---- between the hot kernels (SURVEY.md 8(f) row f1): the grand products and the lookup permutation of create_proof -------
 * halo2_proofs 0.2.0 plonk/permutation/prover.rs (Argument::commit), plonk/lookup/prover.rs (Argument::commit_permuted,
 * Permuted::commit_product) and ff::BatchInvert.  which_field as in trp_field_op (0 = scalar field of the ctx's curve).
 * Blinding rows are the caller's (its RNG): overwrite the tail of z / the permuted columns after the call.              */
/* out[i] = mul[i] / a[i] (d_mul == NULL: 1 / a[i]); a[i] == 0 gives 0, as ff::BatchInvert leaves zeros alone.  out may alias a. */
int trp_dev_batch_invert(trp_ctx* ctx, int which_field, const uint64_t* d_a, const uint64_t* d_mul, uint64_t* d_out, size_t n);
int trp_batch_invert(trp_ctx* ctx, int which_field, uint64_t* a /* in place */, size_t n);
/* z[0] = init (NULL: 1), z[i] = z[i-1] * v[i-1] for i < n_out <= n_in + 1.  z may alias v. */
int trp_dev_grand_product(trp_ctx* ctx, int which_field, const uint64_t* d_v, size_t n_in, const uint64_t* d_init /* device, 1 elem */,
                          uint64_t* d_z, size_t n_out);
int trp_grand_product(trp_ctx* ctx, int which_field, const uint64_t* v, size_t n_in, const uint64_t init[4], uint64_t* z, size_t n_out);
/* One chunk (m <= 16 columns; halo2 uses cs_degree - 2) of permutation::Argument::commit: z[0] = last_z (NULL: 1),
 *   z[r+1] = z[r] * prod_c (v_c[r] + delta_beta[c] * omega^r + gamma) / prod_c (v_c[r] + beta * sigma_c[r] + gamma),  r + 1 < n,
 * delta_beta[c] = beta * DELTA^(index of column c in the whole argument).  d_last_z is a DEVICE pointer so that chunks chain
 * without a host round trip (pass &z_prev[n - (blinding_factors + 1)]). */
int trp_dev_permutation_product(trp_domain* d, const uint64_t* const* d_values /* host array of m device ptrs */,
                                const uint64_t* const* d_sigmas, size_t m, const uint64_t beta[4], const uint64_t gamma[4],
                                const uint64_t* delta_beta /* m x 4 */, const uint64_t* d_last_z, uint64_t* d_z /* n */);
int trp_permutation_product(trp_domain* d, const uint64_t* const* values, const uint64_t* const* sigmas, size_t m,
                            const uint64_t beta[4], const uint64_t gamma[4], const uint64_t* delta_beta, const uint64_t last_z[4],
                            uint64_t* z);
/* lookup::Permuted::commit_product: z[0] = 1, z[r+1] = z[r] * (a[r] + beta)(s[r] + gamma) / ((a'[r] + beta)(s'[r] + gamma)),
 * r + 1 < n_out <= n; a, s = compressed input / table expressions, a', s' = their permuted forms (all n values). */
int trp_dev_lookup_product(trp_domain* d, const uint64_t* d_input, const uint64_t* d_table, const uint64_t* d_perm_input,
                           const uint64_t* d_perm_table, const uint64_t beta[4], const uint64_t gamma[4], uint64_t* d_z, size_t n_out);
int trp_lookup_product(trp_domain* d, const uint64_t* input, const uint64_t* table, const uint64_t* perm_input,
                       const uint64_t* perm_table, const uint64_t beta[4], const uint64_t gamma[4], uint64_t* z, size_t n_out);
/* lookup::prover::permute_expression_pair over the first `rows` (= usable) rows of the compressed input / table expressions
 * (scalar field): perm_input = input sorted by canonical value; perm_table[r] = perm_input[r] at every first occurrence,
 * the left-over table values (ascending) fill the repeated rows from the end.  *all_found = 0 when some input value is
 * absent from the table (halo2 returns Error::ConstraintSystemFailure).  Synchronises the ctx stream. */
int trp_dev_permute_expression_pair(trp_ctx* ctx, const uint64_t* d_input, const uint64_t* d_table, size_t rows,
                                    uint64_t* d_perm_input, uint64_t* d_perm_table, int* all_found);
int trp_permute_expression_pair(trp_ctx* ctx, const uint64_t* input, const uint64_t* table, size_t rows, uint64_t* perm_input,
                                uint64_t* perm_table, int* all_found);

/* ---- opening phase (SURVEY.md 8(f) row f2): halo2_proofs 0.2.0 arithmetic.rs {eval_polynomial, compute_inner_product,
 * kate_division, parallel_generator_collapse} and the round body of poly/commitment/prover.rs create_proof (the IPA) ------- */
/* out[j] = sum_i polys[j * stride + i] * x^i, i < n, for j < m: m evaluations at ONE point (the evaluations at x * omega^rot) */
int trp_dev_eval_polynomials(trp_ctx* ctx, int which_field, const uint64_t* d_polys, size_t stride, size_t n, size_t m,
                             const uint64_t x[4], uint64_t* d_out /* m x 4 */);
/* the same for m polynomials that live in separate device buffers: d_poly_ptrs is a HOST array of m device pointers (the ~700
 * openings of create_proof are evaluations of separately allocated polynomials at four points: x, x*omega, x*omega^-1, x*omega^-(bf+1)) */
int trp_dev_eval_polynomials_at(trp_ctx* ctx, int which_field, const uint64_t* const* d_poly_ptrs, size_t n, size_t m, const uint64_t x[4],
                                uint64_t* d_out /* m x 4 */);
/* d_out[i] = sum_j scalars[j] * d_poly_ptrs[j][i], i < n: the random linear combinations of poly/multiopen/prover.rs (q_polys folded
 * with powers of x_1, the final polynomial with powers of x_4).  d_poly_ptrs: HOST array of m device pointers; scalars: HOST array
 * of m Montgomery field elements; d_out must not alias an input. */
int trp_dev_linear_combination(trp_ctx* ctx, int which_field, const uint64_t* const* d_poly_ptrs, const uint64_t* scalars, size_t n, size_t m,
                               uint64_t* d_out);
int trp_eval_polynomial(trp_ctx* ctx, int which_field, const uint64_t* coeffs, size_t n, const uint64_t x[4], uint64_t out[4]);
/* out[j] = <a_j, b_j>, vectors j at d_a + j * a_stride / d_b + j * b_stride elements (stride 0 = shared vector) */
int trp_dev_inner_products(trp_ctx* ctx, int which_field, const uint64_t* d_a, size_t a_stride, const uint64_t* d_b, size_t b_stride,
                           size_t n, size_t m, uint64_t* d_out);
int trp_compute_inner_product(trp_ctx* ctx, int which_field, const uint64_t* a, const uint64_t* b, size_t n, uint64_t out[4]);
/* d_out[i] = x^i, i < n  (the vector b of the inner-product argument) */
int trp_dev_powers(trp_ctx* ctx, int which_field, const uint64_t x[4], size_t n, uint64_t* d_out);
/* kate_division: q (n - 1 coefficients) = (p(X) - p(b)) / (X - b) for the n coefficients of p */
int trp_dev_kate_division(trp_ctx* ctx, int which_field, const uint64_t* d_coeffs, size_t n, const uint64_t b[4], uint64_t* d_q);
int trp_kate_division(trp_ctx* ctx, int which_field, const uint64_t* coeffs, size_t n, const uint64_t b[4], uint64_t* q);
/* IPA round: a[i] += a[i + half] * u, i < half  (p' with u^-1, b with u) */
int trp_dev_fold(trp_ctx* ctx, int which_field, uint64_t* d_a, size_t half, const uint64_t u[4]);
/* The IPA round without collapsing the generators: after j rounds G'_i = sum_t s_t G_{t cur + i} (cur = n / 2^j, s = the 2^j
 * products of the round challenges), so L_j = <p'_hi, G'_lo> and R_j = <p'_lo, G'_hi> are fixed-base MSMs over the ORIGINAL
 * generators with the scalars p'[.] * s_t.  Writes the two scalar columns for the base indices [lo, lo + count) (a rank's slice of
 * the generators when the point range is split between devices): d_out[b - lo] for L_j, d_out[col_stride + b - lo] for R_j.
 * d_p: the cur live entries of p'; d_s: n / cur entries. */
int trp_dev_ipa_round_scalars(trp_ctx* ctx, int which_field, const uint64_t* d_p, const uint64_t* d_s, size_t cur, size_t lo, size_t count,
                              size_t col_stride, uint64_t* d_out);
/* d_out[2 t] = d_s[t], d_out[2 t + 1] = d_s[t] * u, t < m: the s vector after a round with challenge u (d_out must not alias d_s) */
int trp_dev_ipa_s_double(trp_ctx* ctx, int which_field, const uint64_t* d_s, size_t m, const uint64_t u[4], uint64_t* d_out);
/* parallel_generator_collapse: g[i] = g[i] + [u] g[i + half], i < half, normalised affine points (identity = 0,0); u Montgomery */
int trp_dev_generator_collapse(trp_ctx* ctx, uint64_t* d_g /* 2 * half affine points */, size_t half, const uint64_t u[4]);
/* best_multiexp over caller-owned DEVICE bases (no precomputed table): the round MSMs over the collapsing G' */
int trp_dev_msm_var(trp_ctx* ctx, const uint64_t* d_bases /* n x 8 */, const uint64_t* d_scalars /* m x n x 4 */, size_t n, size_t m,
                    uint64_t* d_out_jacobian /* m x 12 */);

/* ---- parameter generation (SURVEY.md 8(f) row f3): halo2_proofs 0.2.0 poly::commitment::Params::new(k), reached from
 * /root/reference/src/test_utils.rs:21,89, and the pasta_curves 0.4.1 routines it calls (hashtocurve.rs, curves.rs) ----------- */
/* CurveExt::hash_to_curve(domain_prefix) of the ctx's curve ("pallas" / "vesta") applied to n messages: expand_message_xmd over
 * BLAKE2b-512, simplified SWU onto the iso-curve, sum of the two images, 3-isogeny.  Affine Montgomery results (identity = 0,0).
 * Device form: message i = msg_prefix ++ (append_index ? u32_le(first_index + i) : nothing) -- Params::new hashes
 * [0] ++ u32_le(i) for g[i], [1] for w and [2] for u.  Host form: n messages of msg_len bytes each. */
int trp_dev_hash_to_curve(trp_ctx* ctx, const char* domain_prefix, const uint8_t* msg_prefix /* host */, size_t prefix_len,
                          int append_index, uint64_t first_index, size_t n, uint64_t* d_out /* n x 8 */);
int trp_hash_to_curve(trp_ctx* ctx, const char* domain_prefix, const uint8_t* messages /* n x msg_len */, size_t msg_len, size_t n,
                      uint64_t* out /* n x 8 */);
/* arithmetic::best_fft instantiated over curve points (the `Group` instance Params::new uses for g -> g_lagrange): in place over
 * 2^log_n normalised affine points, natural order in and out, out[k] = sum_j [omega^(j k)] in[j]; omega (order 2^log_n) and the
 * optional scale (every output multiplied by it; NULL = none) are Montgomery elements of the curve's SCALAR field. */
int trp_dev_group_fft(trp_ctx* ctx, uint64_t* d_points /* 2^log_n x 8 */, unsigned log_n, const uint64_t omega[4], const uint64_t* scale);
int trp_group_fft(trp_ctx* ctx, uint64_t* points, unsigned log_n, const uint64_t omega[4], const uint64_t* scale);
/* Params::new(k): g[i] = hash_to_curve("Halo2-Parameters")([0] ++ u32_le(i)), g_lagrange = group iFFT of g (alpha^-1 =
 * ROOT_OF_UNITY_INV^(2^(S-k)), then * TWO_INV^k), w = hash([1]), u = hash([2]).  n = 2^k affine points each. */
int trp_params_new(trp_ctx* ctx, unsigned k, uint64_t* g, uint64_t* g_lagrange, uint64_t w[8], uint64_t u[8]);
int trp_dev_params_new(trp_ctx* ctx, unsigned k, uint64_t* d_g, uint64_t* d_g_lagrange, uint64_t* d_wu /* w then u: 2 x 8 */);

/* Bulk random field elements from a 32-byte key drawn from the caller's RNG: d_out[i] = Field::random over the byte stream
 * BLAKE2b-512(key ++ u64_le(first_counter + i)), i.e. pasta_curves' from_u512 of the 64-byte digest, Montgomery form.  The random
 * polynomials of create_proof (vanishing::Argument::commit, the IPA's S) draw 2^k scalars each from the caller's RNG in halo2; a
 * device-resident prover expands a seed here instead (deterministic, the same on every GPU of a multi-GPU proof). */
int trp_dev_random_field(trp_ctx* ctx, int which_field, const uint8_t key[32], uint64_t first_counter, size_t n, uint64_t* d_out);

/* ---- glue / debug: elementwise field kernels over the ctx's scalar (field=0) or base (field=1) field ----
 * op: 0 add, 1 sub, 2 mul, 3 inv(a), 4 sqr(a).  Host pointers.  Used by parity tests of K1 and by K7 callers. */
int trp_field_op(trp_ctx* ctx, int which_field, int op, const uint64_t* a, const uint64_t* b, uint64_t* out, size_t n);
/* device-pointer form; op | 16 broadcasts ONE element at d_b over d_a (e.g. multiply a column by R^2 to enter
 * Montgomery form, or by a challenge) */
int trp_dev_field_op(trp_ctx* ctx, int which_field, int op, const uint64_t* d_a, const uint64_t* d_b, uint64_t* d_out, size_t n);

/* ---- microbenchmarks used by bench.py to measure the integer-pipe roofline denominator -------------------
 * kind 0: independent 32x32+64 wide MACs with carry-out (IMAD.WIDE.U32 + carry count), 1: 32-bit IMAD,
 * 2: IADD3.X carry chains, 3: carry-chained wide MACs as in the field multiplier (IMAD.WIDE.U32.X; the wide-MAC peak),
 * 4: field mul, 5: field add/sub, 10: IMAD.WIDE + IADD3 mix, 11: DFMA.
 * Returns achieved G-ops/s in *out_gops (ops = wide MACs / thread-level instructions / field muls). */
int trp_microbench(trp_ctx* ctx, int kind, int iters, double* out_gops);

#ifdef __cplusplus
}
#endif
#endif /* TR_PROVER_H */
