// K6: extended-domain evaluation of the quotient polynomial's numerator,  h_ext[r] = sum_j y^j * expr_j(row r).
//
// Replaces halo2_proofs::poly::Evaluator::evaluate(&ast, domain) (poly/evaluator.rs, halo2_proofs 0.2.0 @ a95945254dcc,
// Cargo.lock:619-621) as driven by plonk::vanishing::Argument::construct inside create_proof
// (/root/reference/src/test_utils.rs:41,96).  The CPU routine interprets an `Ast<ExtendedLagrangeCoeff>` chunk by chunk
// on rayon threads; the expression set comes from the reference's gates and lookups (SURVEY.md Appendix B, e.g.
// /root/reference/src/circuits/sprod.rs:65-90).
//
// Here the host lowers the AST once into a straight-line program over a small virtual register file
// (tiny-ram-halo2_b200/poly.py) and ONE kernel runs it for every row: a thread owns a row, the virtual registers
// live in shared memory as two 16-byte planes ([reg][thread], conflict-free 128-bit accesses), column values are
// read with coalesced 32-byte loads at (row + rotation * step) mod rows.  The same kernel serves two data layouts:
//   * whole extended domain: columns hold 2^ext_k values, rotation step 2^(ext_k - k)            (what halo2 does)
//   * one size-n coset of it: columns hold n values produced by trp_dev_coeff_to_coset, step 1; the result is
//     written interleaved (row * 2^(ext_k-k) + coset) so that 2^(ext_k-k) calls assemble h_ext without ever
//     materialising the extended columns (700 columns x 256 MiB at k = 20 would not fit; SURVEY.md section 7).
#include "common.cuh"
#include "qlower.h"

#include <cstdlib>
#include <algorithm>
#include <cstring>

using namespace ff;

namespace {

enum QOp : uint32_t {
  Q_LOAD = 0,    // dst = cols[a][(row + (int)b * step) mod rows]
  Q_CONST = 1,   // dst = consts[a]
  Q_ADD = 2, Q_SUB = 3, Q_MUL = 4,   // dst = a (op) b
  Q_NEG = 5, Q_SQR = 6, Q_DBL = 7,   // dst = op(a)
  Q_COSETX = 8,  // dst = zeta * ext_omega^(global row): the value of X on the extended coset (Ast::LinearTerm)
  Q_STORE = 9,   // out[row] = a
  Q_MULC = 10, Q_ADDC = 11, Q_SUBC = 12,   // dst = a (op) consts[b]
  Q_NOPS = 13
};

struct QParams {
  const uint4* prog;     // lowered program in the staged encoding (qlower::stage), qlower::PAD NOPs appended
  unsigned n_instr, n_regs, bd_log;
  const uint4* consts;
  unsigned rows_log, step, out_stride, out_off, x_stride, x_off, ext_log;
  // row-slice mode (nrows > 0): the columns hold rows [row0 - halo_before, row0 + nrows + halo_after) of the coset (cyclic
  // neighbours copied in by the caller), thread t evaluates coset row row0 + t and stores out[t]
  unsigned row0, nrows, halo_before;
  const uint4* tw_ext;   // ext_omega^i, i < 2^(ext_log-1)
  uint4* out;
};

// One thread = one row.  The lowered program (qlower.h) is in accumulator form: the previous result stays in hardware registers
// (acc); an instruction first reloads acc from the virtual register file (shared memory, two 16-byte planes [reg][thread]) unless
// its operand a IS the previous result, combines it with operand b -- register file, constant table, a column at (row +
// rotation), the coset-X table -- and stores acc back unless nobody will read it from the register file.  One case per
// (operation, source of b), so that no operand is ever moved between registers.  The instructions arrive in the staged encoding
// of qlower::stage: register operands are slot offsets, a column operand is the column's address, so the only arithmetic left per
// instruction is the row index of a column read; the next instruction is fetched while the current one executes.
template <class PR>
__global__ void __launch_bounds__(128) quotient_vm_kernel(QParams p) {
  using namespace qlower;
  extern __shared__ uint4 smem[];
  const unsigned tid = threadIdx.x;
  uint4* plane0 = smem + tid;
  uint4* plane1 = plane0 + ((size_t)p.n_regs << p.bd_log);
  const bool slice = p.nrows != 0;
  const unsigned rows = slice ? p.nrows : 1u << p.rows_log;
  const unsigned gid = blockIdx.x * blockDim.x + tid;
  // surplus threads of the last block recompute a valid row and never store
  const unsigned row = slice ? (gid < rows ? gid : rows - 1) : (gid & (rows - 1));
  const bool live = gid < rows;
  const unsigned idx0 = slice ? row + p.halo_before : row, idx_mask = slice ? 0xffffffffu : rows - 1, idx_step = slice ? 1u : p.step;
  auto rd = [&](unsigned slot) -> Fe<PR> {
    const uint4 lo = plane0[slot], hi = plane1[slot];
    Fe<PR> r;
    r.v[0] = lo.x; r.v[1] = lo.y; r.v[2] = lo.z; r.v[3] = lo.w; r.v[4] = hi.x; r.v[5] = hi.y; r.v[6] = hi.z; r.v[7] = hi.w;
    return r;
  };
  auto cst = [&](unsigned i) -> Fe<PR> { return fe_load_ro<PR>(p.consts + 2 * (size_t)i); };
  Fe<PR> acc = fe_zero<PR>();
  uint4 ins = __ldg(p.prog);
  for (unsigned pc = 0; pc < p.n_instr; ++pc) {
    const uint4 nxt = __ldg(p.prog + pc + 1);
    const unsigned fl = ins.x >> 5;
    if (!(fl & (F_FWD_A | F_NO_A))) acc = rd(ins.y & 0xffffu);
    auto col = [&]() -> Fe<PR> {
      const unsigned idx = (idx0 + (unsigned)(((int)ins.y >> 16) * (int)idx_step)) & idx_mask;
      const uint4* base = reinterpret_cast<const uint4*>(((unsigned long long)ins.w << 32) | ins.z);
      return fe_load_ro<PR>(base + 2 * (size_t)idx);
    };
    switch (ins.x & 31u) {
      case K_MOV_CONST: acc = cst(ins.z); break;
      case K_MOV_COL: acc = col(); break;
      case K_MOV_REG: acc = rd(ins.z); break;
      case K_MOV_X: {
        const unsigned g = (row + p.row0) * p.x_stride + p.x_off, half = 1u << (p.ext_log - 1);
        acc = fe_load_ro<PR>(p.tw_ext + 2 * (size_t)(g & (half - 1)));
        if (g & half) acc = fe_neg(acc);
        break;
      }
      case K_ADD_REG: acc = fe_add(acc, rd(ins.z)); break;
      case K_ADD_CONST: acc = fe_add(acc, cst(ins.z)); break;
      case K_ADD_COL: acc = fe_add(acc, col()); break;
      case K_SUB_REG: acc = fe_sub(acc, rd(ins.z)); break;
      case K_SUB_CONST: acc = fe_sub(acc, cst(ins.z)); break;
      case K_SUB_COL: acc = fe_sub(acc, col()); break;
      case K_RSUB_REG: acc = fe_sub(rd(ins.z), acc); break;
      case K_RSUB_CONST: acc = fe_sub(cst(ins.z), acc); break;
      case K_RSUB_COL: acc = fe_sub(col(), acc); break;
      case K_MUL_REG: acc = fe_mul(acc, rd(ins.z)); break;
      case K_MUL_CONST: acc = fe_mul(acc, cst(ins.z)); break;
      case K_MUL_COL: acc = fe_mul(acc, col()); break;
      case K_MUL_A: acc = fe_mul(acc, acc); break;
      case K_NEG: acc = fe_neg(acc); break;
      case K_DBL: acc = fe_dbl(acc); break;
      case K_STORE:
        if (live) fe_store(p.out + 2 * ((size_t)row * p.out_stride + p.out_off), acc);
        break;
      default: break;
    }
    if (!(fl & F_NOWB)) {
      const unsigned slot = ins.x >> 8;
      plane0[slot] = make_uint4(acc.v[0], acc.v[1], acc.v[2], acc.v[3]);
      plane1[slot] = make_uint4(acc.v[4], acc.v[5], acc.v[6], acc.v[7]);
    }
    ins = nxt;
  }
}

int validate_program(trp_ctx* ctx, const uint32_t* prog, size_t n_instr, unsigned n_regs, size_t n_consts, size_t n_cols) {
  bool stores = false;
  for (size_t i = 0; i < n_instr; ++i) {
    const uint32_t op = prog[4 * i], dst = prog[4 * i + 1], a = prog[4 * i + 2], b = prog[4 * i + 3];
    bool ok = op < Q_NOPS;
    if (ok) switch (op) {
      case Q_LOAD: ok = dst < n_regs && a < n_cols && ((int)b >= -32768 && (int)b <= 32767); break;
      case Q_CONST: ok = dst < n_regs && a < n_consts; break;
      case Q_ADD: case Q_SUB: case Q_MUL: ok = dst < n_regs && a < n_regs && b < n_regs; break;
      case Q_NEG: case Q_SQR: case Q_DBL: ok = dst < n_regs && a < n_regs; break;
      case Q_COSETX: ok = dst < n_regs; break;
      case Q_STORE: ok = a < n_regs; stores = true; break;
      default: ok = dst < n_regs && a < n_regs && b < n_consts; break;
    }
    if (!ok) TRP_FAIL(ctx, TRP_E_INVALID, "quotient program: instruction %zu is malformed (op %u dst %u a %u b %u)", i, op, dst, a, b);
  }
  if (!stores) TRP_FAIL(ctx, TRP_E_INVALID, "quotient program never stores a result");
  return TRP_OK;
}

// threads per CTA for a program of n_regs virtual registers (the register file is n_regs x threads x 32 B of shared memory)
bool vm_geometry(unsigned n_regs, unsigned* threads, unsigned* bd_log) {
  *threads = 128; *bd_log = 7;
  while (*threads > 32 && (size_t)n_regs * *threads * 32 > 200 * 1024) { *threads >>= 1; --*bd_log; }
  return (size_t)n_regs * *threads * 32 <= 200 * 1024;
}

// what stage_tables leaves at the front of the arena
struct Staged {
  const uint4* prog; size_t n_instr; unsigned n_regs;     // lowered program, staged encoding
  const uint4* consts;
  char* after;
};

int launch_vm(trp_domain* d, const Staged& st, int coset, uint4* d_out, unsigned row0 = 0, unsigned nrows = 0, unsigned halo_before = 0) {
  trp_ctx* ctx = d->ctx;
  QParams p;
  p.prog = st.prog; p.n_instr = (unsigned)st.n_instr; p.n_regs = st.n_regs; p.consts = st.consts;
  p.ext_log = d->ext_k;
  const unsigned period = 1u << (d->ext_k - d->k);
  const bool contiguous = coset >= 0 && (coset & TRP_Q_CONTIGUOUS);
  if (coset >= 0) coset &= ~TRP_Q_CONTIGUOUS;
  if (coset < 0) { p.rows_log = d->ext_k; p.step = period; p.out_stride = 1; p.out_off = 0; p.x_stride = 1; p.x_off = 0; }
  else {
    p.rows_log = d->k; p.step = 1; p.x_stride = period; p.x_off = (unsigned)coset;
    p.out_stride = contiguous ? 1 : period; p.out_off = contiguous ? 0 : (unsigned)coset;
  }
  p.row0 = row0; p.nrows = nrows; p.halo_before = halo_before;
  if (nrows) { p.out_stride = 1; p.out_off = 0; }
  const void* tw = nullptr;
  TRP_TRY(trp_get_powers(ctx, d->field, d->ext_k, d->ext_omega, &tw));
  p.tw_ext = (const uint4*)tw;
  p.out = d_out;
  unsigned threads, bd_log;
  if (!vm_geometry(st.n_regs, &threads, &bd_log))
    TRP_FAIL(ctx, TRP_E_INVALID, "quotient program needs %u registers (max %u)", st.n_regs, 200 * 1024 / (32 * 32));
  p.bd_log = bd_log;
  size_t smem = (size_t)st.n_regs * threads * 32;
  const size_t rows = nrows ? (size_t)nrows : (size_t)1 << p.rows_log;
  unsigned blocks = (unsigned)((rows + threads - 1) / threads);
  auto go = [&](auto tag) -> int {
    typedef decltype(tag) PR;
    if (smem > 48 * 1024)
      TRP_CUDA(ctx, cudaFuncSetAttribute(quotient_vm_kernel<PR>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    ProfScope ps(ctx, PROF_QUOTIENT, (double)rows);      // work = rows evaluated (x the program's multiplications, known to the caller)
    quotient_vm_kernel<PR><<<blocks, threads, smem, ctx->stream>>>(p);
    TRP_LAUNCHED(ctx);
    return TRP_OK;
  };
  return d->field == 0 ? go(FpParams()) : go(FqParams());
}

constexpr unsigned MAX_QUOTIENT_PARTS = 64;   // = the most cosets a domain has (trp_domain::coset_gen)
constexpr unsigned COMBINE_Q = 8;             // output pieces per thread (grid.y covers the rest)
struct PartsShape { unsigned n_parts, q_out, q[MAX_QUOTIENT_PARTS]; };

// out[q * n + t] = sum_p sum_i A_p[q][i] * P_p[i * n + t] over the parts p with q < Q_p: part p holds the remainders of its values
// on cosets 0 .. Q_p - 1 (P_p[i], rows after those of the earlier parts) and A_p is its Q_p x Q_p constant matrix (the matrices back
// to back in A).  A thread owns pieces q0 .. q0 + 7 of one coefficient index, kept in registers; each input element it needs is
// read once.
template <class PR>
__global__ void cosets_combine_kernel(const uint4* P, const uint4* A, PartsShape sh, size_t n, uint4* out) {
  size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n) return;
  const unsigned q0 = blockIdx.y * COMBINE_Q;
  Fe<PR> acc[COMBINE_Q];
#pragma unroll
  for (unsigned q = 0; q < COMBINE_Q; ++q) acc[q] = fe_zero<PR>();
  size_t row = 0, a_off = 0;
  for (unsigned p = 0; p < sh.n_parts; ++p) {
    const unsigned Q = sh.q[p];
    if (Q > q0)
      for (unsigned i = 0; i < Q; ++i) {
        const Fe<PR> v = fe_load<PR>(P + 2 * ((row + i) * n + t));
#pragma unroll
        for (unsigned q = 0; q < COMBINE_Q; ++q)
          if (q0 + q < Q) acc[q] = fe_add(acc[q], fe_mul(v, fe_load_ro<PR>(A + 2 * (a_off + (q0 + q) * Q + i))));
      }
    row += Q; a_off += (size_t)Q * Q;
  }
#pragma unroll
  for (unsigned q = 0; q < COMBINE_Q; ++q)
    if (q0 + q < sh.q_out) fe_store(out + 2 * ((q0 + q) * n + t), acc[q]);
}

// A' = V^-1 * diag(1 / ((gamma_i - 1) n))  (or diag(1/n) without the vanishing division), V[i][q] = gamma_i^q,
// gamma_i = (zeta * ext_omega^i)^n; host-side field arithmetic (ff.cuh compiles for the host)
template <class PR>
int build_combine_matrix(trp_domain* d, unsigned Q, int divide, std::vector<Fe<PR>>& out) {
  auto from64 = [](const uint64_t* l) { Fe<PR> r; for (int i = 0; i < 4; ++i) { r.v[2 * i] = (uint32_t)l[i]; r.v[2 * i + 1] = (uint32_t)(l[i] >> 32); } return r; };
  const uint64_t n = 1ULL << d->k;
  uint32_t e[2] = {(uint32_t)n, (uint32_t)(n >> 32)};
  const Fe<PR> one = fe_one<PR>();
  std::vector<Fe<PR>> gamma(Q), M(Q * 2 * Q);
  for (unsigned i = 0; i < Q; ++i) gamma[i] = fe_pow(from64(d->coset_gen[i]), e, 2);
  // Gauss-Jordan on [V | I]
  for (unsigned i = 0; i < Q; ++i) {
    Fe<PR> pw = one;
    for (unsigned q = 0; q < Q; ++q) { M[i * 2 * Q + q] = pw; pw = fe_mul(pw, gamma[i]); M[i * 2 * Q + Q + q] = (q == i) ? one : fe_zero<PR>(); }
  }
  for (unsigned c = 0; c < Q; ++c) {
    unsigned piv = c;
    while (piv < Q && fe_is_zero(M[piv * 2 * Q + c])) ++piv;
    if (piv == Q) TRP_FAIL(d->ctx, TRP_E_INVALID, "internal: singular coset Vandermonde matrix");
    if (piv != c) for (unsigned x = 0; x < 2 * Q; ++x) std::swap(M[piv * 2 * Q + x], M[c * 2 * Q + x]);
    Fe<PR> inv = fe_inv(M[c * 2 * Q + c]);
    for (unsigned x = 0; x < 2 * Q; ++x) M[c * 2 * Q + x] = fe_mul(M[c * 2 * Q + x], inv);
    for (unsigned r = 0; r < Q; ++r) {
      if (r == c || fe_is_zero(M[r * 2 * Q + c])) continue;
      Fe<PR> f = M[r * 2 * Q + c];
      for (unsigned x = 0; x < 2 * Q; ++x) M[r * 2 * Q + x] = fe_sub(M[r * 2 * Q + x], fe_mul(f, M[c * 2 * Q + x]));
    }
  }
  Fe<PR> nf = fe_zero<PR>(); nf.v[d->k >> 5] = 1u << (d->k & 31);
  const Fe<PR> ninv = fe_inv(fe_to_mont(nf));
  out.resize(Q * Q);
  for (unsigned i = 0; i < Q; ++i) {
    Fe<PR> s = ninv;
    if (divide) s = fe_mul(s, fe_inv(fe_sub(gamma[i], one)));
    for (unsigned q = 0; q < Q; ++q) out[q * Q + i] = fe_mul(M[q * 2 * Q + Q + i], s);   // (V^-1)[q][i] * s_i
  }
  return TRP_OK;
}

template <class PR>
int cosets_to_coeff_run(trp_domain* d, uint64_t* d_vals, const PartsShape& sh, uint64_t* d_out, int divide) {
  trp_ctx* ctx = d->ctx;
  const size_t n = (size_t)1 << d->k;
  std::vector<Fe<PR>> A;
  for (unsigned p = 0; p < sh.n_parts; ++p) {
    std::vector<Fe<PR>> Ap;
    TRP_TRY(build_combine_matrix<PR>(d, sh.q[p], divide, Ap));
    A.insert(A.end(), Ap.begin(), Ap.end());
  }
  const bool need_tmp = trp_ntt_passes(d->k) > 1;
  const size_t a_bytes = ws_align(A.size() * 32);
  TRP_TRY(trp_ws_reserve(ctx, a_bytes + (need_tmp ? n * 32 : 0)));
  char* w = (char*)ctx->ws;
  TRP_CUDA(ctx, cudaMemcpyAsync(w, A.data(), A.size() * 32, cudaMemcpyHostToDevice, ctx->stream));
  TRP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));   // A is a local
  size_t row = 0;
  for (unsigned p = 0; p < sh.n_parts; ++p)
    for (unsigned i = 0; i < sh.q[p]; ++i, ++row) {
      // P'_i[t] = c_i^-t * iNTT_omega(values)[t]: the coset-i remainder h_p mod (X^n - gamma_i), up to the factors folded into A_p
      uint64_t cinv[4];
      {
        Fe<PR> c; for (int l = 0; l < 4; ++l) { c.v[2 * l] = (uint32_t)d->coset_gen[i][l]; c.v[2 * l + 1] = (uint32_t)(d->coset_gen[i][l] >> 32); }
        Fe<PR> ci = fe_inv(c);
        for (int l = 0; l < 4; ++l) cinv[l] = (uint64_t)ci.v[2 * l] | ((uint64_t)ci.v[2 * l + 1] << 32);
      }
      const void* post = nullptr;
      TRP_TRY(trp_get_powers(ctx, d->field, d->k + 1, cinv, &post));
      uint64_t* v = d_vals + 4 * row * n;
      TRP_TRY(trp_ntt_impl(ctx, d->field, v, v, 1, d->k, d->omega_inv, n, n, (unsigned)n, nullptr, 0, post, (unsigned)n, (unsigned)n,
                           need_tmp ? w + a_bytes : nullptr));
    }
  cosets_combine_kernel<PR><<<dim3((unsigned)((n + 127) / 128), (sh.q_out + COMBINE_Q - 1) / COMBINE_Q), 128, 0, ctx->stream>>>((const uint4*)d_vals, (const uint4*)w, sh, n, (uint4*)d_out);
  TRP_LAUNCHED(ctx);
  return TRP_OK;
}

struct Locked {
  std::lock_guard<std::mutex> g;
  explicit Locked(trp_ctx* c) : g(c->mu) { cudaSetDevice(c->device); }
};

// lower the caller's program (cached: a prover evaluates the same few programs on its cosets, proof after proof), encode it for this launch
// (qlower::stage: slot offsets, column addresses) and put program / constants at the front of the arena.  col_ptrs = the columns'
// device addresses, or NULL if the caller will upload the columns itself right behind the tables, own_col_bytes apart.
int stage_tables(trp_domain* d, const uint32_t* program, size_t n_instr, unsigned n_regs, const uint64_t* consts, size_t n_consts,
                 const uint64_t* const* col_ptrs, size_t n_cols, size_t own_col_bytes, size_t extra, Staged* st) {
  trp_ctx* ctx = d->ctx;
  auto& progs = ctx->q_progs;
  size_t hit = 0;
  while (hit < progs.size() && !(progs[hit].src.size() == n_instr * 4 && progs[hit].src_regs == n_regs && progs[hit].src_consts == n_consts &&
                                 memcmp(progs[hit].src.data(), program, n_instr * 16) == 0))
    ++hit;
  if (hit == progs.size()) {
    trp_ctx::QProgram e;
    if (!qlower::lower(program, n_instr, n_regs, n_consts, e.low, &e.low_regs))
      TRP_FAIL(ctx, TRP_E_INVALID, "quotient program: column index above %u", qlower::MAX_COLS - 1);
    e.src.assign(program, program + n_instr * 4);
    e.src_regs = n_regs; e.src_consts = n_consts;
    if (progs.size() == 16) progs.pop_back();
    progs.insert(progs.begin(), std::move(e));
  } else if (hit > 0) {
    std::rotate(progs.begin(), progs.begin() + hit, progs.begin() + hit + 1);
  }
  const trp_ctx::QProgram& q = progs.front();
  unsigned threads, bd_log;
  if (!vm_geometry(q.low_regs, &threads, &bd_log))
    TRP_FAIL(ctx, TRP_E_INVALID, "quotient program needs %u registers (max %u)", q.low_regs, 200 * 1024 / (32 * 32));
  const size_t low_bytes = q.low.size() * 4;                          // includes the trailing NOPs
  size_t b_prog = ws_align(low_bytes), b_c = ws_align((n_consts + 1) * 32);   // + zeta
  TRP_TRY(trp_ws_reserve(ctx, b_prog + b_c + extra));
  char* w = (char*)ctx->ws;
  std::vector<uint64_t> addr(n_cols ? n_cols : 1);
  for (size_t c = 0; c < n_cols; ++c) addr[c] = col_ptrs ? (uint64_t)(uintptr_t)col_ptrs[c] : (uint64_t)(uintptr_t)(w + b_prog + b_c + c * own_col_bytes);
  if (!qlower::stage(q.low, q.low_regs, bd_log, addr.data(), n_cols, ctx->q_staged))
    TRP_FAIL(ctx, TRP_E_INVALID, "quotient program: a rotation beyond +-32767 rows or too many registers");
  TRP_CUDA(ctx, cudaMemcpyAsync(w, ctx->q_staged.data(), low_bytes, cudaMemcpyHostToDevice, ctx->stream));
  if (n_consts) TRP_CUDA(ctx, cudaMemcpyAsync(w + b_prog, consts, n_consts * 32, cudaMemcpyHostToDevice, ctx->stream));
  TRP_CUDA(ctx, cudaMemcpyAsync(w + b_prog + n_consts * 32, d->g_coset, 32, cudaMemcpyHostToDevice, ctx->stream));   // consts[n_consts] = zeta
  // the host arrays may be reused by the caller as soon as we return
  TRP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  st->prog = (const uint4*)w; st->n_instr = q.low.size() / 4 - qlower::PAD; st->n_regs = q.low_regs;
  st->consts = (const uint4*)(w + b_prog);
  st->after = w + b_prog + b_c;
  return TRP_OK;
}

}  // namespace

extern "C" {

int trp_dev_quotient_eval(trp_domain* d, const uint32_t* program, size_t n_instr, unsigned n_regs, const uint64_t* consts,
                          size_t n_consts, const uint64_t* const* d_cols, size_t n_cols, int coset, uint64_t* d_out) {
  if (!d) return TRP_E_INVALID;
  trp_ctx* ctx = d->ctx;
  Locked l(ctx);
  if (!program || !n_instr || !d_out || (n_consts && !consts) || (n_cols && !d_cols)) TRP_FAIL(ctx, TRP_E_INVALID, "NULL buffer");
  if (n_regs == 0 || (coset >= 0 && (coset & ~TRP_Q_CONTIGUOUS) >= (int)(1u << (d->ext_k - d->k))))
    TRP_FAIL(ctx, TRP_E_INVALID, "bad register count or coset index");
  TRP_TRY(validate_program(ctx, program, n_instr, n_regs, n_consts, n_cols));
  for (size_t c = 0; c < n_cols; ++c) if (!d_cols[c]) TRP_FAIL(ctx, TRP_E_INVALID, "column %zu is NULL", c);
  Staged st;
  TRP_TRY(stage_tables(d, program, n_instr, n_regs, consts, n_consts, d_cols, n_cols, 0, 0, &st));
  return launch_vm(d, st, coset, (uint4*)d_out);
}

// Row-slice form of the coset evaluation (the multi-GPU quotient: a coset's rows are split between the devices): the columns
// hold the coset's rows [row0 - halo_before, row0 + nrows + halo_after) (cyclic), the program may rotate by -halo_before ..
// +halo_after rows, d_out receives the nrows results.
int trp_dev_quotient_eval_rows(trp_domain* d, const uint32_t* program, size_t n_instr, unsigned n_regs, const uint64_t* consts,
                               size_t n_consts, const uint64_t* const* d_cols, size_t n_cols, unsigned coset, size_t row0, size_t nrows,
                               unsigned halo_before, unsigned halo_after, uint64_t* d_out) {
  if (!d) return TRP_E_INVALID;
  trp_ctx* ctx = d->ctx;
  Locked l(ctx);
  if (!program || !n_instr || !d_out || (n_consts && !consts) || (n_cols && !d_cols)) TRP_FAIL(ctx, TRP_E_INVALID, "NULL buffer");
  if (n_regs == 0 || coset >= (1u << (d->ext_k - d->k))) TRP_FAIL(ctx, TRP_E_INVALID, "bad register count or coset index");
  const size_t n = (size_t)1 << d->k;
  if (nrows == 0 || row0 >= n || nrows > n - row0) TRP_FAIL(ctx, TRP_E_INVALID, "row slice [%zu, %zu) is outside the coset", row0, row0 + nrows);
  TRP_TRY(validate_program(ctx, program, n_instr, n_regs, n_consts, n_cols));
  for (size_t i = 0; i < n_instr; ++i)
    if (program[4 * i] == Q_LOAD) {
      const int rot = (int)program[4 * i + 3];
      if (rot < -(int)halo_before || rot > (int)halo_after)
        TRP_FAIL(ctx, TRP_E_INVALID, "quotient program rotates by %d rows, the slice carries -%u .. +%u", rot, halo_before, halo_after);
    }
  for (size_t c = 0; c < n_cols; ++c) if (!d_cols[c]) TRP_FAIL(ctx, TRP_E_INVALID, "column %zu is NULL", c);
  Staged st;
  TRP_TRY(stage_tables(d, program, n_instr, n_regs, consts, n_consts, d_cols, n_cols, 0, 0, &st));
  return launch_vm(d, st, (int)coset, (uint4*)d_out, (unsigned)row0, (unsigned)nrows, halo_before);
}

// host-pointer form over the whole extended domain (what poly::Evaluator::evaluate returns): columns are uploaded,
// the result is downloaded.  Meant for parity tests and small domains; a prover keeps columns on the device.
int trp_quotient_eval(trp_domain* d, const uint32_t* program, size_t n_instr, unsigned n_regs, const uint64_t* consts,
                      size_t n_consts, const uint64_t* const* cols, size_t n_cols, uint64_t* out_ext) {
  if (!d) return TRP_E_INVALID;
  trp_ctx* ctx = d->ctx;
  Locked l(ctx);
  if (!program || !n_instr || !out_ext || (n_consts && !consts) || (n_cols && !cols)) TRP_FAIL(ctx, TRP_E_INVALID, "NULL buffer");
  if (n_regs == 0) TRP_FAIL(ctx, TRP_E_INVALID, "bad register count");
  TRP_TRY(validate_program(ctx, program, n_instr, n_regs, n_consts, n_cols));
  for (size_t c = 0; c < n_cols; ++c) if (!cols[c]) TRP_FAIL(ctx, TRP_E_INVALID, "column %zu is NULL", c);
  const size_t EN = (size_t)1 << d->ext_k;
  Staged st;
  TRP_TRY(stage_tables(d, program, n_instr, n_regs, consts, n_consts, nullptr, n_cols, EN * 32, (n_cols + 1) * EN * 32, &st));
  char* after = st.after;                               // the staged program addresses column c at after + c * EN * 32
  for (size_t c = 0; c < n_cols; ++c)
    TRP_CUDA(ctx, cudaMemcpyAsync(after + c * EN * 32, cols[c], EN * 32, cudaMemcpyHostToDevice, ctx->stream));
  char* d_out = after + n_cols * EN * 32;
  TRP_TRY(launch_vm(d, st, -1, (uint4*)d_out));
  TRP_CUDA(ctx, cudaMemcpyAsync(out_ext, d_out, EN * 32, cudaMemcpyDeviceToHost, ctx->stream));
  TRP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return TRP_OK;
}

// Evaluations of `batch` coefficient-form columns (n each) on the coset (zeta * ext_omega^coset) * <omega>:
// out[i] = p(zeta * ext_omega^(coset + i * 2^(ext_k-k))), i.e. rows coset, coset + 2^(ext_k-k), ... of coeff_to_extended.
int trp_dev_coeff_to_coset(trp_domain* d, const uint64_t* d_coeff, uint64_t* d_out, size_t batch, unsigned coset) {
  if (!d) return TRP_E_INVALID;
  trp_ctx* ctx = d->ctx;
  Locked l(ctx);
  if (batch && (!d_coeff || !d_out)) TRP_FAIL(ctx, TRP_E_INVALID, "NULL buffer");
  if (coset >= (1u << (d->ext_k - d->k))) TRP_FAIL(ctx, TRP_E_INVALID, "coset index %u out of range", coset);
  const size_t n = (size_t)1 << d->k;
  const void* pw = nullptr;   // (zeta * ext_omega^coset)^i, i < n
  TRP_TRY(trp_get_powers(ctx, d->field, d->k + 1, d->coset_gen[coset], &pw));
  const bool need_tmp = trp_ntt_passes(d->k) > 1 && d_coeff == d_out;
  size_t cols = batch > 65535 ? 65535 : batch;
  if (need_tmp) {
    size_t fit = ((size_t)4 << 30) / (n * 32);
    if (fit < 1) fit = 1;
    if (cols > fit) cols = fit;
    TRP_TRY(trp_ws_reserve(ctx, cols * n * 32));
  }
  for (size_t b0 = 0; b0 < batch; b0 += cols) {
    size_t nb = batch - b0 < cols ? batch - b0 : cols;
    TRP_TRY(trp_ntt_impl(ctx, d->field, d_coeff + 4 * b0 * n, d_out + 4 * b0 * n, nb, d->k, d->omega, n, n, (unsigned)n, pw,
                         (unsigned)n, nullptr, 0, (unsigned)n, need_tmp ? ctx->ws : nullptr));
  }
  return TRP_OK;
}

// The same for columns scattered in memory: d_src_tab is a DEVICE array of batch column addresses (n coefficients each), the
// results go to d_out contiguously (column i at d_out[i * n ..]).  A prover expands on each coset only the columns that the
// constraints evaluated there read, without copying them together first.
int trp_dev_coeff_to_coset_gather(trp_domain* d, const uint64_t* const* d_src_tab, uint64_t* d_out, size_t batch, unsigned coset) {
  if (!d) return TRP_E_INVALID;
  trp_ctx* ctx = d->ctx;
  Locked l(ctx);
  if (batch && (!d_src_tab || !d_out)) TRP_FAIL(ctx, TRP_E_INVALID, "NULL buffer");
  if (coset >= (1u << (d->ext_k - d->k))) TRP_FAIL(ctx, TRP_E_INVALID, "coset index %u out of range", coset);
  const size_t n = (size_t)1 << d->k;
  const void* pw = nullptr;   // (zeta * ext_omega^coset)^i, i < n
  TRP_TRY(trp_get_powers(ctx, d->field, d->k + 1, d->coset_gen[coset], &pw));
  for (size_t b0 = 0; b0 < batch; b0 += 65535) {
    size_t nb = batch - b0 < 65535 ? batch - b0 : 65535;
    TRP_TRY(trp_ntt_impl(ctx, d->field, nullptr, d_out + 4 * b0 * n, nb, d->k, d->omega, n, n, (unsigned)n, pw, (unsigned)n, nullptr, 0,
                         (unsigned)n, nullptr, (const void* const*)(d_src_tab + b0)));
  }
  return TRP_OK;
}

// Recover the n * ncos coefficients of a polynomial of degree < n * ncos from its values on the first ncos size-n cosets
// (zeta * ext_omega^i) * <omega>, i < ncos: per coset an inverse NTT gives h mod (X^n - gamma_i), and one ncos x ncos
// constant matrix (inverse Vandermonde in gamma_i = (zeta ext_omega^i)^n) applied per coefficient index undoes the
// wrap-around.  With divide_by_vanishing the input is the quotient NUMERATOR and is divided by X^n - 1 (the constant
// gamma_i - 1 on coset i).  Produces exactly extended_to_coeff(divide_by_vanishing_poly(.)) of the full extended
// domain while evaluating only ncos = j - 1 of its 2^(ext_k - k) cosets (5 of 8 for the TinyRAM circuit).
int trp_dev_cosets_to_coeff(trp_domain* d, uint64_t* d_vals, unsigned ncos, uint64_t* d_out_coeff, int divide_by_vanishing) {
  return trp_dev_cosets_to_coeff_parts(d, d_vals, &ncos, 1, ncos, d_out_coeff, divide_by_vanishing);
}

// The same for a polynomial given as a SUM of parts h = sum_p h_p, deg h_p < n * ncos[p]: part p brings its values on the first
// ncos[p] cosets (rows after those of the earlier parts), and the coefficients of all parts are summed into ncos_out pieces of n.
// Each part is recovered exactly as above (its own ncos[p] x ncos[p] inverse Vandermonde), so a part of low degree is evaluated
// on fewer cosets, and the sum equals trp_dev_cosets_to_coeff of the whole h on ncos_out cosets coefficient for coefficient.
int trp_dev_cosets_to_coeff_parts(trp_domain* d, uint64_t* d_vals, const unsigned* ncos, unsigned n_parts, unsigned ncos_out,
                                  uint64_t* d_out_coeff, int divide_by_vanishing) {
  if (!d) return TRP_E_INVALID;
  trp_ctx* ctx = d->ctx;
  Locked l(ctx);
  if (!d_vals || !d_out_coeff || !ncos) TRP_FAIL(ctx, TRP_E_INVALID, "NULL buffer");
  if (n_parts == 0 || n_parts > MAX_QUOTIENT_PARTS) TRP_FAIL(ctx, TRP_E_INVALID, "n_parts = %u out of range (1 .. %u)", n_parts, MAX_QUOTIENT_PARTS);
  const unsigned t_period = 1u << (d->ext_k - d->k);
  if (ncos_out == 0 || ncos_out > t_period) TRP_FAIL(ctx, TRP_E_INVALID, "ncos_out = %u out of range", ncos_out);
  PartsShape sh{};
  sh.n_parts = n_parts; sh.q_out = ncos_out;
  for (unsigned p = 0; p < n_parts; ++p) {
    if (ncos[p] == 0 || ncos[p] > ncos_out) TRP_FAIL(ctx, TRP_E_INVALID, "part %u: ncos = %u out of range (1 .. %u)", p, ncos[p], ncos_out);
    sh.q[p] = ncos[p];
  }
  return d->field == 0 ? cosets_to_coeff_run<FpParams>(d, d_vals, sh, d_out_coeff, divide_by_vanishing)
                       : cosets_to_coeff_run<FqParams>(d, d_vals, sh, d_out_coeff, divide_by_vanishing);
}

}  // extern "C"
