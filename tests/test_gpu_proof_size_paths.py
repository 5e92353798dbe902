"""GPU tests of the paths a proof takes only at proof size, each against the oracle:

- trp_dev_coeff_to_coset_gather (the quotient's coset NTTs reading their columns through a device table of addresses): scattered,
  repeated and interior-row sources, every coset index, single- and multi-pass sizes, k = 19 and 20 in both fields (with
  trp_dev_coeff_to_coset in and out of place), and the 65 535-column chunking;
- trp_dev_cosets_to_coeff_parts (a quotient given as a sum of parts of different degrees): the prover's part shape and others,
  more than 8 output pieces (a second row of the combine grid), the most parts the entry point takes, the prover's shape at
  k = 19 and 20;
- GpuBackend._commit_many at k = 18, where the backend keeps a narrow c = 13 table over g_lagrange ++ [w] for mostly-zero columns
  and commits grand-product columns by parts over the prefix sums of g_lagrange: which table each batch takes, and every
  commitment against the oracle's MSM over g_lagrange ++ [w];
- one real k = 20 TinyRAM proof (the benchmark's workload) with all of the above probed, verified by the package's verifier."""
import ctypes
import gc
import os
import random

import numpy as np
import pytest

from util import O, pm, make_points, scalars_uniform, scalars_tinyram, affine_of

from test_gpu_quotient_split import split_probe

pytestmark = pytest.mark.gpu

BY_PARTS = os.environ.get("TRP_COMMIT_BY_PARTS", "1") != "0"


@pytest.fixture(scope="module")
def pkg():
    import __graft_entry__ as ge
    return ge.load_package()


@pytest.fixture(scope="module")
def ctxs(pkg):
    return {O.VESTA: pkg.Context(0, pkg.VESTA), O.PALLAS: pkg.Context(0, pkg.PALLAS)}


def _u64(t):
    return t.cpu().numpy().view(np.uint64)


def _dev(arr):
    import torch
    return torch.from_numpy(np.ascontiguousarray(arr).view(np.int64)).cuda()


def _gather(ctx, dom, ptrs, out, coset):
    import torch
    tab = torch.tensor(list(ptrs), dtype=torch.int64).cuda()
    torch.cuda.synchronize()
    rc = ctx.lib.trp_dev_coeff_to_coset_gather(dom.handle, tab.data_ptr(), out.data_ptr(), len(ptrs), coset)
    ctx.sync()
    return rc


# ---- trp_dev_coeff_to_coset_gather ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("curve", [O.VESTA, O.PALLAS])
@pytest.mark.parametrize("j", [6, 17])
@pytest.mark.parametrize("k", [1, 4, 10, 11, 12])
def test_coset_gather_against_the_oracle(pkg, ctxs, curve, j, k):
    """eight table entries over seven columns: three inside one larger tensor (starting 3 rows in, so no column is aligned to a
    multiple of n), four allocated separately, listed out of order and one of them twice; every coset of the extended domain"""
    import torch
    ctx, field = ctxs[curve], O.SCALAR_FIELD[curve]
    dom = pkg.EvaluationDomain(ctx, j, k)
    n = 1 << k
    period = dom.extended_len() // n
    host = O.random_field_mont(field, 7 * n, 300 + 20 * k + j).reshape(7, n, 4)
    big_host = np.concatenate([O.random_field_mont(field, 3, 1), host[:3].reshape(-1, 4), O.random_field_mont(field, 4, 2)])
    big = _dev(big_host)
    own = [_dev(host[c]) for c in range(3, 7)]
    ptr = lambda c: big[3 + c * n].data_ptr() if c < 3 else own[c - 3].data_ptr()
    order = [2, 5, 0, 3, 5, 6, 1, 4]
    ext = O.coeff_to_extended(field, j, k, host)                         # (7, period * n, 4)
    out = torch.empty((len(order), n, 4), dtype=torch.int64, device="cuda")
    for cs in range(period):
        out.fill_(-1)
        assert _gather(ctx, dom, [ptr(c) for c in order], out, cs) == 0
        assert np.array_equal(_u64(out), ext[order][:, cs::period]), cs
    assert np.array_equal(_u64(big), big_host)                          # the sources are read only
    for c in range(3, 7):
        assert np.array_equal(_u64(own[c - 3]), host[c])
    dom.free()


def test_coset_gather_k20(pkg, ctxs):
    """Vesta at k = 20, the quotient's size in the benchmark (_coset_gather_at_proof_size)"""
    _coset_gather_at_proof_size(pkg, ctxs, O.VESTA, 20)


@pytest.mark.parametrize("curve,k", [(O.PALLAS, 20), (O.VESTA, 19), (O.PALLAS, 19)])
def test_coset_gather_k19_k20(pkg, ctxs, curve, k):
    """the other field, and k = 19, where only the first pass is specialised (_coset_gather_at_proof_size)"""
    _coset_gather_at_proof_size(pkg, ctxs, curve, k)


def _coset_gather_at_proof_size(pkg, ctxs, curve, k):
    """two columns (the specialised first pass reads them through the table at k = 19 and 20) on the first and the last coset,
    against the oracle, and trp_dev_coeff_to_coset on a contiguous copy against the oracle too: out of place (the destination
    holds the intermediate) and in place (through the scratch buffer)"""
    import torch
    ctx, field, j = ctxs[curve], O.SCALAR_FIELD[curve], 6
    dom = pkg.EvaluationDomain(ctx, j, k)
    n = 1 << k
    period = dom.extended_len() // n
    host = O.random_field_mont(field, 2 * n, 320 + k).reshape(2, n, 4)
    ext = O.coeff_to_extended(field, j, k, host)
    big = _dev(np.concatenate([host[0], O.random_field_mont(field, 5, 3)]))     # column 0 at row 0 of a longer tensor
    own = _dev(host[1])
    contiguous = torch.stack([own, big[:n]])                                     # the gathered order: 1, 0
    out = torch.empty((2, n, 4), dtype=torch.int64, device="cuda")
    ref = torch.empty_like(out)
    for cs in (0, period - 1):
        want = np.stack([ext[1, cs::period], ext[0, cs::period]])
        out.fill_(-1)
        assert _gather(ctx, dom, [own.data_ptr(), big.data_ptr()], out, cs) == 0
        assert np.array_equal(_u64(out), want), cs
        ref.fill_(-1)
        torch.cuda.synchronize()
        ctx.check(ctx.lib.trp_dev_coeff_to_coset(dom.handle, contiguous.data_ptr(), ref.data_ptr(), 2, cs))
        ctx.sync()
        assert np.array_equal(_u64(ref), want), cs
        ref.copy_(contiguous)
        torch.cuda.synchronize()
        ctx.check(ctx.lib.trp_dev_coeff_to_coset(dom.handle, ref.data_ptr(), ref.data_ptr(), 2, cs))
        ctx.sync()
        assert np.array_equal(_u64(ref), want), ("in place", cs)
    assert np.array_equal(_u64(own), host[1]) and np.array_equal(_u64(big[:n]), host[0])
    assert np.array_equal(_u64(contiguous), host[[1, 0]])
    dom.free()
    del ext, out, ref, big, own, contiguous
    torch.cuda.empty_cache()


@pytest.mark.parametrize("curve", [O.VESTA, O.PALLAS])
def test_coset_gather_chunks_of_65535_columns(pkg, ctxs, curve):
    """65 537 columns at k = 1 in a shuffled table: the launches are split at 65 535 columns, and the second launch must read
    the table from entry 65 535 on"""
    import torch
    ctx, field, j, k = ctxs[curve], O.SCALAR_FIELD[curve], 6, 1
    dom = pkg.EvaluationDomain(ctx, j, k)
    n, m = 1 << k, 65537
    period = dom.extended_len() // n
    host = O.random_field_mont(field, m * n, 330).reshape(m, n, 4)
    src = _dev(host)
    perm = np.random.default_rng(5).permutation(m)
    ext = O.coeff_to_extended(field, j, k, host)[perm]
    out = torch.empty((m, n, 4), dtype=torch.int64, device="cuda")
    for cs in (0, period - 1):
        out.fill_(-1)
        assert _gather(ctx, dom, (src.data_ptr() + perm * (n * 32)).tolist(), out, cs) == 0
        assert np.array_equal(_u64(out), ext[:, cs::period]), cs
    assert np.array_equal(_u64(src), host)
    dom.free()


def test_coset_gather_rejects_bad_arguments(pkg, ctxs):
    import torch
    ctx = ctxs[O.VESTA]
    dom = pkg.EvaluationDomain(ctx, 6, 4)
    n = 16
    src = _dev(O.random_field_mont(O.FP, n, 340))
    out = torch.full((1, n, 4), -1, dtype=torch.int64, device="cuda")
    tab = torch.tensor([src.data_ptr()], dtype=torch.int64).cuda()
    torch.cuda.synchronize()
    lib = ctx.lib
    assert lib.trp_dev_coeff_to_coset_gather(dom.handle, None, None, 0, 0) == 0                       # nothing to do
    assert lib.trp_dev_coeff_to_coset_gather(dom.handle, None, out.data_ptr(), 1, 0) == -1            # a column, no table
    assert lib.trp_dev_coeff_to_coset_gather(dom.handle, tab.data_ptr(), None, 1, 0) == -1            # no output
    assert lib.trp_dev_coeff_to_coset_gather(dom.handle, tab.data_ptr(), out.data_ptr(), 1, 8) == -1  # coset >= period
    ctx.sync()
    assert (out == -1).all()
    assert lib.trp_dev_coeff_to_coset_gather(dom.handle, tab.data_ptr(), out.data_ptr(), 1, 7) == 0
    ctx.sync()
    dom.free()


# ---- trp_dev_cosets_to_coeff_parts --------------------------------------------------------------------------------------------------
def _coset_values(field, j, k, a, Q, divide):
    """(Q, n, 4): the values of the polynomial with coefficients a (degree < Q n) on cosets 0 .. Q - 1 of the extended domain,
    from the oracle's FFT over the whole extended domain; divide: times gamma_i - 1 on coset i, i.e. the numerator a (X^n - 1)"""
    F = pm.Fp if field == O.FP else pm.Fq
    dm = pm.EvaluationDomain(F, j, k)
    n, ek = 1 << k, dm.extended_k
    period = (1 << ek) // n
    mont = lambda vals: O.to_mont(field, O.ints_to_limbs([v % F.p for v in vals]))
    zeta = mont([1, dm.g_coset, dm.g_coset_inv])                          # a(zeta X): coefficient i times zeta^(i mod 3)
    padded = np.zeros((1 << ek, 4), dtype=np.uint64)
    padded[:len(a)] = O.field_op(field, "mul", a, zeta[np.arange(len(a)) % 3])
    h_ext = O.fft(field, padded, ek, mont([dm.extended_omega])[0])
    vals = np.stack([h_ext[i::period] for i in range(Q)])
    if divide:
        for i in range(Q):
            gamma = pow(dm.g_coset * pow(dm.extended_omega, i, F.p), n, F.p)
            vals[i] = O.field_op(field, "mul", vals[i], np.repeat(mont([gamma - 1]), n, axis=0))
    return vals


PART_SHAPES = [(6, [1, 2, 3, 4, 5], 5),           # the prover's shape (degrees 2 .. 6)
               (6, [5, 4, 3, 2, 1], 5),
               (6, [3, 3, 3], 3),                 # equal parts, and one part: also the same bytes as trp_dev_cosets_to_coeff
               (6, [5], 5),
               (6, [2, 1], 5),                    # pieces 2 .. 4 stay zero
               (17, [16, 9, 3, 1], 16),           # 16 pieces: the combine grid's second row (pieces 8 .. 15)
               (17, [1, 16, 3, 9], 16)]           # parts below that row come first: its threads must still step over them


def _parts_case(curve, k, divide, shape, **kw):
    j, parts, ncos_out = PART_SHAPES[shape]
    return pytest.param(curve, k, divide, shape, id="j%d-%s-out%d-%d-%d-%d" % (j, "_".join(map(str, parts)), ncos_out, divide, k, curve), **kw)


# every shape at k = 3 .. 14, and the prover's shape at k = 19 and 20 (the specialised pass: at k = 20 the last one scales by the
# table of coset-power inverses) with the division, and at k = 19 without it
PARTS_CASES = [_parts_case(curve, k, divide, shape) for shape in range(len(PART_SHAPES)) for divide in (0, 1) for k in (3, 10, 11, 14)
               for curve in (O.VESTA, O.PALLAS)]
PARTS_CASES += [_parts_case(curve, k, divide, 0) for k, divide in ((19, 1), (20, 1), (19, 0)) for curve in (O.VESTA, O.PALLAS)]


@pytest.mark.parametrize("curve,k,divide,shape", PARTS_CASES)
def test_cosets_to_coeff_parts_against_the_oracle(pkg, ctxs, curve, k, divide, shape):
    """part p: random coefficients a_p of degree < Q_p n, its values on cosets 0 .. Q_p - 1 (times gamma_i - 1 with the vanishing
    division); the result must be sum_p a_p, zero-padded to ncos_out pieces.  k = 11 and 14 take the multi-pass inverse NTT."""
    import torch
    j, parts, ncos_out = PART_SHAPES[shape]
    ctx, field = ctxs[curve], O.SCALAR_FIELD[curve]
    dom = pkg.EvaluationDomain(ctx, j, k)
    n = 1 << k
    coeffs = [O.random_field_mont(field, Q * n, 400 + 31 * k + 7 * shape + p) for p, Q in enumerate(parts)]
    vals = np.concatenate([_coset_values(field, j, k, a, Q, divide) for a, Q in zip(coeffs, parts)])
    want = np.zeros((ncos_out * n, 4), dtype=np.uint64)
    for a in coeffs:
        want[:len(a)] = O.field_op(field, "add", want[:len(a)], a)
    d_vals = _dev(vals)
    out = torch.full((ncos_out * n, 4), -1, dtype=torch.int64, device="cuda")
    qs = (ctypes.c_uint * len(parts))(*parts)
    torch.cuda.synchronize()
    ctx.check(ctx.lib.trp_dev_cosets_to_coeff_parts(dom.handle, d_vals.data_ptr(), qs, len(parts), ncos_out, out.data_ptr(), divide))
    ctx.sync()
    got = _u64(out)
    assert np.array_equal(got, want)
    assert not got[max(parts) * n:].any()
    if len(set(parts)) == 1:                  # equal parts sum coset by coset: the one-part entry point on the summed values
        Q = parts[0]
        summed = vals[:Q].copy()
        for p in range(1, len(parts)):
            summed = O.field_op(field, "add", summed.reshape(-1, 4), vals[p * Q:(p + 1) * Q].reshape(-1, 4)).reshape(Q, n, 4)
        d_sum = _dev(summed)
        one = torch.full((Q * n, 4), -1, dtype=torch.int64, device="cuda")
        torch.cuda.synchronize()
        ctx.check(ctx.lib.trp_dev_cosets_to_coeff(dom.handle, d_sum.data_ptr(), Q, one.data_ptr(), divide))
        ctx.sync()
        assert np.array_equal(_u64(one), got[:Q * n])
    dom.free()
    if k >= 19:
        del d_vals, out
        torch.cuda.empty_cache()


@pytest.mark.parametrize("k", [3, 11])
def test_cosets_to_coeff_parts_64_parts(pkg, ctxs, k):
    """the most parts the entry point takes (one per coset a domain can have): 64 parts of one coset each; 65 are rejected"""
    import torch
    ctx, field, j = ctxs[O.VESTA], O.FP, 6
    dom = pkg.EvaluationDomain(ctx, j, k)
    n = 1 << k
    coeffs = [O.random_field_mont(field, n, 500 + p) for p in range(65)]
    vals = np.concatenate([_coset_values(field, j, k, a, 1, 1) for a in coeffs])
    want = np.zeros((2 * n, 4), dtype=np.uint64)
    for a in coeffs[:64]:
        want[:n] = O.field_op(field, "add", want[:n], a)
    d_vals = _dev(vals)
    out = torch.full((2 * n, 4), -1, dtype=torch.int64, device="cuda")
    torch.cuda.synchronize()
    assert ctx.lib.trp_dev_cosets_to_coeff_parts(dom.handle, d_vals.data_ptr(), (ctypes.c_uint * 65)(*[1] * 65), 65, 2, out.data_ptr(), 1) == -1
    ctx.sync()
    assert (out == -1).all() and np.array_equal(_u64(d_vals), vals)     # rejected before anything ran
    ctx.check(ctx.lib.trp_dev_cosets_to_coeff_parts(dom.handle, d_vals.data_ptr(), (ctypes.c_uint * 64)(*[1] * 64), 64, 2, out.data_ptr(), 1))
    ctx.sync()
    assert np.array_equal(_u64(out), want)
    dom.free()


# ---- GpuBackend._commit_many at k = 18: the narrow table and the commitment by parts ------------------------------------------------
class MsmLog:
    """stands in for GpuBackend.lib: records the bases handle and column count of every trp_dev_msm_batch, forwards every call"""

    def __init__(self, lib):
        self._lib, self.calls = lib, []

    def __getattr__(self, name):
        return getattr(self._lib, name)

    def trp_dev_msm_batch(self, ctx, bases, scalars, n, m, out):
        self.calls.append((getattr(bases, "value", bases), m))
        return self._lib.trp_dev_msm_batch(ctx, bases, scalars, n, m, out)


def table_names(be):
    names = {be.params.g_lagrange.handle.value: "default", be.params.g.handle.value: "g"}
    if be._gl_sparse is not None:
        names[be._gl_sparse.handle.value] = "narrow"
    if be._gl_prefix is not None:
        names[be._gl_prefix.handle.value] = "prefix"
    return names


def oracle_commit(be, col, blind):
    """the oracle's MSM of col ++ [blind] over g_lagrange ++ [w], on the non-zero scalars only; (x, y) or None"""
    curve = O.VESTA if be.p == O.MODULUS[O.FP] else O.PALLAS
    field = O.SCALAR_FIELD[curve]
    sc = np.concatenate([np.asarray(col, dtype=np.uint64).reshape(-1, 4), O.to_mont(field, O.ints_to_limbs([blind % be.p]))])
    pts = np.concatenate([np.asarray(be.params.g_lagrange_points).reshape(-1, 8), np.asarray(be.params.w).reshape(1, 8)])
    nz = np.flatnonzero(sc.any(axis=1))
    if not len(nz):
        return None
    out = O.msm(curve, np.ascontiguousarray(sc[nz]), np.ascontiguousarray(pts[nz]))
    return tuple(O.limbs_to_ints(O.from_mont(O.BASE_FIELD[curve], out.reshape(2, 4)))) if out.any() else None


def _backend18(pkg, curve):
    be = pkg.plonk.GpuBackend(pkg.Context(0, curve), 18, 6)
    be.lib = MsmLog(be.lib)
    return be


@pytest.fixture(scope="module")
def be18(pkg):
    be = _backend18(pkg, pkg.VESTA)
    yield be
    be.close()


@pytest.fixture(scope="module")
def be18_pallas(pkg):
    be = _backend18(pkg, pkg.PALLAS)
    yield be
    be.close()


def _commit(be, cols, blinds, **hints):
    """commit_lagrange_many of host columns: (commitments, [(table, columns) per batch])"""
    n0, names = len(be.lib.calls), table_names(be)
    got = be.commit_lagrange_many([_dev(c) for c in cols], list(blinds), **hints)
    return got, [(names.get(h, "?"), m) for h, m in be.lib.calls[n0:]]


def _field(be):
    return O.FP if be.p == O.MODULUS[O.FP] else O.FQ


def _mont(be, vals):
    return O.to_mont(_field(be), O.ints_to_limbs([v % be.p for v in vals]))


def _grand_product_column(be, head, c, bf, seed):
    """a random head, the constant c up to row n - bf - 1, bf random blinding rows"""
    n = be.n
    col = np.repeat(_mont(be, [c]), n, axis=0)
    col[:head] = O.random_field_mont(_field(be), head, seed)
    col[n - bf:] = O.random_field_mont(_field(be), bf, seed + 1)
    return col


def _nonzero_rows(col, blind):
    return int(col.any(axis=1).sum()) + (blind != 0)


def test_sparse_head_takes_the_narrow_table(be18):
    be = be18
    assert be._gl_sparse is not None and be._gl_sparse.describe()["c"] == 13
    col = np.zeros((be.n, 4), dtype=np.uint64)
    col[:1 << 14] = O.random_field_mont(O.FP, 1 << 14, 600)
    blind = 0x1234567 << 200
    got, used = _commit(be, [col], [blind], sparse=True)
    assert used == [("narrow", 1)]
    assert got == [oracle_commit(be, col, blind)]


def test_sparse_threshold(be18):
    """a batch with at most n / 10 non-zero rows (the blind's row counted) takes the narrow table, one row more the default one"""
    be, n = be18, be18.n
    lim = n // 10
    rng = np.random.default_rng(7)
    blind = 98765
    for extra, table in ((0, "narrow"), (1, "default")):
        col = np.zeros((n, 4), dtype=np.uint64)
        rows = rng.choice(n, lim - 1 + extra, replace=False)
        col[rows] = O.random_field_mont(O.FP, len(rows), 610 + extra)
        assert _nonzero_rows(col, blind) == lim + extra
        got, used = _commit(be, [col], [blind], sparse=True)
        assert used == [(table, 1)], extra
        assert got == [oracle_commit(be, col, blind)], extra


def _runs_batch(be, seed):
    """three grand-product-shaped columns and one that is constant up to row n - 2 and changes only at row n - 1; in the flattened
    batch each column's row n - 1, its blind and the next column's row 0 all differ (the rows _commit_many patches)"""
    n, bf = be.n, 5
    cols = [_grand_product_column(be, h, c, bf, seed + 10 * i) for i, (h, c) in enumerate([(1000, 1), (1, 0x5555), (20000, be.p - 3)])]
    last = np.repeat(_mont(be, [77]), n, axis=0)
    last[n - 1] = _mont(be, [78])[0]
    cols.append(last)
    blinds = [seed * 1000 + i + 1 for i in range(len(cols))]
    for i, col in enumerate(cols):
        b = _mont(be, [blinds[i]])[0]
        nxt = cols[(i + 1) % len(cols)][0]
        assert not (col[n - 1] == b).all() and not (col[n - 1] == nxt).all() and not (b == nxt).all()
    return cols, blinds


def test_grand_product_columns_take_the_prefix_table(be18):
    be = be18
    cols, blinds = _runs_batch(be, 7)
    got, used = _commit(be, cols, blinds, runs=True)
    assert used == [("prefix" if BY_PARTS else "default", 4)]
    assert got == [oracle_commit(be, c, b) for c, b in zip(cols, blinds)]


def test_pallas_narrow_and_prefix_tables(be18_pallas):
    be = be18_pallas
    col = np.zeros((be.n, 4), dtype=np.uint64)
    col[5000:5000 + (1 << 14)] = O.random_field_mont(O.FQ, 1 << 14, 620)
    got, used = _commit(be, [col], [3], sparse=True)
    assert used == [("narrow", 1)] and got == [oracle_commit(be, col, 3)]
    cols, blinds = _runs_batch(be, 8)
    got, used = _commit(be, cols[:3], blinds[:3], runs=True)
    assert used == [("prefix" if BY_PARTS else "default", 3)]
    assert got == [oracle_commit(be, c, b) for c, b in zip(cols[:3], blinds[:3])]


def test_sparse_and_runs_hints_together(be18):
    """the prover's call for permuted lookup columns: a mostly-zero column takes the narrow table, a column with a non-zero
    default takes the prefix table, and a batch of both (dense as a whole) the prefix table"""
    be, n = be18, be18.n
    zero_heavy = np.zeros((n, 4), dtype=np.uint64)
    zero_heavy[:1 << 14] = O.random_field_mont(O.FP, 1 << 14, 630)
    default = _grand_product_column(be, 1 << 14, 9, 6, 640)
    got, used = _commit(be, [zero_heavy], [11], sparse=True, runs=True)
    assert used == [("narrow", 1)] and got == [oracle_commit(be, zero_heavy, 11)]
    got, used = _commit(be, [default], [12], sparse=True, runs=True)
    assert used == [("prefix" if BY_PARTS else "default", 1)] and got == [oracle_commit(be, default, 12)]
    got, used = _commit(be, [zero_heavy, default], [11, 12], sparse=True, runs=True)
    assert used == [("prefix" if BY_PARTS else "default", 2)]
    assert got == [oracle_commit(be, zero_heavy, 11), oracle_commit(be, default, 12)]


def test_dense_columns_take_the_default_table(be18):
    be = be18
    cols = [O.random_field_mont(O.FP, be.n, 650 + i) for i in range(2)]
    blinds = [5, 6]
    want = [oracle_commit(be, c, b) for c, b in zip(cols, blinds)]
    for hints in ({"sparse": True}, {"runs": True}, {"sparse": True, "runs": True}):
        got, used = _commit(be, cols, blinds, **hints)
        assert used == [("default", 2)], hints
        assert got == want, hints


def test_33_columns_come_back_in_order(be18):
    """33 columns are committed as two batches of 17 and 16; every column is different, the results must keep their order"""
    be, n = be18, be18.n
    rng = np.random.default_rng(9)
    cols, blinds = [], []
    for i in range(33):
        col = np.zeros((n, 4), dtype=np.uint64)
        col[rng.choice(n, 40, replace=False)] = O.random_field_mont(O.FP, 40, 700 + i)
        cols.append(col); blinds.append(1000 + i)
    want = [oracle_commit(be, c, b) for c, b in zip(cols, blinds)]
    got, used = _commit(be, cols, blinds)
    assert used == [("default", 17), ("default", 16)]
    assert got == want
    got, used = _commit(be, cols, blinds, sparse=True)
    assert used == [("narrow", 17), ("narrow", 16)]
    assert got == want


def test_zero_column_with_zero_blind_is_the_identity(be18):
    be = be18
    col = np.zeros((be.n, 4), dtype=np.uint64)
    for hints, table in (({}, "default"), ({"sparse": True}, "narrow"), ({"runs": True}, "prefix" if BY_PARTS else "default")):
        got, used = _commit(be, [col], [0], **hints)
        assert used == [(table, 1)], hints
        assert got == [None], hints


def test_narrow_table_at_2_20_points(pkg, ctxs):
    """the window the backend forces on its tables from k = 18 on, over the 2^20 + 1 bases of a k = 20 proof"""
    ctx = ctxs[O.VESTA]
    n = (1 << 20) + 1
    pts = make_points(O.VESTA, n, seed=23)
    uniform, tinyram = scalars_uniform(O.VESTA, n, 24), scalars_tinyram(O.VESTA, n, 25)
    bases = pkg.Bases(ctx, pts, 13 << 8)
    try:
        info = bases.describe()
        assert info["c"] == 13 and info["precomputed"], info
        got = pkg.best_multiexp(ctx, np.stack([uniform, tinyram]), bases)
        assert np.array_equal(affine_of(O.VESTA, got[0]), O.msm(O.VESTA, uniform, pts))
        assert np.array_equal(affine_of(O.VESTA, got[1]), O.msm(O.VESTA, tinyram, pts))
    finally:
        bases.free()


# ---- one k = 20 proof of the benchmark's workload, probed (last: it holds most of the card while it runs) ---------------------------
def test_k20_proof_probed(pkg):
    """TinyRamCircuit<32, 8> at k = 20 on Vesta, as bench.py proves it: keygen and the proof use every commitment table, the
    first column of the first batch on each table matches the oracle's MSM over 2^20 + 1 points, the split quotient satisfies h(x) (x^n - 1) =
    sum_p N_p(x) on the host, and the package's verifier accepts the proof"""
    import torch
    try:
        _prove_k20_probed(pkg)
    finally:                                  # the backend and its columns are gone once the helper has returned
        gc.collect()
        torch.cuda.empty_cache()


def _prove_k20_probed(pkg):
    PL = pkg.plonk
    from tiny_ram_halo2_b200 import programs, tinyram as TR, verifier as V
    tr = programs.longest_loop(32)
    circ, fixed, copies, adv, inst = TR.build(PL, tr, 20, dense=False)
    seen, first = {}, {}

    class Probe(split_probe(PL, seen, monolithic=False, x_seed=20)):
        def _commit_many(self, bases, vecs, blinds, *args, **kw):
            n0 = len(self.lib.calls)
            out = super()._commit_many(bases, vecs, blinds, *args, **kw)
            b0 = 0
            for h, m in self.lib.calls[n0:]:
                name = self._names.get(h)
                if name in ("default", "narrow", "prefix") and name not in first:
                    first[name] = (_u64(vecs[b0]).copy(), blinds[b0], out[b0])
                b0 += m
            return out

    be = Probe(pkg.Context(0, pkg.VESTA), 20, circ.cs.degree())

    def counts():
        out = {}
        for h, m in be.lib.calls:
            name = be._names.get(h, "?")
            b, c = out.get(name, (0, 0))
            out[name] = (b + 1, c + m)
        be.lib.calls.clear()
        return out

    try:
        be.lib = MsmLog(be.lib)
        be._names = table_names(be)
        pk = PL.keygen(be, circ.cs, TR.device_columns(be, fixed), copies)
        in_keygen = counts()
        d_adv, d_inst = TR.device_columns(be, adv), TR.device_columns(be, inst)
        rnd = random.Random(20)
        proof = PL.create_proof(be, pk, d_inst, d_adv, lambda: rnd.randrange(be.p), PL.Blake2bWrite(be.q, be.p))
        in_proof = counts()
        print("k = 20, MSM batches / columns per table: keygen", in_keygen, "proof", in_proof)
        # the proof commits every Lagrange column through the narrow or the prefix table; keygen's fixed and permutation
        # columns take the default one
        assert {"narrow", "prefix"} <= set(in_proof) and "default" in in_keygen, (in_keygen, in_proof)
        assert set(first) == {"default", "narrow", "prefix"}
        for name, (col, blind, got) in first.items():
            assert got == oracle_commit(be, col, blind), name
        lhs, rhs = seen["identity"]
        assert lhs == rhs, "h(x) (x^n - 1) != sum_p N_p(x) at k = 20"
        assert V.verify_proof(be, pk.vk, V.SingleVerifier(be), d_inst, V.Blake2bRead(proof, be.q, be.p)) is None
    finally:
        be.close()
