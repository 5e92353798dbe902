"""GPU parity tests: every hot-path entry point of the C ABI against the CPU oracle, bit-exact.

All calls go through libtrp.so's extern "C" surface (via the ctypes mirror package).  Results are compared as
canonical objects: field vectors limb-for-limb, group elements after normalisation to affine (the Jacobian
representative best_multiexp returns is not unique on the CPU either)."""
import numpy as np
import pytest

from util import O, pm, FIELDS, make_points, scalars_uniform, scalars_tinyram, affine_of, generator
from test_ff_carry_cpu import _edges

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def pkg():
    import __graft_entry__ as ge
    return ge.load_package()


@pytest.fixture(scope="module")
def ctxs(pkg):
    return {O.VESTA: pkg.Context(0, pkg.VESTA), O.PALLAS: pkg.Context(0, pkg.PALLAS)}


# ---- K1 field arithmetic --------------------------------------------------------------------------------------
@pytest.mark.parametrize("curve", [O.VESTA, O.PALLAS])
@pytest.mark.parametrize("which", [0, 1])
def test_field_ops(ctxs, curve, which):
    """every pair of the carry-bound operands of test_ff_carry_cpu (0, 1, p - 1, 2^254 - 1, R, all-ones low limbs, the top word
    at its maximum, ...) through the device's add, sub and mul, sqr and inv on each of them, then uniform random operands"""
    ctx = ctxs[curve]
    field = O.SCALAR_FIELD[curve] if which == 0 else O.BASE_FIELD[curve]
    edge = _edges(FIELDS[field])
    a = np.concatenate([O.ints_to_limbs([x for x in edge for _ in edge]), O.random_field_mont(field, 4000, 1)])
    b = np.concatenate([O.ints_to_limbs([y for _ in edge for y in edge]), O.random_field_mont(field, 4000, 2)])
    for op in ("add", "sub", "mul"):
        assert np.array_equal(ctx.field_op(op, a, b, which_field=which), O.field_op(field, op, a, b)), op
    one = np.concatenate([O.ints_to_limbs(edge), O.random_field_mont(field, 4000, 3)])
    assert np.array_equal(ctx.field_op("sqr", one, which_field=which), O.field_op(field, "sqr", one))
    assert np.array_equal(ctx.field_op("inv", one[:300], which_field=which), O.field_op(field, "inv", one[:300]))


# ---- K4 NTT ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("curve", [O.VESTA, O.PALLAS])
@pytest.mark.parametrize("log_n", list(range(22)) + [23])
def test_best_fft(pkg, ctxs, curve, log_n):
    """every pass plan up to 2^21 and 2^23 (2^22 and 2^24 are below): one pass up to 2^10, two generic passes 2^11 .. 2^18, the
    specialised first pass with a generic second one at 2^19, both passes specialised at 2^20, three passes from 2^21 on"""
    ctx = ctxs[curve]
    field = O.SCALAR_FIELD[curve]
    F = FIELDS[field]
    omega = O.to_mont(field, O.ints_to_limbs([F.root_of_unity(log_n)]))[0]
    batch = 3 if log_n <= 13 else 2 if log_n <= 20 else 1
    a = O.random_field_mont(field, batch << log_n, 30 + log_n).reshape(batch, 1 << log_n, 4)
    got = pkg.best_fft(ctx, a, omega, log_n)
    for b in range(batch):
        assert np.array_equal(got[b], O.fft(field, a[b], log_n, omega)), (log_n, b)


def test_best_fft_rejects_bad_length(pkg, ctxs):
    ctx = ctxs[O.VESTA]
    omega = O.to_mont(O.FP, O.ints_to_limbs([pm.Fp.root_of_unity(4)]))[0]
    with pytest.raises(ValueError):
        pkg.best_fft(ctx, np.zeros((15, 4), dtype=np.uint64), omega, 4)


def test_ntt_roundtrip_2_20(pkg, ctxs):
    """size-independent property at BASELINE size: iNTT(NTT(a)) * n^-1 == a (lagrange_to_coeff o coeff_to_lagrange)."""
    ctx = ctxs[O.VESTA]
    dom = pkg.EvaluationDomain(ctx, 6, 20)
    a = O.random_field_mont(O.FP, 1 << 20, 31)
    lag = dom.coeff_to_lagrange(a)
    assert np.array_equal(dom.lagrange_to_coeff(lag), a)
    # and one spot-check of the forward transform against the oracle at full size
    assert np.array_equal(lag, O.fft(O.FP, a, 20, dom.omega))


# ---- K5 EvaluationDomain ---------------------------------------------------------------------------------------
@pytest.mark.parametrize("curve", [O.VESTA, O.PALLAS])
@pytest.mark.parametrize("j,k", [(6, 1), (6, 4), (6, 8), (6, 11), (3, 5), (4, 6), (9, 7), (2, 6)])
def test_domain_transforms(pkg, ctxs, curve, j, k):
    ctx = ctxs[curve]
    field = O.SCALAR_FIELD[curve]
    dom = pkg.EvaluationDomain(ctx, j, k)
    ek, om, eom = O.domain_info(field, j, k)
    assert dom.extended_k == ek
    assert np.array_equal(dom.omega, om) and np.array_equal(dom.extended_omega, eom)
    n = 1 << k
    cols = O.random_field_mont(field, 3 * n, 50 + k).reshape(3, n, 4)
    coeff = dom.lagrange_to_coeff(cols)
    assert np.array_equal(coeff, O.lagrange_to_coeff(field, j, k, cols).reshape(3, n, 4))
    ext = dom.coeff_to_extended(coeff)
    assert np.array_equal(ext, O.coeff_to_extended(field, j, k, coeff))
    h = O.random_field_mont(field, 1 << ek, 60 + k)
    for divide in (False, True):
        got = dom.extended_to_coeff(h, divide_by_vanishing_poly=divide)
        assert np.array_equal(got, O.extended_to_coeff(field, j, k, h, divide=divide)), divide
    # extended_to_coeff undoes coeff_to_extended (upper coefficients are zero)
    back = dom.extended_to_coeff(ext[1])
    assert np.array_equal(back[:n], coeff[1]) and not back[n:].any()


# ---- K3 MSM ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("curve", [O.VESTA, O.PALLAS])
@pytest.mark.parametrize("flags", [1, 2])      # 1 = per-window bucket sets, 2 = precomputed multiples
@pytest.mark.parametrize("n", [0, 1, 2, 5, 33, 1000, (1 << 12) + 1])
def test_best_multiexp_small(pkg, ctxs, curve, flags, n):
    ctx = ctxs[curve]
    pts = make_points(curve, max(n, 1))[:n]
    sc = scalars_uniform(curve, max(n, 1), 20 + n)[:n]
    bases = pkg.Bases(ctx, pts, flags)
    got = pkg.best_multiexp(ctx, sc, bases)
    want = O.msm(curve, sc, pts) if n else np.zeros(8, dtype=np.uint64)
    assert np.array_equal(affine_of(curve, got), want)


@pytest.mark.parametrize("flags", [1, 2])
def test_best_multiexp_edge_cases(pkg, ctxs, flags):
    """zero / one / p-1 scalars, repeated bases (P + P), inverse pairs (P - P), identity bases, all-equal scalars."""
    curve = O.VESTA
    ctx = ctxs[curve]
    n = 600
    pts = make_points(curve, n, 77)
    p = O.MODULUS[O.FP]
    pts[1] = pts[0]                                   # duplicate base
    neg = pts[2].copy()
    negy = O.field_op(O.FQ, "sub", np.zeros((1, 4), dtype=np.uint64), neg[4:].reshape(1, 4))[0]
    pts[3, :4] = neg[:4]; pts[3, 4:] = negy           # pts[3] = -pts[2]
    pts[7] = 0                                        # identity base
    canon = O.from_mont(O.FP, scalars_uniform(curve, n, 5))
    special = [0, 1, p - 1, 2, (1 << 16) - 1, 1 << 16, (1 << 15), (1 << 255) % p, p - 2]
    for i, v in enumerate(special):
        canon[10 + i] = O.ints_to_limbs([v])[0]
    canon[0] = canon[1] = O.ints_to_limbs([5])[0]     # 5*P + 5*P
    canon[2] = canon[3] = O.ints_to_limbs([9])[0]     # 9*P - 9*P
    sc = O.to_mont(O.FP, canon)
    bases = pkg.Bases(ctx, pts, flags)
    assert np.array_equal(affine_of(curve, pkg.best_multiexp(ctx, sc, bases)), O.msm(curve, sc, pts))
    # all scalars equal (one bucket per window receives everything), all ones, all zero
    for v in (1, 0, 0x1234567, p - 1):
        sc = O.to_mont(O.FP, np.tile(O.ints_to_limbs([v]), (n, 1)))
        assert np.array_equal(affine_of(curve, pkg.best_multiexp(ctx, sc, bases)), O.msm(curve, sc, pts)), v
    # all bases equal: every bucket add hits the doubling path
    same = np.tile(pts[5], (n, 1))
    b2 = pkg.Bases(ctx, same, flags)
    sc = scalars_uniform(curve, n, 9)
    assert np.array_equal(affine_of(curve, pkg.best_multiexp(ctx, sc, b2)), O.msm(curve, sc, same))
    # prefix MSM (n smaller than the loaded bases) and a batch of columns
    sc3 = scalars_uniform(curve, 3 * 100, 10).reshape(3, 100, 4)
    got = pkg.best_multiexp(ctx, sc3, bases)
    for k in range(3):
        assert np.array_equal(affine_of(curve, got[k]), O.msm(curve, sc3[k], pts[:100]))


def test_best_multiexp_rejects_length_mismatch(pkg, ctxs):
    ctx = ctxs[O.VESTA]
    bases = pkg.Bases(ctx, make_points(O.VESTA, 8))
    with pytest.raises(ValueError):
        pkg.best_multiexp(ctx, np.zeros((9, 4), dtype=np.uint64), bases)


@pytest.mark.parametrize("shape", ["uniform", "tinyram"])
def test_best_multiexp_2_16(pkg, ctxs, shape):
    curve = O.VESTA
    ctx = ctxs[curve]
    n = (1 << 16) + 1
    pts = make_points(curve, n)
    sc = scalars_uniform(curve, n) if shape == "uniform" else scalars_tinyram(curve, n)
    bases = pkg.Bases(ctx, pts)
    assert np.array_equal(affine_of(curve, pkg.best_multiexp(ctx, sc, bases)), O.msm(curve, sc, pts))


def test_commit_lagrange_linearity_2_20(pkg, ctxs):
    """BASELINE size (k = 20): commit(a) + commit(b) == commit(a + b) with independent blinds, both scalar shapes;
    plus a direct oracle comparison of one of the three MSMs."""
    curve = O.VESTA
    ctx = ctxs[curve]
    k = 20
    n = 1 << k
    pts = make_points(curve, 2 * n + 1)
    params = pkg.Params(ctx, k, pts[:n], pts[n:2 * n], pts[2 * n])
    a = scalars_uniform(curve, n, 1); b = scalars_tinyram(curve, n, 2)
    ra, rb = scalars_uniform(curve, 2, 3)
    ab = ctx.field_op("add", a, b); rab = ctx.field_op("add", ra.reshape(1, 4), rb.reshape(1, 4))[0]
    ca = affine_of(curve, params.commit_lagrange(a, ra))
    cb = affine_of(curve, params.commit_lagrange(b, rb))
    cab = affine_of(curve, params.commit_lagrange(ab, rab))
    assert np.array_equal(O.point_add(curve, ca, cb), cab)
    want = O.msm(curve, np.concatenate([b, rb.reshape(1, 4)]), np.concatenate([pts[n:2 * n], pts[2 * n:2 * n + 1]]))
    assert np.array_equal(cb, want)


def test_point_range_split_and_points_sum(pkg, ctxs):
    """SURVEY 8(e)-2 on one device: the MSM over [0, n) equals trp_points_sum of the MSMs over G disjoint slices (each with
    its own pre-sharded base handle); also the identity / single-element / cancelling cases of trp_points_sum."""
    import ctypes
    from tiny_ram_halo2_b200 import parallel as PL
    from tiny_ram_halo2_b200._lib import ptr
    curve = O.VESTA
    ctx = ctxs[curve]
    n, G = 3001, 4
    pts = make_points(curve, n)
    sc = scalars_uniform(curve, n, 12)
    parts = np.zeros((G, 3, 4), dtype=np.uint64)
    for r in range(G):
        lo, hi = PL.split_point_range(n, G, r)
        parts[r] = pkg.best_multiexp(ctx, sc[lo:hi], pkg.Bases(ctx, pts[lo:hi]))
    out = np.zeros((3, 4), dtype=np.uint64)
    ctx.check(ctx.lib.trp_points_sum(ctx.handle, ptr(parts), G, ptr(out)))
    assert np.array_equal(affine_of(curve, out), O.msm(curve, sc, pts))
    # identity inputs, P + (-P), empty sum
    neg = parts[0].copy()
    neg[1] = O.field_op(O.FQ, "sub", np.zeros((1, 4), dtype=np.uint64), parts[0][1].reshape(1, 4))[0]
    for arr, want in ((np.stack([parts[0], neg]), np.zeros(8, dtype=np.uint64)),
                      (np.stack([np.zeros((3, 4), dtype=np.uint64), parts[1]]), affine_of(curve, parts[1])),
                      (np.stack([parts[2], parts[2]]), O.point_add(curve, affine_of(curve, parts[2]), affine_of(curve, parts[2])))):
        ctx.check(ctx.lib.trp_points_sum(ctx.handle, ptr(np.ascontiguousarray(arr)), len(arr), ptr(out)))
        assert np.array_equal(affine_of(curve, out), want)
    ctx.check(ctx.lib.trp_points_sum(ctx.handle, None, 0, ptr(out)))
    assert not out.any()


@pytest.mark.parametrize("curve", [O.VESTA, O.PALLAS])
@pytest.mark.parametrize("n", [1, 15, 16, 17, 4097, 70001])
def test_points_prefix_sum(pkg, ctxs, curve, n):
    """trp_dev_points_prefix_sum against a sequential sum with the oracle's point addition: identity inputs, P + P (the doubling
    case), P + (-P) (a prefix that IS the identity), chunk / segment boundaries (16 points per thread, 256 chunks per segment)"""
    import torch
    if curve == O.PALLAS and n > 4097:
        pytest.skip("one curve is enough at this size")
    ctx = ctxs[curve]
    pts = make_points(curve, n).copy()
    base = O.BASE_FIELD[curve]
    neg = lambda P: np.concatenate([P[:4], O.field_op(base, "sub", np.zeros((1, 4), dtype=np.uint64), P[4:].reshape(1, 4))[0]])
    if n >= 15:
        pts[1] = neg(pts[0])                  # prefix[1] = identity
        pts[3] = pts[2]                       # the accumulator equals the next input: the exact P + P case
        pts[4] = 0                            # an identity input
        pts[7] = neg(pts[6])
    if n >= 4097:
        pts[16 * 256 - 1] = 0
        pts[16 * 256] = pts[16 * 256 - 2]
    want = np.zeros((n, 8), dtype=np.uint64)
    acc = np.zeros(8, dtype=np.uint64)
    for i in range(n):
        acc = O.point_add(curve, acc, pts[i])
        want[i] = acc
    d = torch.from_numpy(pts.view(np.int64)).cuda()
    out = torch.empty_like(d)
    torch.cuda.synchronize()
    ctx.check(ctx.lib.trp_dev_points_prefix_sum(ctx.handle, d.data_ptr(), n, out.data_ptr()))
    ctx.sync()
    assert np.array_equal(out.cpu().numpy().view(np.uint64).reshape(n, 8), want)
    ctx.check(ctx.lib.trp_dev_points_prefix_sum(ctx.handle, d.data_ptr(), n, d.data_ptr()))          # in place
    ctx.sync()
    assert np.array_equal(d.cpu().numpy().view(np.uint64).reshape(n, 8), want)


def test_commitment_by_parts(pkg, ctxs):
    """sum_i z_i G_i = sum_j (z_j - z_{j+1}) Q_j with Q = prefix sums of G (z_n = 0): the identity behind GpuBackend's commitment
    of grand-product columns through their sparse differences; both sides on the device, and against the oracle's MSM"""
    import torch
    curve = O.VESTA
    ctx = ctxs[curve]
    n = 6000
    G = make_points(curve, n)
    rng = np.random.default_rng(3)
    vals = scalars_uniform(curve, 40, 9)
    z = np.zeros((n, 4), dtype=np.uint64)
    i = 0
    while i < n:                               # runs of equal values, some of them zero, a dense stretch in the middle
        ln = int(rng.integers(1, 400)) if not (2000 <= i < 2300) else 1
        z[i:i + ln] = 0 if rng.random() < 0.2 else vals[int(rng.integers(0, 40))]
        i += ln
    d = torch.from_numpy(G.view(np.int64)).cuda()
    torch.cuda.synchronize()
    ctx.check(ctx.lib.trp_dev_points_prefix_sum(ctx.handle, d.data_ptr(), n, d.data_ptr()))
    ctx.sync()
    Q = d.cpu().numpy().view(np.uint64).reshape(n, 8)
    field = O.SCALAR_FIELD[curve]
    e = z.copy()
    e[:n - 1] = O.field_op(field, "sub", z[:n - 1], z[1:])
    direct = pkg.best_multiexp(ctx, z, pkg.Bases(ctx, G))
    by_parts = pkg.best_multiexp(ctx, e, pkg.Bases(ctx, Q))
    assert np.array_equal(affine_of(curve, by_parts), affine_of(curve, direct))
    assert np.array_equal(affine_of(curve, direct), O.msm(curve, z, G))
    assert int((e != 0).any(axis=1).sum()) < int((z != 0).any(axis=1).sum()) // 3


# ---- the upper half of BASELINE.json configs[1] / configs[2]: 2^22 and 2^24, compared with the oracle byte for byte ---------
_LARGE = {}


def _large_msm_case(log_n):
    """inputs and the oracle's answer, computed once per size (the oracle's best_multiexp takes ~10-40 s on the host cores)"""
    if log_n not in _LARGE:
        n = (1 << log_n) + 1                                   # commit_lagrange shape: n + 1 with the blind's base
        pts = make_points(O.VESTA, n)
        sc = scalars_uniform(O.VESTA, n, 20 + log_n)
        sc[n // 2:n // 2 + 1000] = scalars_tinyram(O.VESTA, 1000, 41)         # a run of 0/1 and small scalars inside the uniform ones
        _LARGE.clear()                                         # one size at a time: 2^24 points are 1 GiB on the host
        _LARGE[log_n] = (pts, sc, O.msm(O.VESTA, sc, pts))
    return _LARGE[log_n]


@pytest.mark.parametrize("log_n,flags", [(22, 2), (22, 1), (24, 2), (24, 1)])
def test_best_multiexp_2_22_2_24(pkg, ctxs, log_n, flags):
    """flags 2 = precomputed window multiples (the default table), 1 = one bucket set per window (no table)"""
    ctx = ctxs[O.VESTA]
    pts, sc, want = _large_msm_case(log_n)
    bases = pkg.Bases(ctx, pts, flags)
    try:
        info = bases.describe()
        assert info["precomputed"] == (flags == 2)
        assert np.array_equal(affine_of(O.VESTA, pkg.best_multiexp(ctx, sc, bases)), want), info
    finally:
        bases.free()


@pytest.mark.parametrize("curve", [O.VESTA, O.PALLAS])
@pytest.mark.parametrize("log_n", [22, 24])
def test_best_fft_2_22_2_24(pkg, ctxs, curve, log_n):
    ctx = ctxs[curve]
    field = O.SCALAR_FIELD[curve]
    omega = O.to_mont(field, O.ints_to_limbs([FIELDS[field].root_of_unity(log_n)]))[0]
    a = O.random_field_mont(field, 1 << log_n, 30 + log_n)
    got = pkg.best_fft(ctx, a, omega, log_n)
    want = O.fft(field, a, log_n, omega)
    assert np.array_equal(got, want)
    # and back: the inverse transform with omega^-1, scaled by 2^-log_n, returns the input (size-independent property)
    omega_inv = O.field_op(field, "inv", omega.reshape(1, 4))[0]
    back = pkg.best_fft(ctx, got, omega_inv, log_n)
    ninv = O.to_mont(field, O.ints_to_limbs([pow(1 << log_n, -1, O.MODULUS[field])]))
    assert np.array_equal(O.field_op(field, "mul", back, np.repeat(ninv, 1 << log_n, axis=0)), a)


@pytest.mark.parametrize("k", [20, 22])
def test_domain_transforms_k20_k22(pkg, ctxs, k):
    """lagrange_to_coeff / coeff_to_extended / extended_to_coeff at the proof sizes of configs[3] / configs[4] (extended domains
    of 2^23 and 2^25 values), each against the oracle"""
    ctx = ctxs[O.VESTA]
    j = 6
    dom = pkg.EvaluationDomain(ctx, j, k)
    n = 1 << k
    col = O.random_field_mont(O.FP, n, 50 + k).reshape(1, n, 4)
    coeff = dom.lagrange_to_coeff(col)
    assert np.array_equal(coeff, O.lagrange_to_coeff(O.FP, j, k, col).reshape(1, n, 4))
    ext = dom.coeff_to_extended(coeff)
    assert np.array_equal(ext, O.coeff_to_extended(O.FP, j, k, coeff))
    back = dom.extended_to_coeff(ext[0])
    assert np.array_equal(back[:n], coeff[0]) and not back[n:].any()
    h = O.random_field_mont(O.FP, 1 << dom.extended_k, 60 + k)
    assert np.array_equal(dom.extended_to_coeff(h, divide_by_vanishing_poly=True), O.extended_to_coeff(O.FP, j, k, h, divide=True))
    dom.free()


def test_tma_staged_ntt_pass_matches_the_default(pkg):
    """the opt-in TMA-staged pass kernel (TRP_NTT_TMA=1: cp.async.bulk.tensor + mbarrier tile loads, csrc/ntt.cu) against the
    oracle, in a subprocess because the switch is read once per process: forward NTTs of 2^11 .. 2^20 (two- and three-level pass
    plans), lagrange_to_coeff, the zero-padded coeff_to_extended and a coset transform through the device entry points"""
    import os, subprocess, sys, textwrap
    code = textwrap.dedent("""
        import sys
        sys.path.insert(0, %r); sys.path.insert(0, %r)
        import numpy as np
        from util import O, pm
        import __graft_entry__ as ge
        pkg = ge.load_package()
        ctx = pkg.Context(0, pkg.VESTA)
        for log_n in (11, 13, 16, 20):
            omega = O.to_mont(O.FP, O.ints_to_limbs([pm.Fp.root_of_unity(log_n)]))[0]
            a = O.random_field_mont(O.FP, 2 << log_n, 90 + log_n).reshape(2, 1 << log_n, 4)
            got = pkg.best_fft(ctx, a, omega, log_n)
            for b in range(2):
                assert np.array_equal(got[b], O.fft(O.FP, a[b], log_n, omega)), log_n
        for j, k in ((6, 11), (6, 14), (3, 12)):
            dom = pkg.EvaluationDomain(ctx, j, k)
            n = 1 << k
            cols = O.random_field_mont(O.FP, 2 * n, 70 + k).reshape(2, n, 4)
            coeff = dom.lagrange_to_coeff(cols)
            assert np.array_equal(coeff, O.lagrange_to_coeff(O.FP, j, k, cols).reshape(2, n, 4))
            assert np.array_equal(dom.coeff_to_extended(coeff), O.coeff_to_extended(O.FP, j, k, coeff))
            h = O.random_field_mont(O.FP, 1 << dom.extended_k, 60 + k)
            assert np.array_equal(dom.extended_to_coeff(h, divide_by_vanishing_poly=True), O.extended_to_coeff(O.FP, j, k, h, divide=True))
        print("tma ok")
    """) % (os.path.dirname(os.path.dirname(os.path.abspath(__file__))), os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, "-c", code], env={**os.environ, "TRP_NTT_TMA": "1"}, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0 and "tma ok" in out.stdout, out.stderr[-3000:]
