"""GPU parity of the kernel paths that only multi-GPU proofs and proof-size inputs reach: the row-sliced quotient program
(trp_dev_quotient_eval_rows), the inner-product argument at k = 10 / 12 and its point-range split, the point prefix sum past its
third scan level, tile scans of more than 256 tiles (grand product, batch inversion, kate_division) and
trp_dev_linear_combination with the regrouping of the sharded backend.

Sharding is emulated on ONE device: each rank's arguments go through the same entry points in turn, and the partial results are
combined the way the sharded code combines them.  Every expected value comes from the oracle (oracle/oracle.cpp through
oracle.py, or Python ints); the few comparisons between two device paths are extra cross-checks on top of that."""
import random

import numpy as np
import pytest

from util import O, pm, make_points, generator, affine_of, FIELDS

pytestmark = pytest.mark.gpu

TRP_E_INVALID = -1


@pytest.fixture(scope="module")
def pkg():
    import __graft_entry__ as ge
    return ge.load_package()


@pytest.fixture(scope="module")
def P(pkg):
    from tiny_ram_halo2_b200 import poly
    return poly


@pytest.fixture(scope="module")
def ctxs(pkg):
    # torch tensor operations and trp_dev_* calls share one stream, so the calls below are ordered without explicit fences
    out = {O.VESTA: pkg.Context(0, pkg.VESTA), O.PALLAS: pkg.Context(0, pkg.PALLAS)}
    for ctx in out.values():
        ctx.bind_torch_stream()
    return out


# ---- helpers ---------------------------------------------------------------------------------------------------------------
def limbs(vals):
    """canonical ints -> (n, 4) uint64 limbs"""
    return np.frombuffer(b"".join(int(v).to_bytes(32, "little") for v in vals), dtype=np.uint64).reshape(-1, 4).copy()


def to_ints(arr):
    b = np.ascontiguousarray(arr, dtype=np.uint64).tobytes()
    return [int.from_bytes(b[i:i + 32], "little") for i in range(0, len(b), 32)]


def mont(field, vals):
    return O.to_mont(field, limbs(vals))


def unmont(field, arr):
    return to_ints(O.from_mont(field, arr))


def dev(arr):
    import torch
    return torch.from_numpy(np.ascontiguousarray(arr, dtype=np.uint64).view(np.int64)).cuda()


def host(t):
    return t.cpu().numpy().view(np.uint64)


def mont_powers(field, x, n):
    """(n, 4) Montgomery x^i, i < n, by doubling with the oracle's vector multiplication"""
    out = np.empty((n, 4), dtype=np.uint64)
    out[0] = mont(field, [1])[0]
    m, xm = 1, np.asarray(x, dtype=np.uint64).reshape(1, 4)
    while m < n:
        c = min(m, n - m)
        out[m:m + c] = O.field_op(field, "mul", out[:c], np.repeat(xm, c, axis=0))
        xm = O.field_op(field, "mul", xm, xm)
        m += c
    return out


def rejects(ctx, call):
    """call() must fail with TRP_E_INVALID before any kernel is launched"""
    before = ctx.launches
    rc = call()
    assert rc == TRP_E_INVALID, rc
    assert ctx.launches == before


# ---- A. row-sliced quotient: trp_dev_quotient_eval_rows ------------------------------------------------------------------------
class Coset:
    """coefficient columns moved to one size-n coset on the device (trp_dev_coeff_to_coset), the X values of that coset, and the
    oracle's evaluation of a program over the whole coset"""

    def __init__(self, ctx, dom, coeff, cs):
        import torch
        self.ctx, self.dom, self.cs = ctx, dom, cs
        self.field = O.SCALAR_FIELD[ctx.curve]
        self.n = dom.n
        self.d_coeff = dev(coeff)
        self.d_cols = torch.empty_like(self.d_coeff)
        ctx.check(ctx.lib.trp_dev_coeff_to_coset(dom.handle, self.d_coeff.data_ptr(), self.d_cols.data_ptr(), len(coeff), cs))
        self.h_cols = host(self.d_cols)
        p = O.MODULUS[self.field]
        zeta, eom = unmont(self.field, np.stack([dom.g_coset, dom.extended_omega]))
        x0 = mont(self.field, [zeta * pow(eom, cs, p) % p])[0]
        # X on coset cs: zeta * ext_omega^(cs + i * 2^(ext_k - k)) = (zeta * ext_omega^cs) * omega^i
        self.xs = O.field_op(self.field, "mul", mont_powers(self.field, dom.omega, self.n), np.repeat(x0.reshape(1, 4), self.n, axis=0))

    def want(self, P, prog):
        consts = P._to_mont_limbs(prog.consts, O.MODULUS[self.field])
        return O.quotient_vm(self.field, prog.code, prog.n_regs, consts, list(self.h_cols), self.n, self.xs, self.n)

    def whole(self, ev, prog):
        """the same coset through trp_dev_quotient_eval, contiguous output (cross-check)"""
        import torch
        from tiny_ram_halo2_b200._lib import Q_CONTIGUOUS
        out = torch.zeros((self.n, 4), dtype=torch.int64, device="cuda")
        ev.evaluate_device(prog, self.dom, [c.data_ptr() for c in self.d_cols], out.data_ptr(), coset=self.cs | Q_CONTIGUOUS)
        return host(out)

    def slice_cols(self, row0, nrows, hb, ha):
        """rows [row0 - hb, row0 + nrows + ha) of every column, cyclic"""
        import torch
        idx = (torch.arange(nrows + hb + ha, device="cuda") + (row0 - hb)) % self.n
        return self.d_cols[:, idx].contiguous()

    def run_rows(self, ev, prog, cols, row0, nrows, hb, ha):
        import torch
        out = torch.full((nrows, 4), -1, dtype=torch.int64, device="cuda")
        ev.evaluate_device_rows(prog, self.dom, [c.data_ptr() for c in cols], out.data_ptr(), self.cs, row0, nrows, hb, ha)
        return host(out)


def halo_program(P, hb, ha, y):
    """gate-like folds whose rotations reach exactly -hb and +ha, plus X terms (LinearTerm) so that row0 enters the X index"""
    A, B, C, S = (P.Poly(i) for i in range(4))
    exprs = [S * (A * B - C),
             A.with_rotation(-hb) * B.with_rotation(ha) - C,
             S * (A.with_rotation(ha) + P.LinearTerm(y) * C.with_rotation(-hb)),
             P.LinearTerm(1) * A + B.with_rotation(-hb) * B.with_rotation(-hb)]
    h = P.ConstantTerm(0)
    for e in exprs:
        h = h * y + e
    return h


def deep_program(P, depth):
    """nested DistributePowers: each level keeps its base and accumulator live, ~2 registers per level"""
    h = P.Poly(0)
    for d in range(depth):
        h = P.DistributePowers([h, P.Poly(d % 4, (d % 3) - 1) * P.LinearTerm(d + 2)], P.Poly((d + 1) % 4))
    return h


def compile_ast(P, ast, curve=O.VESTA):
    """lower an Ast with the constants reduced modulo the curve's scalar field (what Evaluator.compile does)"""
    return P.compile_ast(ast, O.MODULUS[O.SCALAR_FIELD[curve]])


Y = 0x1234567890abcdef1234567890abcdef1234567890abcdef


@pytest.mark.parametrize("curve", [O.VESTA, O.PALLAS])
def test_quotient_rows_match_the_oracle(pkg, P, ctxs, curve):
    from tiny_ram_halo2_b200 import parallel as PL
    import torch
    ctx = ctxs[curve]
    field = O.SCALAR_FIELD[curve]
    j, k = 6, 10
    dom = pkg.EvaluationDomain(ctx, j, k)
    n = dom.n
    period = dom.extended_len() // n
    coeff = O.random_field_mont(field, 4 * n, 300 + curve).reshape(4, n, 4)
    ev = P.new_evaluator(ctx)
    cos = {cs: Coset(ctx, dom, coeff, cs) for cs in (0, 3, period - 1)}

    def check(c, prog, want, row0, nrows, hb, ha, cols=None):
        cols = c.slice_cols(row0, nrows, hb, ha) if cols is None else cols
        got = c.run_rows(ev, prog, cols, row0, nrows, hb, ha)
        assert np.array_equal(got, want[row0:row0 + nrows]), (c.cs, row0, nrows, hb, ha)

    # every slice of G = 1, 2, 4, 8 devices with the sharded backend's halo, input packed by parallel.pack_row_slices
    H = 16
    prog = compile_ast(P, halo_program(P, H, H, Y), curve)
    for c in cos.values():
        want = c.want(P, prog)
        assert np.array_equal(c.whole(ev, prog), want), c.cs
        for G in (1, 2, 4, 8):
            S = n // G
            send = torch.zeros((G, 4, S + 2 * H, 4), dtype=torch.int64, device="cuda")
            PL.pack_row_slices(c.d_cols, 4, n, G, H, H, send)
            for r in range(G):
                row0, nrows = PL.row_slice_bounds(n, G, r)
                check(c, prog, want, row0, nrows, H, H, cols=send[r])
    # asymmetric halos (TinyRAM reads rows -6 .. +1) and a one-sided halo, the program rotating by exactly -hb and +ha
    c = cos[3]
    for hb, ha in ((6, 1), (0, 16), (1, 0)):
        prog = compile_ast(P, halo_program(P, hb, ha, Y), curve)
        want = c.want(P, prog)
        for r in range(4):
            check(c, prog, want, *PL.row_slice_bounds(n, 4, r), hb, ha)
        # short slices at both ends of the coset: the halo wraps below row 0 and above row n - 1
        for nrows in (1, 2, 127, 128, 129, 300, 777):
            for row0 in (0, n - nrows, 5, n - nrows - 3):
                check(c, prog, want, row0, nrows, hb, ha)
    # a register-hungry program: fewer than 128 threads per CTA
    prog = compile_ast(P, deep_program(P, 27), curve)
    assert prog.n_regs > 50
    c = cos[period - 1]
    want = c.want(P, prog)
    for row0, nrows in ((0, n), (0, 129), (n - 200, 200), (n // 2 - 65, 130), (n - 1, 1)):
        check(c, prog, want, row0, nrows, 1, 1)


def test_quotient_rows_tinyram_shape(pkg, P, ctxs):
    """j = 6, k = 20 (the flagship proof's domain), one coset split over 8 devices as ShardedGpuBackend.quotient does it: halo 16
    on both sides, slices packed by parallel.pack_row_slices, a TinyRAM-like program rotating by -6 .. +1 with X terms"""
    from tiny_ram_halo2_b200 import parallel as PL
    import torch
    ctx = ctxs[O.VESTA]
    j, k, G, H, ncols = 6, 20, 8, 16, 6
    dom = pkg.EvaluationDomain(ctx, j, k)
    n = dom.n
    coeff = O.random_field_mont(O.FP, ncols * n, 320).reshape(ncols, n, 4)
    c = Coset(ctx, dom, coeff, 4)
    col = [P.Poly(i) for i in range(ncols)]
    s = col[5]
    exprs = [s * (col[0].with_rotation(1) - col[0] - col[1]),
             s * col[2] * (col[2] - 1),
             (col[3].with_rotation(-6) + col[4].with_rotation(-3)) * col[1].with_rotation(1) - col[0],
             s * P.LinearTerm(5) * col[4].with_rotation(-1) + P.LinearTerm(1),
             col[1] * col[2] * col[3] * col[4].with_rotation(-6)]
    h = P.ConstantTerm(0)
    for e in exprs:
        h = h * Y + e
    ev = P.new_evaluator(ctx)
    prog = compile_ast(P, h)
    want = c.want(P, prog)
    S = n // G
    send = torch.zeros((G, ncols, S + 2 * H, 4), dtype=torch.int64, device="cuda")
    PL.pack_row_slices(c.d_cols, ncols, n, G, H, H, send)
    got = np.concatenate([c.run_rows(ev, prog, send[r], r * S, S, H, H) for r in range(G)])
    assert np.array_equal(got, want)
    assert np.array_equal(c.whole(ev, prog), want)


def test_quotient_rows_rejections(pkg, P, ctxs):
    """malformed slices fail with TRP_E_INVALID before anything is launched, and the output is left alone"""
    import torch
    from tiny_ram_halo2_b200._lib import Q_CONTIGUOUS, ptr
    import ctypes
    ctx = ctxs[O.VESTA]
    dom = pkg.EvaluationDomain(ctx, 6, 8)
    n = dom.n
    period = dom.extended_len() // n
    cols = torch.zeros((4, n, 4), dtype=torch.int64, device="cuda")
    out = torch.full((n, 4), 7, dtype=torch.int64, device="cuda")
    ev = P.new_evaluator(ctx)

    def call(prog, coset, row0, nrows, hb, ha):
        consts = P._to_mont_limbs(prog.consts, ev.modulus)
        code = np.ascontiguousarray(prog.code)
        colp = (ctypes.c_void_p * 4)(*[c.data_ptr() for c in cols])
        return lambda: ctx.lib.trp_dev_quotient_eval_rows(dom.handle, ptr(code), len(code), prog.n_regs, ptr(consts), len(prog.consts),
                                                          colp, 4, coset, row0, nrows, hb, ha, out.data_ptr())

    ok = compile_ast(P, halo_program(P, 6, 1, Y))
    ctx.check(call(ok, 1, 0, 64, 6, 1)())                                 # the well-formed call runs
    out.fill_(7)
    A = P.Poly(0)
    rejects(ctx, call(compile_ast(P, A.with_rotation(2) * A), 1, 0, 64, 6, 1))      # reads beyond the halo after the slice
    rejects(ctx, call(compile_ast(P, A.with_rotation(-7) + A), 1, 0, 64, 6, 1))     # ... and before it
    rejects(ctx, call(ok, 1, n - 10, 11, 6, 1))                                 # row0 + nrows > n
    rejects(ctx, call(ok, 1, n, 1, 6, 1))                                       # row0 == n
    rejects(ctx, call(ok, 1, 0, 0, 6, 1))                                       # nrows == 0
    rejects(ctx, call(ok, period, 0, 64, 6, 1))                                 # no such coset
    rejects(ctx, call(ok, 1 | Q_CONTIGUOUS, 0, 64, 6, 1))                       # the layout flag is not a coset index here
    assert (host(out) == 7).all()


# ---- B. the inner-product argument at k = 10 / 12, whole and point-range split -----------------------------------------------
class Transcript:
    """Deterministic stand-in for the Blake2b transcript (as in test_gpu_ipa.py): records what is written, challenges come from a
    seeded stream."""

    def __init__(self, seed, p):
        self.rng, self.p, self.log = random.Random(seed), p, []

    def write_point(self, P):
        self.log.append(("point", np.asarray(P, dtype=np.uint64).copy()))

    def write_scalar(self, s):
        self.log.append(("scalar", s))

    def squeeze_challenge_scalar(self):
        return self.rng.randrange(1, self.p)


def oracle_ipa(curve, k, g, w, u, rand, transcript, p_poly, p_blind, x_3):
    """pm.ipa_create_proof line for line, with the oracle's MSM (O.msm) and generator collapse (O.generator_collapse) in place of
    the Python curve model.  g: (n, 8) affine limbs; w, u: (8,).  Returns each round's state: p' and s (the challenge products,
    G'_i = sum_t s_t G_{t cur + i}) as Python ints, the U / W scalars, L_j and R_j."""
    field = O.SCALAR_FIELD[curve]
    F = FIELDS[field]
    p, n = F.p, 1 << k
    uw = np.stack([u, w])
    s_poly = [rand() for _ in range(n)]
    s_at_x3 = pm.eval_polynomial(F, s_poly, x_3)
    s_poly[0] = (s_poly[0] - s_at_x3) % p
    s_poly_blind = rand()
    transcript.write_point(O.msm(curve, mont(field, s_poly + [s_poly_blind]), np.concatenate([g, w.reshape(1, 8)])))
    xi = transcript.squeeze_challenge_scalar()
    z = transcript.squeeze_challenge_scalar()
    p_prime = [(s * xi + c) % p for s, c in zip(s_poly, p_poly)]
    v = pm.eval_polynomial(F, p_prime, x_3)
    p_prime[0] = (p_prime[0] - v) % p
    f = (s_poly_blind * xi + p_blind) % p
    b, cur = [], 1
    for _ in range(n):
        b.append(cur)
        cur = cur * x_3 % p
    g_prime, s = g.copy(), [1]
    rounds = []
    for j in range(k):
        half = 1 << (k - j - 1)
        value_l_j = pm.compute_inner_product(F, p_prime[half:], b[:half])
        value_r_j = pm.compute_inner_product(F, p_prime[:half], b[half:])
        l_rand, r_rand = rand(), rand()
        l_j = O.msm(curve, mont(field, p_prime[half:] + [value_l_j * z % p, l_rand]), np.concatenate([g_prime[:half], uw]))
        r_j = O.msm(curve, mont(field, p_prime[:half] + [value_r_j * z % p, r_rand]), np.concatenate([g_prime[half:], uw]))
        rounds.append({"p": list(p_prime), "s": list(s), "u_coef": (value_l_j * z % p, value_r_j * z % p), "w_coef": (l_rand, r_rand),
                       "L": l_j, "R": r_j})
        transcript.write_point(l_j)
        transcript.write_point(r_j)
        u_j = transcript.squeeze_challenge_scalar()
        u_j_inv = F.inv(u_j)
        for i in range(half):
            p_prime[i] = (p_prime[i] + p_prime[i + half] * u_j_inv) % p
            b[i] = (b[i] + b[i + half] * u_j) % p
        p_prime, b = p_prime[:half], b[:half]
        g_prime = O.generator_collapse(curve, g_prime, limbs([u_j])[0])
        s = [e for t in s for e in (t, t * u_j % p)]
        f = (f + l_rand * u_j_inv + r_rand * u_j) % p
    assert len(p_prime) == 1
    transcript.write_scalar(p_prime[0])
    transcript.write_scalar(f)
    return rounds


def ipa_inputs(curve, k):
    field = O.SCALAR_FIELD[curve]
    F = FIELDS[field]
    rng = random.Random(500 + k)
    n = 1 << k
    g = make_points(curve, n, 60 + k)
    gen = generator(curve)
    w, u = (O.point_mul(curve, limbs([rng.randrange(1, F.p)])[0], gen) for _ in range(2))
    p_poly = [rng.randrange(F.p) for _ in range(n)]
    p_blind, x_3 = rng.randrange(F.p), rng.randrange(F.p)
    draws = [rng.randrange(F.p) for _ in range(n + 1 + 2 * k)]
    return g, w, u, p_poly, p_blind, x_3, draws


@pytest.mark.parametrize("curve", [O.VESTA, O.PALLAS])
@pytest.mark.parametrize("k", [10, 12])
def test_ipa_create_proof_against_collapse_oracle(pkg, ctxs, curve, k):
    """ipa.create_proof (round scalars over the resident table, no generator collapse) against the collapse-based oracle IPA,
    transcript entry for entry; then every round's L_j / R_j recomputed rank by rank for G = 2, 4, 8 devices as the point-range
    split of ipa.create_proof does it (round scalars over [lo, lo + n / G), U / W terms on rank 0, MSM over the rank's own table,
    trp_dev_points_sum of the partial sums)"""
    import torch
    ctx = ctxs[curve]
    field = O.SCALAR_FIELD[curve]
    F = FIELDS[field]
    n = 1 << k
    g, w, u, p_poly, p_blind, x_3, draws = ipa_inputs(curve, k)
    it1, it2 = iter(draws), iter(draws)
    t_want = Transcript(9, F.p)
    rounds = oracle_ipa(curve, k, g, w, u, lambda: next(it1), t_want, p_poly, p_blind, x_3)
    params = pkg.ipa.IpaParams(ctx, k, g, w, u)
    try:
        t_got = Transcript(9, F.p)
        pkg.ipa.create_proof(params, lambda: next(it2), t_got, mont(field, p_poly), p_blind, x_3)
        assert len(t_got.log) == len(t_want.log) == 1 + 2 * k + 2
        for i, ((kind_g, val_g), (kind_w, val_w)) in enumerate(zip(t_got.log, t_want.log)):
            assert kind_g == kind_w, i
            assert (np.array_equal(val_g, val_w) if kind_g == "point" else val_g == val_w), i
        lib = ctx.lib
        seen = set()
        for j, st in enumerate(rounds):
            cur = n >> j
            d_p, d_s = dev(mont(field, st["p"])), dev(mont(field, st["s"]))
            d_u, d_w = dev(mont(field, list(st["u_coef"]))), dev(mont(field, list(st["w_coef"])))
            for G in (2, 4, 8):
                cnt = n // G
                seen.add("cur > cnt" if cur > cnt else "cur < cnt" if cur < cnt else "cur == cnt")
                parts = torch.zeros((G, 2, 12), dtype=torch.int64, device="cuda")
                for r in range(G):
                    lo = r * cnt
                    if cur > cnt and lo % cur >= cur // 2:
                        seen.add("slice in the high half")
                    cols = torch.zeros((2, cnt + 2, 4), dtype=torch.int64, device="cuda")
                    ctx.check(lib.trp_dev_ipa_round_scalars(ctx.handle, 0, d_p.data_ptr(), d_s.data_ptr(), cur, lo, cnt, cnt + 2, cols.data_ptr()))
                    if r == 0:
                        cols[:, cnt] = d_u
                        cols[:, cnt + 1] = d_w
                    ctx.check(lib.trp_dev_msm_batch(ctx.handle, params.table(r, G), cols.data_ptr(), cnt + 2, 2, parts[r].data_ptr()))
                sums = torch.zeros((2, 12), dtype=torch.int64, device="cuda")
                for c_ in range(2):
                    part = parts[:, c_].contiguous()
                    ctx.check(lib.trp_dev_points_sum(ctx.handle, part.data_ptr(), G, sums[c_].data_ptr()))
                got = host(sums).reshape(2, 3, 4)
                assert np.array_equal(affine_of(curve, got[0]), st["L"]), (j, G)
                assert np.array_equal(affine_of(curve, got[1]), st["R"]), (j, G)
        assert seen >= {"cur > cnt", "cur < cnt", "slice in the high half"}
    finally:
        params.free()


@pytest.mark.parametrize("curve", [O.VESTA, O.PALLAS])
def test_ipa_round_scalars_and_s_double_elementwise(ctxs, curve):
    """trp_dev_ipa_round_scalars and trp_dev_ipa_s_double element by element against Python ints, several CTAs each, slices that
    start inside the low half, straddle the middle and start in the high half; padding past `count` is left alone"""
    import torch
    ctx = ctxs[curve]
    field = O.SCALAR_FIELD[curve]
    F = FIELDS[field]
    rng = random.Random(77)
    n, cur = 1 << 12, 1 << 10
    half = cur // 2
    pv = [rng.randrange(F.p) for _ in range(cur)]
    sv = [rng.randrange(F.p) for _ in range(n // cur)]
    sv[1] = 0
    sv[2] = 1
    d_p, d_s = dev(mont(field, pv)), dev(mont(field, sv))
    for lo, count in ((0, n), (300, 1500), (half, 700), (cur + half - 3, 1000), (n - 513, 513), (n - 1, 1)):
        stride = count + 5
        out = torch.full((2, stride, 4), 3, dtype=torch.int64, device="cuda")
        ctx.check(ctx.lib.trp_dev_ipa_round_scalars(ctx.handle, 0, d_p.data_ptr(), d_s.data_ptr(), cur, lo, count, stride, out.data_ptr()))
        got = host(out)
        want0, want1 = [], []
        for b in range(lo, lo + count):
            t, i = divmod(b, cur)
            if i < half:
                want0.append(pv[half + i] * sv[t] % F.p); want1.append(0)
            else:
                want0.append(0); want1.append(pv[i - half] * sv[t] % F.p)
        assert unmont(field, got[0, :count]) == want0, (lo, count)
        assert unmont(field, got[1, :count]) == want1, (lo, count)
        assert (got[:, count:] == 3).all()
    for m in (1, 257, 700, 2048):
        s_in = [rng.randrange(F.p) for _ in range(m)]
        s_in[0] = 0
        u = rng.randrange(1, F.p)
        d_in = dev(mont(field, s_in))
        out = torch.zeros((2 * m + 1, 4), dtype=torch.int64, device="cuda")
        um = mont(field, [u])[0]
        ctx.check(ctx.lib.trp_dev_ipa_s_double(ctx.handle, 0, d_in.data_ptr(), m, um.ctypes.data, out.data_ptr()))
        got = host(out)
        assert unmont(field, got[:2 * m]) == [e for t in s_in for e in (t, t * u % F.p)], m
        assert not got[2 * m].any()
    assert ctx.lib.trp_dev_ipa_s_double(ctx.handle, 0, d_in.data_ptr(), m, um.ctypes.data, d_in.data_ptr()) == TRP_E_INVALID


# ---- C. point prefix sums across the super-segment level ----------------------------------------------------------------------
CHUNK, SEGMENT = 16, 16 * 256                 # points per thread chunk; points per segment (256 chunks)
SUPER = SEGMENT * 256                         # points per super-segment (256 segments): 2^20


def progression_scalars(curve, seed=21):
    """k0, k1 of make_points(curve, n, seed): point i is (k0 + i k1) G"""
    rng = np.random.Generator(np.random.PCG64(seed))
    q = O.MODULUS[O.SCALAR_FIELD[curve]]
    k0 = int.from_bytes(rng.bytes(32), "little") % q
    k1 = int.from_bytes(rng.bytes(32), "little") % q
    return k0, k1


@pytest.mark.parametrize("n", [SUPER, SUPER + 1, 4 * SUPER])
def test_points_prefix_sum_super_segments(ctxs, n):
    """trp_dev_points_prefix_sum at 2^20 (one full super-segment, the k = 20 base set), 2^20 + 1 (a second super-segment of one
    point) and 2^22 (the k = 22 base set).  Identity inputs, doublings (the running sum equals the next input) and cancellations
    (a prefix that IS the identity) sit at segment and super-segment boundaries.  Every output is checked at once by one random
    linear combination, sum_j c_j Q_j = sum_i (sum_{j >= i} c_j) P_i, with two oracle MSMs; the outputs next to every segment
    boundary are also compared exactly with the closed form of the progression."""
    import torch
    curve = O.VESTA
    ctx = ctxs[curve]
    q = O.MODULUS[O.SCALAR_FIELD[curve]]
    gen = generator(curve)
    pts = make_points(curve, n).copy()
    k0, k1 = progression_scalars(curve)
    assert np.array_equal(pts[0], O.point_mul(curve, limbs([k0])[0], gen))
    ovr = {}                                  # index -> scalar of the replacement input (0 = the identity)

    def prefix_scalar(j):
        s = ((j + 1) * k0 + j * (j + 1) // 2 * k1) % q
        return (s + sum(v - (k0 + i * k1) for i, v in ovr.items() if i <= j)) % q

    def point_of(s):
        return np.zeros(8, dtype=np.uint64) if s % q == 0 else O.point_mul(curve, limbs([s % q])[0], gen)

    def put(i, s):
        if 0 <= i < n:
            ovr[i] = s % q
            pts[i] = point_of(s)

    for b in range(SEGMENT, n, SEGMENT):
        m = b // SEGMENT
        if b % SUPER == 0:
            put(b - 1, 0)                                  # an identity input closes the super-segment
            if (b // SUPER) % 2:
                put(b, -prefix_scalar(b - 1))              # ... the next input cancels the running sum: Q_b is the identity
                put(b + 2, (k0 + (b + 1) * k1))            # P + P inside the chunk after it (Q_{b+1} = P_{b+1})
            else:
                put(b, prefix_scalar(b - 1))               # the first input of the super-segment equals the running sum
        elif m % 97 == 1:
            put(b, prefix_scalar(b - 1))                   # doubling across a segment boundary
        elif m % 97 == 2:
            put(b - 1, 0)                                  # an identity as a segment's last input
        elif m % 97 == 3:
            put(b, -prefix_scalar(b - 1))                  # cancellation at a segment's first input
    d_in = dev(pts)
    d_out = torch.empty_like(d_in)
    ctx.check(ctx.lib.trp_dev_points_prefix_sum(ctx.handle, d_in.data_ptr(), n, d_out.data_ptr()))
    Q = host(d_out).reshape(n, 8).copy()
    # exact values at the ends and next to every segment (and super-segment) boundary
    idx = sorted({0, n - 1} | {j for b in range(SEGMENT, n, SEGMENT) for j in (b - 1, b, b + 1) if j < n} |
                 {j for i in ovr for j in (i - 1, i, i + 1) if 0 <= j < n})
    for j in idx:
        assert np.array_equal(Q[j], point_of(prefix_scalar(j))), j
    if n > SUPER:
        assert not Q[SUPER].any()
    # every output: O.msm(c, Q) == O.msm(suffix sums of c, P); draw the suffix sums S and take c_j = S_j - S_{j+1}
    S = O.random_field_mont(O.FP, n, 900 + n % 7)
    c = S.copy()
    c[:n - 1] = O.field_op(O.FP, "sub", S[:n - 1], S[1:])
    assert np.array_equal(O.msm(curve, c, Q), O.msm(curve, S, pts))
    if n == SUPER + 1:                        # in place gives the same bytes
        ctx.check(ctx.lib.trp_dev_points_prefix_sum(ctx.handle, d_in.data_ptr(), n, d_in.data_ptr()))
        assert np.array_equal(host(d_in).reshape(n, 8), Q)


# ---- D. tile scans of more than 256 tiles ---------------------------------------------------------------------------------------
def running_product(vals, init, p):
    out, run = [], init
    for v in vals:
        out.append(run)
        run = run * v % p
    out.append(run)
    return out


@pytest.mark.parametrize("curve,n_in,n_out", [(O.VESTA, 1 << 20, (1 << 20) - 6), (O.VESTA, 1 << 20, (1 << 20) + 1),
                                              (O.VESTA, (1 << 20) + 2049, (1 << 20) + 2049), (O.PALLAS, (1 << 20) + 2049, (1 << 20) + 2049),
                                              (O.VESTA, (1 << 21) + 3, (1 << 21) + 3)])
def test_grand_product_many_tiles(ctxs, curve, n_in, n_out):
    """trp_dev_grand_product past 256 tiles of 2048 values: 2, 3 and 5 tiles per thread of the tile scan, tile counts that are not
    multiples of 256 (the top threads own no tile), every output against a Python-int running product"""
    import torch
    ctx = ctxs[curve]
    field = O.SCALAR_FIELD[curve]
    p = O.MODULUS[field]
    v = O.random_field_mont(field, n_in, n_in % 1000)
    init = random.Random(n_in).randrange(1, p)
    d_v, d_init = dev(v), dev(mont(field, [init]))
    d_z = torch.zeros((n_out, 4), dtype=torch.int64, device="cuda")
    ctx.check(ctx.lib.trp_dev_grand_product(ctx.handle, 0, d_v.data_ptr(), n_in, d_init.data_ptr(), d_z.data_ptr(), n_out))
    want = running_product(unmont(field, v), init, p)[:n_out]
    assert unmont(field, host(d_z)) == want
    # in place (z aliases v) when n_out == n_in
    if n_out == n_in:
        ctx.check(ctx.lib.trp_dev_grand_product(ctx.handle, 0, d_v.data_ptr(), n_in, d_init.data_ptr(), d_v.data_ptr(), n_out))
        assert unmont(field, host(d_v)) == want


def test_grand_product_rejects_more_outputs_than_inputs_allow(ctxs):
    import torch
    ctx = ctxs[O.VESTA]
    n_in, n_out = (1 << 20) - 6, 1 << 20
    d_v = torch.zeros((n_in, 4), dtype=torch.int64, device="cuda")
    d_z = torch.zeros((n_out, 4), dtype=torch.int64, device="cuda")
    rejects(ctx, lambda: ctx.lib.trp_dev_grand_product(ctx.handle, 0, d_v.data_ptr(), n_in, None, d_z.data_ptr(), n_out))


@pytest.mark.parametrize("curve", [O.VESTA, O.PALLAS])
def test_batch_invert_many_tiles(ctxs, curve):
    import torch
    ctx = ctxs[curve]
    field = O.SCALAR_FIELD[curve]
    n = (1 << 20) + 2049
    a = O.random_field_mont(field, n, 31 + curve)
    rng = np.random.default_rng(5)
    a[rng.integers(0, n, 3000)] = 0                        # scattered zeros
    a[2048 * 300:2048 * 300 + 2048] = 0                    # a whole tile of zeros
    a[n - 2049:n - 2040] = 0                               # zeros in the last, partial tile
    d_a = dev(a)
    d_out = torch.empty_like(d_a)
    ctx.check(ctx.lib.trp_dev_batch_invert(ctx.handle, 0, d_a.data_ptr(), None, d_out.data_ptr(), n))
    assert np.array_equal(host(d_out), O.field_op(field, "inv", a))


@pytest.mark.parametrize("curve", [O.VESTA, O.PALLAS])
def test_kate_division_many_tiles(ctxs, curve):
    """trp_dev_kate_division (the additive, reversed form of the tile scan) at 2^20 + 2049 coefficients, output by output"""
    import torch
    ctx = ctxs[curve]
    field = O.SCALAR_FIELD[curve]
    F = FIELDS[field]
    n = (1 << 20) + 2049
    a = O.random_field_mont(field, n, 41 + curve)
    b = random.Random(curve).randrange(2, F.p)
    d_a = dev(a)
    d_q = torch.zeros((n - 1, 4), dtype=torch.int64, device="cuda")
    bm = mont(field, [b])[0]
    ctx.check(ctx.lib.trp_dev_kate_division(ctx.handle, 0, d_a.data_ptr(), n, bm.ctypes.data, d_q.data_ptr()))
    assert unmont(field, host(d_q)) == pm.kate_division(F, unmont(field, a), b)


# ---- E. trp_dev_linear_combination ---------------------------------------------------------------------------------------------
def lincomb(ctx, field, cols, scal_mont, n, out):
    """trp_dev_linear_combination over separately allocated device columns; returns the C return code"""
    import ctypes
    tab = (ctypes.c_void_p * max(len(cols), 1))(*[c.data_ptr() for c in cols])
    sc = np.ascontiguousarray(scal_mont, dtype=np.uint64).reshape(-1, 4)
    return ctx.lib.trp_dev_linear_combination(ctx.handle, 0, tab, sc.ctypes.data, n, len(cols), out.data_ptr())


def lincomb_oracle(field, cols, scal_mont):
    acc = np.zeros_like(cols[0])
    for c, s in zip(cols, scal_mont):
        acc = O.field_op(field, "add", acc, O.field_op(field, "mul", c, np.repeat(s.reshape(1, 4), len(c), axis=0)))
    return acc


@pytest.mark.parametrize("curve,m,n", [(O.VESTA, m, n) for m in (0, 1, 2, 700) for n in (1, 255, 257, (1 << 16) + 1)] +
                         [(O.PALLAS, 2, 257), (O.PALLAS, 40, 4099), (O.VESTA, 40, 1 << 20)])
def test_linear_combination(ctxs, curve, m, n):
    """sum_j scalars[j] * polys[j] against O.field_op sums, scalars including 0, 1 and p - 1; m = 0 zero-fills the output; and the
    sharded backend's grouping (block-wise partial sums over parallel.block_range, then the G partials with weights 1) gives the
    same bytes for G = 2, 4, 8"""
    import torch
    from tiny_ram_halo2_b200 import parallel as PL
    ctx = ctxs[curve]
    field = O.SCALAR_FIELD[curve]
    p = O.MODULUS[field]
    host_cols = [O.random_field_mont(field, n, 1000 * m + j) for j in range(m)]
    cols = [dev(c) for c in host_cols]                     # separate allocations, not one strided block
    scal = O.random_field_mont(field, max(m, 1), 7 + m)[:m]
    for j, v in enumerate([p - 1, 1, 0][:m]):           # one term alone is never the trivial 0 * poly
        scal[j] = mont(field, [v])[0]
    out = torch.full((n, 4), 5, dtype=torch.int64, device="cuda")
    ctx.check(lincomb(ctx, field, cols, scal, n, out))
    got = host(out).copy()
    if m == 0:
        assert not got.any()
        return
    assert np.array_equal(got, lincomb_oracle(field, host_cols, scal))
    if m < 4:
        return
    one = mont(field, [1])
    for G in (2, 4, 8):
        parts = []
        for r in range(G):
            _, lo, hi = PL.block_range(m, G, r)
            part = torch.full((n, 4), 9, dtype=torch.int64, device="cuda")
            ctx.check(lincomb(ctx, field, cols[lo:hi], scal[lo:hi], n, part))
            parts.append(part)
        total = torch.full((n, 4), 9, dtype=torch.int64, device="cuda")
        ctx.check(lincomb(ctx, field, parts, np.repeat(one, G, axis=0), n, total))
        assert np.array_equal(host(total), got), G


def test_linear_combination_rejects_aliasing(ctxs):
    ctx = ctxs[O.VESTA]
    n = 300
    cols = [dev(O.random_field_mont(O.FP, n, 60 + j)) for j in range(3)]
    before = [host(c).copy() for c in cols]
    scal = O.random_field_mont(O.FP, 3, 61)
    for j in range(3):
        rejects(ctx, lambda: lincomb(ctx, O.FP, cols, scal, n, cols[j]))
    assert all(np.array_equal(host(c), b) for c, b in zip(cols, before))
