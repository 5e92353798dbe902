"""Oracle for SURVEY.md 8(f) row f4: an independent verify_proof and a pure-Python backend for the host prover.

TEST INFRASTRUCTURE ONLY (see pasta_model.py's header): the product never imports this.

  * verify_proof      restates halo2_proofs 0.2.0 plonk::verify_proof with the IPA strategy (plonk/verifier.rs,
                      plonk/{permutation,lookup,vanishing}/verifier.rs, poly/multiopen/verifier.rs, poly/commitment/verifier.rs;
                      reached from the reference at src/test_utils.rs:56-70,111-118) over Python big ints.  It shares NO code with
                      the prover: its own transcript reader, its own expression evaluation (duck-typed on the node class names of
                      plonk.Expression), its own point-set construction.  A proof it accepts satisfies every identity of the
                      protocol at the challenge points, which pins commitments, quotient, evaluations, multiopen and the IPA
                      TOGETHER (the reference's own tests check exactly this accept/reject bit).
  * PythonBackend     the whole backend interface of tiny-ram-halo2_b200/plonk.py (BACKEND_METHODS) over pasta_model /
                      params_model, so that the tests can run the SAME host protocol logic on the CPU and compare proof bytes
                      with the GPU backend's.  Each batch method is the loop over its single-item operation.
PARITY UNPINNED against a Rust run (no halo2 golden proof exists in /root/reference); see plonk.py's header for the one
known deviation (transcript_repr)."""
from __future__ import annotations

import hashlib

import pasta_model as pm
import params_model as prm


# ---- backend for plonk.create_proof / keygen --------------------------------------------------------------------------------------
class PythonBackend:
    leaves_are_coefficients = False     # the quotient's leaves are evaluations on the extended domain

    def __init__(self, curve: pm.Curve, k: int, cs_degree: int, params=None):
        self.C, self.F = curve, curve.scalar
        self.k, self.n, self.j = k, 1 << k, cs_degree
        self.p, self.q = curve.scalar.p, curve.base.p
        self.params = params if params is not None else prm.params_new(curve, k)
        self.dom = pm.EvaluationDomain(self.F, cs_degree, k)
        self.extended_k = self.dom.extended_k
        self.omega, self.omega_inv, self.delta = self.dom.omega, self.dom.omega_inv, self.F.DELTA

    def rotate_omega(self, x, rotation):
        return self.dom.rotate_omega(x, rotation)

    # -- vectors are plain lists of n canonical ints
    def vec(self, values):
        if len(values) > self.n:
            raise ValueError("column longer than the domain")
        return [v % self.p for v in values] + [0] * (self.n - len(values))

    def set_rows(self, v, start, values):
        v[start:start + len(values)] = [x % self.p for x in values]
        return v

    def set_rows_many(self, vs, start, values):
        for v, vals in zip(vs, values):
            self.set_rows(v, start, vals)

    def random_vec(self, rand): return [rand() for _ in range(self.n)]

    def mul_add(self, acc, s, v):
        return list(v) if acc is None else [(a * s + c) % self.p for a, c in zip(acc, v)]

    def sub_low(self, v, low):
        out = list(v)
        for i, r in enumerate(low):
            out[i] = (out[i] - r) % self.p
        return out

    def sigma_vecs(self, m, moved):
        p, n = self.p, self.n
        om = [1] * n
        for j in range(1, n):
            om[j] = om[j - 1] * self.omega % p
        dl = [pow(self.delta, i, p) for i in range(max(m, 1))]
        out = [[dl[i] * om[j] % p for j in range(n)] for i in range(m)]
        for (i, j), (i2, j2) in moved.items():
            out[i][j] = dl[i2] * om[j2] % p
        return out

    def sigma_swap_blocks(self, sigmas, blocks):
        for i, r, i2, r2, rows in blocks:
            for t in range(rows):
                sigmas[i][r + t] = self.rotate_omega(pow(self.delta, i2, self.p), r2 + t)
                sigmas[i2][r2 + t] = self.rotate_omega(pow(self.delta, i, self.p), r + t)
        return sigmas

    def compress(self, exprs, theta, values_of):
        p, n = self.p, self.n
        out = [0] * n
        for e in exprs:
            for r in range(n):
                out[r] = (out[r] * theta + _eval_expr(e, p, lambda q: values_of[q.kind][q.column][(r + q.rotation) % n])) % p
        return out

    def commit_lagrange(self, values, blind):
        return self.C.best_multiexp(list(values) + [blind], self.params["g_lagrange"] + [self.params["w"]])

    def commit(self, coeffs, blind):
        return self.C.best_multiexp(list(coeffs) + [blind], self.params["g"] + [self.params["w"]])

    def commit_lagrange_many(self, vecs, blinds, sparse=False, runs=False): return [self.commit_lagrange(v, b) for v, b in zip(vecs, blinds)]
    def commit_many(self, vecs, blinds): return [self.commit(v, b) for v, b in zip(vecs, blinds)]

    def lagrange_to_coeff(self, values): return self.dom.lagrange_to_coeff(list(values))
    def lagrange_to_coeff_many(self, vs): return [self.lagrange_to_coeff(v) for v in vs]
    def coeff_to_extended(self, coeffs): return self.dom.coeff_to_extended(list(coeffs))
    def coeff_to_extended_static(self, coeffs): return self.coeff_to_extended(coeffs)

    def begin_proof(self, n_polys): pass
    def end_proof(self): pass
    def _wait(self): pass

    def quotient_pieces(self, pk, challenges, build_h, build_parts, resolve):
        ast, keys = build_h(*challenges)                # the whole folded numerator
        return self.quotient(ast, [resolve(k) for k in keys])

    def quotient(self, ast, ext_polys):
        h = pm.evaluate_ast(self.dom, ast, ext_polys)
        h = self.dom.extended_to_coeff(self.dom.divide_by_vanishing_poly(h))
        return [h[i * self.n:(i + 1) * self.n] for i in range(self.j - 1)]

    def eval_polynomial(self, coeffs, x): return pm.eval_polynomial(self.F, coeffs, x)
    def eval_polynomials_at(self, vs, x): return [self.eval_polynomial(v, x) for v in vs]
    def linear_combination(self, vs, scalars): return [sum(s * c for s, c in zip(scalars, col)) % self.p for col in zip(*vs)]
    def kate_division(self, coeffs, b): return pm.kate_division(self.F, list(coeffs), b) + [0]

    def permutation_commit(self, values, sigmas, beta, gamma, chunk_len, blinding_factors, rand, after_chunk):
        return pm.permutation_commit(self.F, self.omega, self.n, values, sigmas, beta, gamma, chunk_len, blinding_factors, rand, after_chunk)

    def permute_expression_pair(self, inp, tab, usable_rows):
        r = pm.permute_expression_pair(self.F, inp, tab, usable_rows)
        if r is None:
            raise ValueError("ConstraintSystemFailure: lookup input value not present in the table")
        return r[0] + [0] * (self.n - usable_rows), r[1] + [0] * (self.n - usable_rows)

    def lookup_product(self, ci, ct, pi, pt, beta, gamma, blinding_factors, rand):
        return pm.lookup_commit_product(self.F, self.n, ci, ct, pi, pt, beta, gamma, blinding_factors, rand)

    def lookups_commit_permuted(self, lookups, theta, values_of, usable, bf, rand):
        """lookup::Argument::commit_permuted for each lookup in turn: A' and S' get their blinding rows, then their two blinds"""
        out = []
        for inputs, tables in lookups:
            ci, ct = self.compress(inputs, theta, values_of), self.compress(tables, theta, values_of)
            pi, pt = self.permute_expression_pair(ci, ct, usable)
            self.set_rows(pi, usable, [rand() for _ in range(bf + 1)])
            self.set_rows(pt, usable, [rand() for _ in range(bf + 1)])
            out.append({"ci": ci, "ct": ct, "pi": pi, "pt": pt, "pi_blind": rand(), "pt_blind": rand()})
        return out

    def lookup_products(self, lookups, beta, gamma, bf, rand):
        """Permuted::commit_product for each lookup in turn: Z with its blinding rows, then its blind"""
        for L in lookups:
            L["z"] = self.lookup_product(L["ci"], L["ct"], L["pi"], L["pt"], beta, gamma, bf, rand)
            L["z_blind"] = rand()

    def ipa_create_proof(self, rand, transcript, p_poly, p_blind, x_3):
        pm.ipa_create_proof(self.C, self.k, self.params["g"], self.params["w"], self.params["u"], rand, transcript, list(p_poly), p_blind, x_3)

    # -- what the product's own verifier (tiny-ram-halo2_b200/verifier.py) asks of a backend beyond the prover's interface
    def fixed_points(self): return self.params["g"][0], self.params["w"], self.params["u"]

    def ipa_s_vector(self, us, init=1):
        s = [init % self.p]
        for u_j in reversed(us):
            s = s + [v * u_j % self.p for v in s]
        return s

    def msm_points(self, scalars, points): return self.C.best_multiexp(list(scalars), list(points))


# ---- verifier -------------------------------------------------------------------------------------------------------------------------
class VerifyError(Exception):
    pass


class Blake2bRead:
    """transcript.rs Blake2bRead<_, _, Challenge255<_>>"""

    def __init__(self, proof: bytes, curve: pm.Curve):
        self.state = hashlib.blake2b(digest_size=64, person=b"Halo2-Transcript")
        self.buf, self.pos, self.C = bytes(proof), 0, curve

    def _take(self, n):
        if self.pos + n > len(self.buf):
            raise VerifyError("proof too short")
        b = self.buf[self.pos:self.pos + n]
        self.pos += n
        return b

    def common_point(self, P):
        if P is None:
            raise VerifyError("point at infinity in the transcript")
        self.state.update(b"\x01" + P[0].to_bytes(32, "little") + P[1].to_bytes(32, "little"))

    def common_scalar(self, s):
        self.state.update(b"\x02" + s.to_bytes(32, "little"))

    def read_point(self):
        b = self._take(32)
        x = int.from_bytes(b, "little") & ((1 << 255) - 1)
        if x >= self.C.base.p:
            raise VerifyError("non-canonical point encoding")
        if b == bytes(32):
            raise VerifyError("point at infinity in the proof")
        y = self.C.base.sqrt((x * x * x + self.C.B) % self.C.base.p)
        if y is None:
            raise VerifyError("point is not on the curve")
        if (y & 1) != (b[31] >> 7):
            y = self.C.base.p - y
        self.common_point((x, y))
        return (x, y)

    def read_scalar(self):
        s = int.from_bytes(self._take(32), "little")
        if s >= self.C.scalar.p:
            raise VerifyError("non-canonical scalar encoding")
        self.common_scalar(s)
        return s

    def squeeze_challenge_scalar(self):
        self.state.update(b"\x00")
        return int.from_bytes(self.state.copy().digest(), "little") % self.C.scalar.p


def _eval_expr(e, p, query):
    kind = type(e).__name__
    if kind == "Constant": return e.value % p
    if kind == "Query": return query(e)
    if kind == "Negated": return -_eval_expr(e.a, p, query) % p
    if kind == "Sum": return (_eval_expr(e.a, p, query) + _eval_expr(e.b, p, query)) % p
    if kind == "Product": return _eval_expr(e.a, p, query) * _eval_expr(e.b, p, query) % p
    if kind == "Scaled": return _eval_expr(e.a, p, query) * e.scalar % p
    raise TypeError(kind)


def _interpolate_eval(points, evals, x, p):
    """value at x of the polynomial of degree < len(points) through (points, evals)"""
    acc = 0
    for j, (xj, yj) in enumerate(zip(points, evals)):
        num, den = 1, 1
        for i, xi in enumerate(points):
            if i != j:
                num = num * (x - xi) % p
                den = den * (xj - xi) % p
        acc = (acc + yj * num % p * pow(den, -1, p)) % p
    return acc


def verify_proof(curve: pm.Curve, params: dict, vk, instances, proof: bytes) -> bool:
    """plonk::verify_proof for one proof.  params: params_model.params_new(curve, k); vk: an object with k, cs, cs_degree,
    fixed_commitments, permutation_commitments, transcript_repr (plonk.VerifyingKey).  True iff the proof is accepted."""
    try:
        _verify(curve, params, vk, instances, proof)
        return True
    except VerifyError as e:
        verify_proof.last_error = str(e)
        return False


verify_proof.last_error = None


def _verify(C, params, vk, instances, proof):
    F = C.scalar
    p, k, cs = F.p, vk.k, vk.cs
    n = 1 << k
    dom = pm.EvaluationDomain(F, vk.cs_degree, k)
    bf = max(3, max(list(cs.num_advice_queries) + [1])) + 2
    usable = n - (bf + 1)
    chunk_len = vk.cs_degree - 2
    t = Blake2bRead(proof, C)
    t.common_scalar(vk.transcript_repr)
    if len(instances) != cs.num_instance:
        raise VerifyError("InvalidInstances")
    inst_commitments = []
    for col in instances:
        if len(col) > usable:
            raise VerifyError("InstanceTooLarge")
        vals = [v % p for v in col] + [0] * (n - len(col))
        cm = C.best_multiexp(vals + [1], params["g_lagrange"] + [params["w"]])
        t.common_point(cm)
        inst_commitments.append(cm)
    adv_commitments = [t.read_point() for _ in range(cs.num_advice)]
    theta = t.squeeze_challenge_scalar()
    lk_permuted = [(t.read_point(), t.read_point()) for _ in cs.lookups]
    beta = t.squeeze_challenge_scalar()
    gamma = t.squeeze_challenge_scalar()
    n_sets = (len(cs.permutation) + chunk_len - 1) // chunk_len
    perm_commitments = [t.read_point() for _ in range(n_sets)]
    lk_products = [t.read_point() for _ in cs.lookups]
    random_commitment = t.read_point()
    y = t.squeeze_challenge_scalar()
    h_commitments = [t.read_point() for _ in range(vk.cs_degree - 1)]
    x = t.squeeze_challenge_scalar()
    q_i, q_a, q_f = cs.queries["instance"], cs.queries["advice"], cs.queries["fixed"]
    inst_evals = [t.read_scalar() for _ in q_i]
    adv_evals = [t.read_scalar() for _ in q_a]
    fix_evals = [t.read_scalar() for _ in q_f]
    random_eval = t.read_scalar()
    sigma_evals = [t.read_scalar() for _ in cs.permutation]
    perm_evals = []
    for i in range(n_sets):
        e, ne = t.read_scalar(), t.read_scalar()
        perm_evals.append((e, ne, t.read_scalar() if i + 1 < n_sets else None))
    lk_evals = [tuple(t.read_scalar() for _ in range(5)) for _ in cs.lookups]     # z, z_next, a, a_inv, s

    # ---- the vanishing identity at x ---------------------------------------------------------------------------------------------------
    xn = pow(x, n, p)
    if xn == 1:
        raise VerifyError("x lies in the domain")
    def l_i(rotation):            # Lagrange basis polynomial of row `rotation mod n`, at x
        w = dom.rotate_omega(1, rotation)
        return (xn - 1) * pow(n, -1, p) % p * w % p * pow((x - w) % p, -1, p) % p
    l_last = l_i(-(bf + 1))
    l_blind = sum(l_i(-r) for r in range(1, bf + 1)) % p
    l_0 = l_i(0)
    evals_of = {"instance": (q_i, inst_evals), "advice": (q_a, adv_evals), "fixed": (q_f, fix_evals)}

    def query(e):
        qs, ev = evals_of[e.kind]
        return ev[qs.index((e.column, e.rotation))]

    terms = [_eval_expr(g, p, query) for g in cs.gates]
    active = (1 - (l_last + l_blind)) % p
    if n_sets:
        terms.append(l_0 * (1 - perm_evals[0][0]) % p)
        zl = perm_evals[-1][0]
        terms.append(l_last * (zl * zl - zl) % p)
        for i in range(1, n_sets):
            terms.append(l_0 * (perm_evals[i][0] - perm_evals[i - 1][2]) % p)
        for i in range(n_sets):
            cols = cs.permutation[i * chunk_len:(i + 1) * chunk_len]
            left, right = perm_evals[i][1], perm_evals[i][0]
            cur_delta = beta * x % p * pow(F.DELTA, i * chunk_len, p) % p
            for off, (kind, c) in enumerate(cols):
                qs, ev = evals_of[kind]
                v = ev[qs.index((c, 0))]
                left = left * ((v + beta * sigma_evals[i * chunk_len + off] + gamma) % p) % p
                right = right * ((v + cur_delta + gamma) % p) % p
                cur_delta = cur_delta * F.DELTA % p
            terms.append((left - right) * active % p)
    for (inputs, tables), (z, z_next, a, a_inv, s) in zip(cs.lookups, lk_evals):
        comp = lambda es: __import__("functools").reduce(lambda acc, e: (acc * theta + _eval_expr(e, p, query)) % p, es, 0)
        terms.append(l_0 * (1 - z) % p)
        terms.append(l_last * (z * z - z) % p)
        terms.append((z_next * (a + beta) % p * (s + gamma) - z * (comp(inputs) + beta) % p * (comp(tables) + gamma)) % p * active % p)
        terms.append(l_0 * (a - s) % p)
        terms.append((a - s) * (a - a_inv) % p * active % p)
    expected_h = 0
    for v in terms:
        expected_h = (expected_h * y + v) % p
    expected_h = expected_h * pow(xn - 1, -1, p) % p
    h_commitment = None
    for cm in reversed(h_commitments):
        h_commitment = C.add(C.mul(xn, h_commitment), cm)

    # ---- queries, in the prover's order ------------------------------------------------------------------------------------------------------
    rot = dom.rotate_omega
    x_next, x_inv, x_last = rot(x, 1), rot(x, -1), rot(x, -(bf + 1))
    Q = []      # (commitment key, commitment point, point, eval)
    for (c, r), e in zip(q_i, inst_evals): Q.append((("i", c), inst_commitments[c], rot(x, r), e))
    for (c, r), e in zip(q_a, adv_evals): Q.append((("a", c), adv_commitments[c], rot(x, r), e))
    for i in range(n_sets):
        Q.append((("pz", i), perm_commitments[i], x, perm_evals[i][0]))
        Q.append((("pz", i), perm_commitments[i], x_next, perm_evals[i][1]))
    for i in reversed(range(n_sets - 1)):
        Q.append((("pz", i), perm_commitments[i], x_last, perm_evals[i][2]))
    for li, ((ca, cs_), cz, (z, z_next, a, a_inv, s)) in enumerate(zip(lk_permuted, lk_products, lk_evals)):
        Q.append((("lz", li), cz, x, z))
        Q.append((("la", li), ca, x, a))
        Q.append((("ls", li), cs_, x, s))
        Q.append((("la", li), ca, x_inv, a_inv))
        Q.append((("lz", li), cz, x_next, z_next))
    for (c, r), e in zip(q_f, fix_evals): Q.append((("f", c), vk.fixed_commitments[c], rot(x, r), e))
    for i, e in enumerate(sigma_evals): Q.append((("sg", i), vk.permutation_commitments[i], x, e))
    Q.append((("h",), h_commitment, x, expected_h))
    Q.append((("rnd",), random_commitment, x, random_eval))

    # ---- multiopen ---------------------------------------------------------------------------------------------------------------------------
    x_1 = t.squeeze_challenge_scalar()
    x_2 = t.squeeze_challenge_scalar()
    pidx = {}
    for _, _, pt, _ in Q:
        pidx.setdefault(pt, len(pidx))
    order, per = [], {}
    for key, cm, pt, e in Q:
        if key not in per:
            per[key] = {"cm": cm, "pts": {}}
            order.append(key)
        per[key]["pts"][pidx[pt]] = e
    set_of = {}
    for key in order:
        set_of.setdefault(tuple(sorted(per[key]["pts"])), len(set_of))
    inv_pidx = {v: kx for kx, v in pidx.items()}
    point_sets = [None] * len(set_of)
    for ps, si in set_of.items():
        point_sets[si] = [inv_pidx[i] for i in ps]
    q_commitments = [None] * len(set_of)
    q_eval_sets = [[0] * len(ps) for ps in point_sets]
    for key in order:
        ps = tuple(sorted(per[key]["pts"]))
        si = set_of[ps]
        q_commitments[si] = C.add(C.mul(x_1, q_commitments[si]), per[key]["cm"])
        q_eval_sets[si] = [(acc * x_1 + per[key]["pts"][i]) % p for acc, i in zip(q_eval_sets[si], ps)]
    q_prime_commitment = t.read_point()
    x_3 = t.squeeze_challenge_scalar()
    u = [t.read_scalar() for _ in point_sets]
    x_4 = t.squeeze_challenge_scalar()
    msm_eval = 0
    for points, evals, proof_eval in zip(point_sets, q_eval_sets, u):
        ev = (proof_eval - _interpolate_eval(points, evals, x_3, p)) % p
        for pt in points:
            if (x_3 - pt) % p == 0:
                raise VerifyError("x_3 hits an opening point")
            ev = ev * pow((x_3 - pt) % p, -1, p) % p
        msm_eval = (msm_eval * x_2 + ev) % p
    P_commit, v = q_prime_commitment, msm_eval
    for cm, ui in zip(q_commitments, u):
        P_commit = C.add(C.mul(x_4, P_commit), cm)
        v = (v * x_4 + ui) % p

    # ---- inner product argument: poly/commitment/verifier.rs --------------------------------------------------------------------------------------
    g, w, U = params["g"], params["w"], params["u"]
    s_commitment = t.read_point()
    xi = t.squeeze_challenge_scalar()
    z = t.squeeze_challenge_scalar()
    lhs = C.add(C.add(P_commit, C.neg(C.mul(v, g[0]))), C.mul(xi, s_commitment))
    us = []
    for _ in range(k):
        l, r = t.read_point(), t.read_point()
        u_j = t.squeeze_challenge_scalar()
        if u_j == 0:
            raise VerifyError("zero challenge")
        lhs = C.add(lhs, C.add(C.mul(F.inv(u_j), l), C.mul(u_j, r)))
        us.append(u_j)
    c, f = t.read_scalar(), t.read_scalar()
    # b = prod_j (1 + u_j x_3^(2^(k-1-j))); G'_0 = <s, G> with s_i = prod_j u_j^(bit (k-1-j) of i)
    b, s = 1, [1]
    for j, u_j in enumerate(us):
        b = b * (1 + u_j * pow(x_3, 1 << (k - 1 - j), p)) % p
    for u_j in reversed(us):
        s = s + [v_ * u_j % p for v_ in s]
    g0 = C.best_multiexp(s, g)
    rhs = C.add(C.add(C.mul(c, g0), C.mul(c * b % p * z % p, U)), C.mul(f, w))
    if lhs != rhs:
        raise VerifyError("the opening proof does not verify")
    if t.pos != len(t.buf):
        raise VerifyError("trailing bytes in the proof")
