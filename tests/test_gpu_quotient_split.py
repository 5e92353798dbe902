"""GpuBackend.quotient_parts (the numerator split by constraint degree, each part on the cosets its degree needs, recovered with
trp_dev_cosets_to_coeff_parts) against the whole numerator: one program of the sum of the parts on all j - 1 cosets, every
column expanded with trp_dev_coeff_to_coset, then trp_dev_cosets_to_coeff.  The j - 1 pieces of h must be equal bit for bit.

Both GPU paths could share a bug (a wrong degree bound in split_by_degree, a wrong program constant, a wrong leaf), so the probe
also checks the quotient identity h(x) (x^n - 1) = sum_p N_p(x) at a random x with no GPU code at all: every leaf's coefficients
are downloaded and evaluated by the oracle, every part's Ast is walked on the host."""
import random

import numpy as np
import pytest

from util import O, pm

import plonk_circuits
import tinyram_programs as TP

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def pkg():
    import __graft_entry__ as ge
    return ge.load_package()


def _whole(PL, P, be, parts):
    """the sum of the parts as ONE Ast over the union of their leaves, and those leaves' polynomials"""
    index, polys, total = {}, [], None
    for _, prog_ast, leaves in parts:
        ast, mine = prog_ast, leaves
        memo = {}

        def remap(a):
            r = memo.get(id(a))
            if r is None:
                if isinstance(a, P.Poly):
                    c = mine[a.index]
                    if id(c) not in index:
                        index[id(c)] = len(polys); polys.append(c)
                    r = P.Poly(index[id(c)], a.rotation)
                elif isinstance(a, (P.Add, P.Mul)): r = type(a)(remap(a.a), remap(a.b))
                elif isinstance(a, P.Scale): r = P.Scale(remap(a.a), a.scalar)
                elif isinstance(a, P.DistributePowers): r = P.DistributePowers([remap(t) for t in a.terms], remap(a.base))
                else: r = a
                memo[id(a)] = r
            return r
        part = remap(ast)
        total = part if total is None else total + part
    return total, polys


def _monolithic(PL, P, be, ast, polys):
    from tiny_ram_halo2_b200._lib import Q_CONTIGUOUS
    t, n, ncos = be.torch, be.n, be.j - 1
    prog = P.compile_ast(ast, be.p)
    vals = t.empty((ncos, n, 4), dtype=t.int64, device="cuda")
    tmp = t.empty((len(polys), n, 4), dtype=t.int64, device="cuda")
    for cs in range(ncos):
        ptrs = []
        for i, c in enumerate(polys):
            if id(c) in be._static:
                ptrs.append(be._static[id(c)][cs].data_ptr())
            else:
                be.ctx.check(be.lib.trp_dev_coeff_to_coset(be.dom.handle, c.data_ptr(), tmp[i].data_ptr(), 1, cs))
                ptrs.append(tmp[i].data_ptr())
        be.ev.evaluate_device(prog, be.dom, ptrs, vals[cs].data_ptr(), coset=cs | Q_CONTIGUOUS)
    h = t.empty((ncos, n, 4), dtype=t.int64, device="cuda")
    be.ctx.check(be.lib.trp_dev_cosets_to_coeff(be.dom.handle, vals.data_ptr(), ncos, h.data_ptr(), 1))
    return h.cpu().numpy()


def _host_eval(P, ast, leaf, x, p):
    """the value at x of an Ast whose Poly leaves are given by leaf(index, rotation), with halo2's node semantics
    (LinearTerm(s) = s X, DistributePowers = fold(0, |acc, t| acc * base + t)); shared subtrees are evaluated once"""
    memo = {}

    def ev(a):
        r = memo.get(id(a))
        if r is None:
            if isinstance(a, P.Poly): r = leaf(a.index, a.rotation)
            elif isinstance(a, P.Add): r = (ev(a.a) + ev(a.b)) % p
            elif isinstance(a, P.Mul): r = ev(a.a) * ev(a.b) % p
            elif isinstance(a, P.Scale): r = ev(a.a) * a.scalar % p
            elif isinstance(a, P.LinearTerm): r = a.scalar * x % p
            elif isinstance(a, P.ConstantTerm): r = a.scalar % p
            elif isinstance(a, P.DistributePowers):
                base, r = ev(a.base), 0
                for t in a.terms:
                    r = (r * base + ev(t)) % p
            else: raise TypeError(type(a))
            memo[id(a)] = r
        return r

    import sys
    old = sys.getrecursionlimit(); sys.setrecursionlimit(max(old, 100000))
    try:
        return ev(ast)
    finally:
        sys.setrecursionlimit(old)


def quotient_identity(P, be, parts, pieces, x):
    """(h(x) (x^n - 1), sum_p N_p(x)) for parts [(ncos, Ast, leaf polynomials in coefficient form)] and the pieces of h, every
    value computed on the host: each leaf is downloaded once and evaluated by the oracle at omega^rot x for the rotations the
    Asts read it at"""
    assert be.leaves_are_coefficients
    p, n = be.p, be.n
    field = O.FP if p == O.MODULUS[O.FP] else O.FQ
    omega = O.limbs_to_ints(O.from_mont(field, O.domain_info(field, be.j, be.k)[1]))[0]
    at = lambda pt: O.limbs_to_ints(O.from_mont(field, pt))[0]
    mont = lambda v: O.to_mont(field, O.ints_to_limbs([v % p]))[0]

    def host_eval(col, pt):
        return at(O.eval_polynomial(field, col.cpu().numpy().view(np.uint64).reshape(-1, 4), mont(pt)))

    rots = {}                                # id(leaf) -> (leaf, rotations read)
    for _, ast, polys in parts:
        memo, stack = set(), [ast]
        while stack:
            a = stack.pop()
            if id(a) in memo:
                continue
            memo.add(id(a))
            if isinstance(a, P.Poly):
                rots.setdefault(id(polys[a.index]), (polys[a.index], set()))[1].add(a.rotation)
            elif isinstance(a, (P.Add, P.Mul)): stack += [a.a, a.b]
            elif isinstance(a, P.Scale): stack.append(a.a)
            elif isinstance(a, P.DistributePowers): stack += list(a.terms) + [a.base]
    value = {}
    for key, (col, rs) in rots.items():
        host = np.ascontiguousarray(col.cpu().numpy().view(np.uint64))
        assert host.shape == (n, 4)
        for r in rs:
            pt = x * pow(omega if r >= 0 else pow(omega, -1, p), abs(r), p) % p
            value[(key, r)] = at(O.eval_polynomial(field, host, mont(pt)))
    rhs = 0
    for _, ast, polys in parts:
        rhs += _host_eval(P, ast, lambda i, r, polys=polys: value[(id(polys[i]), r)], x, p)
    hx, xn = 0, pow(x, n, p)
    for piece in reversed(pieces):
        hx = (hx * xn + host_eval(piece, x)) % p
    return hx * (xn - 1) % p, rhs % p


def split_probe(PL, seen, monolithic=True, x_seed=5):
    """a GpuBackend whose quotient_parts records the split pieces, the whole-numerator pieces (monolithic=True) and both sides
    of the host-side quotient identity at a random x"""
    P = PL.P
    rx = random.Random(x_seed)

    class Probe(PL.GpuBackend):
        def quotient_parts(self, parts):
            pieces = super().quotient_parts(parts)
            with_ast = [(q, self._ast_of[id(prog)], leaves) for q, prog, leaves in parts]
            seen["split"] = np.stack([p_.cpu().numpy() for p_ in pieces])
            if monolithic:
                ast, polys = _whole(PL, P, self, with_ast)
                seen["whole"] = _monolithic(PL, P, self, ast, polys)
            seen["ncos"] = [q for q, _, _ in parts]
            seen["identity"] = quotient_identity(P, self, with_ast, pieces, rx.randrange(1, self.p))
            return pieces

        def quotient_part_programs(self, pk, build_parts, challenges, n_perm_columns):
            asts = build_parts(*challenges)
            progs = super().quotient_part_programs(pk, build_parts, challenges, n_perm_columns)
            self._ast_of = {id(prog): ast for (_, prog, _), (_, ast, _) in zip(progs, asts)}
            return progs

    return Probe


CASES = [("standard", 4, "vesta"), ("standard-no-lookup", 5, "vesta"), ("standard-wide-lookup", 6, "vesta"),
         ("standard", 4, "pallas"), ("standard-no-lookup", 5, "pallas"), ("standard-wide-lookup", 6, "pallas"),
         ("tinyram-w8", 6, "vesta"), ("tinyram-w8", 9, "vesta"),
         ("tinyram-w8", 11, "vesta"), ("tinyram-w16", 12, "vesta")]      # k >= 11: the coset NTTs take more than one pass


@pytest.mark.parametrize("name,k,curve", CASES, ids=[f"{n}-{k}" + ("" if c == "vesta" else f"-{c}") for n, k, c in CASES])
def test_split_quotient_equals_the_whole_numerator(pkg, name, k, curve):
    PL, P = pkg.plonk, pkg.poly
    from tiny_ram_halo2_b200 import tinyram as TR, trace as T
    C = {"vesta": pm.Vesta, "pallas": pm.Pallas}[curve]
    if name.startswith("standard"):
        cs, fixed, copies, adv, inst = plonk_circuits.standard(PL, with_lookup=name != "standard-no-lookup", wide_lookup=name.endswith("wide-lookup"))
    else:
        circ, fixed, copies, adv, inst = TR.build(PL, TP.answer_only(T, int(name[len("tinyram-w"):])), k)
        cs = circ.cs
    seen = {}
    ctx = pkg.Context(0, {"vesta": pkg.VESTA, "pallas": pkg.PALLAS}[curve])
    be = split_probe(PL, seen)(ctx, k, cs.degree())
    pk = PL.keygen(be, cs, fixed, copies)
    rnd = random.Random(11)
    for _ in range(2):                       # the second proof takes the cached programs
        seen.clear()
        PL.create_proof(be, pk, inst, adv, lambda: rnd.randrange(C.scalar.p), PL.Blake2bWrite(C.base.p, C.scalar.p))
        assert seen["split"].shape == seen["whole"].shape and np.array_equal(seen["split"], seen["whole"])
        assert len(seen["ncos"]) >= 1 and max(seen["ncos"]) <= cs.degree() - 1
        lhs, rhs = seen["identity"]
        assert lhs == rhs, "h(x) (x^n - 1) != sum_p N_p(x)"
    be.close()


def test_parts_entry_point_rejects_bad_shapes(pkg):
    import torch
    ctx = pkg.Context(0, pkg.VESTA)
    dom = pkg.EvaluationDomain(ctx, 6, 4)
    d = torch.zeros((8, 16, 4), dtype=torch.int64, device="cuda")
    import ctypes
    qs = lambda *v: (ctypes.c_uint * len(v))(*v)
    assert ctx.lib.trp_dev_cosets_to_coeff_parts(dom.handle, d.data_ptr(), qs(1, 2), 2, 5, d[3].data_ptr(), 1) == 0
    assert ctx.lib.trp_dev_cosets_to_coeff_parts(dom.handle, d.data_ptr(), qs(1, 6), 2, 5, d[3].data_ptr(), 1) == -1    # part above ncos_out
    assert ctx.lib.trp_dev_cosets_to_coeff_parts(dom.handle, d.data_ptr(), qs(0), 1, 5, d[3].data_ptr(), 1) == -1       # empty part
    assert ctx.lib.trp_dev_cosets_to_coeff_parts(dom.handle, d.data_ptr(), qs(1), 1, 9, d[3].data_ptr(), 1) == -1       # > 8 cosets
    assert ctx.lib.trp_dev_cosets_to_coeff_parts(dom.handle, d.data_ptr(), qs(1), 0, 5, d[3].data_ptr(), 1) == -1       # no part
