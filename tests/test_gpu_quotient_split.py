"""GpuBackend.quotient_parts (the numerator split by constraint degree, each part on the cosets its degree needs, recovered with
trp_dev_cosets_to_coeff_parts) against the whole numerator: one program of the sum of the parts on all j - 1 cosets, every
column expanded with trp_dev_coeff_to_coset, then trp_dev_cosets_to_coeff.  The j - 1 pieces of h must be equal bit for bit."""
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


CASES = [("standard", 4), ("standard-no-lookup", 5), ("standard-wide-lookup", 6), ("tinyram-w8", 6), ("tinyram-w8", 9)]


@pytest.mark.parametrize("name,k", CASES)
def test_split_quotient_equals_the_whole_numerator(pkg, name, k):
    PL, P = pkg.plonk, pkg.poly
    from tiny_ram_halo2_b200 import tinyram as TR, trace as T
    C = pm.Vesta
    if name.startswith("standard"):
        cs, fixed, copies, adv, inst = plonk_circuits.standard(PL, with_lookup=name != "standard-no-lookup", wide_lookup=name.endswith("wide-lookup"))
    else:
        circ, fixed, copies, adv, inst = TR.build(PL, TP.answer_only(T, 8), k)
        cs = circ.cs
    seen = {}

    class Probe(PL.GpuBackend):
        def quotient_parts(self, parts):
            pieces = super().quotient_parts(parts)
            seen["split"] = np.stack([p_.cpu().numpy() for p_ in pieces])
            ast, polys = _whole(PL, P, self, [(q, self._ast_of[id(prog)], leaves) for q, prog, leaves in parts])
            seen["whole"] = _monolithic(PL, P, self, ast, polys)
            seen["ncos"] = [q for q, _, _ in parts]
            return pieces

        def quotient_part_programs(self, pk, build_parts, challenges, n_perm_columns):
            asts = build_parts(*challenges)
            progs = super().quotient_part_programs(pk, build_parts, challenges, n_perm_columns)
            self._ast_of = {id(prog): ast for (_, prog, _), (_, ast, _) in zip(progs, asts)}
            return progs

    ctx = pkg.Context(0, pkg.VESTA)
    be = Probe(ctx, k, cs.degree())
    pk = PL.keygen(be, cs, fixed, copies)
    rnd = random.Random(11)
    for _ in range(2):                       # the second proof takes the cached programs
        seen.clear()
        PL.create_proof(be, pk, inst, adv, lambda: rnd.randrange(C.scalar.p), PL.Blake2bWrite(C.base.p, C.scalar.p))
        assert seen["split"].shape == seen["whole"].shape and np.array_equal(seen["split"], seen["whole"])
        assert len(seen["ncos"]) >= 1 and max(seen["ncos"]) <= cs.degree() - 1


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
