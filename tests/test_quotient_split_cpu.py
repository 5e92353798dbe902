"""The quotient numerator split by constraint degree (plonk.split_by_degree): for TinyRamCircuit<32, 8> the parts must add up to
the folded numerator create_proof commits to, and evaluating each part only on the cosets its degree needs must spare exactly
144 of the coset NTTs the whole numerator takes: 141 of advice columns, 3 of one lookup's columns (DESIGN.md section 9)."""
import collections
import random

import pytest


@pytest.fixture(scope="module")
def mods():
    import __graft_entry__ as ge
    ge.load_package()
    from tiny_ram_halo2_b200 import plonk, poly, tinyram
    return plonk, poly, tinyram


def _split(PL, cs, p, delta, seed):
    rnd = random.Random(seed)
    theta, beta, gamma, y = (rnd.randrange(p) for _ in range(4))
    exprs, keys = PL.quotient_constraints(cs, cs.degree(), p, delta, theta, beta, gamma)
    return exprs, keys, y, PL.split_by_degree(exprs, keys, y, cs.degree(), p)


def test_parts_sum_to_the_folded_numerator(mods):
    """sum_d N_d(x) == N(x) at a random point, every leaf a random polynomial of n = 64 coefficients (the oracle evaluates);
    every part's degree bound is at most ncos + 1, and a part references only its own leaves"""
    import pasta_model as pm
    import plonk_model as VM
    PL, P, TR = mods
    cs = TR.TinyRamCircuit(PL, 32).cs
    be = VM.PythonBackend(pm.Vesta, 6, cs.degree())
    p = be.p
    exprs, keys, y, parts = _split(PL, cs, p, be.delta, 3)
    h = P.ConstantTerm(0)
    for e in exprs:
        h = h * y + e
    rnd = random.Random(4)
    poly_of = {k: [rnd.randrange(p) for _ in range(be.n)] for k in keys}
    x = rnd.randrange(p)
    want = PL.eval_ast_at_point(be, h, [poly_of[k] for k in keys], x)
    got = 0
    for ncos, ast, pkeys in parts:
        assert PL.ast_degree(ast) <= ncos + 1 and len(set(pkeys)) == len(pkeys)
        got += PL.eval_ast_at_point(be, ast, [poly_of[k] for k in pkeys], x)
    assert got % p == want
    assert [ncos for ncos, _, _ in parts] == [1, 2, 3, 4, 5]
    assert sorted({k for _, _, pkeys in parts for k in pkeys}, key=keys.index) == keys


def test_coset_transforms_spared(mods):
    """per-proof columns (advice, instance, lookup and permutation products; key material has its cosets precomputed) are expanded
    only on the cosets of the parts that read them: 94 advice columns are read by nothing above degree 5, 16 by nothing above 4
    and 5 by nothing above 3 (141 NTTs), and the Z, A', S' columns of the one degree-5 lookup by nothing above 5 (3 NTTs)"""
    PL, P, TR = mods
    cs = TR.TinyRamCircuit(PL, 32).cs
    p = P._MODULUS[0]
    exprs, keys, y, parts = _split(PL, cs, p, pow(5, 1 << 32, p), 5)
    static = lambda k: isinstance(k, str) or k[0] in (PL.FIXED, "sigma")
    last = {}
    for ncos, _, pkeys in parts:
        for k in pkeys:
            if not static(k):
                last[k] = max(last.get(k, 0), ncos)
    spared = collections.Counter()
    for k, q in last.items():
        spared[k[0]] += cs.degree() - 1 - q
    assert +spared == collections.Counter({PL.ADVICE: 94 + 2 * 16 + 3 * 5, "lookup_z": 1, "lookup_a": 1, "lookup_s": 1})
