"""CPU tests of the row-f4 host logic (tiny-ram-halo2_b200/plonk.py: ConstraintSystem, keygen, create_proof, the Blake2b
transcript) run over the oracle's PythonBackend, against the independent verifier oracle/plonk_model.verify_proof."""
import random

import pytest

from util import pm

import params_model as prm
import plonk_model as VM
import plonk_circuits


@pytest.fixture(scope="module")
def PL():
    import __graft_entry__ as ge
    ge.load_package()
    from tiny_ram_halo2_b200 import plonk
    return plonk


def _prove(PL, C, k, seed=1, mutate=None, **kw):
    cs, fixed, copies, adv, inst = plonk_circuits.standard(PL, **kw)
    if mutate:
        mutate(adv, inst, fixed)
    be = VM.PythonBackend(C, k, cs.degree())
    pk = PL.keygen(be, cs, fixed, copies)
    rnd = random.Random(seed)
    tr = PL.Blake2bWrite(C.base.p, C.scalar.p)
    proof = PL.create_proof(be, pk, inst, adv, lambda: rnd.randrange(C.scalar.p), tr)
    return be, pk, inst, proof


@pytest.mark.parametrize("C", [pm.Vesta, pm.Pallas], ids=["vesta", "pallas"])
@pytest.mark.parametrize("kw", [dict(with_lookup=True), dict(with_lookup=False), dict(with_lookup=True, wide_lookup=True)],
                         ids=["lookup", "no-lookup", "wide-lookup"])
def test_proof_verifies(PL, C, kw):
    be, pk, inst, proof = _prove(PL, C, 4, **kw)
    assert VM.verify_proof(C, be.params, pk.vk, inst, proof)
    # soundness smoke: wrong public input, flipped bytes, truncated proof are all rejected
    assert not VM.verify_proof(C, be.params, pk.vk, [[inst[0][0] + 1]], proof)
    for pos in (0, 40, len(proof) // 2, len(proof) - 1):
        bad = bytearray(proof); bad[pos] ^= 1
        assert not VM.verify_proof(C, be.params, pk.vk, inst, bytes(bad))
    assert not VM.verify_proof(C, be.params, pk.vk, inst, proof[:-32])
    assert not VM.verify_proof(C, be.params, pk.vk, inst, proof + bytes(32))


def test_unsatisfied_circuits_do_not_verify(PL):
    C = pm.Vesta
    def break_gate(adv, inst, fixed): adv[2][0] += 1                 # a + b != c on row 0 (also breaks the copy c[0] = a[1])
    be, pk, inst, proof = _prove(PL, C, 4, mutate=break_gate)
    assert not VM.verify_proof(C, be.params, pk.vk, inst, proof)
    def break_copy(adv, inst, fixed): inst[0][0] += 1                # public input differs from the copied cell
    be, pk, inst, proof = _prove(PL, C, 4, mutate=break_copy)
    assert not VM.verify_proof(C, be.params, pk.vk, inst, proof)
    def break_lookup(adv, inst, fixed): adv[0][3] = 9; adv[1][3] = 9      # a = 9 is not in the table 0..7 (copy a[3] = b[3] kept)
    with pytest.raises(ValueError):
        _prove(PL, C, 4, mutate=break_lookup)


def test_proof_layout_and_determinism(PL):
    C = pm.Vesta
    be, pk, inst, p1 = _prove(PL, C, 4, seed=7)
    _, _, _, p2 = _prove(PL, C, 4, seed=7)
    _, _, _, p3 = _prove(PL, C, 4, seed=8)
    assert p1 == p2 and p1 != p3
    # the bytes themselves are frozen (tests/golden/proof_digests.json): with a fixed-seed blinding RNG the serialized proof must not
    # move when the host logic is reworked; the GPU tests hold the device proofs against this backend's bytes
    import hashlib, json, os
    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "proof_digests.json")) as f:
        want = json.load(f)["standard_k4_seed7_vesta"]
    assert (len(p1), hashlib.sha256(p1).hexdigest(), hex(pk.vk.transcript_repr)) == (want["bytes"], want["sha256"], want["transcript_repr"])
    cs = pk.vk.cs
    n_sets = 2
    points = cs.num_advice + 2 * len(cs.lookups) + n_sets + len(cs.lookups) + 1 + (pk.vk.cs_degree - 1) + 1 + 1 + 2 * be.k
    n_q = sum(len(v) for v in cs.queries.values())
    scalars = n_q + 1 + len(cs.permutation) + (3 * n_sets - 1) + 5 * len(cs.lookups) + 2
    assert (len(p1) - 32 * (points + scalars)) % 32 == 0
    n_point_sets = (len(p1) - 32 * (points + scalars)) // 32
    assert 1 <= n_point_sets <= 5
    assert cs.degree() == 5 and cs.blinding_factors() == 5


def test_multiopen_point_sets(PL):
    """construct_intermediate_sets on the pattern create_proof produces: sets are keyed by the SET of points of a commitment"""
    qs = [("a", 10), ("a", 11), ("b", 10), ("c", 11), ("c", 10), ("d", 12), ("d", 10)]
    cmap, point_sets = PL.construct_intermediate_sets(qs, lambda q: q[0], lambda q: q[1], lambda q: (q[0], q[1]))
    assert [cd["set_index"] for cd in cmap] == [0, 1, 0, 2]
    assert point_sets == [[10, 11], [10], [10, 12]]
    assert cmap[2]["evals"] == [("c", 10), ("c", 11)]
    F = pm.Fp
    pts, ev = [3, 5, 11], [7, 1, 20]
    coeffs = PL.lagrange_interpolate(pts, ev, F.p)
    assert [pm.eval_polynomial(F, coeffs, x) for x in pts] == ev


def test_keygen_permutation_cycles(PL):
    cs, fixed, copies, adv, inst = plonk_circuits.standard(PL)
    F = pm.Fp
    n = 16
    omega = F.root_of_unity(4)
    sig = PL.build_sigmas(cs, n, F.p, omega, F.DELTA, copies)
    ident = [[pow(F.DELTA, i, F.p) * pow(omega, j, F.p) % F.p for j in range(n)] for i in range(len(cs.permutation))]
    # sigma is a permutation of the identity labels that fixes every cell outside the copy constraints
    assert sorted(v for col in sig for v in col) == sorted(v for col in ident for v in col)
    moved = {(i, j) for i in range(len(sig)) for j in range(n) if sig[i][j] != ident[i][j]}
    col_of = {kc: i for i, kc in enumerate(cs.permutation)}
    touched = {(col_of[(k_, c)], r) for pair in copies for (k_, c, r) in pair}
    assert moved == touched


def test_permutation_mapping_is_sparse_and_cyclic(PL):
    """chains and repeated copies merge into one cycle; untouched cells never enter the mapping (keygen is O(copies))"""
    cs = PL.ConstraintSystem()
    a, b = cs.advice_column(), cs.advice_column()
    cs.enable_equality(PL.ADVICE, a); cs.enable_equality(PL.ADVICE, b)
    A = PL.ADVICE
    copies = [((A, a, 0), (A, b, 5)), ((A, b, 5), (A, a, 9)), ((A, a, 9), (A, a, 0)), ((A, b, 1), (A, b, 2)), ((A, a, 3), (A, a, 3))]
    m = PL.permutation_mapping(cs, 1 << 20, copies)
    assert set(m) == {(0, 0), (1, 5), (0, 9), (1, 1), (1, 2)}
    # following the mapping from any cell of the 3-cycle visits all three cells and returns
    cell, seen = (0, 0), []
    for _ in range(3):
        seen.append(cell); cell = m[cell]
    assert cell == (0, 0) and set(seen) == {(0, 0), (1, 5), (0, 9)}
    assert m[(1, 1)] == (1, 2) and m[(1, 2)] == (1, 1)
    with pytest.raises(ValueError):
        PL.permutation_mapping(cs, 16, [((A, a, 0), (PL.FIXED, 0, 0))])
    with pytest.raises(ValueError):
        PL.permutation_mapping(cs, 16, [((A, a, 0), (A, b, 16))])


def test_copy_blocks_are_swaps_only_when_nothing_else_touches_them(PL):
    """keygen's block path (row-range swaps on the device) must equal the general cycle merge of the expanded constraints"""
    cs = PL.ConstraintSystem()
    cols = [cs.advice_column() for _ in range(4)]
    inst = cs.instance_column()
    A, I = PL.ADVICE, PL.INSTANCE
    for c in cols: cs.enable_equality(A, c)
    cs.enable_equality(I, inst)
    n = 64
    copies = [PL.CopyBlock((I, inst, 0), (A, cols[0], 0), 16),          # clean 2-cycles
              PL.CopyBlock((A, cols[1], 4), (A, cols[2], 8), 10),       # overlaps the next block in column 2 -> general path
              PL.CopyBlock((A, cols[2], 12), (A, cols[3], 0), 6),
              PL.CopyBlock((A, cols[3], 20), (A, cols[3], 24), 8),      # overlaps itself (shifted copy within a column) -> general path
              PL.CopyBlock((A, cols[1], 40), (A, cols[3], 40), 5),      # touched by a single pair below -> general path
              ((A, cols[1], 42), (A, cols[0], 50)),
              PL.CopyBlock((A, cols[0], 30), (A, cols[0], 30), 3)]      # a cell copied onto itself: no-op
    want = PL.permutation_mapping(cs, n, copies)
    pairs, blocks = PL._split_disjoint_blocks(cs, n, list(copies))
    got = PL.permutation_mapping(cs, n, pairs)
    assert len(blocks) == 1
    for (i, r, i2, r2, rows) in blocks:
        for t in range(rows):
            assert (i, r + t) not in got and (i2, r2 + t) not in got
            got[(i, r + t)], got[(i2, r2 + t)] = (i2, r2 + t), (i, r + t)
    assert got == want
    with pytest.raises(ValueError):
        PL._split_disjoint_blocks(cs, n, [PL.CopyBlock((A, cols[0], 60), (A, cols[1], 0), 8)])


def test_copy_blocks_nested_in_a_wide_block_take_the_general_path(PL):
    """a wide block overlaps blocks that are not its neighbours in sorted order (A = rows 0..100, B = 10..20, C = 50..60 of one
    column): none of the three may become a device-side swap, and the result must equal the cycle merge of the expanded pairs"""
    cs = PL.ConstraintSystem()
    cols = [cs.advice_column() for _ in range(5)]
    A = PL.ADVICE
    for c in cols: cs.enable_equality(A, c)
    n = 128
    copies = [PL.CopyBlock((A, cols[0], 0), (A, cols[1], 0), 100),
              PL.CopyBlock((A, cols[0], 10), (A, cols[2], 0), 10),
              PL.CopyBlock((A, cols[0], 50), (A, cols[3], 0), 10),
              PL.CopyBlock((A, cols[4], 0), (A, cols[4], 64), 32)]      # untouched by the others: stays a swap
    want = PL.permutation_mapping(cs, n, copies)
    pairs, blocks = PL._split_disjoint_blocks(cs, n, list(copies))
    assert blocks == [(4, 0, 4, 64, 32)]
    got = PL.permutation_mapping(cs, n, pairs)
    for (i, r, i2, r2, rows) in blocks:
        for t in range(rows):
            assert (i, r + t) not in got and (i2, r2 + t) not in got
            got[(i, r + t)], got[(i2, r2 + t)] = (i2, r2 + t), (i, r + t)
    assert got == want
    # a single pair inside the wide block, far from any block start
    copies2 = [PL.CopyBlock((A, cols[0], 0), (A, cols[1], 0), 100), PL.CopyBlock((A, cols[2], 5), (A, cols[3], 5), 4),
               ((A, cols[0], 77), (A, cols[4], 3))]
    pairs2, blocks2 = PL._split_disjoint_blocks(cs, n, list(copies2))
    assert blocks2 == [(2, 5, 3, 5, 4)]


def test_cached_quotient_program_equals_a_fresh_compile_in_quotient_pieces(PL):
    """GpuBackend.quotient_program keeps the compiled quotient program of a proving key and patches the challenge-dependent
    constants (theta, beta, gamma, y, beta * DELTA^i).  Run here over the oracle's PythonBackend: for two proofs of the same key
    (the second one takes the cached path) the patched program must equal a fresh compile of that proof's Ast, for the small
    test circuit and for the real TinyRamCircuit (lookups with theta, a 47-chunk permutation)."""
    import random
    import numpy as np
    from util import pm
    import plonk_model as VM
    import plonk_circuits
    import tinyram_programs as TP
    import __graft_entry__ as ge
    ge.load_package()
    from tiny_ram_halo2_b200 import poly as P, tinyram as TR, trace as T
    C = pm.Vesta

    class Stop(Exception):
        pass

    class Probe(VM.PythonBackend):
        checked = 0

        def quotient_pieces(self, pk, challenges, build_h, build_parts, resolve):
            got = PL.GpuBackend.quotient_program(self, pk, build_h, challenges, len(pk.vk.cs.permutation))
            assert got is not None
            prog, keys = got
            ast, keys_fresh = build_h(*challenges)
            fresh = P.compile_ast(ast, self.p)
            assert keys == keys_fresh and (prog.code == fresh.code).all() and prog.consts == fresh.consts and prog.n_regs == fresh.n_regs
            Probe.checked += 1
            if self.stop_after_check:
                raise Stop()
            return super().quotient_pieces(pk, challenges, build_h, build_parts, resolve)     # the proof must still verify

    rnd = random.Random(5)
    rand = lambda: rnd.randrange(C.scalar.p)
    cs, fixed, copies, adv, inst = plonk_circuits.standard(PL, wide_lookup=True)
    be = Probe(C, 4, cs.degree()); be.stop_after_check = False
    pk = PL.keygen(be, cs, fixed, copies)
    for _ in range(2):
        proof = PL.create_proof(be, pk, inst, adv, rand, PL.Blake2bWrite(C.base.p, C.scalar.p))
        assert VM.verify_proof(C, be.params, pk.vk, inst, proof)
    assert Probe.checked == 2 and pk._quotient_program[id(be)]
    circ, fixed, copies, adv, inst = TR.build(PL, TP.answer_only(T, 8), 6)
    be = Probe(C, 6, circ.cs.degree()); be.stop_after_check = True
    pk = PL.keygen(be, circ.cs, fixed, copies)
    for _ in range(2):
        with pytest.raises(Stop):
            PL.create_proof(be, pk, inst, adv, rand, PL.Blake2bWrite(C.base.p, C.scalar.p))
    assert Probe.checked == 4
    slots = pk._quotient_program[id(be)][2]
    names = {s[0] for s in slots if s is not None}
    assert names == {"theta", "beta", "gamma", "y", "beta_delta"}


def test_summation_by_parts_commitment_identity():
    """sum_i z_i G_i = sum_j (z_j - z_{j+1}) Q_j, Q_j = G_0 + ... + G_j, z_n = 0 -- what plonk.GpuBackend._commit_many(runs=True) relies
    on to commit halo2's grand-product columns (constant over the rows a circuit leaves unused) through their sparse differences;
    checked here with the oracle's affine group law on a column with runs, zeros and a change in the last row"""
    import random
    import pasta_model as pm
    C = pm.Vesta
    r = C.scalar.p
    rng = random.Random(17)
    n = 24
    G, P = [], C.G
    for _ in range(n):
        P = C.add(C.double(P), C.G)
        G.append(P)
    z, v = [], 0
    for i in range(n):
        if rng.random() < 0.3:
            v = rng.choice([0, rng.randrange(r)])
        z.append(v)
    z[-1] = rng.randrange(r)
    def smul(k, P):
        acc, k = None, k % r
        while k:
            if k & 1:
                acc = C.add(acc, P)
            P = C.double(P)
            k >>= 1
        return acc
    direct = None
    for zi, Gi in zip(z, G):
        direct = C.add(direct, smul(zi, Gi))
    Q, acc = [], None
    for Gi in G:
        acc = C.add(acc, Gi)
        Q.append(acc)
    e = [(z[j] - (z[j + 1] if j + 1 < n else 0)) % r for j in range(n)]
    by_parts = None
    for ej, Qj in zip(e, Q):
        by_parts = C.add(by_parts, smul(ej, Qj))
    assert by_parts == direct and direct is not None
    assert sum(1 for x in e if x) < n
