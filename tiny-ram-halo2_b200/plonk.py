"""Mirror of halo2_proofs::plonk::{ConstraintSystem, keygen_vk, keygen_pk, create_proof} and of the Blake2b transcript
(plonk/{circuit,keygen,prover}.rs, plonk/{permutation,lookup,vanishing}/prover.rs, poly/multiopen/prover.rs, transcript.rs of
halo2_proofs 0.2.0 @ a95945254dcc, the un-vendored dependency the reference calls at /root/reference/src/test_utils.rs:21-49)
-- SURVEY.md 8(f) row f4: the proof assembly that strings the hot kernels together and produces the serialized proof.

The protocol logic below (phase order, RNG draw order, transcript order, query order, point-set construction) is host code,
as it is in the reference; every piece of field / group arithmetic goes through a BACKEND object (BACKEND_METHODS below):

    GpuBackend (this file)      the product: libtrp.so through the ctypes mirrors (commitment / domain / poly / permutation /
                                lookup / ipa).  There is no CPU fallback; constructing it without a GPU raises TrpError.
    oracle/plonk_model.py       test infrastructure only: the same interface over the Python big-int model, used by the
                                tests as the checker (identical proof bytes), next to an independent verify_proof.

Values at this level are canonical Python ints; points are affine (x, y) int tuples, None = identity.  The witness is
supplied as columns (circuit synthesis / layouting stay with the caller, as north_star keeps them on the Rust side).

Deviation that cannot be avoided here: VerifyingKey::transcript_repr hashes Rust's `{:?}` rendering of the pinned key; the same
BLAKE2b construction is applied to OUR canonical text rendering (pinned_text), so proofs are self-consistent with
oracle/plonk_model.verify_proof but the first transcript scalar differs from a Rust run's."""
from __future__ import annotations

import hashlib
from dataclasses import dataclass, field
from typing import Callable, List, Optional, Sequence, Tuple

from . import poly as P

ADVICE, FIXED, INSTANCE = "advice", "fixed", "instance"


# ---- plonk::Expression ------------------------------------------------------------------------------------------------------------
class Expression:
    def __add__(self, o): return Sum(self, _lift(o))
    __radd__ = __add__
    def __neg__(self): return Negated(self)
    def __sub__(self, o): return Sum(self, Negated(_lift(o)))
    def __rsub__(self, o): return Sum(_lift(o), Negated(self))
    def __mul__(self, o): return Scaled(self, o) if isinstance(o, int) else Product(self, o)
    def __rmul__(self, o): return Scaled(self, o)


def _lift(x):
    return Constant(x) if isinstance(x, int) else x


@dataclass(eq=False)
class Constant(Expression):
    value: int
    def degree(self): return 0


@dataclass(eq=False)
class Query(Expression):
    kind: str
    column: int
    rotation: int
    def degree(self): return 1


@dataclass(eq=False)
class Negated(Expression):
    a: Expression
    def degree(self): return self.a.degree()


@dataclass(eq=False)
class Sum(Expression):
    a: Expression
    b: Expression
    def degree(self): return max(self.a.degree(), self.b.degree())


@dataclass(eq=False)
class Product(Expression):
    a: Expression
    b: Expression
    def degree(self): return self.a.degree() + self.b.degree()


@dataclass(eq=False)
class Scaled(Expression):
    a: Expression
    scalar: int
    def degree(self): return self.a.degree()


def evaluate_expression(e: Expression, p: int, query: Callable[[Query], int]) -> int:
    """Expression::evaluate over field elements (the verifier's use, and row-wise compression of lookup expressions)"""
    if isinstance(e, Constant): return e.value % p
    if isinstance(e, Query): return query(e)
    if isinstance(e, Negated): return -evaluate_expression(e.a, p, query) % p
    if isinstance(e, Sum): return (evaluate_expression(e.a, p, query) + evaluate_expression(e.b, p, query)) % p
    if isinstance(e, Product): return evaluate_expression(e.a, p, query) * evaluate_expression(e.b, p, query) % p
    if isinstance(e, Scaled): return evaluate_expression(e.a, p, query) * e.scalar % p
    raise TypeError(type(e))


# ---- plonk::ConstraintSystem ------------------------------------------------------------------------------------------------------
class ConstraintSystem:
    """The subset of plonk::ConstraintSystem the prover reads: columns, ordered queries, gate polynomials, lookups, the
    permutation's columns.  Selectors are plain fixed columns here (halo2 compresses them into fixed columns at keygen)."""

    def __init__(self):
        self.num_advice = self.num_fixed = self.num_instance = 0
        self.queries = {ADVICE: [], FIXED: [], INSTANCE: []}     # ordered (column, rotation), as cs.*_queries
        self.num_advice_queries: List[int] = []
        self.gates: List[Expression] = []
        self.lookups: List[Tuple[List[Expression], List[Expression]]] = []
        self.permutation: List[Tuple[str, int]] = []
        self.minimum_degree: Optional[int] = None

    def advice_column(self):
        self.num_advice += 1; self.num_advice_queries.append(0); return self.num_advice - 1

    def fixed_column(self):
        self.num_fixed += 1; return self.num_fixed - 1

    def instance_column(self):
        self.num_instance += 1; return self.num_instance - 1

    def query(self, kind: str, column: int, rotation: int = 0) -> Query:
        """meta.query_advice / query_fixed / query_instance: registers (column, rotation) on first use"""
        if (column, rotation) not in self.queries[kind]:
            self.queries[kind].append((column, rotation))
            if kind == ADVICE:
                self.num_advice_queries[column] += 1
        return Query(kind, column, rotation)

    def enable_equality(self, kind: str, column: int):
        self.query(kind, column, 0)
        if (kind, column) not in self.permutation:
            self.permutation.append((kind, column))

    def create_gate(self, polys: Sequence[Expression]):
        self.gates.extend(polys)

    def lookup(self, pairs: Sequence[Tuple[Expression, Expression]]):
        self.lookups.append(([a for a, _ in pairs], [t for _, t in pairs]))

    def query_index(self, kind, column, rotation):
        return self.queries[kind].index((column, rotation))

    def degree(self) -> int:
        degree = 3                                              # permutation::Argument::required_degree
        for inputs, tables in self.lookups:
            di = max([1] + [e.degree() for e in inputs]); dt = max([1] + [e.degree() for e in tables])
            degree = max(degree, max(4, 2 + di + dt))           # lookup::Argument::required_degree
        degree = max([degree] + [g.degree() for g in self.gates])
        return max(degree, self.minimum_degree or 1)

    def blinding_factors(self) -> int:
        factors = max(self.num_advice_queries + [1])
        return max(3, factors) + 2

    def minimum_rows(self) -> int:
        return self.blinding_factors() + 3

    def pinned_text(self) -> str:
        def ex(e):
            if isinstance(e, Constant): return f"Constant({e.value:#x})"
            if isinstance(e, Query): return f"{e.kind.capitalize()}({e.column}, {e.rotation})"
            if isinstance(e, Negated): return f"Negated({ex(e.a)})"
            if isinstance(e, Sum): return f"Sum({ex(e.a)}, {ex(e.b)})"
            if isinstance(e, Product): return f"Product({ex(e.a)}, {ex(e.b)})"
            return f"Scaled({ex(e.a)}, {e.scalar:#x})"
        return (f"PinnedConstraintSystem {{ num_fixed_columns: {self.num_fixed}, num_advice_columns: {self.num_advice}, "
                f"num_instance_columns: {self.num_instance}, gates: [{', '.join(ex(g) for g in self.gates)}], "
                f"advice_queries: {self.queries[ADVICE]}, instance_queries: {self.queries[INSTANCE]}, fixed_queries: {self.queries[FIXED]}, "
                f"permutation: {self.permutation}, lookups: [{', '.join('(' + ', '.join(ex(e) for e in a) + ' -> ' + ', '.join(ex(e) for e in t) + ')' for a, t in self.lookups)}], "
                f"minimum_degree: {self.minimum_degree} }}")


# ---- transcript.rs: Blake2bWrite<_, _, Challenge255<_>> ---------------------------------------------------------------------------
class Blake2bWrite:
    """BLAKE2b-512 personalised "Halo2-Transcript"; prefixes 0 (challenge), 1 (point), 2 (scalar); points enter the hash as
    x || y (32-byte little-endian each) and the proof as the 32-byte compressed encoding; a challenge is the 64-byte digest
    read little-endian and reduced (Challenge255 / from_bytes_wide)."""

    def __init__(self, base_modulus: int, scalar_modulus: int):
        self.state = hashlib.blake2b(digest_size=64, person=b"Halo2-Transcript")
        self.q, self.p = base_modulus, scalar_modulus
        self.proof = bytearray()

    def common_point(self, pt):
        if pt is None:
            raise ValueError("cannot write points at infinity to the transcript")
        self.state.update(b"\x01" + pt[0].to_bytes(32, "little") + pt[1].to_bytes(32, "little"))

    def common_scalar(self, s):
        self.state.update(b"\x02" + (s % self.p).to_bytes(32, "little"))

    def write_point(self, pt):
        self.common_point(pt)
        b = bytearray(pt[0].to_bytes(32, "little"))
        b[31] |= (pt[1] & 1) << 7
        self.proof += b

    def write_scalar(self, s):
        self.common_scalar(s)
        self.proof += (s % self.p).to_bytes(32, "little")

    def squeeze_challenge_scalar(self) -> int:
        self.state.update(b"\x00")
        return int.from_bytes(self.state.copy().digest(), "little") % self.p

    def finalize(self) -> bytes:
        return bytes(self.proof)


def transcript_repr(text: str, p: int) -> int:
    """VerifyingKey::from_parts: BLAKE2b-512 personalised "Halo2-Verify-Key" over len(text) (u64 LE) || text, from_bytes_wide"""
    h = hashlib.blake2b(digest_size=64, person=b"Halo2-Verify-Key")
    h.update(len(text).to_bytes(8, "little") + text.encode())
    return int.from_bytes(h.digest(), "little") % p


# ---- keys -------------------------------------------------------------------------------------------------------------------------
@dataclass
class VerifyingKey:
    k: int
    cs: ConstraintSystem
    cs_degree: int
    fixed_commitments: list
    permutation_commitments: list
    transcript_repr: int


@dataclass
class ProvingKey:
    vk: VerifyingKey
    fixed_values: list
    fixed_polys: list
    fixed_cosets: list
    sigma_values: list
    sigma_polys: list
    sigma_cosets: list
    l0: object
    l_blind: object
    l_last: object


@dataclass(frozen=True)
class CopyBlock:
    """`rows` consecutive copy constraints (kind, column, row0 + t) == (kind', column', row0' + t), t < rows: what a loop of
    assign_advice_from_instance / copy_advice over a region produces (e.g. /root/reference/src/circuits/tables/prog.rs:206-216).
    Equivalent to its expansion into pairs; keygen handles blocks that touch no other constraint without expanding them."""
    left: Tuple[str, int, int]
    right: Tuple[str, int, int]
    rows: int


def expand_copies(copies):
    """the copy constraints as plain ((kind, column, row), (kind, column, row)) pairs"""
    for c in copies:
        if isinstance(c, CopyBlock):
            (lk, lc, lr), (rk, rc, rr) = c.left, c.right
            for t in range(c.rows):
                yield ((lk, lc, lr + t), (rk, rc, rr + t))
        else:
            yield c


def _split_disjoint_blocks(cs: ConstraintSystem, n: int, copies):
    """(pairs, blocks): blocks = the CopyBlocks whose cells occur in no other copy constraint (their cycles are the 2-cycles
    left <-> right, so sigma is a swap of two row ranges), as (column, row0, column', row0', rows) over cs.permutation indices;
    every other constraint is returned expanded in `pairs`."""
    col_of = {kc: i for i, kc in enumerate(cs.permutation)}
    blocks = [c for c in copies if isinstance(c, CopyBlock)]
    pairs = [c for c in copies if not isinstance(c, CopyBlock)]
    spans = []                                  # (column, lo, hi, block index)
    for bi, b in enumerate(blocks):
        for kind, col, r0 in (b.left, b.right):
            if (kind, col) not in col_of:
                raise ValueError("copy constraint on a column without enable_equality")
            if not (0 <= r0 and r0 + b.rows <= n):
                raise ValueError("copy constraint outside the domain")
            spans.append((col_of[(kind, col)], r0, r0 + b.rows, bi))
    spans.sort()
    shared = set()
    cur_col, max_hi, owner = None, 0, None     # interval sweep per column: the running maximum `hi` and the block that set it
    for c, lo, hi, b in spans:                  # (a wide span overlaps spans that are not its neighbours in sorted order)
        if c != cur_col:
            cur_col, max_hi, owner = c, hi, b
            continue
        if lo < max_hi:
            shared.update((owner, b))
        if hi > max_hi:
            max_hi, owner = hi, b
    if pairs and blocks:
        import bisect
        starts = [(c, lo) for c, lo, _, _ in spans]
        for pair in pairs:
            for kind, col, r in pair:
                i = bisect.bisect_right(starts, (col_of.get((kind, col), -1), r)) - 1
                if i >= 0 and spans[i][0] == col_of.get((kind, col), -1) and spans[i][1] <= r < spans[i][2]:
                    shared.add(spans[i][3])
    out, ordered, bi = [], [], 0                # halo2 merges cycles in the order of the copy calls: keep that order
    for c in copies:
        if not isinstance(c, CopyBlock):
            ordered.append(c)
            continue
        b = c
        if bi in shared or b.left[:2] == b.right[:2] and abs(b.left[2] - b.right[2]) < b.rows:
            ordered.extend(expand_copies([b]))
        elif b.rows:
            out.append((col_of[b.left[:2]], b.left[2], col_of[b.right[:2]], b.right[2], b.rows))
        bi += 1
    pairs = ordered
    return pairs, out


def permutation_mapping(cs: ConstraintSystem, n: int, copies):
    """permutation::keygen::Assembly: cycles of the copy constraints (copy -> merge the two cycles, smaller into larger).
    Returns {(column, row): (column', row')} for the cells whose image differs from themselves; column = index into
    cs.permutation.  copies: ((kind, column, row), (kind, column, row)) pairs.  Cells no copy touches never enter the dict,
    so keygen stays O(copies) however large n is."""
    col_of = {kc: i for i, kc in enumerate(cs.permutation)}
    mapping, aux, sizes = {}, {}, {}
    for (lk, lc, lr), (rk, rc, rr) in expand_copies(copies):
        if (lk, lc) not in col_of or (rk, rc) not in col_of:
            raise ValueError("copy constraint on a column without enable_equality")
        left, right = (col_of[(lk, lc)], lr), (col_of[(rk, rc)], rr)
        if not (0 <= lr < n and 0 <= rr < n):
            raise ValueError("copy constraint outside the domain")
        lcyc, rcyc = aux.get(left, left), aux.get(right, right)
        if lcyc == rcyc:
            continue
        if sizes.get(lcyc, 1) < sizes.get(rcyc, 1):
            lcyc, rcyc = rcyc, lcyc
        sizes[lcyc] = sizes.get(lcyc, 1) + sizes.get(rcyc, 1)
        i = rcyc
        while True:
            aux[i] = lcyc
            i = mapping.get(i, i)
            if i == rcyc:
                break
        ml, mr = mapping.get(left, left), mapping.get(right, right)
        mapping[left], mapping[right] = mr, ml
    return {c: t for c, t in mapping.items() if c != t}


def build_sigmas(cs: ConstraintSystem, n: int, p: int, omega: int, delta: int, copies):
    """build_pk's sigma values as dense int lists: sigma_i[j] = delta^i' * omega^j' for the cell (i', j') that (i, j) maps to"""
    m = len(cs.permutation)
    moved = permutation_mapping(cs, n, copies)
    om = [1] * n
    for j in range(1, n):
        om[j] = om[j - 1] * omega % p
    dl = [1] * max(m, 1)
    for i in range(1, m):
        dl[i] = dl[i - 1] * delta % p
    out = [[dl[i] * om[j] % p for j in range(n)] for i in range(m)]
    for (i, j), (i2, j2) in moved.items():
        out[i][j] = dl[i2] * om[j2] % p
    return out


# ---- the backend interface: all that keygen and create_proof ask of a backend, and every backend implements all of it --------------
# (GpuBackend, sharded_backend.ShardedGpuBackend, oracle/plonk_model.PythonBackend).  A batch method means the loop over its
# single-item operation; v is a vector of n values, bf the number of blinding factors.
BACKEND_ATTRIBUTES = ("n", "p", "q", "k", "j", "extended_k", "omega", "delta",   # 2^k rows, moduli, cs degree, domain constants
                      "leaves_are_coefficients")       # the quotient's leaves stay in coefficient form (debug=True needs it)
BACKEND_METHODS = (
    "rotate_omega",               # (x, rotation) -> omega^rotation x
    "vec",                        # (values) -> v, zero-padded to n rows
    "set_rows",                   # (v, start, values) -> v with v[start : start + len(values)] = values
    "set_rows_many",              # (vs, start, values): set_rows(vs[i], start, values[i]) for each i
    "random_vec",                 # (rand) -> a random v
    "mul_add",                    # (acc, s, v) -> acc s + v (v when acc is None)
    "sub_low",                    # (v, low) -> v - low on the first len(low) coefficients
    "sigma_vecs",                 # (m, moved) -> m columns of identity labels delta^i omega^j, moved cells relabelled
    "sigma_swap_blocks",          # (sigmas, blocks) -> sigmas, each block's two row ranges exchanging their identity labels
    "commit",                     # (v, blind) -> the commitment over g (coefficient form)
    "commit_many",                # (vs, blinds) -> [commit]
    "commit_lagrange_many",       # (vs, blinds, sparse=, runs=) -> commitments over g_lagrange; sparse / runs are density hints
    "lagrange_to_coeff",          # (v) -> coefficients
    "lagrange_to_coeff_many",     # (vs) -> [lagrange_to_coeff]
    "coeff_to_extended",          # (coeffs) -> the quotient's leaf for a proof's polynomial
    "coeff_to_extended_static",   # (coeffs) -> the same for key material, which the backend may cache
    "begin_proof",                # (n_polys): a proof starts and will bring n_polys polynomials to coefficient form
    "end_proof",                  # (): the proof is done (keygen calls it too)
    "_wait",                      # (): block until the enqueued work has finished (phase timings)
    "lookups_commit_permuted",    # (lookups, theta, values_of, usable, bf, rand) -> per lookup {ci, ct, pi, pt, pi_blind, pt_blind}
    "permutation_commit",         # (values, sigmas, beta, gamma, chunk_len, bf, rand, after_chunk): after_chunk(z) per chunk
    "lookup_products",            # (lookups, beta, gamma, bf, rand): sets each lookup's z and z_blind
    "quotient_pieces",            # (pk, challenges, build_h, build_parts, resolve) -> the j - 1 pieces of h(X)
    "eval_polynomial",            # (coeffs, x) -> value
    "eval_polynomials_at",        # (vs, x) -> [eval_polynomial]
    "linear_combination",         # (vs, scalars) -> sum_j scalars[j] vs[j]
    "kate_division",              # (coeffs, b) -> (coeffs - coeffs(b)) / (X - b)
    "ipa_create_proof",           # (rand, transcript, p_poly, p_blind, x_3): the opening argument
)


def keygen(backend, cs: ConstraintSystem, fixed_values, copies=()) -> ProvingKey:
    """keygen_vk + keygen_pk.  fixed_values: one column per fixed column -- a list of at most n ints (zero-padded) or a
    backend vector."""
    n, p = backend.n, backend.p
    backend.end_proof()                        # key material never lives in a proof's polynomial arena
    if n < cs.minimum_rows():
        raise ValueError("NotEnoughRowsAvailable")
    if backend.j != cs.degree():
        raise ValueError("the backend's EvaluationDomain was built for a different constraint-system degree")
    if len(fixed_values) != cs.num_fixed:
        raise ValueError("one column per fixed column")
    fixed_values = [backend.vec(v) for v in fixed_values]
    fixed_commitments = backend.commit_lagrange_many(fixed_values, [1] * len(fixed_values))          # Blind::default() = 1
    pairs, blocks = _split_disjoint_blocks(cs, n, list(copies))     # row-range swaps for the blocks no other constraint touches
    sigma_values = backend.sigma_swap_blocks(backend.sigma_vecs(len(cs.permutation), permutation_mapping(cs, n, pairs)), blocks)
    permutation_commitments = backend.commit_lagrange_many(sigma_values, [1] * len(sigma_values))
    pt = lambda c: "Identity" if c is None else f"({c[0]:#066x}, {c[1]:#066x})"
    text = (f"PinnedVerificationKey {{ base_modulus: {backend.q:#066x}, scalar_modulus: {p:#066x}, domain: PinnedEvaluationDomain {{ k: {backend.k}, "
            f"extended_k: {backend.extended_k}, omega: {backend.omega:#066x} }}, cs: {cs.pinned_text()}, "
            f"fixed_commitments: [{', '.join(pt(c) for c in fixed_commitments)}], permutation: VerifyingKey {{ commitments: "
            f"[{', '.join(pt(c) for c in permutation_commitments)}] }} }}")
    vk = VerifyingKey(backend.k, cs, cs.degree(), fixed_commitments, permutation_commitments, transcript_repr(text, p))
    fixed_polys = [backend.lagrange_to_coeff(v) for v in fixed_values]
    sigma_polys = [backend.lagrange_to_coeff(v) for v in sigma_values]
    bf = cs.blinding_factors()
    static = backend.coeff_to_extended_static      # key material: cosets may be cached
    ext = lambda lag: static(backend.lagrange_to_coeff(lag))
    l0 = backend.vec([1])
    l_blind = backend.set_rows(backend.vec([]), n - bf, [1] * bf)
    l_last = backend.set_rows(backend.vec([]), n - bf - 1, [1])
    return ProvingKey(vk, fixed_values, fixed_polys, [static(c) for c in fixed_polys], sigma_values, sigma_polys,
                      [static(c) for c in sigma_polys], ext(l0), ext(l_blind), ext(l_last))


# ---- poly/multiopen: construct_intermediate_sets -----------------------------------------------------------------------------------
def construct_intermediate_sets(queries, commitment_key: Callable, point_of: Callable, eval_of: Callable):
    """poly::multiopen::construct_intermediate_sets.  Returns (commitment_map, point_sets): commitment_map is a list of dicts
    {commitment, set_index, point_indices, evals} in order of first appearance; point_sets[set] lists that set's points."""
    point_index_map = {}
    for q in queries:
        point_index_map.setdefault(point_of(q), len(point_index_map))
    inverse = {v: k for k, v in point_index_map.items()}
    cmap, where = [], {}
    for q in queries:
        key = commitment_key(q)
        if key not in where:
            where[key] = len(cmap)
            cmap.append({"commitment": q, "point_indices": [], "set_index": None, "evals": None})
        pi = point_index_map[point_of(q)]
        if pi not in cmap[where[key]]["point_indices"]:
            cmap[where[key]]["point_indices"].append(pi)
    point_idx_sets = {}
    for cd in cmap:
        point_idx_sets.setdefault(tuple(sorted(cd["point_indices"])), len(point_idx_sets))
    for cd in cmap:
        cd["evals"] = [None] * len(cd["point_indices"])
    for q in queries:
        cd = cmap[where[commitment_key(q)]]
        pset = tuple(sorted(cd["point_indices"]))
        cd["set_index"] = point_idx_sets[pset]
        cd["evals"][pset.index(point_index_map[point_of(q)])] = eval_of(q)
    point_sets = [None] * len(point_idx_sets)
    for pset, idx in point_idx_sets.items():
        point_sets[idx] = [inverse[i] for i in pset]
    return cmap, point_sets


def lagrange_interpolate(points, evals, p):
    """arithmetic::lagrange_interpolate: coefficients (low -> high) of the polynomial of degree < len(points) through the pairs"""
    m = len(points)
    if m == 1:
        return [evals[0] % p]
    out = [0] * m
    for j in range(m):
        num, den = [1], 1
        for i in range(m):
            if i == j:
                continue
            nxt = [0] * (len(num) + 1)
            for d, c in enumerate(num):
                nxt[d] = (nxt[d] - c * points[i]) % p
                nxt[d + 1] = (nxt[d + 1] + c) % p
            num = nxt
            den = den * (points[j] - points[i]) % p
        s = evals[j] * pow(den, -1, p) % p
        for d, c in enumerate(num):
            out[d] = (out[d] + c * s) % p
    return out


# ---- plonk::create_proof -----------------------------------------------------------------------------------------------------------
@dataclass
class _Opening:
    poly: list          # coefficient form
    blind: int
    point: int
    eval: int = 0


def eval_ast_at_point(B, ast, polys, x):
    """value at X = x of an Ast whose leaves are coefficient-form polynomials (debug aid: the vanishing identity at one point)"""
    p = B.p
    memo = {}

    def go(a):
        if isinstance(a, P.Poly):
            key = (a.index, a.rotation)
            if key not in memo:
                memo[key] = B.eval_polynomial(polys[a.index], B.rotate_omega(x, a.rotation))
            return memo[key]
        if isinstance(a, P.Add): return (go(a.a) + go(a.b)) % p
        if isinstance(a, P.Mul): return go(a.a) * go(a.b) % p
        if isinstance(a, P.Scale): return go(a.a) * a.scalar % p
        if isinstance(a, P.LinearTerm): return a.scalar * x % p
        if isinstance(a, P.ConstantTerm): return a.scalar % p
        if isinstance(a, P.DistributePowers):
            base, acc = go(a.base), 0
            for t in a.terms:
                acc = (acc * base + go(t)) % p
            return acc
        raise TypeError(type(a))

    import sys
    old = sys.getrecursionlimit(); sys.setrecursionlimit(max(old, 100000))
    try:
        return go(ast)
    finally:
        sys.setrecursionlimit(old)


def quotient_constraints(cs: ConstraintSystem, cs_degree: int, p: int, delta: int, theta_: int, beta_: int, gamma_: int):
    """every constraint of the vanishing argument as a poly::Ast over symbolic leaves, in halo2's order: (exprs, leaf keys in
    leaf-index order).  Its SHAPE depends on the constraint system only; the challenges enter as constants."""
    leaves, keys = {}, []
    bf, chunk_len = cs.blinding_factors(), cs_degree - 2

    def leaf(key):
        if key not in leaves:
            leaves[key] = len(keys)
            keys.append(key)
        return P.Poly(leaves[key], 0)

    def to_ast(e):
        if isinstance(e, Constant): return P.ConstantTerm(e.value % p)
        if isinstance(e, Query): return leaf((e.kind, e.column)).with_rotation(e.rotation)
        if isinstance(e, Negated): return -to_ast(e.a)
        if isinstance(e, Sum): return to_ast(e.a) + to_ast(e.b)
        if isinstance(e, Product): return to_ast(e.a) * to_ast(e.b)
        return to_ast(e.a) * (e.scalar % p)

    l0, l_blind, l_last = leaf("l0"), leaf("l_blind"), leaf("l_last")
    one = P.ConstantTerm(1)
    active = one - (l_last + l_blind)
    exprs = [to_ast(g) for g in cs.gates]
    if cs.permutation:                          # one grand product per chunk of chunk_len columns
        zs = [leaf(("perm_z", i)) for i in range(-(-len(cs.permutation) // chunk_len))]
        exprs.append(l0 * (one - zs[0]))
        exprs.append(l_last * (zs[-1] * zs[-1] - zs[-1]))
        for i in range(1, len(zs)):
            exprs.append(l0 * (zs[i] - zs[i - 1].with_rotation(-(bf + 1))))
        for i, z in enumerate(zs):
            cols = cs.permutation[i * chunk_len:(i + 1) * chunk_len]
            left, right = z.with_rotation(1), z
            cur_delta = beta_ * pow(delta, i * chunk_len, p) % p
            for off, (kk, c) in enumerate(cols):
                col = leaf((kk, c))
                sig = leaf(("sigma", i * chunk_len + off))
                left = left * (col + sig * beta_ + gamma_)
                right = right * (col + P.LinearTerm(cur_delta) + gamma_)
                cur_delta = cur_delta * delta % p
            exprs.append((left - right) * active)
    for li, (inputs, tables) in enumerate(cs.lookups):
        z, a, s = leaf(("lookup_z", li)), leaf(("lookup_a", li)), leaf(("lookup_s", li))
        comp = lambda es: P.DistributePowers([to_ast(e) for e in es], P.ConstantTerm(theta_)) if len(es) > 1 else to_ast(es[0])
        exprs.append(l0 * (one - z))
        exprs.append(l_last * (z * z - z))
        exprs.append((z.with_rotation(1) * (a + beta_) * (s + gamma_) - z * (comp(inputs) + beta_) * (comp(tables) + gamma_)) * active)
        exprs.append(l0 * (a - s))
        exprs.append(((a - s) * (a - a.with_rotation(-1))) * active)
    return exprs, keys


def ast_degree(ast, memo=None) -> int:
    """upper bound on the degree in X of an Ast whose leaves have degree < n, in units of n (halo2's bound: a leaf and X count 1)"""
    memo = {} if memo is None else memo
    key = id(ast)
    if key not in memo:
        if isinstance(ast, (P.Poly, P.LinearTerm)): d = 1
        elif isinstance(ast, P.ConstantTerm): d = 0
        elif isinstance(ast, P.Add): d = max(ast_degree(ast.a, memo), ast_degree(ast.b, memo))
        elif isinstance(ast, P.Mul): d = ast_degree(ast.a, memo) + ast_degree(ast.b, memo)
        elif isinstance(ast, P.Scale): d = ast_degree(ast.a, memo)
        elif isinstance(ast, P.DistributePowers): d = max([ast_degree(ast.base, memo) * (len(ast.terms) - 1)] + [ast_degree(t, memo) for t in ast.terms])
        else: raise TypeError(type(ast))
        memo[key] = d
    return memo[key]


def split_by_degree(exprs, keys, y, cs_degree, p):
    """The folded numerator N = sum_i y^(m-1-i) exprs[i] as parts N_d, one per degree bound d of the constraints: every expr
    vanishes on the domain by itself, so h_d = N_d / (X^n - 1) has degree < (d - 1) n and needs only d - 1 cosets, and sum_d h_d is
    the quotient h.  Returns [(d - 1, Ast, leaf keys)] by increasing d; each part keeps its terms' powers of y (y^gap constants
    between its terms) and numbers its own leaves.  Degrees below 2 join d = 2 (a degree-1 numerator that vanishes on the
    domain is zero); a bound above cs_degree would break the monolithic quotient too, and raises."""
    memo = {}
    groups = {}
    for i, e in enumerate(exprs):
        d = max(ast_degree(e, memo), 2)
        if d > cs_degree:
            raise ValueError(f"constraint {i} has degree {d} > the constraint system's degree {cs_degree}")
        groups.setdefault(d, []).append(i)
    m, out = len(exprs), []
    for d in sorted(groups):
        acc, last = None, None
        for i in groups[d]:
            e = exprs[i]
            acc = e if acc is None else acc * P.ConstantTerm(pow(y, i - last, p)) + e
            last = i
        if m - 1 - last:
            acc = acc * P.ConstantTerm(pow(y, m - 1 - last, p))
        local, rebuilt = {}, {}

        def remap(a):                       # the part's own leaf numbering; shared subtrees stay shared (x * x stays a square)
            r = rebuilt.get(id(a))
            if r is not None:
                return r
            if isinstance(a, P.Poly):
                r = P.Poly(local.setdefault(a.index, len(local)), a.rotation)
            elif isinstance(a, (P.Add, P.Mul)):
                r = type(a)(remap(a.a), remap(a.b))
            elif isinstance(a, P.Scale):
                r = P.Scale(remap(a.a), a.scalar)
            elif isinstance(a, P.DistributePowers):
                r = P.DistributePowers([remap(t) for t in a.terms], remap(a.base))
            else:
                r = a
            rebuilt[id(a)] = r
            return r

        import sys
        old = sys.getrecursionlimit(); sys.setrecursionlimit(max(old, 100000))
        try:
            ast = remap(acc)
        finally:
            sys.setrecursionlimit(old)
        out.append((d - 1, ast, [keys[g] for g in sorted(local, key=local.get)]))
    return out


def create_proof(backend, pk: ProvingKey, instances, advice, rand: Callable[[], int], transcript: Blake2bWrite, debug: bool = False,
                 timings: Optional[dict] = None) -> bytes:
    """plonk::create_proof for ONE circuit instance.  instances: one column per instance column, advice: one per advice column
    -- lists of at most usable_rows ints, or backend vectors of n values whose blinding rows are overwritten here.  rand()
    draws one uniformly random scalar (the caller's RNG: every draw happens in halo2's order).  Polynomials are opaque backend
    vectors throughout; only scalars, points and the few interpolation coefficients live on the host.  Returns the proof
    bytes (also left in `transcript`)."""
    B = backend
    vk, cs = pk.vk, pk.vk.cs
    n, p, k = B.n, B.p, B.k
    bf = cs.blinding_factors()
    usable = n - (bf + 1)
    rot = B.rotate_omega
    if len(instances) != cs.num_instance or len(advice) != cs.num_advice:
        raise ValueError("InvalidInstances / wrong number of advice columns")
    transcript.common_scalar(vk.transcript_repr)
    chunks = -(-len(cs.permutation) // (vk.cs_degree - 2)) if cs.permutation else 0
    B.begin_proof(cs.num_instance + cs.num_advice + 3 * len(cs.lookups) + chunks)     # instance, advice, (A', S', Z) per lookup, Z per chunk
    import time as _time
    _t = [_time.perf_counter()]

    def tick(name):                            # wall-clock per phase; an asynchronous backend is drained first so that the
        if timings is not None:                # time lands in the phase that enqueued the work (a handful of waits per proof)
            B._wait()
            now = _time.perf_counter()
            timings[name] = timings.get(name, 0.0) + now - _t[0]
            _t[0] = now

    def column(col, what):
        if isinstance(col, (list, tuple)) and len(col) > usable:
            raise ValueError(f"{what} column longer than the usable rows")
        return B.vec(col)

    # commit_lagrange_many's hints (the backend checks the density itself): sparse = mostly zero (instance / advice / permuted lookup
    # columns of a circuit that uses a fraction of its rows); runs = constant over the rows a circuit leaves unused (grand products,
    # permuted lookup columns with a non-zero default), so the row-to-row differences are sparse (GpuBackend._commit_many)

    # ---- instance columns: commit (not written, only absorbed) -------------------------------------------------------------
    inst_values = [column(c, "InstanceTooLarge: instance") for c in instances]
    for cm in B.commit_lagrange_many(inst_values, [1] * len(inst_values), sparse=True):
        transcript.common_point(cm)
    inst_polys = B.lagrange_to_coeff_many(inst_values)
    inst_cosets = [B.coeff_to_extended(c) for c in inst_polys]
    tick("instance")

    # ---- advice columns --------------------------------------------------------------------------------------------------------
    adv_values = [column(c, "advice") for c in advice]
    B.set_rows_many(adv_values, usable, [[rand() for _ in range(usable, n)] for _ in adv_values])
    adv_blinds = [rand() for _ in adv_values]
    for cm in B.commit_lagrange_many(adv_values, adv_blinds, sparse=True):
        transcript.write_point(cm)
    adv_polys = B.lagrange_to_coeff_many(adv_values)
    adv_cosets = [B.coeff_to_extended(c) for c in adv_polys]
    values_of = {ADVICE: adv_values, FIXED: pk.fixed_values, INSTANCE: inst_values}
    tick("advice")

    # ---- lookups: commit_permuted -------------------------------------------------------------------------------------------------
    theta = transcript.squeeze_challenge_scalar()
    lookups = B.lookups_commit_permuted(cs.lookups, theta, values_of, usable, bf, rand)
    for L, pi_poly, pt_poly in zip(lookups, *[B.lagrange_to_coeff_many([L[nm] for L in lookups]) for nm in ("pi", "pt")]):
        L["pi_poly"], L["pt_poly"] = pi_poly, pt_poly
    # the commitments do not feed the RNG, so they are computed as one batch and written in halo2's order
    for cm in B.commit_lagrange_many([L[nm] for L in lookups for nm in ("pi", "pt")], [L[nm + "_blind"] for L in lookups for nm in ("pi", "pt")],
                                     sparse=True, runs=True):
        transcript.write_point(cm)
    tick("lookups_permuted")

    # ---- permutation and lookup grand products ----------------------------------------------------------------------------------------
    beta = transcript.squeeze_challenge_scalar()
    gamma = transcript.squeeze_challenge_scalar()
    chunk_len = vk.cs_degree - 2
    perm_sets = []

    def after_chunk(z):                        # halo2 draws the chunk's blind right after its blinding rows
        perm_sets.append({"z": z, "blind": rand()})

    if cs.permutation:
        B.permutation_commit([values_of[kk][c] for kk, c in cs.permutation], pk.sigma_values, beta, gamma, chunk_len, bf, rand, after_chunk)
    for cm in B.commit_lagrange_many([S["z"] for S in perm_sets], [S["blind"] for S in perm_sets], runs=True):
        transcript.write_point(cm)
    for S, poly in zip(perm_sets, B.lagrange_to_coeff_many([S["z"] for S in perm_sets])):
        S["poly"] = poly
        S["coset"] = B.coeff_to_extended(poly)
    B.lookup_products(lookups, beta, gamma, bf, rand)
    for cm in B.commit_lagrange_many([L["z"] for L in lookups], [L["z_blind"] for L in lookups], runs=True):
        transcript.write_point(cm)
    for L, poly in zip(lookups, B.lagrange_to_coeff_many([L["z"] for L in lookups])):
        L["z_poly"] = poly
    tick("grand_products")

    # ---- vanishing argument: random polynomial ------------------------------------------------------------------------------------------
    random_poly = B.random_vec(rand)
    random_blind = rand()
    transcript.write_point(B.commit(random_poly, random_blind))

    # ---- quotient --------------------------------------------------------------------------------------------------------------------
    y = transcript.squeeze_challenge_scalar()
    cos_of = {ADVICE: adv_cosets, FIXED: pk.fixed_cosets, INSTANCE: inst_cosets}

    def build_h(theta_, beta_, gamma_, y_):
        """the folded constraint polynomial sum_i y^(m-1-i) expr_i as one Ast: (h_ast, leaf keys)"""
        exprs, keys = quotient_constraints(cs, vk.cs_degree, p, B.delta, theta_, beta_, gamma_)
        h = P.ConstantTerm(0)
        for e in exprs:
            h = h * y_ + e
        return h, keys

    def build_parts(theta_, beta_, gamma_, y_):
        """the same sum split by constraint degree (quotient_parts)"""
        exprs, keys = quotient_constraints(cs, vk.cs_degree, p, B.delta, theta_, beta_, gamma_)
        return split_by_degree(exprs, keys, y_, vk.cs_degree, p)

    def resolve(key):                           # the polynomial of THIS proof behind a leaf key
        if isinstance(key, str):
            return getattr(pk, key)             # l0, l_blind, l_last
        tag = key[0]
        if tag == "perm_z": return perm_sets[key[1]]["coset"]
        if tag == "sigma": return pk.sigma_cosets[key[1]]
        if tag in ("lookup_z", "lookup_a", "lookup_s"):
            L = lookups[key[1]]
            name = {"lookup_z": "z_poly", "lookup_a": "pi_poly", "lookup_s": "pt_poly"}[tag]
            if name + "_ext" not in L:
                L[name + "_ext"] = B.coeff_to_extended(L[name])
            return L[name + "_ext"]
        return cos_of[tag][key[1]]

    # The backend picks the form of the numerator (the whole Ast, or parts by degree) and may keep the compiled programs of a
    # proving key, whose code depends on the constraint system only (GpuBackend.quotient_program).
    challenges = (theta, beta, gamma, y)
    pieces = B.quotient_pieces(pk, challenges, build_h, build_parts, resolve)      # the j - 1 pieces (n coefficients each) of h(X)
    if debug:        # h(X) (X^n - 1) must equal the folded constraint polynomial: checked at a point outside the domain
        if not B.leaves_are_coefficients:
            raise ValueError("debug=True needs a backend whose quotient leaves stay in coefficient form (GpuBackend)")
        h_ast, keys = build_h(*challenges)
        xd = 0x1234567890abcdef1234567890abcdef % p
        lhs = eval_ast_at_point(B, h_ast, [resolve(k_) for k_ in keys], xd)
        hx, xdn = 0, pow(xd, n, p)
        for piece in reversed(pieces):
            hx = (hx * xdn + B.eval_polynomial(piece, xd)) % p
        if lhs != hx * (xdn - 1) % p:
            raise AssertionError("the quotient does not satisfy h(X) (X^n - 1) = sum_i y^i expr_i(X): unsatisfied circuit or a "
                                 "fault in the quotient phase")
    h_blinds = [rand() for _ in pieces]
    for cm in B.commit_many(pieces, h_blinds):
        transcript.write_point(cm)
    tick("quotient")

    # ---- evaluations -----------------------------------------------------------------------------------------------------------------
    x = transcript.squeeze_challenge_scalar()
    xn = pow(x, n, p)
    polys_of = {ADVICE: adv_polys, FIXED: pk.fixed_polys, INSTANCE: inst_polys}
    cache = {}

    def ev(poly, point):                       # every opened value is computed once (transcript and multiopen share them)
        return cache[(id(poly), point)]

    h_poly, h_blind = None, 0
    for piece, b in zip(reversed(pieces), reversed(h_blinds)):
        h_poly = B.mul_add(h_poly, xn, piece)
        h_blind = (h_blind * xn + b) % p
    x_next, x_inv, x_last = rot(x, 1), rot(x, -1), rot(x, -(bf + 1))
    # nothing below feeds the transcript back into x: all openings are computed up front, point by point
    want = [(polys_of[kind][c], rot(x, r)) for kind in (INSTANCE, ADVICE, FIXED) for c, r in cs.queries[kind]]
    want += [(random_poly, x), (h_poly, x)] + [(sp, x) for sp in pk.sigma_polys]
    for i, S in enumerate(perm_sets):
        want += [(S["poly"], x), (S["poly"], x_next)] + ([(S["poly"], x_last)] if i + 1 < len(perm_sets) else [])
    for L in lookups:
        want += [(L["z_poly"], x), (L["z_poly"], x_next), (L["pi_poly"], x), (L["pi_poly"], x_inv), (L["pt_poly"], x)]
    by_point = {}
    for poly, pt_ in want:
        if (id(poly), pt_) not in cache:
            cache[(id(poly), pt_)] = None
            by_point.setdefault(pt_, []).append(poly)
    for pt_, polys_ in by_point.items():
        for poly, val in zip(polys_, B.eval_polynomials_at(polys_, pt_)):
            cache[(id(poly), pt_)] = val
    for kind in (INSTANCE, ADVICE, FIXED):
        for c, r in cs.queries[kind]:
            transcript.write_scalar(ev(polys_of[kind][c], rot(x, r)))
    transcript.write_scalar(ev(random_poly, x))
    for sp in pk.sigma_polys:
        transcript.write_scalar(ev(sp, x))
    for i, S in enumerate(perm_sets):
        transcript.write_scalar(ev(S["poly"], x))
        transcript.write_scalar(ev(S["poly"], x_next))
        if i + 1 < len(perm_sets):
            transcript.write_scalar(ev(S["poly"], x_last))
    for L in lookups:
        for poly, pt_ in ((L["z_poly"], x), (L["z_poly"], x_next), (L["pi_poly"], x), (L["pi_poly"], x_inv), (L["pt_poly"], x)):
            transcript.write_scalar(ev(poly, pt_))
    tick("evaluations")

    # ---- multiopen ---------------------------------------------------------------------------------------------------------------------
    qs: List[_Opening] = []
    for c, r in cs.queries[INSTANCE]:
        qs.append(_Opening(inst_polys[c], 1, rot(x, r)))
    for c, r in cs.queries[ADVICE]:
        qs.append(_Opening(adv_polys[c], adv_blinds[c], rot(x, r)))
    for S in perm_sets:
        qs.append(_Opening(S["poly"], S["blind"], x))
        qs.append(_Opening(S["poly"], S["blind"], x_next))
    for S in list(reversed(perm_sets))[1:]:
        qs.append(_Opening(S["poly"], S["blind"], x_last))
    for L in lookups:
        qs.append(_Opening(L["z_poly"], L["z_blind"], x))
        qs.append(_Opening(L["pi_poly"], L["pi_blind"], x))
        qs.append(_Opening(L["pt_poly"], L["pt_blind"], x))
        qs.append(_Opening(L["pi_poly"], L["pi_blind"], x_inv))
        qs.append(_Opening(L["z_poly"], L["z_blind"], x_next))
    for c, r in cs.queries[FIXED]:
        qs.append(_Opening(pk.fixed_polys[c], 1, rot(x, r)))
    for sp in pk.sigma_polys:
        qs.append(_Opening(sp, 1, x))
    qs.append(_Opening(h_poly, h_blind, x))
    qs.append(_Opening(random_poly, random_blind, x))
    for q in qs:
        q.eval = ev(q.poly, q.point)

    x_1 = transcript.squeeze_challenge_scalar()
    x_2 = transcript.squeeze_challenge_scalar()
    cmap, point_sets = construct_intermediate_sets(qs, lambda q: (id(q.poly), q.blind), lambda q: q.point, lambda q: q.eval)
    ns = len(point_sets)
    q_blinds = [0] * ns
    q_eval_sets = [[0] * len(ps) for ps in point_sets]
    members = [[] for _ in range(ns)]
    for cd in cmap:
        s, o = cd["set_index"], cd["commitment"]
        members[s].append(o.poly)
        q_blinds[s] = (q_blinds[s] * x_1 + o.blind) % p
        q_eval_sets[s] = [(a * x_1 + e) % p for a, e in zip(q_eval_sets[s], cd["evals"])]
    # q_polys[s] = sum_j x_1^(r - 1 - j) * member_j: halo2's Horner fold over the set's members, in one pass over the inputs
    q_polys = [B.linear_combination(polys_, [pow(x_1, len(polys_) - 1 - j, p) for j in range(len(polys_))]) for polys_ in members]
    q_prime = None
    for points, evals, poly in zip(point_sets, q_eval_sets, q_polys):
        cur = B.sub_low(poly, lagrange_interpolate(points, evals, p))
        for pt_ in points:
            cur = B.kate_division(cur, pt_)
        q_prime = B.mul_add(q_prime, x_2, cur)
    q_prime_blind = rand()
    transcript.write_point(B.commit(q_prime, q_prime_blind))
    x_3 = transcript.squeeze_challenge_scalar()
    for qp in q_polys:
        transcript.write_scalar(B.eval_polynomial(qp, x_3))
    x_4 = transcript.squeeze_challenge_scalar()
    p_poly, p_blind = q_prime, q_prime_blind
    for qp, qb in zip(q_polys, q_blinds):
        p_poly = B.mul_add(p_poly, x_4, qp)
        p_blind = (p_blind * x_4 + qb) % p
    tick("multiopen")
    B.ipa_create_proof(rand, transcript, p_poly, p_blind, x_3)
    tick("ipa")
    B.end_proof()
    return transcript.finalize()


# ---- the product backend: libtrp.so, device resident ----------------------------------------------------------------------------------
class GpuBackend:
    """Backend of keygen / create_proof over the CUDA library.  Every polynomial is a torch int64 tensor (n, 4) of Montgomery
    limbs in HBM and every operation is a trp_dev_* entry point of include/tr_prover.h; the host sees scalars and points only.
    The quotient is evaluated coset by coset from coefficient form (j - 1 cosets, trp_dev_cosets_to_coeff), so no
    extended-domain column is ever materialised.  No CPU fallback: constructing it without a GPU raises TrpError."""
    leaves_are_coefficients = True                # coeff_to_extended keeps coefficient form (cosets are expanded in the quotient)

    def __init__(self, ctx, k: int, cs_degree: int, params=None):
        import ctypes
        import os
        import numpy as np
        import torch
        from . import ipa as _ipa, permutation as _perm
        from .commitment import Params
        from .domain import EvaluationDomain
        self.np, self.torch, self.ct, self._ipa = np, torch, ctypes, _ipa
        self.ctx, self.lib, self.k, self.n, self.j = ctx, ctx.lib, k, 1 << k, cs_degree
        self.p = _perm._MODULUS[ctx.curve]
        self.q = _perm._MODULUS[1 - ctx.curve]
        self.R, self.Rq = (1 << 256) % self.p, (1 << 256) % self.q
        self.Rinv, self.Rqinv = pow(self.R, -1, self.p), pow(self.Rq, -1, self.q)
        # ONE stream for torch's kernels, the library's kernels and NCCL: the ctx is pointed at a torch stream that is made this
        # thread's current stream, so everything the prover enqueues is ordered by the stream itself: a hand-over between torch
        # and the library needs no fence, and the host only waits when it reads a result (.cpu()).  (Round 1 kept the library on
        # its own non-blocking stream and fenced every call with a device-wide synchronize: ~3 000 fences per proof at k = 20.)
        self.stream = ctx.bind_torch_stream()                  # one per process and device, shared by every backend and ctx
        self.params = params if params is not None else Params.new(ctx, k)
        self.dom = EvaluationDomain(ctx, cs_degree, k)
        self.extended_k = self.dom.extended_k
        self.omega = self._ints(self.dom.omega.reshape(1, 4))[0]
        self.omega_inv = pow(self.omega, -1, self.p)
        self.delta = pow(5, 1 << 32, self.p)
        self.ipa_params = _ipa.IpaParams(ctx, k, self.params.g_points, self.params.w, self.params.u)
        # a second, NARROW window table over g_lagrange ++ [w] for columns that are mostly zero (TinyRAM's instance / advice /
        # permuted lookup columns use 2^16 of the 2^20 rows): what is left of such an MSM is the bucket reduction, whose cost is
        # the 2^(c-1) buckets (profiles/msm_variants_r02.md: c = 13 2.17 ms per 8 columns against 3.3 ms at the dense c = 17)
        self._gl_sparse = None
        if k >= 18:
            from .arithmetic import Bases
            self._gl_sparse = Bases(ctx, np.concatenate([self.params.g_lagrange_points, self.params.w.reshape(1, 8)]), 13 << 8)
        # a third table over Q ++ [w], Q_j = g_lagrange_0 + ... + g_lagrange_j (trp_dev_points_prefix_sum): summation by parts,
        #     sum_i z_i G_i = sum_j (z_j - z_{j+1}) Q_j   (z_n = 0),
        # commits a column through its DIFFERENCES, which are sparse whenever the column rarely changes from row to row.  halo2's
        # grand-product columns do exactly that: on the rows a circuit leaves unused every factor of the permutation / lookup
        # product is 1, so Z is dense in value but constant over 15/16 of TinyRAM's rows (and some permuted lookup columns hold a
        # non-zero default there).  Same group element, same proof bytes; 78 of the 86 dense MSMs of a proof become sparse ones.
        self._gl_prefix = None
        if os.environ.get("TRP_COMMIT_BY_PARTS", "1") != "0":
            from .arithmetic import Bases
            d_q = self.torch.from_numpy(np.ascontiguousarray(self.params.g_lagrange_points).view(np.int64)).cuda()
            self.ctx.check(self.lib.trp_dev_points_prefix_sum(self.ctx.handle, d_q.data_ptr(), self.n, d_q.data_ptr()))
            q_host = d_q.cpu().numpy().view(np.uint64).reshape(self.n, 8)
            self._gl_prefix = Bases(ctx, np.concatenate([q_host, self.params.w.reshape(1, 8)]), (13 << 8) if k >= 18 else 0)
            del d_q
        self.ev = P.new_evaluator(ctx)
        self._static, self._static_keep = {}, []
        self.static_budget_bytes = 48 << 30
        self._arena, self._arena_used, self._arena_slot, self._arena_on, self._coset_buf = None, 0, {}, False, None

    def close(self):
        """release the library-side handles (MSM tables of the opening, the domain); torch tensors follow Python's lifetime"""
        if getattr(self, "ipa_params", None) is not None:
            self.ipa_params.free(); self.ipa_params = None
        if getattr(self, "dom", None) is not None:
            self.dom.free(); self.dom = None
        self._static.clear(); self._static_keep.clear()
        self._arena, self._arena_slot, self._arena_on, self._coset_buf = None, {}, False, None

    # -- conversions between canonical ints and Montgomery limb arrays (host side: scalars, points, short lists)
    def _limbs(self, vals, mod=None, R=None):
        np = self.np
        mod, R = mod or self.p, R or self.R
        buf = b"".join((v % mod * R % mod).to_bytes(32, "little") for v in vals)
        return np.frombuffer(buf, dtype=np.uint64).reshape(len(vals), 4).copy()

    def _ints(self, arr, mod=None, Rinv=None):
        mod, Rinv = mod or self.p, Rinv or self.Rinv
        raw = self.np.ascontiguousarray(arr, dtype=self.np.uint64).reshape(-1, 4).tobytes()
        return [int.from_bytes(raw[i:i + 32], "little") * Rinv % mod for i in range(0, len(raw), 32)]

    def _m(self, v):                      # one scalar -> host limbs pointer argument
        from ._lib import ptr
        return ptr(self._limbs([v])[0])

    def _dev(self, limbs):
        return self.torch.from_numpy(self.np.ascontiguousarray(limbs).view(self.np.int64)).cuda()

    def _new(self, rows=None, zero=False):
        f = self.torch.zeros if zero else self.torch.empty
        return f((self.n if rows is None else rows, 4), dtype=self.torch.int64, device="cuda")

    def _wait(self):
        self.stream.synchronize()

    def _point(self, d_jac):
        jac = d_jac.cpu().numpy().view(self.np.uint64).reshape(3, 4)
        if not jac[2].any():
            return None
        x, y = self._ints(jac[:2], self.q, self.Rqinv)
        return (x, y)

    def rotate_omega(self, x, rotation):
        return x * pow(self.omega if rotation >= 0 else self.omega_inv, abs(rotation), self.p) % self.p

    # -- vectors
    def vec(self, values):
        if hasattr(values, "data_ptr"):
            if tuple(values.shape) != (self.n, 4) or values.dtype != self.torch.int64 or not values.is_cuda:
                raise ValueError("device columns must be (n, 4) int64 cuda tensors of Montgomery limbs")
            return values
        if len(values) > self.n:
            raise ValueError("column longer than the domain")
        v = self._new(zero=True)
        if len(values):
            v[:len(values)] = self._dev(self._limbs(values))
        return v

    def set_rows(self, v, start, values):
        if len(values):
            v[start:start + len(values)] = self._dev(self._limbs(values))
        return v

    def set_rows_many(self, vs, start, values):
        """vs[i][start : start + len(values[i])] = values[i] with ONE host -> device copy"""
        flat = [x for vals in values for x in vals]
        if not flat:
            return
        d = self._dev(self._limbs(flat))
        off = 0
        for v, vals in zip(vs, values):
            if vals:
                v[start:start + len(vals)] = d[off:off + len(vals)]
                off += len(vals)

    def random_vec(self, rand):
        key = getattr(rand, "bulk_key", None)          # optional: 32 bytes of the caller's RNG, expanded on the device
        if key is not None:
            out = self._new()
            self.ctx.check(self.lib.trp_dev_random_field(self.ctx.handle, 0, key(), 0, self.n, out.data_ptr()))
            return out
        bulk = getattr(rand, "vector", None)           # optional bulk draw: (n, 4) Montgomery limbs
        return self._dev(bulk(self.n)) if bulk else self._dev(self._limbs([rand() for _ in range(self.n)]))

    def mul_add(self, acc, s, v):
        if acc is None:
            return v.clone()
        out = self._new()
        d_s = self._dev(self._limbs([s]))
        self.ctx.check(self.lib.trp_dev_field_op(self.ctx.handle, 0, 2 | 16, acc.data_ptr(), d_s.data_ptr(), out.data_ptr(), self.n))
        self.ctx.check(self.lib.trp_dev_field_op(self.ctx.handle, 0, 0, out.data_ptr(), v.data_ptr(), out.data_ptr(), self.n))
        return out

    def sub_low(self, v, low):
        out = v.clone()
        cur = self._ints(out[:len(low)].cpu().numpy().view(self.np.uint64))
        return self.set_rows(out, 0, [(c - r) % self.p for c, r in zip(cur, low)])

    def sigma_vecs(self, m, moved):
        base = self._new()
        self.ctx.check(self.lib.trp_dev_powers(self.ctx.handle, 0, self._m(self.omega), self.n, base.data_ptr()))
        out, dl = [], 1
        for i in range(m):
            v = self._new()
            d_s = self._dev(self._limbs([dl]))
            self.ctx.check(self.lib.trp_dev_field_op(self.ctx.handle, 0, 2 | 16, base.data_ptr(), d_s.data_ptr(), v.data_ptr(), self.n))
            out.append(v)
            dl = dl * self.delta % self.p
        if moved:                                      # patch the cells the copy constraints move: one scatter per column
            top = max(j2 for _, (_, j2) in moved.items())
            om = [1] * (top + 1)
            for j in range(1, top + 1):
                om[j] = om[j - 1] * self.omega % self.p
            dls = [pow(self.delta, i, self.p) for i in range(m)]
            per_col = {}
            for (i, j), (i2, j2) in moved.items():
                per_col.setdefault(i, ([], []))
                per_col[i][0].append(j); per_col[i][1].append(dls[i2] * om[j2] % self.p)
            for i, (rws, vals) in per_col.items():
                idx = self.torch.tensor(rws, dtype=self.torch.int64, device="cuda")
                out[i][idx] = self._dev(self._limbs(vals))
        return out

    def sigma_swap_blocks(self, sigmas, blocks):
        """blocks: (column, row0, column', row0', rows) 2-cycles left <-> right that no other constraint touches: the two row
        ranges exchange their identity labels delta^column * omega^row (device copies, nothing per cell on the host)"""
        if not blocks:
            return sigmas
        base = self._new()
        self.ctx.check(self.lib.trp_dev_powers(self.ctx.handle, 0, self._m(self.omega), self.n, base.data_ptr()))
        scal = {}
        for (i, r, i2, r2, rows) in blocks:
            for (dst, d0, src, s0) in ((i, r, i2, r2), (i2, r2, i, r)):
                if src not in scal:
                    scal[src] = self._dev(self._limbs([pow(self.delta, src, self.p)]))
                self.ctx.check(self.lib.trp_dev_field_op(self.ctx.handle, 0, 2 | 16, base[s0:s0 + rows].data_ptr(), scal[src].data_ptr(),
                                                         sigmas[dst][d0:d0 + rows].data_ptr(), rows))
        return sigmas

    # -- commitments and transforms
    def _commit(self, bases, v, blind):
        t = self.torch
        stage = t.cat([v, self._dev(self._limbs([blind]))])
        out = t.zeros(12, dtype=t.int64, device="cuda")
        self.ctx.check(self.lib.trp_dev_msm_batch(self.ctx.handle, bases.handle, stage.data_ptr(), self.n + 1, 1, out.data_ptr()))
        return self._point(out)

    def commit_lagrange(self, v, blind): return self._commit(self.params.g_lagrange, v, blind)
    def commit(self, v, blind): return self._commit(self.params.g, v, blind)

    def _commit_many(self, bases, vecs, blinds, batch=32, sparse=False, runs=False):
        """several commitments over the same bases as batched MSMs (trp_dev_msm_batch processes the columns concurrently).
        sparse: the caller expects mostly-zero columns; batches whose non-zero rows are below 10 % go to the narrow table.
        runs: the caller expects columns that rarely change from row to row (grand products over a partly used circuit): the
        batch is committed by parts -- its row-to-row differences over the prefix sums of the bases -- if those are below 10 %."""
        t, n, results = self.torch, self.n, []
        if len(vecs) > batch:                        # equal batches (33 columns: 17 + 16, not 32 + 1)
            nb = -(-len(vecs) // batch)
            batch = -(-len(vecs) // nb)
        for b0 in range(0, len(vecs), batch):
            vs, bs = vecs[b0:b0 + batch], blinds[b0:b0 + batch]
            stage = t.empty((len(vs), n + 1, 4), dtype=t.int64, device="cuda")
            for i, v in enumerate(vs):
                stage[i, :n] = v
            stage[:, n] = self._dev(self._limbs(bs))
            use = bases
            if sparse and self._gl_sparse is not None and bases is self.params.g_lagrange:
                if int((stage != 0).any(dim=-1).sum()) * 10 <= len(vs) * n:
                    use = self._gl_sparse
            if runs and use is bases and self._gl_prefix is not None and bases is self.params.g_lagrange:
                # e_j = z_j - z_{j+1} (j < n - 1), e_{n-1} = z_{n-1}; the blind keeps its own base w
                diff = t.empty_like(stage)
                flat_in, flat_out = stage.view(-1, 4), diff.view(-1, 4)
                self.ctx.check(self.lib.trp_dev_field_op(self.ctx.handle, 0, 1, flat_in.data_ptr(), flat_in[1:].data_ptr(), flat_out.data_ptr(),
                                                         flat_in.shape[0] - 1))
                diff[:, n - 1:] = stage[:, n - 1:]
                if int((diff != 0).any(dim=-1).sum()) * 10 <= len(vs) * n:
                    use, stage = self._gl_prefix, diff
            res = t.zeros((len(vs), 12), dtype=t.int64, device="cuda")
            self.ctx.check(self.lib.trp_dev_msm_batch(self.ctx.handle, use.handle, stage.data_ptr(), n + 1, len(vs), res.data_ptr()))
            results.append(res)
        out = []
        if results:                                  # ONE device -> host read for the whole call
            jac = t.cat(results).cpu().numpy().view(self.np.uint64).reshape(-1, 3, 4)
            for j in jac:
                out.append(None if not j[2].any() else tuple(self._ints(j[:2], self.q, self.Rqinv)))
        return out

    def commit_lagrange_many(self, vecs, blinds, sparse=False, runs=False):
        return self._commit_many(self.params.g_lagrange, vecs, blinds, sparse=sparse, runs=runs)
    def commit_many(self, vecs, blinds): return self._commit_many(self.params.g, vecs, blinds)

    # -- the verifier's three extras (verifier.py): the fixed points, the challenges' s vector, a variable-base MSM
    def fixed_points(self):
        pt = lambda arr: tuple(self._ints(self.np.asarray(arr, dtype=self.np.uint64).reshape(-1, 8)[0].reshape(2, 4), self.q, self.Rqinv))
        return pt(self.params.g_points), pt(self.params.w), pt(self.params.u)

    def ipa_s_vector(self, us, init=1):
        """commitment::compute_s on the device: s[0] = init, then one broadcast multiplication per round doubles the filled
        prefix (s[len .. 2 len) = s[0 .. len) * u_j, last round first)"""
        s = self._new(zero=True)
        s[:1] = self._dev(self._limbs([init]))
        filled = 1
        for u_j in reversed(us):
            d_u = self._dev(self._limbs([u_j]))
            self.ctx.check(self.lib.trp_dev_field_op(self.ctx.handle, 0, 2 | 16, s[:filled].data_ptr(), d_u.data_ptr(),
                                                     s[filled:2 * filled].data_ptr(), filled))
            filled *= 2
        if filled != self.n:
            raise ValueError("one challenge per round: len(us) must equal k")
        return s

    def msm_points(self, scalars, points):
        """sum_i scalars[i] * points[i] over caller-supplied affine points (trp_dev_msm_var: no table, one bucket set per window)"""
        t = self.torch
        if not scalars:
            return None
        d_pts = self._dev(self._limbs([c for pt in points for c in pt], self.q, self.Rq).reshape(len(points), 8))
        d_sc = self._dev(self._limbs(scalars))
        out = t.zeros(12, dtype=t.int64, device="cuda")
        self.ctx.check(self.lib.trp_dev_msm_var(self.ctx.handle, d_pts.data_ptr(), d_sc.data_ptr(), len(scalars), 1, out.data_ptr()))
        return self._point(out)

    # -- per-proof polynomial arena: create_proof announces how many polynomials it will bring to coefficient form; they are then
    #    laid out in ONE (count, n, 4) block, which the quotient's batched coset NTT reads in place (no 15.5 GiB staging copy at
    #    k = 20).  Polynomials made outside a proof (keygen) never come from the arena.
    def begin_proof(self, n_polys):
        t = self.torch
        n_polys += self._arena_padding()
        if self._arena is None or self._arena.shape[0] < n_polys:
            self._arena = None
            self._arena = t.empty((n_polys, self.n, 4), dtype=t.int64, device="cuda")
        self._arena_used, self._arena_slot, self._arena_on = 0, {}, True

    def end_proof(self):
        self._arena_on = False            # the views handed out stay valid until the next begin_proof

    def _arena_padding(self):
        return 0

    def lagrange_to_coeff(self, v):
        if self._arena_on and self._arena_used < self._arena.shape[0]:
            c = self._arena[self._arena_used]
            self._arena_slot[id(c)] = (self._arena_used, c)      # the view is kept alive: id() must stay unique
            self._arena_used += 1
            c.copy_(v)
        else:
            c = v.clone()
        self.ctx.check(self.lib.trp_dev_lagrange_to_coeff(self.dom.handle, c.data_ptr(), 1))
        return c

    def lagrange_to_coeff_many(self, vs):
        """the same for a batch: inside a proof the results are consecutive arena slots, transformed by ONE batched iNTT"""
        k = len(vs)
        if not (self._arena_on and k and self._arena_used + k <= self._arena.shape[0]):
            return [self.lagrange_to_coeff(v) for v in vs]
        first = self._arena_used
        out = []
        for v in vs:
            c = self._arena[self._arena_used]
            self._arena_slot[id(c)] = (self._arena_used, c)
            self._arena_used += 1
            c.copy_(v)
            out.append(c)
        self.ctx.check(self.lib.trp_dev_lagrange_to_coeff(self.dom.handle, self._arena[first].data_ptr(), k))
        return out

    def coeff_to_extended(self, c):
        return c                          # lazy: the quotient evaluates cosets straight from coefficient form

    def coeff_to_extended_static(self, c):
        """key material (fixed / sigma / Lagrange-selector polynomials): its evaluations on the j - 1 cosets are computed once
        and kept in HBM ((j - 1) * 32 B per row), so a proof only transforms its own columns"""
        ncos = self.j - 1
        held = sum(v.numel() for v in self._static.values()) * 8
        if held + ncos * self.n * 32 > self.static_budget_bytes:
            return c
        vals = self.torch.empty((ncos, self.n, 4), dtype=self.torch.int64, device="cuda")
        for cs in range(ncos):
            self.ctx.check(self.lib.trp_dev_coeff_to_coset(self.dom.handle, c.data_ptr(), vals[cs].data_ptr(), 1, cs))
        self._static[id(c)] = vals
        self._static_keep.append(c)       # id() stays unique while the tensor is alive
        return c

    def _run_program(self, ast, columns, out, coset):
        from ._lib import Q_CONTIGUOUS
        prog = P.compile_ast(ast, self.p)
        self.ev.evaluate_device(prog, self.dom, [c.data_ptr() for c in columns], out.data_ptr(), coset=coset | Q_CONTIGUOUS)

    def quotient_program(self, pk, build_h, challenges, n_perm_columns):
        """The compiled quotient program of `pk` with this proof's challenges patched in, or None (then the caller builds and
        compiles the Ast as usual).  The program's CODE depends on the constraint system only; its constants are literals of the
        gates or one of theta, beta, gamma, y, beta * DELTA^i.  The first proof of a key compiles the Ast twice -- with the real
        challenges and with a probe set -- and explains every constant slot by exactly one of those formulas; later proofs
        evaluate the formulas (microseconds) instead of rebuilding and recompiling the Ast (~60 ms of Python at 8 000
        instructions, during which the GPU would idle: the challenge y is the last thing the transcript yields before the
        quotient).  Any slot that cannot be explained disables the cache for that key."""
        return GpuBackend._cached_program(self, pk, id(self), build_h, challenges, n_perm_columns)   # self may be another backend (tests)

    def quotient_part_programs(self, pk, build_parts, challenges, n_perm_columns):
        """[(ncos, Program, leaf keys)] of create_proof's build_parts: one program per constraint degree, each cached like the
        whole one (a part's constants may also be powers of y); a part the cache cannot explain is compiled afresh"""
        built = {}

        def parts_at(ch):
            if ch not in built:
                built[ch] = build_parts(*ch)
            return built[ch]

        cache = pk.__dict__.setdefault("_quotient_program", {})
        shape = cache.get((id(self), "parts"))
        if shape is None:                         # the degrees depend on the constraint system only
            shape = cache[(id(self), "parts")] = [ncos for ncos, _, _ in parts_at(tuple(challenges))]
        out = []
        for i, ncos in enumerate(shape):
            got = self._cached_program(pk, (id(self), "part", i), lambda *ch, i=i: parts_at(ch)[i][1:], challenges, n_perm_columns)
            if got is None:
                return [(q, P.compile_ast(ast, self.p), keys) for q, ast, keys in parts_at(tuple(challenges))]
            out.append((ncos, got[0], got[1]))
        return out

    def _cached_program(self, pk, cache_key, build, challenges, n_perm_columns):
        p = self.p
        cache = pk.__dict__.setdefault("_quotient_program", {})
        entry = cache.get(cache_key)
        if entry is None:
            real = tuple(c % p for c in challenges)
            probe = tuple((c * 0x9e3779b97f4a7c15 + 0x632be59bd9b4e019 + i) % p for i, c in enumerate(real))
            ast_r, keys_r = build(*real)
            ast_p, keys_p = build(*probe)
            prog_r, prog_p = P.compile_ast(ast_r, p), P.compile_ast(ast_p, p)
            entry = False
            if keys_r == keys_p and prog_r.code.shape == prog_p.code.shape and (prog_r.code == prog_p.code).all() and len(prog_r.consts) == len(prog_p.consts):
                def formulas(ch, max_gap):
                    theta, beta, gamma, y = ch
                    f = {("theta",): theta, ("beta",): beta, ("gamma",): gamma, ("y",): y}
                    d = beta
                    for i in range(n_perm_columns):
                        f[("beta_delta", i)] = d
                        d = d * self.delta % p
                    yp = y
                    for e in range(2, max_gap + 1):             # split_by_degree's y^gap between the terms of a part
                        yp = yp * y % p
                        f[("y_pow", e)] = yp
                    return f
                fr, fp = formulas(real, 1024), formulas(probe, 1024)
                by_value = {}
                for name in fr:
                    by_value.setdefault((fr[name], fp[name]), name)
                slots = []
                for vr, vp in zip(prog_r.consts, prog_p.consts):
                    if vr == vp:
                        slots.append(None)                      # a literal of the constraint system
                        continue
                    name = by_value.get((vr, vp))
                    if name is None:
                        slots = None
                        break
                    slots.append(name)
                if slots is not None:
                    max_gap = max([name[1] for name in slots if name is not None and name[0] == "y_pow"], default=1)
                    entry = (prog_r, keys_r, slots, formulas, max_gap)
            cache[cache_key] = entry
            if entry:
                return entry[0], entry[1]
            return None
        if entry is False:
            return None
        prog, keys, slots, formulas, max_gap = entry
        f = formulas(tuple(c % p for c in challenges), max_gap)
        consts = [v if name is None else f[name] for v, name in zip(prog.consts, slots)]
        return P.Program(prog.code, consts, prog.n_regs, prog.n_cols), keys

    def quotient_pieces(self, pk, challenges, build_h, build_parts, resolve):
        """one program per constraint degree, each evaluated on the cosets its degree needs"""
        parts = self.quotient_part_programs(pk, build_parts, challenges, len(pk.vk.cs.permutation))
        return self.quotient_parts([(ncos, prog, [resolve(k_) for k_ in keys]) for ncos, prog, keys in parts])

    def quotient_parts(self, parts):
        """h(X) from the numerator given by parts [(ncos, Program, leaf polynomials)]: part p is evaluated on cosets 0 .. ncos - 1
        only, and coset c expands only the coefficient columns that the parts evaluated there read (one gathered batch of NTTs;
        key material comes from its precomputed cosets).  Columns are numbered by the last coset that needs them, so coset c's
        columns are a prefix of coset 0's and keep their slot.  Returns the j - 1 pieces of h (n coefficients each)."""
        from ._lib import Q_CONTIGUOUS
        t, n, ncos_out = self.torch, self.n, self.j - 1
        last = {}                                  # id -> (last coset + 1, polynomial) of every column transformed here
        for ncos, _, polys in parts:
            for c in polys:
                if id(c) not in self._static and last.get(id(c), (0,))[0] < ncos:
                    last[id(c)] = (ncos, c)
        order = sorted(last.values(), key=lambda e: -e[0])                # stable: first-use order within a coset count
        slot = {id(c): s_ for s_, (_, c) in enumerate(order)}
        count = [sum(1 for q, _ in order if q > cs) for cs in range(ncos_out)]
        tab = t.tensor([c.data_ptr() for _, c in order] or [0], dtype=t.int64).cuda()
        if self._coset_buf is None or self._coset_buf.shape[0] < len(order):   # kept across proofs: a fresh 15.5 GiB block per proof
            self._coset_buf = None                                              # costs the caching allocator 0.1 s every other proof
            self._coset_buf = t.empty((max(len(order), 1), n, 4), dtype=t.int64, device="cuda")
        buf = self._coset_buf
        row = [0]
        for ncos, _, _ in parts:
            row.append(row[-1] + ncos)
        vals = t.empty((row[-1], n, 4), dtype=t.int64, device="cuda")
        for cs in range(ncos_out):
            if count[cs]:
                self.ctx.check(self.lib.trp_dev_coeff_to_coset_gather(self.dom.handle, tab.data_ptr(), buf.data_ptr(), count[cs], cs))
            for pi, (ncos, prog, polys) in enumerate(parts):
                if cs < ncos:
                    ptrs = [buf[slot[id(c)]].data_ptr() if id(c) in slot else self._static[id(c)][cs].data_ptr() for c in polys]
                    self.ev.evaluate_device(prog, self.dom, ptrs, vals[row[pi] + cs].data_ptr(), coset=cs | Q_CONTIGUOUS)
        h = t.empty((ncos_out, n, 4), dtype=t.int64, device="cuda")
        qs = (self.ct.c_uint * len(parts))(*[ncos for ncos, _, _ in parts])
        self.ctx.check(self.lib.trp_dev_cosets_to_coeff_parts(self.dom.handle, vals.data_ptr(), qs, len(parts), ncos_out, h.data_ptr(), 1))
        return [h[i] for i in range(ncos_out)]

    def eval_polynomial(self, v, x):
        out = self._new(1)
        self.ctx.check(self.lib.trp_dev_eval_polynomials(self.ctx.handle, 0, v.data_ptr(), self.n, self.n, 1, self._m(x), out.data_ptr()))
        return self._ints(out.cpu().numpy().view(self.np.uint64))[0]

    def eval_polynomials_at(self, vs, x):
        """the values of many separately allocated polynomials at ONE point: one library call (trp_dev_eval_polynomials_at)"""
        if not vs:
            return []
        out = self._new(len(vs))
        tab = (self.ct.c_void_p * len(vs))(*[v.data_ptr() for v in vs])
        self.ctx.check(self.lib.trp_dev_eval_polynomials_at(self.ctx.handle, 0, tab, self.n, len(vs), self._m(x), out.data_ptr()))
        return self._ints(out.cpu().numpy().view(self.np.uint64))

    def linear_combination(self, vs, scalars):
        """sum_j scalars[j] * vs[j] in one pass (trp_dev_linear_combination)"""
        out = self._new()
        tab = (self.ct.c_void_p * len(vs))(*[v.data_ptr() for v in vs])
        sc = self._limbs(scalars)
        from ._lib import ptr
        self.ctx.check(self.lib.trp_dev_linear_combination(self.ctx.handle, 0, tab, ptr(sc), self.n, len(vs), out.data_ptr()))
        return out

    def kate_division(self, v, b):
        q = self._new(zero=True)
        self.ctx.check(self.lib.trp_dev_kate_division(self.ctx.handle, 0, v.data_ptr(), self.n, self._m(b), q.data_ptr()))
        return q

    # -- lookups and permutation
    def compress(self, exprs, theta, values_of):
        leaves, cols = {}, []

        def to_ast(e):
            if isinstance(e, Constant): return P.ConstantTerm(e.value % self.p)
            if isinstance(e, Query):
                key = (e.kind, e.column)
                if key not in leaves:
                    leaves[key] = len(cols); cols.append(values_of[e.kind][e.column])
                return P.Poly(leaves[key], e.rotation)
            if isinstance(e, Negated): return -to_ast(e.a)
            if isinstance(e, Sum): return to_ast(e.a) + to_ast(e.b)
            if isinstance(e, Product): return to_ast(e.a) * to_ast(e.b)
            return to_ast(e.a) * (e.scalar % self.p)

        ast = P.ConstantTerm(0)
        for e in exprs:
            ast = ast * theta + to_ast(e)
        out = self._new()
        self._run_program(ast, cols, out, 0)          # coset 0, contiguous: rows = n, rotations step by one row
        return out

    def permute_expression_pair(self, inp, tab, usable_rows):
        from .lookup import ConstraintSystemFailure
        pa, ps = self._new(zero=True), self._new(zero=True)
        ok = self.ct.c_int(1)
        self.ctx.check(self.lib.trp_dev_permute_expression_pair(self.ctx.handle, inp.data_ptr(), tab.data_ptr(), usable_rows, pa.data_ptr(),
                                                                ps.data_ptr(), self.ct.byref(ok)))
        if not ok.value:
            raise ConstraintSystemFailure("lookup input value not present in the table")
        return pa, ps

    def permutation_commit(self, values, sigmas, beta, gamma, chunk_len, blinding_factors, rand, after_chunk):
        from ._lib import ptr
        n, p, ct = self.n, self.p, self.ct
        deltaomega, last, sets = 1, None, []
        for lo in range(0, len(values), chunk_len):
            cols = list(range(lo, min(lo + chunk_len, len(values))))
            dbeta = self._limbs([deltaomega * pow(self.delta, c - lo, p) % p * beta % p for c in cols])
            deltaomega = deltaomega * pow(self.delta, len(cols), p) % p
            vptr = (ct.c_void_p * len(cols))(*[values[c].data_ptr() for c in cols])
            sptr = (ct.c_void_p * len(cols))(*[sigmas[c].data_ptr() for c in cols])
            z = self._new()
            self.ctx.check(self.lib.trp_dev_permutation_product(self.dom.handle, vptr, sptr, len(cols), self._m(beta), self._m(gamma), ptr(dbeta),
                                                                None if last is None else last[n - (blinding_factors + 1)].data_ptr(), z.data_ptr()))
            self.set_rows(z, n - blinding_factors, [rand() for _ in range(blinding_factors)])
            last = z
            sets.append(z)
            after_chunk(z)
        return sets

    def lookup_product(self, ci, ct_, pi, pt, beta, gamma, blinding_factors, rand):
        z = self._new()
        self.ctx.check(self.lib.trp_dev_lookup_product(self.dom.handle, ci.data_ptr(), ct_.data_ptr(), pi.data_ptr(), pt.data_ptr(), self._m(beta),
                                                       self._m(gamma), z.data_ptr(), self.n - blinding_factors))
        return self.set_rows(z, self.n - blinding_factors, [rand() for _ in range(blinding_factors)])

    def lookups_commit_permuted(self, lookups, theta, values_of, usable, bf, rand):
        out = []
        for inputs, tables in lookups:
            ci, ct_ = self.compress(inputs, theta, values_of), self.compress(tables, theta, values_of)
            pi, pt = self.permute_expression_pair(ci, ct_, usable)
            self.set_rows(pi, usable, [rand() for _ in range(bf + 1)])
            self.set_rows(pt, usable, [rand() for _ in range(bf + 1)])
            out.append({"ci": ci, "ct": ct_, "pi": pi, "pt": pt, "pi_blind": rand(), "pt_blind": rand()})
        return out

    def lookup_products(self, lookups, beta, gamma, bf, rand):
        for L in lookups:
            L["z"] = self.lookup_product(L["ci"], L["ct"], L["pi"], L["pt"], beta, gamma, bf, rand)
            L["z_blind"] = rand()

    def ipa_create_proof(self, rand, transcript, p_poly, p_blind, x_3):
        outer = self

        class _Adapter:
            def write_point(self, limbs):
                x, y = outer._ints(outer.np.asarray(limbs, dtype=outer.np.uint64).reshape(2, 4), outer.q, outer.Rqinv)
                transcript.write_point(None if (x, y) == (0, 0) else (x, y))
            def write_scalar(self, s): transcript.write_scalar(s)
            def squeeze_challenge_scalar(self): return transcript.squeeze_challenge_scalar()

        bulk = (lambda n_: self.random_vec(rand)) if hasattr(rand, "bulk_key") else getattr(rand, "vector", None)
        self._ipa.create_proof(self.ipa_params, rand, _Adapter(), p_poly, p_blind, x_3, rand_vector=bulk, dist=self._ipa_dist())

    def _ipa_dist(self):
        return None                       # sharded_backend.ShardedGpuBackend divides the opening's rounds between its ranks
