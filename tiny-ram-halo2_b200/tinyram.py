"""The reference's TinyRamCircuit<WORD_BITS, REG_COUNT> restated over plonk.ConstraintSystem: the real gates, lookups, equality
columns and witness of the circuit whose create_proof this repo accelerates (SURVEY.md 8(f) row f4; BASELINE.json configs[0]).

configure  -- /root/reference/src/circuits/mod.rs:48-60: ProgConfig::configure (tables/prog.rs:139-161), ExeChip::configure
              (tables/exe.rs:535-790) with every gadget it instantiates, then the dynamic lookup of the execution table's
              (pc, program line) in the program table (tables/prog.rs:163-193).  Columns are allocated, and cells queried, in the
              reference's order, so column indices and query order are the reference's.
synthesize -- circuits/mod.rs:62-75: the three fixed tables (even_bits.rs:56-74, pow.rs:21-66, out_table.rs:133-215), the
              program region (prog.rs:195-233) and the execution region (exe.rs:792-1080), rows of both regions starting at 0
              (SimpleFloorPlanner: the regions use disjoint columns).  Unassigned cells are 0, as in the real prover.
program_instance -- tables/prog.rs:38-60.

What this mirror has to decide for itself (halo2 fork internals that are not in /root/reference):
  * selectors are one fixed column each (s_prog is never queried and s_table is complex, so halo2's selector compression leaves
    them alone; first_line is the only simple selector used in a gate);
  * lookup-table columns are fixed columns whose unused rows repeat row 0 (SimpleTableLayouter's default fill);
  * `Expression::SelectorExpression` (fork) is the identity;
  * the fork's dynamic table: one extra fixed "tag" column, 1 on the rows `add_row` marked; `lookup_dynamic` becomes the
    lookup  [sel, sel * e_1, ...] in [tag, col_1, ...]  -- UNVERIFIED against the fork, it is absent from this machine.
Two witness details where following the reference to the letter would make its own gates unsatisfiable are noted at the code
(`reg_operand_value`, `a_flag`)."""
from __future__ import annotations

from typing import Callable, Dict, List, Optional, Tuple

from . import trace as T

U64_MAX = (1 << 64) - 1
OUT_NAMES = ("and", "xor", "or", "sum", "prod", "ssum", "sprod", "mod", "shift", "flag1", "flag2", "flag3", "flag4")   # Out::new order

# OutPut::OUT per instruction (tables/aux/out.rs:157-348)
OUT = {
    "And": ("and", "flag1", "flag2"), "Or": ("or", "flag1", "flag2"), "Xor": ("xor", "flag1", "flag2"), "Not": ("xor", "flag1", "flag2"),
    "Add": ("sum",), "Sub": ("sum",), "Mull": ("prod", "flag1", "flag2"), "UMulh": ("prod", "flag1", "flag2"),
    "SMulh": ("sprod", "flag1", "flag2"), "UDiv": ("mod", "flag1", "flag2", "flag3"), "UMod": ("mod", "flag1", "flag2", "flag3"),
    "Shl": ("shift", "flag4"), "Shr": ("shift", "flag4"), "Cmpe": ("xor", "flag1", "flag2"), "Cmpa": ("sum",), "Cmpae": ("sum",),
    "Cmpg": ("ssum",), "Cmpge": ("ssum",), "Mov": ("xor",), "CMov": ("mod",), "Jmp": ("xor",), "CJmp": ("mod",), "CnJmp": ("mod",),
    "LoadW": (), "StoreW": ("xor",), "Answer": (),
}
# rows of the Out table, in assignment order (out_table.rs:137-213)
OUT_TABLE_ORDER = ("And", "Or", "Xor", "Not", "Add", "Sub", "Mull", "UMulh", "SMulh", "UDiv", "UMod", "Shl", "Shr", "Cmpe", "Cmpa",
                   "Cmpae", "Cmpg", "Cmpge", "Mov", "CMov", "Jmp", "CJmp", "CnJmp", "StoreW", "LoadW", "Answer")


def selections(ins: T.Instruction):
    """TempVarSelectorsRow::from(&Instruction) (tables/aux.rs:95-407): (a, b, c, d, changed registers, changed pc, changed flag)"""
    n, ri, rj, a = ins.name, ins.ri, ins.rj, ins.a
    A = ("A", a)
    if n in ("And", "Or", "Xor"):
        return A, ("Reg", rj), ("RegN", ri), ("Unset",), (ri,), False, True
    if n == "Not":
        return A, ("MaxWord",), ("RegN", ri), ("Unset",), (ri,), False, True
    if n == "Add":
        return A, ("Reg", rj), ("RegN", ri), ("Zero",), (ri,), False, True
    if n == "Sub":
        return A, ("RegN", ri), ("Reg", rj), ("Zero",), (ri,), False, True
    if n in ("Mull", "Shl"):
        return A, ("Reg", rj), ("NonDet",), ("RegN", ri), (ri,), False, True
    if n in ("UMulh", "SMulh", "Shr"):
        return A, ("Reg", rj), ("RegN", ri), ("NonDet",), (ri,), False, True
    if n == "UDiv":
        return ("NonDet",), ("RegN", ri), A, ("Reg", rj), (ri,), False, True
    if n == "UMod":
        return ("RegN", ri), ("NonDet",), A, ("Reg", rj), (ri,), False, True
    if n == "Cmpe":
        return A, ("Reg", ri), ("NonDet",), ("Unset",), (), False, True
    if n in ("Cmpa", "Cmpg"):
        return ("Reg", ri), ("NonDet",), A, ("Zero",), (), False, True
    if n in ("Cmpae", "Cmpge"):
        return ("Reg", ri), ("NonDet",), A, ("One",), (), False, True
    if n == "Mov":
        return A, ("RegN", ri), ("Zero",), ("Unset",), (ri,), False, False
    if n == "CMov":
        return ("RegN", ri), A, ("Zero",), ("Reg", ri), (ri,), False, False
    if n == "Jmp":
        return A, ("PcN",), ("Zero",), ("Unset",), (), True, False
    if n == "CJmp":
        return ("PcN",), A, ("Zero",), ("PcPlusOne",), (), True, False
    if n == "CnJmp":
        return ("PcN",), ("PcPlusOne",), ("Zero",), A, (), True, False
    if n == "LoadW":
        return ("VAddr",), ("Reg", ri), ("Zero",), ("Zero",), (ri,), False, False
    if n == "StoreW":
        return ("VAddr",), ("RegN", ri), ("Zero",), ("Zero",), (), False, False
    if n == "Answer":
        return A, ("Pc",), ("Zero",), ("Zero",), (), False, False
    raise ValueError(n)


class ProgramLine:
    """ProgramLine<W, R, C> (tables/prog.rs:21-26, 62-79): opcode, immediate and the 92 TempVarSelectors columns, allocated in
    the order of SelectorsA/B/C/D::new_columns (aux.rs:587-600, 724-740, 870-883, 995-1011) and ChangedSelectors::new
    (changed.rs:26-33)."""

    def __init__(self, new_col: Callable[[], int], R: int):
        regs = lambda: [new_col() for _ in range(R)]
        self.opcode, self.immediate = new_col(), new_col()
        self.a = {"pc_next": new_col(), "reg": regs(), "reg_next": regs(), "a": new_col(), "v_addr": new_col(), "non_det": new_col()}
        self.b = {"pc": new_col(), "pc_next": new_col(), "pc_plus_one": new_col(), "reg": regs(), "reg_next": regs(), "a": new_col(),
                  "non_det": new_col(), "max_word": new_col()}
        self.c = {"reg": regs(), "reg_next": regs(), "a": new_col(), "non_det": new_col(), "zero": new_col()}
        self.d = {"pc": new_col(), "reg": regs(), "reg_next": regs(), "a": new_col(), "non_det": new_col(), "zero": new_col(),
                  "one": new_col()}
        self.ch = {"regs": regs(), "pc": new_col(), "flag": new_col()}

    def to_vec(self) -> List[int]:
        """ProgramLine::to_vec = the order of ProgramLine::map (prog.rs:106-128); ChangedSelectors::map visits pc, flag, regs
        (changed.rs:73-81), everything else in allocation order"""
        if getattr(self, "_vec", None) is None:
            out = [self.opcode, self.immediate]
            for part in (self.a, self.b, self.c, self.d):
                for v in part.values():
                    out.extend(v if isinstance(v, list) else [v])
            self._vec = out + [self.ch["pc"], self.ch["flag"]] + self.ch["regs"]
        return list(self._vec)

    def row_values(self, ins: T.Instruction) -> Dict[int, int]:
        """ProgramLine::assign_cells for one line (prog.rs:81-104): {column: value}"""
        sa, sb, sc, sd, ch_regs, ch_pc, ch_flag = selections(ins)
        vals = {c: 0 for c in self.to_vec()}
        vals[self.opcode], vals[self.immediate] = ins.opcode, ins.immediate()

        def set_sel(part, s):                       # From<SelectionX> for SelectorsX<bool> (aux.rs:562-585, 742-768, 885-905, 1013-1041)
            kind = s[0]
            if kind == "A":
                if isinstance(s[1], T.Imm): vals[part["a"]] = 1
                else: vals[part["reg"][s[1].index]] = 1
            elif kind == "Reg": vals[part["reg"][s[1]]] = 1
            elif kind == "RegN": vals[part["reg_next"][s[1]]] = 1
            elif kind == "PcN": vals[part["pc_next"]] = 1
            elif kind == "Pc": vals[part["pc"]] = 1
            elif kind == "PcPlusOne":
                if "pc_plus_one" in part: vals[part["pc_plus_one"]] = 1
                else: vals[part["pc"]] = 1; vals[part["one"]] = 1           # SelectionD::PcPlusOne sets pc AND one
            elif kind == "VAddr": vals[part["v_addr"]] = 1
            elif kind == "NonDet": vals[part["non_det"]] = 1
            elif kind == "MaxWord": vals[part["max_word"]] = 1
            elif kind == "Zero": vals[part["zero"]] = 1
            elif kind == "One": vals[part["one"]] = 1
            elif kind != "Unset": raise ValueError(kind)

        for part, s in ((self.a, sa), (self.b, sb), (self.c, sc), (self.d, sd)):
            set_sel(part, s)
        for r in ch_regs:
            vals[self.ch["regs"][r]] = 1
        vals[self.ch["pc"]], vals[self.ch["flag"]] = int(ch_pc), int(ch_flag)
        return vals


class EvenBits:
    """EvenBitsConfig (tables/even_bits.rs:88-203): word column, its even / odd halves, the advice selectors that enable it"""
    def __init__(self, word, even, odd):
        self.word, self.even, self.odd = word, even, odd


class Signed:
    """SignedConfig (tables/signed.rs:12-21)"""
    def __init__(self, word: EvenBits, msb, word_sigma, check_sign: EvenBits):
        self.word, self.msb, self.word_sigma, self.check_sign = word, msb, word_sigma, check_sign


def even_bits_at(i: int) -> int:
    """even_bits.rs:219-231: spread the bits of i to the even positions"""
    r, c = 0, 0
    while i:
        r += (i & 1) << (2 * c)
        i >>= 1; c += 1
    return r


def even_bits_table(count: int) -> List[int]:
    """[even_bits_at(i) for i in range(count)], count <= 2^32, by the usual mask-and-shift bit spreading on a uint64 array"""
    import numpy as np
    if count > 1 << 32:
        raise ValueError("even-bits table beyond 2^32 rows")
    x = np.arange(count, dtype=np.uint64)
    for shift, mask in ((16, 0x0000FFFF0000FFFF), (8, 0x00FF00FF00FF00FF), (4, 0x0F0F0F0F0F0F0F0F), (2, 0x3333333333333333),
                        (1, 0x5555555555555555)):
        x = (x | (x << np.uint64(shift))) & np.uint64(mask)
    return x.tolist()


_EVEN_MASK = int.from_bytes(bytes([0x55] * 32), "little")
_ODD_MASK = int.from_bytes(bytes([0xAA] * 32), "little")


def decompose(word: int) -> Tuple[int, int]:
    """even_bits.rs:253-270: even bits of the 32-byte repr; odd bits of the LOWER 128 bits shifted right by one"""
    return word & _EVEN_MASK, ((word & _ODD_MASK) & ((1 << 128) - 1)) >> 1


_NO_GADGET = frozenset(("Add", "Sub", "Mull", "UMulh", "Cmpa", "Cmpae", "CMov", "Jmp", "CJmp", "CnJmp", "LoadW", "StoreW", "Answer", "Not"))


def _batch_inverse(values: List[int], p: int) -> List[int]:
    """the inverses modulo p of `values` with ONE modular inversion (prefix products); zeros stay zero"""
    prefix, run = [], 1
    for v in values:
        prefix.append(run)
        if v:
            run = run * v % p
    inv = pow(run, -1, p)
    out = [0] * len(values)
    for i in range(len(values) - 1, -1, -1):
        v = values[i]
        if v:
            out[i] = inv * prefix[i] % p
            inv = inv * v % p
    return out


def program_instance(prog: List[T.Instruction], word_bits: int, reg_count: int = 8, arrays: bool = False) -> List[List[int]]:
    """tables/prog.rs:38-60: the 94 instance columns; the program is padded to TABLE_LEN lines with its terminal Answer.
    arrays: the columns as uint64 numpy arrays (same values)"""
    table_len = 1 << (word_bits // 2)
    if not prog or prog[-1].name != "Answer":
        raise ValueError("Empty programs are invalid / the last instruction must be Answer")
    if len(prog) > table_len:
        raise ValueError("program longer than the program table")
    counter = iter(range(1 << 30))
    line = ProgramLine(lambda: next(counter), reg_count)
    n_cols = len(line.to_vec())
    pad = table_len - len(prog)                         # the terminal Answer, repeated
    if arrays:                                          # the same cells written into one uint64 matrix (every value is below 2^64)
        import numpy as np
        mat = np.zeros((n_cols, table_len), dtype=np.uint64)
        rows_of = {}
        for off, ins in enumerate(prog):
            if id(ins) not in rows_of:
                rows_of[id(ins)] = [(c, v) for c, v in line.row_values(ins).items() if v]
            for c, v in rows_of[id(ins)]:
                mat[c, off] = v
        if pad:
            for c, v in line.row_values(prog[-1]).items():
                if v:
                    mat[c, len(prog):] = v
        return [mat[c] for c in range(n_cols)]
    cols = [[0] * table_len for _ in range(n_cols)]
    rows_of = {}
    for off, ins in enumerate(prog):
        if id(ins) not in rows_of:
            rows_of[id(ins)] = line.row_values(ins)
        for c, v in rows_of[id(ins)].items():
            if v:
                cols[c][off] = v
    if pad:
        for c, v in line.row_values(prog[-1]).items():
            if v:
                cols[c][len(prog):] = [v] * pad
    return cols


class TinyRamCircuit:
    """configure() at construction; synthesize(trace) -> (fixed, copies, advice); the ConstraintSystem is .cs"""

    def __init__(self, PL, word_bits: int, reg_count: int = 8, with_prog: bool = True):
        """with_prog=False is the reference's ExeCircuit (tables/exe.rs:1082-1116): the execution table alone, no program table,
        no instance columns, no dynamic lookup"""
        if word_bits % 8 or not 8 <= word_bits <= 32:
            raise ValueError("WORD_BITS must be 8, 16, 24 or 32")
        self.PL, self.W, self.R, self.with_prog = PL, word_bits, reg_count, with_prog
        self.table_len = 1 << (word_bits // 2)                   # ExeConfig::TABLE_LEN = ProgConfig::TABLE_LEN (exe.rs:106, prog.rs:137)
        self.cs = PL.ConstraintSystem()
        self.gate_names: List[str] = []
        self._configure()

    # ---- helpers -----------------------------------------------------------------------------------------------------------------
    def _adv(self, col, rot=0): return self.cs.query(self.PL.ADVICE, col, rot)
    def _fix(self, col, rot=0): return self.cs.query(self.PL.FIXED, col, rot)

    def _gate(self, name, selector, polys):
        """meta.create_gate(name, |meta| Constraints::with_selector(selector, polys))"""
        self.cs.create_gate([selector * p for p in polys])
        self.gate_names += [name] * len(polys)

    def _new_tracked(self):
        c = self.cs.advice_column()
        self.intermediate.append(c)
        return c

    def _even_bits(self, word, s_even_bits) -> EvenBits:
        """EvenBitsConfig::configure (even_bits.rs:115-173): even / odd columns, the decompose gate and the two table lookups,
        enabled by s_table * (sum of the advice selectors)"""
        cfg = EvenBits(word, self._new_tracked(), self._new_tracked())

        def sel():
            s_table = self._fix(self.s_table)
            e = None
            for c in s_even_bits:
                q = self._adv(c)
                e = q if e is None else e + q
            return s_table * e if e is not None else s_table

        s = sel()
        lhs, rhs, out = self._adv(cfg.even), self._adv(cfg.odd), self._adv(word)
        self._gate("decompose", s, [lhs + self.PL.Constant(2) * rhs - out])
        s = sel(); e = self._adv(cfg.even)
        self.cs.lookup([(s * e, self._fix(self.t_even))])
        s = sel(); o = self._adv(cfg.odd)
        self.cs.lookup([(s * o, self._fix(self.t_even))])
        return cfg

    def _signed(self, s_signed, word: EvenBits) -> Signed:
        """SignedConfig::configure (signed.rs:24-111)"""
        C = self.PL.Constant
        msb, word_sigma, cs_exp = self._new_tracked(), self._new_tracked(), self._new_tracked()
        check_sign = self._even_bits(cs_exp, s_signed)
        cfg = Signed(word, msb, word_sigma, check_sign)
        one, two, mx = C(1), C(2), C(1 << self.W)
        word_odd = self._adv(word.odd)
        q_msb = self._adv(msb)
        q_ws = self._adv(word_sigma)
        sigma = -q_msb * two * q_ws + q_ws
        q_word = self._adv(word.word)
        q_cs = self._adv(check_sign.word)
        s_table = self._fix(self.s_table)
        e = None
        for c in s_signed:
            q = self._adv(c)
            e = q if e is None else e + q
        sel = s_table * e if e is not None else s_table
        self._gate("signed", sel, [(-q_msb * mx + q_word) - sigma,
                                   (word_odd + (one - two * q_msb) * C(1 << (self.W - 2)) - q_cs)])
        return cfg

    def _sigma(self, s: Signed):
        """a_sigma = -msb * 2 * word_sigma + word_sigma (ssum.rs:83-85, sprod.rs:73-75)"""
        ws = self._adv(s.word_sigma)
        msb = self._adv(s.msb)
        return -msb * self.PL.Constant(2) * ws + ws

    # ---- configure (circuits/mod.rs:48-60) -----------------------------------------------------------------------------------------------
    def _configure(self):
        PL, cs, W, R = self.PL, self.cs, self.W, self.R
        A, F, I, C = PL.ADVICE, PL.FIXED, PL.INSTANCE, PL.Constant
        adv, fix = self._adv, self._fix

        # ProgConfig::configure (prog.rs:139-161)
        if self.with_prog:
            self.s_prog = cs.fixed_column()                                    # meta.selector(): never queried by a gate
            self.prog_input = ProgramLine(cs.instance_column, R)
            self.prog_table = ProgramLine(cs.advice_column, R)
            self.prog_pc = cs.fixed_column()
            self.dyn_tag = cs.fixed_column()                                   # create_dynamic_table (fork): the table's tag column
            for c in self.prog_input.to_vec(): cs.enable_equality(I, c)
            for c in self.prog_table.to_vec(): cs.enable_equality(A, c)

        # ExeChip::configure_instructions (exe.rs:535-767)
        self.time = cs.fixed_column()
        self.pc = cs.advice_column()
        self.line = ProgramLine(cs.advice_column, R)
        self.reg = [cs.advice_column() for _ in range(R)]
        self.flag, self.address, self.value = cs.advice_column(), cs.advice_column(), cs.advice_column()
        self.out = {n: cs.advice_column() for n in OUT_NAMES}
        self.first_line = cs.fixed_column()                                    # meta.selector()
        self.s_table = cs.fixed_column()                                       # meta.complex_selector()
        self.s_trace = cs.advice_column()
        self.t_even = cs.fixed_column()                                        # EvenBitsTable
        self.t_pow_values, self.t_pow_powers = cs.fixed_column(), cs.fixed_column()
        self.t_out_opcode = cs.fixed_column()
        self.t_out = {n: cs.fixed_column() for n in OUT_NAMES}
        self.t_out_continue = cs.fixed_column()
        out = self.out

        # CorrectOutConfig::configure (out_table.rs:23-83)
        s_table = fix(self.s_table)
        s_next = adv(self.s_trace, 1)
        s_cur = adv(self.s_trace)
        opcode = adv(self.line.opcode)
        oq = {n: adv(out[n]) for n in OUT_NAMES}
        pairs = [(s_next, self.t_out_continue), (opcode + C(1), self.t_out_opcode)]
        pairs += [(oq[n], self.t_out[n]) for n in ("and", "xor", "or", "sum", "ssum", "prod", "sprod", "mod", "shift", "flag1", "flag2", "flag3", "flag4")]
        cs.lookup([(s_table * s_cur * e, fix(t)) for e, t in pairs])

        self.intermediate: List[int] = []                                      # TrackColumns (exe.rs:563, assign.rs:29-52)
        # TempVars::configure (exe/temp_vars.rs:29-123): the four words are NOT tracked
        ta, tb, tc, td = (cs.advice_column() for _ in range(4))
        self.tv_a = self._even_bits(ta, [out[n] for n in ("mod", "and", "or", "xor", "ssum", "sprod")])
        self.tv_b = self._even_bits(tb, [out[n] for n in ("mod", "sum", "ssum", "sprod", "flag4")])
        self.tv_c = self._even_bits(tc, [out[n] for n in ("xor", "prod", "shift", "ssum", "sprod")])
        self.tv_d = self._even_bits(td, [out[n] for n in ("prod", "sprod")])
        a_w, b_w, c_w, d_w = ta, tb, tc, td

        def gsel(name):                       # s_table * s_<gadget>
            return fix(self.s_table) * adv(out[name])

        # Flag1Config (flag1.rs:23-47)
        s = gsel("flag1"); c_ = adv(c_w); flag_n = adv(self.flag, 1)
        self._gate("flag1", s, [flag_n * c_])
        # Flag2Config (flag2.rs:28-60)
        self.a_flag = self._new_tracked()
        s = gsel("flag2"); c_ = adv(c_w); flag_n = adv(self.flag, 1); a_flag = adv(self.a_flag)
        self._gate("flag2", s, [(flag_n + c_) * a_flag - C(1)])
        # Flag3Config (flag3.rs:29-92) over r_decompose, which the shift gadget shares
        flag3_r = self._new_tracked()
        self.r_dec = self._even_bits(flag3_r, [out["flag3"], out["shift"]])
        one, two = C(1), C(2)
        s = gsel("flag3")
        a_, b_, c_ = adv(a_w), adv(b_w), adv(c_w)
        flag_n = adv(self.flag, 1)
        re, ro, r_ = adv(self.r_dec.even), adv(self.r_dec.odd), adv(self.r_dec.word)
        self._gate("flag3", s, [b_ * flag_n + (one - flag_n) * (c_ - a_ - one - two * ro - re),
                                c_ * ((c_ - a_ - one) - r_)])
        # SumConfig (sum.rs:56-100)
        s = gsel("sum"); a_, b_, c_, d_ = adv(a_w), adv(b_w), adv(c_w), adv(d_w); flag_n = adv(self.flag, 1)
        self._gate("sum", s, [a_ + b_ - c_ - (C(1 << W) * flag_n) + d_])
        # ModConfig (modulo.rs:28-66)
        s = gsel("mod"); a_, b_, c_, d_ = adv(a_w), adv(b_w), adv(c_w), adv(d_w); flag_n = adv(self.flag, 1)
        self._gate("mod", s, [flag_n * (b_ - d_) + d_ - b_ * c_ - a_])
        # a's second decomposition, then LogicConfig (exe.rs:626-648, logic.rs:47-190)
        self.a_decomp = self._even_bits(a_w, [out[n] for n in ("and", "xor", "ssum")])
        lg = [out[n] for n in ("and", "xor", "or")]
        self.logic_b = self._even_bits(b_w, lg)
        self.even_sum = self._even_bits(self._new_tracked(), lg)
        self.odd_sum = self._even_bits(self._new_tracked(), lg)
        for lhs, rhs, res in ((self.a_decomp.even, self.logic_b.even, self.even_sum.word), (self.a_decomp.odd, self.logic_b.odd, self.odd_sum.word)):
            l_, r_, s_ = adv(lhs), adv(rhs), adv(res)
            st = fix(self.s_table); sa, sx, so = adv(out["and"]), adv(out["xor"]), adv(out["or"])
            self._gate("l_add", st * (sa + sx + so), [l_ + r_ - s_])
        s = gsel("and"); eo, oo, res = adv(self.even_sum.odd), adv(self.odd_sum.odd), adv(c_w)
        self._gate("and", s, [eo + C(2) * oo - res])
        s = gsel("xor"); ee, oe, res = adv(self.even_sum.even), adv(self.odd_sum.even), adv(c_w)
        self._gate("xor", s, [ee + C(2) * oe - res])
        s = gsel("or")
        ee, eo, oe, oo, res = adv(self.even_sum.even), adv(self.even_sum.odd), adv(self.odd_sum.even), adv(self.odd_sum.odd), adv(c_w)
        self._gate("or", s, [(ee + C(2) * oe) + (eo + C(2) * oo) - res])
        # ProdConfig (prod.rs:44-77)
        s = gsel("prod"); a_, b_, c_, d_ = adv(a_w), adv(b_w), adv(c_w), adv(d_w)
        self._gate("prod", s, [a_ * b_ - d_ - C(1 << W) * c_])
        # signed views of a, b, c (exe.rs:661-698)
        self.signed_a = self._signed([out["ssum"]], self.a_decomp)
        self.b_decomp = self._even_bits(b_w, [out["sprod"]])
        self.signed_b = self._signed([out["sprod"]], self.b_decomp)
        self.c_decomp = self._even_bits(c_w, [out["ssum"]])
        self.signed_c = self._signed([out["ssum"]], self.c_decomp)
        # SSumConfig (ssum.rs:50-101)
        s = gsel("ssum")
        a_s = self._sigma(self.signed_a); b_ = adv(b_w); c_s = self._sigma(self.signed_c); d_ = adv(d_w); flag_n = adv(self.flag, 1)
        self._gate("ssum", s, [a_s + b_ - c_s - (C(1 << W) * flag_n) + d_])
        # SProdConfig (sprod.rs:45-94)
        s = gsel("sprod")
        a_s, b_s, c_s = self._sigma(self.signed_a), self._sigma(self.signed_b), self._sigma(self.signed_c); d_ = adv(d_w)
        self._gate("sprod", s, [a_s * b_s - d_ - C(1 << W) * c_s])
        # ShiftConfig (shift.rs:72-168)
        self.a_shift, self.a_power = self._new_tracked(), self._new_tracked()
        s = gsel("shift")
        a_, b_, c_, d_ = adv(a_w), adv(b_w), adv(c_w), adv(d_w)
        r_o, r_e = adv(self.r_dec.odd), adv(self.r_dec.even)
        q_shift, q_power = adv(self.a_shift), adv(self.a_power)
        self._gate("shift", s, [q_shift * (q_shift - C(1)),
                                (C(1) - q_shift) * (C(W) - a_ - (C(2) * r_o) - r_e),
                                q_power * b_ - d_ - C(1 << W) * c_])
        s_shift, a_ = adv(out["shift"]), adv(a_w)
        q_shift, q_power = adv(self.a_shift), adv(self.a_power)
        cs.lookup([(s_shift * (a_ + q_shift * (C(W) - a_)), fix(self.t_pow_values)),
                   ((s_shift * q_power) + C(1) - (s_shift * C(1)), fix(self.t_pow_powers))])
        # Flag4Config (flag4.rs:29-65)
        self.lsb_b, self.b_flag = self._new_tracked(), self._new_tracked()
        s = gsel("flag4")
        q_bf, msb_b, lsb_b, flag_n = adv(self.b_flag), adv(self.signed_b.msb), adv(self.lsb_b), adv(self.flag, 1)
        self._gate("flag4", s, [flag_n - (q_bf * msb_b) - ((C(1) - q_bf) * lsb_b)])

        # ExeChip::configure (exe.rs:769-790): unchanged, trace_len gates, temp-var selector gates
        def trace_next():                     # TableSelector::query_trace_next (tables/mod.rs:45-53)
            return fix(self.s_table) * adv(self.s_trace, 1)

        def trace_cur():                      # TableSelector::query (tables/mod.rs:35-43)
            return fix(self.s_table) * adv(self.s_trace)

        ch = self.line.ch
        s_ext = trace_next()
        ch_pc = adv(ch["pc"]); pc_n = adv(self.pc, 1); pc_ = adv(self.pc)
        ch_flag = adv(ch["flag"]); flag_n = adv(self.flag, 1); flag_ = adv(self.flag)
        polys = [(C(1) - ch_pc) * (pc_ + C(1) - pc_n), (C(1) - ch_flag) * (flag_ - flag_n)]
        for ch_r, r in zip(ch["regs"], self.reg):
            q_ch = adv(ch_r); r_n = adv(r, 1); r_c = adv(r)
            polys.append((C(1) - q_ch) * (r_c - r_n))
        self._gate("unchanged", s_ext, polys)                                  # changed.rs:83-121

        first = fix(self.first_line); s_tr = adv(self.s_trace)                 # exe.rs:148-168
        polys = [C(1) - s_tr, adv(self.pc), adv(self.flag)] + [adv(r) for r in self.reg]
        self._gate("start_trace", first, polys)
        ans, big = C(T.OPCODES["Answer"]), C(U64_MAX)                          # exe.rs:170-193
        st = fix(self.s_table); s_tr = adv(self.s_trace); s_tr_n = adv(self.s_trace, 1); opc = adv(self.line.opcode)
        contiguous = s_tr - s_tr_n
        may_change = big - (s_tr * big) + opc - ans
        self._gate("contiguous_trace", st, [contiguous * may_change])

        sa, sb, sc, sd = self.line.a, self.line.b, self.line.c, self.line.d

        def pc_gate(sel_col, tv, nm):          # exe.rs:195-215
            q_s = adv(sel_col); pc_ = adv(self.pc); t = adv(tv)
            st = fix(self.s_table); s_tr = adv(self.s_trace, 1)
            self._gate(f"tv.{nm}.pc", st * s_tr * q_s, [pc_ - t])

        def pc_plus_one_gate(sel_col, tv, nm):  # exe.rs:217-236
            q_s = adv(sel_col); pc_ = adv(self.pc); t = adv(tv)
            self._gate(f"tv.{nm}.pc+1", trace_next() * q_s, [(pc_ + C(1)) - t])

        def pc_next_gate(sel_col, tv, nm):     # exe.rs:238-265
            q_s = adv(sel_col); pc_n = adv(self.pc, 1); t = adv(tv)
            self._gate(f"tv.{nm}.pc_next", trace_next() * q_s, [pc_n - t])

        def reg_gate(sel_cols, tv, nm):        # exe.rs:267-289
            for i, sc_ in enumerate(sel_cols):
                q_s = adv(sc_); r = adv(self.reg[i]); t = adv(tv)
                self._gate(f"tv.{nm}.reg[{i}]", trace_cur() * q_s, [r - t])

        def reg_next_gate(sel_cols, tv, nm):   # exe.rs:291-317
            for i, sc_ in enumerate(sel_cols):
                q_s = adv(sc_); r = adv(self.reg[i], 1); t = adv(tv)
                self._gate(f"tv.{nm}.reg_next[{i}]", trace_next() * q_s, [r - t])

        def immediate_gate(sel_col, tv, nm):   # exe.rs:319-339
            q_s = adv(sel_col); imm = adv(self.line.immediate); t = adv(tv)
            self._gate(f"tv.{nm}.a", trace_cur() * q_s, [imm - t])

        def simple_gate(kind, sel_col, tv, nm, poly_of):     # vaddr / one / zero / max_word gates (exe.rs:341-428)
            q_s = adv(sel_col)
            pre = adv(self.value) if kind == "vaddr" else None
            t = adv(tv)
            st = fix(self.s_table); s_tr = adv(self.s_trace)
            self._gate(f"tv.{nm}.{kind}", st * s_tr * q_s, [poly_of(pre, t)])

        # configure_selectors_a .. d (exe.rs:430-498)
        pc_next_gate(sa["pc_next"], a_w, "a"); reg_gate(sa["reg"], a_w, "a"); reg_next_gate(sa["reg_next"], a_w, "a")
        immediate_gate(sa["a"], a_w, "a"); simple_gate("vaddr", sa["v_addr"], a_w, "a", lambda v, t: v - t)
        pc_gate(sb["pc"], b_w, "b"); pc_next_gate(sb["pc_next"], b_w, "b"); pc_plus_one_gate(sb["pc_plus_one"], b_w, "b")
        reg_gate(sb["reg"], b_w, "b"); reg_next_gate(sb["reg_next"], b_w, "b"); immediate_gate(sb["a"], b_w, "b")
        simple_gate("max_word", sb["max_word"], b_w, "b", lambda _, t: C((1 << W) - 1) - t)
        reg_gate(sc["reg"], c_w, "c"); reg_next_gate(sc["reg_next"], c_w, "c"); immediate_gate(sc["a"], c_w, "c")
        simple_gate("zero", sc["zero"], c_w, "c", lambda _, t: t)
        pc_gate(sd["pc"], d_w, "d"); reg_gate(sd["reg"], d_w, "d"); reg_next_gate(sd["reg_next"], d_w, "d")
        immediate_gate(sd["a"], d_w, "d"); simple_gate("zero", sd["zero"], d_w, "d", lambda _, t: t)
        simple_gate("one", sd["one"], d_w, "d", lambda _, t: C(1) - t)

        if not self.with_prog:
            return
        # prog_config.lookup (circuits/mod.rs:52-57 -> prog.rs:163-193): the fork's lookup_dynamic
        s_tr = adv(self.s_trace)
        pc_ = adv(self.pc)
        table_map = [(pc_, (F, self.prog_pc))]
        for exe_col, prog_col in zip(self.line.to_vec(), self.prog_table.to_vec()):
            table_map.append((adv(exe_col), (A, prog_col)))
        cs.lookup([(s_tr, fix(self.dyn_tag))] + [(s_tr * e, cs.query(kind, col)) for e, (kind, col) in table_map])

    # ---- synthesize (circuits/mod.rs:62-75) ---------------------------------------------------------------------------------------------
    def synthesize(self, trace: Optional[T.Trace], n: int, a_flag_rand: Optional[Callable[[], int]] = None,
                   reg_operand_value: bool = True, arrays: bool = False):
        """Returns (fixed, copies, advice): fixed = one FixedColumn (assigned prefix + fill value) per fixed column, advice = one
        sparse {row: value} dict per advice column, copies = the copy constraints of assign_advice_from_instance (one plonk.CopyBlock per column pair).  Values are
        canonical ints of the circuit field.

        reg_operand_value: push_temp_var_vals takes a REGISTER operand's temp-var value to be the register's INDEX
        (`ImmediateOrRegName::RegName(r) => r.0.into()`, aux.rs:419-427) although the selector it sets is reg[r], whose gate
        (exe.rs:267-289) demands the register's VALUE; True (default) assigns the value, False reproduces the reference.
        a_flag_rand: flag2.rs:70 fills a_flag with F::random(OsRng) when c + flag_next = 0; here a_flag_rand() or 0.
        arrays: columns whose cells depend on the instruction alone (the program line's selector vector, the Out row) and the
        fixed range columns come back as uint64 numpy arrays instead of lists (same values; device_columns uploads them without
        a list round trip)."""
        PL, cs, W, R, TL = self.PL, self.cs, self.W, self.R, self.table_len
        p = PL_FIELD_MODULUS
        A, I = PL.ADVICE, PL.INSTANCE
        if TL > n:
            raise ValueError("NotEnoughRowsAvailable")
        fixed = [[] for _ in range(cs.num_fixed)]                # the assigned prefix of each column; (prefix, fill) pairs are returned
        fill = [0] * cs.num_fixed
        for col in ((self.s_prog, self.dyn_tag, self.prog_pc) if self.with_prog else ()) + ((self.first_line, self.s_table, self.time) if trace is not None else ()):
            fixed[col] = [0] * TL
        rows_cap = max(TL, len(trace.exe) + 1 if trace is not None else 0)
        advice: List[list] = [[None] * rows_cap for _ in range(cs.num_advice)]     # None = unassigned (columns_to_lists trims / zero-fills)
        copies = []

        # ExeChip::construct: the three lookup tables (exe.rs:519-533); unused rows repeat row 0 (SimpleTableLayouter)
        def table(cols_rows):
            for col, rows in cols_rows.items():
                fixed[col], fill[col] = list(rows), rows[0]

        import numpy as np
        ones = (lambda: np.ones(TL, dtype=np.uint64)) if arrays else (lambda: [1] * TL)
        ramp = (lambda: np.arange(TL, dtype=np.uint64)) if arrays else (lambda: list(range(TL)))
        table({self.t_even: even_bits_table(TL)})                                                           # even_bits.rs:56-74
        table({self.t_pow_values: list(range(W)) + [W],
               self.t_pow_powers: [(1 << i) % (1 << W) for i in range(W)] + [0]})                          # pow.rs:21-66
        rows = [(T.OPCODES[nm] + 1, OUT[nm], nm != "Answer") for nm in OUT_TABLE_ORDER] + [(0, (), False)]  # out_table.rs:133-215
        table({self.t_out_opcode: [r[0] for r in rows], self.t_out_continue: [int(r[2]) for r in rows],
               **{self.t_out[nm]: [int(nm in r[1]) for r in rows] for nm in OUT_NAMES}})

        # ProgConfig::assign_prog (prog.rs:195-233): the program table is a copy of the instance columns
        if self.with_prog:
            for ic, tc in zip(self.prog_input.to_vec(), self.prog_table.to_vec()):
                copies.append(PL.CopyBlock((I, ic, 0), (A, tc, 0), TL))
            fixed[self.s_prog], fixed[self.dyn_tag], fixed[self.prog_pc] = ones(), ones(), ramp()

        if trace is not None:
            if trace.word_bits != W or trace.reg_count != R:
                raise ValueError("trace of a different machine")
            exe = trace.exe
            if len(exe) > TL - 1:
                raise ValueError("trace longer than TABLE_LEN - 1")
            # ExeChip::assign_trace (exe.rs:792-1080).  The reference assigns row by row; the same cells are written here
            # column by column where a column's value depends on the instruction alone (one table row per distinct instruction,
            # gathered with numpy), then the machine state and the temporary variables, then -- row by row, in the reference's
            # order, last write wins -- what the instruction's gadget assigns, and `value` last.
            import numpy as np
            fixed[self.first_line][0] = 1
            fixed[self.s_table], fixed[self.time] = ones(), ramp()
            ne = len(exe)
            advice[self.s_trace][:ne] = [1] * ne
            # -- static part: intermediate fill, opcode, immediate, the selector vector of the line, the Out row
            kinds, kind_of, templates = {}, [0] * ne, []
            for off, step in enumerate(exe):
                ins = step.instruction
                ki = kinds.get(id(ins))
                if ki is None:
                    ki = kinds[id(ins)] = len(templates)
                    tm = {c: U64_MAX for c in self.intermediate}
                    tm[self.line.opcode], tm[self.line.immediate] = ins.opcode, ins.immediate()
                    for c, v in self.line.row_values(ins).items():
                        if c not in (self.line.opcode, self.line.immediate):
                            tm[c] = v
                    for nm in OUT_NAMES:
                        tm[self.out[nm]] = int(nm in OUT[ins.name])
                    templates.append(tm)
                kind_of[off] = ki
            if ne:
                static_cols = list(templates[0])
                if any(list(tm) != static_cols for tm in templates):
                    raise AssertionError("internal: the static columns do not depend on the instruction")
                table_ = np.array([[tm[c] % p for c in static_cols] for tm in templates], dtype=np.uint64)     # all below 2^64
                gathered = table_[np.array(kind_of, dtype=np.int64)]
                untouched = (set(self.line.to_vec()) | set(self.out.values())) if arrays else ()     # nothing below writes these
                for j_, c in enumerate(static_cols):
                    if c in untouched:
                        advice[c] = np.ascontiguousarray(gathered[:, j_])
                    else:
                        advice[c][:ne] = gathered[:, j_].tolist()
            # -- machine state
            advice[self.pc][:ne] = [st.pc for st in exe]
            for r_, rc in enumerate(self.reg):
                advice[rc][:ne] = [st.regs[r_] % p for st in exe]
            advice[self.flag][:ne] = [int(st.flag) for st in exe]
            # -- temporary variables and their even / odd halves (temp_vars.rs:125-169), a_flag (flag2.rs:62-74)
            sel_cache = {}
            tvs = [self._temp_var_vals(exe, off, reg_operand_value, p, sel_cache) for off in range(ne)]
            m128 = (1 << 128) - 1
            for idx, cfg in enumerate((self.tv_a, self.tv_b, self.tv_c, self.tv_d)):
                words = [t[idx] for t in tvs]
                advice[cfg.word][:ne] = words
                advice[cfg.even][:ne] = [w & _EVEN_MASK for w in words]
                advice[cfg.odd][:ne] = [((w & _ODD_MASK) & m128) >> 1 for w in words]
            sums = [(tvs[off][2] + (int(exe[off + 1].flag) if off + 1 < ne else 0)) % p for off in range(ne)]
            advice[self.a_flag][:ne] = [x if x else (a_flag_rand() % p if a_flag_rand else 0) for x in _batch_inverse(sums, p)]
            # -- the gadget of the row's instruction
            cur = [0]
            def put(col, v):
                advice[col][cur[0]] = v % p
            for off, step in enumerate(exe):
                ins = step.instruction
                nm = ins.name
                if nm in _NO_GADGET:
                    continue
                cur[0] = off
                ta, tb, tc, td = tvs[off]
                if nm == "And":
                    self._assign_logic(put, ta, tb, lambda x, y: x & y)
                elif nm in ("Xor", "Cmpe", "Mov"):
                    self._assign_logic(put, ta, tb, lambda x, y: x ^ y)
                elif nm == "Or":
                    self._assign_logic(put, ta, tb, lambda x, y: x | y)
                elif nm in ("Cmpg", "Cmpge"):                                                           # ssum.rs:103-115
                    self._assign_signed(put, self.signed_a, ta & ((1 << 128) - 1))
                    self._assign_signed(put, self.signed_c, tc & ((1 << 128) - 1))
                    self._assign_decompose(put, self.signed_c.word, tc)
                elif nm == "SMulh":                                                                     # sprod.rs:96-112
                    self._assign_signed(put, self.signed_a, ta & ((1 << 128) - 1))
                    self._assign_signed(put, self.signed_b, tb & ((1 << 128) - 1))
                    self._assign_decompose(put, self.signed_b.word, tb)
                    self._assign_signed(put, self.signed_c, tc & ((1 << 128) - 1))
                    self._assign_decompose(put, self.signed_c.word, tc)
                elif nm in ("UMod", "UDiv"):                                                            # flag3.rs:94-113
                    r = 0 if tc == 0 else (tc - ta - 1) % p
                    put(self.r_dec.word, r)
                    self._assign_decompose(put, self.r_dec, r)
                elif nm in ("Shl", "Shr"):
                    bits = ins.a.value if isinstance(ins.a, T.Imm) else step.regs[ins.a.index]
                    self._assign_shift(put, bits)                                                       # shift.rs:170-211
                    b64 = tb & ((1 << 128) - 1)
                    if b64 >= 1 << 64:
                        raise OverflowError("tb does not fit u64")
                    put(self.lsb_b, b64 & 1)                                                            # flag4.rs:67-91
                    put(self.b_flag, int(nm == "Shl"))
                    self._assign_signed(put, self.signed_b, b64)
            advice[self.value][:ne] = [(st.v_addr or 0) % p for st in exe]
            advice[self.s_trace][ne] = 0
        return [FixedColumn(pre, f) for pre, f in zip(fixed, fill)], copies, advice

    def assign_instance(self, advice, instances):
        """assign_advice_from_instance: the program-table advice cells take the instance values (prog.rs:206-216)"""
        TL = self.table_len
        for ic, tc in zip(self.prog_input.to_vec(), self.prog_table.to_vec()):
            if not isinstance(instances[ic], list):          # program_instance(arrays=True): TABLE_LEN values each
                advice[tc] = instances[ic].copy()
                continue
            col = list(instances[ic][:TL])
            advice[tc][:TL] = col + [0] * (TL - len(col))
        return advice

    # ---- witness helpers -------------------------------------------------------------------------------------------------------------
    def _assign_decompose(self, put, cfg: EvenBits, word: int):
        e, o = decompose(word)
        put(cfg.even, e); put(cfg.odd, o)
        return e, o

    def _assign_logic(self, put, lhs, rhs, op):
        """LogicConfig::assign_logic + assign_and / xor / or (logic.rs:192-279); res is the temp var c's word column"""
        le, lo = self._assign_decompose(put, self.a_decomp, lhs)
        re, ro = self._assign_decompose(put, self.logic_b, rhs)
        put(self.even_sum.word, le + re); self._assign_decompose(put, self.even_sum, le + re)
        put(self.odd_sum.word, lo + ro); self._assign_decompose(put, self.odd_sum, lo + ro)
        m = (1 << 128) - 1
        put(self.tv_c.word, op(lhs & m, rhs & m))

    def _assign_signed(self, put, cfg: Signed, word: int):
        """SignedConfig::assign_signed (signed.rs:113-164)"""
        W = self.W
        msb = (word >> (W - 1)) & 1
        put(cfg.msb, msb)
        put(cfg.word_sigma, abs(-msb * (1 << W) + word))
        _e, o = self._assign_decompose(put, cfg.word, word)
        cs_ = o + (1 - 2 * msb) * (1 << (W - 2))
        if cs_ < 0:
            raise AssertionError("assertion failed: cs >= 0")
        self._assign_decompose(put, cfg.check_sign, cs_)
        put(cfg.check_sign.word, cs_)

    def _assign_shift(self, put, shift_bits: int):
        W = self.W
        put(self.a_shift, int(W < shift_bits))
        if shift_bits >= 64:
            raise OverflowError("attempt to multiply with overflow")           # 2u64.pow(shift_bits)
        put(self.a_power, 0 if shift_bits == W else 1 << shift_bits)
        r = 0 if shift_bits > W else W - shift_bits
        put(self.r_dec.word, r)
        self._assign_decompose(put, self.r_dec, r)

    def _temp_var_vals(self, steps, i, reg_operand_value, p, sel_cache=None):
        """TempVarSelectorsRow::push_temp_var_vals (aux.rs:409-560): the values of the temporary variables a, b, c, d"""
        W = self.W
        step = steps[i]
        ins = step.instruction
        mask32 = 0xFFFFFFFF
        sel = sel_cache.get(id(ins)) if sel_cache is not None else None       # one `selections` per distinct instruction of a trace
        if sel is None:
            sel = selections(ins)[:4]
            if sel_cache is not None:
                sel_cache[id(ins)] = sel
        sa, sb, sc, sd = sel
        get = lambda op: op.value if isinstance(op, T.Imm) else step.regs[op.index]     # ImmediateOrRegName::get

        def a_of(op):
            if isinstance(op, T.Imm): return op.value
            return step.regs[op.index] if reg_operand_value else op.index

        def common(s):
            k = s[0]
            if k == "Zero" or k == "Unset": return 0
            if k == "Reg": return step.regs[s[1]]
            if k == "RegN": return steps[i + 1].regs[s[1]]
            if k == "A": return a_of(s[1])
            if k == "Pc": return step.pc
            if k == "PcN": return steps[i + 1].pc
            if k == "PcPlusOne": return step.pc + 1
            if k == "VAddr": return step.v_addr
            if k == "MaxWord": return (1 << W) - 1
            if k == "One": return 1
            return None

        nm = ins.name
        ta = common(sa)
        if ta is None:                                                                   # SelectionA::NonDet
            if nm != "UDiv": raise RuntimeError("Unhandled non-deterministic advice")
            av = get(ins.a)
            ta = 0 if av == 0 else step.regs[ins.rj] % av
        tb = common(sb)
        if tb is None:                                                                   # SelectionB::NonDet
            if nm == "UMod":
                av = get(ins.a)
                tb = 0 if av == 0 else step.regs[ins.rj] // av
            elif nm in ("Cmpa", "Cmpg"):
                x, c = step.regs[ins.ri], a_of(ins.a)
                tb = ((1 << W) - (x - c) if x > c else c - x) & mask32
            elif nm in ("Cmpae", "Cmpge"):
                x, c = step.regs[ins.ri], a_of(ins.a)
                tb = ((1 << W) - 1 - (x - c) if x >= c else c - x - 1) & mask32
            else:
                raise RuntimeError("Unhandled non-deterministic advice")
        tc = common(sc)
        if tc is None:                                                                   # SelectionC::NonDet
            if nm == "Mull":
                tc = ((step.regs[ins.rj] * get(ins.a)) >> W) & ((1 << W) - 1)
            elif nm == "Cmpe":
                tc = step.regs[ins.ri] ^ get(ins.a)
            elif nm == "Shl":
                av, b = get(ins.a), step.regs[ins.rj]
                d = (b << av) & ((1 << W) - 1)
                assert d == steps[i + 1].regs[ins.ri]
                num = (1 << av) * b - d                                                  # shift::non_det_c (shift.rs:219-226)
                tc = abs(num) // (1 << W) * (1 if num >= 0 else -1)
                if tc < 0: raise OverflowError("non_det_c: negative")
            else:
                raise RuntimeError("Unhandled non-deterministic advice")
        td = common(sd)
        if td is None:                                                                   # SelectionD::NonDet
            if nm == "UMulh":
                td = (step.regs[ins.rj] * get(ins.a)) & ((1 << W) - 1)
            elif nm == "SMulh":
                _u, lower, _f = T.smulh_eval(get(ins.a), step.regs[ins.rj], W)
                td = lower
            elif nm == "Shr":
                av, b = get(ins.a), step.regs[ins.rj]
                c = b >> av
                assert c == steps[i + 1].regs[ins.ri]
                td = ((1 << av) * b - (1 << W) * c) % p                                  # shift::non_det_d (shift.rs:214-217)
            else:
                raise RuntimeError("Unhandled non-deterministic advice")
        return ta & mask32, tb & mask32, tc % p, td % p


class FixedColumn:
    """a fixed column as its assigned prefix and the value of every row after it (0, or row 0 of a lookup table)"""
    def __init__(self, prefix: List[int], fill: int = 0):
        self.prefix, self.fill = prefix, fill

    def dense(self, n: int) -> List[int]:
        return self.prefix + [self.fill] * (n - len(self.prefix))


PL_FIELD_MODULUS = 0x40000000000000000000000000000000224698fc094cf91b992d30ed00000001   # pasta Fp: the circuit field (test_utils.rs:2)


def columns_to_lists(advice: List[list]) -> List[List[int]]:
    """columns with None for unassigned cells -> dense lists just long enough to hold the assigned rows (create_proof zero-pads)"""
    out = []
    for col in advice:
        if not isinstance(col, list):          # a uint64 array of synthesize(arrays=True): every row of it is assigned
            out.append(col)
            continue
        m = len(col)
        if m and col[-1] is None:
            if col.count(None) == m:
                m = 0
            else:
                while col[m - 1] is None:
                    m -= 1
        dense = col[:m]
        if None in dense:
            dense = [0 if v is None else v for v in dense]
        out.append(dense)
    return out


def build(PL, trace: T.Trace, k: int, keygen_from_empty_circuit: bool = False, dense: bool = True, with_prog: bool = True,
          arrays: bool = False, **kw):
    """The whole of `TinyRamCircuit { trace }` + program_instance: returns (circuit, fixed, copies, advice, instances) ready for
    plonk.keygen / plonk.create_proof at n = 2^k (reference: mock_prover_test, circuits/mod.rs:364-375, uses k = 2 + W / 2).
    with_prog=False builds the reference's ExeCircuit (no program table, `instances` is empty).
    keygen_from_empty_circuit: the fixed columns are those of `TinyRamCircuit::default()` (trace: None), which is what
    gen_proofs_and_verify hands keygen_vk / keygen_pk (test_utils.rs:22-25): the execution table's selectors are then all off.
    dense=False leaves the fixed columns as FixedColumn (prefix, fill) pairs (large n).
    arrays=True (the upload path of bench.py): columns that are cheap to make as uint64 numpy arrays come back as such."""
    circ = TinyRamCircuit(PL, trace.word_bits, trace.reg_count, with_prog=with_prog)
    n = 1 << k
    fixed, copies, advice = circ.synthesize(trace, n, arrays=arrays, **kw)
    if keygen_from_empty_circuit:
        fixed, _, _ = circ.synthesize(None, n)
    instances = []
    if with_prog:
        instances = program_instance(trace.prog, trace.word_bits, trace.reg_count, arrays=arrays)
        circ.assign_instance(advice, instances)
    if dense:
        fixed = [f.dense(n) for f in fixed]
    return circ, fixed, copies, columns_to_lists(advice), instances


def device_columns(be, columns) -> list:
    """Upload columns to plonk.GpuBackend vectors.  columns: lists of canonical ints (zero-padded to n), uint64 arrays
    (build(arrays=True)) or FixedColumn.  Columns
    whose values all fit 64 bits take a fast path: the u64 values go up as limb 0 and are brought to Montgomery form on the device
    (one multiplication by R^2 through trp_dev_field_op)."""
    import numpy as np
    torch = be.torch
    r2 = be._dev(be._limbs([be.R]))
    out = []
    for col in columns:
        prefix, fill = (col.prefix, col.fill) if isinstance(col, FixedColumn) else (col, 0)
        if len(prefix) > be.n:
            raise ValueError("column longer than the domain")
        arr = _column_u64(prefix) if fill < 1 << 64 else None
        if arr is not None:
            v = torch.zeros((be.n, 4), dtype=torch.int64, device="cuda")       # only the assigned prefix crosses PCIe
            if fill:
                v[:, 0] = int(np.uint64(fill).view(np.int64)) if fill >= 1 << 63 else fill
            if len(arr):
                v[:len(arr), 0] = torch.from_numpy(arr.view(np.int64)).cuda()
            be.ctx.check(be.lib.trp_dev_field_op(be.ctx.handle, 0, 2 | 16, v.data_ptr(), r2.data_ptr(), v.data_ptr(), be.n))
        else:
            v = be.vec(prefix.tolist() if isinstance(prefix, np.ndarray) else prefix)
            if fill:
                v[len(prefix):] = be._dev(be._limbs([fill]))
        out.append(v)
    return out


def _column_u64(prefix):
    """the column as a contiguous uint64 array if every value fits 64 bits (device_columns' fast path), else None.  Columns that
    build(arrays=True) already made as uint64 arrays pass through without the list round trip."""
    import numpy as np
    if isinstance(prefix, np.ndarray):
        return np.ascontiguousarray(prefix) if prefix.dtype == np.uint64 else None
    if not prefix:
        return np.zeros(0, dtype=np.uint64)
    if max(prefix) >= 1 << 64:
        return None
    return np.array(prefix, dtype=np.uint64)


class HostWitness:
    """A proof's witness columns (instance + advice as synthesize() returns them) packed once into PINNED host memory, in the
    form that crosses PCIe: columns whose values fit 64 bits as u64 prefixes (the rows the circuit assigns), the few wide ones
    as 4 x u64 canonical limbs.  upload(be) is the per-proof host -> device step of the end-to-end path: two asynchronous
    copies, a scatter per column on the device and ONE multiplication by R^2 over the whole block (Montgomery form).
    bytes = what a proof sends over PCIe (bench.py's e2e.h2d_bytes_per_step)."""

    def __init__(self, be, columns):
        import numpy as np
        torch = be.torch
        self.n, self.ncols = be.n, len(columns)
        narrow, wide, self.meta = [], [], []
        off_n = off_w = 0
        for col in columns:
            if isinstance(col, FixedColumn):
                raise ValueError("witness columns only (fixed columns are key material)")
            if len(col) > be.n:
                raise ValueError("column longer than the domain")
            arr = _column_u64(col)
            if arr is not None:
                self.meta.append((0, off_n, len(arr))); narrow.append(arr); off_n += len(arr)
            else:
                vals = col.tolist() if isinstance(col, np.ndarray) else col
                limbs = np.frombuffer(b"".join((v % be.p).to_bytes(32, "little") for v in vals), dtype=np.uint64).reshape(len(vals), 4)
                self.meta.append((1, off_w, len(vals))); wide.append(limbs); off_w += len(vals)
        cat = lambda parts, shape: np.concatenate(parts) if parts else np.zeros(shape, dtype=np.uint64)
        self.narrow = torch.from_numpy(cat(narrow, (0,)).view(np.int64)).pin_memory()
        self.wide = torch.from_numpy(cat(wide, (0, 4)).view(np.int64).reshape(-1, 4)).pin_memory()
        self.bytes = self.narrow.numel() * 8 + self.wide.numel() * 8

    def upload(self, be, out=None):
        """-> (ncols, n, 4) device block of Montgomery columns (views of it are plonk.GpuBackend vectors)"""
        torch = be.torch
        d_n = self.narrow.cuda(non_blocking=True)
        d_w = self.wide.cuda(non_blocking=True)
        if out is None:
            out = torch.empty((self.ncols, self.n, 4), dtype=torch.int64, device="cuda")
        out.zero_()
        for c, (kind, off, ln) in enumerate(self.meta):
            if not ln:
                continue
            if kind == 0:
                out[c, :ln, 0] = d_n[off:off + ln]
            else:
                out[c, :ln] = d_w[off:off + ln]
        r2 = be._dev(be._limbs([be.R]))
        be.ctx.check(be.lib.trp_dev_field_op(be.ctx.handle, 0, 2 | 16, out.data_ptr(), r2.data_ptr(), out.data_ptr(), self.ncols * self.n))
        return out
