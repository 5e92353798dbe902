"""CPU tests of the TinyRAM witness generator's row logic (csrc/tinyram_witness.h: the code trp_dev_tinyram_witness runs one thread
per trace step).  Its host build (tests/tinyram_witness_host_shim.cpp), fed the packed inputs the device gets
(tinyram.witness_inputs), must give tinyram.build's instance and advice columns bit for bit, and must fail where synthesize fails,
with the same exception and at the same trace row."""
import ctypes
import dataclasses
import importlib.util
import os
import random
import subprocess

import numpy as np
import pytest

import tinyram_programs as TP

HERE = os.path.dirname(os.path.abspath(__file__))
SO = os.path.join(HERE, "_tinyram_witness_host_shim.so")


@pytest.fixture(scope="module")
def mods():
    import __graft_entry__ as ge
    ge.load_package()
    from tiny_ram_halo2_b200 import plonk, programs, tinyram, trace
    return plonk, tinyram, trace, programs


@pytest.fixture(scope="module")
def shim():
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-x", "c++", os.path.join(HERE, "tinyram_witness_host_shim.cpp"),
                           "-o", SO])
    lib = ctypes.CDLL(SO)
    vp, sz, u = ctypes.c_void_p, ctypes.c_size_t, ctypes.c_uint
    lib.trw_host_run.argtypes = [u, u, ctypes.c_int, vp, sz, vp, vp, sz, vp, vp, sz]
    lib.trw_host_run.restype = ctypes.c_uint64
    return lib


def witness_cases(mods):
    """make_witness_digests.cases (the traces whose witness digests are frozen) and the option variants it digests"""
    PL, TR, T, programs = mods
    spec = importlib.util.spec_from_file_location("make_witness_digests", os.path.join(HERE, "golden", "make_witness_digests.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    out = []
    for name, (tr, k) in mod.cases(T, programs).items():
        out.append((name, tr, {}))
        if name in ("load_and_answer_w8", "loop_w8", "loop_w16_short"):
            out += [(name + "/exe", tr, {"with_prog": False}), (name + "/reg_index", tr, {"reg_operand_value": False})]
    return out


def limbs_of(values):
    """canonical ints -> (len, 4) uint64 limbs"""
    return np.frombuffer(b"".join(int(v).to_bytes(32, "little") for v in values), dtype=np.uint64).reshape(-1, 4)


def ints_of(limbs):
    raw = np.ascontiguousarray(limbs).tobytes()
    return [int.from_bytes(raw[i:i + 32], "little") for i in range(0, len(raw), 32)]


def host_block(mods, shim, tr, with_prog=True, reg_operand_value=True):
    """the shim's (n_cols, rows, 4) canonical block, a_flag inverted as trp_dev_tinyram_witness inverts it; raises the
    witness generator's failure as tinyram.witness_error"""
    PL, TR, T, _ = mods
    circ = TR.TinyRamCircuit(PL, tr.word_bits, tr.reg_count, with_prog=with_prog)
    steps, ins, prog, cm = TR.witness_inputs(circ, tr)
    rows = max(circ.table_len, len(tr.exe) + 1)
    out = np.zeros((circ.cs.num_instance + circ.cs.num_advice, rows, 4), dtype=np.uint64)
    vp = lambda a: a.ctypes.data_as(ctypes.c_void_p)
    err = shim.trw_host_run(circ.W, circ.R, int(reg_operand_value) | (2 if with_prog else 0), vp(steps), len(steps), vp(ins), vp(prog),
                            len(prog), vp(cm), vp(out), rows)
    if err:
        raise TR.witness_error(err & 0xFF, (err >> 8) & 0xFFFFFFFF)
    ne, col = len(tr.exe), out[cm[4]]
    col[:ne] = limbs_of(TR._batch_inverse(ints_of(col[:ne]), TR.PL_FIELD_MODULUS)).reshape(ne, 4)
    return out


def expected_block(mods, tr, rows, **kw):
    """tinyram.build's instance + advice columns as a zero-padded (n_cols, rows, 4) block of canonical limbs"""
    PL, TR, T, _ = mods
    k = max(tr.word_bits // 2, (rows - 1).bit_length())
    _, _, _, adv, inst = TR.build(PL, tr, k, dense=False, arrays=True, **kw)
    cols = list(inst) + list(adv)
    out = np.zeros((len(cols), rows, 4), dtype=np.uint64)
    for c, col in enumerate(cols):
        arr = TR._column_u64(col)
        if arr is not None:
            out[c, :len(arr), 0] = arr
        elif len(col):
            out[c, :len(col)] = limbs_of(list(col))
    return out


def assert_same(got, want, what):
    if not np.array_equal(got, want):
        c, r = np.argwhere((got != want).any(axis=2))[0]
        raise AssertionError(f"{what}: first difference at block column {c}, row {r}: {ints_of(got[c, r])} != {ints_of(want[c, r])}")


def check_trace(mods, shim, tr, what, **kw):
    got = host_block(mods, shim, tr, **kw)
    assert_same(got, expected_block(mods, tr, got.shape[1], **kw), what)


def test_equals_build_on_the_frozen_witness_cases(mods, shim):
    """every trace of make_witness_digests (W = 8 / 16 / 32, bench.py's 65 521-step trace included) and its /exe and /reg_index
    variants"""
    for name, tr, kw in witness_cases(mods):
        check_trace(mods, shim, tr, name, **kw)


@pytest.mark.parametrize("W", [8, 16, 24])
def test_equals_build_on_single_instruction_programs(mods, shim, W):
    """every single-instruction program of tests/tinyram_programs.py, immediate and register operands, both reg_operand_value
    settings (W = 32 is the frozen cases' and the random programs')"""
    PL, TR, T, _ = mods
    rnd = random.Random(W)
    top = 1 << W
    for name in TP.THREE_OPERAND + TP.TWO_OPERAND:
        for _ in range(3):
            a = rnd.randrange(1, min(W, 32)) if name in ("Shl", "Shr") else rnd.randrange(top)
            b = rnd.randrange(top)
            check_trace(mods, shim, TP.mov_named(T, W, name, a, b), f"{name} W={W} a={a} b={b}")
            ctor = getattr(T, name)                                   # the operand in register 0, which Mov loads with b
            ins = ctor(1, 0, T.Reg(0)) if name in TP.THREE_OPERAND else ctor(0, T.Reg(0))
            if name in ("Shl", "Shr"):
                b = rnd.randrange(1, min(W, 32))
            tr = TP.mov_ins_answer(T, W, ins, b)
            for rov in (True, False):
                check_trace(mods, shim, tr, f"{name} W={W} reg operand, b={b}, reg_operand_value={rov}", reg_operand_value=rov)
    check_trace(mods, shim, TP.answer_only(T, W), f"answer_only W={W}")
    check_trace(mods, shim, TP.load_and_answer(T, W, 1, 2), f"load_and_answer W={W}")


def test_equals_build_on_random_programs(mods, shim):
    """random straight-line programs over every instruction (all eight registers, Not's 32-bit result included)"""
    PL, TR, T, _ = mods
    rnd = random.Random(99)
    three = TP.THREE_OPERAND
    two = ("Cmpe", "Cmpa", "Cmpae", "Cmpg", "Cmpge", "Mov", "CMov", "Not")
    for trial in range(40):
        W = rnd.choice((8, 16, 24, 32))
        prog = [T.Mov(rnd.randrange(8), T.Imm(rnd.randrange(1 << W))) for _ in range(3)]
        for _ in range(rnd.randrange(1, 11)):                           # at most 14 steps: TABLE_LEN - 1 at W = 8
            if rnd.random() < 0.5:
                name = rnd.choice(three)
                operand = T.Imm(rnd.randrange(1, 8)) if name in ("Shl", "Shr") else (
                    T.Imm(rnd.randrange(1 << W)) if rnd.random() < 0.6 else T.Reg(rnd.randrange(8)))
                prog.append(getattr(T, name)(rnd.randrange(8), rnd.randrange(8), operand))
            else:
                operand = T.Imm(rnd.randrange(1 << W)) if rnd.random() < 0.6 else T.Reg(rnd.randrange(8))
                prog.append(getattr(T, rnd.choice(two))(rnd.randrange(8), operand))
        prog.append(T.Answer(T.Imm(1)))
        try:
            tr = T.eval_program(prog, T.Mem(W, [1]))
        except AssertionError:                                          # SMulh of a register beyond the word (trace.smulh_eval)
            continue
        check_trace(mods, shim, tr, f"trial {trial}", reg_operand_value=rnd.random() < 0.7)


def _with_step(tr, i, **changes):
    exe = list(tr.exe)
    exe[i] = dataclasses.replace(exe[i], **changes)
    return dataclasses.replace(tr, exe=exe)


def _regs(step, **set_):
    regs = list(step.regs)
    for r, v in set_.items():
        regs[int(r[1:])] = v
    return tuple(regs)


def _same_failure(mods, shim, tr, exc, row, **kw):
    PL, TR, T, _ = mods
    with pytest.raises(exc):
        TR.build(PL, tr, max(6, tr.word_bits // 2 + 1), **kw)
    with pytest.raises(exc) as got:
        host_block(mods, shim, tr, **kw)
    assert got.value.row == row, (got.value, row)
    return got.value


def test_failures_match_synthesize(mods, shim):
    """each failure synthesize can meet, on traces edited after the interpreter: the same exception type, at the known row"""
    PL, TR, T, _ = mods
    W = 8
    shl = TP.mov_ins_answer(T, W, T.Shl(1, 0, T.Reg(2)), 5)               # Mov r0 5; Shl r1 r0 r2; Answer
    shr = TP.mov_ins_answer(T, W, T.Shr(1, 0, T.Reg(2)), 200)
    # Shl / Shr: the next step does not hold the shifted register (AssertionError at the shift's row)
    for tr in (shl, shr):
        bad = _with_step(tr, 2, regs=_regs(tr.exe[2], r1=tr.exe[2].regs[1] ^ 1))
        _same_failure(mods, shim, bad, AssertionError, 1)
    # a trace cut after a step whose temporary variables read the next step (IndexError)
    add = TP.mov_named(T, W, "Add", 7, 9)
    _same_failure(mods, shim, dataclasses.replace(add, exe=add.exe[:2]), IndexError, 1)
    _same_failure(mods, shim, dataclasses.replace(shl, exe=shl.exe[:2]), IndexError, 1)
    # a shift by 64 or more (OverflowError in the gadget phase), behind an earlier failure-free row
    for tr in (shl, shr):
        big = _with_step(_with_step(tr, 1, regs=_regs(tr.exe[1], r2=70)), 2, regs=_regs(tr.exe[2], r1=0))
        _same_failure(mods, shim, big, OverflowError, 1)
    # a temporary-variable failure beats a gadget failure of an earlier row
    two = [T.Mov(0, T.Imm(5)), T.Shl(1, 0, T.Reg(2)), T.Add(3, 0, T.Imm(1)), T.Answer(T.Imm(1))]
    tr = T.eval_program(two, T.Mem(W, [1]))
    tr = _with_step(_with_step(tr, 1, regs=_regs(tr.exe[1], r2=70)), 2, regs=_regs(tr.exe[2], r1=0))
    _same_failure(mods, shim, dataclasses.replace(tr, exe=tr.exe[:3]), IndexError, 2)
    # SMulh's sign assertion (trace.smulh_eval) on a register beyond the word, as Not leaves one
    y = next(y for y in range(256, 1 << 16) if _smulh_fails(T, 4, y, W))
    sm = TP.mov_ins_answer(T, W, T.SMulh(1, 0, T.Imm(4)), 3)
    _same_failure(mods, shim, _with_step(sm, 1, regs=_regs(sm.exe[1], r0=y)), AssertionError, 1)


def _smulh_fails(T, a, b, W):
    try:
        T.smulh_eval(a, b, W)
    except AssertionError:
        return True
    return False


def test_shifts_beyond_the_word(mods, shim):
    """shift amounts in [W, 64): Shl's tc beyond 64 bits and Shr's td as a full field element, against build"""
    PL, TR, T, _ = mods
    for W, amount in ((8, 8), (8, 40), (32, 33), (32, 63), (16, 3)):
        for name in ("Shl", "Shr"):
            tr = TP.mov_ins_answer(T, W, getattr(T, name)(1, 0, T.Reg(2)), 0xB7)
            tr = _with_step(_with_step(tr, 1, regs=_regs(tr.exe[1], r2=amount)), 2,
                            regs=_regs(tr.exe[2], r1=(0xB7 << amount) & ((1 << W) - 1) if name == "Shl" else 0xB7 >> amount))
            check_trace(mods, shim, tr, f"{name} by {amount} at W={W}")


def test_unhandled_nondeterministic_advice(mods, shim, monkeypatch):
    """RuntimeError("Unhandled non-deterministic advice"): no instruction selects it, so the selection table is patched -- for
    build and for the packed instruction table alike -- to ask for non-deterministic advice where none is defined"""
    PL, TR, T, _ = mods
    orig = TR.selections

    def patched(ins):
        s = orig(ins)
        return (s[0], s[1], s[2], ("NonDet",)) + s[4:] if ins.name == "Add" else s
    monkeypatch.setattr(TR, "selections", patched)
    tr = T.eval_program([T.Mov(0, T.Imm(1)), T.Mov(1, T.Imm(2)), T.Add(2, 0, T.Imm(3)), T.Answer(T.Imm(1))], T.Mem(8, [1]))
    _same_failure(mods, shim, tr, RuntimeError, 2)


def test_packed_inputs(mods):
    """the formats of include/tr_prover.h: one instruction row per distinct instruction, L = 9 R + 22 line values, the column map's
    roles on the configured columns"""
    PL, TR, T, programs = mods
    tr = programs.counting_loop(16, 3, programs.mixed_body(16))
    circ = TR.TinyRamCircuit(PL, 16, 8)
    steps, ins, prog, cm = TR.witness_inputs(circ, tr)
    L = 9 * 8 + 22
    assert steps.shape == (len(tr.exe), 12) and ins.shape == (len(set(tr.prog)), 16 + L + 13) and len(prog) == len(tr.prog)
    assert [int(x) for x in steps[:, 0]] == [st.pc for st in tr.exe]
    assert all(int(ins[int(steps[i, 3]), 0]) == st.instruction.opcode for i, st in enumerate(tr.exe))
    assert all(int(prog[st.pc]) == int(steps[i, 3]) for i, st in enumerate(tr.exe))
    n_inst = circ.cs.num_instance
    assert cm[0] == n_inst + circ.pc and cm[4] == n_inst + circ.a_flag
    assert len(cm) == 60 + 8 + 13 + 3 * L + 1 + len(circ.intermediate)
    assert list(cm[60 + 8 + 13 + 2 * L:60 + 8 + 13 + 3 * L]) == circ.prog_input.to_vec()
    with pytest.raises(ValueError):
        TR.witness_inputs(circ, T.eval_program([T.Mov(0, T.Imm(1 << 32)), T.Answer(T.Imm(1))], T.Mem(16, [1])))
