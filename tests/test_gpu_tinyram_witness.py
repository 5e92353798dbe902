"""GPU tests of tinyram.device_witness (trp_dev_tinyram_witness): the witness block made on the device from the packed trace must
equal the host path's block -- tinyram.build + HostWitness.upload -- bit for bit, a k = 20 proof made from it must be byte for byte
the proof made from the host block, and the failures of synthesize must come back as the same exceptions."""
import dataclasses
import importlib.util
import os

import pytest

import tinyram_programs as TP

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))


@pytest.fixture(scope="module")
def env():
    import __graft_entry__ as ge
    pkg = ge.load_package()
    from tiny_ram_halo2_b200 import programs, tinyram, trace
    return pkg, pkg.plonk, tinyram, trace, programs, pkg.Context(0, pkg.VESTA)


_backends = {}


def _backend(env, k):
    pkg, PL, TR, T, programs, ctx = env
    if k not in _backends:
        _backends[k] = PL.GpuBackend(ctx, k, 6)
    return _backends[k]


def _cases(env):
    pkg, PL, TR, T, programs, ctx = env
    spec = importlib.util.spec_from_file_location("make_witness_digests", os.path.join(HERE, "golden", "make_witness_digests.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    out = []
    for name, (tr, k) in mod.cases(T, programs).items():
        out.append((name, tr, k, {}))
        if name in ("load_and_answer_w8", "loop_w8", "loop_w16_short"):
            out += [(name + "/exe", tr, k, {"with_prog": False}), (name + "/reg_index", tr, k, {"reg_operand_value": False})]
    return out


def _host_block(env, be, tr, k, **kw):
    PL, TR = env[1], env[2]
    _, _, _, adv, inst = TR.build(PL, tr, k, dense=False, arrays=True, **kw)
    return TR.HostWitness(be, list(inst) + list(adv)).upload(be)


def test_device_block_equals_host_block(env):
    """every trace of make_witness_digests (bench.py's 65 521-step trace at k = 20 included) and its /exe and /reg_index variants,
    plus the single-instruction programs with register operands"""
    import torch
    pkg, PL, TR, T, programs, ctx = env
    cases = _cases(env)
    for W in (8, 16):
        for name in TP.THREE_OPERAND + TP.TWO_OPERAND:
            ins = getattr(T, name)(1, 0, T.Reg(0)) if name in TP.THREE_OPERAND else getattr(T, name)(0, T.Reg(0))
            cases.append((f"{name}_reg_w{W}", TP.mov_ins_answer(T, W, ins, 3 if name in ("Shl", "Shr") else 0xA5), W // 2 + 2, {}))
    for name, tr, k, kw in cases:
        be = _backend(env, k)
        want = _host_block(env, be, tr, k, **kw)
        got = TR.device_witness(be, tr, **kw)
        assert got.shape == want.shape and torch.equal(got, want), name
        del got, want


def test_out_buffer_reuse(env):
    import torch
    pkg, PL, TR, T, programs, ctx = env
    tr = programs.counting_loop(16, 3, programs.mixed_body(16))
    be = _backend(env, 11)
    first = TR.device_witness(be, tr)
    buf = torch.full_like(first, -1)
    again = TR.device_witness(be, tr, out=buf)
    assert again.data_ptr() == buf.data_ptr() and torch.equal(again, first)
    with pytest.raises(ValueError):
        TR.device_witness(be, tr, out=buf[:, :10])
    with pytest.raises(ValueError):
        TR.device_witness(be, tr, a_flag_rand=lambda: 1)


def test_failures_raise_the_host_exceptions(env):
    """the trace edits of tests/test_tinyram_witness_cpu.py: the same exception as build(), at the same row"""
    pkg, PL, TR, T, programs, ctx = env
    be = _backend(env, 6)

    def step(tr, i, **regs):
        exe = list(tr.exe)
        r = list(exe[i].regs)
        for name, v in regs.items():
            r[int(name[1:])] = v
        exe[i] = dataclasses.replace(exe[i], regs=tuple(r))
        return dataclasses.replace(tr, exe=exe)

    shl = TP.mov_ins_answer(T, 8, T.Shl(1, 0, T.Reg(2)), 5)
    add = TP.mov_named(T, 8, "Add", 7, 9)
    cases = [(step(shl, 2, r1=shl.exe[2].regs[1] ^ 1), AssertionError, 1),
             (dataclasses.replace(add, exe=add.exe[:2]), IndexError, 1),
             (step(step(shl, 1, r2=70), 2, r1=0), OverflowError, 1)]
    for tr, exc, row in cases:
        with pytest.raises(exc):
            TR.build(PL, tr, 6)
        with pytest.raises(exc) as got:
            TR.device_witness(be, tr)
        assert got.value.row == row
    bad_prog = dataclasses.replace(add, prog=add.prog[:-1])                 # the program must end with Answer: program_instance's check
    with pytest.raises(ValueError):
        TR.build(PL, bad_prog, 6)
    with pytest.raises(ValueError):
        TR.device_witness(be, bad_prog)


def test_k20_proof_from_the_device_block(env):
    """bench.py's trace at k = 20: the proof from the device block, with the reproducible RNG at a fixed seed, is byte for byte the
    proof from the host block, and the package's verifier accepts it"""
    from tiny_ram_halo2_b200 import rng as RNG, verifier as V
    pkg, PL, TR, T, programs, ctx = env
    k = 20
    be = _backend(env, k)
    tr = programs.longest_loop(32)
    circ, fixed, copies, adv, inst = TR.build(PL, tr, k, dense=False, arrays=True)
    pk = PL.keygen(be, circ.cs, TR.device_columns(be, fixed), copies)
    n_inst = len(inst)
    host = TR.HostWitness(be, list(inst) + list(adv)).upload(be)
    proofs = []
    for block in (host, TR.device_witness(be, tr)):
        cols = [block[i] for i in range(block.shape[0])]
        rng = RNG.ScalarStreamRng(be.p, bytes(range(32)))
        proofs.append(PL.create_proof(be, pk, cols[:n_inst], cols[n_inst:], rng, PL.Blake2bWrite(be.q, be.p)))
    assert proofs[0] == proofs[1]
    V.verify_proof(be, pk.vk, V.SingleVerifier(be), [host[i] for i in range(n_inst)], V.Blake2bRead(proofs[1], be.q, be.p))
