"""The Montgomery product of csrc/ff.cuh defers two carries per reduction round (the m*p2 carry caught in one register, and
m >> 2 of the 2^254 term carried into the next round's word).  These tests drive every product through its plain-C twin on
operands that push those carries and the top words to their bounds, and check each result against Python big ints."""
import ctypes
import os
import random
import subprocess

import numpy as np
import pytest

import pasta_model as pm
import oracle as O

HERE = os.path.dirname(os.path.abspath(__file__))


@pytest.fixture(scope="module")
def shim(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("ff_carry") / "ff_host_shim.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-x", "c++", os.path.join(HERE, "ff_host_shim.cpp"), "-o", so])
    return ctypes.CDLL(so)


def _run(shim, fid, op, a, b):
    A = O.ints_to_limbs(a); B = O.ints_to_limbs(b); R = np.zeros_like(A)
    shim.ffh_op(fid, op, A.ctypes.data_as(ctypes.c_void_p), B.ctypes.data_as(ctypes.c_void_p),
                R.ctypes.data_as(ctypes.c_void_p), ctypes.c_size_t(len(a)))
    return O.limbs_to_ints(R)


def _edges(F):
    p = F.p
    e = [0, 1, 2, p - 1, p - 2, p - 3, (p - 1) // 2, (p + 1) // 2, (1 << 254) - 1, 1 << 254, F.R, F.R2, F.Rinv, F.R * F.R2 % p,
         (1 << 32) - 1, (1 << 64) - 1, (1 << 128) - 1, (1 << 224) - 1]
    # all-ones low limbs below p: p - 1 with its low k 32-bit limbs set to ones, and 2^254 - 1 with its low limbs cleared
    for k in range(1, 8):
        ones = (1 << (32 * k)) - 1
        e += [x for x in ((p - 1) | ones, ((1 << 254) - 1) & ~ones, p - 1 - ones) if 0 <= x < p]
    # the top word at its maximum below p with every lower limb at 0 or all ones
    e += [(p >> 224) << 224, ((p >> 224) << 224) - 1]
    return sorted({x % p for x in e})


@pytest.mark.parametrize("fid,F", [(0, pm.Fp), (1, pm.Fq)])
def test_mul_and_sqr_at_carry_bounds(shim, fid, F):
    p, Ri = F.p, F.Rinv
    edge = _edges(F)
    a = [x for x in edge for _ in edge]
    b = [y for _ in edge for y in edge]
    assert _run(shim, fid, 2, a, b) == [x * y * Ri % p for x, y in zip(a, b)]
    assert _run(shim, fid, 4, edge, edge) == [x * x * Ri % p for x in edge]


@pytest.mark.parametrize("fid,F", [(0, pm.Fp), (1, pm.Fq)])
def test_mul_and_sqr_random(shim, fid, F):
    p, Ri = F.p, F.Rinv
    rnd = random.Random(1234 + fid)
    # uniform operands, and operands whose limbs are each 0, 1, 2^32 - 2 or 2^32 - 1 (most carries out of every limb)
    extreme = lambda: sum(rnd.choice((0, 1, 0xfffffffe, 0xffffffff)) << (32 * i) for i in range(8)) % p
    a = [rnd.randrange(p) for _ in range(3000)] + [extreme() for _ in range(3000)]
    b = [rnd.randrange(p) for _ in range(3000)] + [extreme() for _ in range(3000)]
    assert _run(shim, fid, 2, a, b) == [x * y * Ri % p for x, y in zip(a, b)]
    assert _run(shim, fid, 4, a, b) == [x * x * Ri % p for x in a]


@pytest.mark.parametrize("fid,F", [(0, pm.Fp), (1, pm.Fq)])
def test_mont_conversions_and_inverse(shim, fid, F):
    p, Ri = F.p, F.Rinv
    edge = _edges(F)
    assert _run(shim, fid, 5, edge, edge) == [x * Ri % p for x in edge]
    assert _run(shim, fid, 6, edge, edge) == [x * F.R % p for x in edge]
    for x, r in zip(edge, _run(shim, fid, 3, edge, edge)):
        assert r == 0 if x == 0 else r * x * Ri % p == F.R
