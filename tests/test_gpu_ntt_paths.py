"""GPU tests of the NTT's device-resident entry points (the ones the prover calls) at the sizes where the pass plan changes
shape, each against the oracle bit for bit, in both fields.

A transform of 2^L values runs ceil(L / 10) passes.  The plans and the kernels their passes launch:

    2^0 .. 2^10   one generic pass                                  test_gpu_parity.py::test_best_fft, test_dev_ntt (10)
    2^11 .. 2^18  two generic passes                                test_best_fft, test_dev_ntt (11, 18)
    2^19          a specialised first pass (s = 10, c = 1) and a    test_best_fft, test_dev_ntt (19),
                  generic second one (lo = 10, s = 9, c = 2)        test_dev_domain_transforms (k or extended_k = 19)
    2^20          two specialised passes                            test_best_fft, test_dev_ntt (20),
                                                                    test_dev_domain_transforms (k or extended_k = 20)
    2^21 .. 2^24  three generic passes (the last one of 7 stages    test_best_fft, test_dev_ntt (21),
                  at 2^21 and 2^23)                                 test_gpu_parity.py::test_best_fft_2_22_2_24

The 7 specialised instances of ntt_pass_spec_kernel per field (csrc/ntt.cu), and what launches each of them:

    first pass, no scaling            trp_dev_ntt at 2^19 / 2^20 (test_dev_ntt, test_dev_ntt_chunks_of_128_columns);
                                      trp_dev_extended_to_coeff without the division at extended_k 19 / 20
                                      (test_dev_domain_transforms)
    first pass, one scalar            trp_dev_extended_to_coeff with the division at (j, k) = (2, 19), (2, 20): the extended
                                      domain is the domain, so 1 / (X^n - 1) is one constant (test_dev_domain_transforms)
    first pass, table                 trp_dev_coeff_to_coset at k = 19 / 20, in and out of place
                                      (test_dev_ntt_chunks_of_128_columns; test_gpu_proof_size_paths.py::test_coset_gather_k20,
                                      test_coset_gather_k19_k20)
    first pass, gathered, table       trp_dev_coeff_to_coset_gather at k = 19 / 20 (test_coset_gather_k20, test_coset_gather_k19_k20)
    last pass, no scaling             trp_dev_ntt at 2^20; trp_dev_coeff_to_extended at extended_k = 20 (test_dev_domain_transforms)
    last pass, one scalar             trp_dev_lagrange_to_coeff at k = 20 (1 / n; test_dev_domain_transforms,
                                      test_dev_ntt_chunks_of_128_columns)
    last pass, table                  trp_dev_cosets_to_coeff_parts at k = 20 (the coset-power inverses;
                                      test_gpu_proof_size_paths.py::test_cosets_to_coeff_parts_against_the_oracle)

trp_dev_coeff_to_extended pads its input and trp_dev_extended_to_coeff truncates its output with a period-3 scaling (zeta), so
those passes run the generic kernel whatever the size: at extended_k = 20 a generic first pass and a specialised last one for
coeff_to_extended, the reverse for extended_to_coeff, and two generic passes for extended_to_coeff with the division at j > 2
(the divisor table has period 2^(extended_k - k)).

dev_ntt_inplace and the in-place trp_dev_coeff_to_coset split a batch into chunks whose scratch fits 4 GiB: 128 columns at
k = 20.  A proof's 263 advice columns cross that boundary twice; test_dev_ntt_chunks_of_128_columns crosses it once."""
import gc

import numpy as np
import pytest

from util import O, FIELDS

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def pkg():
    import __graft_entry__ as ge
    return ge.load_package()


@pytest.fixture(scope="module")
def ctxs(pkg):
    return {O.VESTA: pkg.Context(0, pkg.VESTA), O.PALLAS: pkg.Context(0, pkg.PALLAS)}


def _u64(t):
    return t.cpu().numpy().view(np.uint64)


def _dev(arr):
    import torch
    return torch.from_numpy(np.ascontiguousarray(arr).view(np.int64)).cuda()


def _free_device_memory():
    import torch
    gc.collect()
    torch.cuda.empty_cache()


def _root(field, log_n):
    return O.to_mont(field, O.ints_to_limbs([FIELDS[field].root_of_unity(log_n)]))[0]


def _times(field, col, lam):
    """lam * col, with the oracle's multiplication"""
    return O.field_op(field, "mul", col, np.ascontiguousarray(np.broadcast_to(lam, col.shape)))


# ---- trp_dev_ntt -------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("curve", [O.VESTA, O.PALLAS])
@pytest.mark.parametrize("log_n", [10, 11, 18, 19, 20, 21])
def test_dev_ntt(pkg, ctxs, curve, log_n):
    """three columns in place: uniform values; every value p - 1 (the largest carries into every butterfly's add); one value at
    index 2^(L-1) + 2^10 + 3 and zeros elsewhere, whose set bits are butterflied in every pass, so its transform v * omega^(i j)
    shows a wrong twiddle exponent at the output index it lands on"""
    from tiny_ram_halo2_b200._lib import ptr
    import torch
    ctx, field = ctxs[curve], O.SCALAR_FIELD[curve]
    n = 1 << log_n
    omega = _root(field, log_n)
    cols = np.zeros((3, n, 4), dtype=np.uint64)
    cols[0] = O.random_field_mont(field, n, 800 + log_n)
    cols[1] = O.ints_to_limbs([O.MODULUS[field] - 1])
    imp = ((1 << (log_n - 1)) | (1 << 10) | 3) & (n - 1)
    cols[2, imp] = O.random_field_mont(field, 1, 900 + log_n)[0]
    d = _dev(cols)
    torch.cuda.synchronize()
    ctx.check(ctx.lib.trp_dev_ntt(ctx.handle, d.data_ptr(), 3, log_n, ptr(omega)))
    ctx.sync()
    got = _u64(d)
    for c in range(3):
        assert np.array_equal(got[c], O.fft(field, cols[c], log_n, omega)), c
    del d
    _free_device_memory()


# ---- the EvaluationDomain transforms at extended_k = 19 and 20 --------------------------------------------------------------------
@pytest.mark.parametrize("curve", [O.VESTA, O.PALLAS])
@pytest.mark.parametrize("j,k", [(6, 17), (5, 18), (3, 19), (2, 19), (2, 20)])
def test_dev_domain_transforms(pkg, ctxs, curve, j, k):
    """trp_dev_lagrange_to_coeff (in place), trp_dev_coeff_to_extended (the destination holds the intermediate) and
    trp_dev_extended_to_coeff with the division off and on, on device tensors, against the oracle's EvaluationDomain"""
    import torch
    ctx, field = ctxs[curve], O.SCALAR_FIELD[curve]
    dom = pkg.EvaluationDomain(ctx, j, k)
    ek, n = dom.extended_k, 1 << k
    assert ek == O.domain_info(field, j, k)[0] and ek in (19, 20)
    lag = O.random_field_mont(field, 2 * n, 1000 + 10 * j + k).reshape(2, n, 4)
    d = _dev(lag)
    torch.cuda.synchronize()
    ctx.check(ctx.lib.trp_dev_lagrange_to_coeff(dom.handle, d.data_ptr(), 2))
    ctx.sync()
    coeff = O.lagrange_to_coeff(field, j, k, lag).reshape(2, n, 4)
    assert np.array_equal(_u64(d), coeff)

    coeff = O.random_field_mont(field, 2 * n, 1100 + 10 * j + k).reshape(2, n, 4)
    src = _dev(coeff)
    ext = torch.full((2, 1 << ek, 4), -1, dtype=torch.int64, device="cuda")
    torch.cuda.synchronize()
    ctx.check(ctx.lib.trp_dev_coeff_to_extended(dom.handle, src.data_ptr(), ext.data_ptr(), 2))
    ctx.sync()
    assert np.array_equal(_u64(ext), O.coeff_to_extended(field, j, k, coeff))
    assert np.array_equal(_u64(src), coeff)
    del src, ext

    h = O.random_field_mont(field, 1 << ek, 1200 + 10 * j + k)
    for divide in (0, 1):
        d_h = _dev(h)
        out = torch.full(((j - 1) * n, 4), -1, dtype=torch.int64, device="cuda")
        torch.cuda.synchronize()
        ctx.check(ctx.lib.trp_dev_extended_to_coeff(dom.handle, d_h.data_ptr(), out.data_ptr(), divide))
        ctx.sync()
        assert np.array_equal(_u64(out), O.extended_to_coeff(field, j, k, h, divide=divide)), divide
    dom.free()
    del d, d_h, out
    _free_device_memory()


# ---- the 128-column chunks of a k = 20 batch ----------------------------------------------------------------------------------------
@pytest.mark.parametrize("curve", [O.VESTA, O.PALLAS])
def test_dev_ntt_chunks_of_128_columns(pkg, curve):
    """130 columns at k = 20 (chunks of 128 + 2) through trp_dev_lagrange_to_coeff, then trp_dev_ntt and then trp_dev_coeff_to_coset
    in place on the last coset, each on the previous one's output.  Column c is lam_c * a_(c mod 3) for three random columns a_r,
    so by linearity the exact reference of every column is lam_c times the oracle's transform of a_(c mod 3)"""
    import torch
    from tiny_ram_halo2_b200._lib import ptr
    field, j, k, m = O.SCALAR_FIELD[curve], 6, 20, 130
    n = 1 << k
    ctx = pkg.Context(0, curve)                  # its own scratch (4 GiB at this size), released when the test ends
    try:
        dom = pkg.EvaluationDomain(ctx, j, k)
        period = dom.extended_len() // n
        a = [O.random_field_mont(field, n, 1300 + r) for r in range(3)]
        lam = O.random_field_mont(field, m, 1310)
        d = torch.empty((m, n, 4), dtype=torch.int64, device="cuda")
        for c in range(m):
            d[c] = _dev(_times(field, a[c % 3], lam[c]))

        def check(step, ref):
            for c in range(m):
                assert np.array_equal(_u64(d[c]), _times(field, ref[c % 3], lam[c])), (step, c)

        torch.cuda.synchronize()
        ctx.check(ctx.lib.trp_dev_lagrange_to_coeff(dom.handle, d.data_ptr(), m))
        ctx.sync()
        ref = [O.lagrange_to_coeff(field, j, k, x) for x in a]
        check("lagrange_to_coeff", ref)
        ctx.check(ctx.lib.trp_dev_ntt(ctx.handle, d.data_ptr(), m, k, ptr(dom.omega)))
        ctx.sync()
        ref = [O.fft(field, x, k, dom.omega) for x in ref]
        check("ntt", ref)
        ctx.check(ctx.lib.trp_dev_coeff_to_coset(dom.handle, d.data_ptr(), d.data_ptr(), m, period - 1))
        ctx.sync()
        ref = [O.coeff_to_extended(field, j, k, x)[0, period - 1::period].copy() for x in ref]
        check("coeff_to_coset", ref)
        dom.free()
        del d
    finally:
        ctx.close()
        _free_device_memory()
