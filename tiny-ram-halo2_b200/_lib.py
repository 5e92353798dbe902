"""ctypes binding of libtrp.so (include/tr_prover.h).  Fails loudly when the library or a GPU is missing."""
from __future__ import annotations

import ctypes
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "libtrp.so")

PALLAS, VESTA = 0, 1
Q_CONTIGUOUS = 0x10000

TRP_OK, TRP_E_INVALID, TRP_E_CUDA, TRP_E_OOM, TRP_E_NODEVICE = 0, -1, -2, -3, -4
_ERR_NAMES = {-1: "TRP_E_INVALID", -2: "TRP_E_CUDA", -3: "TRP_E_OOM", -4: "TRP_E_NODEVICE"}

# every symbol include/tr_prover.h declares (tests check that the library exports them all)
EXPORTED_SYMBOLS = [
    "trp_ctx_create", "trp_ctx_destroy", "trp_last_error", "trp_ctx_set_stream", "trp_ctx_sync",
    "trp_ctx_launch_count", "trp_version", "trp_prof_enable", "trp_prof_reset", "trp_prof_get", "trp_prof_get_work",
    "trp_bases_load", "trp_dev_bases_load", "trp_bases_load_ex", "trp_dev_bases_load_ex", "trp_bases_len", "trp_bases_describe", "trp_bases_free",
    "trp_msm", "trp_msm_batch", "trp_dev_msm_batch", "trp_dev_points_progression", "trp_dev_points_prefix_sum", "trp_points_sum", "trp_dev_points_sum",
    "trp_ntt", "trp_dev_ntt",
    "trp_domain_create", "trp_domain_free", "trp_domain_extended_k", "trp_domain_constants",
    "trp_lagrange_to_coeff", "trp_dev_lagrange_to_coeff", "trp_coeff_to_lagrange",
    "trp_coeff_to_extended", "trp_dev_coeff_to_extended", "trp_extended_to_coeff", "trp_dev_extended_to_coeff",
    "trp_dev_quotient_eval", "trp_dev_quotient_eval_rows", "trp_quotient_eval", "trp_dev_coeff_to_coset", "trp_dev_coeff_to_coset_gather",
    "trp_dev_cosets_to_coeff", "trp_dev_cosets_to_coeff_parts",
    "trp_field_op", "trp_dev_field_op", "trp_microbench",
    "trp_dev_batch_invert", "trp_batch_invert", "trp_dev_grand_product", "trp_grand_product",
    "trp_dev_permutation_product", "trp_permutation_product", "trp_dev_lookup_product", "trp_lookup_product",
    "trp_dev_permute_expression_pair", "trp_permute_expression_pair",
    "trp_dev_eval_polynomials", "trp_dev_eval_polynomials_at", "trp_dev_linear_combination", "trp_eval_polynomial", "trp_dev_inner_products", "trp_compute_inner_product", "trp_dev_powers",
    "trp_dev_kate_division", "trp_kate_division", "trp_dev_random_field", "trp_dev_fold", "trp_dev_ipa_round_scalars", "trp_dev_ipa_s_double", "trp_dev_generator_collapse", "trp_dev_msm_var",
    "trp_dev_hash_to_curve", "trp_hash_to_curve", "trp_dev_group_fft", "trp_group_fft", "trp_params_new", "trp_dev_params_new",
    "trp_dev_tinyram_witness",
]


class TrpError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"{_ERR_NAMES.get(code, code)}: {msg}")
        self.code = code


def lib_path() -> str:
    return _SO


def build_library(force: bool = False, jobs: int = 8) -> str:
    """Compile csrc/*.cu for sm_100a into libtrp.so (nvcc cross-compiles without a GPU)."""
    csrc = os.path.join(_HERE, "csrc")
    cmd = ["make", "-C", csrc, f"-j{jobs}"]
    if force:
        cmd.append("-B")
    subprocess.check_call(cmd, stdout=subprocess.DEVNULL)
    return _SO


_lib = None


def load_library():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(_SO):
        raise TrpError(TRP_E_NODEVICE, f"{_SO} is missing: build it with __graft_entry__.build() "
                                       "(there is no CPU fallback)")
    L = ctypes.CDLL(_SO)
    vp, sz, u, i = ctypes.c_void_p, ctypes.c_size_t, ctypes.c_uint, ctypes.c_int
    L.trp_ctx_create.argtypes = [ctypes.POINTER(vp), i, i]
    L.trp_ctx_destroy.argtypes = [vp]; L.trp_ctx_destroy.restype = None
    L.trp_last_error.argtypes = [vp]; L.trp_last_error.restype = ctypes.c_char_p
    L.trp_ctx_set_stream.argtypes = [vp, vp]
    L.trp_ctx_sync.argtypes = [vp]
    L.trp_ctx_launch_count.argtypes = [vp]; L.trp_ctx_launch_count.restype = ctypes.c_uint64
    L.trp_version.restype = ctypes.c_char_p
    L.trp_prof_enable.argtypes = [vp, i]
    L.trp_prof_reset.argtypes = [vp]
    L.trp_prof_get.argtypes = [vp, i, ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_uint64)]
    L.trp_prof_get_work.argtypes = [vp, i, ctypes.POINTER(ctypes.c_double)]
    L.trp_bases_load.argtypes = [vp, vp, sz, ctypes.POINTER(vp)]
    L.trp_dev_bases_load.argtypes = [vp, vp, sz, ctypes.POINTER(vp)]
    L.trp_bases_load_ex.argtypes = [vp, vp, sz, i, ctypes.POINTER(vp)]
    L.trp_dev_bases_load_ex.argtypes = [vp, vp, sz, i, ctypes.POINTER(vp)]
    L.trp_bases_len.argtypes = [vp]; L.trp_bases_len.restype = sz
    L.trp_bases_describe.argtypes = [vp, vp]
    L.trp_bases_free.argtypes = [vp]; L.trp_bases_free.restype = None
    L.trp_msm.argtypes = [vp, vp, vp, sz, vp]
    L.trp_msm_batch.argtypes = [vp, vp, vp, sz, sz, vp]
    L.trp_dev_msm_batch.argtypes = [vp, vp, vp, sz, sz, vp]
    L.trp_dev_points_progression.argtypes = [vp, vp, vp, sz, vp]
    L.trp_dev_points_prefix_sum.argtypes = [vp, vp, sz, vp]
    L.trp_points_sum.argtypes = [vp, vp, sz, vp]
    L.trp_dev_points_sum.argtypes = [vp, vp, sz, vp]
    L.trp_ntt.argtypes = [vp, vp, sz, u, vp]
    L.trp_dev_ntt.argtypes = [vp, vp, sz, u, vp]
    L.trp_domain_create.argtypes = [vp, u, u, ctypes.POINTER(vp)]
    L.trp_domain_free.argtypes = [vp]; L.trp_domain_free.restype = None
    L.trp_domain_extended_k.argtypes = [vp]; L.trp_domain_extended_k.restype = u
    L.trp_domain_constants.argtypes = [vp, vp]
    L.trp_lagrange_to_coeff.argtypes = [vp, vp, sz]
    L.trp_dev_lagrange_to_coeff.argtypes = [vp, vp, sz]
    L.trp_coeff_to_lagrange.argtypes = [vp, vp, sz]
    L.trp_coeff_to_extended.argtypes = [vp, vp, vp, sz]
    L.trp_dev_coeff_to_extended.argtypes = [vp, vp, vp, sz]
    L.trp_extended_to_coeff.argtypes = [vp, vp, vp, i]
    L.trp_dev_extended_to_coeff.argtypes = [vp, vp, vp, i]
    L.trp_dev_quotient_eval.argtypes = [vp, vp, sz, u, vp, sz, vp, sz, i, vp]
    L.trp_dev_quotient_eval_rows.argtypes = [vp, vp, sz, u, vp, sz, vp, sz, u, sz, sz, u, u, vp]
    L.trp_quotient_eval.argtypes = [vp, vp, sz, u, vp, sz, vp, sz, vp]
    L.trp_dev_coeff_to_coset.argtypes = [vp, vp, vp, sz, u]
    L.trp_dev_coeff_to_coset_gather.argtypes = [vp, vp, vp, sz, u]
    L.trp_dev_cosets_to_coeff.argtypes = [vp, vp, u, vp, i]
    L.trp_dev_cosets_to_coeff_parts.argtypes = [vp, vp, vp, u, u, vp, i]
    L.trp_field_op.argtypes = [vp, i, i, vp, vp, vp, sz]
    L.trp_dev_field_op.argtypes = [vp, i, i, vp, vp, vp, sz]
    L.trp_microbench.argtypes = [vp, i, i, ctypes.POINTER(ctypes.c_double)]
    L.trp_dev_batch_invert.argtypes = [vp, i, vp, vp, vp, sz]
    L.trp_batch_invert.argtypes = [vp, i, vp, sz]
    L.trp_dev_grand_product.argtypes = [vp, i, vp, sz, vp, vp, sz]
    L.trp_grand_product.argtypes = [vp, i, vp, sz, vp, vp, sz]
    L.trp_dev_permutation_product.argtypes = [vp, vp, vp, sz, vp, vp, vp, vp, vp]
    L.trp_permutation_product.argtypes = [vp, vp, vp, sz, vp, vp, vp, vp, vp]
    L.trp_dev_lookup_product.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp, sz]
    L.trp_lookup_product.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp, sz]
    L.trp_dev_permute_expression_pair.argtypes = [vp, vp, vp, sz, vp, vp, ctypes.POINTER(i)]
    L.trp_permute_expression_pair.argtypes = [vp, vp, vp, sz, vp, vp, ctypes.POINTER(i)]
    L.trp_dev_eval_polynomials.argtypes = [vp, i, vp, sz, sz, sz, vp, vp]
    L.trp_dev_eval_polynomials_at.argtypes = [vp, i, vp, sz, sz, vp, vp]
    L.trp_dev_linear_combination.argtypes = [vp, i, vp, vp, sz, sz, vp]
    L.trp_eval_polynomial.argtypes = [vp, i, vp, sz, vp, vp]
    L.trp_dev_inner_products.argtypes = [vp, i, vp, sz, vp, sz, sz, sz, vp]
    L.trp_compute_inner_product.argtypes = [vp, i, vp, vp, sz, vp]
    L.trp_dev_powers.argtypes = [vp, i, vp, sz, vp]
    L.trp_dev_kate_division.argtypes = [vp, i, vp, sz, vp, vp]
    L.trp_kate_division.argtypes = [vp, i, vp, sz, vp, vp]
    L.trp_dev_fold.argtypes = [vp, i, vp, sz, vp]
    L.trp_dev_random_field.argtypes = [vp, i, ctypes.c_char_p, ctypes.c_uint64, sz, vp]
    L.trp_dev_ipa_round_scalars.argtypes = [vp, i, vp, vp, sz, sz, sz, sz, vp]
    L.trp_dev_ipa_s_double.argtypes = [vp, i, vp, sz, vp, vp]
    L.trp_dev_generator_collapse.argtypes = [vp, vp, sz, vp]
    L.trp_dev_msm_var.argtypes = [vp, vp, vp, sz, sz, vp]
    L.trp_dev_hash_to_curve.argtypes = [vp, ctypes.c_char_p, vp, sz, i, ctypes.c_uint64, sz, vp]
    L.trp_hash_to_curve.argtypes = [vp, ctypes.c_char_p, vp, sz, sz, vp]
    L.trp_dev_group_fft.argtypes = [vp, vp, u, vp, vp]
    L.trp_group_fft.argtypes = [vp, vp, u, vp, vp]
    L.trp_params_new.argtypes = [vp, u, vp, vp, vp, vp]
    L.trp_dev_params_new.argtypes = [vp, u, vp, vp, vp]
    L.trp_dev_tinyram_witness.argtypes = [vp, u, u, i, vp, sz, vp, sz, vp, sz, vp, sz, vp, sz, sz, ctypes.POINTER(ctypes.c_uint64),
                                          ctypes.POINTER(i)]
    _lib = L
    return L


def as_u64(a, copy=False):
    a = np.ascontiguousarray(a, dtype=np.uint64)
    return a.copy() if copy else a


def ptr(a):
    """host numpy array -> void*; int -> device pointer as void*."""
    if a is None:
        return None
    if isinstance(a, int):
        return ctypes.c_void_p(a)
    return a.ctypes.data_as(ctypes.c_void_p)


class Context:
    """One device + one stream + one commitment curve (trp_ctx).  curve = VESTA is what the reference uses
    (Params<EqAffine>, src/test_utils.rs:12,21): scalars / NTT field Fp, point coordinates Fq."""

    def __init__(self, device: int = 0, curve: int = VESTA):
        self.lib = load_library()
        h = ctypes.c_void_p()
        rc = self.lib.trp_ctx_create(ctypes.byref(h), device, curve)
        if rc != TRP_OK:
            why = {TRP_E_NODEVICE: "no CUDA device is visible (this backend has no CPU fallback)",
                   TRP_E_INVALID: "invalid device or curve id"}.get(rc, "context creation failed")
            raise TrpError(rc, why)
        self.handle = h
        self.device, self.curve = device, curve

    def check(self, rc):
        if rc != TRP_OK:
            raise TrpError(rc, self.lib.trp_last_error(self.handle).decode())

    def set_stream(self, cuda_stream_ptr):
        self.check(self.lib.trp_ctx_set_stream(self.handle, ctypes.c_void_p(cuda_stream_ptr or 0)))

    def sync(self):
        self.check(self.lib.trp_ctx_sync(self.handle))

    _TORCH_STREAMS = {}

    def bind_torch_stream(self):
        """Make torch and this ctx share ONE CUDA stream (one per process and device, made torch's current stream): code that
        mixes torch tensor operations with trp_dev_* calls is then ordered by the stream itself -- no fences between the two.
        Returns the torch stream.  (A ctx starts on its own non-blocking stream, which torch's streams do not synchronise with.)"""
        import torch
        st = Context._TORCH_STREAMS.get(self.device)
        if st is None:
            torch.cuda.synchronize(self.device)
            st = Context._TORCH_STREAMS[self.device] = torch.cuda.Stream(device=self.device)
        if torch.cuda.current_stream(self.device) != st:
            torch.cuda.synchronize(self.device)
            torch.cuda.set_stream(st)
        self.set_stream(st.cuda_stream)
        return st

    @property
    def launches(self) -> int:
        return int(self.lib.trp_ctx_launch_count(self.handle))

    def field_op(self, op, a, b=None, which_field=0):
        code = {"add": 0, "sub": 1, "mul": 2, "inv": 3, "sqr": 4}[op]
        a = as_u64(a); out = np.empty_like(a)
        bb = as_u64(b) if b is not None else None
        self.check(self.lib.trp_field_op(self.handle, which_field, code, ptr(a), ptr(bb), ptr(out), a.size // 4))
        return out

    def microbench(self, kind, iters=256) -> float:
        v = ctypes.c_double()
        self.check(self.lib.trp_microbench(self.handle, kind, iters, ctypes.byref(v)))
        return v.value

    PROF_PHASES = ("msm_sort", "msm_accum_l1", "msm_levels", "msm_reduce", "ntt_pass", "quotient_vm", "products", "lookup_sort")

    def prof_enable(self, on=True):
        self.check(self.lib.trp_prof_enable(self.handle, int(on)))

    def prof_reset(self):
        self.check(self.lib.trp_prof_reset(self.handle))

    def prof_get(self):
        """{phase: (total_ms, spans)} measured with CUDA events on the ctx stream."""
        out = {}
        for idx, name in enumerate(self.PROF_PHASES):
            ms, cnt = ctypes.c_double(), ctypes.c_uint64()
            self.check(self.lib.trp_prof_get(self.handle, idx, ctypes.byref(ms), ctypes.byref(cnt)))
            out[name] = (ms.value, int(cnt.value))
        return out

    def prof_work(self):
        """{phase: algorithmic units of the timed spans} (trp_prof_get_work)"""
        out = {}
        for idx, name in enumerate(self.PROF_PHASES):
            w = ctypes.c_double()
            self.check(self.lib.trp_prof_get_work(self.handle, idx, ctypes.byref(w)))
            out[name] = w.value
        return out

    def close(self):
        if getattr(self, "handle", None):
            self.lib.trp_ctx_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
