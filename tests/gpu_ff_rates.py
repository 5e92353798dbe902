"""Ad-hoc measurement (not a test): the rates that the Pasta field multiplier (csrc/ff.cuh) bounds, one JSON line.

  fe_mul_gops  trp_microbench kind 4: Fq Montgomery products per second (two dependent chains per thread, all SMs)
  ntt_ms       one batched NTT of 8 x 2^20 Fp elements (trp_dev_ntt), device resident
  msm_ms       one MSM step of 8 columns x (2^20 + 1) Vesta points, uniform scalars (trp_dev_msm_batch), device resident,
               with the msm_accum_l1 share from the library's phase timers

The quotient program is timed per phase by bench.py (roofline.phase_share_of_step).  Run it once per build, on the same card,
alternating builds, and compare the lines; env TAG labels the line, REPS sets the timed repetitions (default 10)."""
import ctypes
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import __graft_entry__ as ge

pkg = ge.load_package()
from tiny_ram_halo2_b200 import synthetic
from tiny_ram_halo2_b200._lib import ptr

REPS = int(os.environ.get("REPS", "10"))
K, B = 20, 8


def timed(stream, fn, reps=REPS, warm=3):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(reps):
        fn()
    e1.record(stream)
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def main():
    ctx = pkg.Context(0, pkg.VESTA)
    stream = torch.cuda.Stream()
    ctx.set_stream(stream.cuda_stream)
    lib = ctx.lib
    out = {"tag": os.environ.get("TAG", ""), "device": torch.cuda.get_device_name(0)}
    out["fe_mul_gops"] = round(max(ctx.microbench(4, 512) for _ in range(3)), 1)

    dom = pkg.EvaluationDomain(ctx, 6, K)
    a = torch.randint(0, 1 << 62, (B, 1 << K, 4), dtype=torch.int64, device="cuda")
    out["ntt_ms"] = round(timed(stream, lambda: ctx.check(lib.trp_dev_ntt(ctx.handle, a.data_ptr(), B, K, ptr(dom.omega)))), 4)
    del a

    n = (1 << K) + 1
    d_pts = torch.empty((n, 8), dtype=torch.int64, device="cuda")
    torch.cuda.synchronize()
    synthetic.device_points(ctx, n, d_pts.data_ptr())
    ctx.sync()
    hb = ctypes.c_void_p()
    ctx.check(lib.trp_dev_bases_load(ctx.handle, d_pts.data_ptr(), n, ctypes.byref(hb)))
    ctx.sync()
    d_sc = torch.from_numpy(synthetic.random_scalars(n, 20, B).view(np.int64)).cuda()
    d_out = torch.zeros((B, 12), dtype=torch.int64, device="cuda")
    torch.cuda.synchronize()
    step = lambda: ctx.check(lib.trp_dev_msm_batch(ctx.handle, hb, d_sc.data_ptr(), n, B, d_out.data_ptr()))
    out["msm_ms"] = round(timed(stream, step), 4)
    ctx.prof_reset(); ctx.prof_enable(True)
    for _ in range(REPS):
        step()
    torch.cuda.synchronize()
    prof = ctx.prof_get()
    ctx.prof_enable(False)
    acc_ms, acc_launches = prof["msm_accum_l1"]
    out["msm_accum_l1_ms_per_step"] = round(acc_ms / REPS, 4)
    out["msm_checksum"] = int(d_out.cpu().numpy().view(np.uint64).sum() & 0xffffffff)
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
