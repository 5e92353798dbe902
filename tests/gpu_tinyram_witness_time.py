"""Times trace -> witness block for bench.py's trace (programs.longest_loop(32), 65 521 steps, k = 20) both ways, in one process,
alternating the two paths:
  host    tinyram.build(arrays=True) + HostWitness + upload        (what bench.py's setup and e2e leg do)
  device  device_witness: the packing (tinyram.witness_inputs, also timed alone) and trp_dev_tinyram_witness
Each timing ends in a device synchronise.  Also: the device span of device_witness from CUDA events, its kernels from
torch.profiler (a separate pass), the bytes each path sends host -> device, and the card's name and power limit.
usage: python tests/gpu_tinyram_witness_time.py [reps] [out.json]"""
import json
import subprocess
import sys
import time

import torch

sys.path.insert(0, ".")
import __graft_entry__ as ge

pkg = ge.load_package()
from tiny_ram_halo2_b200 import plonk as PL, programs, tinyram as TR  # noqa: E402

reps = int(sys.argv[1]) if len(sys.argv) > 1 else 5
out_path = sys.argv[2] if len(sys.argv) > 2 else None
K = 20
ctx = pkg.Context(0, pkg.VESTA)
be = PL.GpuBackend(ctx, K, 6)
tr = programs.longest_loop(32)
card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()


def host_path(out=None):
    _, _, _, adv, inst = TR.build(PL, tr, K, dense=False, arrays=True)
    hw = TR.HostWitness(be, list(inst) + list(adv))
    return hw.upload(be, out), hw.bytes


host_block, host_bytes = host_path()
dev_block = TR.device_witness(be, tr)
assert torch.equal(host_block, dev_block), "device block differs from the host block"
circ = TR.TinyRamCircuit(PL, 32, 8)
steps, ins, prog, colmap = TR.witness_inputs(circ, tr)
dev_bytes = steps.nbytes + ins.nbytes + prog.nbytes + colmap.nbytes

rows = []
for _ in range(reps):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    host_path(host_block)
    torch.cuda.synchronize()
    t1 = time.perf_counter()
    TR.witness_inputs(circ, tr)
    t2 = time.perf_counter()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    TR.device_witness(be, tr, out=dev_block)
    e1.record()
    torch.cuda.synchronize()
    t3 = time.perf_counter()
    rows.append({"host_s": t1 - t0, "pack_s": t2 - t1, "device_s": t3 - t2, "device_span_ms": e0.elapsed_time(e1)})

with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
    TR.device_witness(be, tr, out=dev_block)
    torch.cuda.synchronize()
kernels = {}
for ev in prof.key_averages():
    if ev.device_time_total > 0:
        kernels[ev.key] = round(ev.device_time_total / 1e3, 4)           # ms

med = lambda key: sorted(r[key] for r in rows)[len(rows) // 2]
result = {"card": card, "k": K, "steps": len(tr.exe), "reps": reps, "block_shape": list(dev_block.shape),
          "host_path_s_median": round(med("host_s"), 4), "device_path_s_median": round(med("device_s"), 4),
          "pack_s_median": round(med("pack_s"), 4),
          "device_span_ms_median": round(med("device_span_ms"), 3), "kernels_ms": kernels,
          "h2d_bytes": {"host_path": host_bytes, "device_path": dev_bytes}, "runs": rows}
print(json.dumps(result, indent=1))
if out_path:
    with open(out_path, "w") as f:
        json.dump(result, f, indent=1)
