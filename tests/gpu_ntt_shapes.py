"""Ad-hoc measurement (not a test): the NTT at the shapes a k = 20 proof runs, one JSON line with a digest per output.

  fwd8_ms      trp_dev_ntt, 8 x 2^20, no scaling
  l2c32_ms     trp_dev_lagrange_to_coeff, 32 x 2^20 (1/N scalar on the last pass)
  coset32_ms   trp_dev_coeff_to_coset, 32 x 2^20 (table of n powers on the first pass)
  gather32_ms  trp_dev_coeff_to_coset_gather, 32 x 2^20 (the same, columns read through a device address table)

Inputs are seeded, so the *_dig fields (SHA-256 prefixes of the outputs) must agree between builds.  argv[1], if given, is the
repository tree to load the package from (default: this one), so that two builds can be run alternately; env TAG labels
the line."""
import hashlib, json, os, sys
root = sys.argv[1] if len(sys.argv) > 1 else os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, root)
import torch
import __graft_entry__ as ge
pkg = ge.load_package()
from tiny_ram_halo2_b200._lib import ptr
REPS = 20
K = 20

def timed(stream, fn, reps=REPS, warm=3):
    for _ in range(warm): fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(reps): fn()
    e1.record(stream)
    torch.cuda.synchronize()
    return round(e0.elapsed_time(e1) / reps, 4)

def digest(t):
    torch.cuda.synchronize()
    return hashlib.sha256(t.cpu().numpy().tobytes()).hexdigest()[:16]

ctx = pkg.Context(0, pkg.VESTA)
stream = torch.cuda.Stream()
ctx.set_stream(stream.cuda_stream)
lib = ctx.lib
out = {"tag": os.environ.get("TAG", ""), "device": torch.cuda.get_device_name(0)}
dom = pkg.EvaluationDomain(ctx, 6, K)
g = torch.Generator(device="cuda"); g.manual_seed(7)
def rnd(b):  # below 2^248: canonical in both Pasta fields
    a = torch.randint(0, 1 << 62, (b, 1 << K, 4), dtype=torch.int64, device="cuda", generator=g)
    a[..., 3] &= (1 << 56) - 1
    torch.cuda.synchronize()  # written on torch's stream, read on the ctx's: the values must be there before the transform runs
    return a
a = rnd(8)
out["fwd8_ms"] = timed(stream, lambda: ctx.check(lib.trp_dev_ntt(ctx.handle, a.data_ptr(), 8, K, ptr(dom.omega))))
b = rnd(8); ctx.check(lib.trp_dev_ntt(ctx.handle, b.data_ptr(), 8, K, ptr(dom.omega))); out["fwd_dig"] = digest(b)
B = 32
c = rnd(B)
out["l2c32_ms"] = timed(stream, lambda: ctx.check(lib.trp_dev_lagrange_to_coeff(dom.handle, c.data_ptr(), B)))
d = rnd(B); ctx.check(lib.trp_dev_lagrange_to_coeff(dom.handle, d.data_ptr(), B)); out["l2c_dig"] = digest(d)
src = rnd(B); dst = torch.empty_like(src)
out["coset32_ms"] = timed(stream, lambda: ctx.check(lib.trp_dev_coeff_to_coset(dom.handle, src.data_ptr(), dst.data_ptr(), B, 1)))
out["coset_dig"] = digest(dst)
tab = torch.tensor([src[i].data_ptr() for i in reversed(range(B))], dtype=torch.int64, device="cuda")
out["gather32_ms"] = timed(stream, lambda: ctx.check(lib.trp_dev_coeff_to_coset_gather(dom.handle, tab.data_ptr(), dst.data_ptr(), B, 3)))
out["gather_dig"] = digest(dst)
print(json.dumps(out), flush=True)
