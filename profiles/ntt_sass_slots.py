"""Static SASS check of the specialised NTT pass kernels (csrc/ntt.cu), no GPU needed.

Compiles ntt.cu for sm_100a, reads `cuobjdump -sass`, and for every ntt_pass_spec_kernel instance reports:
  regs, spill    registers and spill bytes (ptxas -v)
  div            I2F / MUFU instructions (a runtime 32-bit division or modulo); must be 0
  muls           field multiplications in the static code: IMAD.WIDE.U32.X count / the same count in one fe_mul
  slots/mul      fmaheavy issue slots (IMAD.WIDE* = 2, every other IMAD* = 1) per multiplication, i.e. per radix-2
                 butterfly plus the scaling multiplications; the multiplier alone is the `fe_mul` row.
The unit loops are not unrolled (#pragma unroll 1), so the static code holds each radix-4 group once and the ratio is the
executed one.  Usage: python profiles/ntt_sass_slots.py [--check]   (--check: exit 1 if an instance divides or spills)
"""
import collections
import os
import re
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "tiny-ram-halo2_b200", "csrc")
CUDA = os.environ.get("CUDA_HOME", "/usr/local/cuda")
NVCC = [os.path.join(CUDA, "bin", "nvcc"), "-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a",
        "--expt-relaxed-constexpr", "-Xptxas", "-v", "-cubin", "-I", CSRC]

ONE_MUL = r"""
#include "ff.cuh"
extern "C" __global__ void one_fe_mul(const uint4* a, const uint4* b, uint4* out) {
  ff::fe_store(out, ff::fe_mul(ff::fe_load<ff::FpParams>(a), ff::fe_load<ff::FpParams>(b)));
}
"""


def compile_sass(src, tmp, name):
    cubin = os.path.join(tmp, name + ".cubin")
    r = subprocess.run(NVCC + [src, "-o", cubin], capture_output=True, text=True, check=True)
    sass = subprocess.run([os.path.join(CUDA, "bin", "cuobjdump"), "-sass", cubin], capture_output=True, text=True,
                          check=True).stdout
    return sass, r.stderr


def functions(sass):
    out = {}
    for blk in re.split(r"\n\s*Function : ", sass)[1:]:
        name = blk.split("\n", 1)[0].strip()
        ops = collections.Counter(m.group(1) for m in re.finditer(
            r"/\*[0-9a-f]{4,}\*/\s+(?:@!?U?P[T0-9]+\s+)?([A-Z][A-Z0-9_.]*)", blk))
        out[name] = ops
    return out


def ptxas_info(log):
    info = {}
    for blk in log.split("Function properties for ")[1:]:
        name = blk.split("\n", 1)[0].strip()
        regs = re.search(r"Used (\d+) registers", blk)
        sp = re.search(r"(\d+) bytes spill stores, (\d+) bytes spill loads", blk)
        info[name] = (int(regs.group(1)) if regs else -1, int(sp.group(1)) + int(sp.group(2)) if sp else 0)
    return info


def slots(ops):
    return sum((2 if k.startswith("IMAD.WIDE") else 1) * v for k, v in ops.items() if k.startswith("IMAD"))


def demangle(name):
    d = subprocess.run(["c++filt", name], capture_output=True, text=True).stdout.strip()
    m = re.search(r"ntt_pass_spec_kernel<ff::(\w+)Params, (.*)>\(", d)
    return f"{m.group(1)}<{m.group(2)}>" if m else d


def main():
    check = "--check" in sys.argv
    with tempfile.TemporaryDirectory() as tmp:
        one = os.path.join(tmp, "one_mul.cu")
        with open(one, "w") as f:
            f.write(ONE_MUL)
        ref = functions(compile_sass(one, tmp, "one_mul")[0])["one_fe_mul"]
        sass, log = compile_sass(os.path.join(CSRC, "ntt.cu"), tmp, "ntt")
    wide_per_mul = ref["IMAD.WIDE.U32.X"]
    print(f"fe_mul alone: {slots(ref)} fmaheavy slots, {wide_per_mul} IMAD.WIDE.U32.X")
    info = ptxas_info(log)
    print(f"{'instance <S, C, first, last, pre, post, gather>':68s} regs  spill  div  muls  slots/mul")
    bad = False
    for name, ops in functions(sass).items():
        if "ntt_pass_spec_kernel" not in name:
            continue
        regs, spill = info.get(name, (-1, -1))
        div = sum(v for k, v in ops.items() if k.startswith(("I2F", "MUFU")))
        muls = ops["IMAD.WIDE.U32.X"] / wide_per_mul
        print(f"{demangle(name):68s} {regs:4d} {spill:6d} {div:4d} {muls:5.1f} {slots(ops) / muls:9.1f}")
        bad |= div > 0 or spill > 0
    if check and bad:
        sys.exit(1)


if __name__ == "__main__":
    main()
