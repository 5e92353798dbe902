#!/usr/bin/env python
"""bench.py -- headline benchmark of the prover hot path on B200: ONE real create_proof at k = 20.

Workload (BASELINE.json: "TinyRAM create_proof time at k=20", configs[3]): plonk.create_proof of the reference's
TinyRamCircuit<32, 8> (tiny-ram-halo2_b200/tinyram.py: its real gates, lookups and witness) for a 65 521-step trace that fills
the 2^16-row execution table, n = 2^20 rows, Vesta / IPA, Blake2b transcript, serialized proof -- the unit of work of the
reference's only prover entry point (/root/reference/src/test_utils.rs:37-51).  A step = one proof.  Metric: proofs per second
(1 / create_proof seconds), whole job.

  python bench.py [--gpus N] [--steps K] [--warmup W]       # this repo's CUDA path
  python bench.py --impl reference [...]                     # CPU restatement (oracle/), per-phase sampled, same workload
  python bench.py --dump-outputs DIR [...]                   # also write the last timed proof as DIR/proof.npy

The prover's RNG is keyed by a fixed seed, so with the same arguments every run proves the same witness with the same
blinding and the last timed proof is the same bytes: two builds can be compared output for output.

N > 1 (torchrun, one rank per GPU) is STRONG scaling of the same single proof: sharded_backend.ShardedGpuBackend divides the
commitments, the Lagrange -> coefficient transforms, the lookups, the permutation chunks and the quotient (NTTs by column
block, program by row slice) between the ranks; the proof bytes are identical on every rank and for every N.

value  device-resident: the witness columns are in HBM when the timed region starts.
e2e    the same through the host-facing path: the witness starts in pinned host memory every step (tinyram.HostWitness),
       is uploaded, proved, and the proof bytes end on the host.
extras (N = 1): the other two parts of BASELINE.json's composite metric -- MSM Mpts/s (8 x (2^20 + 1) commit_lagrange-shaped
       columns, device resident and through trp_msm_batch with host buffers) and NTT GB/s against both rooflines.
Inputs exceed L2 by orders of magnitude (15.5 GiB of per-proof polynomials), so no flush is needed between steps.
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True          # the benchmark writes nothing into the tree it runs from (which may be read-only)

K_LOG = int(os.environ.get("TRP_BENCH_K", "20"))          # 20 is the benchmark; smaller values are for dry runs of this file
WORD_BITS = 32 if K_LOG >= 17 else 2 * (K_LOG - 2)
N_POINTS = (1 << K_LOG) + 1
M_COLS = 8
METRIC = "tinyram_create_proof_throughput"
UNIT = "proofs/s"
WORKLOAD = (f"one plonk.create_proof of the reference's TinyRamCircuit<{WORD_BITS}, 8> (tinyram.py) at k = {K_LOG}: a trace that fills the "
            f"2^{WORD_BITS // 2}-row execution table, Vesta/IPA, Blake2b transcript, serialized proof (BASELINE.json configs[3])")
FMUL_PER_MIXED_ADD = 10          # XYZZ madd-2008-s: 8M + 2S (SURVEY.md 8d)
MACS_PER_FMUL = 128              # generic 8x8-limb CIOS: 64 product + 64 reduction 32x32->64 MACs
DTYPE = "u32x8 (255-bit Montgomery)"
RNG_SEED = hashlib.sha256(b"bench.py create_proof").digest()


def _config(extra=None):
    c = {"workload": WORKLOAD, "k": K_LOG, "word_bits": WORD_BITS, "curve": "vesta", "rng": "AES-256-CTR keyed by a fixed seed (RNG_SEED); random polynomials = a 32-byte key of that stream expanded on the device (BLAKE2b counter mode)",
         "l2_policy": "inputs larger than L2 (15.5 GiB of per-proof polynomials at k = 20)"}
    if extra:
        c.update(extra)
    return c


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.lines, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def stop(self, t0, t1):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, smax, reasons = [], [], set()
        for ts, line in self.lines:
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                clk, mx = float(f[1]), float(f[2])
            except ValueError:
                continue
            if t0 - 0.05 <= ts <= t1 + 0.15:
                sm.append(clk); smax.append(mx)
                for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                    if val.lower().startswith("active"):
                        reasons.add(name)
        if not sm:   # region shorter than the sampling period: fall back to all samples
            for ts, line in self.lines:
                f = [x.strip() for x in line.split(",")]
                try:
                    sm.append(float(f[1])); smax.append(float(f[2]))
                except (ValueError, IndexError):
                    pass
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return json.load(f), "measured (MEASURED_PEAKS.json)"
    return {"hbm_gbs": 6650.0, "sm_max_mhz": 1965.0}, "fallback (B200_PROFILING.md)"


def _traffic_from_profiles(kernel, pattern):
    """dram bytes per launch of a kernel from the newest committed ncu capture, if any (profiles/*.json)."""
    import glob
    scale = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9, "Tbyte": 1e12}
    for p in sorted(glob.glob(os.path.join(ROOT, "profiles", pattern)), reverse=True):
        try:
            with open(p) as f:
                rows = json.load(f)
            vals = [sum(float(r[k]) * scale[r[k + ".unit"]] for k in ("dram__bytes_read.sum", "dram__bytes_write.sum"))
                    for r in rows if kernel in r.get("kernel", "")]
            if vals:
                return int(sum(vals) / len(vals)), os.path.relpath(p, ROOT)
        except Exception:
            continue
    return None, None


def _load_workload(pkg, arrays=True):
    """trace, circuit, fixed columns, copy constraints, advice and instance columns of the benchmark circuit (host synthesis)"""
    from tiny_ram_halo2_b200 import plonk as PL, programs, tinyram as TR
    tr = programs.longest_loop(WORD_BITS)
    circ, fixed, copies, adv, inst = TR.build(PL, tr, K_LOG, dense=False, arrays=arrays)
    return tr, circ, fixed, copies, adv, inst


# -------------------------------------------------------------------------------------------------------------
# CPU arm: the oracle's restatement of halo2_proofs 0.2.0 on the host cores, per-phase SAMPLED
# -------------------------------------------------------------------------------------------------------------
class CpuProofSampler:
    """create_proof of the same circuit on the host cores, sampled phase by phase (BASELINE.md section 3; the Rust prover cannot be
    built here, and a full k = 20 proof of the C++ restatement takes ~10 minutes): every hot routine of halo2's create_proof is
    timed ONCE at full size (or on a stated fraction of its rows) with all host threads and multiplied by the number of times
    SURVEY.md Appendix C's flow calls it for this constraint system.  Counted: commit_lagrange MSMs (sparse advice-shaped and
    dense), coefficient-basis commits, lagrange_to_coeff, coeff_to_extended (halo2 materialises every extended coset),
    the quotient program over the extended domain, extended_to_coeff, the openings' evaluations, the IPA's round MSMs and
    generator collapse.  Not counted (minor on the CPU as well): witness synthesis, lookup permutation, grand-product scans,
    multiopen's linear combinations, transcript hashing -- so the estimate favours the CPU."""

    def __init__(self):
        sys.path.insert(0, os.path.join(ROOT, "oracle")); sys.path.insert(0, os.path.join(ROOT, "tests"))
        import __graft_entry__ as ge
        import oracle as O
        self.O, self.cores = O, O.hw_threads()
        ge.load_package()
        from tiny_ram_halo2_b200 import plonk as PL, poly as P, tinyram as TR, trace as T
        # the constraint system and the quotient program do not depend on k: take them from the smallest instance of the circuit
        import random
        import plonk_model as VM
        import pasta_model as pm
        import tinyram_programs as TP
        circ, fixed, copies, adv, inst = TR.build(PL, TP.answer_only(T, 8), 6)
        cs = circ.cs

        class _Stop(Exception):
            pass

        be = VM.PythonBackend(pm.Vesta, 6, cs.degree())
        captured = {}

        def grab(ast, ext):
            captured["ast"], captured["leaves"] = ast, len(ext)
            raise _Stop()

        be.quotient = grab
        pk = PL.keygen(be, cs, fixed, copies)
        rnd = random.Random(1)
        try:
            PL.create_proof(be, pk, inst, adv, lambda: rnd.randrange(be.p), PL.Blake2bWrite(pm.Vesta.base.p, be.p))
        except _Stop:
            pass
        self.prog = P.compile_ast(captured["ast"], be.p)
        self.p = be.p
        chunks = -(-len(cs.permutation) // (cs.degree() - 2)) if cs.permutation else 0
        L = len(cs.lookups)
        nq = sum(len(cs.queries[kind]) for kind in cs.queries)
        self.counts = {
            "msm_sparse": cs.num_instance + cs.num_advice + 2 * L,          # commit_lagrange of instance / advice / permuted lookup columns
            "msm_dense": chunks + L + 1 + (cs.degree() - 1) + 1 + 1,        # Z columns; random poly, h pieces, q', the IPA's S (coefficient basis)
            "lagrange_to_coeff": cs.num_instance + cs.num_advice + 3 * L + chunks,
            "coeff_to_extended": cs.num_instance + cs.num_advice + 3 * L + chunks,
            "quotient_rows": 1 << (K_LOG + 3), "extended_to_coeff": 1,
            "evaluations": nq + 2 + len(cs.permutation) + 3 * chunks + 5 * L,
            "ipa_rounds": K_LOG}
        self.shape = {"advice": cs.num_advice, "instance": cs.num_instance, "lookups": L, "permutation_chunks": chunks,
                      "program": self.prog.counts(), "leaves": captured["leaves"]}
        self._inputs = None

    def _prepare(self):
        O = self.O
        from util import make_points
        n = 1 << K_LOG
        rng = np.random.Generator(np.random.PCG64(20))
        dense = rng.integers(0, 1 << 64, size=(n + 1, 4), dtype=np.uint64); dense[:, 3] &= np.uint64((1 << 62) - 1)
        sparse = np.zeros((n + 1, 4), dtype=np.uint64)
        rows = min(1 << 16, n)
        small = np.zeros((rows, 4), dtype=np.uint64)
        kind = rng.random(rows)
        small[:, 0] = np.where(kind < 0.9, rng.integers(0, 2, rows, dtype=np.uint64), rng.integers(0, 1 << 32, rows, dtype=np.uint64))
        sparse[:rows] = O.to_mont(O.FP, small)
        sparse[n - 6:] = dense[:7]                                       # blinding rows + the blind
        pts = make_points(O.VESTA, n + 1)
        sample_rows = 1 << 12
        cols = [O.random_field_mont(O.FP, sample_rows, 100 + i) for i in range(8)]
        consts = O.to_mont(O.FP, O.ints_to_limbs(self.prog.consts))
        self._inputs = dict(n=n, dense=dense, sparse=sparse, pts=pts, sample_rows=sample_rows, cols=cols, consts=consts,
                            omega=None)
        _, om, _ = O.domain_info(O.FP, 6, K_LOG)
        self._inputs["omega"] = om

    def sample(self):
        """one bounded sample: every routine once; returns (estimated seconds of one create_proof, per-phase seconds, sample seconds)"""
        if self._inputs is None:
            self._prepare()
        O, I, T, c = self.O, self._inputs, self.cores, self.counts
        n = I["n"]
        t_all = time.perf_counter()

        def timed(fn):
            t = time.perf_counter(); fn(); return time.perf_counter() - t

        per = {}
        per["msm_dense"] = timed(lambda: O.msm(O.VESTA, I["dense"], I["pts"], threads=T)) * c["msm_dense"]
        per["msm_sparse"] = timed(lambda: O.msm(O.VESTA, I["sparse"], I["pts"], threads=T)) * c["msm_sparse"]
        col = I["dense"][:n].reshape(1, n, 4)
        per["lagrange_to_coeff"] = timed(lambda: O.lagrange_to_coeff(O.FP, 6, K_LOG, col, threads=T)) * c["lagrange_to_coeff"]
        ext = {}
        per["coeff_to_extended"] = timed(lambda: ext.setdefault("e", O.coeff_to_extended(O.FP, 6, K_LOG, col, threads=T))) * c["coeff_to_extended"]
        per["extended_to_coeff"] = timed(lambda: O.extended_to_coeff(O.FP, 6, K_LOG, ext["e"][0], divide=True, threads=T))
        del ext
        # the quotient program on sample_rows rows (every leaf read from one of 8 small in-cache columns: favours the CPU)
        sr = I["sample_rows"]
        cols = [I["cols"][i % 8] for i in range(self.prog.n_cols)]
        per["quotient"] = timed(lambda: O.quotient_vm(O.FP, self.prog.code, self.prog.n_regs, I["consts"], cols, sr, I["cols"][0], sr,
                                                      threads=T)) * (c["quotient_rows"] / sr)
        x = O.random_field_mont(O.FP, 1, 7)[0]
        per["evaluations"] = timed(lambda: O.eval_polynomial(O.FP, I["dense"][:n], x, threads=T)) * c["evaluations"]
        # IPA: round j has two MSMs of n / 2^(j+1) points and a collapse of as many scalar multiplications: geometric sum = 2 x round 0
        half = n // 2
        per["ipa_msm"] = timed(lambda: O.msm(O.VESTA, I["dense"][:half], I["pts"][:half], threads=T)) * 2 * 2
        cs_n = min(1 << 11, half)
        u = O.ints_to_limbs([0x1234567890abcdef1234567890abcdef1234567890abcdef1234567890abcdef % self.p])[0]
        per["ipa_collapse"] = timed(lambda: O.generator_collapse(O.VESTA, I["pts"][:2 * cs_n], u, threads=T)) * (half / cs_n) * 2
        return sum(per.values()), per, time.perf_counter() - t_all

    def describe(self, per, sample_s):
        return {"kind": "port", "cores": self.cores, "method": "sampled",
                "sample": (f"every hot routine of halo2 0.2.0's create_proof timed once per step on {self.cores} host threads (oracle/liboracle.so, the C++ "
                           f"restatement; the Rust crate cannot be built here) at k = {K_LOG} and multiplied by its call count for this constraint system: "
                           f"{json.dumps(self.counts)}; the quotient program on {self._inputs['sample_rows']} rows of 8 in-cache columns; witness synthesis, "
                           "lookup permutation, grand-product scans, multiopen and hashing not counted (the estimate favours the CPU)"),
                "phase_seconds": {k: round(v, 2) for k, v in per.items()}, "sample_seconds": round(sample_s, 1), "circuit": self.shape}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    S = CpuProofSampler()
    for _ in range(max(min(args.warmup, 1), 0)):
        S.sample()
    ests, per, sample_s = [], None, 0.0
    t0 = time.perf_counter()
    for _ in range(args.steps):
        est, per, sample_s = S.sample()
        ests.append(est)
    wall = time.perf_counter() - t0
    est = statistics.median(ests)
    value = 1.0 / est
    cpu = S.describe(per, sample_s)
    cpu.update({"value": value, "unit": UNIT, "estimated_create_proof_seconds": round(est, 1)})
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": est * 1e3, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": DTYPE, "data": "synthetic", "config": _config(),
            "cpu_baseline": cpu, "sample_wall_seconds_per_step": round(wall / max(args.steps, 1), 1),
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


# -------------------------------------------------------------------------------------------------------------
# GPU arm
# -------------------------------------------------------------------------------------------------------------
def run_gpu(args):
    import torch
    import torch.distributed as dist
    import __graft_entry__ as ge

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- this backend has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    d = None
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        d = dist

    pkg = ge.load_package()
    from tiny_ram_halo2_b200 import plonk as PL, tinyram as TR, verifier as V
    from tiny_ram_halo2_b200.sharded_backend import ShardedGpuBackend, ShardedRng
    ctx = pkg.Context(local_rank, pkg.VESTA)

    # ---- setup (untimed): witness synthesis on the host, Params::new, upload, keygen ----------------------------------------
    t0 = time.perf_counter()
    tr, circ, fixed, copies, adv, inst = _load_workload(pkg)
    t_witness = time.perf_counter() - t0
    cs = circ.cs
    t0 = time.perf_counter()
    be = ShardedGpuBackend(ctx, K_LOG, cs.degree(), d)
    be._wait(); t_params = time.perf_counter() - t0
    stream = be.stream
    t0 = time.perf_counter()
    d_fixed = TR.device_columns(be, fixed)
    host_witness = TR.HostWitness(be, list(inst) + list(adv))             # pinned: the end-to-end leg's input
    block = host_witness.upload(be)
    be._wait(); t_upload = time.perf_counter() - t0
    n_inst = len(inst)
    t0 = time.perf_counter()
    pk = PL.keygen(be, cs, d_fixed, copies)
    be._wait(); t_keygen = time.perf_counter() - t0
    rng = ShardedRng(be.p, d, "cuda", seed=RNG_SEED)                       # the same stream on every rank and in every run

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def prove(src_block):
        # create_proof overwrites the advice columns' blinding rows (the last 6 of 2^k) with fresh randomness on every call and
        # reads nothing else of them, so the resident block serves every step as it is
        cols = [src_block[i] for i in range(src_block.shape[0])]
        return PL.create_proof(be, pk, cols[:n_inst], cols[n_inst:], rng, PL.Blake2bWrite(be.q, be.p))

    proof = None
    for _ in range(max(args.warmup, 3)):
        proof = prove(block)
    barrier()

    # ---- timed region: K proofs, CUDA events on the prover's stream ---------------------------------------------------------------
    ctx.prof_reset(); ctx.prof_enable(True)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        time.sleep(0.25)
    launches0 = ctx.launches
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    w0 = time.time()
    e0.record(stream)
    for _ in range(args.steps):
        proof = prove(block)
    e1.record(stream)
    barrier()
    w1 = time.time()
    elapsed_ms = e0.elapsed_time(e1)
    launches = ctx.launches - launches0
    clocks = sampler.stop(w0, w1) if rank == 0 else None
    prof, work = ctx.prof_get(), ctx.prof_work()
    ctx.prof_enable(False)
    t = torch.tensor([elapsed_ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    elapsed_ms = float(t.item())
    seconds = elapsed_ms * 1e-3 / args.steps
    value = 1.0 / seconds
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, proof)

    # ---- end to end: the witness starts in pinned host memory every step, the proof bytes end on the host ----------------------------
    up = torch.empty_like(block)

    def e2e_step():
        return prove(host_witness.upload(be, up))

    e2e_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        proof_e2e = e2e_step()
    barrier()
    e2e_s = time.perf_counter() - t0
    t = torch.tensor([e2e_s], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_seconds = float(t.item()) / args.steps

    # ---- the proof is checked in band: the package's verifier on the device, and the same bytes on every rank ---------------------
    d_inst = [block[i] for i in range(n_inst)]
    t0 = time.perf_counter()
    try:
        V.verify_proof(be, pk.vk, V.SingleVerifier(be), d_inst, V.Blake2bRead(proof_e2e, be.q, be.p))
        verified, verify_err = True, None
        bad = bytearray(proof_e2e); bad[len(bad) // 3] ^= 2
        try:
            V.verify_proof(be, pk.vk, V.SingleVerifier(be), d_inst, V.Blake2bRead(bytes(bad), be.q, be.p))
            tamper_rejected = False
        except V.VerifyError:
            tamper_rejected = True
    except V.VerifyError as e:
        verified, verify_err, tamper_rejected = False, str(e), None
    t_verify = time.perf_counter() - t0
    digest = hashlib.sha256(proof_e2e).digest()
    same = True
    if world > 1:
        tt = torch.tensor(list(digest), dtype=torch.uint8, device="cuda")
        parts = [torch.empty_like(tt) for _ in range(world)]
        dist.all_gather(parts, tt)
        same = all(bool(torch.equal(parts[0], q)) for q in parts)

    if rank == 0:
        peaks, peak_src = _peaks()
        # integer-multiply peak, measured now: carry-chained 32x32+64 wide MACs (SASS: IMAD.WIDE.U32[.X] only); cross-check: the
        # 32-bit IMAD issue rate / 2 (a wide MAC occupies two fmaheavy issue slots on sm_100a, profiles/int_pipe_r01.md)
        int_peak_gmacs = max(ctx.microbench(3, 512), ctx.microbench(0, 512))
        imad32_g = ctx.microbench(1, 512)
        peak = int_peak_gmacs / 1e3
        share = {k: round(v[0] / elapsed_ms, 4) for k, v in prof.items() if v[1]}
        # dominant kernel of a proof: the NTT pass kernel (every polynomial goes Lagrange -> coefficients once and coefficients ->
        # coset values on j - 1 cosets).  work = radix-2 butterflies of the launches timed (trp_prof_get_work), 1 butterfly = 1 Fmul
        ntt_ms, ntt_launches = prof["ntt_pass"]
        butterflies = work["ntt_pass"]
        ntt_tmacs = butterflies * MACS_PER_FMUL / (ntt_ms * 1e-3) / 1e12 if ntt_ms else 0.0
        traffic, traffic_src = _traffic_from_profiles("ntt_pass_reg_kernel", "ncu_ntt_r*.json")
        log_n = K_LOG
        passes = -(-log_n // 10)
        bytes_alg = butterflies / (log_n / 2.0) * 64 if log_n else 0       # butterflies / (N/2 log N) transforms x 2 N x 32 B each
        roofline = {"bound": "int32-pipe", "kernel": "ntt_pass_reg_kernel", "achieved": ntt_tmacs, "peak": peak, "unit": "TMAC/s",
                    "frac": ntt_tmacs / peak if peak else None,
                    "traffic": traffic, "traffic_unit": "dram bytes read+written per launch of 8 columns x 2^20 (ncu --set full)", "traffic_source": traffic_src,
                    "peak_source": "wide-MAC (IMAD.WIDE.U32.X chain) microbenchmark run in this process; MEASURED_PEAKS.json has no integer peak. "
                                   "SURVEY 8(d)'s model: 1 Fmul = 128 wide MACs = 256 IMAD slots",
                    "imad32_tops": imad32_g / 1e3, "launch_ms": ntt_ms / max(ntt_launches, 1), "launches_timed": ntt_launches,
                    "algorithmic_macs_per_launch": butterflies * MACS_PER_FMUL / max(ntt_launches, 1),
                    "model": f"radix-2 butterflies of every pass launched x {MACS_PER_FMUL} MAC (1 Fmul per butterfly); {passes} passes per 2^{log_n} transform",
                    "hbm": {"algorithmic_bytes": bytes_alg, "gbs": bytes_alg / (ntt_ms * 1e-3) / 1e9 if ntt_ms else None,
                            "peak_gbs": peaks.get("hbm_gbs"), "peak_source": peak_src,
                            "note": "a 255-bit NTT is ~14x above the HBM balance point (SURVEY.md 0.5): the binding roofline is the integer pipe"},
                    "phase_share_of_step": share,
                    "other_kernels": "msm_accum_l1 (uniform scalars) and quotient_vm against the same peak: extras.msm.roofline, profiles/"}
        cpu = None
        if world == 1 and not args.no_cpu:
            try:
                S = CpuProofSampler()
                est, per, sample_s = S.sample()
                cpu = S.describe(per, sample_s)
                cpu.update({"value": 1.0 / est, "unit": UNIT, "estimated_create_proof_seconds": round(est, 1)})
            except Exception as e:      # the headline line must still print
                cpu = {"error": repr(e)}
        extras = None
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
                "ms_per_step": seconds * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
                "dtype": DTYPE, "data": "synthetic",
                "config": _config({"parallelism": ("one GPU" if world == 1 else
                                                   f"one proof over {world} GPUs: commitments / iNTTs / lookups / permutation chunks by column, quotient NTTs by column block and program by row slice; openings and IPA replicated"),
                                   "trace_steps": len(tr.exe), "advice": cs.num_advice, "instance": cs.num_instance, "fixed": cs.num_fixed,
                                   "gates": len(cs.gates), "lookups": len(cs.lookups), "equality_columns": len(cs.permutation), "degree": cs.degree()}),
                "create_proof_seconds": seconds, "proof_bytes": len(proof_e2e), "proof_sha256": hashlib.sha256(proof_e2e).hexdigest(),
                "verified": verified, "verify_error": verify_err, "tampered_proof_rejected": tamper_rejected, "verify_seconds": round(t_verify, 3),
                "proof_identical_on_all_ranks": same,
                "roofline": roofline, "cpu_baseline": cpu, "clocks": clocks,
                "e2e": {"value": 1.0 / e2e_seconds, "unit": UNIT, "seconds": e2e_seconds, "h2d_bytes_per_step": host_witness.bytes,
                        "d2h_bytes_per_step": len(proof_e2e),
                        "scope": "witness columns (instance + advice) from pinned host memory -> device, create_proof, proof bytes on the host; "
                                 "witness SYNTHESIS (host, unchanged Rust in the integration) is setup.witness_synthesis_s"},
                "gpu_launches": launches,
                "setup": {"witness_synthesis_s": round(t_witness, 3), "params_new_and_tables_s": round(t_params, 3), "upload_s": round(t_upload, 3),
                          "keygen_s": round(t_keygen, 3), "torch_peak_gib": round(torch.cuda.max_memory_allocated() / 2**30, 1)},
                "extras": None}
    # ---- extras (one GPU): the MSM and NTT lines of BASELINE.json's composite metric ---------------------------------------------
    if world == 1 and not args.no_extras:
        del up, block, host_witness
        be.close(); be = None; pk = None
        import gc
        gc.collect(); torch.cuda.empty_cache()
        try:
            line["extras"] = measure_extras(pkg, ctx, stream, peaks, peak_src, peak)
        except Exception as e:
            line["extras"] = {"error": repr(e)}
    if rank == 0:
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    ok = verified and same
    sys.exit(0 if ok else 1)


def dump_outputs(out_dir, proof: bytes):
    """What a caller of create_proof receives from the last timed step: the serialized proof, one float32 per byte (exact)."""
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "proof.npy"), np.frombuffer(proof, dtype=np.uint8).astype(np.float32))


def measure_extras(pkg, ctx, stream, peaks, peak_src, int_peak_tmacs):
    """MSM Mpts/s and NTT GB/s (BASELINE.json configs[1] / configs[2] at 2^20), device resident and through the host-buffer C ABI"""
    import ctypes
    import torch
    from tiny_ram_halo2_b200 import synthetic
    from tiny_ram_halo2_b200._lib import ptr
    out = {}
    lib = ctx.lib
    n, m, steps = N_POINTS, M_COLS, 10
    # ---- MSM: 8 commit_lagrange-shaped columns of 2^20 + 1 Vesta points, uniform scalars ----------------------------------------
    d_pts = torch.empty((n, 8), dtype=torch.int64, device="cuda")
    torch.cuda.synchronize()
    synthetic.device_points(ctx, n, d_pts.data_ptr())
    hb = ctypes.c_void_p()
    ctx.check(lib.trp_dev_bases_load(ctx.handle, d_pts.data_ptr(), n, ctypes.byref(hb)))
    ctx.sync()
    desc = (ctypes.c_uint * 3)()
    ctx.check(lib.trp_bases_describe(hb, desc))
    c_bits, windows, precomp = int(desc[0]), int(desc[1]), bool(desc[2])
    h_scalars = torch.from_numpy(synthetic.random_scalars(n, 20, m).view(np.int64)).pin_memory()
    d_scalars = h_scalars.cuda()
    d_out = torch.zeros((m, 12), dtype=torch.int64, device="cuda")
    torch.cuda.synchronize()
    step = lambda: ctx.check(lib.trp_dev_msm_batch(ctx.handle, hb, d_scalars.data_ptr(), n, m, d_out.data_ptr()))
    for _ in range(3):
        step()
    torch.cuda.synchronize()
    ctx.prof_reset(); ctx.prof_enable(True)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(steps):
        step()
    e1.record(stream)
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    prof = ctx.prof_get()
    ctx.prof_enable(False)
    h_out = torch.zeros((m, 12), dtype=torch.int64).pin_memory()
    e2e = lambda: ctx.check(lib.trp_msm_batch(ctx.handle, hb, h_scalars.data_ptr(), n, m, h_out.data_ptr()))
    e2e(); torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(steps):
        e2e()
    torch.cuda.synchronize()
    e2e_ms = (time.perf_counter() - t0) / steps * 1e3
    acc_ms, acc_launches = prof["msm_accum_l1"]
    per_launch_ms = acc_ms / max(acc_launches, 1)
    # windows that actually receive digits: ceil(255 / c) (scalars are 255 bits; a 16th window at c = 17 only takes carries)
    live_windows = min(windows, -(-255 // c_bits))
    macs = m * n * live_windows * FMUL_PER_MIXED_ADD * MACS_PER_FMUL
    traffic, traffic_src = _traffic_from_profiles("msm_accum_l1", "ncu_accum_r*.json")
    out["msm"] = {"workload": f"{m} columns x (2^{K_LOG}+1) Vesta points, uniform Fp scalars, one resident base table (BASELINE.json configs[1])",
                  "Mpts_per_s": m * n / ms / 1e3, "ms_per_step": ms, "window_bits": c_bits, "windows": windows, "precomputed_bases": precomp,
                  "e2e_Mpts_per_s": m * n / e2e_ms / 1e3, "e2e_h2d_bytes_per_step": m * n * 32, "e2e_d2h_bytes_per_step": m * 96,
                  "e2e_matches_device_path": bool(torch.equal(h_out.cuda(), d_out)),
                  "roofline": {"bound": "int32-pipe", "kernel": "msm_accum_l1_seg_kernel", "achieved": macs / (per_launch_ms * 1e-3) / 1e12,
                               "peak": int_peak_tmacs, "unit": "TMAC/s", "frac": macs / (per_launch_ms * 1e-3) / 1e12 / int_peak_tmacs,
                               "launch_ms": per_launch_ms, "traffic": traffic, "traffic_source": traffic_src,
                               "model": f"cols*n*W*{FMUL_PER_MIXED_ADD} Fmul x {MACS_PER_FMUL} MAC, cols={m}, W={live_windows} windows with digits (table has {windows}), c={c_bits}",
                               "phase_ms_per_step": {k: round(v[0] / steps, 3) for k, v in prof.items() if v[1]}}}
    try:
        sys.path.insert(0, os.path.join(ROOT, "oracle")); sys.path.insert(0, os.path.join(ROOT, "tests"))
        import oracle as O
        cores = O.hw_threads()
        pts_h = d_pts.cpu().numpy().view(np.uint64)
        sc_h = h_scalars.numpy().view(np.uint64)
        t0 = time.perf_counter()
        want = O.msm(O.VESTA, sc_h[0], pts_h, threads=cores)
        dt = time.perf_counter() - t0
        got = O.jacobian_to_affine(O.VESTA, d_out[0].cpu().numpy().view(np.uint64).reshape(3, 4))
        out["msm"]["cpu_baseline"] = {"Mpts_per_s": n / dt / 1e6, "cores": cores, "kind": "port", "equals_gpu_result": bool(np.array_equal(got, want)),
                                      "sample": f"one best_multiexp of 2^{K_LOG}+1 points on {cores} threads (oracle/liboracle.so), column 0 of the GPU step"}
    except Exception as e:
        out["msm"]["cpu_baseline"] = {"error": repr(e)}
    lib.trp_bases_free(hb)
    del d_pts, d_scalars
    # ---- batched NTT, BASELINE configs[2]: 8 columns x 2^20 over Fp, in place, device resident (256 MiB > L2) ---------------------
    logn, batch = K_LOG, 8
    N = 1 << logn
    a = torch.randint(0, 1 << 62, (batch, N, 4), dtype=torch.int64, device="cuda")
    dom = pkg.EvaluationDomain(ctx, 6, logn)
    fn = lambda: ctx.check(lib.trp_dev_ntt(ctx.handle, a.data_ptr(), batch, logn, ptr(dom.omega)))
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    reps = 10
    e0.record(stream)
    for _ in range(reps):
        fn()
    e1.record(stream)
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    gbs = batch * N * 64 / (ms * 1e-3) / 1e9
    tmacs = batch * (N // 2) * logn * MACS_PER_FMUL / (ms * 1e-3) / 1e12
    out["ntt"] = {"workload": f"{batch} columns x 2^{logn} forward NTT over Fp, in place, device resident", "ms": ms,
                  "algorithmic_gbs": gbs, "hbm_peak_gbs": peaks.get("hbm_gbs"), "hbm_frac": gbs / peaks.get("hbm_gbs"),
                  "hbm_peak_source": peak_src, "algorithmic_tmacs": tmacs, "int_peak_tmacs": int_peak_tmacs,
                  "int_frac": tmacs / int_peak_tmacs, "bound": "int32-pipe (SURVEY.md 0.5: 255-bit NTT is ~14x above the HBM balance point)",
                  "model": "bytes = 2*N*32 per column; MACs = (N/2)*log2(N)*128 per column"}
    try:
        host = O.random_field_mont(O.FP, N, 30)
        omega = np.ascontiguousarray(dom.omega, dtype=np.uint64)
        O.fft(O.FP, host[: 1 << 12], 12, omega, threads=cores)
        t0 = time.perf_counter()
        O.fft(O.FP, host, logn, omega, threads=cores)
        dt = time.perf_counter() - t0
        out["ntt"]["cpu_baseline"] = {"ms_per_column": dt * 1e3, "algorithmic_gbs": N * 64 / dt / 1e9, "cores": cores, "kind": "port",
                                      "sample": f"one 2^{logn} best_fft over Fp on {cores} threads, oracle/liboracle.so"}
    except Exception as e:
        out["ntt"]["cpu_baseline"] = {"error": repr(e)}
    del a
    dom.free()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-extras", action="store_true", help="skip the MSM and NTT lines that follow the headline (N = 1)")
    ap.add_argument("--no-cpu", action="store_true", help="skip the sampled CPU baseline (N = 1)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the proof of the last timed step as DIR/proof.npy (float32, one per byte)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        if args.dump_outputs:
            ap.error("--dump-outputs: the reference arm samples phase timings and produces no proof")
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
