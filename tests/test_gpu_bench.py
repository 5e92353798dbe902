"""GPU test of bench.py --dump-outputs on a small instance of the benchmark circuit (TRP_BENCH_K = 10): the proof of the last
timed step is written as float32 bytes, and two runs with the same arguments write the same proof (the prover's RNG is
keyed by a fixed seed), so two builds of the project can be compared output for output."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(out_dir):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "2", "--warmup", "1", "--no-cpu",
                        "--no-extras", "--dump-outputs", str(out_dir)], env={**os.environ, "TRP_BENCH_K": "10"},
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    lines = [json.loads(l) for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    return lines[0], np.load(os.path.join(out_dir, "proof.npy"))


def test_dump_outputs_is_the_same_proof_in_every_run(tmp_path):
    line, a = _run(tmp_path / "a")
    assert line["steps"] == 2 and line["verified"] is True
    assert a.dtype == np.float32 and a.shape == (line["proof_bytes"],)
    assert np.array_equal(a, np.round(a)) and a.min() >= 0 and a.max() <= 255
    _, b = _run(tmp_path / "b")
    assert np.array_equal(a, b)
