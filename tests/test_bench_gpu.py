"""GPU: `bench.py --dump-outputs` writes the embeddings of the last timed step, and two runs with the same arguments write
the same array (seeded inputs, deterministic kernels), so two builds can be compared output for output."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run_bench(out_dir, steps):
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--forward-only", "--clips", "96", "--steps", str(steps), "--warmup", "1",
           "--dump-outputs", str(out_dir)]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    return json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])


def test_bench_dump_outputs_is_repeatable(tmp_path):
    a = run_bench(tmp_path / "a", 2)
    b = run_bench(tmp_path / "b", 3)
    assert a["steps"] == 2 and b["steps"] == 3
    assert sorted(os.listdir(tmp_path / "a")) == ["embeddings.npy"]
    ea, eb = np.load(tmp_path / "a" / "embeddings.npy"), np.load(tmp_path / "b" / "embeddings.npy")
    assert ea.dtype == np.float32 and ea.shape == (96, 256)
    assert np.allclose(np.linalg.norm(ea, axis=1), 1.0, atol=1e-5)
    assert np.array_equal(ea, eb)
