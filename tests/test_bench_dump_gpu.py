"""GPU: `bench.py --dump-outputs DIR` writes what the last timed step returned, and the same arguments give the same
outputs from run to run whatever the number of timed steps (small test model, so each run takes seconds)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run_bench(steps, out_dir):
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(steps), "--warmup", "1", "--model", "test-en",
           "--batch", "3", "--beam", "2", "--decode-steps", "12", "--no-cpu-baseline", "--no-gpu-baseline",
           "--dump-outputs", str(out_dir)]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    assert json.loads(lines[0])["steps"] == steps
    return {f[:-4]: np.load(os.path.join(out_dir, f)) for f in sorted(os.listdir(out_dir))}


@pytest.mark.gpu
def test_bench_dump_outputs_repeatable(tmp_path):
    a = run_bench(1, tmp_path / "a")
    b = run_bench(2, tmp_path / "b")
    assert sorted(a) == ["avg_logprob", "no_speech_prob", "tokens"]
    assert all(v.dtype == np.float64 for v in a.values())
    assert a["tokens"].shape[0] == a["avg_logprob"].shape[0] == a["no_speech_prob"].shape[0] == 3
    assert (a["tokens"][:, 0] >= 0).all() and np.isfinite(a["avg_logprob"]).all()
    for k in a:
        assert np.array_equal(a[k], b[k]), k
