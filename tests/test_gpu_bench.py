"""bench.py on the GPU: --steps sets the number of timed steps, and --dump-outputs writes what the last of them returned,
the same arrays from run to run for the same arguments."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

pytestmark = pytest.mark.gpu


def _bench(out_dir):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "tiny", "--steps", "3", "--warmup", "3",
                          "--no-cpu-baseline", "--dump-outputs", str(out_dir)], capture_output=True, text=True, timeout=900,
                         cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    return json.loads(lines[0])


def test_bench_dumps_the_outputs_of_its_last_timed_step(tmp_path):
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    runs = [tmp_path / "a", tmp_path / "b"]
    for d in runs:
        line = _bench(d)
        assert line["steps"] == 3 and line["config"]["envs_per_gpu"] == 64
    a, b = ({f[:-4]: np.load(d / f) for f in sorted(os.listdir(d))} for d in runs)
    assert set(a) == {"obs", "reward", "strehl"}
    assert a["obs"].shape == (64, 9, 9) and a["reward"].shape == a["strehl"].shape == (64,)
    for k in a:
        assert a[k].dtype == np.float32 and np.isfinite(a[k]).all(), k
        assert np.array_equal(a[k], b[k]), k
    assert np.abs(a["obs"]).max() > 0 and (a["strehl"] > 0).all()
