"""bench.py contract checks that need no GPU: the reference arm prints one JSON line with the agreed keys, and the
non-zero ranks of a torchrun launch stay silent."""
import json
import os
import subprocess
import sys

from oracle import ref_harness

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(env_extra=None):
    env = dict(os.environ)
    env.update(env_extra or {})
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "tiny",
                          "--steps", "1", "--warmup", "0"], capture_output=True, text=True, timeout=300, env=env, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    return [ln for ln in out.stdout.splitlines() if ln.startswith("{")]


def test_reference_arm_prints_one_contract_line():
    lines = _run()
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "closed-loop AO env-steps/sec (batched envs)" and d["unit"] == "env-steps/s"
    assert d["higher_is_better"] is True and d["value"] > 0 and d["gpu_launches"] == 0
    # "reference" = the unmodified reference, when a copy of it is present; "port" otherwise
    assert d["cpu_baseline"]["kind"] == ("reference" if ref_harness.reference_available() else "port")
    assert d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["steps"] >= 2 and d["ms_per_step"] > 0          # the steps really timed, not the requested ones
    assert d["e2e"] == {"value": d["value"], "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["config"]["workload"] == "tiny" and d["vs_baseline"] is None


def test_reference_arm_other_ranks_are_silent():
    assert _run({"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"}) == []


def test_dump_outputs_writes_float_arrays_within_the_size_limit(tmp_path, monkeypatch):
    import numpy as np
    import torch
    import bench
    bench.dump_outputs(tmp_path / "one", {"obs": torch.ones(9, 9), "reward": torch.tensor(2, dtype=torch.int32)}, 1)
    one = {f: np.load(tmp_path / "one" / f) for f in os.listdir(tmp_path / "one")}
    assert {k: (v.dtype, v.shape) for k, v in one.items()} == {"obs.npy": (np.float32, (1, 9, 9)), "reward.npy": (np.float32, (1,))}
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", 4000)
    obs = torch.arange(100 * 20, dtype=torch.float64).reshape(100, 20)
    for d in ("a", "b"):
        bench.dump_outputs(tmp_path / d, {"obs": obs, "reward": obs[:, 0].float()}, 100)
    a, b = ({f: np.load(tmp_path / d / f) for f in os.listdir(tmp_path / d)} for d in ("a", "b"))
    assert set(a) == {"obs.npy", "reward.npy", "env_index.npy"} and sum(v.nbytes for v in a.values()) <= 4000
    assert all(np.array_equal(a[k], b[k]) for k in a)                   # a fixed sample
    idx = a["env_index.npy"].astype(np.int64)
    assert a["obs.npy"].dtype == np.float64 and np.array_equal(a["obs.npy"], obs.numpy()[idx])
    assert a["reward.npy"].dtype == np.float32 and np.array_equal(a["reward.npy"], obs.numpy()[idx, 0])
