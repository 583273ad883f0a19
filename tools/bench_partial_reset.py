"""Per-environment episode resets at cfg3 (40 x 40 lenslets, three layers, 1024 environments):

1. OOPAO.reset_envs for k = 1, 16, 128 and 1024 environments, next to Atmosphere.generateNewPhaseScreen in the same process
   (device time from CUDA events around `--reps` calls after a warm-up; host time per call; launches per call);
2. env-steps/s of GymnasiumVectorSH in a device-resident loop (action = gain * newest observation) with episode_length=500
   and staggered episodes (about two resets per call at 1024 environments), against the same wrapper with
   episode_length=None (no resets), alternated over `--rounds` rounds.

Usage: python tools/bench_partial_reset.py [--reps 20] [--steps 300] [--warmup 30] [--rounds 3] [--out FILE.json]"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def build(dev, B=1024, nS=40, nL=3):
    import bench
    from rlao_b200.OOPAOEnv.OOPAOEnvRazor import OOPAO
    env = OOPAO()
    env.set_params_file("rlao_b200.Conf.parameter_file_synthetic_SHWFS", "")
    env.set_params(bench.make_args(nS, nL), "shackhartmann", gainCL=0.5, n_envs=B, device=dev, rng="philox", seed=1)
    env.atm.generateNewPhaseScreen(17)
    env.dm.coefs = 0
    env.tel * env.dm * env.wfs
    return env


def device_info():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                            os.environ.get("CUDA_VISIBLE_DEVICES", "0").split(",")[0]], capture_output=True, text=True,
                           timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        q = f"unavailable ({e})"
    return name, q


def timed(fn, reps):
    """(device ms per call from CUDA events, host ms per call, launches per call) over `reps` calls."""
    from rlao_b200 import _lib
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    n0, t0 = _lib.launch_count(), time.perf_counter()
    e0.record()
    for r in range(reps):
        fn(r)
    e1.record()
    torch.cuda.synchronize()
    host = (time.perf_counter() - t0) * 1e3 / reps
    return e0.elapsed_time(e1) / reps, host, (_lib.launch_count() - n0) / reps


def reset_times(env, reps, rounds):
    B, rng = env.n_envs, np.random.RandomState(0)
    out = {}
    for _ in range(rounds):                              # alternating: every variant sees the same state of the machine
        for k in (1, 16, 128, 1024):
            ids = [np.sort(rng.choice(B, size=k, replace=False)) for _ in range(reps)]
            env.reset_envs(ids[0], 1)                    # warm-up (also computes the next frame: later calls reuse it)
            dev_ms, host_ms, launches = timed(lambda r: env.reset_envs(ids[r], 1000 + r), reps)
            out.setdefault(f"reset_envs_k{k}", []).append(dict(device_ms=dev_ms, host_ms=host_ms, launches=launches))
        env.atm.generateNewPhaseScreen(5)
        dev_ms, host_ms, launches = timed(lambda r: env.atm.generateNewPhaseScreen(2000 + r), reps)
        out.setdefault("generateNewPhaseScreen", []).append(dict(device_ms=dev_ms, host_ms=host_ms, launches=launches))
    med = lambda v, key: sorted(x[key] for x in v)[len(v) // 2]
    return {name: dict(device_ms_median=med(v, "device_ms"), host_ms_median=med(v, "host_ms"), launches=v[0]["launches"],
                       rounds=v) for name, v in out.items()}


def wrapper_rates(envs, steps, warmup, rounds):
    from rlao_b200 import _lib
    from rlao_b200.OOPAOEnv.gymnasium_api import GymnasiumVectorSH
    vecs = {"staggered_500": GymnasiumVectorSH(envs[0], n_history=2, episode_length=500, stagger_episodes=True),
            "no_resets": GymnasiumVectorSH(envs[1], n_history=2, episode_length=None)}
    obs = {k: v.reset(seed=3)[0] for k, v in vecs.items()}
    stats = {k: dict(env_steps_per_s=[], resets_per_call=[], launches_per_call=[]) for k in vecs}

    def run(k, n):
        v, o = vecs[k], obs[k]
        resets = 0
        for _ in range(n):
            resets += int(v._pending.sum())
            o = v.step(v.env.gainCL * o[:, 0])[0]
        obs[k] = o
        return resets
    for k in vecs:
        run(k, warmup)
    for _ in range(rounds):
        for k, v in vecs.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            n0 = _lib.launch_count()
            e0.record()
            resets = run(k, steps)
            e1.record()
            torch.cuda.synchronize()
            s = stats[k]
            s["env_steps_per_s"].append(v.num_envs * steps / (e0.elapsed_time(e1) * 1e-3))
            s["resets_per_call"].append(resets / steps)
            s["launches_per_call"].append((_lib.launch_count() - n0) / steps)
    for s in stats.values():
        s["median_env_steps_per_s"] = sorted(s["env_steps_per_s"])[len(s["env_steps_per_s"]) // 2]
    return stats


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--steps", type=int, default=300)
    ap.add_argument("--warmup", type=int, default=30)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_partial_reset: needs a CUDA device")
    dev = torch.device("cuda:0")
    name, power = device_info()
    result = dict(device=name, power_limit_and_max_sm_clock=power, workload="cfg3 (40x40 SH, 3 layers), 1024 environments",
                  date=time.strftime("%Y-%m-%d"), reps=args.reps, steps=args.steps, rounds=args.rounds)
    envs = [build(dev), build(dev)]
    result["reset"] = reset_times(envs[0], args.reps, args.rounds)
    print(json.dumps({"reset": {k: v["device_ms_median"] for k, v in result["reset"].items()}}), flush=True)
    result["wrapper"] = wrapper_rates(envs, args.steps, args.warmup, args.rounds)
    print(json.dumps({"wrapper": {k: v["median_env_steps_per_s"] for k, v in result["wrapper"].items()}}), flush=True)
    if args.out:
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
