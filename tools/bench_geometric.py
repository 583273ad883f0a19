"""Geometric against diffractive Shack-Hartmann: throughput of the device-resident integrator loop (env.step on the
device, action = gain * observation) for cfg2, cfg3 and cfg5, both sensors in one process and timed alternately, plus the
geometric kernel alone (aoenv_shwfs_geometric as the step calls it: atmosphere OPD + the DM in factored form, pupil
statistics, GEMM operand planes) from CUDA events, its algorithmic bytes and their rate against the 7.7 TB/s data-sheet
bandwidth of one B200.

Usage: python tools/bench_geometric.py [--steps 200] [--warmup 20] [--rounds 3] [--kernel-reps 200] [--out FILE.json]"""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

HBM_BYTES_PER_S = 7.7e12                  # NVIDIA HGX B200 data sheet, per GPU
L2_BYTES = 126 * 2 ** 20
WORKLOADS = {"cfg2": (20, 1, 1024), "cfg3": (40, 3, 1024), "cfg5": (80, 5, 256)}


def build(nS, nL, B, geometric, dev):
    import types
    from rlao_b200.Conf.parameter_file_synthetic_SHWFS import initializeParameterFile, layer_profile
    from rlao_b200.OOPAOEnv.OOPAOEnvRazor import OOPAO
    args = types.SimpleNamespace(r0=0.13, L0=25, nSubaperture=nS, nLoop=None, gainCL=0.5, is_geometric=geometric,
                                 **layer_profile(nL))
    env = OOPAO()
    env.set_params_file(initializeParameterFile(args), "")
    env.set_params(args, "shackhartmann", gainCL=0.5, n_envs=B, device=dev, rng="philox", seed=1)
    env.atm.generateNewPhaseScreen(17)
    env.dm.coefs = 0
    env.tel * env.dm * env.wfs
    return env


def loop(env, obs, steps):
    """Device-resident loop; returns (last observation, ms) from CUDA events around `steps` steps."""
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(steps):
        obs, _, _, _, _ = env.step(None, env.gainCL * obs)
    e1.record()
    torch.cuda.synchronize()
    return obs, e0.elapsed_time(e1)


def kernel_time(env, reps):
    """aoenv_shwfs_geometric on the environment's current atmosphere and DM commands, CUDA events over `reps` launches
    (each call also resets the statistics: two launches)."""
    from rlao_b200 import gemm
    wfs, B = env.wfs, env.n_envs
    planes = wfs._signal_planes if gemm.uses_tensor_cores(B) else None
    run = lambda: wfs._run_geometric(env.atm._opd, env.dm.surface_ref(), wfs._signal, 1.0 / wfs.slopes_units, planes,
                                     wfs._stats)
    for _ in range(5):
        run()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(reps):
        run()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps * 1e3


def algorithmic_bytes(env):
    """Bytes the measurement has to move, from shapes: per environment the OPD (R*R float32), the nAct T rows of the DM
    (nAct * R float32), slopes (2 nV float32) + their two bf16 planes, the statistics (4 float64); once per launch the
    pupil, flux and the DM row weights."""
    wfs, dm, B = env.wfs, env.dm, env.n_envs
    R, nV = env.tel.resolution, wfs.nValidSubaperture
    per_env = R * R * 4 + dm.nAct * R * 4 + 2 * nV * 4 + 2 * 2 * nV * 2 + 4 * 8
    shared = 2 * R * R * 4 + R * 2 * 12 * 4
    return B * per_env + shared, B * R * R * 4


def device_info():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                            os.environ.get("CUDA_VISIBLE_DEVICES", "0").split(",")[0]], capture_output=True, text=True,
                           timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        q = f"unavailable ({e})"
    return name, q


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--kernel-reps", type=int, default=200)
    ap.add_argument("--workloads", default="cfg2,cfg3,cfg5")
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_geometric: needs a CUDA device")
    dev = torch.device("cuda:0")
    name, power = device_info()
    result = dict(device=name, power_limit_and_max_sm_clock=power, steps=args.steps, rounds=args.rounds,
                  date=time.strftime("%Y-%m-%d"), workloads={})
    for wl in args.workloads.split(","):
        nS, nL, B = WORKLOADS[wl]
        envs = {"diffractive": build(nS, nL, B, False, dev), "geometric": build(nS, nL, B, True, dev)}
        obs = {k: e.reset_soft() for k, e in envs.items()}
        for k, e in envs.items():
            obs[k], _ = loop(e, obs[k], args.warmup)
        rates = {k: [] for k in envs}
        for _ in range(args.rounds):                     # alternating: both see the same state of the shared machine
            for k, e in envs.items():
                obs[k], ms = loop(e, obs[k], args.steps)
                rates[k].append(B * args.steps / (ms * 1e-3))
        assert all(e._native is not None for e in envs.values())
        us = kernel_time(envs["geometric"], args.kernel_reps)
        nbytes, opd_bytes = algorithmic_bytes(envs["geometric"])
        row = dict(n_envs=B, nSubap=nS, layers=nL,
                   env_steps_per_s={k: dict(median=sorted(v)[len(v) // 2], all=v) for k, v in rates.items()},
                   geometric_over_diffractive=sorted(rates["geometric"])[args.rounds // 2]
                   / sorted(rates["diffractive"])[args.rounds // 2],
                   geometric_kernel_us=us, algorithmic_bytes=nbytes, achieved_GBps=nbytes / (us * 1e-6) / 1e9,
                   share_of_hbm_datasheet=nbytes / (us * 1e-6) / HBM_BYTES_PER_S,
                   opd_fits_l2=opd_bytes < L2_BYTES,
                   strehl_mean={k: float(e._strehl.float().mean()) for k, e in envs.items()})
        result["workloads"][wl] = row
        print(json.dumps({wl: row}), flush=True)
        del envs, obs
        torch.cuda.empty_cache()
    if args.out:
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
