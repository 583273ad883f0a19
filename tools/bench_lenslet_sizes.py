"""Shack-Hartmann lenslets of n = 6, 8, 10 and 12 pixels: throughput of the device-resident integrator loop (env.step on the
device, action = gain * observation) at 20 x 20 lenslets (R = 20 n), one layer, 1024 environments, all sizes in one process
and timed alternately; plus the spots kernel alone (aoenv_shwfs_frame_dm as the step calls it: atmosphere OPD + the DM in
factored form, lit-first order, per-environment maximum, pupil statistics) from CUDA events, and the FP32 rate of its DFT
arithmetic: 12 n^3 FMA per lit lenslet (two pruned 2n-point passes of n inputs, radix-2 split), 2 FLOP each.

Usage: python tools/bench_lenslet_sizes.py [--steps 200] [--warmup 20] [--rounds 3] [--kernel-reps 200] [--out FILE.json]"""
import argparse
import ctypes
import json
import math
import os
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from bench_geometric import device_info, loop  # noqa: E402

# FP32 FMA rate of one B200 measured by tools/microbench/ffma2_rate.cu (DESIGN.md section 4): the reference for the share
FP32_FLOPS = 72e12
SIZES = (6, 8, 10, 12)


def build(n, B, dev):
    import types
    from rlao_b200.Conf.parameter_file_synthetic_SHWFS import initializeParameterFile, layer_profile
    from rlao_b200.OOPAOEnv.OOPAOEnvRazor import OOPAO
    args = types.SimpleNamespace(r0=0.13, L0=25, nSubaperture=20, nPixelPerSubap=n, nLoop=None, gainCL=0.5,
                                 **layer_profile(1))
    env = OOPAO()
    env.set_params_file(initializeParameterFile(args), "")
    env.set_params(args, "shackhartmann", gainCL=0.5, n_envs=B, device=dev, rng="philox", seed=1)
    env.atm.generateNewPhaseScreen(17)
    env.dm.coefs = 0
    env.tel * env.dm * env.wfs
    return env


def spots_kernel_us(env, reps):
    """aoenv_shwfs_frame_dm on the environment's current atmosphere and DM commands, CUDA events over `reps` calls (each
    call is two launches: the reset of the maxima and statistics, then the spots kernel)."""
    from rlao_b200 import _lib
    wfs, B, R = env.wfs, env.n_envs, env.tel.resolution
    b_t, dm = wfs._second_term(env.dm.surface_ref())
    assert b_t is None and dm is not None
    lib, st = _lib.load(), _lib.stream_ptr(wfs.device)
    scale = ctypes.c_float(2 * math.pi / env.source.wavelength)

    def run():
        _lib.check(lib.aoenv_shwfs_frame_dm(
            _lib.ptr(env.atm._opd), None, ctypes.byref(dm), _lib.ptr(wfs._lit_first), _lib.ptr(env.tel._pupil_f),
            _lib.ptr(wfs._amp), _lib.ptr(wfs._valid_u8), B, wfs.nSubap, wfs.n_pix_subap, scale, None, 0,
            _lib.ptr(wfs._frame), _lib.ptr(wfs._envmax), _lib.ptr(wfs._stats), st), "shwfs_frame_dm")
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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--kernel-reps", type=int, default=200)
    ap.add_argument("--envs", type=int, default=1024)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_lenslet_sizes: needs a CUDA device")
    dev, B = torch.device("cuda:0"), args.envs
    name, power = device_info()
    result = dict(device=name, power_limit_and_max_sm_clock=power, steps=args.steps, rounds=args.rounds, n_envs=B,
                  nSubap=20, layers=1, fp32_reference_flops=FP32_FLOPS, date=time.strftime("%Y-%m-%d"), sizes={})
    envs = {n: build(n, B, dev) for n in SIZES}
    obs = {n: e.reset_soft() for n, e in envs.items()}
    for n, e in envs.items():
        obs[n], _ = loop(e, obs[n], args.warmup)
    rates = {n: [] for n in envs}
    for _ in range(args.rounds):                         # alternating: every size sees the same state of the shared machine
        for n, e in envs.items():
            obs[n], ms = loop(e, obs[n], args.steps)
            rates[n].append(B * args.steps / (ms * 1e-3))
    assert all(e._native is not None for e in envs.values())
    for n, e in envs.items():
        us = spots_kernel_us(e, args.kernel_reps)
        n_lit = e.wfs.nValidSubaperture
        dft_flop = 2 * 12 * n ** 3 * n_lit * B
        row = dict(resolution=e.tel.resolution, lit_lenslets=n_lit,
                   env_steps_per_s=dict(median=sorted(rates[n])[args.rounds // 2], all=rates[n]),
                   spots_kernel_us=us, dft_flop=dft_flop, dft_tflops=dft_flop / (us * 1e-6) / 1e12,
                   dft_share_of_fp32_reference=dft_flop / (us * 1e-6) / FP32_FLOPS,
                   strehl_mean=float(e._strehl.float().mean()))
        result["sizes"][str(n)] = row
        print(json.dumps({n: row}), flush=True)
    if args.out:
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
