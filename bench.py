#!/usr/bin/env python
"""bench.py — closed-loop AO env-steps/s (batched environments) on N B200s, next to the CPU baseline.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--workload cfg3|cfg2|cfg1|tiny]

A "step" is one `env.step` of every environment on every GPU (integrator policy action = gainCL * obs).
Default workload (BASELINE.json configs[2], the one the 1e6 env-steps/s target is quoted on): 8 m telescope,
40x40 SH-WFS, 41x41 DM, 3-layer von Karman atmosphere, 1024 environments PER GPU (8192 on 8 GPUs, weak scaling).
Prints ONE JSON line (see the task contract): value = device-timed throughput with inputs resident in HBM,
e2e = same metric through the host-facing TorchWrapper (pinned host action in, host obs/reward/Strehl out,
copies inside the timed region), roofline of the dominant kernel, cpu_baseline (oracle port on host cores).
Extra keys: `e2e_lookahead` (the same loop through TorchWrapper(lookahead=True), opt-in), `kernels` (per C-ABI entry point,
CUDA events, separate pass), `roofline.fp32` when the dominant kernel is the FMA-bound SH-WFS transform.
Other workloads: --workload cfg1|cfg2|cfg3noise|cfg4|cfg4lowflux|cfg5|cfg5psf|tiny; --policy po4ao runs ConvPolicy rollouts.
--dump-outputs DIR writes what the last timed step of the device-resident loop returned (obs, reward, Strehl; the last
rollout step's obs and reward and the reward sums with --policy po4ao) as DIR/<name>.npy.  The environments, atmosphere and
policy weights are seeded, so the same arguments give the same inputs and two builds can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time
import types

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (nSubap, nLayers, envs per GPU, description, options)
    "cfg3": (40, 3, 1024, "8m 40x40 SH-WFS, 41x41 DM (1353 act), 3-layer VK atmosphere, integrator, noise off", {}),
    "cfg3noise": (40, 3, 1024, "cfg3 with the reference environment's default camera: photon noise, RON 14 e-, QE 0.56, dark 5, "
                               "FWC 1e4, 10-bit ADC (OOPAOEnvRazor.py:243-250,332-333)", {"noise": True}),
    "cfg2": (20, 1, 1024, "8m 20x20 SH-WFS, 21x21 DM (357 act), 1-layer VK atmosphere, integrator, noise off", {}),
    "cfg4": (20, 1, 4096, "8m 20x20 SH-WFS, 21x21 DM, 1 layer, Razor-like camera: photon noise, RON 14 e-, QE 0.56, dark 5, "
                          "FWC 1e4, 10-bit ADC", {"noise": True}),
    "cfg4lowflux": (20, 1, 4096, "cfg4 at magnitude 12", {"noise": True, "magnitude": 12}),
    "cfg5": (80, 5, 256, "8m 80x80 SH-WFS, 81x81 DM (5209 act), 5-layer VK atmosphere, integrator, noise off", {}),
    "cfg5psf": (80, 5, 256, "cfg5 with the science-PSF Strehl (zero padding 4, N=1920) as the per-step reward",
                {"psf": (4, 32)}),
    "cfg1": (20, 1, 1, "8m 20x20 SH-WFS, 21x21 DM, 1 layer, single env", {}),
    "tiny": (8, 2, 64, "8m 8x8 SH-WFS test system", {}),
}


def make_args(nSubap, nLayers, opts=None):
    from rlao_b200.Conf.parameter_file_synthetic_SHWFS import layer_profile
    prof = layer_profile(nLayers)
    opts = opts or {}
    extra = {k: opts[k] for k in ("noise", "magnitude") if k in opts}
    return types.SimpleNamespace(r0=0.13, L0=25, nSubaperture=nSubap, nLoop=None, gainCL=0.5, **prof, **extra)


def oracle_config(nSubap, nLayers, opts=None):
    from oracle.ao_oracle import AOConfig, DetectorConfig
    from oracle.golden_configs import RAZOR_DETECTOR
    from rlao_b200.Conf.parameter_file_synthetic_SHWFS import layer_profile
    prof = layer_profile(nLayers)
    opts = opts or {}
    extra = {}
    if opts.get("noise"):
        extra["detector"] = DetectorConfig(**RAZOR_DETECTOR)
    if "magnitude" in opts:
        extra["magnitude"] = float(opts["magnitude"])
    return AOConfig(**extra, nSubap=nSubap, windSpeed=[float(v) for v in prof["windSpeed"]],
                    windDirection=[float(v) for v in prof["windDirection"]], fractionalR0=prof["fractionalR0"],
                    altitude=[0.0] * nLayers, nZernike=50, nLoop=4096)


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, arrays, n_envs):
    """--dump-outputs: writes each of `arrays` (tensors with the environment axis first, or squeezed away when n_envs == 1)
    as <out_dir>/<name>.npy, float64 kept, everything else as float32.  Past DUMP_LIMIT_BYTES in all, the same fixed seeded
    sample of environments is taken from every array and its indices are written as env_index.npy."""
    import numpy as np
    host = {}
    for name, t in arrays.items():
        a = t.detach().cpu().numpy() if hasattr(t, "detach") else np.asarray(t)
        a = a.astype(np.float64 if a.dtype == np.float64 else np.float32)
        host[name] = a[None] if n_envs == 1 else a
    total = sum(a.nbytes for a in host.values())
    if total > DUMP_LIMIT_BYTES:
        keep = max(1, DUMP_LIMIT_BYTES // (total // n_envs + 8))          # + 8: the environment's entry in env_index
        idx = np.sort(np.random.default_rng(0).choice(n_envs, size=keep, replace=False))
        host = {name: a[idx] for name, a in host.items()}
        host["env_index"] = idx.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in host.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


# ---------------------------------------------------------------------------------------------------------
# clocks
# ---------------------------------------------------------------------------------------------------------
class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region (the recipe's clocks line).  Uses NVML in a
    thread of this process (clock + event-reason queries only: `nvidia-smi --query-gpu=...,power.draw -lms` stalls
    kernel launches for tens of milliseconds per sample, which showed up as a 2x slowdown of launch-heavy loops);
    falls back to an `nvidia-smi` poller when the NVML binding is missing."""
    Q = "index,clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown," \
        "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
    PERIOD = 0.004

    def __init__(self, gpu_index):
        self.rows, self.gpu, self.proc, self.nvml, self._stop = [], gpu_index, None, None, threading.Event()

    def _physical_index(self):
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        if vis:
            ids = [v.strip() for v in vis.split(",") if v.strip()]
            if self.gpu < len(ids) and ids[self.gpu].isdigit():
                return int(ids[self.gpu])
        return self.gpu

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nvml = pynvml
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(self._physical_index())
            self.max_sm = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
            threading.Thread(target=self._poll_nvml, daemon=True).start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self._physical_index()), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _poll_nvml(self):
        nv = self.nvml
        names = (("hw_slowdown", nv.nvmlClocksEventReasonHwSlowdown), ("hw_thermal_slowdown", nv.nvmlClocksEventReasonHwThermalSlowdown),
                 ("sw_thermal_slowdown", nv.nvmlClocksEventReasonSwThermalSlowdown), ("sw_power_cap", nv.nvmlClocksEventReasonSwPowerCap))
        while not self._stop.is_set():
            try:
                sm = float(nv.nvmlDeviceGetClockInfo(self.handle, nv.NVML_CLOCK_SM))
                mask = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.handle))
                self.rows.append((time.time(), sm, self.max_sm, [n for n, bit in names if mask & bit]))
            except Exception:
                pass
            self._stop.wait(self.PERIOD)

    def _read(self):
        for line in self.proc.stdout:
            r = [x.strip() for x in line.split(",")]
            try:
                reasons = [n for n, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7])
                           if v.lower().startswith("active")]
                self.rows.append((time.time(), float(r[1]), float(r[2]), reasons))
            except Exception:
                pass

    def stop(self, t0, t1):
        if self.nvml is None and self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no NVML binding and no nvidia-smi"]}
        time.sleep(2 * self.PERIOD)
        self._stop.set()
        if self.proc is not None:
            self.proc.terminate()
        rows = [r for r in self.rows if t0 <= r[0] <= t1 + 2 * self.PERIOD] or self.rows[-3:]
        sm = sorted(r[1] for r in rows)
        reasons = sorted({n for r in rows for n in r[3]})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": rows[-1][2] if rows else None, "reasons": reasons,
                "samples": len(sm), "source": "nvml" if self.nvml is not None else "nvidia-smi"}


# ---------------------------------------------------------------------------------------------------------
# CPU arm (oracle port of the reference step)
# ---------------------------------------------------------------------------------------------------------
def _cpu_worker(env, seed, n_steps, q):
    import numpy as np
    try:
        from threadpoolctl import threadpool_limits
        ctx = threadpool_limits(1)
    except Exception:
        import contextlib
        ctx = contextlib.nullcontext()
    with ctx:
        obs = env.new_episode(seed)
        for i in range(3):
            obs, *_ = env.step(i, env.gainCL * obs)
        t0 = time.perf_counter()
        for i in range(n_steps):
            obs, *_ = env.step(3 + i, env.gainCL * obs)
        q.put((time.perf_counter() - t0, float(np.abs(obs).max())))


def cpu_env(nSubap, nLayers, reconstructor=None, opts=None):
    from oracle.ao_oracle import EnvOracle
    return EnvOracle(oracle_config(nSubap, nLayers, opts), reconstructor=reconstructor)


def reference_env(nSubap, nLayers, opts=None):
    """The UNMODIFIED reference (OOPAO + the drl4ao Razor environment) from the build container's reference tree or, on
    the GPU box, from the copy build() staged under oracle/_ref/; None when neither is there."""
    from oracle import ref_harness
    if not ref_harness.reference_available():
        return None
    return ref_harness.ReferenceStepper(oracle_config(nSubap, nLayers, opts))


def time_cpu(env, n_procs, n_steps):
    """`n_procs` forked workers (read-only operators shared copy-on-write), one environment each, one BLAS
    thread each; returns env-steps/s summed over workers."""
    import multiprocessing as mp
    ctx = mp.get_context("fork")
    q = ctx.Queue()
    procs = [ctx.Process(target=_cpu_worker, args=(env, 100 + r, n_steps, q)) for r in range(n_procs)]
    t0 = time.perf_counter()
    for p in procs:
        p.start()
    res = [q.get() for _ in procs]
    for p in procs:
        p.join()
    wall = time.perf_counter() - t0
    worst = max(r[0] for r in res)
    return n_procs * n_steps / worst, worst, wall


def run_reference_arm(args):
    """--impl reference: the reference's own CPU implementation of the step on all host cores (the unmodified OOPAO +
    drl4ao environment staged under oracle/_ref/ by build(); the oracle port only if that copy is missing), same
    metric/config keys.  A "step" of this arm is one env.step of every worker process's environment; the line reports
    the steps it really timed."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    nS, nL, B, desc, opts = WORKLOADS[args.workload]
    cores = os.cpu_count() or 1
    n_procs = max(1, min(cores, 64))
    t_init = time.perf_counter()
    env, kind = None, "reference"
    try:
        env = reference_env(nS, nL, opts)
    except Exception as ex:
        print(f"reference import failed ({ex!r}); timing the oracle port", file=sys.stderr)
    if env is None:
        env, kind = cpu_env(nS, nL, opts=opts), "port"
    t_init = time.perf_counter() - t_init
    per_step = {8: 0.004, 20: 0.02, 40: 0.12, 80: 0.8}.get(nS, 0.1)          # s per env-step of one process (survey figures)
    n_steps = max(2, int(min(30.0, 1.0 * max(1, args.steps)) / per_step))     # bounded sample: <= 30 s of stepping per worker
    n_warm = max(1, min(args.warmup, 3))
    time_cpu(env, n_procs, n_warm)
    value, worst, wall = time_cpu(env, n_procs, n_steps)
    note = ("UNMODIFIED reference (OOPAO + MAIN_CODE/OOPAOEnv/OOPAOEnvRazor.py, numpy float64; skimage.transform.warp through the "
            "documented restatement oracle/warp018.py)" if kind == "reference" else "oracle port (numpy float64) of the OOPAO/drl4ao step")
    line = {
        "impl": "reference", "metric": "closed-loop AO env-steps/sec (batched envs)", "value": value, "unit": "env-steps/s",
        "n_gpus": args.gpus, "steps": n_steps, "warmup": n_warm + 3, "ms_per_step": 1e3 * worst / n_steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": args.workload, "description": desc, "envs": n_procs, "requested_steps": args.steps,
                   "note": note + ", one environment per host process"},
        "cpu_baseline": {"value": value, "unit": "env-steps/s", "cores": n_procs, "kind": kind,
                         "sample": f"{n_procs} processes x {n_steps} steps of one env each (1 BLAS thread), init {t_init:.1f}s excluded"},
        "e2e": {"value": value, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------------------------------
class KernelTimer:
    """Wraps the C-ABI entry points with CUDA events on the launching stream (used in a separate pass after the
    timed region) to attribute device time to each kernel family."""

    def __init__(self, lib, torch):
        self.lib, self.torch, self.events, self.saved = lib, torch, [], {}

    def __enter__(self):
        from rlao_b200 import _lib
        for name in _lib.PROTOTYPES:
            fn = getattr(self.lib, name)
            self.saved[name] = fn
            setattr(self.lib, name, self._wrap(name, fn))
        return self

    def _wrap(self, name, fn):
        torch = self.torch

        def call(*a):
            key = name
            if name in ("aoenv_gemm_tn", "aoenv_gemm_tn_tc"):
                key = f"{name}[N={a[7]},K={a[8]}]"
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            rc = fn(*a)
            e1.record()
            self.events.append((key, e0, e1))
            return rc
        return call

    def __exit__(self, *exc):
        for name, fn in self.saved.items():
            setattr(self.lib, name, fn)

    def summary(self, n_steps):
        self.torch.cuda.synchronize()
        out = {}
        for key, e0, e1 in self.events:
            d = out.setdefault(key, [0.0, 0])
            d[0] += e0.elapsed_time(e1)
            d[1] += 1
        return {k: {"ms_per_step": v[0] / n_steps, "calls_per_step": v[1] / n_steps, "ms_per_call": v[0] / v[1]} for k, v in out.items()}


def pin_to_gpu_numa_node(local_rank, world):
    """One process per GPU on one host: keep this rank's threads (and therefore its first-touch pinned buffers) on the CPUs
    NVML reports as local to its GPU, split evenly between the ranks that share them.  Returns a short description."""
    try:
        import pynvml
        pynvml.nvmlInit()
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        ids = [int(v) for v in vis.split(",")] if vis and all(v.strip().isdigit() for v in vis.split(",")) else list(range(world))
        words = (os.cpu_count() + 63) // 64
        sets = []
        for g in ids[:world]:
            mask = pynvml.nvmlDeviceGetCpuAffinity(pynvml.nvmlDeviceGetHandleByIndex(g), words)
            sets.append(frozenset(64 * w + b for w, m in enumerate(mask) for b in range(64) if (m >> b) & 1))
        mine = sets[local_rank]
        allowed = sorted(mine & set(os.sched_getaffinity(0)))
        sharers = [r for r in range(len(sets)) if sets[r] == mine]
        if not allowed or len(sharers) == 0:
            return "no NUMA information"
        k, n = sharers.index(local_rank), len(sharers)
        per = max(1, len(allowed) // n)
        cpus = allowed[k * per:(k + 1) * per] or allowed
        os.sched_setaffinity(0, cpus)
        return f"{len(cpus)} CPUs local to GPU {ids[local_rank]} ({cpus[0]}-{cpus[-1]})"
    except Exception as ex:                       # affinity is an optimisation, never a requirement
        return f"not pinned ({type(ex).__name__})"


def run_gpu_arm(args):
    import torch
    import torch.distributed as dist
    from rlao_b200 import _lib
    from rlao_b200.OOPAOEnv.OOPAOEnvRazor import OOPAO
    from rlao_b200.PO4AO.util_simple import TorchWrapper

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    pinned = pin_to_gpu_numa_node(local, world) if world > 1 else "single rank"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    nS, nL, B, desc, opts = WORKLOADS[args.workload]
    if args.envs:
        B = args.envs
    env = OOPAO()
    env.set_params_file("rlao_b200.Conf.parameter_file_synthetic_SHWFS", "")
    env.set_params(make_args(nS, nL, opts), args.wfs, gainCL=0.5, n_envs=B, device=dev, rng="philox", seed=1,
                   env_offset=rank * B)
    if args.wfs == "pyramid":
        desc = desc.replace("SH-WFS", "Pyramid WFS (modulation 3 lambda/D, 20 modulation points, the library's own FFT kernels)")
    env.atm.generateNewPhaseScreen(17)
    env.dm.coefs = 0
    env.tel * env.dm * env.wfs
    obs = env.reset_soft()
    gain = env.gainCL
    if opts.get("psf"):
        env.psf_reward = tuple(opts["psf"])

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident loop ------------------------------------------------------------------------
    for i in range(args.warmup):
        obs, reward, strehl, _, _ = env.step(None, gain * obs)
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
        time.sleep(0.25)
    l0 = _lib.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    t_wall0 = time.time()
    if os.environ.get("AOENV_PROFILE_REGION"):      # lets `ncu --profile-from-start off` see only the timed region
        torch.cuda.profiler.start()
    e0.record()
    for i in range(args.steps):
        obs, reward, strehl, _, _ = env.step(None, gain * obs)
    e1.record()
    barrier()
    if os.environ.get("AOENV_PROFILE_REGION"):
        torch.cuda.profiler.stop()
    t_wall1 = time.time()
    ms = e0.elapsed_time(e1)
    launches = _lib.launch_count() - l0
    clocks = sampler.stop(t_wall0, t_wall1) if rank == 0 else None
    # copies: the environment keeps the returned tensors as its own state, and reset_soft() below writes into them
    last_step = {"obs": obs.clone(), "reward": reward.clone(), "strehl": strehl.clone()} if args.dump_outputs else None
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max = float(t[0])
    value = world * B * args.steps / (ms_max * 1e-3)
    sr_mean = float(strehl.float().mean())

    # ---- end-to-end through the host-facing wrapper (pinned host buffers, copies inside the timed region) ----
    # the host-side "policy" (action = gain * obs on 1.7M floats) may use this rank's share of the host cores
    # (torchrun pins OMP_NUM_THREADS=1 by default)
    torch.set_num_threads(max(1, min(16, len(os.sched_getaffinity(0)) if world > 1 else (os.cpu_count() or 1))))
    wrapped = TorchWrapper(env, host_io=True)
    obs_h = wrapped.reset_soft()
    # The policy works IN PLACE on the pinned observation the wrapper returned (the caller owns it until step t+2) and hands
    # it back as the action: a separate output array makes the multiply move 3 x 6.9 MB per rank and step (read, write-
    # allocate, write) instead of 2 x, and eight ranks doing that on one host are bound by its memory bandwidth — measured
    # at N = 8 with 4 threads per rank: 0.54 ms of the 1.38 ms step were this multiply (profiles/r2_v8_e2e_sweep_8gpu.json).
    for i in range(max(3, args.warmup)):
        torch.mul(obs_h, gain, out=obs_h)
        obs_h, reward_h, strehl_h, _, _ = wrapped.step(None, obs_h)
    barrier()
    e0.record()
    for i in range(args.steps):
        torch.mul(obs_h, gain, out=obs_h)
        obs_h, reward_h, strehl_h, _, _ = wrapped.step(None, obs_h)
    e1.record()
    barrier()
    t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_value = world * B * args.steps / (float(t[0]) * 1e-3)

    # experiment hook (AOENV_BENCH_E2E_SWEEP="1,2,4"): the strict loop again with other thread counts for the host policy
    e2e_sweep = None
    if os.environ.get("AOENV_BENCH_E2E_SWEEP"):
        e2e_sweep = {}
        for nt in [int(v) for v in os.environ["AOENV_BENCH_E2E_SWEEP"].split(",")]:
            torch.set_num_threads(nt)
            for i in range(5):
                torch.mul(obs_h, gain, out=obs_h)
                obs_h, reward_h, strehl_h, _, _ = wrapped.step(None, obs_h)
            barrier()
            t_host = 0.0
            e0.record()
            for i in range(args.steps):
                th0 = time.perf_counter()
                torch.mul(obs_h, gain, out=obs_h)
                t_host += time.perf_counter() - th0
                obs_h, reward_h, strehl_h, _, _ = wrapped.step(None, obs_h)
            e1.record()
            barrier()
            t = torch.tensor([e0.elapsed_time(e1), t_host * 1e3], dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
            e2e_sweep[str(nt)] = {"value": world * B * args.steps / (float(t[0]) * 1e-3), "policy_ms_per_step": float(t[1]) / args.steps}

    # same loop with the opt-in lookahead wrapper (frame t+1 is measured while the host works on step t)
    ahead = TorchWrapper(env, host_io=True, lookahead=True)
    obs_h = ahead.reset_soft()
    for i in range(max(3, args.warmup)):
        torch.mul(obs_h, gain, out=obs_h)
        obs_h, reward_h, strehl_h, _, _ = ahead.step(None, obs_h)
    barrier()
    e0.record()
    for i in range(args.steps):
        torch.mul(obs_h, gain, out=obs_h)
        obs_h, reward_h, strehl_h, _, _ = ahead.step(None, obs_h)
    e1.record()
    barrier()
    ahead.flush()
    t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_ahead = world * B * args.steps / (float(t[0]) * 1e-3)
    nAct2 = env.nActuator ** 2
    h2d, d2h = B * nAct2 * 4, B * nAct2 * 4 + 2 * B * 4

    # ---- per-kernel attribution + roofline of the dominant kernel (rank 0) -----------------------------------
    roofline, kernels = None, None
    if rank == 0:
        n_prof = min(args.steps, 10)
        # attribution needs the step call by call, on one stream: the library-sequenced entry points (aoenv_atm_update,
        # aoenv_sh_step) and the side-stream atmosphere are switched off for this pass only
        saved = (env.native_step, env.atm.native_update, env.atm.pipelined)
        torch.cuda.synchronize()
        env.atm._join_prefetch(consume=True)
        env.native_step, env.atm.native_update, env.atm.pipelined = False, False, False
        with KernelTimer(_lib.load(), torch) as kt:
            o = env._sq(env._obs).clone()
            for i in range(n_prof):
                o, *_ = env.step(None, gain * o)
        env.native_step, env.atm.native_update, env.atm.pipelined = saved
        kernels = kt.summary(n_prof)
        roofline = dominant_roofline(kernels, env, B)
    if world > 1:
        dist.barrier()

    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        try:
            t0 = time.perf_counter()
            orc = cpu_env(nS, nL, reconstructor=env.reconstructor.cpu().numpy(), opts=opts)
            n_cpu = 100 if nS >= 40 else 400
            v, worst, wall = time_cpu(orc, 1, n_cpu)
            cpu_baseline = {"value": v, "unit": "env-steps/s", "cores": 1, "kind": "port",
                            "sample": f"{n_cpu} steps of one environment of the same optical configuration, one process, one BLAS thread "
                                      f"(oracle port, float64; setup {time.perf_counter() - t0 - wall:.1f}s excluded)"}
        except Exception as ex:          # the baseline must never take the GPU number down with it
            cpu_baseline = {"value": None, "unit": "env-steps/s", "cores": 1, "kind": "port", "sample": f"failed: {ex!r}"}

    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, last_step, B)
    if rank == 0:
        line = {
            "metric": "closed-loop AO env-steps/sec (batched envs)", "value": value, "unit": "env-steps/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_max / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": args.workload, "description": desc, "envs_per_gpu": B, "total_envs": world * B,
                       "policy": "integrator gainCL=0.5, leak=0.99", "rng": "philox",
                       "reconstructor": "50-mode Zernike modal (the reference's default, OOPAOEnvRazor.py:256-337)",
                       "l2": "per-step working set (layer maps) %.0f MB per GPU exceeds the 126 MB L2" % (
                           env.atm._maps.numel() * 4 / 2 / 1e6),
                       "mean_strehl_last_step": sr_mean, "host_affinity": pinned},
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": "env-steps/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "host_policy": "action = gainCL * obs, in place on the pinned observation returned by the previous step"},
            "e2e_lookahead": {"value": e2e_ahead, "unit": "env-steps/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                              "note": "TorchWrapper(lookahead=True), opt-in; `e2e` is the strict wrapper"},
            "gpu_launches": launches,
            **({"e2e_sweep": e2e_sweep} if e2e_sweep else {}),
            "roofline": roofline,
            "step_roofline": step_roofline(env, B, ms_max / args.steps),
            "cpu_baseline": cpu_baseline,
            "kernels": kernels,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def dominant_roofline(kernels, env, B):
    """Algorithmic bytes / flops per launch (SURVEY.md section 8 d; DESIGN.md 'Kernels') of the kernel family with
    the largest share of the step, against the measured peaks."""
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = peaks.get("hbm_gbs", 6650.0)
    tc_peak = peaks.get("bf16_tflops_sustained", 1400.0)
    src = "measured (MEASURED_PEAKS.json)" if peaks else "fallback (B200_PROFILING.md)"
    R, L, M = env.tel.resolution, env.atm.nLayer, env.atm._M
    P, nA, nSig = R * R, env.dm.nValidAct, env.wfs.nSignal
    top = max(kernels, key=lambda k: kernels[k]["ms_per_step"])
    ms = kernels[top]["ms_per_call"]
    traffic = None
    try:     # DRAM bytes per launch from the committed ncu capture of this workload (profiles/)
        t = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic_cfg3.json")))
        if t.get("envs_per_gpu") == B and (R, L) == (240, 3):
            traffic = t.get(top)          # null until an ncu capture of this kernel is committed
    except Exception:
        pass
    if top.startswith("aoenv_gemm_tn"):
        N = int(top.split("N=")[1].split(",")[0])
        K = {P: nA, nA: nSig}.get(N, env.atm._nI + env.atm._nO)
        flops = 2.0 * B * N * K
        ach = flops / (ms * 1e-3) / 1e12
        if top.startswith("aoenv_gemm_tn_tc"):
            parts = 3 if N == env.atm._nO else 2
            n_mma = {2: 3, 3: 6}[parts]
            return {"kernel": top, "bound": "tensor", "achieved": ach * n_mma, "peak": tc_peak, "unit": "TFLOP/s",
                    "frac": ach * n_mma / tc_peak, "traffic": None, "fp32_equivalent_tflops": ach,
                    "peak_source": src + f", bf16 dense sustained; achieved counts the {n_mma} bf16 MMAs issued per FP32-grade "
                                         "product (algorithmic 2*M*N*K flops x " + str(n_mma) + ")"}
        return {"kernel": top, "bound": "tensor", "achieved": ach, "peak": tc_peak, "unit": "TFLOP/s", "frac": ach / tc_peak,
                "traffic": None, "peak_source": src + ", bf16 dense sustained; this kernel runs FP32 SIMT"}
    per_env_all = {
        "aoenv_dm_surface_separable": P * 4 + nA * 4,
        "aoenv_atm_phase": L * M * M * 4 + P * 4,
        "aoenv_shwfs_frame": 3 * P * 4,
        "aoenv_shwfs_frame_dm": 2 * P * 4 + (env.dm.nAct + 14) * R * 4,           # atmosphere OPD in, frame out, T = C gx rows in
        "aoenv_shwfs_fused": P * 4 + nSig * 4 + (env.dm.nAct + 14) * R * 4,      # OPD in, slopes out, T = C gx rows in
        "aoenv_dm_rows": nA * 4 + env.dm.nAct * R * 4,
        "aoenv_shwfs_slopes": P * 4 + nSig * 4,
        "aoenv_atm_ring": 2 * (4 * M - 4) * 4,
        "aoenv_atm_compact": 2 * M * M * 4,
        "aoenv_atm_gather": 2 * (env.atm._nI + env.atm._nO) * 4,
        "aoenv_command_update": 3 * nA * 4 + env.nActuator ** 2 * 4,
        "aoenv_observe": nA * 4 + env.nActuator ** 2 * 4,
    }
    if "aoenv_dm_rows" not in kernels:             # the frame kernel read a surface from memory (no factored DM this run)
        per_env_all["aoenv_shwfs_frame_dm"] = 3 * P * 4
    per_env = per_env_all.get(top, 0)
    ach = per_env * B / (ms * 1e-3) / 1e9
    out = {"kernel": top, "bound": "hbm", "achieved": ach, "peak": hbm_peak, "unit": "GB/s", "frac": ach / hbm_peak,
           "traffic": traffic, "peak_source": src}
    # algorithmic HBM GB/s of every streaming kernel of the step (same definition as `achieved`)
    out["all_streaming_kernels_gbs"] = {k: round(per_env_all[k] * B / (kernels[k]["ms_per_call"] * 1e-3) / 1e9, 1)
                                        for k in kernels if k in per_env_all}
    if top in ("aoenv_shwfs_frame", "aoenv_shwfs_frame_dm", "aoenv_shwfs_fused"):
        # This kernel is bound by the FP32 FMA pipe (ncu: profiles/), so the roofline is the FP32 one: algorithmic flops =
        # the two pruned DFT passes on the n non-zero inputs with the radix-2 split (4 n^3 + 8 n^3 FMA per lit lenslet,
        # DESIGN.md section 4) and, for the fused kernel, the banded DM surface (W FMA per pixel + the T = C gx stage).
        # Field generation, |.|^2, binning, statistics and centroids are not counted.  The HBM figures stay as
        # `hbm_model` (algorithmic bytes: OPD in, commands in, slopes out; the camera frame only when it is written).
        n = env.wfs.n_pix_subap if hasattr(env.wfs, "n_pix_subap") else R // env.wfs.nSubap
        fma = (4 * n ** 3 + 8 * n ** 3) * int(env.wfs.nValidSubaperture)
        what = "pruned DFT passes"
        if top in ("aoenv_shwfs_fused", "aoenv_shwfs_frame_dm"):
            tb = env.dm.fused_tables()
            if tb is not None:
                win = env.wfs._dm_windows(tb)
                fma += (win[0] if win else 14) * P               # row half of the separable surface (the column half is aoenv_dm_rows)
                what += " + banded DM surface (row half)"
        tflops = 2.0 * fma * B / (ms * 1e-3) / 1e12
        out = {"kernel": top, "bound": "fp32", "achieved": tflops, "peak": 72.3, "unit": "TFLOP/s", "frac": tflops / 72.3,
               "traffic": traffic, "flops_counted": what,
               "peak_source": "FP32 FMA peak measured on this pool's B200 (tools/microbench/ffma2_rate.cu: FFMA and FFMA2 both "
                              "72.3 TFLOP/s; nominal 148 SM x 128 x 2 x 1.965 GHz = 74.4); MEASURED_PEAKS.json holds no FP32 figure",
               "hbm_model": {"algorithmic_bytes_per_launch": per_env * B, "achieved_gbs": ach, "frac_of_hbm_peak": ach / hbm_peak,
                             "hbm_peak_gbs": hbm_peak, "peak_source": src},
               "all_streaming_kernels_gbs": out["all_streaming_kernels_gbs"]}
    return out


def step_roofline(env, B, ms_per_step):
    """Whole-step HBM figure on SURVEY.md section 8(d)'s compulsory bytes per env-step: every layer map read once, one map
    write-back per expected add_row, commands, slopes, observation, reward and Strehl."""
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak = peaks.get("hbm_gbs", 6650.0)
    R, L, M = env.tel.resolution, env.atm.nLayer, env.atm._M
    nA, nSig, nAct2 = env.dm.nValidAct, env.wfs.nSignal, env.nActuator ** 2
    f = sum(float(abs(ly.ratio).max()) for ly in env.atm._layers)
    per_env = L * M * M * 4 + f * M * M * 4 + 3 * nA * 4 + nSig * 4 + nAct2 * 4 + 8
    gbs = per_env * B / (ms_per_step * 1e-3) / 1e9
    return {"algorithmic_bytes_per_env_step": per_env, "add_row_events_per_step": f, "achieved_gbs": gbs, "peak_gbs": hbm_peak,
            "frac": gbs / hbm_peak, "peak_source": "measured (MEASURED_PEAKS.json)" if peaks else "fallback (B200_PROFILING.md)"}


def run_po4ao_arm(args):
    """SURVEY.md section 8(d) cfg 2: policy-driven rollouts (ConvPolicy, n_history = 20, random weights) of all
    environments in lock-step, telemetry histories and the replay buffer on the device."""
    import torch
    import torch.distributed as dist
    from rlao_b200 import _lib
    from rlao_b200.PO4AO import mbrl
    from rlao_b200.PO4AO.conv_models_simple import ConvPolicy, EnsembleDynamics
    from rlao_b200.PO4AO.util_simple import EfficientExperienceReplay, TorchWrapper
    from rlao_b200.OOPAOEnv.OOPAOEnvRazor import OOPAO

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    nS, nL, B, desc, opts = WORKLOADS[args.workload]
    if args.envs:
        B = args.envs
    n_history = 20
    base = OOPAO()
    base.set_params_file("rlao_b200.Conf.parameter_file_synthetic_SHWFS", "")
    base.set_params(make_args(nS, nL, opts), "shackhartmann", gainCL=0.5, n_envs=B, device=dev, rng="philox", seed=1,
                    env_offset=rank * B)
    env = TorchWrapper(base, host_io=False)
    nA = env.nActuator
    torch.manual_seed(5)
    policy = ConvPolicy(env.xvalid, env.yvalid, 0.0, env.F.float(), n_history).to(dev)
    dynamics = EnsembleDynamics(env.xvalid, env.yvalid, n_history).to(dev)
    replay = EfficientExperienceReplay((nA, nA), (nA, nA), max_size=(args.steps + args.warmup) * B, device=dev, n_envs=B)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def episode(n, it):
        return mbrl.run(env, None, None, None, replay, policy, dynamics, n_history, n, warmup_ts=0, sigma=0.0, episode=1,
                        iteration=it)

    episode(args.warmup, 1)
    replay.clear()
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
        time.sleep(0.25)
    base.atm.generateNewPhaseScreen(93234 * 2)
    base.dm.coefs = 0
    base.tel * base.dm * base.wfs
    l0 = _lib.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    t_wall0 = time.time()
    e0.record()
    sr, reward_sum, _, _, obs_last, rewards, _ = mbrl.run(env, None, None, None, replay, policy, dynamics, n_history, args.steps,
                                                          warmup_ts=0, sigma=0.0, episode=1, iteration=2, new_screen=False)
    e1.record()
    barrier()
    t_wall1 = time.time()
    ms = e0.elapsed_time(e1)
    launches = _lib.launch_count() - l0
    clocks = sampler.stop(t_wall0, t_wall1) if rank == 0 else None
    if rank == 0 and args.dump_outputs:          # before the breakdown below steps the environment again
        dump_outputs(args.dump_outputs, {"obs": obs_last, "reward": rewards[-1], "reward_sum": reward_sum}, B)
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max = float(t[0])

    # where the time goes: the policy forward alone, and the environment step alone
    obs = torch.randn((B, 1, nA, nA), device=dev)
    hist = torch.randn((B, 2 * (n_history - 1), nA, nA), device=dev)
    with torch.no_grad():
        for _ in range(3):
            policy(obs, hist)
        e0.record()
        for _ in range(10):
            policy(obs, hist)
        e1.record()
    torch.cuda.synchronize()
    ms_policy = e0.elapsed_time(e1) / 10
    act = torch.zeros((B, nA, nA), device=dev)
    e0.record()
    for i in range(10):
        base._step_views(None, act)
    e1.record()
    torch.cuda.synchronize()
    ms_env = e0.elapsed_time(e1) / 10
    if rank == 0:
        flops = 2 * 9 * nA * nA * ((2 * n_history - 1) * 64 + 64 * 64 + 64) * B
        line = {
            "metric": "closed-loop AO env-steps/sec (batched envs)", "value": world * B * args.steps / (ms_max * 1e-3),
            "unit": "env-steps/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_max / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": args.workload, "description": desc, "envs_per_gpu": B, "total_envs": world * B,
                       "policy": "PO4AO ConvPolicy n_history=20 (random weights, PyTorch/cuDNN, TF32 convolutions as PyTorch "
                                 "defaults), histories + replay on the device", "rng": "philox",
                       "mean_strehl": sr},
            "clocks": clocks, "e2e": None, "gpu_launches": launches,
            "breakdown_ms": {"policy_forward": ms_policy, "env_step": ms_env,
                             "policy_tflops": flops / (ms_policy * 1e-3) / 1e12},
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="cfg3", choices=list(WORKLOADS))
    ap.add_argument("--envs", type=int, default=0, help="environments per GPU (default: the workload's)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--wfs", default="shackhartmann", choices=["shackhartmann", "pyramid"],
                    help="pyramid: the papyrus-style environment (SURVEY.md section 8 f-3)")
    ap.add_argument("--policy", default="integrator", choices=["integrator", "po4ao"],
                    help="po4ao: ConvPolicy (n_history 20) rollouts through rlao_b200.PO4AO.mbrl.run with a GPU replay")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last of them returned (obs, reward, ...; rank 0's environments) "
                         "as DIR/<name>.npy, at most 64 MB in all; the inputs are seeded, so two builds can be compared")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the GPU path; --impl reference has none")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    if args.impl == "reference":
        run_reference_arm(args)
    elif args.policy == "po4ao":
        run_po4ao_arm(args)
    else:
        run_gpu_arm(args)


if __name__ == "__main__":
    main()
