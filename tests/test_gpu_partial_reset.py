"""Per-environment episode resets on the device (OOPAO.reset_envs -> Atmosphere.reset_envs: aoenv_vk_screens_envs,
aoenv_atm_gather_envs + GEMM + aoenv_atm_ring_envs, aoenv_atm_phase_envs) and the vector wrapper GymnasiumVectorSH.

Most cases run a cfg2-size system (20 x 20 lenslets) with three layers, so that the layers' add_rows group, at 64 or 256
environments; the wrapper runs at cfg3 / 1024.  Resets cover environments 0 and B - 1, a single environment and the whole
batch."""
import functools
import math

import numpy as np
import pytest
import torch

import bench
from parity_util import rel_err

pytestmark = pytest.mark.gpu

B_SMALL = 64
# (step before which reset_envs runs, environments, seed): 0 and B - 1, one environment, a mixed set
RESETS = ((3, (0, 17, B_SMALL - 1), 101), (8, (5,), 102), (14, (0, 5, 40), 103))
UNTOUCHED = sorted(set(range(B_SMALL)) - {e for _, ids, _ in RESETS for e in ids})
RESET = sorted({e for _, ids, _ in RESETS for e in ids})
STEPS = 20

# name -> (AOENV_STEP_NATIVE, AOENV_ATM_PREFETCH, AOENV_ATM_NATIVE, camera noise, geometric sensor)
MODES = {
    "native_prefetch": ("1", "force", "1", False, False),
    "native_inline": ("1", "0", "1", False, False),
    "calls_prefetch": ("0", "force", "1", False, False),
    "calls_inline": ("0", "0", "1", False, False),
    "python_atm": ("1", "0", "0", False, False),
    "noise": ("1", "force", "1", True, False),
    "geometric": ("1", "0", "1", False, True),
}


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    return torch.device("cuda:0")


def build(dev, B=B_SMALL, nS=20, nL=3, mode="native_prefetch", seed=1):
    """An environment built as bench.py builds its own, in one of MODES."""
    import os
    from rlao_b200.OOPAOEnv.OOPAOEnvRazor import OOPAO
    step_native, prefetch, atm_native, noise, geometric = MODES[mode]
    saved = {k: os.environ.get(k) for k in ("AOENV_STEP_NATIVE", "AOENV_ATM_PREFETCH", "AOENV_ATM_NATIVE")}
    os.environ.update(AOENV_STEP_NATIVE=step_native, AOENV_ATM_PREFETCH=prefetch, AOENV_ATM_NATIVE=atm_native)
    try:
        args = bench.make_args(nS, nL, {"noise": True} if noise else {})
        if geometric:
            args.is_geometric = True
        env = OOPAO()
        env.set_params_file("rlao_b200.Conf.parameter_file_synthetic_SHWFS", "")
        env.set_params(args, "shackhartmann", gainCL=0.5, n_envs=B, device=dev, rng="philox", seed=seed)
    finally:
        for k, v in saved.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v
    env.atm.generateNewPhaseScreen(17)
    env.dm.coefs = 0
    env.tel * env.dm * env.wfs
    return env, env.reset_soft()


def _cpu(t):
    return t.detach().cpu().clone()


@functools.lru_cache(maxsize=None)
def trajectory(mode, with_resets):
    """STEPS integrator steps (closed loop on the environment's own observation); per step the step's outputs, the
    slopes and the rms diagnostics, and at the end every layer's window and extrema."""
    dev = torch.device("cuda:0")
    env, obs = build(dev, mode=mode)
    out = {k: [] for k in ("obs", "reward", "strehl", "slopes", "total", "residual")}
    for i in range(STEPS):
        for at, ids, seed in (RESETS if with_resets else ()):
            if at == i:
                env.reset_envs(list(ids), seed)
        obs, reward, strehl, _, _ = env.step(i, env.gainCL * obs)
        for k, v in (("obs", obs), ("reward", reward), ("strehl", strehl), ("slopes", env.wfs._signal),
                     ("total", env._total_now), ("residual", env._residual_now)):
            out[k].append(_cpu(v))
    out = {k: torch.stack(v) for k, v in out.items()}
    out["maps"] = [_cpu(ly.mapShift) for ly in env.atm._layers]
    out["ext"] = _cpu(env.atm._ext)
    out["events"] = [ly.events for ly in env.atm._layers]
    out["native"] = env._native is not None
    del env
    torch.cuda.empty_cache()
    return out


@pytest.mark.parametrize("mode", list(MODES))
def test_untouched_environments_are_bit_identical(dev, mode):
    twin, got = trajectory(mode, False), trajectory(mode, True)
    assert got["native"] == (MODES[mode][0] == "1")
    u = torch.tensor(UNTOUCHED)
    for k in ("obs", "reward", "strehl", "slopes", "total", "residual"):
        assert torch.equal(got[k][:, u], twin[k][:, u]), k
        assert not torch.equal(got[k][4:, torch.tensor(RESET)], twin[k][4:, torch.tensor(RESET)]), k
    for i in range(len(got["maps"])):
        assert torch.equal(got["maps"][i][u], twin["maps"][i][u]), ("canvas", i)
        assert torch.equal(got["ext"][i][:, u], twin["ext"][i][:, u]), ("extrema", i)
    assert got["events"] == twin["events"]                     # the add_row counters did not move


@pytest.mark.parametrize("pair", [("native_prefetch", "native_inline"), ("native_inline", "calls_inline"),
                                  ("calls_prefetch", "calls_inline"), ("native_inline", "python_atm")])
def test_reset_environments_do_not_depend_on_the_path(dev, pair):
    a, b = trajectory(pair[0], True), trajectory(pair[1], True)
    for k in ("obs", "reward", "strehl", "slopes", "total", "residual"):
        assert torch.equal(a[k], b[k]), k
    if MODES[pair[0]][1] == MODES[pair[1]][1]:     # with prefetch the layers end one frame ahead of the last step
        for i in range(len(a["maps"])):
            assert torch.equal(a["maps"][i], b["maps"][i]), ("canvas", i)


def _unpack(packed):
    """Value of a packed extremum (csrc/atm.cu: monotone key << 32 | position)."""
    key = ((packed >> 32) & 0xFFFFFFFF) ^ 0x80000000
    key = torch.where(key >= 2 ** 31, key - 2 ** 32, key).to(torch.int32)
    bits = torch.where(key >= 0, key, key ^ 0x7FFFFFFF)
    return bits.view(torch.float32)


SUBSETS = [(0, B_SMALL - 1), (23,), tuple(range(B_SMALL))]


@pytest.mark.parametrize("ids", SUBSETS, ids=["ends", "one", "all"])
def test_new_screens_ring_extrema_and_phase(dev, ids):
    from rlao_b200 import _lib
    env, _ = build(dev, mode="native_inline")
    twin, _ = build(dev, mode="native_inline")
    atm, seed = env.atm, 555
    env.step(0, torch.zeros((B_SMALL, env.nActuator, env.nActuator), device=dev))
    before = [ly.mapShift.clone() for ly in atm._layers]
    atm.reset_envs(list(ids), seed)
    torch.cuda.synchronize()
    assert atm._prefetched
    idx = torch.tensor(ids, device=dev)
    k, L, M, nI, nO, K = len(ids), atm.nLayer, atm._M, atm._nI, atm._nO, atm._K
    # screens: environment e's interior equals its interior after generateNewPhaseScreen(seed).  Both are the same Philox
    # draws through two split-bf16 (3 parts, ~2^-24) DFT-matrix products; the batch composition only changes the GEMM's
    # K split, so they agree to float32 rounding of the synthesis: |diff| <= 1e-5 max |screen|.
    twin.atm.generateNewPhaseScreen(seed)
    for i in range(L):
        got = atm._layers[i].mapShift[idx, 1:-1, 1:-1].double()
        want = twin.atm._layers[i].mapShift[idx, 1:-1, 1:-1].double()
        assert rel_err(got.cpu().numpy(), want.cpu().numpy()) < 1e-5, ("screen", i)
    # ring: the environment's own row of X = [A | B] zx in float64 from the device's zx (one group of all three layers)
    assert atm._group_max >= L
    from rlao_b200 import gemm
    parts = atm._W_op.parts
    if gemm.uses_tensor_cores(L * k):          # the tensor-core product reads the split-bf16 planes the gather wrote
        zx = atm._zx_planes.reshape(-1)[:parts * L * k * K].reshape(parts, L * k, K).double().sum(0)
    else:                                      # a few rows: the exact-FP32 kernel on the float32 copy
        zx = atm._zx[:L * k].double()
    W = atm._W.double()
    want_x, mag = zx @ W.T, zx.abs() @ W.abs().T
    outer = torch.ones((M, M), dtype=torch.bool, device=dev)
    outer[1:-1, 1:-1] = False
    inner_rc = atm._inner_rc.long()
    for i in range(L):
        win = atm._layers[i].mapShift[idx]
        rows = slice(i * k, (i + 1) * k)
        ring = win[:, outer].double()
        assert float(((ring - want_x[rows, :nO]).abs() / mag[rows, :nO]).max()) < 2.0 ** -16, ("ring", i)
        z = win[:, inner_rc[:, 0], inner_rc[:, 1]].double()
        assert float(((zx[rows, :nI] - z).abs() / z.abs().clamp_min(1e-30)).max()) < 2.0 ** -16, ("Z", i)
        # extrema blocks: window, interior, current origin
        ext = atm._ext[i][:, idx]
        assert torch.equal(_unpack(ext[0, :, 0]), win.reshape(k, -1).min(1).values)
        assert torch.equal(_unpack(ext[0, :, 1]), win.reshape(k, -1).max(1).values)
        assert torch.equal(_unpack(ext[1, :, 0]), win[:, 1:-1, 1:-1].reshape(k, -1).min(1).values)
        assert torch.equal(_unpack(ext[1, :, 1]), win[:, 1:-1, 1:-1].reshape(k, -1).max(1).values)
        oy, ox = atm._org[i]
        assert (ext[2, :, 0] == ((1 << 32) | (oy * atm._pitch + ox))).all()
        # xi is not the layer's next per-frame draw (that stream is keyed by the add_row counter, which did not move)
        ly = atm._layers[i]
        scratch = torch.zeros((B_SMALL, K), dtype=torch.float32, device=dev)
        _lib.check(_lib.load().aoenv_atm_gather(atm._win_ptr(i), B_SMALL, M, atm._pitch, atm._env_stride, 0, 0,
                                                _lib.ptr(atm._inner_rc), nI, nO, None, ly.philox_seed,
                                                ((ly.events << 8) | i) + (atm.env_offset << 40), _lib.ptr(scratch), K, None,
                                                parts, _lib.stream_ptr(dev)), "atm_gather")
        xi_next = scratch[idx, nI:nI + nO].double()
        assert float((zx[rows, nI:nI + nO] - xi_next).abs().min()) > 0, ("xi", i)
    # phase: the reset environments' rows of the next frame = a whole-batch recompute on the patched canvases, bit for bit
    full = torch.empty_like(atm._opd_next)
    atm._publish(full)
    torch.cuda.synchronize()
    assert torch.equal(full, atm._opd_next)
    # the untouched environments' windows did not change
    others = torch.tensor(sorted(set(range(B_SMALL)) - set(ids)), dtype=torch.long, device=dev)
    if others.numel():
        for i in range(L):
            assert not torch.equal(atm._layers[i].mapShift[idx], before[i][idx])
            assert torch.equal(atm._layers[i].mapShift[others], before[i][others])


def test_events_do_not_move_and_flat_mirror_at_the_first_step(dev):
    env, obs = build(dev, mode="native_prefetch")
    twin, obs_t = build(dev, mode="native_prefetch")
    ids = [0, 9, B_SMALL - 1]
    for i in range(4):
        obs = env.step(i, env.gainCL * obs)[0]
        obs_t = twin.step(i, twin.gainCL * obs_t)[0]
    env.reset_envs(np.array([i in ids for i in range(B_SMALL)]), 7)
    act = torch.randn((B_SMALL, env.nActuator, env.nActuator), device=dev, generator=torch.Generator(dev).manual_seed(3))
    env.step(4, act)
    twin.step(4, act)
    torch.cuda.synchronize()
    assert [ly.events for ly in env.atm._layers] == [ly.events for ly in twin.atm._layers]
    t = torch.tensor(ids, device=dev)
    assert torch.equal(env._residual_now[t], env._total_now[t])          # flat mirror: the sensor sees the atmosphere alone
    assert not torch.equal(twin._residual_now[t], twin._total_now[t])
    nA = env.dm.nValidAct
    want = env._action_tensor(act)[:, env._act_idx.long()] * np.float32(1e-6)
    assert torch.equal(env.dm._coefs[t, :nA], want[t])                   # the command is this step's action alone
    assert torch.equal(env._dm_prev[t, :nA], want[t])


def test_reset_screen_statistics(dev):
    """Structure function of the reset screens against the reference algorithm with its own MT19937 streams (the check of
    test_gpu_reset.py); pre- and post-reset screens of one environment are uncorrelated; two seeds differ."""
    from rlao_b200.tools import vonkarman as vk
    B = 256
    env, _ = build(dev, B=B, mode="native_inline")
    atm = env.atm
    pre = [ly.mapShift[:, 1:-1, 1:-1].double().clone() for ly in atm._layers]
    atm.reset_envs(np.ones(B, dtype=bool), 4242)
    post = torch.cat([ly.mapShift[:, 1:-1, 1:-1].double() for ly in atm._layers])        # 768 screens
    N, delta = atm._ops.layer_res, atm._ops.layer_D / atm._ops.layer_res
    ref = np.stack([vk.screen_reference_rng(atm.r0, atm.L0, N, delta, 1000 + k) for k in range(192)])
    for sep in (1, 4, 16):
        dx = float(((post[:, :, sep:] - post[:, :, :-sep]) ** 2).mean())
        dy = float(((post[:, sep:, :] - post[:, :-sep, :]) ** 2).mean())
        wx = ((ref[:, :, sep:] - ref[:, :, :-sep]) ** 2).mean()
        wy = ((ref[:, sep:, :] - ref[:, :-sep, :]) ** 2).mean()
        tol = 0.08 if sep <= 4 else 0.15
        assert abs(dx / wx - 1) < tol and abs(dy / wy - 1) < tol, (sep, dx / wx, dy / wy)
    d = lambda a: (a[:, :, 1:] - a[:, :, :-1]).reshape(a.shape[0], -1)
    a, b = d(pre[0][:64]), d(post[:64])
    c = ((a - a.mean(1, keepdim=True)) * (b - b.mean(1, keepdim=True))).sum(1) / (a.std(1) * b.std(1) * (a.shape[1] - 1))
    assert float(c.abs().max()) < 0.3 and float(c.abs().mean()) < 0.06, c
    atm.reset_envs([3], 4243)
    assert not torch.equal(atm._layers[0].mapShift[3, 1:-1, 1:-1].double(), post[3])


def test_checkpoint_right_after_reset_resumes_bit_identically(dev):
    env, obs = build(dev, mode="native_prefetch")
    for i in range(3):
        obs = env.step(i, env.gainCL * obs)[0]
    env.reset_envs([0, 31, B_SMALL - 1], 9)
    st = env.state_dict()
    assert st["atm_opd_next"] is not None
    other, _ = build(dev, mode="native_prefetch", seed=5)
    other.load_state_dict(st)
    o1 = o2 = obs
    for i in range(3, 8):
        o1, r1, s1, _, _ = env.step(i, env.gainCL * o1)
        o2, r2, s2, _, _ = other.step(i, other.gainCL * o2)
        assert torch.equal(o1, o2) and torch.equal(r1, r2) and torch.equal(s1, s2), i


def test_vector_wrapper_ignores_the_actions_of_resetting_environments_at_cfg3_size(dev):
    """GymnasiumVectorSH at 1024 environments, episode_length 50, staggered: garbage actions on the rows that reset at a
    call give the same run, bit for bit, as zero actions there."""
    from rlao_b200.OOPAOEnv.gymnasium_api import GymnasiumVectorSH
    B, L = 1024, 50
    runs = []
    for garbage in (True, False):
        env, _ = build(dev, B=B, nS=40, nL=3, mode="native_prefetch")
        vec = GymnasiumVectorSH(env, n_history=2, delay=1, episode_length=L, stagger_episodes=True)
        obs, _ = vec.reset(seed=77)
        gen = torch.Generator(dev).manual_seed(1)
        rec, n_reset = [], 0
        for t in range(60):
            act = env.gainCL * obs[:, 0]
            rows = torch.as_tensor(vec._pending, device=dev)
            n_reset += int(vec._pending.sum())
            junk = torch.randn(act.shape, device=dev, generator=gen) * 1e3
            act = torch.where(rows[:, None, None], junk if garbage else torch.zeros_like(act), act)
            obs, reward, terminated, truncated, info = vec.step(act)
            assert not terminated.any() and int(truncated.sum()) <= math.ceil(B / L)
            rec.append((_cpu(obs), _cpu(reward), truncated.copy()))
        assert n_reset >= B                                    # every environment reset at least once
        runs.append(rec)
        del vec, env
        torch.cuda.empty_cache()
    for (o1, r1, t1), (o2, r2, t2) in zip(*runs):
        assert torch.equal(o1, o2) and torch.equal(r1, r2) and np.array_equal(t1, t2)
