"""Geometric Shack-Hartmann sensor on the GPU (aoenv_shwfs_geometric / _f64, the geometric part of aoenv_sh_step) against
the geometric oracle (oracle/ao_oracle.py, DESIGN.md section 2) and against the diffractive path's pupil statistics."""
import ctypes
import math

import numpy as np
import pytest
import torch

from oracle.ao_oracle import AOConfig, flux_map, source_properties, telescope_pupil
from oracle.golden_configs import CONFIGS, EPISODE_SEED, STEPS
from parity_util import new_episode, rel_err
from geometric_oracle import GeometricEnvOracle, GeometricShackHartmannOracle
from test_geometric_cpu import build_geometric_env

pytestmark = pytest.mark.gpu

SLOPE_TOL = 1e-4
STATS_TOL = 1e-9


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    return torch.device("cuda:0")


def _np(t):
    return t.detach().double().cpu().numpy()


def _opds(R, count, seed, scale=0.4e-6):
    rs = np.random.RandomState(seed)
    yy, xx = np.mgrid[:R, :R] / R
    out = []
    for _ in range(count):
        c = rs.normal(size=5)
        out.append(scale * (c[0] * xx + c[1] * yy + c[2] * np.sin(7 * xx + 3 * yy) + c[3] * np.cos(11 * yy) * xx
                            + 0.3 * c[4] * np.sin(23 * xx * yy)) + 0.05 * scale * rs.normal(size=(R, R)))
    return np.stack(out)


def _frame_stats(wfs, opd_a, opd_b=None, dm=None):
    """Pupil statistics of the diffractive frame kernel on the same input."""
    from rlao_b200 import _lib
    B, R = opd_a.shape[0], opd_a.shape[1]
    frame = torch.empty((B, R, R), dtype=torch.float32, device=opd_a.device)
    envmax = torch.zeros((B,), dtype=torch.int32, device=opd_a.device)
    stats = torch.zeros((B, 4), dtype=torch.float64, device=opd_a.device)
    _lib.check(_lib.load().aoenv_shwfs_frame_dm(
        _lib.ptr(opd_a), _lib.ptr(opd_b), ctypes.byref(dm) if dm is not None else None, None, _lib.ptr(wfs.telescope._pupil_f),
        _lib.ptr(wfs._amp), _lib.ptr(wfs._valid_u8), B, wfs.nSubap, wfs.n_pix_subap,
        ctypes.c_float(2 * math.pi / wfs.telescope.src.wavelength), None, 0, _lib.ptr(frame), _lib.ptr(envmax), _lib.ptr(stats),
        _lib.stream_ptr(opd_a.device)), "shwfs_frame_dm")
    return _np(stats)


@pytest.mark.parametrize("nS", [8, 20, 40])
@pytest.mark.parametrize("n", [4, 6, 8])
def test_geometric_kernels_vs_oracle(dev, nS, n):
    from rlao_b200.ShackHartmann import ShackHartmann
    from rlao_b200.Source import Source
    from rlao_b200.Telescope import Telescope
    cfg = AOConfig(nSubap=nS, nPixPerSubap=n)
    R, B = cfg.resolution, 3
    tel = Telescope(R, cfg.diameter, cfg.samplingTime, n_envs=B, device=dev)
    Source(cfg.opticalBand, cfg.magnitude) * tel
    wfs = ShackHartmann(nS, tel, cfg.lightRatio, is_geometric=True)
    assert wfs.is_geometric and wfs.cam.frame is None
    pupil = telescope_pupil(R)
    wl, nph = source_properties(cfg.opticalBand, cfg.magnitude)
    orc = GeometricShackHartmannOracle(cfg, pupil, flux_map(pupil, nph, cfg.samplingTime, cfg.diameter), wl)
    assert np.array_equal(wfs.valid_subapertures, orc.valid)
    assert np.all(wfs.reference_slopes_maps == 0)
    assert rel_err(wfs.slopes_units, orc.slopes_units) < 2e-6
    wfs.slopes_units = orc.slopes_units                  # identical inputs for the comparisons below
    a32 = _opds(R, B, 5).astype(np.float32)
    b32 = _opds(R, B, 6, scale=0.1e-6).astype(np.float32)
    a, b = torch.as_tensor(a32, device=dev), torch.as_tensor(b32, device=dev)
    # tel * wfs: one OPD term
    tel.OPD_no_pupil = a
    tel * wfs
    got = _np(wfs.signal)
    for e in range(B):
        assert rel_err(got[e], orc.measure(a32[e].astype(np.float64) * 2 * np.pi / wl)) < SLOPE_TOL, (e, "slopes")
    assert rel_err(_np(wfs.signal_2D)[2], orc.signal_2D) < SLOPE_TOL
    # two OPD terms + statistics, against the oracle and the frame kernel's statistics
    slopes = torch.zeros_like(wfs._signal)
    stats = torch.zeros((B, 4), dtype=torch.float64, device=dev)
    wfs._run_geometric(a, b, slopes, 1.0 / wfs.slopes_units, None, stats)
    tot = (a + b).cpu().numpy().astype(np.float64)
    got = _np(slopes)[:, :wfs.nSignal]
    for e in range(B):
        assert rel_err(got[e], orc.measure(tot[e] * 2 * np.pi / wl)) < SLOPE_TOL, (e, "slopes, two terms")
    assert rel_err(_np(stats), _frame_stats(wfs, a, b)) < STATS_TOL
    # calibration-grade twin (multi-frame branch)
    frames = wfs.measure_frames(a) * wfs.slopes_units
    want = orc.measure_multi(a32.astype(np.float64) * 2 * np.pi / wl).T * orc.slopes_units
    assert rel_err(_np(frames), want) < 1e-9


def test_inline_dm_vs_materialised_surface(dev):
    """The separable DM evaluated while staging (factored form) against the surface read from memory: float32 rounding;
    pupil statistics identical to the frame kernel's on the same factored input."""
    from rlao_b200.DeformableMirror import DMSurfaceRef
    cfg = CONFIGS["cfg1"]()
    env = build_geometric_env(cfg, n_envs=4, rng="philox", seed=2, device=dev)
    wfs, dm = env.wfs, env.dm
    assert dm.lazy_surface
    rs = np.random.RandomState(1)
    dm.coefs = torch.as_tensor(rs.normal(size=(4, dm.nValidAct)) * 3e-8, dtype=torch.float32, device=dev)
    ref = dm.surface_ref()
    assert isinstance(ref, DMSurfaceRef)
    opd_a = env.atm._opd
    b_t, dm_struct = wfs._second_term(ref)
    assert b_t is None and dm_struct is not None
    s_inline = torch.zeros_like(wfs._signal)
    st_inline = torch.zeros((4, 4), dtype=torch.float64, device=dev)
    wfs._run_geometric(opd_a, ref, s_inline, 1.0 / wfs.slopes_units, None, st_inline)
    surface = ref.tensor()
    s_mat = torch.zeros_like(wfs._signal)
    wfs._run_geometric(opd_a, surface, s_mat, 1.0 / wfs.slopes_units)
    assert rel_err(_np(s_inline), _np(s_mat)) < 2e-5
    assert rel_err(_np(st_inline), _frame_stats(wfs, opd_a, dm=dm_struct)) < STATS_TOL


@pytest.mark.parametrize("name", ["cfg1", "cfg3"])
def test_closed_loop_trace_vs_geometric_oracle(dev, name):
    """20 x 20 and 40 x 40 lenslets, rng='reference': the environment and the geometric oracle environment in lock-step,
    every step driven with the oracle's own action (identical inputs).  No threshold, so no knife-edge exclusion."""
    cfg = CONFIGS[name]()
    env = build_geometric_env(cfg, n_envs=1, rng="reference", device=dev)
    orc = GeometricEnvOracle(cfg)
    assert np.array_equal(env.wfs.valid_subapertures, orc.wfs.valid)
    assert rel_err(env.wfs.slopes_units, orc.wfs.slopes_units) < 2e-6
    assert rel_err(_np(env.calib_zonal.D), orc.D_zonal) < 1e-6
    env.set_reconstructor(orc.reconstructor)
    env.wfs.slopes_units = float(orc.wfs.slopes_units)
    obs = new_episode(env, EPISODE_SEED)
    obs_o = orc.new_episode(EPISODE_SEED)
    assert rel_err(_np(env.wfs.signal), orc.wfs.signal) < 2e-4
    for i in range(STEPS[name]):
        action = cfg.gainCL * obs_o
        obs, reward, strehl, done, info = env.step(i, torch.as_tensor(action, dtype=torch.float32, device=dev))
        obs_o, reward_o, strehl_o, _, _ = orc.step(i, action)
        assert rel_err(_np(env.wfs.signal), orc.wfs.signal) < 2e-4, (i, "slopes")
        assert abs(float(strehl) - strehl_o) <= 1e-3 * strehl_o + 1e-30, (i, "strehl")    # (float32 underflow)
        assert rel_err(_np(obs), obs_o) < 1e-3, (i, "obs")
    assert env._native is not None                       # the default path: aoenv_atm_update + aoenv_sh_step


def test_native_step_is_bit_identical_to_call_by_call(dev):
    """aoenv_sh_step (geometric part) against the entry points called one by one, with the next frame's atmosphere on the
    side stream or in line; 32 environments so that the reconstruction runs on the tensor cores from the bf16 planes."""
    cfg = CONFIGS["tiny"]()
    cfg.windSpeed, cfg.windDirection = [40.0, 75.0], [20.0, 250.0]

    def run(one_call, prefetch, steps=10):
        env = build_geometric_env(cfg, n_envs=32, rng="philox", seed=4, device=dev, canvas_slack=4)
        env.atm.pipelined = "force" if prefetch else False
        env.native_step = one_call
        obs = new_episode(env, 9)
        out = [obs.cpu().clone()]
        for i in range(steps):
            obs, reward, strehl, _, _ = env.step(i, 0.4 * obs)
            out += [obs.cpu().clone(), reward.cpu().clone(), strehl.cpu().clone(), env.wfs.signal.cpu().clone()]
        torch.cuda.synchronize()
        assert (env._native is not None) == one_call and env.atm._prefetched == prefetch
        return out

    base = run(False, False)
    for kw in (dict(one_call=True, prefetch=False), dict(one_call=True, prefetch=True), dict(one_call=False, prefetch=True)):
        got = run(**kw)
        assert all(torch.equal(x, y) for x, y in zip(base, got)), kw
