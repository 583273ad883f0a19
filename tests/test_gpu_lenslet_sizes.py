"""Lenslets of 10 and 12 pixels on the GPU: the spots kernel (materialised surface and DM in place), the slopes, the camera,
the float64 calibration and the geometric sensor against the float64 oracles; the closed loop at 20 x 20 lenslets against
the oracle environment; the two-call step against the call-by-call one, also at 1024 environments."""
import math

import numpy as np
import pytest
import torch

from oracle.ao_oracle import AOConfig, EnvOracle, ShackHartmannOracle, flux_map, source_properties, telescope_pupil
from oracle.golden_configs import CONFIGS, EPISODE_SEED
from parity_util import build_env, knife_edge_lenslets, new_episode, rel_err
from geometric_oracle import GeometricEnvOracle, GeometricShackHartmannOracle
from test_geometric_cpu import build_geometric_env
from rlao_b200 import _lib

pytestmark = pytest.mark.gpu

WIDE = (10, 12)
FRAME_TOL = 2e-4
SLOPE_TOL = 1e-4


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


def _sensor(dev, nS, n, B, geometric=False, magnitude=None):
    from rlao_b200.ShackHartmann import ShackHartmann
    from rlao_b200.Source import Source
    from rlao_b200.Telescope import Telescope
    cfg = AOConfig(nSubap=nS, nPixPerSubap=n)
    if magnitude is not None:
        cfg.magnitude = magnitude
    R = cfg.resolution
    tel = Telescope(R, cfg.diameter, cfg.samplingTime, n_envs=B, device=dev)
    Source(cfg.opticalBand, cfg.magnitude) * tel
    wfs = ShackHartmann(nS, tel, cfg.lightRatio, is_geometric=geometric)
    pupil = telescope_pupil(R)
    wl, nph = source_properties(cfg.opticalBand, cfg.magnitude)
    orc = (GeometricShackHartmannOracle if geometric else ShackHartmannOracle)(
        cfg, pupil, flux_map(pupil, nph, cfg.samplingTime, cfg.diameter), wl)
    return cfg, tel, wfs, orc, pupil, wl


def _slopes_vs_oracle(got, want, orc, what):
    """Slopes to SLOPE_TOL of the array's maximum, lenslets with a pixel at the centroiding threshold excluded."""
    maps = orc.maps_intensity
    edge = knife_edge_lenslets(maps, orc.threshold_cog * maps.max())
    keep = np.concatenate([~edge, ~edge])
    assert edge.sum() <= max(2, 0.02 * orc.nValid), (what, "knife-edge lenslets", int(edge.sum()))
    assert np.abs(got - want)[keep].max() < SLOPE_TOL * np.abs(want).max(), what


@pytest.mark.parametrize("nS", [8, 20])
@pytest.mark.parametrize("n", WIDE)
def test_frame_slopes_and_calibration_vs_oracle(dev, nS, n):
    cfg, tel, wfs, orc, pupil, wl = _sensor(dev, nS, n, 3)
    assert wfs.n_pix_subap == n and np.array_equal(wfs.valid_subapertures, orc.valid)
    # float64 calibration: reference slopes and slope units
    assert rel_err(wfs.reference_slopes_maps, orc.reference_slopes_maps) < 1e-6
    assert rel_err(wfs.slopes_units, orc.slopes_units) < 1e-6
    wfs.slopes_units = orc.slopes_units                  # identical inputs for the comparisons below
    R = cfg.resolution
    tel.OPD_no_pupil = torch.as_tensor(_opds(R, 3, 5), dtype=torch.float32, device=dev)
    tel * wfs
    got_sig, got_frame, envmax = _np(wfs.signal), _np(wfs.cam.frame), wfs._envmax.cpu().numpy()
    opd32 = _np(tel.OPD_no_pupil)
    for e in range(3):
        want = orc.measure(opd32[e] * pupil * 2 * np.pi / wl)
        assert rel_err(got_frame[e], orc.frame) < FRAME_TOL, (e, "frame")
        _slopes_vs_oracle(got_sig[e], want, orc, (e, "slopes"))
        # the per-environment maximum the threshold uses: over the pixels of the lit lenslets
        lit = np.kron(wfs.valid_subapertures, np.ones((n, n), dtype=bool))
        i = int(envmax[e])
        assert np.float32(got_frame[e][lit].max()) == np.int32(i if i >= 0 else i ^ 0x7fffffff).view(np.float32)
    # calibration-grade multi-frame measurement (interaction-matrix pushes: one threshold for the batch)
    frames = wfs.measure_frames(tel.OPD_no_pupil)
    want = orc.measure_multi(opd32 * 2 * np.pi / wl)
    assert rel_err(_np(frames), want.T) < 1e-6
    # the alternative frame implementations stay at 4, 6, 8 pixels and say so
    lib = _lib.load()
    prev = lib.aoenv_set_wfs6_variant(3)
    try:
        with pytest.raises(RuntimeError, match="alternative frame variant"):
            tel * wfs
    finally:
        lib.aoenv_set_wfs6_variant(prev)


@pytest.mark.parametrize("n", WIDE)
def test_inline_dm_frame_vs_materialised_surface(dev, n):
    """aoenv_shwfs_frame_dm with the separable DM evaluated in place (lit-first order) against the frame of the surface read
    from memory: float32 rounding of the surface; the pupil statistics agree as well."""
    from rlao_b200.DeformableMirror import DMSurfaceRef
    cfg = CONFIGS["cfg1"]()
    cfg.nPixPerSubap = n
    B = 4
    env = build_env(cfg, n_envs=B, rng="philox", seed=2, device=dev)
    wfs, dm = env.wfs, env.dm
    assert dm.lazy_surface
    rs = np.random.RandomState(1)
    dm.coefs = torch.as_tensor(rs.normal(size=(B, dm.nValidAct)) * 3e-8, dtype=torch.float32, device=dev)
    ref = dm.surface_ref()
    assert isinstance(ref, DMSurfaceRef)
    b_t, dm_struct = wfs._second_term(ref)
    assert b_t is None and dm_struct is not None and dm_struct.WL == 14
    opd_a, R = env.atm._opd, env.tel.resolution
    scale = 2 * math.pi / env.source.wavelength

    def run(second):
        frame = torch.empty((B, R, R), dtype=torch.float32, device=dev)
        envmax = torch.zeros((B,), dtype=torch.int32, device=dev)
        stats = torch.zeros((B, 4), dtype=torch.float64, device=dev)
        slopes = torch.zeros_like(wfs._signal)
        wfs._run(opd_a, second, env.tel._pupil_f, scale, False, None, frame, envmax, stats, slopes, wfs._ref_xy,
                 1.0 / wfs.slopes_units)
        return _np(frame), _np(stats), _np(slopes)
    f_in, st_in, s_in = run(ref)
    f_mat, st_mat, s_mat = run(ref.tensor())
    assert rel_err(f_in, f_mat) < 2e-5
    assert rel_err(st_in[:, :2], st_mat[:, :2]) < 1e-9                 # the atmosphere's sums do not involve the DM
    # (the total is centred on a different pixel value in place: compare variances)
    P = float(env.tel.pixelArea)
    var = lambda st: st[:, 3] / P - (st[:, 2] / P) ** 2
    assert rel_err(var(st_in), var(st_mat)) < 1e-4
    assert rel_err(s_in, s_mat) < 1e-3


@pytest.mark.parametrize("n", WIDE)
def test_camera_noise_statistics(dev, n):
    """The camera pass at the new sizes: photon noise (index of dispersion 1), rounded Gaussian read noise, independent
    streams across environments; the per-environment maximum is taken after the camera, over the lit lenslets."""
    B = 256
    cfg, tel, wfs, orc, pupil, wl = _sensor(dev, 8, n, B, magnitude=10)
    tel.resetOPD()
    tel * wfs
    ideal = _np(wfs.cam.frame[0])
    lit = ideal > 0.02 * ideal.max()
    lit_lenslets = np.kron(wfs.valid_subapertures, np.ones((n, n), dtype=bool))
    wfs.cam.photonNoise = True
    tel * wfs
    f1 = _np(wfs.cam.frame)
    assert np.all(f1 == np.round(f1)) and f1.min() >= 0
    mean, var = f1.mean(axis=0), f1.var(axis=0)
    assert abs(mean[lit].mean() / ideal[lit].mean() - 1) < 0.01
    assert abs((var[lit] / mean[lit]).mean() - 1) < 0.05
    assert abs(np.corrcoef((f1[0] - ideal)[lit], (f1[1] - ideal)[lit])[0, 1]) < 0.1
    em = wfs._envmax.cpu().numpy()
    em = np.where(em >= 0, em, em ^ 0x7fffffff).astype(np.int32).view(np.float32)
    assert np.array_equal(em, f1[:, lit_lenslets].max(axis=1).astype(np.float32))
    wfs.cam.photonNoise = False
    wfs.cam.readoutNoise = 14
    tel * wfs
    r = _np(wfs.cam.frame) - ideal
    assert abs(r[:, ~lit].std() - 14) < 0.3 and abs(r[:, ~lit].mean()) < 0.2
    assert np.abs(r[:, ~lit] - np.round(r[:, ~lit])).max() < 1e-3


@pytest.mark.parametrize("nS", [8, 20])
@pytest.mark.parametrize("n", WIDE)
def test_geometric_slopes_vs_oracle(dev, nS, n):
    cfg, tel, wfs, orc, pupil, wl = _sensor(dev, nS, n, 3, geometric=True)
    assert np.array_equal(wfs.valid_subapertures, orc.valid)
    assert rel_err(wfs.slopes_units, orc.slopes_units) < 1e-6
    wfs.slopes_units = orc.slopes_units
    a32 = _opds(cfg.resolution, 3, 5).astype(np.float32)
    tel.OPD_no_pupil = torch.as_tensor(a32, device=dev)
    tel * wfs
    got = _np(wfs.signal)
    for e in range(3):
        assert rel_err(got[e], orc.measure(a32[e].astype(np.float64) * 2 * np.pi / wl)) < SLOPE_TOL, e
    frames = wfs.measure_frames(tel.OPD_no_pupil) * wfs.slopes_units
    want = orc.measure_multi(a32.astype(np.float64) * 2 * np.pi / wl).T * orc.slopes_units
    assert rel_err(_np(frames), want) < 1e-9


@pytest.mark.parametrize("n", WIDE)
def test_closed_loop_trace_vs_oracle(dev, n):
    """20 x 20 lenslets of n pixels (R = 20 n), rng='reference': the environment and the oracle environment in lock-step,
    every step driven with the oracle's action; the parity tests' tolerances and knife-edge rule."""
    cfg = CONFIGS["cfg1"]()
    cfg.nPixPerSubap = n
    env = build_env(cfg, n_envs=1, rng="reference", device=dev)
    orc = EnvOracle(cfg)
    nV = env.wfs.nValidSubaperture
    assert env.tel.resolution == 20 * n and np.array_equal(env.wfs.valid_subapertures, orc.wfs.valid)
    assert rel_err(env.wfs.slopes_units, orc.wfs.slopes_units) < 1e-6
    assert rel_err(env.wfs.reference_slopes_maps, orc.wfs.reference_slopes_maps) < 1e-6
    # (the pushes are float32 DM surfaces here, float64 in the oracle: the tolerance of the existing interaction-matrix test)
    assert rel_err(_np(env.calib_zonal.D), orc.D_zonal) < 1e-5
    assert rel_err(_np(env.reconstructor), orc.reconstructor) < 2e-4
    env.set_reconstructor(orc.reconstructor)
    env.wfs.slopes_units = float(orc.wfs.slopes_units)
    obs = new_episode(env, EPISODE_SEED)
    obs_o = orc.new_episode(EPISODE_SEED)
    assert rel_err(_np(obs), obs_o) < 2e-4
    for i in range(12):
        action = cfg.gainCL * obs_o
        obs, reward, strehl, done, info = env.step(i, torch.as_tensor(action, dtype=torch.float32, device=dev))
        obs_o, reward_o, strehl_o, _, _ = orc.step(i, action)
        assert rel_err(_np(env.wfs.cam.frame), orc.wfs.frame) < FRAME_TOL, (i, "frame")
        assert abs(float(strehl) - strehl_o) <= 1e-3 * strehl_o + 1e-30, (i, "strehl")
        maps = orc.wfs.maps_intensity
        edge = knife_edge_lenslets(maps, orc.wfs.threshold_cog * maps.max())
        keep = np.concatenate([~edge, ~edge])
        assert edge.sum() <= max(2, 0.02 * nV), (i, "knife-edge lenslets", int(edge.sum()))
        sig = _np(env.wfs.signal)
        assert np.abs(sig - orc.wfs.signal)[keep].max() < 2 * SLOPE_TOL * np.abs(orc.wfs.signal).max(), (i, "slopes")
        assert rel_err(_np(obs), obs_o) < (1e-3 if not edge.any() else 1e-2), (i, "obs")
    assert env._native is not None                       # the default path: aoenv_atm_update + aoenv_sh_step


def _run_steps(build, one_call, steps, noise=False):
    env = build()
    env.native_step = one_call
    if noise:
        env.wfs.cam.photonNoise, env.wfs.cam.readoutNoise = True, 3.0
    obs = new_episode(env, 9)
    out = [obs.cpu().clone()]
    for i in range(steps):
        obs, reward, strehl, _, _ = env.step(i, 0.4 * obs)
        out += [obs.cpu().clone(), reward.cpu().clone(), strehl.cpu().clone(), env.wfs.signal.cpu().clone()]
    torch.cuda.synchronize()
    assert (env._native is not None) == one_call
    return env, out


@pytest.mark.parametrize("n", WIDE)
@pytest.mark.parametrize("mode", ["diffractive", "noisy", "geometric"])
def test_native_step_is_bit_identical_to_call_by_call(dev, n, mode):
    """aoenv_sh_step against the entry points called one by one; 32 environments, so the reconstruction runs on the tensor
    cores from the bf16 planes."""
    cfg = CONFIGS["tiny"]()
    cfg.nPixPerSubap = n
    cfg.windSpeed, cfg.windDirection = [40.0, 75.0], [20.0, 250.0]
    if mode == "geometric":
        build = lambda: build_geometric_env(cfg, n_envs=32, rng="philox", seed=4, device=dev, canvas_slack=4)
    else:
        build = lambda: build_env(cfg, n_envs=32, rng="philox", seed=4, device=dev, canvas_slack=4)
    _, base = _run_steps(build, False, 8, noise=mode == "noisy")
    _, got = _run_steps(build, True, 8, noise=mode == "noisy")
    assert all(torch.equal(x, y) for x, y in zip(base, got))


def test_benchmark_batch_size(dev):
    """1024 environments of 20 x 20 lenslets of 12 pixels (R = 240), the benchmark's loop shape: the two-call step equals the
    call-by-call one bit for bit, and the slopes of sampled environments (both sides of warp and CTA boundaries, the last
    one) follow the float64 oracle on the OPD each of them saw."""
    cfg = CONFIGS["cfg1"]()
    cfg.nPixPerSubap = 12
    B = 1024

    build = lambda: build_env(cfg, n_envs=B, rng="philox", seed=17, device=dev)
    env, got = _run_steps(build, True, 3)
    _, base = _run_steps(build, False, 3)
    assert all(torch.equal(x, y) for x, y in zip(base, got))
    from rlao_b200 import gemm
    assert gemm.uses_tensor_cores(B)
    pupil = telescope_pupil(cfg.resolution)
    wl, nph = source_properties(cfg.opticalBand, cfg.magnitude)
    orc = ShackHartmannOracle(cfg, pupil, flux_map(pupil, nph, cfg.samplingTime, cfg.diameter), wl)
    assert rel_err(env.wfs.slopes_units, orc.slopes_units) < 1e-6
    orc.slopes_units = env.wfs.slopes_units
    opd = env.tel.OPD                                     # the OPD the last measurement saw, [B, R, R]
    sig = _np(env.wfs.signal)
    for e in (0, 1, 31, 32, 127, 128, 511, 777, B - 2, B - 1):
        want = orc.measure(_np(opd[e]) * pupil * 2 * np.pi / wl)
        _slopes_vs_oracle(sig[e], want, orc, (e, "slopes"))
