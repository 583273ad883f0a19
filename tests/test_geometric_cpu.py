"""Geometric Shack-Hartmann sensor without a GPU: the oracle's definition (DESIGN.md section 2) checked on its own and
against the diffractive oracle, and the environment's host layer driven through the CPU stand-in of the library."""
import types

import numpy as np
import pytest

from oracle.ao_oracle import AOConfig, ShackHartmannOracle, flux_map, source_properties, telescope_pupil
from oracle.golden_configs import CONFIGS, EPISODE_SEED
import fake_backend_geometric
from geometric_oracle import GeometricEnvOracle, GeometricShackHartmannOracle
from parity_util import new_episode, param_from_config, rel_err


def sensor(nSubap, n, geometric):
    cfg = AOConfig(nSubap=nSubap, nPixPerSubap=n)
    pupil = telescope_pupil(cfg.resolution)
    wl, nph = source_properties(cfg.opticalBand, cfg.magnitude)
    return (GeometricShackHartmannOracle if geometric else ShackHartmannOracle)(cfg, pupil, flux_map(pupil, nph, cfg.samplingTime, cfg.diameter), wl), wl


def full_ramp(R):
    ramp = np.linspace(0, np.pi, R, endpoint=False)
    tip = np.tile(ramp[None, :], (R, 1))
    return tip / np.std(tip)                        # the normalisation of the slope-unit ramps (full-ramp std)


@pytest.mark.parametrize("axis", [1, 0])
def test_oracle_ramp_reads_its_amplitude(axis):
    wfs, wl = sensor(20, 6, True)
    assert np.all(wfs.reference_slopes_maps == 0)
    a = 30e-9
    tip = full_ramp(wfs.R)
    opd = a * (tip if axis == 1 else tip.T)
    s = wfs.measure(opd * 2 * np.pi / wl)
    nV = wfs.nValid
    on, off = (s[:nV], s[nV:]) if axis == 1 else (s[nV:], s[:nV])
    assert np.allclose(on, a * 2 * np.pi / wl, rtol=1e-12, atol=0)
    assert np.abs(off).max() < 1e-12 * a * 2 * np.pi / wl


def test_oracle_piston_invariance_and_linearity():
    wfs, wl = sensor(8, 6, True)
    R = wfs.R
    rs = np.random.RandomState(3)
    p1, p2 = rs.normal(size=(R, R)), rs.normal(size=(R, R))
    s1, s2 = wfs.measure(p1).copy(), wfs.measure(p2).copy()
    assert np.allclose(wfs.measure(p1 + 7.5), s1, rtol=0, atol=1e-12 * np.abs(s1).max())
    assert np.allclose(wfs.measure(2.0 * p1 - 3.0 * p2), 2.0 * s1 - 3.0 * s2, rtol=0, atol=1e-12 * np.abs(s1).max())
    multi = wfs.measure_multi(np.stack([p1, p2]))
    assert np.allclose(multi[:, 0], s1, rtol=0, atol=0) and np.allclose(multi[:, 1], s2, rtol=0, atol=0)


@pytest.mark.parametrize("n", [4, 6, 8])
def test_oracle_agrees_with_diffractive_on_fully_lit_lenslets(n):
    """Smooth aberrations defined on the whole grid: the two sensors agree where no pupil edge crosses the lenslet."""
    geo, wl = sensor(20, n, True)
    dif, _ = sensor(20, n, False)
    assert np.array_equal(geo.valid, dif.valid)
    R = geo.R
    x = np.linspace(-1, 1, R)
    X, Y = np.meshgrid(x, x)
    full = (geo.photon_per_subap == geo.photon_per_subap.max())[geo.valid_1d]
    full2 = np.concatenate([full, full])
    for k, rms in enumerate((5e-9, 20e-9, 50e-9)):
        rs = np.random.RandomState(k)
        c = rs.normal(size=6)
        opd = c[0] * X + c[1] * Y + c[2] * X * Y + c[3] * (X ** 2 - Y ** 2) + c[4] * (2 * X ** 2 + 2 * Y ** 2 - 1) + c[5] * X ** 3
        opd *= rms / np.std(opd[geo.pupil])
        phase = opd * 2 * np.pi / wl
        sg = geo.measure(phase).copy()
        sd = dif.measure(phase * dif.pupil).copy()
        err = np.linalg.norm(sg[full2] - sd[full2]) / np.linalg.norm(sd[full2])
        assert err < 0.05, (n, rms, err)


def build_geometric_env(cfg, n_envs=1, rng="reference", seed=0, device=None, canvas_slack=32):
    """parity_util.build_env with the geometric sensor."""
    from rlao_b200.OOPAOEnv.OOPAOEnvRazor import OOPAO
    param = param_from_config(cfg)
    param["is_geometric"] = True
    env = OOPAO()
    env.set_params_file(param, "")
    env.set_params(types.SimpleNamespace(), "shackhartmann", gainCL=cfg.gainCL, n_envs=n_envs, rng=rng, seed=seed,
                   device=device, canvas_slack=canvas_slack)
    env.leak = cfg.leak
    return env


@pytest.fixture
def fake(monkeypatch):
    return fake_backend_geometric.install(monkeypatch)


@pytest.mark.parametrize("native", [True, False])
def test_env_step_sequence_matches_geometric_oracle_on_cpu(fake, monkeypatch, native):
    monkeypatch.setenv("AOENV_STEP_NATIVE", "1" if native else "0")
    cfg = CONFIGS["tiny"]()
    env = build_geometric_env(cfg)
    assert env.wfs.is_geometric and env.wfs._frame is None
    with pytest.raises(NotImplementedError):
        env.wfs.is_geometric = False
    orc = GeometricEnvOracle(cfg)
    assert env.dm.nValidAct == orc.nValidAct
    assert np.array_equal(env.wfs.valid_subapertures, orc.wfs.valid)
    assert np.all(env.wfs.reference_slopes_maps == 0)
    assert rel_err(env.wfs.slopes_units, orc.wfs.slopes_units) < 1e-5
    assert rel_err(env.reconstructor.cpu().numpy(), orc.reconstructor) < 2e-3
    obs = new_episode(env, EPISODE_SEED)
    obs_o = orc.new_episode(EPISODE_SEED)
    assert rel_err(obs.numpy(), obs_o) < 5e-4
    counter = env.wfs.cam.frame_counter
    for i in range(12):
        obs, reward, strehl, done, info = env.step(i, cfg.gainCL * obs)
        obs_o, reward_o, strehl_o, _, _ = orc.step(i, cfg.gainCL * obs_o)
        assert rel_err(env.wfs.signal.numpy(), orc.wfs.signal) < 2e-4, i
        assert rel_err(obs.numpy(), obs_o) < 2e-3, i
        assert abs(float(reward) - reward_o) < 2e-3 * abs(reward_o), i
        assert abs(float(strehl) - strehl_o) < 1e-3, i
        assert abs(float(env.total[i]) - orc.total[i]) < 1e-3 * orc.total[i]
        assert abs(float(env.residual[i]) - orc.residual[i]) < 2e-3 * orc.residual[i]
    assert (env._native is not None) == native
    assert env.wfs.cam.frame_counter == counter          # the camera is not used
    assert env.wfs.cam.frame is None


def test_geometric_signal_2d_and_light_ratio(fake):
    cfg = CONFIGS["tiny"]()
    env = build_geometric_env(cfg)
    wfs = env.wfs
    env.tel.resetOPD()
    R = env.tel.resolution
    a = 20e-9
    wfs.wfs_measure(phase_in=full_ramp(R) * a * 2 * np.pi / env.source.wavelength)
    s = wfs.signal.numpy()
    nV = wfs.nValidSubaperture
    assert np.allclose(s[:nV], a * 2 * np.pi / env.source.wavelength, rtol=1e-4)
    assert np.abs(s[nV:]).max() < 1e-4 * np.abs(s[:nV]).max()
    s2 = wfs.signal_2D.numpy()
    assert s2.shape == (2 * wfs.nSubap, wfs.nSubap)
    assert np.allclose(s2[:wfs.nSubap][wfs.valid_subapertures], s[:nV])
    n_before = wfs.nValidSubaperture
    wfs.lightRatio = 0.9
    assert wfs.nValidSubaperture < n_before and wfs.is_geometric
    assert np.all(wfs.reference_slopes_maps == 0)
