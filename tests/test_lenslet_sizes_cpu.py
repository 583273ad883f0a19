"""Lenslets of 10 and 12 pixels without a GPU: the sizes the sensor accepts, the float64 oracle's properties at every
compiled size, the DM window the in-place surface needs, and the environment's host layer (calibration, call-by-call and
two-call steps, diffractive and geometric) driven through the CPU stand-in of the library."""
import importlib
import types

import numpy as np
import pytest

from oracle.ao_oracle import AOConfig, EnvOracle, ShackHartmannOracle, flux_map, source_properties, telescope_pupil
from oracle.golden_configs import CONFIGS, EPISODE_SEED
import fake_backend_geometric
from geometric_oracle import GeometricEnvOracle
from parity_util import build_env, new_episode, param_from_config, rel_err

SIZES = (4, 6, 8, 10, 12)


def test_sensor_accepts_the_compiled_sizes_only():
    sh = importlib.import_module("rlao_b200.ShackHartmann")
    assert sh._SUPPORTED_N == SIZES
    for n in (5, 7, 14):
        tel = types.SimpleNamespace(src=types.SimpleNamespace(type="NGS"), device="cpu", n_envs=1, resolution=8 * n)
        with pytest.raises(NotImplementedError, match=r"compiled sizes are \(4, 6, 8, 10, 12\)"):
            sh.ShackHartmann(8, tel, 0.5)


def oracle_sensor(nSubap, n):
    cfg = AOConfig(nSubap=nSubap, nPixPerSubap=n)
    pupil = telescope_pupil(cfg.resolution)
    wl, nph = source_properties(cfg.opticalBand, cfg.magnitude)
    return ShackHartmannOracle(cfg, pupil, flux_map(pupil, nph, cfg.samplingTime, cfg.diameter), wl), wl


@pytest.mark.parametrize("n", SIZES)
def test_oracle_properties(n):
    """Flat wavefront -> zero slopes; a tip ramp of amplitude a (the slope-unit ramp) reads a 2 pi / lambda on X and
    nothing on Y (on average); piston does not move the spots; small wavefronts add."""
    wfs, wl = oracle_sensor(8, n)
    R, nV, pupil = wfs.R, wfs.nValid, wfs.pupil
    assert np.all(wfs.measure(np.zeros((R, R))) == 0)
    tip = np.tile(np.linspace(0, np.pi, R, endpoint=False)[None, :], (R, 1))
    tip = tip / np.std(tip[pupil.astype(int)])
    for a in (-10e-9, 5e-9, 15e-9):
        s = wfs.measure(pupil * tip * a * 2 * np.pi / wl).copy()
        # to the nonlinearity the five-ramp linear fit of the slope units leaves (a few per cent at the edge lenslets)
        assert abs(s[:nV].mean() - a * 2 * np.pi / wl) < 0.1 * abs(a * 2 * np.pi / wl), (n, a)
        # partially lit edge lenslets see some Y; the pupil's symmetry cancels it in the mean
        assert abs(s[nV:].mean()) < 1e-9 * abs(a * 2 * np.pi / wl)
    rs = np.random.RandomState(n)
    x = np.linspace(-1, 1, R)
    X, Y = np.meshgrid(x, x)

    def smooth(k):
        c = rs.normal(size=4)
        opd = c[0] * X + c[1] * Y + c[2] * X * Y + c[3] * (X ** 2 - Y ** 2)
        return pupil * opd * (3e-9 / np.std(opd[pupil > 0])) * 2 * np.pi / wl
    p1, p2 = smooth(0), smooth(1)
    s1, s2 = wfs.measure(p1).copy(), wfs.measure(p2).copy()
    scale = np.abs(s1).max()
    assert np.allclose(wfs.measure(p1 + 2.3 * pupil), s1, rtol=0, atol=1e-9 * scale)
    assert rel_err(wfs.measure(p1 + p2), s1 + s2) < 2e-2
    assert rel_err(wfs.measure(-0.5 * p1), -0.5 * s1) < 2e-2


@pytest.fixture
def fake(monkeypatch):
    return fake_backend_geometric.install(monkeypatch)


def wide_config(n):
    cfg = CONFIGS["tiny"]()
    cfg.nPixPerSubap = n
    return cfg


def build(cfg, geometric):
    from rlao_b200.OOPAOEnv.OOPAOEnvRazor import OOPAO
    if not geometric:
        return build_env(cfg)
    param = param_from_config(cfg)
    param["is_geometric"] = True
    env = OOPAO()
    env.set_params_file(param, "")
    env.set_params(types.SimpleNamespace(), "shackhartmann", gainCL=cfg.gainCL, n_envs=1, rng="reference")
    env.leak = cfg.leak
    return env


@pytest.mark.parametrize("n", [10, 12])
@pytest.mark.parametrize("geometric", [False, True])
@pytest.mark.parametrize("native", [True, False])
def test_env_calibrates_and_steps_at_wide_lenslets(fake, monkeypatch, n, geometric, native):
    """set_params with nPixelPerSubap = 10 / 12: the calibration (interaction matrix, reconstructor) and the closed loop
    follow the float64 oracle; the default step is the two-call one (the in-place DM window exists at these sizes)."""
    monkeypatch.setenv("AOENV_STEP_NATIVE", "1" if native else "0")
    cfg = wide_config(n)
    env = build(cfg, geometric)
    assert env.wfs.n_pix_subap == n and env.tel.resolution == 8 * n and env.wfs.is_geometric == geometric
    win = env.wfs._dm_windows(env.dm.fused_tables())
    assert win is not None and win[0] == 14
    orc = GeometricEnvOracle(cfg) if geometric else EnvOracle(cfg)
    assert env.dm.nValidAct == orc.nValidAct
    assert np.array_equal(env.wfs.valid_subapertures, orc.wfs.valid)
    assert rel_err(env.wfs.slopes_units, orc.wfs.slopes_units) < 1e-5
    assert rel_err(env.reconstructor.cpu().numpy(), orc.reconstructor) < 2e-3
    obs = new_episode(env, EPISODE_SEED)
    obs_o = orc.new_episode(EPISODE_SEED)
    assert rel_err(obs.numpy(), obs_o) < 5e-4
    for i in range(8):
        obs, reward, strehl, done, info = env.step(i, cfg.gainCL * obs)
        obs_o, reward_o, strehl_o, _, _ = orc.step(i, cfg.gainCL * obs_o)
        assert rel_err(env.wfs.signal.numpy(), orc.wfs.signal) < 2e-4, i
        assert rel_err(obs.numpy(), obs_o) < 2e-3, i
        assert abs(float(reward) - reward_o) < 2e-3 * abs(reward_o), i
        assert abs(float(env.total[i]) - orc.total[i]) < 1e-3 * orc.total[i]
        assert abs(float(env.residual[i]) - orc.residual[i]) < 2e-3 * orc.residual[i]
    assert (env._native is not None) == native


def test_window_height_does_not_grow_with_the_lenslet(fake):
    """The in-place DM window counts actuator rows: a lenslet spans about one actuator pitch whatever its pixel count,
    so the default mirror needs the same WL at every size."""
    for n in SIZES:
        env = build(wide_config(n), False)
        assert env.wfs._dm_windows_host(env.dm.fused_tables())[0] == 14, n


def test_fused_kernel_rejects_wide_lenslets(fake, monkeypatch):
    monkeypatch.setenv("AOENV_WFS", "fused")
    with pytest.raises(NotImplementedError, match="fused WFS kernel"):
        build(wide_config(10), False)
