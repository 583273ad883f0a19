"""Mirror and lenslet-grid geometries that select their own kernel variants, without a GPU: which variant each geometry
selects (band width of the separable mirror, height of the in-place DM window, lazy or materialised surface, residue of
the pupil size and of the atmosphere's layer size mod 4, two-call or call-by-call step), pinned so that a change of a
threshold cannot silently move tests/test_gpu_geometries.py off the kernels it exists to run; and the float64 influence
functions of a mis-registered mirror, restated from OOPAO and checked against the mirror's own."""
import dataclasses
import math
import types

import numpy as np
import pytest

from oracle.ao_oracle import dm_geometry, dm_modes
from oracle.golden_configs import CONFIGS, EPISODE_SEED
import fake_backend_geometric
from parity_util import new_episode, param_from_config

MISREG = dict(shiftX=0.07, shiftY=-0.04, radialScaling=0.02, tangentialScaling=-0.01)

# nSubap x n pixels per lenslet, mechanical coupling, mirror.  `n` is the default lenslet size of the geometry.
GEOMETRIES = {
    "wl18": dict(nSubap=16, n=6, coupling=0.7),              # influence bands of 16 columns, DM windows of 18 rows
    "unbanded": dict(nSubap=16, n=6, coupling=0.75),         # bands wider than 16: unbanded kernel, materialised surface
    "misreg": dict(nSubap=20, n=6, coupling=0.35, misreg=MISREG),   # separable, off the lenslet grid
    "razor": dict(nSubap=20, n=6, coupling=0.35, razor=True),      # explicit coordinates: dense contraction
    "odd42": dict(nSubap=7, n=6, coupling=0.35),             # R = 42
    "odd50": dict(nSubap=5, n=10, coupling=0.35),            # R = 50
}
WL18_SIZES = (4, 6, 8, 10, 12)

# What each geometry selects: separable band width W (None: no separable tables), DM window height WL (None: the surface
# is materialised), R mod 4, layer size M mod 4, and whether env.step takes the two-call native step.
SELECTIONS = {
    "wl18": dict(W=16, WL=18, R4=0, M4=2, native=True),
    "unbanded": dict(W=0, WL=None, R4=0, M4=2, native=False),
    "misreg": dict(W=12, WL=14, R4=0, M4=2, native=True),
    "razor": dict(W=None, WL=None, R4=0, M4=2, native=False),
    "odd42": dict(W=12, WL=14, R4=2, M4=0, native=True),
    "odd50": dict(W=12, WL=14, R4=2, M4=0, native=True),
}


def geometry_config(name, n=None):
    """oracle AOConfig of a geometry (two layers of the 'tiny' configuration)."""
    g = GEOMETRIES[name]
    cfg = CONFIGS["tiny"]()
    cfg.nSubap, cfg.nPixPerSubap, cfg.mechCoupling = g["nSubap"], n or g["n"], g["coupling"]
    if g.get("razor"):
        cfg.dm_geometry = "razor"
    return cfg


def cartesian_mask(cfg):
    """The default mirror's valid-actuator mask [nAct, nAct]: the razor geometry is given this mask explicitly."""
    return dm_geometry(dataclasses.replace(cfg, dm_geometry="cartesian"))[2]


def build_geometry_env(name, n=None, n_envs=1, rng="reference", seed=0, device=None, geometric=False, canvas_slack=32,
                       cfg_overrides=None):
    """(cfg, env) of a geometry, as parity_util.build_env builds the default one; `cfg_overrides`: AOConfig fields."""
    from rlao_b200.OOPAOEnv.OOPAOEnvRazor import OOPAO
    cfg = geometry_config(name, n)
    for k, v in (cfg_overrides or {}).items():
        setattr(cfg, k, v)
    g = GEOMETRIES[name]
    p = param_from_config(cfg)
    p.update(g.get("misreg", {}))
    if g.get("razor"):
        p["dm_geometry"] = "razor"
        p["boolActMask"] = cartesian_mask(cfg).astype(int)
    p["is_geometric"] = geometric
    env = OOPAO()
    env.set_params_file(p, "")
    env.set_params(types.SimpleNamespace(), "shackhartmann", gainCL=cfg.gainCL, n_envs=n_envs, rng=rng, seed=seed,
                   device=device, canvas_slack=canvas_slack)
    env.leak = cfg.leak
    return cfg, env


def influence_functions(cfg, misreg=None):
    """OOPAO/DeformableMirror.py:286-341,494-514 in float64 numpy: the Cartesian mirror's valid actuators (chosen before
    the mis-registration), moved by anamorphosis, rotation and shift, with anisotropic Gaussian influence functions on the
    grid linspace(0, 1, R) * R.  OOPAO passes (tangentialScaling, radialScaling) as (mRad, mNorm) to its anamorphosis, and
    widens the Gaussian by (1 + radialScaling) along x and (1 + tangentialScaling) along y.  Returns modes [R*R, nValid]
    and, for a mirror without rotation and anamorphosis angle, its separable factors gx [nAct, R] (per actuator column)
    and gy [nAct, R] (per actuator row): modes[:, k] = gy[row k] (outer) gx[column k]."""
    m = dict(rotationAngle=0.0, shiftX=0.0, shiftY=0.0, anamorphosisAngle=0.0, tangentialScaling=0.0, radialScaling=0.0)
    m.update(misreg or {})
    D, R, nS = cfg.diameter, cfg.resolution, cfg.nSubap
    nAct, pitch = nS + 1, D / nS
    x = np.linspace(-D / 2, D / 2, nAct)
    X, Y = np.meshgrid(x, x)
    xs, ys = X.reshape(-1), Y.reshape(-1)
    r = np.hypot(xs, ys)
    valid = (r > cfg.centralObstruction * D / 2 - 0.5 * pitch) & (r <= D / 2 + 0.7533 * pitch)

    def moved(x0, y0):
        th = math.radians(m["anamorphosisAngle"])
        mRad, mNorm = 1 + m["tangentialScaling"], 1 + m["radialScaling"]
        cross = mNorm * math.sin(2 * th) / 2 - mRad * math.sin(2 * th) / 2
        x3 = x0 * (mRad * math.cos(th) ** 2 + mNorm * math.sin(th) ** 2) + y0 * cross
        y3 = y0 * (mRad * math.sin(th) ** 2 + mNorm * math.cos(th) ** 2) + x0 * cross
        rot = math.radians(m["rotationAngle"])
        x4, y4 = x3 * math.cos(rot) - y3 * math.sin(rot), y3 * math.cos(rot) + x3 * math.sin(rot)
        return x4 - m["shiftX"], y4 - m["shiftY"]

    xIF, yIF = moved(xs[valid], ys[valid])
    base = (R / nS) / math.sqrt(2 * math.log(1 / cfg.mechCoupling))
    cx, cy = (1 + m["radialScaling"]) * base, (1 + m["tangentialScaling"]) * base
    th = math.radians(m["anamorphosisAngle"])
    a = math.cos(th) ** 2 / (2 * cx ** 2) + math.sin(th) ** 2 / (2 * cy ** 2)
    b = -math.sin(2 * th) / (4 * cx ** 2) + math.sin(2 * th) / (4 * cy ** 2)
    c = math.sin(th) ** 2 / (2 * cx ** 2) + math.cos(th) ** 2 / (2 * cy ** 2)
    g = np.linspace(0, 1, R) * R
    dx = g[None, None, :] - (R / 2 + xIF * R / D)[:, None, None]
    dy = g[None, :, None] - (R / 2 + yIF * R / D)[:, None, None]
    modes = np.exp(-(a * dx ** 2 + 2 * b * dx * dy + c * dy ** 2)).reshape(len(xIF), R * R).T.copy()
    gx = gy = None
    if m["rotationAngle"] == 0 and m["anamorphosisAngle"] == 0:
        xc, yc = moved(x, x)                                   # (x3 = x mRad and y3 = y mNorm at zero angle)
        gx = np.exp(-a * (g[None, :] - (R / 2 + xc * R / D)[:, None]) ** 2)
        gy = np.exp(-c * (g[None, :] - (R / 2 + yc * R / D)[:, None]) ** 2)
    return modes, valid.reshape(nAct, nAct), gx, gy


def reference_modes(cfg, name):
    """float64 influence functions [R*R, nValid] of a geometry's mirror and, if it is separable, its column factors
    [nAct, R]: the oracle's for the razor geometry, the restatement above for the Cartesian ones."""
    if GEOMETRIES[name].get("razor"):
        xIF, yIF, _, sigma = dm_geometry(cfg, cartesian_mask(cfg))
        return dm_modes(cfg, xIF, yIF, sigma)[0], None
    modes, _, gx, _ = influence_functions(cfg, GEOMETRIES[name].get("misreg"))
    return modes, gx


@pytest.fixture
def fake(monkeypatch):
    return fake_backend_geometric.install(monkeypatch)


def _mirror(cfg, misreg=None, n_envs=1):
    from rlao_b200.DeformableMirror import DeformableMirror
    from rlao_b200.MisRegistration import MisRegistration
    from rlao_b200.Source import Source
    from rlao_b200.Telescope import Telescope
    tel = Telescope(cfg.resolution, cfg.diameter, cfg.samplingTime, n_envs=n_envs)
    Source(cfg.opticalBand, cfg.magnitude) * tel
    mr = MisRegistration()
    for k, v in (misreg or {}).items():
        setattr(mr, k, v)
    return tel, DeformableMirror(tel, cfg.nSubap, cfg.mechCoupling, misReg=mr)


def test_restated_influence_functions_are_the_oracles_without_misregistration():
    cfg = geometry_config("odd42")
    modes, valid, gx, gy = influence_functions(cfg)
    xIF, yIF, mask, sigma = dm_geometry(cfg)
    want, wgx, wgy = dm_modes(cfg, xIF, yIF, sigma)
    assert np.array_equal(valid, mask)
    assert np.abs(modes - want).max() < 1e-13
    # the factors are per actuator column / row of the full grid, the oracle's per valid actuator
    rows, cols = np.nonzero(mask)
    assert np.abs(gx[cols] - wgx).max() < 1e-13 and np.abs(gy[rows] - wgy).max() < 1e-13


@pytest.mark.parametrize("misreg", [dict(shiftX=0.07, shiftY=-0.04), dict(radialScaling=0.02, tangentialScaling=-0.01),
                                    MISREG])
def test_misregistered_mirror_modes_equal_the_restatement(fake, misreg):
    """dm.modes (float64) of a shifted / scaled mirror against OOPAO's influence functions restated above; the mirror stays
    separable, and its factors reproduce the same modes.  The GPU tests use the restatement as their float64 reference."""
    cfg = geometry_config("misreg")
    _, dm = _mirror(cfg, misreg)
    modes, valid, gx, gy = influence_functions(cfg, misreg)
    assert np.array_equal(dm.validAct.reshape(valid.shape), valid)
    got = dm.modes.double().numpy()
    assert got.shape == modes.shape
    assert np.abs(got - modes).max() < 1e-12
    assert dm._sep is not None                                 # shifts and scalings keep the separable kernels
    rows, cols = np.nonzero(valid)
    R = cfg.resolution
    sep = (gy[rows][:, :, None] * gx[cols][:, None, :]).reshape(len(rows), R * R).T
    assert np.abs(sep - modes).max() < 1e-12
    assert np.abs(dm._sep["gy_host"] - gy).max() < 1e-12
    # and the mis-registration does move the mirror: the restatement is not the oracle's unshifted mirror
    xIF, yIF, _, sigma = dm_geometry(cfg)
    assert np.abs(dm_modes(cfg, xIF, yIF, sigma)[0] - modes).max() > 1e-2


@pytest.mark.parametrize("n", WL18_SIZES)
def test_wl18_selects_the_18_row_window_at_every_lenslet_size(fake, n):
    """16 x 16 lenslets, coupling 0.7: bands of 16 actuator columns (dm_separable_banded_kernel<16>, dm_rows W = 16) and
    lenslet rows whose bands span 15-18 actuator rows (shwfs_frame_kernel<n, 18>, shwfs_frame_wide_kernel<n, 18>,
    shwfs_geometric_kernel<n, V, 18>)."""
    from rlao_b200.ShackHartmann import ShackHartmann
    cfg = geometry_config("wl18", n)
    tel, dm = _mirror(cfg)
    wfs = ShackHartmann(cfg.nSubap, tel, cfg.lightRatio)
    t = dm.fused_tables()
    assert t is not None and t["W"] == 16
    WL, ilr, _ = wfs._dm_windows_host(t)
    assert WL == 18
    # a window of 14 would not do: some lenslet row needs more than 14 actuator rows
    by = t["by_host"]
    need = (by[:, 1].reshape(cfg.nSubap, n).max(axis=1) - ilr + 1).max()
    assert 14 < need <= 18


@pytest.mark.parametrize("name", list(GEOMETRIES))
def test_geometry_selects_its_kernel_variant(fake, name):
    """Each geometry of tests/test_gpu_geometries.py selects the variant that file is there to run."""
    want = SELECTIONS[name]
    cfg, env = build_geometry_env(name)
    dm, wfs, R = env.dm, env.wfs, env.tel.resolution
    assert R == cfg.resolution
    if want["W"] is None:
        assert dm._sep is None and dm.fused_tables() is None
    else:
        assert dm._sep is not None and dm._sep["W"] == want["W"]
    tables = dm.fused_tables()
    if want["WL"] is None:
        assert tables is None and not dm.lazy_surface
    else:
        assert tables is not None and dm.lazy_surface
        assert wfs._dm_windows_host(tables)[0] == want["WL"]
    assert R % 4 == want["R4"]
    assert env.atm._M % 4 == want["M4"]
    obs = new_episode(env, EPISODE_SEED)
    for i in range(2):
        obs, *_ = env.step(i, cfg.gainCL * obs)
    assert (env._native is not None) == want["native"]
    if GEOMETRIES[name].get("razor"):
        assert np.array_equal(env.dm_mask, cartesian_mask(cfg).astype(int))
        assert dm.nValidAct == int(cartesian_mask(cfg).sum())
