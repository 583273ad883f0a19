"""Kernel variants that the mirror's and the lenslet grid's geometry select, against float64 (the geometries and their
selections are pinned in tests/test_geometries_cpu.py):

    wl18      16 x {4..12} px, coupling 0.7    banded DM W = 16, in-place DM windows of WL = 18 actuator rows
    unbanded  16 x 6, coupling 0.75            unbanded dm_separable_kernel, materialised surface, call-by-call step
    misreg    20 x 6, shifted and scaled       separable mirror off the lenslet grid, evaluated in place
    razor     20 x 6, explicit coordinates     dense DM contraction (SIMT at 1 environment, tensor cores at 16)
    odd42     7 x 6 (R = 42)                   R = 2 mod 4: float2 geometric kernels, scalar tails, layers M = 0 mod 4
    odd50     5 x 10 (R = 50)                  the same with the wide frame kernel

DM surfaces and T = C gx against modes64 @ coefs; frames, slopes and pupil variances of the spots kernel with the mirror
evaluated in place against ShackHartmannOracle on float64 (atmosphere + mirror); the geometric sensor against its oracle;
the closed loop against the oracle environment; the two-call step against the call-by-call one; and a profiler capture
that shows each instantiation really ran."""
import math

import numpy as np
import pytest
import torch

from oracle.ao_oracle import EnvOracle, ShackHartmannOracle, flux_map, source_properties, telescope_pupil
from oracle.golden_configs import EPISODE_SEED
from parity_util import knife_edge_lenslets, new_episode, rel_err
from geometric_oracle import GeometricShackHartmannOracle
from test_geometries_cpu import GEOMETRIES, SELECTIONS, WL18_SIZES, build_geometry_env, cartesian_mask, reference_modes
from test_gpu_geometric import _frame_stats, _opds, stats_tol

pytestmark = pytest.mark.gpu

FRAME_TOL = 2e-4
SLOPE_TOL = 1e-4
VAR_TOL = 5e-5
SEP_TOL = 2e-6            # separable kernels against float64 modes (test_dm_surface_vs_oracle_and_linearity)
SURFACE_TOL = 1e-4        # the dense contraction (tensor cores at 16 environments)

# geometries whose mirror the spots kernels evaluate in place, with the lenslet size
IN_PLACE = [("wl18", n) for n in WL18_SIZES] + [("misreg", 6), ("odd42", 6), ("odd50", 10)]
SURFACES = [(name, n, 3) for name, n in IN_PLACE] + [("unbanded", 6, 3), ("razor", 6, 1), ("razor", 6, 16)]
LOOPS = [("wl18", 6), ("unbanded", 6), ("misreg", 6), ("razor", 6), ("odd42", 6), ("odd50", 10)]
NATIVE = [("wl18", 6), ("misreg", 6), ("odd42", 6), ("odd50", 10)]


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    return torch.device("cuda:0")


@pytest.fixture(scope="module")
def envs(dev):
    """Environments of 3 (or B) environments per geometry, built once for the module; tests set the state they use."""
    cache = {}

    def get(name, n, B=3, geometric=False):
        key = (name, n, B, geometric)
        if key not in cache:
            cache[key] = build_geometry_env(name, n, n_envs=B, rng="philox", seed=3, device=dev, geometric=geometric)
        return cache[key]
    return get


@pytest.fixture(scope="module")
def modes64():
    """float64 influence functions (and column factors) per (geometry, lenslet size)."""
    cache = {}

    def get(name, cfg):
        key = (name, cfg.resolution)
        if key not in cache:
            cache[key] = reference_modes(cfg, name)
        return cache[key]
    return get


def _np(t):
    return t.detach().double().cpu().numpy()


def _commands(dm, B, seed, scale):
    return (np.random.RandomState(seed).normal(size=(B, dm.nValidAct)) * scale).astype(np.float32)


def _oracle_sensor(cfg, cls=ShackHartmannOracle):
    pupil = telescope_pupil(cfg.resolution)
    wl, nph = source_properties(cfg.opticalBand, cfg.magnitude)
    return cls(cfg, pupil, flux_map(pupil, nph, cfg.samplingTime, cfg.diameter), wl), pupil, wl


def _slopes_vs_oracle(got, want, orc, what):
    """Slopes to SLOPE_TOL of the array's maximum, lenslets with a pixel at the centroiding threshold excluded."""
    maps = orc.maps_intensity
    edge = knife_edge_lenslets(maps, orc.threshold_cog * maps.max())
    keep = np.concatenate([~edge, ~edge])
    assert edge.sum() <= max(2, 0.02 * orc.nValid), (what, "knife-edge lenslets", int(edge.sum()))
    assert np.abs(got - want)[keep].max() < SLOPE_TOL * np.abs(want).max(), what


def _variances_vs_float64(stats, opds, pupil, P):
    """Pupil variances of the atmosphere and of the total OPD from a kernel's statistics [B, 4] against float64."""
    inside = pupil.astype(bool)
    for i, opd in zip((0, 2), opds):
        var = stats[:, i + 1] / P - (stats[:, i] / P) ** 2
        want = np.array([o[inside].var() for o in opd])
        assert np.abs(var / want - 1).max() < VAR_TOL, ("variance", i)


@pytest.mark.parametrize("name,n,B", SURFACES)
def test_dm_surface_vs_float64(dev, envs, modes64, name, n, B):
    """dm.OPD and, for the lazy mirrors, T = C gx (aoenv_dm_rows) against float64 products on the same float32 commands."""
    cfg, env = envs(name, n, B)
    dm, R = env.dm, cfg.resolution
    m64, gx64 = modes64(name, cfg)
    assert m64.shape == (R * R, dm.nValidAct)
    c32 = _commands(dm, B, 7, 1e-7)
    dm.coefs = torch.as_tensor(c32, device=dev)
    c64 = c32.astype(np.float64)
    if SELECTIONS[name]["WL"] is not None:
        assert dm.lazy_surface and not dm._valid[dm._slot]
        T = _np(dm._rows_of(dm._slot))                         # [B, nAct + 18, R]
        nAct = dm.nAct
        C = np.zeros((B, nAct * nAct))
        C[:, dm._sep["act_pos"].cpu().numpy()] = c64
        want_T = C.reshape(B, nAct, nAct) @ gx64               # [B, nAct, R]
        assert rel_err(T[:, :nAct], want_T) < SEP_TOL
        assert not T[:, nAct:].any()                           # the padding rows the windows may run into stay zero
    got = _np(dm.OPD).reshape(B, R, R)
    want = (c64 @ m64.T).reshape(B, R, R)
    assert rel_err(got, want) < (SURFACE_TOL if name == "razor" else SEP_TOL)
    if name == "razor":
        from rlao_b200 import gemm
        assert dm._sep is None and gemm.uses_tensor_cores(B) == (B > 8)


@pytest.mark.parametrize("name,n", IN_PLACE)
def test_spots_slopes_and_variances_with_the_mirror_in_place(dev, envs, modes64, name, n):
    """aoenv_shwfs_frame_dm with the separable mirror evaluated in place (WL = 14 or 18 row windows) against the float64
    oracle on (atmosphere + modes64 @ coefs): frames, slopes (knife-edge lenslets excluded), pupil variances."""
    cfg, env = envs(name, n)
    wfs, dm, tel = env.wfs, env.dm, env.tel
    B, R = 3, cfg.resolution
    orc, pupil, wl = _oracle_sensor(cfg)
    assert np.array_equal(wfs.valid_subapertures, orc.valid)
    assert rel_err(wfs.slopes_units, orc.slopes_units) < 1e-6
    m64, _ = modes64(name, cfg)
    c32 = _commands(dm, B, 11, 5e-8)
    dm.coefs = torch.as_tensor(c32, device=dev)
    ref = dm.surface_ref()
    b_t, dm_struct = wfs._second_term(ref)
    assert b_t is None and dm_struct is not None and dm_struct.WL == SELECTIONS[name]["WL"]
    opd_a = env.atm._opd
    frame = torch.empty((B, R, R), dtype=torch.float32, device=dev)
    envmax = torch.zeros((B,), dtype=torch.int32, device=dev)
    stats = torch.zeros((B, 4), dtype=torch.float64, device=dev)
    slopes = torch.zeros_like(wfs._signal)
    wfs._run(opd_a, ref, tel._pupil_f, 2 * math.pi / wl, False, None, frame, envmax, stats, slopes, wfs._ref_xy,
             1.0 / orc.slopes_units)
    assert not dm._valid[dm._slot]                             # the surface was never written
    a64 = _np(opd_a)
    total = a64 + (c32.astype(np.float64) @ m64.T).reshape(B, R, R)
    got_frame, got_sig, st = _np(frame), _np(slopes)[:, :wfs.nSignal], _np(stats)
    for e in range(B):
        want = orc.measure(total[e] * pupil * 2 * np.pi / wl)
        assert rel_err(got_frame[e], orc.frame) < FRAME_TOL, (e, "frame")
        _slopes_vs_oracle(got_sig[e], want, orc, (e, "slopes"))
    _variances_vs_float64(st, (a64, total), pupil, float(tel.pixelArea))


@pytest.mark.parametrize("name,n", IN_PLACE)
def test_geometric_sensor_vs_oracle(dev, envs, modes64, name, n):
    """aoenv_shwfs_geometric with one OPD term, two terms and the mirror in place (V = 2 at R = 2 mod 4; WL = 18 windows at
    wl18) against the geometric oracle; its pupil statistics against the frame kernel's; the float64 twin."""
    cfg, env = envs(name, n, geometric=True)
    wfs, dm = env.wfs, env.dm
    B, R = 3, cfg.resolution
    orc, pupil, wl = _oracle_sensor(cfg, GeometricShackHartmannOracle)
    assert np.array_equal(wfs.valid_subapertures, orc.valid)
    assert rel_err(wfs.slopes_units, orc.slopes_units) < 2e-6
    inv = 1.0 / orc.slopes_units
    scale = 2 * np.pi / wl
    a = env.atm._opd
    a64 = _np(a)
    b32 = _opds(R, B, 6, scale=0.1e-6).astype(np.float32)
    b = torch.as_tensor(b32, device=dev)
    slopes = torch.zeros_like(wfs._signal)
    stats = torch.zeros((B, 4), dtype=torch.float64, device=dev)

    def check(got, total, what):
        for e in range(B):
            assert rel_err(got[e, :wfs.nSignal], orc.measure(total[e] * scale)) < SLOPE_TOL, (e, what)
    wfs._run_geometric(a, None, slopes, inv)
    check(_np(slopes), a64, "one term")
    wfs._run_geometric(a, b, slopes, inv, None, stats)
    check(_np(slopes), _np(a + b), "two terms")
    assert rel_err(_np(stats), _frame_stats(wfs, a, b)) < stats_tol(n)
    m64, _ = modes64(name, cfg)
    c32 = _commands(dm, B, 13, 5e-8)
    dm.coefs = torch.as_tensor(c32, device=dev)
    ref = dm.surface_ref()
    b_t, dm_struct = wfs._second_term(ref)
    assert b_t is None and dm_struct is not None and dm_struct.WL == SELECTIONS[name]["WL"]
    wfs._run_geometric(a, ref, slopes, inv, None, stats)
    assert not dm._valid[dm._slot]
    total = a64 + (c32.astype(np.float64) @ m64.T).reshape(B, R, R)
    check(_np(slopes), total, "mirror in place")
    assert rel_err(_np(stats), _frame_stats(wfs, a, dm=dm_struct)) < stats_tol(n)
    _variances_vs_float64(_np(stats), (a64, total), pupil, float(env.tel.pixelArea))
    frames = wfs.measure_frames(a) * wfs.slopes_units
    want = orc.measure_multi(a64 * scale).T * orc.slopes_units
    assert rel_err(_np(frames), want) < 1e-9


@pytest.fixture(scope="module")
def atm_ops():
    """Atmosphere operators of the oracle environments, shared between geometries of the same pupil size."""
    return {}


@pytest.mark.parametrize("name,n", LOOPS)
def test_closed_loop_vs_oracle_environment(dev, modes64, atm_ops, name, n):
    """rng='reference', one environment: the environment and the oracle environment in lock step with the same
    reconstructor, every step driven with the oracle's action; the atmosphere at two snapshot steps."""
    cfg, env = build_geometry_env(name, n, n_envs=1, rng="reference", device=dev)
    R = cfg.resolution
    mask = cartesian_mask(cfg) if GEOMETRIES[name].get("razor") else None
    if name == "misreg":
        # the oracle's mirror has no mis-registration: give it the restated influence functions (and the environment's
        # reconstructor: the oracle's own calibration would be of the other mirror)
        orc = EnvOracle(cfg, atm_ops=atm_ops.get(R), reconstructor=_np(env.reconstructor))
        orc.modes = modes64(name, cfg)[0]
        assert orc.modes.shape[1] == orc.nValidAct == env.dm.nValidAct
    else:
        orc = EnvOracle(cfg, atm_ops=atm_ops.get(R), act_mask=mask)
        assert env.dm.nValidAct == orc.nValidAct
        assert rel_err(_np(env.calib_zonal.D), orc.D_zonal) < 1e-5
    atm_ops[R] = orc.atm.ops
    assert np.array_equal(env.wfs.valid_subapertures, orc.wfs.valid)
    assert rel_err(env.wfs.slopes_units, orc.wfs.slopes_units) < 1e-6
    env.set_reconstructor(orc.reconstructor)
    env.wfs.slopes_units = float(orc.wfs.slopes_units)
    nV = env.wfs.nValidSubaperture
    obs = new_episode(env, EPISODE_SEED)
    obs_o = orc.new_episode(EPISODE_SEED)
    assert rel_err(_np(obs), obs_o) < 2e-4
    steps, snaps = 20, (7, 19)
    for i in range(steps):
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
        if not edge.any():
            assert rel_err(_np(obs), obs_o) < 1e-3, (i, "obs")
            assert abs(float(reward) - reward_o) <= 1e-3 * abs(reward_o), (i, "reward")
        else:
            assert rel_err(_np(obs), obs_o) < 1e-2, (i, "obs, knife-edge step")
        if i in snaps:
            assert rel_err(_np(env.atm.OPD), orc.atm.OPD) < 3e-5, (i, "atmosphere")
    assert rel_err(_np(env.total[:steps, 0]), orc.total[:steps]) < 1e-4
    assert rel_err(_np(env.residual[:steps, 0]), orc.residual[:steps]) < 1e-3
    assert (env._native is not None) == SELECTIONS[name]["native"]


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
    return out


@pytest.mark.parametrize("name,n", NATIVE)
@pytest.mark.parametrize("mode", ["diffractive", "noisy", "geometric"])
def test_native_step_is_bit_identical_to_call_by_call(dev, name, n, mode):
    """aoenv_sh_step against the entry points called one by one; 32 environments (reconstruction on the tensor cores),
    winds of several pixels per frame."""
    over = dict(windSpeed=[40.0, 75.0], windDirection=[20.0, 250.0])
    build = lambda: build_geometry_env(name, n, n_envs=32, rng="philox", seed=4, device=dev, geometric=mode == "geometric",
                                       canvas_slack=4, cfg_overrides=over)[1]
    base = _run_steps(build, False, 8, noise=mode == "noisy")
    got = _run_steps(build, True, 8, noise=mode == "noisy")
    assert all(torch.equal(x, y) for x, y in zip(base, got))


def _expected_kernels(name, n, R, geometric):
    sel = SELECTIONS[name]
    WL = sel["WL"] or 0
    if geometric:
        names = [f"shwfs_geometric_kernel<{n},{4 if R % 4 == 0 else 2},{WL}>"]
    else:
        names = [f"shwfs_frame_wide_kernel<{n},{WL}>" if n > 8 else f"shwfs_frame_kernel<{n},{WL}>"]
    if sel["W"] is None:
        names.append("gemm_skinny_kernel")                   # the dense DM product of 3 environments
    elif sel["W"] == 0:
        names.append("dm_separable_kernel")
    else:
        names.append(f"dm_rows_kernel<{sel['W']}>")
    return names + ["atm_phase_kernel"]


@pytest.mark.parametrize("name,n", IN_PLACE + [("unbanded", 6), ("razor", 6)])
def test_the_selected_instantiations_run(dev, envs, name, n, capsys):
    """One step of each geometry under the profiler (CUDA activity): the instantiation the geometry selects is among the
    kernels launched (and the in-place geometries launch no surface kernel)."""
    from torch.profiler import ProfilerActivity, profile
    kinds = [False] + ([True] if (name, n) in IN_PLACE else [])
    for geometric in kinds:
        cfg, env = envs(name, n, geometric=geometric)
        obs = new_episode(env, 5)
        env.step(0, 0.4 * obs)
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            env.step(1, 0.4 * obs)
            torch.cuda.synchronize()
        ran = {e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA}
        for k in _expected_kernels(name, n, cfg.resolution, geometric):
            hits = sorted(r for r in ran if k in r.replace(" ", ""))
            assert hits, (name, n, geometric, k, sorted(ran))
            with capsys.disabled():
                i = hits[0].find(k.split("<")[0])
                print(f"\n{name} n={n} {'geometric' if geometric else 'diffractive'}: {hits[0][i:hits[0].find('(', i)]}")
        if SELECTIONS[name]["WL"] is not None:
            assert not any("dm_separable" in r for r in ran), (name, n, sorted(ran))
        assert (env._native is not None) == SELECTIONS[name]["native"]
