"""Parity of the CUDA path (through the C ABI, via the rlao_b200 host layer) against the CPU oracle and the
golden fixtures recorded from the unmodified reference.  Tolerances (north_star): noise-free slopes and DM
surfaces rel. 1e-4 (of the array's max), Strehl rel. 1e-3, on identical inputs; noisy runs: statistics."""
import math
import os

import numpy as np
import pytest
import torch

from oracle.ao_oracle import (AOConfig, AtmosphereOracle, EnvOracle, ShackHartmannOracle, compute_psf,
                              dm_geometry, dm_modes, flux_map, source_properties, telescope_pupil)
from oracle.golden_configs import CONFIGS, EPISODE_SEED, STEPS
from oracle.make_golden import load as load_golden
from oracle.warp018 import warp_translate
from parity_util import build_env, knife_edge_lenslets, new_episode, rel_err
from rlao_b200 import _lib

pytestmark = pytest.mark.gpu

SLOPE_TOL = 1e-4
SURFACE_TOL = 1e-4
STREHL_TOL = 1e-3


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    return torch.device("cuda:0")


def _np(t):
    return t.detach().double().cpu().numpy()


# ---------------------------------------------------------------------------------------------------------
def test_extension_is_the_code_that_runs(dev):
    from rlao_b200 import _lib
    lib = _lib.load()
    n0 = _lib.launch_count()
    x = torch.randn(8, 16, device=dev)
    w = torch.randn(5, 16, device=dev)
    d = torch.zeros(8, 8, device=dev)
    _lib.check(lib.aoenv_gemm_tn(_lib.ptr(x), 16, _lib.ptr(w), 16, _lib.ptr(d), 8, 8, 5, 16, 1.0, _lib.stream_ptr(dev)))
    torch.cuda.synchronize()
    assert _lib.launch_count() == n0 + 1
    assert rel_err(_np(d[:, :5]), _np(x) @ _np(w).T) < 1e-5


@pytest.mark.parametrize("M,N,K", [(1, 1, 16), (37, 131, 48), (300, 257, 1360), (128, 128, 16), (1024, 980, 2928),
                                   (1, 1353, 2528), (3, 500, 1488), (8, 357, 640), (9, 357, 640)])     # <= 8 rows: the warp-per-column kernel
def test_gemm_tn_vs_float64(dev, M, N, K):
    from rlao_b200 import _lib
    g = torch.Generator(device=dev).manual_seed(M * 7 + N)
    x = torch.randn(M, K, device=dev, generator=g)
    w = torch.randn(N, K, device=dev, generator=g)
    ldd = (N + 3) // 4 * 4
    d = torch.full((M, ldd), float("nan"), device=dev)
    _lib.check(_lib.load().aoenv_gemm_tn(_lib.ptr(x), K, _lib.ptr(w), K, _lib.ptr(d), ldd, M, N, K, 0.5, _lib.stream_ptr(dev)))
    ref = 0.5 * (_np(x) @ _np(w).T)
    assert rel_err(_np(d[:, :N]), ref) < 1e-5
    assert torch.isnan(d[:, N:]).all()          # padding columns are never written


def test_gemm_rejects_bad_arguments(dev):
    from rlao_b200 import _lib
    x = torch.zeros(4, 20, device=dev)
    rc = _lib.load().aoenv_gemm_tn(_lib.ptr(x), 20, _lib.ptr(x), 20, _lib.ptr(x), 20, 4, 4, 20, 1.0, _lib.stream_ptr(dev))
    assert rc != 0 and b"multiple of 16" in _lib.load().aoenv_last_error()


def test_entry_points_reject_bad_arguments(dev):
    """Every entry point validates shapes before launching: negative return code, message in aoenv_last_error, no launch."""
    lib = _lib.load()
    z = torch.zeros(4096, device=dev)
    zp, st = _lib.ptr(z), _lib.stream_ptr(dev)
    n0 = _lib.launch_count()
    cases = [
        (lib.aoenv_atm_gather(zp, 1, 10, 12, 120, 2, 0, zp, 8, 36, None, 0, 0, zp, 64, None, 3, st), b"shift"),
        (lib.aoenv_atm_ring(zp, 1, 10, 12, 120, 0, 35, zp, 36, zp, zp, 0, st), b"ring has"),
        (lib.aoenv_shwfs_frame(zp, None, zp, zp, zp, 1, 4, 5, 1.0, None, 0, zp, zp, None, st), b"pixels per lenslet"),
        (lib.aoenv_shwfs_slopes(zp, zp, 0, zp, 4, zp, 1.0, 0.01, 1, 4, 6, zp, 4, None, 2, st), b"shwfs_slopes"),
        (lib.aoenv_gemm_tn_tc(zp, zp, 12, 2, zp, 8, 4, 4, 12, 1.0, st), b"gemm_tn_tc"),
        (lib.aoenv_split_bf16(zp, 16, 4, 16, 5, zp, 16, st), b"parts"),
        (lib.aoenv_psf_peak(zp, None, zp, zp, zp, zp, 1, 7, 21, 1, 8, 1.0, zp, 16, zp, None, zp, st), b"psf_peak"),
        (lib.aoenv_dm_surface_separable(zp, 2, zp, 4, 2, zp, zp, zp, zp, None, None, None, None, 0, 1, 8, zp, st), b"dm_surface_separable"),
    ]
    for rc, needle in cases:
        assert rc < 0, needle
    # the message of the last failure is retrievable; nothing was launched
    assert b"dm_surface_separable" in lib.aoenv_last_error()
    assert _lib.launch_count() == n0


# ---------------------------------------------------------------------------------------------------------
def _tiny_objects(dev, n_envs=1, cfg=None):
    from rlao_b200.Atmosphere import Atmosphere
    from rlao_b200.Source import Source
    from rlao_b200.Telescope import Telescope
    cfg = cfg or CONFIGS["tiny"]()
    tel = Telescope(cfg.resolution, cfg.diameter, cfg.samplingTime, cfg.centralObstruction, n_envs=n_envs, device=dev)
    src = Source(cfg.opticalBand, cfg.magnitude)
    src * tel
    atm = Atmosphere(tel, cfg.r0, cfg.L0, cfg.windSpeed, cfg.fractionalR0, cfg.windDirection, cfg.altitude, rng="reference")
    return cfg, tel, src, atm


def test_atmosphere_operators_and_screens_vs_oracle(dev):
    cfg, tel, src, atm = _tiny_objects(dev)
    atm.initializeAtmosphere(tel)
    pupil = telescope_pupil(cfg.resolution)
    assert np.array_equal(tel.pupil.astype(bool), pupil)
    orc = AtmosphereOracle(cfg, pupil)
    assert rel_err(_np(atm._ops.A), orc.A) < 1e-8
    assert rel_err(_np(atm._ops.B), orc.B) < 1e-8
    M = atm._M
    for i, lo in enumerate(orc.layers):
        assert rel_err(_np(atm._layers[i].mapShift), lo.map) < 5e-6, f"layer {i} map after init"
    assert rel_err(_np(atm.OPD_no_pupil), orc.OPD_no_pupil) < 2e-6
    for k in range(40):                     # crosses several integer-pixel boundaries on both layers
        atm.update()
        orc.update()
    for i, (ly, lo) in enumerate(zip(atm._layers, orc.layers)):
        assert np.allclose(ly.buff, lo.buff, atol=1e-12)
        assert rel_err(_np(atm._layers[i].mapShift), lo.map) < 1e-5, f"layer {i} map after 40 updates"
    assert rel_err(_np(atm.OPD_no_pupil), orc.OPD_no_pupil) < 1e-5
    assert rel_err(_np(atm.OPD), orc.OPD) < 1e-5


def test_atmosphere_injected_innovations(dev):
    """xi-override hook: the oracle's recorded draws, fed back through xi_queue, reproduce its screens."""
    cfg, tel, src, atm = _tiny_objects(dev)
    atm.initializeAtmosphere(tel)
    orc = AtmosphereOracle(cfg, telescope_pupil(cfg.resolution))
    orc.xi_log.clear()
    for _ in range(25):
        orc.update()
    atm.xi_queue = iter([x[None, :] for x in orc.xi_log])
    for _ in range(25):
        atm.update()
    assert rel_err(_np(atm.OPD_no_pupil), orc.OPD_no_pupil) < 5e-6
    with pytest.raises(StopIteration):
        for _ in range(200):
            atm.update()


def test_sliding_window_canvas_vs_oracle(dev):
    """Fast wind + tiny canvas slack: the window is re-centred every second add_row, extrema are tracked across
    origin moves (rescans when the extremum pixel leaves the window); maps, extrema and OPD must follow the oracle."""
    from rlao_b200.Atmosphere import Atmosphere
    from rlao_b200.Source import Source
    from rlao_b200.Telescope import Telescope
    cfg = CONFIGS["tiny"]()
    cfg.windSpeed, cfg.windDirection = [33.0, 41.0], [30.0, 250.0]      # > 1 px/step, both axes, both signs
    tel = Telescope(cfg.resolution, cfg.diameter, cfg.samplingTime, n_envs=2, device=dev)
    Source(cfg.opticalBand, cfg.magnitude) * tel
    atm = Atmosphere(tel, cfg.r0, cfg.L0, cfg.windSpeed, cfg.fractionalR0, cfg.windDirection, cfg.altitude,
                     rng="reference", canvas_slack=2)
    atm.initializeAtmosphere(tel)
    orc = AtmosphereOracle(cfg, telescope_pupil(cfg.resolution))
    for k in range(30):
        atm.update()
        orc.update()
        if k % 7 == 0:
            assert rel_err(_np(atm.OPD_no_pupil[0]), orc.OPD_no_pupil) < 3e-5, k
    for i, lo in enumerate(orc.layers):
        got = _np(atm._layers[i].mapShift[0])
        assert rel_err(got, lo.map) < 3e-5
        ext = atm._ext[i, 0, 0].cpu().numpy().view(np.uint64)     # block 0: the whole window
        ext_in = atm._ext[i, 1, 0].cpu().numpy().view(np.uint64)  # block 1: its interior
        pitch, (oy, ox) = atm._pitch, atm._org[i]
        inner = np.full_like(got, np.nan)
        inner[1:-1, 1:-1] = got[1:-1, 1:-1]
        for packed, want in ((ext[0], got.min()), (ext[1], got.max()), (ext_in[0], np.nanmin(inner)), (ext_in[1], np.nanmax(inner))):
            pos = int(packed) & 0xffffffff
            r, c = pos // pitch - oy, pos % pitch - ox
            assert got[r, c] == want                             # tracked extremum is the true extremum, at its true position
    assert sum(ly.events for ly in atm._layers) > 8 * atm._S        # the canvases were re-centred many times


def test_tracked_extrema_stay_exact_through_wind_reversals(dev):
    """The clip range of every window (block 0 of the extrema array) and the extrema of its interior (block 1) against
    the canvas itself, after every frame, for 24 environments: diagonal wind, canvas re-centring every few events, and a
    reversal of the wind in mid-run (the ring kernel infers from the previous window origin which lines became interior;
    a wrong line would leave a stale interior extremum behind)."""
    from rlao_b200.Atmosphere import Atmosphere
    from rlao_b200.Source import Source
    from rlao_b200.Telescope import Telescope
    cfg = CONFIGS["tiny"]()
    cfg.windSpeed, cfg.windDirection = [70.0, 50.0], [30.0, 250.0]
    B = 24
    tel = Telescope(cfg.resolution, cfg.diameter, cfg.samplingTime, n_envs=B, device=dev)
    Source(cfg.opticalBand, cfg.magnitude) * tel
    atm = Atmosphere(tel, cfg.r0, cfg.L0, cfg.windSpeed, cfg.fractionalR0, cfg.windDirection, cfg.altitude,
                     rng="philox", canvas_slack=3)
    atm.initializeAtmosphere(tel)
    M, pitch = atm._M, atm._pitch
    rescans = 0
    for k in range(36):
        if k == 12:
            atm.windDirection = [210.0, 70.0]          # both layers turn around
        if k == 24:
            atm.windDirection = [90.0, 180.0]          # pure +y / pure -x
        atm.update()
        torch.cuda.synchronize()
        rescans += int(atm._flag.sum())
        for i in range(atm.nLayer):
            oy, ox = atm._org[i]
            win = atm._maps[i, atm._cur[i], :, oy:oy + M, ox:ox + M]
            ext = atm._ext[i].cpu().numpy().view(np.uint64)
            w = win.cpu().numpy()
            for b in range(B):
                inner = w[b, 1:-1, 1:-1]
                for blk, ref in ((0, w[b]), (1, inner)):
                    for e, want in ((ext[blk, b, 0], ref.min()), (ext[blk, b, 1], ref.max())):
                        pos = int(e) & 0xffffffff
                        r, c = pos // pitch - oy, pos % pitch - ox
                        assert 0 <= r < M and 0 <= c < M and w[b, r, c] == want, (k, i, b, blk)
                        if blk == 1:
                            assert 1 <= r <= M - 2 and 1 <= c <= M - 2, (k, i, b)
    assert sum(ly.events for ly in atm._layers) > 30 and rescans > 0


def test_layers_extruded_together_equal_layers_extruded_one_by_one(dev):
    """Counter-based innovations depend on (layer, event, environment) only: the grouped add_row (one gather / GEMM /
    ring for all layers of a round) must give bit-identical maps, extrema and OPD to the layer-by-layer sequence."""
    from rlao_b200.Atmosphere import Atmosphere
    from rlao_b200.Source import Source
    from rlao_b200.Telescope import Telescope
    cfg = CONFIGS["tiny"]()
    speeds, dirs, frac = [47.0, 21.0, 12.0, 33.0], [10.0, 130.0, 250.0, 300.0], [0.4, 0.3, 0.2, 0.1]

    def build():
        # nine environments: more rows than AOENV_SKINNY_MAX_ROWS, so the grouped and the single-layer products both run on
        # the tensor-core kernel (a product of <= 8 rows takes the exact-FP32 kernel and rounds differently)
        tel = Telescope(cfg.resolution, cfg.diameter, cfg.samplingTime, n_envs=9, device=dev)
        Source(cfg.opticalBand, cfg.magnitude) * tel
        atm = Atmosphere(tel, cfg.r0, cfg.L0, speeds, frac, dirs, [0.0] * 4, rng="philox", seed=5, canvas_slack=6)
        atm.initializeAtmosphere(tel)
        return atm
    a, b = build(), build()
    b.native_update = False                      # a: sequenced by aoenv_atm_update (grouped); b: by the Python methods, one layer at a time
    b._update_layers = lambda: [b._update_layer(i) for i in range(b.nLayer)]
    launches = []
    for k in range(25):
        l0 = _lib.launch_count()
        a.update()
        l1 = _lib.launch_count()
        b.update()
        launches.append((l1 - l0, _lib.launch_count() - l1))
        assert torch.equal(a.OPD_no_pupil, b.OPD_no_pupil), k
    for i in range(4):
        assert torch.equal(a._layers[i].mapShift, b._layers[i].mapShift)
        assert torch.equal(a._ext[i], b._ext[i])
    assert sum(x for x, _ in launches) < sum(y for _, y in launches)      # fewer launches when grouped


@pytest.mark.parametrize("kernel", ["lagrange018", "catmull_rom"])
def test_subpixel_shift_vs_warp_restatement(dev, kernel):
    cfg, tel, src, atm = _tiny_objects(dev)
    atm.warp_kernel = kernel
    atm.initializeAtmosphere(tel)
    M = atm._M
    ly = atm._layers[0]
    for buff in ([0.3, -0.6], [-0.999, 0.001], [0.0, 0.5], [0.75, 0.75]):
        for l2 in atm._layers:
            l2.buff = np.array(buff)
        atm._publish()
        want = 0
        for i in range(atm.nLayer):
            m = _np(atm._layers[i].mapShift)
            sh = warp_translate(m, buff[0], buff[1], kernel=kernel)[1:-1, 1:-1]
            c = sh.shape[0] // 2
            want = want + sh[c - cfg.resolution // 2:c + cfg.resolution // 2, c - cfg.resolution // 2:c + cfg.resolution // 2] * math.sqrt(cfg.fractionalR0[i])
        want = want * 500e-9 / 2 / np.pi
        assert rel_err(_np(atm.OPD_no_pupil), want) < 2e-6, buff


# ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("nS,n", [(8, 6), (5, 4), (4, 8), (20, 6)])
def test_shack_hartmann_vs_oracle(dev, nS, n):
    from rlao_b200.ShackHartmann import ShackHartmann
    from rlao_b200.Source import Source
    from rlao_b200.Telescope import Telescope
    cfg = AOConfig(nSubap=nS, nPixPerSubap=n)
    R = cfg.resolution
    tel = Telescope(R, cfg.diameter, cfg.samplingTime, n_envs=3, device=dev)
    src = Source(cfg.opticalBand, cfg.magnitude)
    src * tel
    wfs = ShackHartmann(nS, tel, cfg.lightRatio)
    pupil = telescope_pupil(R)
    wl, nph = source_properties(cfg.opticalBand, cfg.magnitude)
    orc = ShackHartmannOracle(cfg, pupil, flux_map(pupil, nph, cfg.samplingTime, cfg.diameter), wl)
    assert np.array_equal(wfs.valid_subapertures, orc.valid)
    assert rel_err(wfs.reference_slopes_maps, orc.reference_slopes_maps) < 1e-6
    assert rel_err(wfs.slopes_units, orc.slopes_units) < 2e-6
    wfs.slopes_units = orc.slopes_units          # identical inputs for the comparison below
    rs = np.random.RandomState(5)
    yy, xx = np.mgrid[:R, :R] / R
    opds = []
    for e in range(3):
        c = rs.normal(size=6)
        opd = 0.4e-6 * (c[0] * xx + c[1] * yy + c[2] * np.sin(7 * xx + 3 * yy) + c[3] * np.cos(11 * yy) * xx
                        + 0.3 * c[4] * np.sin(23 * xx * yy)) + 0.05e-6 * rs.normal(size=(R, R))
        opds.append(opd)
    tel.OPD_no_pupil = torch.as_tensor(np.stack(opds), dtype=torch.float32, device=dev)
    tel * wfs
    got_sig, got_frame = _np(wfs.signal), _np(wfs.cam.frame)
    opd32 = _np(tel.OPD_no_pupil)
    for e in range(3):
        want = orc.measure(opd32[e] * pupil * 2 * np.pi / wl)
        assert rel_err(got_frame[e], orc.frame) < 2e-5, (e, "frame")
        assert rel_err(got_sig[e], want) < SLOPE_TOL, (e, "slopes")
    s2d = _np(wfs.signal_2D)
    assert rel_err(s2d[2], orc.signal_2D) < SLOPE_TOL
    # every implementation of the frame kernel gives the same frame as the default one: 3 = term by term on n/2 lanes per
    # lenslet (any n); for 6-pixel lenslets also 1 = factorised (radix 2 x Good-Thomas 2 x 3) on one thread per lenslet and
    # 2 = factorised on three lanes per lenslet; 0 = term by term, one thread per lenslet
    lib = _lib.load()
    wfs.use_fused = False
    tel * wfs
    got_sig, got_frame = _np(wfs.signal), _np(wfs.cam.frame)
    default = lib.aoenv_set_wfs6_variant(-1)
    lib.aoenv_set_wfs6_variant(default)
    for variant in ((0, 1, 2, 3) if n == 6 else (0, 3)):
        prev = lib.aoenv_set_wfs6_variant(variant)
        try:
            tel * wfs
            alt_sig, alt_frame = _np(wfs.signal), _np(wfs.cam.frame)
        finally:
            lib.aoenv_set_wfs6_variant(prev)
        assert rel_err(alt_frame, got_frame) < 5e-6, variant
        assert rel_err(alt_sig, got_sig) < 2e-5, variant
        for e in range(3):
            orc.measure(opd32[e] * pupil * 2 * np.pi / wl)
            assert rel_err(alt_frame[e], orc.frame) < 2e-5, (e, "frame", variant)


def test_shack_hartmann_flat_wavefront_gives_zero_signal_at_full_size(dev):
    from rlao_b200.ShackHartmann import ShackHartmann
    from rlao_b200.Source import Source
    from rlao_b200.Telescope import Telescope
    tel = Telescope(240, 8, 1 / 500, n_envs=5, device=dev)
    src = Source("I", 8)
    src * tel
    wfs = ShackHartmann(40, tel, 0.5)
    assert wfs.nValidSubaperture == 1264 and wfs.nSignal == 2528       # SURVEY.md section 8 size table
    tel.resetOPD()
    tel * wfs
    assert float(wfs.signal.abs().max()) < 1e-5
    # piston invariance: a constant OPD changes nothing
    tel.OPD_no_pupil = torch.full((5, 240, 240), 3e-7, device=dev)
    tel * wfs
    assert float(wfs.signal.abs().max()) < 1e-4


# ---------------------------------------------------------------------------------------------------------
def test_dm_surface_vs_oracle_and_linearity(dev):
    from rlao_b200.DeformableMirror import DeformableMirror
    from rlao_b200.Source import Source
    from rlao_b200.Telescope import Telescope
    cfg = CONFIGS["cfg1"]()
    tel = Telescope(cfg.resolution, cfg.diameter, cfg.samplingTime, n_envs=4, device=dev)
    Source("I", 8) * tel
    dm = DeformableMirror(tel, cfg.nSubap, cfg.mechCoupling)
    xIF, yIF, mask, sigma = dm_geometry(cfg)
    modes, _, _ = dm_modes(cfg, xIF, yIF, sigma)
    assert dm.nValidAct == 357 == modes.shape[1]                         # pinned by manual_m2c.npy (SURVEY section 4)
    assert np.array_equal(dm.validAct.reshape(21, 21), mask)
    assert rel_err(_np(dm.modes), modes) < 1e-12
    rs = np.random.RandomState(1)
    c = rs.normal(size=(4, 357)) * 1e-7
    dm.coefs = torch.as_tensor(c, dtype=torch.float32, device=dev)
    want = (modes @ _np(dm.coefs).T).T.reshape(4, cfg.resolution, cfg.resolution)
    assert dm._sep is not None                                            # default geometry -> separable kernel
    assert rel_err(_np(dm.OPD), want) < 2e-6
    dm.surface_backend = "gemm"                                           # dense tcgen05 contraction of the same thing
    dm.coefs = torch.as_tensor(c, dtype=torch.float32, device=dev)
    assert rel_err(_np(dm.OPD), want) < SURFACE_TOL
    dm.surface_backend = "auto"
    dm.coefs = torch.as_tensor(c, dtype=torch.float32, device=dev)
    a = _np(dm.OPD).copy()
    dm.coefs = torch.as_tensor(2 * c, dtype=torch.float32, device=dev)
    assert rel_err(_np(dm.OPD), 2 * a) < 1e-6                            # linearity
    dm.coefs = 0
    assert float(dm.OPD.abs().max()) == 0.0
    # reference [nValidAct, k] matrix mode (calibration pushes)
    dm.coefs = torch.eye(357, dtype=torch.float32, device=dev)[:, :7] * 1e-9
    assert dm.OPD.shape == (7, cfg.resolution, cfg.resolution)
    assert rel_err(_np(dm.OPD[3]).reshape(-1), modes[:, 3] * 1e-9) < SURFACE_TOL


# ---------------------------------------------------------------------------------------------------------
def _trace(name, dev, steps=None):
    cfg = CONFIGS[name]()
    gold = load_golden(name)
    env = build_env(cfg, n_envs=1, rng="reference", device=dev)
    orc = EnvOracle(cfg)
    return cfg, gold, env, orc


def _knife_edge_lenslets(orc, margin=1e-4):
    """Valid lenslets of the oracle's last measurement having a pixel within `margin` (relative) of the centroiding
    threshold 0.01 * max: the float32 path may legitimately flip such a pixel (SURVEY.md section 7, hard parts)."""
    maps = orc.wfs.maps_intensity
    return knife_edge_lenslets(maps, orc.wfs.threshold_cog * maps.max(), margin)


@pytest.mark.parametrize("name", ["tiny", "cfg1", "cfg3"])
def test_closed_loop_trace_vs_reference_golden(dev, name):
    """Closed-loop trace recorded from the UNMODIFIED reference (tests/golden/<name>.npz).  Every step is driven with
    the reference's own action (gainCL * its observation), so each step sees identical inputs; the oracle runs in
    lock-step (and must reproduce the golden trace) to expose the camera frame of every step."""
    cfg, gold, env, orc = _trace(name, dev)
    assert np.array_equal(env.wfs.valid_subapertures, gold["valid_subapertures"])
    assert np.array_equal(env.dm_mask.astype(bool), gold["validAct"].astype(bool))
    assert rel_err(env.wfs.slopes_units, gold["slopes_units"]) < 2e-6
    assert rel_err(env.wfs.reference_slopes_maps, gold["reference_slopes_maps"]) < 1e-6
    # our GPU-calibrated reconstructor (float64 WFS kernels on float32 DM surfaces) vs the reference's
    assert rel_err(_np(env.reconstructor), orc.reconstructor) < 2e-4
    env.set_reconstructor(orc.reconstructor)          # identical inputs from here on
    env.wfs.slopes_units = float(gold["slopes_units"])
    n, nV = STEPS[name], env.wfs.nValidSubaperture
    obs = new_episode(env, EPISODE_SEED)
    orc.new_episode(EPISODE_SEED)
    assert rel_err(_np(obs), gold["obs0"]) < 2e-4
    assert rel_err(_np(env.wfs.signal), gold["signal0"]) < SLOPE_TOL
    snap = set(int(s) for s in gold["snap_steps"])
    obs_ref = gold["obs0"]
    clean_steps = 0
    for i in range(n):
        action = cfg.gainCL * obs_ref
        obs, reward, strehl, done, info = env.step(i, torch.as_tensor(action, dtype=torch.float32, device=dev))
        orc.step(i, action)
        obs_ref = gold["trace_obs"][i]
        # the oracle IS the reference here (the large fixture stores float32 traces)
        assert rel_err(orc.wfs.signal, gold["trace_signal"][i]) < (1e-7 if gold["trace_signal"].dtype == np.float64 else 3e-7)
        assert rel_err(_np(env.dm.coefs), gold["trace_coefs"][i]) < 1e-6, (i, "coefs")
        assert rel_err(_np(env.wfs.cam.frame), orc.wfs.frame) < 2e-4, (i, "frame")
        assert abs(float(strehl) - gold["trace_strehl"][i]) <= STREHL_TOL * gold["trace_strehl"][i] + 1e-30, (i, "strehl")
        edge = _knife_edge_lenslets(orc)
        keep = np.concatenate([~edge, ~edge])
        assert edge.sum() <= max(2, 0.02 * nV), (i, "too many knife-edge lenslets", int(edge.sum()))
        sig, sig_ref = _np(env.wfs.signal), gold["trace_signal"][i]
        assert np.abs(sig - sig_ref)[keep].max() < 2 * SLOPE_TOL * np.abs(sig_ref).max(), (i, "slopes")
        if not edge.any():
            clean_steps += 1
            # obs is the reconstructed RESIDUAL: once the loop has converged it is ~10x smaller than the DM surface
            # that cancels the turbulence, so surface errors of 1e-5 (relative) show up here at the 1e-4 level
            assert rel_err(_np(obs), gold["trace_obs"][i]) < 1e-3, (i, "obs")
            assert abs(float(reward) - gold["trace_reward"][i]) <= 1e-3 * abs(gold["trace_reward"][i]), (i, "reward")
        else:
            # a flipped threshold pixel moves one lenslet's centroid; its weight in the reconstruction is ~1/nV
            assert rel_err(_np(obs), gold["trace_obs"][i]) < 1e-2, (i, "obs, knife-edge step")
        if i in snap:
            assert rel_err(_np(env.atm.OPD), gold[f"atm_OPD_{i}"]) < 3e-5
            assert rel_err(_np(env.tel.OPD), gold[f"tel_OPD_{i}"]) < SURFACE_TOL
    # with 1264 lenslets x 36 pixels nearly every frame has some pixel within 1e-4 of the threshold
    assert clean_steps >= n // 2 or nV > 1000
    assert rel_err(_np(env.total[:n, 0]), gold["trace_total"]) < 1e-4
    assert rel_err(_np(env.residual[:n, 0]), gold["trace_residual"]) < 1e-3
    assert done is False and "strehl" in info


def test_closed_loop_own_policy_tracks_reference(dev):
    """Free-running loop (the GPU path feeds its own observations back): Strehl and residual stay on the reference's
    trajectory; slopes agree to the tolerance until a knife-edge pixel flips, and to 5 % afterwards."""
    cfg, gold, env, orc = _trace("cfg1", dev)
    env.set_reconstructor(orc.reconstructor)
    n = STEPS["cfg1"]
    obs = new_episode(env, EPISODE_SEED)
    for i in range(n):
        obs, reward, strehl, done, info = env.step(i, cfg.gainCL * obs)
        assert rel_err(_np(env.wfs.signal), gold["trace_signal"][i]) < 5e-2, i
        assert abs(float(strehl) - gold["trace_strehl"][i]) <= 0.02 * gold["trace_strehl"][i] + 1e-30, i
    assert rel_err(_np(env.residual[:n, 0]), gold["trace_residual"]) < 5e-3


def test_dm_with_rotation_uses_the_dense_contraction(dev):
    from rlao_b200.DeformableMirror import DeformableMirror
    from rlao_b200.MisRegistration import MisRegistration
    from rlao_b200.Source import Source
    from rlao_b200.Telescope import Telescope
    tel = Telescope(48, 8, 1 / 500, n_envs=2, device=dev)
    Source("I", 8) * tel
    mis = MisRegistration()
    mis.rotationAngle, mis.shiftX = 3.0, 0.05
    dm = DeformableMirror(tel, 8, 0.35, misReg=mis)
    assert dm._sep is None
    c = torch.randn(2, dm.nValidAct, device=dev) * 1e-7
    dm.coefs = c
    want = (_np(dm.modes) @ _np(c).T).T.reshape(2, 48, 48)
    assert rel_err(_np(dm.OPD), want) < SURFACE_TOL
    shifted = MisRegistration()
    shifted.shiftX, shifted.shiftY, shifted.radialScaling = 0.07, -0.02, 0.01
    dm2 = DeformableMirror(tel, 8, 0.35, misReg=shifted)
    assert dm2._sep is not None                                           # shifts / scalings keep it separable
    dm2.coefs = c[:, :dm2.nValidAct]
    want2 = (_np(dm2.modes) @ _np(c[:, :dm2.nValidAct]).T).T.reshape(2, 48, 48)
    assert rel_err(_np(dm2.OPD), want2) < 2e-6


def test_interaction_matrix_vs_oracle(dev):
    cfg, gold, env, orc = _trace("tiny", dev)
    D = _np(env.calib_zonal.D)
    assert D.shape == orc.D_zonal.shape
    assert rel_err(D, orc.D_zonal) < 1e-5
    # SVD bookkeeping of CalibrationVault
    c = env.calib_CL
    assert rel_err(_np(c.M @ c.D), np.eye(c.D.shape[1])) < 1e-6


# ---------------------------------------------------------------------------------------------------------
def test_psf_peak_vs_oracle(dev):
    from rlao_b200.psf import psf_peak
    cfg, tel, src, atm = _tiny_objects(dev, n_envs=2)
    atm.initializeAtmosphere(tel)
    tel + atm
    pupil = telescope_pupil(cfg.resolution)
    wl, nph = source_properties(cfg.opticalBand, cfg.magnitude)
    fm = flux_map(pupil, nph, cfg.samplingTime, cfg.diameter)
    # well-corrected wavefront: scale the turbulence down so that the peak sits in the core
    opd = atm._opd * 0.05
    peak, win = psf_peak(tel, opd.contiguous(), None, 4, 16, return_window=True)
    for e in range(2):
        psf = compute_psf(pupil, fm, _np(opd[e]) * pupil * 2 * np.pi / wl, 4)
        c = psf.shape[0] // 2
        assert rel_err(_np(win[e]), psf[c - 8:c + 8, c - 8:c + 8]) < 2e-5
        assert abs(float(peak[e]) - psf.max()) < 2e-5 * psf.max()
    # against the full-image torch.fft path of Telescope.computePSF and the golden reference value
    gold = np.load(os.path.join(os.path.dirname(__file__), "golden", "tiny.npz"))
    ph = torch.as_tensor(gold["psf_atm_phase"], dtype=torch.float32, device=dev)
    tel.OPD_no_pupil = (ph * (wl / 2 / np.pi)).unsqueeze(0).expand(2, -1, -1)
    tel.computePSF(4)
    cc = tel.PSF.shape[-1] // 2
    assert rel_err(_np(tel.PSF[0, cc - 8:cc + 8, cc - 8:cc + 8]), gold["psf_atm_crop"]) < 1e-4
    assert abs(float(tel.PSF[0].max()) - gold["psf_atm_max"]) < 1e-4 * gold["psf_atm_max"]


# ---------------------------------------------------------------------------------------------------------
def test_detector_noise_statistics(dev):
    """Noisy WFS frames: Poisson photon noise (variance = mean), rounded Gaussian read noise, dark current, QE,
    full-well clipping and ADC quantisation follow OOPAO/Detector.py:190-301 statistically; streams are independent
    across environments and steps (Philox counters)."""
    from rlao_b200.ShackHartmann import ShackHartmann
    from rlao_b200.Source import Source
    from rlao_b200.Telescope import Telescope
    B = 256
    tel = Telescope(48, 8, 1 / 500, n_envs=B, device=dev)
    src = Source("I", 10)
    src * tel
    wfs = ShackHartmann(8, tel, 0.5)
    tel.resetOPD()
    tel * wfs
    ideal = _np(wfs.cam.frame[0])
    lit = ideal > 0.02 * ideal.max()
    # (1) photon noise only
    wfs.cam.photonNoise = True
    tel * wfs
    f1 = _np(wfs.cam.frame)
    tel * wfs
    f2 = _np(wfs.cam.frame)
    assert np.all(f1 == np.round(f1)) and f1.min() >= 0
    mean, var = f1.mean(axis=0), f1.var(axis=0)
    assert abs(mean[lit].mean() / ideal[lit].mean() - 1) < 0.01
    assert abs((var[lit] / mean[lit]).mean() - 1) < 0.05              # index of dispersion 1
    d01 = (f1[0] - ideal)[lit], (f1[1] - ideal)[lit]
    assert abs(np.corrcoef(*d01)[0, 1]) < 0.1                         # independent across environments
    dt = (f1 - ideal)[:, lit].reshape(-1), (f2 - ideal)[:, lit].reshape(-1)
    assert abs(np.corrcoef(*dt)[0, 1]) < 0.02                         # independent across steps
    # (2) read noise only: round(N(0,1)*RON)
    wfs.cam.photonNoise = False
    wfs.cam.readoutNoise = 14
    tel * wfs
    r = _np(wfs.cam.frame) - ideal
    dark_px = ~lit
    assert abs(r[:, dark_px].std() - 14) < 0.3 and abs(r[:, dark_px].mean()) < 0.2
    resid = _np(wfs.cam.frame)[:, dark_px] - ideal[dark_px]
    assert np.abs(resid - np.round(resid)).max() < 1e-3
    # (3) Razor-like camera: QE, dark current, full well, 10-bit ADC
    wfs.cam.photonNoise, wfs.cam.readoutNoise = True, 0
    wfs.cam.QE, wfs.cam.FWC, wfs.cam.bits, wfs.cam.darkCurrent, wfs.cam.sensor = 0.56, 10000, 10, 5000.0, "CMOS"
    wfs.cam.integrationTime = 1 / 500
    tel * wfs
    q = _np(wfs.cam.frame)
    assert np.all(q == np.round(q)) and q.min() >= 0 and q.max() <= 1023
    expect = np.clip(ideal * 0.56 + 10.0, 0, 10000) / 10000 * 1023
    unsat = lit & (ideal * 0.56 < 8000)
    assert abs((q.mean(axis=0)[unsat] + 0.5).mean() / expect[unsat].mean() - 1) < 0.02
    assert abs(q[:, dark_px].mean() - (10.0 / 10000 * 1023 - 0.5)) < 0.15


def test_poisson_sampler_matches_the_poisson_pmf(dev):
    """Photon-noise draws against scipy's Poisson pmf, pixel by pixel, across the regimes of the sampler (sequential
    inversion below 12, PTRS transformed rejection above, OOPAO/Detector.py:190-206 -> numpy's legacy poisson)."""
    from scipy import stats
    from rlao_b200.ShackHartmann import ShackHartmann
    from rlao_b200.Source import Source
    from rlao_b200.Telescope import Telescope
    B, K = 512, 8
    checked = []
    for mag in (5.0, 9.0, 12.5):
        tel = Telescope(48, 8, 1 / 500, n_envs=B, device=dev)
        Source("I", mag) * tel
        wfs = ShackHartmann(8, tel, 0.5)
        tel.resetOPD()
        tel * wfs
        ideal = _np(wfs.cam.frame[0]).astype(np.float64)
        wfs.cam.photonNoise = True
        draws = []
        for _ in range(K):
            tel * wfs
            draws.append(_np(wfs.cam.frame))
        x = np.concatenate(draws, axis=0).astype(np.int64)              # [K*B, R, R]
        # one pixel per decade of flux present in this frame (+ the two sides of the algorithm switch at 12)
        targets = [0.3, 3.0, 11.0, 13.0, 15.0, 18.0, 40.0, 400.0, 1500.0, 4000.0, 12000.0, 40000.0]
        flat = ideal.reshape(-1)
        for tgt in targets:
            j = int(np.argmin(np.abs(np.log(np.maximum(flat, 1e-9) / tgt))))
            lam = flat[j]
            if not (0.75 * tgt < lam < 1.33 * tgt) or any(abs(lam - c) < 1e-6 * lam for c in checked):
                continue
            s = x.reshape(x.shape[0], -1)[:, j]
            lo, hi = int(stats.poisson.ppf(1e-4, lam)), int(stats.poisson.ppf(1 - 1e-4, lam))
            edges = np.unique(np.round(np.linspace(lo, hi + 1, 24)).astype(int))
            cdf = stats.poisson.cdf(edges - 1, lam)
            p = np.diff(np.concatenate([[0.0], cdf, [1.0]]))                 # (-inf, e0), [e0, e1), ..., [e_last, inf)
            obs = np.histogram(s, bins=np.concatenate([[-1], edges, [10 ** 9]]))[0]
            keep = p * s.size >= 5
            chi2 = (((obs[keep] - p[keep] * s.size) ** 2) / (p[keep] * s.size)).sum()
            pval = stats.chi2.sf(chi2, int(keep.sum()) - 1)
            assert pval > 1e-4, (mag, lam, chi2, pval)
            assert abs(s.mean() - lam) < 5 * np.sqrt(lam / s.size) + 1e-3 * lam, (mag, lam, s.mean())
            checked.append(lam)
    assert min(checked) < 1.0 and max(checked) > 1000 and any(8 < c < 12 for c in checked) and any(12 < c < 20 for c in checked)


def test_dark_current_draws_follow_the_poisson_pmf(dev):
    """Dark-current shot noise (OOPAO/Detector.py:232-238) alone and on top of bright pixels: the draw comes from the
    fifth word of the pixel's Philox block (means below 12) or from block 1 (PTRS, means >= 12); it must be Poisson,
    independent of the photon draw of the same pixel, and survive the trip through the warp queue of the bright pixels."""
    from scipy import stats
    from rlao_b200.ShackHartmann import ShackHartmann
    from rlao_b200.Source import Source
    from rlao_b200.Telescope import Telescope
    B = 512
    tel = Telescope(48, 8, 1 / 500, n_envs=B, device=dev)
    Source("I", 8) * tel
    wfs = ShackHartmann(8, tel, 0.5)
    tel.resetOPD()
    tel * wfs
    ideal = _np(wfs.cam.frame[0]).astype(np.float64)
    wfs.cam.integrationTime = 1 / 500
    for d in (0.05, 3.0, 20.0):
        wfs.cam.photonNoise, wfs.cam.darkCurrent = False, d * 500
        tel * wfs
        x = _np(wfs.cam.frame).astype(np.float64) - ideal
        assert np.abs(x - np.round(x)).max() < 2e-3 * max(1.0, ideal.max() * 1e-4) and x.min() > -0.5
        x = np.round(x).reshape(-1)
        assert abs(x.mean() - d) < 5 * np.sqrt(d / x.size), (d, x.mean())
        assert abs(x.var() / d - 1) < 5 * np.sqrt((2 + 1 / d) / x.size), (d, x.var())
        ks = np.arange(0, int(stats.poisson.ppf(1 - 1e-6, d)) + 1)
        p = stats.poisson.pmf(ks, d)
        obs = np.bincount(x.astype(np.int64), minlength=ks.size)[:ks.size]
        keep = p * x.size >= 5
        chi2 = (((obs[keep] - p[keep] * x.size) ** 2) / (p[keep] * x.size)).sum()
        assert stats.chi2.sf(chi2, int(keep.sum()) - 1) > 1e-4, (d, chi2)
    # with photon noise: mean and variance add, and the two draws of a pixel are uncorrelated (bright = queued pixels)
    wfs.cam.photonNoise, wfs.cam.darkCurrent = True, 3.0 * 500
    tel * wfs
    y = _np(wfs.cam.frame).astype(np.float64)
    assert (ideal > 100.0).sum() > 50
    for sel in (ideal > 100.0, (ideal > 0.5) & (ideal < 10.0)):
        if sel.sum() < 50:
            continue
        m, v = y.mean(axis=0)[sel], y.var(axis=0)[sel]
        assert abs((m - ideal[sel]).mean() - 3.0) < 0.05 * np.sqrt(ideal[sel].mean() + 3.0) + 0.05
        assert abs((v / (ideal[sel] + 3.0)).mean() - 1) < 0.05


def test_extruded_screens_keep_the_von_karman_structure_function(dev):
    """After the window has been regenerated several times over by add_row (float32 maps, split-bf16 tensor-core GEMM for
    X = A Z + B xi), the phase structure function of the maps must still be the von Karman one the operators were
    built for (OOPAO/phaseStats.py:70-133): D(r) = 2 (C(0) - C(r))."""
    from oracle.ao_oracle import vk_covariance_matrix
    from rlao_b200.Atmosphere import Atmosphere
    from rlao_b200.Source import Source
    from rlao_b200.Telescope import Telescope
    R, D, L0, r0, B = 48, 8.0, 25.0, 0.13, 512
    tel = Telescope(R, D, 1 / 500, n_envs=B, device=dev)
    Source("I", 8) * tel
    atm = Atmosphere(tel, r0, L0, [45.0], [1.0], [35.0], [0.0], rng="philox", seed=11)
    atm.initializeAtmosphere(tel)
    ps = atm.ps_loop
    steps = int(4 * atm._M / (45.0 / 500 / ps)) + 1           # the wind carries four window widths of fresh screen in
    for _ in range(steps):
        atm.update()
    m = atm._layers[0].mapShift.double()                       # [B, M, M] radians at 500 nm
    assert torch.isfinite(m).all()
    for sep in (1, 3, 8, 20):
        want = 2 * (vk_covariance_matrix(np.array([0j]), np.array([0j]), L0, r0)[0, 0]
                    - vk_covariance_matrix(np.array([0j]), np.array([sep * ps + 0j]), L0, r0)[0, 0])
        dx = float(((m[:, :, sep:] - m[:, :, :-sep]) ** 2).mean())
        dy = float(((m[:, sep:, :] - m[:, :-sep, :]) ** 2).mean())
        tol = 0.04 if sep <= 8 else 0.08
        assert abs(dx / want - 1) < tol and abs(dy / want - 1) < tol, (sep, dx / want, dy / want)
