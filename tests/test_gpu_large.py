"""Parity at the sizes of BASELINE.json configs[3] and [4] (SURVEY.md section 8 d: cfg4 = 20 x 20 / 4096 environments with
the noisy camera; cfg5 = 80 x 80 SH, 81 x 81 DM, five layers, PSF-Strehl reward): kernels on injected inputs against the
oracle, the shapes of the large contractions against float64, and the closed-loop trace recorded from the unmodified
reference at 80 x 80 (tests/golden/cfg5.npz, oracle/make_golden.py)."""
import math
import os

import numpy as np
import pytest
import torch

from oracle.ao_oracle import (AOConfig, ShackHartmannOracle, compute_psf, dm_geometry, dm_modes, flux_map, source_properties,
                              telescope_pupil)
from oracle.golden_configs import CONFIGS, EPISODE_SEED, STEPS, psf_formula_opd
from oracle.make_golden import load as load_golden
from oracle.warp018 import warp_translate
from parity_util import build_env, new_episode, rel_err
from rlao_b200 import _lib

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden", "cfg5.npz")


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    return torch.device("cuda:0")


def _np(t):
    return t.detach().double().cpu().numpy()


# ---- 80 x 80 wavefront sensor and DM on injected inputs -----------------------------------------------------------
def test_wfs_and_dm_at_80x80_vs_oracle(dev):
    from rlao_b200.DeformableMirror import DeformableMirror
    from rlao_b200.ShackHartmann import ShackHartmann
    from rlao_b200.Source import Source
    from rlao_b200.Telescope import Telescope
    cfg = AOConfig(nSubap=80)
    R, B = cfg.resolution, 2
    tel = Telescope(R, cfg.diameter, cfg.samplingTime, n_envs=B, device=dev)
    Source(cfg.opticalBand, cfg.magnitude) * tel
    wfs = ShackHartmann(80, tel, cfg.lightRatio)
    dm = DeformableMirror(tel, 80, cfg.mechCoupling)
    assert (wfs.nValidSubaperture, wfs.nSignal, dm.nValidAct) == (5024, 10048, 5209)          # SURVEY.md section 8 size table
    pupil = telescope_pupil(R)
    wl, nph = source_properties(cfg.opticalBand, cfg.magnitude)
    orc = ShackHartmannOracle(cfg, pupil, flux_map(pupil, nph, cfg.samplingTime, cfg.diameter), wl)
    assert np.array_equal(wfs.valid_subapertures, orc.valid)
    assert rel_err(wfs.slopes_units, orc.slopes_units) < 2e-6
    rs = np.random.RandomState(8)
    yy, xx = np.mgrid[:R, :R] / R
    opd = np.stack([0.5e-6 * (c[0] * xx + c[1] * yy + c[2] * np.sin(9 * xx + 4 * yy) + 0.3 * c[3] * np.cos(31 * xx * yy))
                    + 0.04e-6 * rs.normal(size=(R, R)) for c in rs.normal(size=(B, 4))])
    coefs = rs.normal(size=(B, dm.nValidAct)) * 1e-7
    dm.coefs = torch.as_tensor(coefs, dtype=torch.float32, device=dev)
    # DM surface (separable kernel; evaluated inside the fused kernel below) vs the float64 influence matrix, one column
    # block at a time (the dense matrix is 9.6 GB)
    xIF, yIF, mask, sigma = dm_geometry(cfg)
    g = np.linspace(0, 1, R) * R
    u0x, u0y = R / 2 + xIF * R / cfg.diameter, R / 2 + yIF * R / cfg.diameter
    gx = np.exp(-((g[None, :] - u0x[:, None]) ** 2) / (2 * sigma ** 2))        # [nA, R] along columns
    gy = np.exp(-((g[None, :] - u0y[:, None]) ** 2) / (2 * sigma ** 2))        # [nA, R] along rows
    want_surf = np.stack([(gy.T * c) @ gx for c in _np(dm.coefs)])              # sum_k c_k gy_k(y) gx_k(x)
    surf = _np(dm.OPD)
    assert rel_err(surf, want_surf) < 2e-6
    a = torch.as_tensor(opd, dtype=torch.float32, device=dev).contiguous()
    total = _np(a) + surf
    for mode in ("kernels", "fused"):
        if mode == "fused":                       # opt-in cluster kernel: DM surface + spots + slopes in one launch
            wfs.use_fused, wfs.keep_frame, dm.lazy_surface = True, True, True
            dm.coefs = torch.as_tensor(coefs, dtype=torch.float32, device=dev)
        wfs._measure_terms(a, dm.surface_ref(), 0)
        if mode == "fused":
            plan = wfs._fused_plans[id(dm.fused_tables())]
            assert plan["cluster"] >= 8 and plan["rows"][-1] == 80       # strips of at most ~10 lenslet rows fit in shared memory
        sig, frame = _np(wfs.signal), _np(wfs.cam.frame)
        for e in range(B):
            want = orc.measure(total[e] * pupil * 2 * np.pi / wl) * orc.slopes_units / wfs.slopes_units
            assert rel_err(frame[e], orc.frame) < 2e-5, (mode, e, "frame")
            assert rel_err(sig[e], want) < 1e-4, (mode, e, "slopes")


def test_atmosphere_phase_at_480px_five_layers_vs_warp_restatement(dev):
    from rlao_b200.Atmosphere import Atmosphere
    from rlao_b200.Source import Source
    from rlao_b200.Telescope import Telescope
    cfg = CONFIGS["cfg5"]()
    R = cfg.resolution
    tel = Telescope(R, cfg.diameter, cfg.samplingTime, n_envs=2, device=dev)
    Source(cfg.opticalBand, cfg.magnitude) * tel
    atm = Atmosphere(tel, cfg.r0, cfg.L0, cfg.windSpeed, cfg.fractionalR0, cfg.windDirection, cfg.altitude, rng="philox", seed=3)
    atm.initializeAtmosphere(tel)
    assert (atm._nO, atm._nI, atm._M) == (1940, 3856, 486)                      # SURVEY.md section 8 size table
    for _ in range(3):                                                          # a few add_row events on every layer
        atm.update()
    buffs = [[0.3, -0.6], [-0.999, 0.001], [0.0, 0.5], [0.75, 0.75], [-0.2, 0.9]]
    for i, ly in enumerate(atm._layers):
        ly.buff = np.array(buffs[i])
    atm._publish()
    want = 0
    for i in range(atm.nLayer):
        m = _np(atm._layers[i].mapShift[0])
        sh = warp_translate(m, buffs[i][0], buffs[i][1], kernel="lagrange018")[1:-1, 1:-1]
        c = sh.shape[0] // 2
        want = want + sh[c - R // 2:c + R // 2, c - R // 2:c + R // 2] * math.sqrt(cfg.fractionalR0[i])
    want = want * 500e-9 / 2 / np.pi
    assert rel_err(_np(atm.OPD_no_pupil[0]), want) < 2e-6


@pytest.mark.parametrize("M,N,K,parts", [(256, 5209, 10048, 2), (1280, 1940, 5796, 3)])
def test_large_contraction_shapes_vs_float64(dev, M, N, K, parts):
    """The reconstruction [5209 x 10048] and the add_row operator [1940 x (3856 + 1940)] of the 80 x 80 system."""
    from rlao_b200 import gemm
    Kp = (K + 15) // 16 * 16
    g = torch.Generator(device=dev).manual_seed(K)
    X, W = torch.zeros(M, Kp, device=dev), torch.zeros(N, Kp, device=dev)
    X[:, :K] = torch.randn(M, K, device=dev, generator=g)
    W[:, :K] = torch.randn(N, K, device=dev, generator=g)
    op = gemm.Operator(W, parts=parts)
    ldd = (N + 3) // 4 * 4
    D = torch.full((M, ldd), float("nan"), device=dev)
    gemm.gemm_tn(X, op, D, M, N, backend="tc")
    ref = X.double() @ W.double().T
    mag = X.double().abs() @ W.double().abs().T
    err = ((D[:, :N].double() - ref).abs() / mag).max().item()
    assert err < (2.0 ** -16 if parts == 2 else 2.0 ** -18)
    assert torch.isnan(D[:, N:]).all()
    # 160 output tiles on 148 SMs run in stream-K order (tiles shared by two CTAs, float atomics on a zeroed D): two
    # addends commute, so a second run must reproduce every bit
    D2 = torch.full((M, ldd), float("nan"), device=dev)
    gemm.gemm_tn(X, op, D2, M, N, backend="tc")
    assert torch.equal(D[:, :N], D2[:, :N])


def test_psf_peak_at_480px_zero_padding_4(dev):
    """Science-PSF Strehl of the 80 x 80 configuration (R 480, zero padding 4 -> N 3840 with oversampling 2): the
    pruned-DFT kernels against the full-image oracle and, when the fixture is there, against the reference's computePSF."""
    from rlao_b200.psf import psf_peak
    from rlao_b200.Source import Source
    from rlao_b200.Telescope import Telescope
    cfg = CONFIGS["cfg5"]()
    R = cfg.resolution
    tel = Telescope(R, cfg.diameter, cfg.samplingTime, n_envs=2, device=dev)
    Source(cfg.opticalBand, cfg.magnitude) * tel
    pupil = telescope_pupil(R)
    wl, nph = source_properties(cfg.opticalBand, cfg.magnitude)
    fm = flux_map(pupil, nph, cfg.samplingTime, cfg.diameter)
    opd = psf_formula_opd(R)
    both = torch.as_tensor(np.stack([opd, 0.5 * opd]), dtype=torch.float32, device=dev).contiguous()
    peak, win = psf_peak(tel, both, None, 4, 32, return_window=True)
    for e, scale in enumerate((1.0, 0.5)):
        psf = compute_psf(pupil, fm, scale * opd * pupil * 2 * np.pi / wl, 4)
        c = psf.shape[0] // 2
        assert rel_err(_np(win[e]), psf[c - 16:c + 16, c - 16:c + 16]) < 2e-5
        assert abs(float(peak[e]) - psf.max()) < 2e-5 * psf.max()
    if os.path.exists(GOLD):
        gold = np.load(GOLD)
        assert rel_err(_np(win[0]), gold["psf_formula_win"]) < 1e-4
        assert abs(float(peak[0]) - gold["psf_formula_max"]) < 1e-4 * gold["psf_formula_max"]


# ---- cfg4: 20 x 20, 4096 environments, noisy camera at low flux ----------------------------------------------------
def test_detector_statistics_at_cfg4_size_low_flux(dev):
    """4096 environments of the 20 x 20 system, magnitude 12, Razor-like camera (photon noise, RON 14 e-, QE 0.56, dark
    5 e-/px/s, FWC 1e4, 10 bit): per-pixel mean / variance across environments against the analytic chain, quantisation,
    independence across environments, frames and shards, and the noisy slopes centred on the noise-free ones."""
    from rlao_b200.ShackHartmann import ShackHartmann
    from rlao_b200.Source import Source
    from rlao_b200.Telescope import Telescope
    B, nS = 4096, 20
    tel = Telescope(120, 8, 1 / 500, n_envs=B, device=dev)
    Source("I", 12) * tel
    wfs = ShackHartmann(nS, tel, 0.5)
    tel.resetOPD()
    tel * wfs
    ideal = _np(wfs.cam.frame[0])
    clean_sig = _np(wfs.signal[0])
    cam = wfs.cam
    cam.photonNoise, cam.readoutNoise, cam.QE, cam.FWC, cam.bits, cam.darkCurrent, cam.sensor = True, 14, 0.56, 10000, 10, 5.0, "CMOS"
    cam.integrationTime = 1 / 500
    tel * wfs
    f1 = wfs.cam.frame.clone()
    s1 = _np(wfs.signal)
    tel * wfs
    f2 = wfs.cam.frame.clone()
    # whole counts, clipped at the top only (Detector.py:190-201 truncates towards zero and clips to [min, 2^bits - 1]:
    # read noise around an empty pixel gives small negative counts)
    assert bool((f1 == f1.round()).all()) and float(f1.min()) > -12 and float(f1.max()) <= 1023
    mean = f1.double().mean(dim=0).cpu().numpy()
    var = f1.double().var(dim=0).cpu().numpy()
    lit = ideal > 0.2 * ideal.max()
    # expectation of the chain (Detector.py:190-301) by Monte Carlo in float64, pixel by pixel: Poisson(photons) x QE +
    # Poisson(dark), full well, + round(N(0,1) RON), ADC frame / FWC * (2^bits - 1) truncated towards zero.  At this flux
    # (a few electrons per pixel under 14 e- of read noise) the truncation is not a plain -1/2 count.
    rs = np.random.RandomState(3)
    lam = ideal[lit]
    K = 4096
    e = rs.poisson(lam[None, :], size=(K, lam.size)) * 0.56 + rs.poisson(5.0 / 500, size=(K, lam.size))
    e = np.clip(e, 0, 10000) + np.round(rs.normal(size=(K, lam.size)) * 14)
    adu = np.trunc(e / 10000 * 1023)
    assert abs(mean[lit].mean() - adu.mean()) < 0.02 * adu.std() + 4 * adu.std() / np.sqrt(K * lam.size / 50)
    assert abs(var[lit].mean() / adu.var(axis=0).mean() - 1) < 0.03
    assert np.corrcoef(mean[lit], adu.mean(axis=0))[0, 1] > 0.5                # brighter pixels read brighter
    d1, d2 = (f1.double() - f1.double().mean(dim=0)), (f2.double() - f2.double().mean(dim=0))
    sel = torch.as_tensor(lit, device=dev)
    c_frames = float((d1[:, sel] * d2[:, sel]).mean() / (d1[:, sel].std() * d2[:, sel].std()))
    assert abs(c_frames) < 5e-3                                                   # independent frames
    c_envs = float((d1[0::2][:, sel] * d1[1::2][:, sel]).mean() / d1[:, sel].var())
    assert abs(c_envs) < 5e-3                                                     # independent environments
    # slopes: unbiased around the noise-free measurement, noise well above float32 error, finite
    assert np.isfinite(s1).all()
    assert np.abs(s1.mean(axis=0) - clean_sig).max() < 6 * s1.std(axis=0).max() / np.sqrt(B) + 0.02 * np.abs(s1).max()
    assert s1.std(axis=0).mean() > 1e-3
    # another shard (env_offset) draws other noise
    wfs.env_offset = B
    cam.frame_counter = 1
    tel * wfs
    assert not torch.equal(wfs.cam.frame, f1)


# ---- the reference's own closed loop at 80 x 80 -----------------------------------------------------------------------
@pytest.mark.skipif(not os.path.exists(GOLD), reason="tests/golden/cfg5.npz not generated (oracle/make_golden.py cfg5)")
def test_closed_loop_trace_cfg5_vs_reference_golden(dev):
    """Trace recorded from the UNMODIFIED reference at 80 x 80 x 5 layers; every step driven with the reference's action.
    The CPU oracle is not run beside it (its set-up takes tens of minutes at this size): the knife-edge lenslet masks of
    every step come from the reference's own spots in the fixture; the reconstructor is the GPU-calibrated one, so `obs`
    is compared at the accuracy the two calibrations agree to."""
    cfg = CONFIGS["cfg5"]()
    gold = load_golden("cfg5")
    env = build_env(cfg, n_envs=1, rng="reference", device=dev)
    assert np.array_equal(env.wfs.valid_subapertures, gold["valid_subapertures"])
    assert np.array_equal(env.dm_mask.astype(bool), gold["validAct"].astype(bool))
    assert rel_err(env.wfs.slopes_units, gold["slopes_units"]) < 2e-6
    assert rel_err(env.wfs.reference_slopes_maps, gold["reference_slopes_maps"]) < 1e-6
    env.wfs.slopes_units = float(gold["slopes_units"])
    n, nV = STEPS["cfg5"], env.wfs.nValidSubaperture
    knife = np.unpackbits(gold["knife_edge"], axis=1)[:, :nV].astype(bool)
    obs = new_episode(env, EPISODE_SEED)
    assert rel_err(_np(env.wfs.signal), gold["signal0"]) < 1e-4
    assert rel_err(_np(obs), gold["obs0"]) < 5e-3
    obs_ref = gold["obs0"].astype(np.float64)
    rows = slice(0, None, int(gold["snap_row_step"]))
    excluded = []
    for i in range(n):
        action = cfg.gainCL * obs_ref
        obs, reward, strehl, done, info = env.step(i, torch.as_tensor(action, dtype=torch.float32, device=dev))
        obs_ref = gold["trace_obs"][i].astype(np.float64)
        assert rel_err(_np(env.dm.coefs), gold["trace_coefs"][i]) < 2e-6, (i, "coefs")
        assert abs(float(strehl) - gold["trace_strehl"][i]) <= 1e-3 * gold["trace_strehl"][i] + 1e-30, (i, "strehl")
        edge = knife[i]
        excluded.append(int(edge.sum()))
        assert edge.sum() <= 0.02 * nV, (i, "too many knife-edge lenslets", int(edge.sum()))
        keep = np.concatenate([~edge, ~edge])
        sig, sig_ref = _np(env.wfs.signal), gold["trace_signal"][i]
        assert np.abs(sig - sig_ref)[keep].max() < 2e-4 * np.abs(sig_ref).max(), (i, "slopes")
        assert rel_err(_np(obs), gold["trace_obs"][i]) < 1e-2, (i, "obs")
        assert abs(float(reward) - gold["trace_reward"][i]) <= 1e-2 * abs(gold["trace_reward"][i]), (i, "reward")
    last = n - 1
    assert rel_err(_np(env.atm.OPD)[rows], gold[f"atm_OPD_{last}"]) < 3e-5
    assert rel_err(_np(env.tel.OPD)[rows], gold[f"tel_OPD_{last}"]) < 1e-4
    assert rel_err(_np(env.wfs.cam.frame)[rows], gold[f"frame_{last}"]) < 2e-4
    assert rel_err(_np(env.total[:n, 0]), gold["trace_total"]) < 1e-4
    assert rel_err(_np(env.residual[:n, 0]), gold["trace_residual"]) < 1e-3
    print("knife-edge lenslets excluded per step:", excluded)
