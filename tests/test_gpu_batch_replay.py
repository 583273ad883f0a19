"""The batched environment step at the benchmark's batch sizes against a float64 restatement, environment by environment.

Every environment is built the way bench.py builds it (bench.make_args, the synthetic parameter file, rng="philox", seed 1,
generateNewPhaseScreen(17), the integrator loop obs = env.step(None, gain * obs)), so the step takes the benchmark's path:
the two library calls aoenv_atm_update + aoenv_sh_step, the reconstruction on the tensor cores from the bf16 slope planes,
the next frame's atmosphere on the side stream where the batch is large enough, add_row products of G * B rows.  For a
sample of environments (both sides of warp, CTA and GEMM tile boundaries, the end of the batch, seeded random ones) every
stage of a step is recomputed in float64 from that environment's own inputs; cheap invariants are checked on all of them.
The Pyramid (cfg2) and the science-PSF reward (cfg5psf) take the other path, one entry point at a time
(OOPAO._measure_frame + _apply_command): the DM surface written to memory by aoenv_dm_surface_separable, the Pyramid's
frames in chunks of environments (aoenv_pyramid_frames) and its torch signal processing, the PSF peak (aoenv_psf_peak).
A kernel that reads or writes another environment's row, a chunk loop that gets an offset wrong, or a kernel that
mishandles the last partial tile, fails here even though its closed-loop numbers would look plausible."""
import math

import numpy as np
import pytest
import torch

import bench
from geometric_oracle import GeometricShackHartmannOracle
from oracle.ao_oracle import ShackHartmannOracle, dm_geometry, flux_map, ring_masks, source_properties, telescope_pupil
from oracle.pyramid_oracle import PyramidOracle
from oracle.warp018 import warp_translate
from parity_util import knife_edge_lenslets, psf_window_f64, rel_err

pytestmark = pytest.mark.gpu

U32 = 2.0 ** -24                 # unit roundoff of float32
SINCOS_ABS = 2.0 ** -21.41       # largest absolute error of __sinf / __cosf on [-pi, pi] (CUDA C Programming Guide)
BAND_CUT = math.exp(-21.0)       # the separable DM tables drop a Gaussian factor below this (DeformableMirror: CUT = 21)
REC_BLOCK_N = 256                # environments per output tile of the reconstruction product (csrc/gemm_tc.cu: launch<2, 256>)
SLOPE_TOL = 1e-4
# Knife-edge lenslets excluded from the slope comparison, as a fraction of the valid ones: at most 1 % of the sampled
# environments' lenslets in one step, and 5 % of any one environment's.  The set comes from the float64 oracle's maps
# alone, so a wrong kernel cannot grow it; the limits only keep the comparison from being hollowed out.  Measured at these
# seeds: 0.14 % (cfg3), 0.18 % (cfg5), 0.3 % (cfg2: about one lenslet of 316 per environment, three in a few).
KNIFE_EDGE_STEP, KNIFE_EDGE_ENV = 0.01, 0.05
WARMUP, CHECKED = 3, 3


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    return torch.device("cuda:0")


def _np(t):
    return t.detach().double().cpu().numpy()


def sampled_envs(B):
    """Environments recomputed in float64: both sides of the warp (32) and CTA (128, 256) boundaries, the last two of the
    batch, the first and last of the reconstruction's last output tile when it is partial, and six seeded random ones."""
    idx = {0, 1, 31, 32, 127, 128, 129, 255, 256, B - 2, B - 1}
    if B % REC_BLOCK_N:
        idx |= {B // REC_BLOCK_N * REC_BLOCK_N, B - 1}
    idx |= {int(i) for i in np.random.default_rng(B).choice(B, size=6, replace=False)}
    return sorted(i for i in idx if 0 <= i < B)


def bench_env(dev, workload, B, geometric=False, wfs="shackhartmann"):
    """The environment of bench.py's GPU arm (same arguments, same episode start, the PSF reward of the workload), its
    first observation and bench.py's oracle configuration of the workload."""
    from rlao_b200.OOPAOEnv.OOPAOEnvRazor import OOPAO
    nS, nL, _, _, opts = bench.WORKLOADS[workload]
    args = bench.make_args(nS, nL, opts)
    if geometric:
        args.is_geometric = True
    env = OOPAO()
    env.set_params_file("rlao_b200.Conf.parameter_file_synthetic_SHWFS", "")
    env.set_params(args, wfs, gainCL=0.5, n_envs=B, device=dev, rng="philox", seed=1, env_offset=0)
    env.atm.generateNewPhaseScreen(17)
    env.dm.coefs = 0
    env.tel * env.dm * env.wfs
    obs = env.reset_soft()
    if opts.get("psf"):
        env.psf_reward = tuple(opts["psf"])
    return env, obs, bench.oracle_config(nS, nL, opts)


def pyramid_oracle(cfg, param):
    """The float64 Pyramid of the parameter file's settings (OOPAO.set_params: n_pix_edge = 2)."""
    pupil = telescope_pupil(cfg.resolution)
    wl, nph = source_properties(cfg.opticalBand, cfg.magnitude)
    return PyramidOracle(pupil, flux_map(pupil, nph, cfg.samplingTime, cfg.diameter), cfg.nSubap, param["modulation"],
                         param["lightThreshold"], n_pix_separation=param["n_pix_separation"], n_pix_edge=2,
                         postProcessing=param["postProcessing"])


class StepReference:
    """Float64 pieces of one environment's step: the sensor oracle, the pupil, and the separable DM surface
    sum_k c_k gy_k(y) gx_k(x) (the dense influence matrix is never built).  sensor: "sh", "geometric" or "pyramid"."""

    def __init__(self, env, cfg, sensor="sh", oracle=None):
        R = cfg.resolution
        self.pupil = telescope_pupil(R)
        self.wl, nph = source_properties(cfg.opticalBand, cfg.magnitude)
        self.flux = flux_map(self.pupil, nph, cfg.samplingTime, cfg.diameter)
        xIF, yIF, act_mask, sigma = dm_geometry(cfg)
        g = np.linspace(0, 1, R) * R
        gx = np.exp(-((g[None, :] - (R / 2 + xIF * R / cfg.diameter)[:, None]) ** 2) / (2 * sigma ** 2))   # [nA, R] columns
        gy = np.exp(-((g[None, :] - (R / 2 + yIF * R / cfg.diameter)[:, None]) ** 2) / (2 * sigma ** 2))   # [nA, R] rows
        self.gx = torch.as_tensor(gx, dtype=torch.float64, device=env.device)
        self.gyT = torch.as_tensor(gy.T.copy(), dtype=torch.float64, device=env.device)
        self.n = R // cfg.nSubap
        W = env.dm._sep["W"]
        assert W in (12, 16)             # the banded surface kernels of dm.cu
        # aoenv_dm_surface_separable (banded) forms T = C gx with W chained FMAs per pixel column and the surface with W
        # chained FMAs per pixel row, from float32 gx and gy tables: every term is off by at most (2 W + 2) u of
        # |c_k| gy_k gx_k, + 1 u for second-order terms; terms whose factor is below the band cut are dropped
        self.sep_terms = 2 * W + 3
        if sensor == "pyramid":
            par = env.param
            self.wfs = pyramid_oracle(cfg, par) if oracle is None else oracle
            w = env.wfs
            assert (par["modulation"], par["n_pix_separation"], par["lightThreshold"]) == (3, 4, 0.1)
            assert par["postProcessing"] == "slopesMaps_incidence_flux" and w.postProcessing == par["postProcessing"]
            assert np.array_equal(w.validI4Q, self.wfs.validI4Q)
            assert (w.nSignal, w.nTheta, w.nRes, w.cam.resolution) == (self.wfs.nSignal, self.wfs.nTheta, self.wfs.nRes,
                                                                       self.wfs.cam_resolution)
            assert w.slopesUnits == 1
            assert rel_err(_np(w.referenceSignal), self.wfs.referenceSignal) < 1e-9
            self.ref2d_env = _np(w.referenceSignal_2D)
        else:
            oracle = GeometricShackHartmannOracle if sensor == "geometric" else ShackHartmannOracle
            self.wfs = oracle(cfg, self.pupil, self.flux, self.wl)
            # the sensor kernels evaluate the surface in float32 from T = C gx (W columns per pixel) and the row windows (WL
            # rows per pixel): every term is off by at most (W + WL + 6) u of |c_k| gy_k gx_k (chained sums, products, tables)
            tables = env.dm.fused_tables()
            self.dm_terms = tables["W"] + env.wfs._dm_windows(tables)[0] + 6
            assert np.array_equal(env.wfs.valid_subapertures, self.wfs.valid)
            assert rel_err(env.wfs.slopes_units, self.wfs.slopes_units) < 2e-6
        # this is the system the environment built
        assert np.array_equal(env.dm_mask.astype(bool), act_mask)
        assert np.array_equal(np.asarray(env.tel.pupil).astype(bool), self.pupil)
        assert abs(env.tel.src.wavelength - self.wl) <= 1e-12 * self.wl

    def surfaces(self, coefs, materialised=False):
        """DM surfaces [k, R, R] of the commands [k, nA] and the bound on the float32 evaluation error of each pixel: by
        the sensor kernel (in place), or by aoenv_dm_surface_separable (materialised)."""
        c = torch.as_tensor(coefs, dtype=torch.float64, device=self.gx.device)
        surf = (self.gyT[None] * c[:, None, :]) @ self.gx
        mag = (self.gyT[None] * c.abs()[:, None, :]) @ self.gx
        if materialised:
            bound = mag * (self.sep_terms * U32) + BAND_CUT * c.abs().sum(dim=1)[:, None, None]
        else:
            bound = mag * (self.dm_terms * U32)
        return surf.cpu().numpy(), bound.cpu().numpy()


def std_bound(f, centre, eps, pupil, n):
    """Bound on how far the kernels' std of the field `f` over the pupil can be from the float64 one.  The sensor kernels
    sum, per lenslet thread, the n x n values d = f - centre and d^2 in float32 (n^2 + 3 roundings of the magnitudes at
    most), then in float64; var = E[d^2] - E[d]^2.  n=None: the sums are float64 (the Pyramid's torch statistics), whose
    rounding is negligible here.  A pointwise error |e| <= eps of the field moves the std by at most rms(eps)."""
    d = (f - centre)[pupil]
    sigma = d.std()
    dvar = 0.0 if n is None else (n * n + 3) * U32 * (d * d).mean() + 2 * abs(d.mean()) * (n * n + 1) * U32 * np.abs(d).mean()
    return np.sqrt((eps[pupil] ** 2).mean()) + dvar / (2 * sigma), sigma


def check_every_env(env, obs, reward, strehl, invalid):
    """On all environments, on the device: finite outputs, nothing at invalid actuators, reward = -||obs||_2.  The kernel's
    float32 sum of squares (nA / 256 terms per thread, a warp tree, 8 warp sums) is within ~40 u of the float64 one at
    every size here, and the square root halves that."""
    B, nA, nSig = env.n_envs, env.dm.nValidAct, env.wfs.nSignal
    for name, t in (("obs", obs), ("reward", reward), ("strehl", strehl), ("slopes", env.wfs._signal[:, :nSig]),
                    ("reconstruction", env._rec[:, :nA]), ("total", env._total_now), ("residual", env._residual_now)):
        assert bool(torch.isfinite(t).all()), name
    flat = obs.reshape(B, -1)
    assert not bool(flat[:, invalid].any()), "obs at invalid actuators"
    norm = torch.linalg.vector_norm(flat.double(), dim=1)
    assert float(((reward.double() + norm).abs() / norm).max()) < 1e-6, "reward"


def noisy_frame_slopes(frame, wfs):
    """Slopes of a camera frame [R, R] in float64: thresholded centre of gravity of every valid lenslet (threshold = 0.01 x
    the maximum over the valid lenslets' pixels; axes as the oracle), minus the sensor's reference, in slope units.  Also
    the lenslets with a pixel that the float32 threshold, threshold_cog * max rounded once, classifies otherwise: the frame
    values are the device's own, so that product is the only place where float32 and float64 can disagree."""
    nS, n = wfs.nSubap, wfs.n_pix_subap
    tiles = frame.reshape(nS, n, nS, n).transpose(0, 2, 1, 3).reshape(nS * nS, n, n)[wfs.valid_subapertures_1D]
    cen = ShackHartmannOracle.centroid(tiles, wfs.threshold_cog)
    slopes = ((cen.T - _np(wfs._ref_xy)) / wfs.slopes_units).reshape(-1)
    top = tiles.max()
    thr32 = float(np.float32(wfs.threshold_cog) * np.float32(top))
    edge = ((tiles < thr32) != (tiles < wfs.threshold_cog * top)).any(axis=(1, 2))
    return slopes, edge


def pyramid_frame_bound(amp, kt, pm_max, nTheta, N, binning):
    """Bound on sum |frame - frame_f64| of aoenv_pyramid_frames, as a fraction of sum frame_f64 (a normwise error model).
    Field of a modulation point: amp exp(i phase), phase = kt + tilt, kt = k (opd + surface) pupil in float64.  The kernel
    sums opd + surface in float32, rounds the products with the float32 phase_turns (phase_scale / 2 pi, three roundings),
    the float32 tilt and the exact phasor reduction (at most 6 u |kt| + 8 u |tilt| + 3 u 2 pi of phase in all), takes
    __sinf / __cosf (SINCOS_ABS) and rounds amp and amp * cos / sin (3 u).  Four float32 transforms of length N = 16 x N2
    follow (Higham, Accuracy and Stability of Numerical Algorithms, Thm 24.2: eps1 = L eta / (1 - L eta),
    eta = u + gamma_4 (sqrt2 + u); the codelets' radix-3 butterflies and extra twiddle products are covered by counting
    L = 2 ceil(log2 N) levels), and the float32 mask product (4 u).  An l2 error eps of the field Y moves
    sum |Y|^2 by at most (2 eps + eps^2) sum |Y|^2.  Intensities: 2 nTheta chained FMAs over the modulation points, the
    1 / N^4 scale (4 u), binning of binning^2 pixels."""
    u = U32
    delta = u * (6 * np.abs(kt) + 8 * pm_max + 3 * 2 * np.pi) + math.sqrt(2) * SINCOS_ABS + 3 * u
    eps_field = math.sqrt(((amp * delta) ** 2).sum() / (amp ** 2).sum())
    L = 2 * math.ceil(math.log2(N))
    eta = u + 4 * u / (1 - 4 * u) * (math.sqrt(2) + u)
    eps = eps_field + 4 * L * eta / (1 - L * eta) + 4 * u
    return 2 * eps + eps * eps + (2 * nTheta + 4 + binning * binning) * u


def psf_peak_bound(amp, kt, peak, N, R, Wu):
    """Bound on |psf_peak - peak_f64| for one environment; peak_f64 = max of the float64 window.  Per pupil pixel
    psf_field_kernel errs on amp exp(i kt) by at most amp (u (6 |kt| + 2 pi + 3) + sqrt2 SINCOS_ABS): the float32 sum
    opd + surface and the product with phase_turns (the piston is not removed, so |kt| is the full phase), the reduced
    angle times 2 pi, __sinf / __cosf, amp and its products.  Stage 1 (split-bf16 field and W1 planes) errs by 2^-16 of
    sum |amp| per component of the row transform; stage 2 by (2 R / slices + slices) chained float32 roundings plus the
    float32 twiddles, of sum |T| <= sum amp.  So every window amplitude |F| / N errs by at most delta = dF / N, and a
    binned pixel, the sum of 2 x 2 squared amplitudes, by at most 4 delta sqrt(P) + 4 delta^2, plus 7 roundings of P."""
    A = amp.sum()
    slices = max(1, 256 // Wu)
    per = -(-R // slices)
    dF = (amp * (U32 * (6 * np.abs(kt) + 2 * np.pi + 3) + math.sqrt(2) * SINCOS_ABS)).sum() \
        + math.sqrt(2) * (2.0 ** -16 + (2 * per + slices + 2) * U32) * A
    delta = dF / N
    return 4 * delta * math.sqrt(peak) + 4 * delta ** 2 + 8 * U32 * peak


def replay(env, obs, ref, mode, prefetch, extra_envs=(), frames_calls=None):
    """WARMUP + CHECKED integrator steps as bench.py runs them; every checked step is recomputed in float64 for the sampled
    environments.  mode: "sh" (diffractive sensor, noise off), "geometric", "noisy" (slopes from the device's own camera
    frame), "pyramid", "psf" (the diffractive sensor with the science-PSF Strehl as the step's Strehl).  extra_envs join
    the sample; frames_calls (Pyramid) is the list of environment counts that aoenv_pyramid_frames has been called with.
    Returns the knife-edge lenslets excluded per checked step (summed over the sampled environments) and, per stage, the
    worst error as a fraction of its bound."""
    dev, B, nA, nSig = env.device, env.n_envs, env.dm.nValidAct, env.wfs.nSignal
    from rlao_b200 import gemm
    for _ in range(WARMUP):
        obs, *_ = env.step(None, env.gainCL * obs)
    torch.cuda.synchronize()
    # the benchmark's path: two library calls per step for the Shack-Hartmann alone, one entry point at a time for the
    # Pyramid and the PSF reward; the next frame prefetched on the side stream where bench.py does it, the reconstruction
    # on the tensor cores
    one_at_a_time = mode in ("pyramid", "psf")
    if one_at_a_time:
        assert env._native_cfg() is None
    else:
        assert env._native is not None
    assert env.atm._prefetched == prefetch
    assert env.atm.can_prefetch() == prefetch
    assert gemm.uses_tensor_cores(B)
    idx = sorted(set(sampled_envs(B)) | {b for b in extra_envs if 0 <= b < B})
    it = torch.as_tensor(idx, device=dev)
    act_idx = env._act_idx.long()
    invalid = torch.as_tensor(~env.dm_mask.astype(bool).reshape(-1), device=dev)
    k = 2 * np.pi / ref.wl
    units = 1.0 if mode == "pyramid" else ref.wfs.slopes_units / env.wfs.slopes_units
    knife, worst = [], {}

    def record(name, err, bound):
        worst[name] = max(worst.get(name, 0.0), float(np.max(err / np.maximum(bound, 1e-300))))

    if mode == "psf":
        zp, win = env.psf_reward
        N, os_ = env.tel.psf_geometry(zp)[:2]
        amp64 = torch.as_tensor(np.sqrt(ref.flux), device=dev)
        amp_np = np.sqrt(ref.flux)
        flat = float(psf_window_f64(amp64, torch.zeros((1,) + ref.pupil.shape, dtype=torch.float64, device=dev), zp, win).max())
        flat_bound = psf_peak_bound(amp_np, 0.0, flat, N, ref.pupil.shape[0], os_ * win)
        record("psf flat peak", abs(float(env._psf_model_max) - flat), flat_bound)
        assert abs(float(env._psf_model_max) - flat) <= flat_bound, ("psf flat peak", float(env._psf_model_max), flat)
        psf_strehl = []
    if mode == "pyramid":
        orc = ref.wfs
        amp_np = np.sqrt(ref.flux / orc.nTheta)
        pm_max = float(np.abs(orc.phase_mod).max())
        binning = orc.nRes // orc.cam_resolution
    for step in range(CHECKED):
        coefs = env.dm.coefs[it]                         # the commands in effect: the DM surface this frame sees
        prev = env._dm_prev[it, :nA].clone()
        assert torch.equal(coefs, prev)
        action = env.gainCL * obs
        if frames_calls is not None:
            frames_calls.clear()
        obs, reward, strehl, _, _ = env.step(None, action)
        torch.cuda.synchronize()
        tag = (mode, B, step)
        check_every_env(env, obs, reward, strehl, invalid)
        if frames_calls is not None:
            chunk = env.wfs._kernel_ws[0][0]
            assert frames_calls == [min(chunk, B - s0) for s0 in range(0, B, chunk)], tag + ("pyramid chunks", frames_calls)

        # reconstruction: the split-bf16 product against float64 on the device's own slopes
        s = env.wfs._signal[it, :nSig].double()
        rec = env._rec[it, :nA]
        want = s @ env.reconstructor.T
        mag = s.abs() @ env.reconstructor.abs().T
        assert float(((rec.double() - want).abs() / mag).max()) < 2.0 ** -16, tag + ("reconstruction",)
        # observation: -rec * 1e6 at the valid actuators, bit for bit
        o = obs[it].reshape(len(idx), -1)
        assert torch.equal(o[:, act_idx], -rec * 1e6), tag + ("obs",)
        # command update: leak * previous + action * 1e-6, and the integrator state is the new command
        new = env.dm.coefs[it]
        want_c = env.leak * _np(prev) + _np(action[it].reshape(len(idx), -1)[:, act_idx]) * 1e-6
        new64 = _np(new)
        for j, b in enumerate(idx):
            assert rel_err(new64[j], want_c[j]) < 1e-6, tag + (b, "command")
        assert torch.equal(env._dm_prev[it, :nA], new), tag + ("dm_prev",)

        opd = _np(env.atm._opd[it])
        surf, surf_err = ref.surfaces(_np(coefs)) if mode != "pyramid" else (None, None)
        if one_at_a_time:
            # the surface this frame saw, written to memory by aoenv_dm_surface_separable (the slot before the command
            # update flipped it)
            seen = env.dm._slot ^ 1
            assert env.dm._valid[seen] and env.dm._coefs_of[seen] is not None
            surf_dev = _np(env.dm._opd[seen][it])
            surf_m, surf_m_err = ref.surfaces(_np(coefs), materialised=True)
            for j, b in enumerate(idx):
                err = np.abs(surf_dev[j] - surf_m[j])
                record("dm surface", err, surf_m_err[j])
                assert (err <= surf_m_err[j]).all(), tag + (b, "dm surface", float(err.max()))
        sig_dev = _np(s)
        total, residual = _np(env._total_now[it]), _np(env._residual_now[it])
        sr = _np(env._strehl[it])                        # the phase Strehl exp(-var), also under a PSF reward
        frames = _np(env.wfs._frame[it]) if mode in ("noisy", "pyramid") else None
        excluded = 0
        for j, b in enumerate(idx):
            if mode == "pyramid":
                # the sensor saw the float32 sum of the atmosphere and the materialised surface; stats are float64 sums
                field = opd[j] + surf_dev[j]
                kt = field * ref.pupil * k
                # frames: the float64 camera frame of the device's own inputs
                orc._propagate(kt)
                f64 = orc.frame
                l1 = np.abs(frames[j] - f64).sum()
                fb = pyramid_frame_bound(amp_np, kt, pm_max, orc.nTheta, orc.nRes, binning) * f64.sum()
                record("pyramid frame (l1)", l1, fb)
                worst["pyramid frame rel_err"] = max(worst.get("pyramid frame rel_err", 0.0), rel_err(frames[j], f64))
                assert l1 <= fb, tag + (b, "pyramid frame", l1 / f64.sum())
                raw64, sig64 = orc.signal_processing()
                norma64, dI = orc.norma, np.abs(frames[j] - f64).max()
                orc.frame = frames[j]
                maps_d, sig_d = orc.signal_processing()
                norma_d = orc.norma
                # slopes, 1: the quadrant arithmetic of the device's own frame, up to the float32 rounding of the stored
                # signal (and the difference of the two float64 reference slopes)
                ref_v = np.abs(orc.referenceSignal_2D)[orc.validSignal]
                dref = np.abs(ref.ref2d_env - orc.referenceSignal_2D)[orc.validSignal]
                b1 = U32 * np.abs(sig_d) + 1e-13 * (np.abs(sig_d) + ref_v) + (1 + U32) * dref
                record("pyramid slopes of the device frame", np.abs(sig_dev[j] - sig_d), b1)
                assert (np.abs(sig_dev[j] - sig_d) <= b1).all(), tag + (b, "pyramid slopes of the device frame")
                # slopes, 2: the float64 frame's slopes within what the frame error can move them
                s_raw = np.abs(sig64 + orc.referenceSignal)
                b2 = (4 * dI + s_raw * abs(norma_d - norma64)) / min(norma_d, norma64) * (1 + 1e-12) + 1e-13 * (s_raw + ref_v)
                record("pyramid slopes vs float64 frame", np.abs(sig_d - sig64), b2)
                assert (np.abs(sig_d - sig64) <= b2).all(), tag + (b, "pyramid slopes vs float64 frame")
                # pupil statistics in float64 over the float32 sum: that rounding and the surface bound only
                c = opd[j][opd.shape[1] // 2, opd.shape[2] // 2]
                d_tot, s_tot = std_bound(opd[j], c, np.zeros_like(field), ref.pupil, None)
                field_ref = opd[j] + surf_m[j]
                d_res, s_res = std_bound(field_ref, c, surf_m_err[j] + U32 * np.abs(field), ref.pupil, None)
            else:
                field = opd[j] + surf[j]
                # slopes
                if mode == "noisy":
                    want_s, edge = noisy_frame_slopes(frames[j], env.wfs)
                elif mode == "geometric":                # the geometric sensor sees the pupil-less OPD
                    want_s, edge = ref.wfs.measure(field * k) * units, np.zeros(env.wfs.nValidSubaperture, dtype=bool)
                else:
                    want_s = ref.wfs.measure(field * ref.pupil * k) * units
                    maps = ref.wfs.maps_intensity
                    edge = knife_edge_lenslets(maps, ref.wfs.threshold_cog * maps.max())
                nV = env.wfs.nValidSubaperture
                assert edge.sum() <= KNIFE_EDGE_ENV * nV, tag + (b, "too many knife-edge lenslets", int(edge.sum()))
                excluded += int(edge.sum())
                keep = np.concatenate([~edge, ~edge])
                assert np.abs(sig_dev[j] - want_s)[keep].max() < SLOPE_TOL * np.abs(want_s).max(), tag + (b, "slopes")
                # pupil statistics: rms of the atmosphere, of the residual, Strehl = exp(-var(phase)); the kernels centre
                # the sums on the atmosphere's centre pixel, and the residual carries the float32 DM surface and the
                # float32 sum atmosphere + surface
                c = opd[j][opd.shape[1] // 2, opd.shape[2] // 2]
                d_tot, s_tot = std_bound(opd[j], c, np.zeros_like(field), ref.pupil, ref.n)
                d_res, s_res = std_bound(field, c, surf_err[j] + U32 * np.abs(field), ref.pupil, ref.n)
                field_ref = field
            record("total", abs(total[j] - 1e9 * s_tot), 1e9 * (1e-5 * s_tot + d_tot))
            assert abs(total[j] - 1e9 * s_tot) <= 1e9 * (1e-5 * s_tot + d_tot), tag + (b, "total")
            record("residual", abs(residual[j] - 1e9 * s_res), 1e9 * (1e-5 * s_res + d_res))
            assert abs(residual[j] - 1e9 * s_res) <= 1e9 * (1e-5 * s_res + d_res), tag + (b, "residual")
            v = (field_ref[ref.pupil] * k).var()
            s_ref = math.exp(-v)
            # ln S = -k^2 var moves by at most k^2 (2 sigma d + d^2); float32 underflow of a barely corrected pupil: 1e-30
            tol = (1e-5 + math.expm1(k * k * (2 * s_res * d_res + d_res ** 2))) * s_ref + 1e-30
            record("phase strehl", abs(sr[j] - s_ref), tol)
            assert abs(sr[j] - s_ref) <= tol, tag + (b, "strehl", sr[j], s_ref)
        if mode == "psf":
            # the step's Strehl = psf_peak(atm + surface) / psf_peak(flat) against the float64 window of the same inputs
            kt = (torch.as_tensor(opd, device=dev) + torch.as_tensor(surf_dev, device=dev)) * torch.as_tensor(ref.pupil, device=dev) * k
            peaks = psf_window_f64(amp64, kt, zp, win).amax(dim=(1, 2)).cpu().numpy()
            kt = kt.cpu().numpy()
            got = _np(strehl[it])
            for j, b in enumerate(idx):
                dP = psf_peak_bound(amp_np, kt[j], peaks[j], N, ref.pupil.shape[0], os_ * win)
                want_sr = peaks[j] / flat
                tol = (dP + want_sr * flat_bound) / (flat - flat_bound) + 2 * U32 * want_sr
                record("psf strehl", abs(got[j] - want_sr), tol)
                assert abs(got[j] - want_sr) <= tol, tag + (b, "psf strehl", got[j], want_sr)
                psf_strehl.append(want_sr)
        if mode not in ("pyramid",):
            nV = env.wfs.nValidSubaperture
            assert excluded <= KNIFE_EDGE_STEP * len(idx) * nV, tag + ("too many knife-edge lenslets", excluded)
        knife.append(excluded)
    if mode == "psf":
        worst["psf strehl range"] = (min(psf_strehl), max(psf_strehl))
    return knife, worst


@pytest.mark.parametrize("workload,B,prefetch", [
    ("cfg2", 1024, False),       # bench sizes
    ("cfg3", 1024, True),
    ("cfg5", 256, True),         # R = 480
    ("cfg2", 1000, False),       # the last environment tile of the reconstruction is partial
    ("cfg2", 9, False),          # one row above the skinny FP32 product: the tensor-core path at its smallest
])
def test_step_replay_shack_hartmann_noise_off(dev, workload, B, prefetch):
    env, obs, cfg = bench_env(dev, workload, B)
    knife, _ = replay(env, obs, StepReference(env, cfg), "sh", prefetch)
    print(f"\n{workload} B={B}: knife-edge lenslets excluded per checked step (sum over {len(sampled_envs(B))} "
          f"environments of {env.wfs.nValidSubaperture} lenslets): {knife}")


def test_step_replay_geometric_sensor_at_cfg3_size(dev):
    """The geometric branch of aoenv_sh_step at 1024 environments: no threshold, so no lenslet is excluded."""
    env, obs, cfg = bench_env(dev, "cfg3", 1024, geometric=True)
    assert env.wfs.is_geometric
    replay(env, obs, StepReference(env, cfg, sensor="geometric"), "geometric", True)


def test_step_replay_noisy_camera_at_cfg4_size(dev):
    """4096 environments with the Razor-like camera: the frame is random, so the slopes are replayed from the device's own
    frame (per-environment maximum and threshold); the rest of the step and the noise-free pupil statistics as above."""
    env, obs, cfg = bench_env(dev, "cfg4", 4096)
    assert env.wfs.cam.photonNoise and env.wfs.cam.readoutNoise > 0
    knife, _ = replay(env, obs, StepReference(env, cfg), "noisy", True)
    print(f"\ncfg4 B=4096: lenslets with a pixel on the float32/float64 threshold boundary per checked step: {knife}")


def _report(name, worst):
    print(f"\n{name}: worst error / bound per stage: " + ", ".join(
        f"{k} {v[0]:.4g}..{v[1]:.4g}" if isinstance(v, tuple) else f"{k} {v:.3g}" for k, v in worst.items()))


@pytest.mark.parametrize("size", ["bench", "two chunks + 1"])
def test_step_replay_pyramid_at_cfg2_size(dev, monkeypatch, size):
    """bench.py --wfs pyramid: cfg2 at 1024 environments (the default), and at 2 chunk + 1 so that the last call of
    aoenv_pyramid_frames holds one environment.  Both sides of the first two chunk boundaries and of the last one are
    sampled; every call of the frames kernel is counted."""
    from rlao_b200 import _lib
    from rlao_b200.Conf.parameter_file_synthetic_SHWFS import initializeParameterFile
    from rlao_b200.Pyramid import Pyramid
    nS, nL, _, _, opts = bench.WORKLOADS["cfg2"]
    cfg = bench.oracle_config(nS, nL, opts)
    orc = pyramid_oracle(cfg, initializeParameterFile(bench.make_args(nS, nL, opts)))
    chunk = Pyramid.frames_chunk(orc.nTheta, orc.nRes, cfg.resolution)
    B = 1024 if size == "bench" else 2 * chunk + 1
    env, obs, _ = bench_env(dev, "cfg2", B, wfs="pyramid")
    assert env.wfs.tag == "pyramid" and env.wfs._kernels_ok()
    ref = StepReference(env, cfg, sensor="pyramid", oracle=orc)
    lib, calls = _lib.load(), []
    frames = lib.aoenv_pyramid_frames

    def counted(*args):
        calls.append(args[7])            # environments in this call
        return frames(*args)
    monkeypatch.setattr(lib, "aoenv_pyramid_frames", counted)
    obs, *_ = env.step(None, env.gainCL * obs)
    assert env.wfs._kernel_ws[0][0] == chunk and B > 2 * chunk
    last = (B - 1) // chunk * chunk                  # first environment of the last chunk
    edges = (chunk - 1, chunk, 2 * chunk - 1, 2 * chunk, last - 1, last)
    knife, worst = replay(env, obs, ref, "pyramid", False, extra_envs=edges, frames_calls=calls)
    _report(f"pyramid cfg2 B={B}: chunk {chunk}, {len(calls)} aoenv_pyramid_frames calls per step {calls}", worst)


def test_step_replay_psf_reward_at_cfg5_size(dev):
    """bench.py --workload cfg5psf: 256 environments, the Shack-Hartmann kernels one at a time, the DM surface written to
    memory at R = 480, the PSF peak at zero padding 4 (N = 3840, oversampling 2) as the step's Strehl."""
    env, obs, cfg = bench_env(dev, "cfg5psf", 256)
    assert env.psf_reward == (4, 32)
    knife, worst = replay(env, obs, StepReference(env, cfg), "psf", True)
    _report(f"cfg5psf B=256: knife-edge lenslets excluded per checked step {knife}", worst)


def test_atmosphere_at_cfg3_size_vs_float64(dev):
    """atm.update() at 1024 environments, sequenced by aoenv_atm_update (in line, so that the workspaces belong to the
    frame just computed): the phase of the sampled environments against the warp restatement of their own windows, and
    every add_row of the frame — interior shifted bit for bit, new ring = the environment's row g * B + b of X in outerMask
    order, X = [A | B] zx in float64, Z = the inner rings of the shifted window."""
    from rlao_b200 import gemm
    B = 1024
    env, obs, cfg = bench_env(dev, "cfg3", B)
    atm = env.atm
    L, M, R, nI, nO, K, parts = atm.nLayer, atm._M, cfg.resolution, atm._nI, atm._nO, atm._K, atm._W_op.parts
    obs, *_ = env.step(None, env.gainCL * obs)
    torch.cuda.synchronize()
    assert env._native is not None and atm._prefetched
    atm.pipelined = False
    atm.update()                         # takes the frame computed ahead; every update() below computes its frame in line
    idx = sampled_envs(B)
    it = torch.as_tensor(idx, device=dev)
    outer = ring_masks(M - 2)[0]
    inner_rc = atm._inner_rc.long().cpu().numpy()
    W = atm._W.double()
    extruded = 0
    for frame in range(6):
        prev = [_np(ly.mapShift[it]) for ly in atm._layers]
        events = [ly.events for ly in atm._layers]
        org, cur = [atm._org[i] for i in range(L)], [atm._cur[i] for i in range(L)]
        atm.update()
        torch.cuda.synchronize()
        assert not atm._prefetched
        maps = [_np(ly.mapShift[it]) for ly in atm._layers]
        assert all(np.isfinite(m).all() for m in maps)
        opd = _np(atm._opd[it])
        for j, b in enumerate(idx):
            want = 0
            for i, ly in enumerate(atm._layers):
                sh = warp_translate(maps[i][j], ly.buff[0], ly.buff[1], kernel=atm.warp_kernel)[1:-1, 1:-1]
                c = sh.shape[0] // 2
                want = want + sh[c - R // 2:c + R // 2, c - R // 2:c + R // 2] * math.sqrt(atm.fractionalR0[i])
            assert rel_err(opd[j], want * atm.wavelength / 2 / np.pi) < 2e-6, (frame, b, "phase")
        # the layers that extruded this frame went through one gather / product / ring, in layer order (group slots)
        ext = [i for i in range(L) if atm._layers[i].events != events[i]]
        if not ext:
            continue
        assert all(atm._layers[i].events == events[i] + 1 for i in ext)       # less than a pixel of wind per frame at cfg3
        G = len(ext)
        assert gemm.uses_tensor_cores(G * B)
        X = atm._X[:G * B, :nO]
        assert bool(torch.isfinite(X).all())
        zx_all = atm._zx_planes.reshape(-1)[:parts * G * B * K].reshape(parts, G * B, K)   # planes of this group's G * B rows
        for g, i in enumerate(ext):
            if atm._cur[i] != cur[i]:
                continue                 # re-centred into the other canvas this frame: the origin no longer tells the step
            sy, sx = org[i][0] - atm._org[i][0], org[i][1] - atm._org[i][1]
            assert (sy, sx) != (0, 0) and abs(sy) <= 1 and abs(sx) <= 1
            rows = g * B + it
            zx = zx_all[:, rows].double().sum(0)
            want_x = zx @ W.T
            mag = zx.abs() @ W.abs().T
            assert float(((X[rows].double() - want_x).abs() / mag).max()) < 2.0 ** -16, (frame, i, "X = [A | B] zx")
            Xs, zxs = _np(X[rows]), zx.cpu().numpy()
            for j, b in enumerate(idx):
                old, new = prev[i][j], maps[i][j]
                assert np.array_equal(new[1:-1, 1:-1], old[1 - sy:M - 1 - sy, 1 - sx:M - 1 - sx]), (frame, i, b, "interior")
                assert np.array_equal(new[outer], Xs[j]), (frame, i, b, "ring")
                z = old[inner_rc[:, 0] - sy, inner_rc[:, 1] - sx]
                assert (np.abs(zxs[j, :nI] - z) <= 2.0 ** -16 * np.abs(z)).all(), (frame, i, b, "Z")
            extruded += 1
    assert extruded > 0
