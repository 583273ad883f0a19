"""Shared helpers for the parity tests."""
import types

import numpy as np


def param_from_config(cfg):
    """oracle.ao_oracle.AOConfig -> parameter dict in the format rlao_b200's env mirror reads
    (same keys as the reference's parameter files, see rlao_b200/Conf/parameter_file_synthetic_SHWFS.py)."""
    d = cfg.detector
    p = dict(
        r0=cfg.r0, L0=cfg.L0, fractionalR0=list(cfg.fractionalR0), windSpeed=list(cfg.windSpeed),
        windDirection=list(cfg.windDirection), altitude=list(cfg.altitude), diameter=cfg.diameter,
        nSubaperture=cfg.nSubap, nPixelPerSubap=cfg.nPixPerSubap, resolution=cfg.resolution,
        samplingTime=cfg.samplingTime, centralObstruction=cfg.centralObstruction, magnitude=cfg.magnitude,
        opticalBand=cfg.opticalBand, nActuator=cfg.nSubap + 1, mechanicalCoupling=cfg.mechCoupling, isM4=False,
        dm_geometry="cartesian", shiftX=0, shiftY=0, rotationAngle=0, anamorphosisAngle=0, radialScaling=0,
        tangentialScaling=0, lightRatio=cfg.lightRatio, threshold_cog=cfg.threshold_cog, shannon_sampling=False,
        cam_photonNoise=d.photonNoise, cam_readoutNoise=d.readoutNoise, cam_sensor=d.sensor, cam_FWC=d.FWC,
        cam_bits=d.bits, cam_QE=d.QE, cam_darkCurrent=d.darkCurrent, nZernike=cfg.nZernike,
        nMeasurements=cfg.nMeasurements, nLoop=cfg.nLoop, gainCL=cfg.gainCL)
    return p


def build_env(cfg, n_envs=1, rng="reference", seed=0, device=None, env_offset=0, canvas_slack=32):
    from rlao_b200.OOPAOEnv.OOPAOEnvRazor import OOPAO
    env = OOPAO()
    env.set_params_file(param_from_config(cfg), "")
    env.set_params(types.SimpleNamespace(), "shackhartmann", gainCL=cfg.gainCL, n_envs=n_envs, rng=rng, seed=seed,
                   device=device, env_offset=env_offset, canvas_slack=canvas_slack)
    env.leak = cfg.leak
    return env


def new_episode(env, seed):
    """Caller pattern of MAIN_CODE/integrator_oopao_razor.py:46-60 / PO4AO/mbrl.py:49-55."""
    env.atm.generateNewPhaseScreen(seed)
    env.dm.coefs = 0
    env.dm_prev = 0 * env.dm_prev
    env.tel * env.dm * env.wfs
    return env.reset_soft()


def knife_edge_lenslets(maps, threshold, margin=1e-4):
    """Lenslets of `maps` [nValid, n, n] having a pixel within `margin` (relative) of the centroiding `threshold`: the
    float32 path may legitimately flip such a pixel (SURVEY.md section 7, hard parts)."""
    return (np.abs(maps - threshold) < margin * threshold).any(axis=(1, 2))


def psf_window_f64(amp, phase, zeroPaddingFactor, window):
    """The central `window` x `window` binned pixels of oracle.ao_oracle.compute_psf (even image sizes), as a matrix DFT in
    float64 on the device of the inputs: amp [R, R], phase [F, R, R] (radians) -> [F, window, window].
    compute_psf takes fftshift(fft2(ifftshift(sup * phasor))) / N of the field padded to N x N, so output row k is
    sum_n sup[n] exp(-2 pi i (k - N/2)(n - N/2) / N) / N over the support rows n = pad + y, and the same along x; the
    half-pixel phasor is applied as the reference rounds it, in complex64."""
    import torch
    R = amp.shape[-1]
    img_res = int(zeroPaddingFactor * R)
    os_ = 1 if zeroPaddingFactor >= 2 else int(np.ceil(2.0 / zeroPaddingFactor))
    if os_ % 2 != img_res % 2:
        os_ += 1
    N = int(np.fix(zeroPaddingFactor * os_ * R))
    pad, img_size = int(np.ceil((N - R) / 2)), img_res * os_
    assert img_res % 2 == 0 and N % 2 == 0 and N == R + 2 * pad and N % 2 == img_size % 2, "even image sizes only"
    dev = phase.device
    n = pad + torch.arange(R, device=dev, dtype=torch.int64)
    phasor = torch.polar(torch.ones(R, R, dtype=torch.float64, device=dev), -np.pi / N * (n[None, :] + n[:, None]).double())
    field = torch.polar(amp.double().expand_as(phase), phase.double()) * phasor.to(torch.complex64).to(torch.complex128)
    lo = int(np.ceil(N / 2) - img_size // 2)                       # compute_psf's crop of the image (shift 0: N, img even)
    c = img_res // 2
    k = lo + os_ * (c - window // 2) + torch.arange(os_ * window, device=dev, dtype=torch.int64)
    m = ((k - N // 2)[:, None] * (n - N // 2)[None, :]) % N          # exact integer phase reduction
    W = torch.polar(torch.ones(m.shape, dtype=torch.float64, device=dev), -2 * np.pi * m.double() / N)
    emf = W @ field @ W.T / N
    psf = emf.abs() ** 2
    return psf.reshape(-1, window, os_, window, os_).sum(dim=(2, 4))


def rel_err(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return np.abs(a - b).max() / max(np.abs(b).max(), 1e-300)
