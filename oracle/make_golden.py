"""Generates tests/golden/*.npz by running the UNMODIFIED reference (/root/reference) in the build
container — TEST INFRASTRUCTURE ONLY.  Usage:  python -m oracle.make_golden [name ...]

Each fixture holds what the reference produced for one named configuration (oracle/golden_configs.py):
init-time quantities (masks, slope units, reference slopes, reconstructor or its digest, atmosphere
operator digests) and a closed-loop integrator trace driven exactly like
MAIN_CODE/integrator_oopao_razor.py:46-70 (generateNewPhaseScreen(17); reset_soft(); action = gainCL*obs;
env.step(i, action)).  The reference detector seeds its noise from the wall clock (OOPAO/Detector.py:127-130);
for the noisy fixture the three RandomState attributes are replaced by RandomState(seed), which keeps the
reference code path untouched and makes its integer frames reproducible.

The OPD and camera-frame snapshots of the trace go to <name>_snapshots.npz beside <name>.npz, so that no fixture file
grows past 1 MB; load() returns the two as one dictionary.
"""
import os
import sys

import numpy as np
from numpy.random import RandomState
from threadpoolctl import threadpool_limits

from . import ref_harness as rh
from .golden_configs import COMPACT, CONFIGS, LITE, STEPS, EPISODE_SEED

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")
DET_SEED = 1234
# BLAS threads the fixtures are recorded and replayed with.  The atmosphere's innovation factor B is the Cholesky factor of
# a Schur complement formed through pinv of an ill-conditioned covariance: OpenBLAS's thread split alone moves its digest by
# up to 4e-6 (relative), far above the 1e-7 the oracle is held to, so the split is fixed rather than left to the host.
BLAS_THREADS = 8


def paths(name, golden_dir=OUT):
    """The fixture of `name`: (<name>.npz, <name>_snapshots.npz)."""
    return os.path.join(golden_dir, name + ".npz"), os.path.join(golden_dir, name + "_snapshots.npz")


def load(name, golden_dir=OUT):
    """Every array of the fixture of `name`, snapshots included, as one dictionary."""
    g = {}
    for path in paths(name, golden_dir):
        with np.load(path) as z:
            g.update((k, z[k]) for k in z.files)
    return g


def digest(a):
    a = np.asarray(a, dtype=np.float64)
    return np.array([a.sum(), np.abs(a).sum(), (a * a).sum(), a.flat[0], a.flat[a.size // 2], a.flat[-1]])


def generate(name):
    cfg = CONFIGS[name]()
    env = rh.build_reference_env(cfg)
    g = {}
    g["pupil"] = np.packbits(env.tel.pupil.astype(bool))
    g["valid_subapertures"] = env.wfs.valid_subapertures
    g["validAct"] = np.reshape(env.dm.validAct, (cfg.nSubap + 1, cfg.nSubap + 1))
    g["slopes_units"] = np.float64(env.wfs.slopes_units)
    g["reference_slopes_maps"] = env.wfs.reference_slopes_maps
    g["nPhoton"] = np.float64(env.source.nPhoton)
    g["wavelength"] = np.float64(env.source.wavelength)
    L = env.atm.layer_1
    g["A_digest"] = digest(L.A)
    g["B_digest"] = digest(L.B)
    g["A_row0"] = L.A[0].copy()
    g["B_diag"] = np.diag(L.B).copy()
    g["modes_digest"] = digest(env.dm.modes)
    g["D_zonal_digest"] = digest(env.calib_zonal.D)
    g["reconstructor_digest"] = digest(env.reconstructor)
    if env.reconstructor.size <= 20000:
        g["reconstructor"] = env.reconstructor
    g["signal_after_build"] = env.wfs.signal.copy()
    # PSF of the flat wavefront and of the current atmosphere (Telescope.py:260-360), zero padding 4
    with rh.quiet():
        env.tel.computePSF(4)
    c = env.tel.PSF.shape[0] // 2
    g["psf_atm_max"] = np.float64(env.tel.PSF.max())
    g["psf_atm_crop"] = env.tel.PSF[c - 8:c + 8, c - 8:c + 8].copy()
    g["psf_atm_phase"] = env.tel.src.phase.copy()
    if name in LITE:
        # PSF of a wavefront given by a formula (golden_configs.psf_formula_opd), so that the test can rebuild the input
        # without a 0.9 MB phase map in the fixture: peak and central 32 x 32 window of tel.computePSF(4)
        from .golden_configs import psf_formula_opd
        env.tel.OPD = psf_formula_opd(cfg.resolution) * env.tel.pupil
        with rh.quiet():
            env.tel.computePSF(4)
        c = env.tel.PSF.shape[0] // 2
        g["psf_formula_max"] = np.float64(env.tel.PSF.max())
        g["psf_formula_win"] = env.tel.PSF[c - 16:c + 16, c - 16:c + 16].copy()
        env.tel.resetOPD()

    if cfg.detector.photonNoise or cfg.detector.readoutNoise:
        env.wfs.cam.random_state_photon_noise = RandomState(DET_SEED)
        env.wfs.cam.random_state_readout_noise = RandomState(DET_SEED + 1)
        env.wfs.cam.random_state_dark_shot_noise = RandomState(DET_SEED + 2)
    elif cfg.detector.darkCurrent:
        env.wfs.cam.random_state_dark_shot_noise = RandomState(DET_SEED + 2)

    n = STEPS[name]
    with rh.quiet():
        env.atm.generateNewPhaseScreen(EPISODE_SEED)
        env.dm.coefs = 0
        env.dm_prev = env.dm.coefs.copy()
        env.tel * env.dm * env.wfs
        obs = env.reset_soft()
    g["obs0"] = obs.copy()
    g["signal0"] = env.wfs.signal.copy()
    g["frame0"] = np.asarray(env.wfs.cam.frame).copy()
    nA = cfg.nSubap + 1
    tr = dict(obs=np.zeros((n, nA, nA)), reward=np.zeros(n), strehl=np.zeros(n), signal=np.zeros((n, env.wfs.nSignal)),
              coefs=np.zeros((n, env.dm.nValidAct)))
    snaps = {}
    lite = name in LITE
    knife = np.zeros((n, env.wfs.nValidSubaperture), dtype=bool)
    rows = slice(0, None, 3) if lite else slice(None)
    for i in range(n):
        with rh.quiet():
            obs, reward, strehl, done, info = env.step(i, env.gainCL * obs)
        tr["obs"][i], tr["reward"][i], tr["strehl"][i] = obs, reward, strehl
        tr["signal"][i] = env.wfs.signal
        tr["coefs"][i] = env.dm.coefs
        if lite:     # lenslets with a pixel within 1e-4 (relative) of the centroiding threshold, from the reference's spots
            maps = env.wfs.maps_intensity
            thr = env.wfs.threshold_cog * maps.max()
            knife[i] = (np.abs(maps - thr) < 1e-4 * thr).any(axis=(1, 2))
        if i in ((n - 1,) if name in COMPACT else (0, n // 2, n - 1)):
            ft = np.float32 if name in COMPACT else np.float64
            snaps[f"atm_OPD_{i}"] = env.atm.OPD.astype(ft)[rows]
            snaps[f"tel_OPD_{i}"] = env.tel.OPD.astype(ft)[rows]
            snaps[f"frame_{i}"] = np.asarray(env.wfs.cam.frame).astype(ft)[rows]
    for k, v in tr.items():
        g["trace_" + k] = v
    g["trace_total"] = env.total[:n].copy()
    g["trace_residual"] = env.residual[:n].copy()
    g["snap_steps"] = np.array([n - 1] if name in COMPACT else [0, n // 2, n - 1])
    if lite:
        g["knife_edge"] = np.packbits(knife, axis=1)
        g["snap_row_step"] = np.int64(3)
        for k in ("frame0", "psf_atm_phase", "psf_atm_crop"):
            g.pop(k, None)
        g["trace_obs"] = g["trace_obs"].astype(np.float32)
        g["obs0"] = g["obs0"].astype(np.float32)
    if name in COMPACT:
        for k in ("frame0", "trace_signal", "trace_coefs", "psf_atm_phase", "signal_after_build", "signal0", "reference_slopes_maps"):
            if k in g:
                g[k] = np.asarray(g[k]).astype(np.float32)
    for i in range(env.atm.nLayer):
        ly = getattr(env.atm, f"layer_{i + 1}")
        g[f"final_buff_{i}"] = ly.buff.copy()
        g[f"final_map_digest_{i}"] = digest(ly.mapShift)
    os.makedirs(OUT, exist_ok=True)
    for path, arrays in zip(paths(name), (g, snaps)):
        np.savez_compressed(path, **arrays)
        print(name, "->", path, os.path.getsize(path) // 1024, "KiB")


if __name__ == "__main__":
    if not rh.reference_available():
        sys.exit("reference not present: golden fixtures can only be regenerated in the build container")
    with threadpool_limits(limits=BLAS_THREADS, user_api="blas"):
        for nm in (sys.argv[1:] or list(CONFIGS)):
            generate(nm)
