"""Drives oracle.ao_oracle.EnvOracle exactly as oracle/make_golden.py drives the reference, returning the
same keys, so a test can diff the two dictionaries (TEST INFRASTRUCTURE ONLY)."""
import numpy as np
from numpy.random import RandomState
from threadpoolctl import threadpool_limits

from .ao_oracle import EnvOracle, compute_psf
from .golden_configs import COMPACT, CONFIGS, STEPS, EPISODE_SEED
from .make_golden import BLAS_THREADS, digest, DET_SEED


def replay_oracle(name, env=None, steps=None):
    """On the BLAS thread count the fixtures were recorded with, whatever the host's core count."""
    with threadpool_limits(limits=BLAS_THREADS, user_api="blas"):
        return _replay_oracle(name, env, steps)


def _replay_oracle(name, env, steps):
    cfg = CONFIGS[name]()
    env = env if env is not None else EnvOracle(cfg, detector_seed=DET_SEED)
    g = {}
    g["pupil"] = np.packbits(env.pupil)
    g["valid_subapertures"] = env.wfs.valid
    g["validAct"] = env.dm_mask
    g["slopes_units"] = np.float64(env.wfs.slopes_units)
    g["reference_slopes_maps"] = env.wfs.reference_slopes_maps
    g["nPhoton"] = np.float64(env.nPhoton)
    g["wavelength"] = np.float64(env.wavelength)
    g["A_digest"] = digest(env.atm.A)
    g["B_digest"] = digest(env.atm.B)
    g["A_row0"] = env.atm.A[0].copy()
    g["B_diag"] = np.diag(env.atm.B).copy()
    g["modes_digest"] = digest(env.modes)
    g["D_zonal_digest"] = digest(env.D_zonal)
    g["reconstructor_digest"] = digest(env.reconstructor)
    if env.reconstructor.size <= 20000:
        g["reconstructor"] = env.reconstructor
    g["signal_after_build"] = env.wfs.signal.copy()
    phase = env.tel_OPD * 2 * np.pi / env.wavelength
    psf = compute_psf(env.pupil, env.fluxMap, phase, 4)
    c = psf.shape[0] // 2
    g["psf_atm_max"] = np.float64(psf.max())
    g["psf_atm_crop"] = psf[c - 8:c + 8, c - 8:c + 8].copy()
    g["psf_atm_phase"] = phase

    # same point at which make_golden.py swaps in the seeded detector streams
    env.cam.rs_photon = RandomState(DET_SEED)
    env.cam.rs_readout = RandomState(DET_SEED + 1)
    env.cam.rs_dark = RandomState(DET_SEED + 2)
    n = steps if steps is not None else STEPS[name]
    obs = env.new_episode(EPISODE_SEED)
    g["obs0"] = obs.copy()
    g["signal0"] = env.wfs.signal.copy()
    g["frame0"] = np.asarray(env.wfs.frame).copy()
    nA = cfg.nSubap + 1
    tr = dict(obs=np.zeros((n, nA, nA)), reward=np.zeros(n), strehl=np.zeros(n),
              signal=np.zeros((n, env.wfs.nSignal)), coefs=np.zeros((n, env.nValidAct)))
    for i in range(n):
        obs, reward, strehl, done, info = env.step(i, env.gainCL * obs)
        tr["obs"][i], tr["reward"][i], tr["strehl"][i] = obs, reward, strehl
        tr["signal"][i] = env.wfs.signal
        tr["coefs"][i] = env.coefs
        if i in ((n - 1,) if name in COMPACT else (0, n // 2, n - 1)):
            g[f"atm_OPD_{i}"] = env.atm.OPD.copy()
            g[f"tel_OPD_{i}"] = env.tel_OPD.copy()
            g[f"frame_{i}"] = np.asarray(env.wfs.frame).copy()
    for k, v in tr.items():
        g["trace_" + k] = v
    g["trace_total"] = env.total[:n].copy()
    g["trace_residual"] = env.residual[:n].copy()
    g["snap_steps"] = np.array([n - 1] if name in COMPACT else [0, n // 2, n - 1])
    for i, ly in enumerate(env.atm.layers):
        g[f"final_buff_{i}"] = ly.buff.copy()
        g[f"final_map_digest_{i}"] = digest(ly.map)
    return g, env
