"""Float64 numpy definition of the geometric Shack-Hartmann sensor (`ShackHartmann(is_geometric=True)`, DESIGN.md section 2)
and of the closed-loop environment that uses it, built on the diffractive oracle of oracle/ao_oracle.py.  TEST
INFRASTRUCTURE ONLY.

PARITY UNPINNED: no reference output covers OOPAO's geometric branch, so the sensor is defined here as the geometric-optics
limit of the diffractive sensor the oracle pins — same lenslets, valid set, axes, signs, signal layout and calibration
procedure; per lenslet the flux-weighted mean of np.gradient of the PUPIL-LESS phase; reference slopes exactly zero; no
camera (noise-free).
"""
import numpy as np

from oracle.ao_oracle import EnvOracle, ShackHartmannOracle, calibration_vault, zernike_modes


class GeometricShackHartmannOracle(ShackHartmannOracle):
    """ShackHartmannOracle's valid set, signal layout and five-ramp slope units, measured geometrically.  `measure` and
    `measure_multi` take the pupil-less phase; the camera is never used."""

    def set_flux(self, fluxMap):
        self.fluxMap = np.asarray(fluxMap, dtype=float)
        super().set_flux(fluxMap)

    def _centroids(self, phase):
        """Geometric slopes of the valid lenslets [nValid, 2] (X, Y) of one phase map [R, R]: np.gradient with unit spacing
        (central differences inside, one-sided first differences on the outer rows and columns; axis 1 -> X, axis 0 -> Y),
        flux-weighted mean over the lenslet's pixels [i*n:(i+1)*n, j*n:(j+1)*n] (not transposed)."""
        nS, n = self.nS, self.n
        gy, gx = np.gradient(np.asarray(phase, dtype=float))
        tiles = lambda img: img.reshape(nS, n, nS, n).transpose(0, 2, 1, 3).reshape(nS * nS, n, n)[self.valid_1d]
        w = self.fluxMap
        sw = tiles(w).sum(axis=(1, 2))
        return np.stack([tiles(w * gx).sum(axis=(1, 2)) / sw, tiles(w * gy).sum(axis=(1, 2)) / sw], axis=1)

    def measure(self, phase):
        self.signal_2D, self.signal = self._signal_from_centroids(self._centroids(phase))
        return self.signal

    def measure_multi(self, phases, rs_photon=None, rs_readout=None):
        sig = np.zeros((self.nSignal, phases.shape[0]))
        for f in range(phases.shape[0]):
            _, sig[:, f] = self._signal_from_centroids(self._centroids(phases[f]))
        self.signal = sig
        return sig

    def _initialize(self):
        """Reference slopes stay zero (a flat wavefront has zero gradient); slope units from the five tip ramps of
        ShackHartmannOracle._initialize (full-ramp-std quirk kept), on the pupil-less ramp."""
        R = self.R
        tip, _ = np.meshgrid(np.linspace(0, np.pi, R, endpoint=False), np.linspace(0, np.pi, R, endpoint=False))
        tip = tip / np.std(tip[self.pupil.astype(int)])
        amp = 10e-9
        mean_slope = np.zeros(5)
        for i in range(5):
            self.measure(tip * (i - 2) * amp * 2 * np.pi / self.wavelength)
            mean_slope[i] = np.mean(self.signal[:self.nValid])
        p = np.polyfit(np.linspace(-2, 2, 5) * amp, mean_slope, deg=1)
        self.slopes_units = np.abs(p[0]) * (self.wavelength / 2 / np.pi)
        self.measure(np.zeros((R, R)))


def geometric_interaction_matrix(wfs, modes, stroke, wavelength, chunk=25):
    """InteractionMatrix (noise off) of the geometric sensor: the measurement is linear and has no shared threshold, so
    D = s(stroke * mode) / stroke, column by column."""
    R = wfs.R
    D = np.zeros((wfs.nSignal, modes.shape[1]))
    for c0 in range(0, modes.shape[1], chunk):
        opd = (modes[:, c0:c0 + chunk] * stroke).T.reshape(-1, R, R)
        D[:, c0:c0 + chunk] = wfs.measure_multi(opd * 2 * np.pi / wavelength) / stroke
    return D


class GeometricEnvOracle(EnvOracle):
    """EnvOracle with the geometric sensor: calibrated the same way (zonal interaction matrix, modal Zernike basis, SVD
    inverse), and the sensor sees the pupil-less OPD (atmosphere + DM surface)."""

    def __init__(self, cfg, atm_ops=None, act_mask=None, detector_seed=0):
        super().__init__(cfg, atm_ops=atm_ops, act_mask=act_mask, detector_seed=detector_seed, reconstructor=np.zeros((1, 1)))
        self.wfs = GeometricShackHartmannOracle(cfg, self.pupil, self.fluxMap, self.wavelength, self.cam)
        if cfg.nZernike > 0:
            Z = zernike_modes(self.pupil, cfg.diameter, cfg.nZernike)
            self.M2C = np.linalg.pinv(self.modes[self.pupil.reshape(-1), :]) @ Z
        else:
            self.M2C = np.eye(self.nValidAct)
        self.D_zonal = geometric_interaction_matrix(self.wfs, self.modes, cfg.stroke, self.wavelength)
        self.calib = calibration_vault(self.D_zonal @ self.M2C)
        self.reconstructor = self.M2C @ self.calib["M"]
        self.F = self.M2C @ np.linalg.pinv(self.M2C)
        self.wfs.measure(np.zeros((cfg.resolution, cfg.resolution)))

    def propagate(self):
        self.tel_OPD_no_pupil = self.tel_OPD_no_pupil + self.dm_OPD
        self.tel_OPD = self.tel_OPD_no_pupil * self.pupil
        self.phase = self.tel_OPD * 2 * np.pi / self.wavelength          # (with the pupil: Strehl)
        return self.wfs.measure(self.tel_OPD_no_pupil * 2 * np.pi / self.wavelength)
