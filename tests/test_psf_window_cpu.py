"""The float64 matrix-DFT window of the science PSF (parity_util.psf_window_f64), which the batched-step replay compares the
PSF-peak kernels with, against the reference definition oracle.ao_oracle.compute_psf: central crop and maximum."""
import numpy as np
import pytest
import torch

from oracle.ao_oracle import compute_psf, flux_map, source_properties, telescope_pupil
from oracle.golden_configs import psf_formula_opd
from parity_util import psf_window_f64, rel_err


@pytest.mark.parametrize("R,zp,window,screens", [
    (48, 4, 32, 3),              # the tiny system
    (48, 2, 16, 1),
    (480, 4, 32, 1),             # cfg5psf: N = 3840, oversampling 2
])
def test_matrix_dft_window_equals_compute_psf(R, zp, window, screens):
    pupil = telescope_pupil(R)
    wl, nph = source_properties("I", 8.0)
    fm = flux_map(pupil, nph, 1.0 / 500, 8.0)
    rng = np.random.default_rng(R + zp)
    # a smooth aberration several radians deep, a piston of tens of radians and a rough part: light spread over the window
    phases = np.stack([(psf_formula_opd(R) * 2 * np.pi / wl * (1 + 4 * s) + 30.0 * (s + 1)
                        + rng.normal(0, 0.3, (R, R))) * pupil for s in range(screens)])
    got = psf_window_f64(torch.as_tensor(np.sqrt(fm)), torch.as_tensor(phases), zp, window).numpy()
    for s in range(screens):
        psf = compute_psf(pupil, fm, phases[s], zp)
        c = psf.shape[0] // 2
        want = psf[c - window // 2:c + window // 2, c - window // 2:c + window // 2]
        assert rel_err(got[s], want) < 1e-12, s
        assert abs(got[s].max() - want.max()) < 1e-12 * want.max(), s
