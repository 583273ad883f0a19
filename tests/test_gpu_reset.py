"""Episode reset on the device (aoenv_vk_screens: Philox spectrum -> two DFT-matrix GEMMs on the tensor cores ->
sub-harmonics; OOPAO/phaseStats.py:190-318 via Atmosphere.generateNewPhaseScreen, OOPAO/Atmosphere.py:560-592):
bit-for-bit the reference's algorithm on injected Gaussian draws, and the right statistics with its own generator."""
import numpy as np
import pytest
import torch
from numpy.random import RandomState

from oracle.golden_configs import CONFIGS
from parity_util import rel_err

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("needs a CUDA device")
    return torch.device("cuda:0")


def _synth_screens(synth, S, seed=1, screen0=0, inject=None):
    N = synth.N
    out = torch.zeros((S, N, N), dtype=torch.float32, device=synth.device)
    synth.generate(seed, screen0, S, out.data_ptr(), N, N * N, inject=inject)
    torch.cuda.synchronize()
    return out


@pytest.mark.parametrize("R", [42, 48, 120, 240])          # (N = R + 4: 46 = 2 mod 4, the others 0 mod 4)
def test_screens_from_injected_draws_equal_the_reference_algorithm(dev, R):
    """The reference draws normal(size=(N,N)) twice from RandomState(seed) (real, imaginary parts) and reuses the head of the
    same stream for the sub-harmonics; fed with those draws the device path must reproduce its screens."""
    from rlao_b200.tools import vonkarman as vk
    N, delta, r0, L0 = R + 4, 8.0 / R, 0.13, 25.0
    synth = vk.ScreenSynth(r0, L0, N, delta, dev)
    seeds = [17, 18, 1017]
    inj = np.zeros((len(seeds), 2, N, N), dtype=np.float32)
    want = []
    for k, sd in enumerate(seeds):
        rs = RandomState(sd)
        inj[k, 0], inj[k, 1] = rs.normal(size=(N, N)), rs.normal(size=(N, N))
        want.append(vk.screen_reference_rng(r0, L0, N, delta, sd))
    got = _synth_screens(synth, len(seeds), inject=inj).double().cpu().numpy()
    for k in range(len(seeds)):
        assert rel_err(got[k], want[k]) < 2e-5, (R, seeds[k])


def test_philox_screens_have_the_reference_statistics(dev):
    """40 x 40 system (N = 244): structure function of 512 device screens against 96 screens of the reference algorithm
    with its own MT19937 streams; independence between screens, shards and seeds."""
    from rlao_b200.tools import vonkarman as vk
    R = 240
    N, delta, r0, L0 = R + 4, 8.0 / R, 0.13, 25.0
    synth = vk.ScreenSynth(r0, L0, N, delta, dev)
    a = _synth_screens(synth, 512, seed=5).double()
    assert torch.isfinite(a).all()
    ref = np.stack([vk.screen_reference_rng(r0, L0, N, delta, 1000 + k) for k in range(96)])
    for sep in (1, 4, 16, 60, 150):
        dx = float(((a[:, :, sep:] - a[:, :, :-sep]) ** 2).mean())
        dy = float(((a[:, sep:, :] - a[:, :-sep, :]) ** 2).mean())
        wx = ((ref[:, :, sep:] - ref[:, :, :-sep]) ** 2).mean()
        wy = ((ref[:, sep:, :] - ref[:, :-sep, :]) ** 2).mean()
        tol = 0.06 if sep <= 16 else 0.15
        assert abs(dx / wx - 1) < tol and abs(dy / wy - 1) < tol, (sep, dx / wx, dy / wy)
    assert abs(float(a.var()) / ref.var() - 1) < 0.15
    # independent streams: other screens, other shard offset, other seed
    # (first differences: the screens themselves are dominated by a handful of large-scale modes, which correlate by chance)
    d = (a[:64, :, 1:] - a[:64, :, :-1]).reshape(64, -1)[:, ::5].cpu().numpy()
    c = np.corrcoef(d)
    assert np.abs(c - np.eye(64)).max() < 0.3 and np.abs(c - np.eye(64)).mean() < 0.06
    b = _synth_screens(synth, 4, seed=5, screen0=512)
    assert not torch.equal(b[0].double(), a[0])
    again = _synth_screens(synth, 4, seed=5, screen0=0)
    # counter-based: screen s of seed 5 does not depend on the batch it is generated in (to GEMM rounding: the small batch
    # takes the split-K path of the tensor-core kernel)
    assert rel_err(again.double().cpu().numpy(), a[:4].cpu().numpy()) < 1e-5
    other = _synth_screens(synth, 4, seed=6)
    assert not torch.equal(other.double(), a[:4])


def test_generate_new_phase_screen_runs_on_the_device(dev):
    """Atmosphere.generateNewPhaseScreen in the production mode (rng='philox'): with the reference-mode draws injected it
    leaves the reference-mode screens in the layer maps (interior; the ring is extruded from each mode's own innovations)."""
    from rlao_b200 import _lib
    from rlao_b200.Atmosphere import Atmosphere
    from rlao_b200.Source import Source
    from rlao_b200.Telescope import Telescope
    cfg = CONFIGS["tiny"]()
    B = 2

    def build(rng):
        tel = Telescope(cfg.resolution, cfg.diameter, cfg.samplingTime, n_envs=B, device=dev)
        Source(cfg.opticalBand, cfg.magnitude) * tel
        atm = Atmosphere(tel, cfg.r0, cfg.L0, cfg.windSpeed, cfg.fractionalR0, cfg.windDirection, cfg.altitude, rng=rng)
        atm.initializeAtmosphere(tel)
        return atm
    ref, phx = build("reference"), build("philox")
    N = ref._ops.layer_res
    seed = 31
    ref.generateNewPhaseScreen(seed)
    inj = []
    for i in range(ref.nLayer):
        z = np.zeros((B, 2, N, N), dtype=np.float32)
        for e in range(B):
            rs = RandomState(seed + i + 104729 * e)           # Atmosphere._new_screens, reference mode
            z[e, 0], z[e, 1] = rs.normal(size=(N, N)), rs.normal(size=(N, N))
        inj.append(z)
    phx.screen_inject = inj
    n0 = _lib.launch_count()
    phx.generateNewPhaseScreen(seed)
    assert _lib.launch_count() - n0 >= 5 * ref.nLayer          # spectrum, GEMM, transpose, GEMM, finish per layer
    for i in range(ref.nLayer):
        a = ref._layers[i].mapShift[:, 1:-1, 1:-1].double().cpu().numpy()
        b = phx._layers[i].mapShift[:, 1:-1, 1:-1].double().cpu().numpy()
        assert rel_err(b, a) < 2e-5, i
    phx.screen_inject = None
    phx.generateNewPhaseScreen(seed)                           # own generator: different, finite, same scale
    m = phx._layers[0].mapShift.double()
    assert torch.isfinite(m).all() and 0.2 < float(m.std()) / float(ref._layers[0].mapShift.double().std()) < 5
