"""Pins the CPU oracle (oracle/ao_oracle.py) against fixtures produced by the UNMODIFIED reference
(tests/golden/*.npz, written by oracle/make_golden.py in the build container)."""
import numpy as np

from oracle.make_golden import load
from oracle.replay import replay_oracle

# digests accumulate ~1e3 terms of mixed sign; traces go through a pinv/SVD chain
RTOL = {"default": 1e-8, "digest": 1e-7}


def _check(name, golden_dir):
    ref = load(name, golden_dir)
    got, _ = replay_oracle(name)
    assert set(ref) == set(got)
    for k in ref:
        a, b = np.asarray(ref[k]), np.asarray(got[k])
        assert a.shape == b.shape, k
        if a.dtype == np.uint8 or a.dtype == bool:
            assert np.array_equal(a, b), k
            continue
        rtol = RTOL["digest"] if "digest" in k else RTOL["default"]
        if a.dtype == np.float32:                      # large fixtures keep float32 snapshots
            rtol = max(rtol, 2e-7)
        scale = max(float(np.abs(a).max()), 1e-300)
        err = np.abs(a.astype(float) - b.astype(float)).max() / scale
        assert err <= rtol, f"{name}:{k} rel err {err:.3e}"


def test_oracle_matches_reference_tiny(golden_dir):
    _check("tiny", golden_dir)


def test_oracle_matches_reference_cfg1(golden_dir):
    _check("cfg1", golden_dir)


def test_oracle_matches_reference_cfg3(golden_dir):
    """The benchmark configuration itself (40x40 SH, 41x41 DM, three layers), one environment, 8 closed-loop steps."""
    _check("cfg3", golden_dir)


def test_oracle_matches_reference_noisy_detector_bit_exact(golden_dir):
    """Razor-like detector (photon + read + dark noise, QE, FWC, 10-bit ADC) with the reference's three
    RandomState streams seeded: the integer camera frames must agree exactly."""
    name = "tiny_noise"
    ref = load(name, golden_dir)
    got, _ = replay_oracle(name)
    for k in ("frame0", "frame_0", f"frame_{ref['snap_steps'][1]}", f"frame_{ref['snap_steps'][2]}"):
        assert np.array_equal(np.asarray(ref[k]).astype(np.int64), np.asarray(got[k]).astype(np.int64)), k
    np.testing.assert_allclose(got["trace_signal"], ref["trace_signal"], rtol=0, atol=1e-7 * np.abs(ref["trace_signal"]).max())
    np.testing.assert_allclose(got["trace_strehl"], ref["trace_strehl"], rtol=1e-8)
