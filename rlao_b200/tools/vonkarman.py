"""Host-side (float64) construction of the von Karman operators and initial screens — init-time only.

Formulas: OOPAO/phaseStats.py:70-133 (covariance with Bessel K_5/6), :190-318 (FFT + sub-harmonic screens,
Schmidt 2010 / Lane 1992); OOPAO/Atmosphere.py:263-286,485-558 (Assemat 2006 predictor A and innovation factor B).
The heavy linear algebra (pinv, Cholesky) runs on the GPU in float64 through torch.linalg.
"""
import math

import numpy as np
import torch

from . import linalg
from numpy.random import RandomState
from scipy.special import kv


def _vk_cov(z1, z2, L0, r0):
    rho = np.abs(z1[:, None] - z2[None, :])
    ratio = (L0 / r0) ** (5.0 / 3)
    c0 = (24.0 * math.gamma(6.0 / 5) / 5) ** (5.0 / 6)
    cst = c0 * math.gamma(11.0 / 6) / (2.0 ** (5.0 / 6) * math.pi ** (8.0 / 3)) * ratio
    var = c0 * math.gamma(11.0 / 6) * math.gamma(5.0 / 6) / (2 * math.pi ** (8.0 / 3)) * ratio
    out = np.full(rho.shape, var)
    nz = rho != 0
    u = 2 * math.pi * rho[nz] / L0
    out[nz] = cst * u ** (5.0 / 6) * kv(5.0 / 6, u)
    return out


def ring_geometry(layer_res, nExtra=2):
    """Boolean masks of the outer ring and of the two rings inside it on the (layer_res+nExtra)^2 map, plus
    their (row, col) lists in numpy boolean-mask order (Atmosphere.py:263-276)."""
    M = layer_res + nExtra
    outer = np.ones((M, M), dtype=bool)
    outer[1:-1, 1:-1] = False
    inner = ~outer
    inner[1 + nExtra:-1 - nExtra, 1 + nExtra:-1 - nExtra] = False
    return outer, inner, np.argwhere(outer).astype(np.int32), np.argwhere(inner).astype(np.int32)


class VKOperators:
    """A, B and the r0-independent covariances they come from."""

    def __init__(self, tel_resolution, diameter, L0, r0, r0_def, device):
        self.r0_def = r0_def
        self.layer_res = tel_resolution + 4                       # Atmosphere.py:218 (fov = 0)
        self.layer_D = self.layer_res * diameter / tel_resolution
        self.outer, self.inner, self.outer_rc, self.inner_rc = ring_geometry(self.layer_res)
        l = np.linspace(0, self.layer_res + 1, self.layer_res + 2) * self.layer_D / (self.layer_res - 1)
        u, v = np.meshgrid(l, l)
        zi = u[self.inner] + 1j * v[self.inner]
        zo = u[self.outer] + 1j * v[self.outer]
        f64 = dict(dtype=torch.float64, device=device)
        ZZt = torch.as_tensor(_vk_cov(zi, zi, L0, r0_def), **f64)
        self.ZXt = torch.as_tensor(_vk_cov(zi, zo, L0, r0_def), **f64)
        self.XXt = torch.as_tensor(_vk_cov(zo, zo, L0, r0_def), **f64)
        ZZt_inv = linalg.pinv(ZZt)
        s = (r0_def / r0) ** (5.0 / 3)
        self.A = (self.ZXt * s).T @ (ZZt_inv / s)
        self.B = self.innovation_factor(r0)

    def innovation_factor(self, r0):
        s = (self.r0_def / r0) ** (5.0 / 3)
        return torch.linalg.cholesky(self.XXt * s - self.A @ (self.ZXt * s))


def _psd(f, r0, L0, l0):
    fm = 5.92 / l0 / (2 * math.pi)
    return 0.023 * r0 ** (-5.0 / 3) * np.exp(-((f / fm) ** 2)) / ((f ** 2 + (1.0 / L0) ** 2) ** (11.0 / 6))


def screen_reference_rng(r0, L0, N, delta, seed, l0=1e-10):
    """One screen with the reference's MT19937 streams (numpy RandomState(seed) for both the FFT part and the
    sub-harmonics, phaseStats.py:268,272) — used for parity runs and small batches."""
    rs_hi, rs_lo = RandomState(seed), RandomState(seed)
    del_f = 1.0 / (N * delta)
    fx = np.arange(-N / 2.0, N / 2.0) * del_f
    fx, fy = np.meshgrid(fx, fx)
    psd = _psd(np.sqrt(fx ** 2 + fy ** 2), r0, L0, l0)
    psd[N // 2, N // 2] = 0
    cn = (rs_hi.normal(size=(N, N)) + 1j * rs_hi.normal(size=(N, N))) * np.sqrt(psd) * del_f
    hi = np.fft.fftshift(np.fft.fft2(np.fft.fftshift(cn))).real
    D = N * delta
    c = np.arange(-N / 2, N / 2) * delta
    x, y = np.meshgrid(c, c)
    lo = np.zeros((N, N), dtype=complex)
    for p in range(1, 4):
        df = 1 / (3 ** p * D)
        gx, gy = np.meshgrid(np.arange(-1, 2) * df, np.arange(-1, 2) * df)
        ps = _psd(np.sqrt(gx ** 2 + gy ** 2), r0, L0, l0)
        ps[1, 1] = 0
        cs = (rs_lo.normal(size=(3, 3)) + 1j * rs_lo.normal(size=(3, 3))) * np.sqrt(ps) * df
        for i in range(2):
            for j in range(2):
                lo += cs[i, j] * np.exp(1j * 2 * np.pi * (gx[i, j] * x + gy[i, j] * y))
    lo = lo.real - lo.real.mean()
    return lo + hi


def screens_device_rng(r0, L0, N, delta, n, generator, device, l0=1e-10):
    """`n` independent screens of the same statistics, drawn with torch's device generator (Philox) and
    transformed with torch.fft — the large-batch path.  Returns float32 [n, N, N]."""
    del_f = 1.0 / (N * delta)
    fx = np.arange(-N / 2.0, N / 2.0) * del_f
    fx, fy = np.meshgrid(fx, fx)
    psd = _psd(np.sqrt(fx ** 2 + fy ** 2), r0, L0, l0)
    psd[N // 2, N // 2] = 0
    amp = torch.as_tensor(np.sqrt(psd) * del_f, dtype=torch.float32, device=device)
    out = torch.empty((n, N, N), dtype=torch.float32, device=device)
    D = N * delta
    c = torch.as_tensor(np.arange(-N / 2, N / 2) * delta, dtype=torch.float32, device=device)
    chunk = max(1, min(n, (1 << 26) // (N * N)))
    for s in range(0, n, chunk):
        m = min(chunk, n - s)
        re = torch.randn((m, N, N), generator=generator, device=device)
        im = torch.randn((m, N, N), generator=generator, device=device)
        cn = torch.complex(re, im) * amp
        hi = torch.fft.fftshift(torch.fft.fft2(torch.fft.fftshift(cn, dim=(-2, -1))), dim=(-2, -1)).real
        lo = torch.zeros((m, N, N), dtype=torch.complex64, device=device)
        for p in range(1, 4):
            df = 1 / (3 ** p * D)
            g = np.arange(-1, 2) * df
            gx, gy = np.meshgrid(g, g)
            ps = _psd(np.sqrt(gx ** 2 + gy ** 2), r0, L0, l0)
            ps[1, 1] = 0
            a = torch.as_tensor(np.sqrt(ps) * df, dtype=torch.float32, device=device)
            cs = torch.complex(torch.randn((m, 3, 3), generator=generator, device=device),
                               torch.randn((m, 3, 3), generator=generator, device=device)) * a
            for i in range(2):
                for j in range(2):
                    ex = torch.polar(torch.ones_like(c), 2 * math.pi * float(gx[i, j]) * c)     # along x (columns)
                    ey = torch.polar(torch.ones_like(c), 2 * math.pi * float(gy[i, j]) * c)     # along y (rows)
                    lo += cs[:, i, j, None, None] * (ey[:, None] * ex[None, :])
        lo = lo.real - lo.real.mean(dim=(-2, -1), keepdim=True)
        out[s:s + m] = lo + hi
    return out


class ScreenSynth:
    """Device-side synthesis of the episode's first screens (aoenv_vk_screens: Philox spectrum, two DFT-matrix GEMMs on the
    tensor cores, sub-harmonics) — OOPAO/phaseStats.py:190-318 for a batch of screens.  Holds the operators of one
    (r0, L0, N, delta): signed spectral amplitude, the two DFT operators in split-bf16 form, the sub-harmonic tables."""

    def __init__(self, r0, L0, N, delta, device, parts=3, l0=1e-10):
        from .. import gemm
        self.N, self.parts, self.device = int(N), parts, device
        N = self.N
        del_f = 1.0 / (N * delta)
        f1 = np.arange(-N / 2.0, N / 2.0) * del_f
        fx, fy = np.meshgrid(f1, f1)
        psd = _psd(np.sqrt(fx ** 2 + fy ** 2), r0, L0, l0)
        psd[N // 2, N // 2] = 0
        k = np.arange(N)
        sign = 1.0 - 2.0 * ((k[:, None] + k[None, :]) % 2)
        t32 = lambda a: torch.as_tensor(np.ascontiguousarray(a), dtype=torch.float32, device=device)
        self.amp = t32(np.sqrt(psd) * del_f * sign)
        # W[y][a] = (-1)^y exp(-2 pi i y a / N), exponent reduced mod N in integers
        ang = -2.0 * np.pi * ((k[:, None] * k[None, :]) % N) / N
        sy = (1.0 - 2.0 * (k % 2))[:, None]
        Wr, Wi = np.cos(ang) * sy, np.sin(ang) * sy
        self.Kp = (2 * N + 15) // 16 * 16
        WA = np.zeros((2 * N, self.Kp))
        WA[:N, :N], WA[:N, N:2 * N] = Wr, -Wi           # Ur = Gr Wr - Gi Wi
        WA[N:, :N], WA[N:, N:2 * N] = Wi, Wr            # Ui = Gr Wi + Gi Wr
        WB = np.zeros((N, self.Kp))
        WB[:, :N], WB[:, N:2 * N] = Wr, -Wi             # Re(U W)
        self.WA, self.WB = gemm.Operator(t32(WA), parts=parts), gemm.Operator(t32(WB), parts=parts)
        # sub-harmonic grids p = 1..3: frequencies (j - 1) df along x, (i - 1) df along y, only i, j in {0, 1} are used
        D = N * delta
        c = np.arange(-N / 2, N / 2) * delta
        ex = np.zeros((3, 2, N), dtype=complex)
        amp_lo = np.zeros((3, 2, 2))
        for p in range(1, 4):
            df = 1 / (3 ** p * D)
            g = np.arange(-1, 2) * df
            gx, gy = np.meshgrid(g, g)
            ps = _psd(np.sqrt(gx ** 2 + gy ** 2), r0, L0, l0)
            ps[1, 1] = 0
            amp_lo[p - 1] = (np.sqrt(ps) * df)[:2, :2]
            for j in range(2):
                ex[p - 1, j] = np.exp(2j * np.pi * g[j] * c)
        pack = lambda z: np.stack([z.real, z.imag], axis=-1)
        self.sh_ex = t32(pack(ex))                      # the y tables are the same numbers (square grid)
        self.h_amp = np.ascontiguousarray(amp_lo, dtype=np.float32)
        self.h_mean = np.ascontiguousarray(pack(ex.mean(axis=2)), dtype=np.float32)

    def generate(self, seed, screen0, S, dst_ptr, pitch, env_stride, inject=None, env_idx=None):
        """Writes S screens into the windows starting at device address dst_ptr (row 1 / column 1 of environment 0); with
        env_idx (int32 device tensor of S environments), screen s goes to environment env_idx[s] from its stream
        screen0 + env_idx[s] (aoenv_vk_screens_envs)."""
        import ctypes as C
        from .. import _lib
        lib, N, Kp, dev = _lib.load(), self.N, self.Kp, self.device
        lda, ldb = (2 * N + 3) // 4 * 4, (N + 3) // 4 * 4
        per_screen = self.parts * N * Kp * 2 + N * (lda + ldb) * 4
        chunk = max(1, min(S, 32767, (768 << 20) // per_screen))
        planes = torch.empty((self.parts, chunk * N, Kp), dtype=torch.bfloat16, device=dev)
        wa = torch.empty((chunk * N, lda), dtype=torch.float32, device=dev)
        wb = torch.empty((chunk * N, ldb), dtype=torch.float32, device=dev)
        f = lambda a: a.ctypes.data_as(C.c_void_p)
        for s0 in range(0, S, chunk):
            m = min(chunk, S - s0)
            if env_idx is not None:
                _lib.check(lib.aoenv_vk_screens_envs(
                    C.c_uint64(seed & 0xFFFFFFFFFFFFFFFF), C.c_uint32(screen0 & 0xFFFFFFFF), _lib.ptr(env_idx[s0:s0 + m]), m, N,
                    _lib.ptr(self.amp), _lib.ptr(self.WA.planes()), _lib.ptr(self.WB.planes()), Kp, self.parts,
                    _lib.ptr(self.sh_ex), _lib.ptr(self.sh_ex), f(self.h_amp), f(self.h_mean), f(self.h_mean), _lib.ptr(planes),
                    _lib.ptr(wa), lda, _lib.ptr(wb), ldb, dst_ptr, pitch, env_stride, _lib.stream_ptr(dev)), "vk_screens_envs")
                continue
            inj = None
            if inject is not None:
                inj = torch.as_tensor(inject[s0:s0 + m], dtype=torch.float32, device=dev).contiguous()
            _lib.check(lib.aoenv_vk_screens(
                C.c_uint64(seed & 0xFFFFFFFFFFFFFFFF), C.c_uint32((screen0 + s0) & 0xFFFFFFFF), m, N, _lib.ptr(self.amp),
                _lib.ptr(inj), _lib.ptr(self.WA.planes()), _lib.ptr(self.WB.planes()), Kp, self.parts, _lib.ptr(self.sh_ex),
                _lib.ptr(self.sh_ex), f(self.h_amp), f(self.h_mean), f(self.h_mean), _lib.ptr(planes), _lib.ptr(wa), lda,
                _lib.ptr(wb), ldb, dst_ptr + 4 * s0 * env_stride, pitch, env_stride, _lib.stream_ptr(dev)), "vk_screens")


def cubic_tap_weights(buff, kernel="lagrange018"):
    """Tap offset (relative to the output pixel) and the four float64 weights of the separable cubic
    interpolation that shifts a map by `buff` pixels (|buff| < 1) along one axis.

    lagrange018 = scikit-image 0.18.3 `bicubic_interpolation` (interpolation.pxd): taps floor(r)-1..floor(r)+2
    combined by the cubic through 4 equispaced nodes, argument (r - first_tap)/3.
    catmull_rom = scikit-image >= 0.19.  Input coordinate of output pixel i is r = i - buff."""
    f = math.floor(-buff)                     # floor(r) - i
    frac = -buff - f                          # in [0, 1)
    off = f - 1
    if kernel == "lagrange018":
        x = (frac + 1.0) / 3.0
        w = [1.0 + x * (-5.5 + x * (9.0 + x * -4.5)), x * (9.0 + x * (-22.5 + x * 13.5)),
             x * (-4.5 + x * (18.0 + x * -13.5)), x * (1.0 + x * (-4.5 + x * 4.5))]
    elif kernel == "catmull_rom":
        x = frac
        w = [0.5 * x * (-1.0 + x * (2.0 - x)), 1.0 + 0.5 * x * x * (-5.0 + 3.0 * x),
             0.5 * x * (1.0 + x * (4.0 - 3.0 * x)), 0.5 * x * x * (x - 1.0)]
    else:
        raise ValueError(f"unknown interpolation kernel {kernel!r}")
    return off, w
