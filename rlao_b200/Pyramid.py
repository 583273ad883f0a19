"""Pyramid — mirror of OOPAO/Pyramid.py for the configuration the drl4ao papyrus environment instantiates
(MAIN_CODE/OOPAOEnv/OOPAOEnv.py:239-249): 4-sided pyramid, PSF centred on four pixels, circular tip-tilt modulation,
`slopesMaps` post-processing; batched over environments (SURVEY.md section 8 f-3, first step).

The two transforms per modulation point (Pyramid.py:469-504: FFT of the padded field, focal-plane mask, inverse FFT),
the intensity accumulation over the modulation points and the detector binning run in the library's own kernels
(aoenv_pyramid_frames, csrc/pyr.cu: hand-written N = 16 x N2 transforms, no cuFFT) for the compiled transform sizes
(N = 128, 288), over chunks of environments that bound the workspaces.  Other sizes and the float64 calibration frames go
through `torch.fft`.  The quadrant arithmetic is batched tensor operations.  Detector noise uses the camera kernel of the
SH path (`Detector.integrate` -> aoenv_detector_integrate).  Parity is pinned through oracle/pyramid_oracle.py, itself
pinned against the unmodified reference (tests/golden/pyramid.npz).
Unsupported reference options raise NotImplementedError.
"""
import math

import numpy as np
import torch

from . import _lib
from .Detector import Detector


class Pyramid:
    def __init__(self, nSubap, telescope, modulation, lightRatio, postProcessing="slopesMaps", psfCentering=True,
                 n_pix_separation=2, calibModulation=50, n_pix_edge=None, extraModulationFactor=0, binning=1,
                 nTheta_user_defined=None, userValidSignal=None, old_mask=False, rooftop=None, delta_theta=0,
                 user_modulation_path=None, pupilSeparationRatio=None, edgePixel=None, zeroPadding=None,
                 max_points_per_pass=8):
        tel = telescope
        self.telescope = tel
        self.device = tel.device
        self.n_envs = tel.n_envs
        if (tel.resolution / nSubap) % 2 != 0:
            raise ValueError("The resolution should be an even number and be a multiple of 2**i where i>=2")
        if tel.src is None:
            raise AttributeError("The telescope was not coupled to any source object! Make sure to couple it with an src object using src*tel")
        if postProcessing not in ("slopesMaps", "slopesMaps_incidence_flux"):
            raise NotImplementedError(f"Pyramid(postProcessing={postProcessing!r}) is out of scope (full-frame signals)")
        for name, val, default in (("psfCentering", psfCentering, True),
                                   ("binning", binning, 1), ("userValidSignal", userValidSignal, None),
                                   ("old_mask", old_mask, False), ("rooftop", rooftop, None),
                                   ("user_modulation_path", user_modulation_path, None),
                                   ("pupilSeparationRatio", pupilSeparationRatio, None), ("edgePixel", edgePixel, None),
                                   ("zeroPadding", zeroPadding, None)):
            if val != default:
                raise NotImplementedError(f"Pyramid({name}={val!r}) is out of scope; only {default!r} is supported")
        self.tag = "pyramid"
        self.nSubap = int(nSubap)
        self.postProcessing = postProcessing
        self.psfCentering = True
        self.binning = 1
        self.delta_theta = delta_theta
        self.extraModulationFactor = extraModulationFactor
        self.nTheta_user_defined = nTheta_user_defined
        self.n_pix_separation = n_pix_separation
        self.n_pix_edge = n_pix_separation // 2 if n_pix_edge is None else n_pix_edge                 # Pyramid.py:237-240
        R = tel.resolution
        self.nRes = int((self.nSubap * 2 + self.n_pix_separation + self.n_pix_edge * 2) * R / self.nSubap)   # :250
        self.zeroPaddingFactor = self.nRes / R
        self.zeroPadding = (self.nRes - R) // 2
        self.center = self.nRes // 2
        self.cam = Detector(round(self.nSubap * self.zeroPaddingFactor))                              # :254
        self.lightRatio = lightRatio
        self.calibModulation = R / 2 - 1 if calibModulation >= R / 2 else calibModulation             # :258-261
        self.delta_Tip = self.delta_Tilt = 0
        self.fov = 206265 * self.nRes / self.zeroPaddingFactor * (tel.src.wavelength / tel.D)
        self.max_points_per_pass = int(max_points_per_pass)
        # step path: the library's own FFT kernels when the transform size is a compiled one (N = 128, 288: the 12 x 12 test
        # system and the 20 x 20 papyrus system); other sizes, and the float64 calibration frames, go through torch.fft
        self.use_kernels = True
        dev = self.device
        lin = np.linspace(-np.pi, np.pi, R)
        tip, tilt = np.meshgrid(lin, lin)                                                             # :285-288
        self._Tip = torch.as_tensor(tip * tel.pupil, dtype=torch.float64, device=dev)
        self._Tilt = torch.as_tensor(tilt * tel.pupil, dtype=torch.float64, device=dev)
        k = torch.arange(self.nRes, dtype=torch.float64, device=dev)
        ph1 = torch.polar(torch.ones_like(k), -math.pi * (self.nRes + 1) / self.nRes * k)             # :291-292, separable
        self._phasor = ph1[:, None] * ph1[None, :]
        self.m = self._phase_mask()
        self._mask = torch.polar(torch.ones_like(self.m), self.m)                                     # :318-323
        self.mask = self._mask
        self.slopesUnits = 1
        self.referenceSignal = 0
        self.referenceSignal_2D = 0
        self.isInitialized = self.isCalibrated = False
        self._signal64 = self._signal_2D = None
        self._signal_is_multi = False
        self._signal_planes = None                      # the environment's reconstruction GEMM splits `_signal` itself
        self.modulation = modulation
        self.initialization(tel)                                                                      # :301-303
        self._lds = (self.nSignal + 15) // 16 * 16
        self._signal = torch.zeros((self.n_envs, self._lds), dtype=torch.float32, device=self.device)
        self._stats = torch.zeros((self.n_envs, 4), dtype=torch.float64, device=self.device)
        self.modulation = modulation
        self.wfs_calibration(tel)
        tel.resetOPD()
        self.wfs_measure()

    # ---- static geometry ----------------------------------------------------------------------------------
    def _phase_mask(self):
        """Pyramid.py:368-388 (get_phase_mask, psf_centering=True)."""
        n_tot, nS = self.nRes, self.nSubap
        norma = (nS + self.n_pix_separation) * (self.telescope.resolution / nS)
        lim = np.pi / 4 - (np.pi / 4) / (n_tot // 2)
        tip, tilt = np.meshgrid(np.linspace(-lim, lim, n_tot // 2), np.linspace(-lim, lim, n_tot // 2))
        h = n_tot // 2
        m = np.zeros((n_tot, n_tot))
        m[:h, :h] = tip * norma + tilt * norma
        m[:h, -h:] = -tip * norma + tilt * norma
        m[-h:, -h:] = -tip * norma - tilt * norma
        m[-h:, :h] = tip * norma - tilt * norma
        return torch.as_tensor(-m, dtype=torch.float64, device=self.device)

    # ---- modulation ---------------------------------------------------------------------------------------
    @property
    def modulation(self):
        return self._modulation

    @modulation.setter
    def modulation(self, val):
        """Pyramid.py:941-984: modulation path, per-point tip/tilt phases; re-calibrates the reference slopes."""
        self._modulation = val
        if val >= self.telescope.resolution // 2:
            raise ValueError("Error the modulation radius is too large for this resolution! Consider using a larger telescope resolution!")
        if val != 0:
            perimeter = np.pi * 2 * val
            self.nTheta = (4 * int(self.extraModulationFactor + np.ceil(perimeter / 4)) if self.nTheta_user_defined is None
                           else self.nTheta_user_defined)
            self.thetaModulation = np.linspace(0 + self.delta_theta, 2 * np.pi + self.delta_theta, self.nTheta, endpoint=False)
            self.modulation_path = [[val * np.cos(t) + self.delta_Tip, val * np.sin(t) + self.delta_Tilt] for t in self.thetaModulation]
            px = torch.as_tensor([p[0] for p in self.modulation_path], dtype=torch.float64, device=self.device)
            py = torch.as_tensor([p[1] for p in self.modulation_path], dtype=torch.float64, device=self.device)
            # the reference keeps these phases in float32 (:960-961)
            self._phase_mod = (px[:, None, None] * self._Tip + py[:, None, None] * self._Tilt).to(torch.float32)
        else:
            self.nTheta = 1
            self._phase_mod = torch.zeros((1,) + tuple(self._Tip.shape), dtype=torch.float32, device=self.device)
        if getattr(self, "isCalibrated", False):
            self.slopesUnits = 1
            self.referenceSignal = 0
            self.referenceSignal_2D = 0
            self.wfs_calibration(self.telescope)

    # ---- propagation --------------------------------------------------------------------------------------
    def _frames(self, phase, precise=False):
        """phase [F, R, R] (radians, pupil-masked) -> detector frames [F, n_cam, n_cam] before the camera chain:
        sum over the modulation points of |IFFT(FFT(padded field * phasor) * mask)|^2 (Pyramid.py:469-504, 581-603),
        binned to the detector pixels (:987-1002, tools.py:409-416)."""
        tel = self.telescope
        R, N, F = tel.resolution, self.nRes, phase.shape[0]
        rdt, cdt = (torch.float64, torch.complex128) if precise else (torch.float32, torch.complex64)
        amp = (torch.as_tensor(np.sqrt(tel.src.fluxMap / self.nTheta) * tel.pupilReflectivity, device=self.device)).to(rdt)
        phasor, mask = self._phasor.to(cdt), self._mask.to(cdt)
        lo = self.center - R // 2
        out = torch.zeros((F, N, N), dtype=rdt, device=self.device)
        step = max(1, self.max_points_per_pass)
        for t0 in range(0, self.nTheta, step):
            pm = self._phase_mod[t0:t0 + step].to(rdt)                                     # [T, R, R]
            field = torch.polar(amp.expand(F, pm.shape[0], R, R), phase.to(rdt)[:, None] + pm[None])
            support = torch.zeros((F, pm.shape[0], N, N), dtype=cdt, device=self.device)
            support[:, :, lo:lo + R, lo:lo + R] = field
            ft = torch.fft.fft2(support * phasor)
            out += (torch.fft.ifft2(ft * mask).abs() ** 2).sum(dim=1)
        n, b = self.cam.resolution, int(round(N / self.cam.resolution))
        return out.reshape(F, n, b, n, b).sum(dim=(2, 4))

    def _kernel_tables(self):
        """Operands of aoenv_pyramid_frames for the current modulation: mask in the transform's digit-scrambled order
        (position j1 N2 + j2 holds frequency j1 + 16 j2, N = 16 N2), tilt ramp, modulation path, amplitude."""
        key = (self.nTheta, float(self._modulation), getattr(self.telescope.src, "_flux_version", 0))
        if getattr(self, "_ktab_key", None) != key:
            tel, N, dev = self.telescope, self.nRes, self.device
            N1, N2 = 16, N // 16
            pos = np.arange(N)
            perm = torch.as_tensor((pos // N2) + N1 * (pos % N2), device=dev)
            mask_s = self._mask.to(torch.complex64)[perm][:, perm].contiguous()
            path = np.asarray(self.modulation_path, dtype=np.float32) if self._modulation != 0 else np.zeros((1, 2), dtype=np.float32)
            amp = np.sqrt(tel.src.fluxMap / self.nTheta) * tel.pupilReflectivity
            self._ktab = dict(
                mask_s=torch.view_as_real(mask_s).contiguous(),
                lin=torch.as_tensor(np.linspace(-np.pi, np.pi, tel.resolution), dtype=torch.float32, device=dev),
                mod=torch.as_tensor(path, dtype=torch.float32, device=dev).contiguous(),
                amp=torch.as_tensor(amp, dtype=torch.float32, device=dev).contiguous())
            self._ktab_key = key
        return self._ktab

    @staticmethod
    def frames_chunk(nTheta, N, R):
        """Most environments per aoenv_pyramid_frames call: the workspaces (nTheta transforms of N x R and N x N complex
        values, one N x N intensity per environment) stay within 2 GiB."""
        return max(1, (2 << 30) // (nTheta * N * (N + R) * 8 + N * N * 4))

    def _frames_kernels(self, opd_a, opd_b):
        """Detector frames [F, n_cam, n_cam] of OPD_no_pupil = opd_a (+ opd_b) through the library's own transform kernels
        (aoenv_pyramid_frames: hand-written N = 16 x N2 FFTs, no cuFFT), environments in chunks that bound the workspaces."""
        tel, lib = self.telescope, _lib.load()
        R, N, F, dev = tel.resolution, self.nRes, opd_a.shape[0], self.device
        n_cam = self.cam.resolution
        tab = self._kernel_tables()
        chunk = min(F, self.frames_chunk(self.nTheta, N, R))
        ws = getattr(self, "_kernel_ws", None)
        if ws is None or ws[0] != (chunk, self.nTheta):
            ws = ((chunk, self.nTheta), torch.empty((chunk, self.nTheta, N, R, 2), dtype=torch.float32, device=dev),
                  torch.empty((chunk, self.nTheta, N, N, 2), dtype=torch.float32, device=dev),
                  torch.empty((chunk, N, N), dtype=torch.float32, device=dev))
            self._kernel_ws = ws
        out = torch.empty((F, n_cam, n_cam), dtype=torch.float32, device=dev)
        for s0 in range(0, F, chunk):
            m = min(chunk, F - s0)
            a = opd_a[s0:s0 + m].contiguous()
            b = None if opd_b is None else opd_b[s0:s0 + m].contiguous()
            _lib.check(lib.aoenv_pyramid_frames(
                _lib.ptr(a), _lib.ptr(b), _lib.ptr(tel._pupil_f), _lib.ptr(tab["amp"]), _lib.ptr(tab["lin"]), _lib.ptr(tab["mod"]),
                _lib.ptr(tab["mask_s"]), m, R, N, self.nTheta, N // n_cam, 2 * math.pi / tel.src.wavelength, _lib.ptr(ws[1]),
                _lib.ptr(ws[2]), _lib.ptr(ws[3]), _lib.ptr(out[s0:s0 + m]), _lib.stream_ptr(dev)), "pyramid_frames")
        return out

    def _kernels_ok(self):
        N, n_cam = self.nRes, self.cam.resolution
        return self.use_kernels and N % n_cam == 0 and bool(_lib.load().aoenv_pyramid_supported(N))

    def _camera(self, frames, env_offset=0):
        """self*self.cam (:987-1002): detector chain on the binned frames."""
        self.pyramidFrame = frames
        if self.cam.integrationTime is None:
            self.cam.integrationTime = self.telescope.samplingTime
        if self.cam.is_ideal():
            self.cam.frame = frames[0] if (self.n_envs == 1 and frames.shape[0] == 1) else frames
        else:
            self.cam._integrated_time += self.telescope.samplingTime       # Pyramid.py:989
            out = self.cam.integrate(frames.to(torch.float32), env_offset)
            self.cam.frame = out[0] if (self.n_envs == 1 and out.shape[0] == 1) else out
        return self.cam.frame

    def grabQuadrant(self, n, cameraFrame=None):
        """Pyramid.py:774-791 (4-sided pyramid, binning 1), on [..., n_cam, n_cam]."""
        f = self.cam.frame if cameraFrame is None else cameraFrame
        e = int(np.round(self.n_pix_separation / 2))
        c = int(np.round(self.cam.resolution / 2))
        m = int(np.ceil(self.nSubap))
        if n == 3:
            return f[..., e + c:e + c + m, e + c:e + c + m]
        if n == 4:
            return f[..., e + c:e + c + m, -e + c - m:-e + c]
        if n == 1:
            return f[..., -e + c - m:-e + c, -e + c - m:-e + c]
        if n == 2:
            return f[..., -e + c - m:-e + c, e + c:e + c + m]
        raise ValueError("quadrant index must be 1..4")

    def signalProcessing(self, cameraFrame=None):
        """Pyramid.py:685-726 (slopesMaps, slopesMaps_incidence_flux): returns (slopes maps [..., 2 nSubap, nSubap],
        slopes [..., nSignal])."""
        f = self.cam.frame if cameraFrame is None else cameraFrame
        v = self._valid_t.to(f.dtype)
        I1, I2, I3, I4 = (self.grabQuadrant(k, f) * v for k in (1, 2, 3, 4))
        I4Q = I1 + I2 + I3 + I4
        if self.postProcessing == "slopesMaps":                         # :689-691
            self.norma = I4Q[..., self._valid_t].mean(dim=-1)
        else:                                                           # :713-716 mean of the camera frame
            self.norma = f.mean(dim=(-2, -1))
        norma = self.norma[..., None, None] if I4Q.ndim == 3 else self.norma
        Sx = (I1 - I2 + I4 - I3) / norma
        Sy = (I1 - I4 + I2 - I3) / norma
        maps = (torch.cat([Sx, Sy], dim=-2) - self.referenceSignal_2D) * self.slopesUnits
        return maps, maps[..., self._valid_signal_t]

    # ---- reference-facing API -----------------------------------------------------------------------------
    def initialization(self, telescope):
        """Pyramid.py:408-450: valid pixels from the flux at a large modulation."""
        telescope.resetOPD()
        self.modulation = self.calibModulation
        zero = torch.zeros((1, telescope.resolution, telescope.resolution), dtype=torch.float64, device=self.device)
        self.initFrame = self._frames(zero, precise=True)[0]
        quads = [self.grabQuadrant(k, self.initFrame) for k in (1, 2, 3, 4)]
        self.I4Q = quads[0] + quads[1] + quads[2] + quads[3]
        self._valid_t = self.I4Q >= self.lightRatio * self.I4Q.max()
        self._valid_signal_t = torch.cat([self._valid_t, self._valid_t], dim=0)
        self.validI4Q = self._valid_t.cpu().numpy()
        self.validSignal = self._valid_signal_t.cpu().numpy()
        self.nSignal = int(self.validSignal.sum())
        self.isInitialized = True

    def wfs_calibration(self, telescope):
        """Pyramid.py:454-466: reference slopes of the flat wavefront at the working modulation (float64)."""
        zero = torch.zeros((1, telescope.resolution, telescope.resolution), dtype=torch.float64, device=self.device)
        frame = self._frames(zero, precise=True)[0]
        self.referenceSignal_2D = 0
        ref2d, ref = self.signalProcessing(frame)
        self.referenceSignal_2D, self.referenceSignal = ref2d, ref
        self.referencePyramidFrame = frame
        self.isCalibrated = True

    def wfs_measure(self, phase_in=None):
        """Pyramid.py:516-603, single-frame branches, for every environment (a stack of k wavefronts other than n_envs
        goes through the multi-frame branch :604-676 and yields signal [nSignal, k])."""
        tel = self.telescope
        lam = tel.src.wavelength
        if phase_in is not None:
            ph = torch.as_tensor(phase_in, dtype=torch.float32, device=self.device)
            tel.OPD = (ph.unsqueeze(0) if ph.ndim == 2 else ph) * (lam / (2 * math.pi))
        a, b = tel._terms()
        if a.shape[0] != self.n_envs:
            self._multi_signal = self.measure_frames(a if b is None else a + b)
            self._signal_is_multi = True
            return
        self._measure_terms(a, b)

    def _measure_terms(self, opd_a, opd_b, env_offset=None):
        """Per-environment measurement on OPD_no_pupil = opd_a (+ opd_b): what tel*wfs and the environment's step run.
        Also leaves the operands of the environment's reconstruction / reward kernels: `_signal` [B, lds] float32 (zero
        padded) and the pupil statistics `_stats` [B, 4] (sum and sum of squares of the atmosphere-only and of the total
        OPD inside the pupil, relative to the value at the pupil centre — the definition of aoenv_shwfs_frame)."""
        tel = self.telescope
        lam, R = tel.src.wavelength, tel.resolution
        env_offset = getattr(self, "env_offset", 0) if env_offset is None else env_offset
        if opd_b is not None and not torch.is_tensor(opd_b):
            opd_b = opd_b.tensor()                                  # DMSurfaceRef: the surface kernel runs now
        opd = opd_a if opd_b is None else opd_a + opd_b
        pupil = tel._pupil_f
        if self._kernels_ok() and opd_a.dtype == torch.float32:
            frames = self._frames_kernels(opd_a, opd_b)
        else:                                                           # transform sizes without a compiled kernel
            frames = self._frames(opd * pupil * (2 * math.pi / lam))
        self._camera(frames, env_offset)
        frame = self.cam.frame if self.cam.frame.ndim == 3 else self.cam.frame.unsqueeze(0)
        self._frame = frame
        maps, sig = self.signalProcessing(frame.to(torch.float64) if self.cam.is_ideal() else frame.to(torch.float32))
        self._signal_2D, self._signal64 = maps, sig
        self._signal[:, :self.nSignal] = sig.to(torch.float32)
        inside = pupil > 0
        ka = opd_a[:, R // 2, R // 2].double()[:, None]
        da = (opd_a.double().reshape(opd_a.shape[0], -1) - ka) * inside.reshape(-1)
        kt = opd[:, R // 2, R // 2].double()[:, None]
        dt = (opd.double().reshape(opd.shape[0], -1) - kt) * inside.reshape(-1)
        self._stats[:, 0], self._stats[:, 1] = da.sum(dim=1), (da * da).sum(dim=1)
        self._stats[:, 2], self._stats[:, 3] = dt.sum(dim=1), (dt * dt).sum(dim=1)
        self._signal_is_multi = False
        self.pyramidSignal_2D, self.pyramidSignal = self.signal_2D, self.signal

    def measure_frames(self, opd):
        """Multi-frame branch (Pyramid.py:604-676): k wavefronts [k, R, R] (OPD_no_pupil, metres), ideal detector, every
        frame processed on its own.  Returns signal [k, nSignal] in float64 (the calibration path)."""
        if not self.cam.is_ideal() and (self.cam.photonNoise or self.cam.readoutNoise):
            raise NotImplementedError("noisy multi-frame measurements are not supported (calibrate with noise='off')")
        tel = self.telescope
        out = []
        for s0 in range(0, opd.shape[0], 16):                      # bounded memory: 16 wavefronts x nTheta points per pass
            ph = opd[s0:s0 + 16].double() * tel._pupil_f.double() * (2 * math.pi / tel.src.wavelength)
            out.append(self.signalProcessing(self._frames(ph, precise=True))[1])
        return torch.cat(out, dim=0)

    def pyramid_propagation(self, telescope):
        self.wfs_measure()

    @property
    def signal(self):
        if self._signal_is_multi:
            return self._multi_signal.T                                # [nSignal, k] as Pyramid.py:676
        return self._signal64[0] if self.n_envs == 1 else self._signal64

    @property
    def signal_2D(self):
        return self._signal_2D[0] if self.n_envs == 1 else self._signal_2D

    def __mul__(self, obj):
        if getattr(obj, "tag", None) != "detector":
            raise AttributeError("Error light propagated to the wrong type of object")
        self._camera(self.pyramidFrame)
        return -1
