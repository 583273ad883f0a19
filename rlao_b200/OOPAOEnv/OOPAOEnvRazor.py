"""Gym-style closed-loop AO environment — mirror of MAIN_CODE/OOPAOEnv/OOPAOEnvRazor.py `class OOPAO`
(Shack-Hartmann branch; twin of OOPAOEnv.py), stepping `n_envs` independent environments in lock-step on one GPU.

    env = OOPAO(); env.set_params_file(param_file, oopao_path); env.set_params(args, "shackhartmann", n_envs=1024)
    obs = env.reset_soft()
    obs, reward, strehl, done, info = env.step(i, action)

`step` follows OOPAOEnvRazor.py:474-514 line by line but never leaves the device: seven kernel launches per
step plus one GEMM-triple per integer-pixel wind shift (see DESIGN.md).  Arrays carry a leading n_envs
dimension (squeezed when n_envs == 1); rewards / Strehl ratios are tensors of shape [n_envs].
"""
import contextlib
import ctypes
import importlib
import math
import os
import types

import numpy as np
import torch

from .. import _lib, gemm
from ..Atmosphere import Atmosphere
from ..DeformableMirror import DeformableMirror, DMSurfaceRef
from ..MisRegistration import MisRegistration
from ..ShackHartmann import ShackHartmann
from ..Source import Source
from ..Telescope import Telescope
from ..Zernike import Zernike
from ..calibration.CalibrationVault import CalibrationVault
from ..calibration.InteractionMatrix import InteractionMatrix
from ..tools import linalg


_NVTX = os.environ.get("AOENV_NVTX", "0") not in ("", "0")


@contextlib.contextmanager
def _range(name):
    """NVTX range around a stage of the step when AOENV_NVTX=1 (timeline profilers); free otherwise."""
    if _NVTX:
        torch.cuda.nvtx.range_push(name)
        try:
            yield
        finally:
            torch.cuda.nvtx.range_pop()
    else:
        yield


class OOPAO:
    metadata = {"render.modes": ["rgb_array"]}

    def __init__(self):
        self.gainCL = None
        self.atm = self.wfs = self.dm = self.misReg = self.tel = self.source = None
        self.M2C_CL = self.calib_CL = self.reconstructor = None
        self.SR = self.total = self.residual = self.wfsSignal = self.OPD = None
        self.action_buffer = []
        self.done = False
        self.param_file = ""
        self.oopao_path = ""
        self.delay = 1
        self.F = 1
        self.name = "OOPAO"
        self.dm_mask = self.nActuator = self.xvalid = self.yvalid = None
        self.leak = 0.99
        self.n_envs = 1
        self.device = None
        self.psf_reward = None        # (zeroPaddingFactor, window) -> Strehl from the PSF peak each step
        self.native_step = os.environ.get("AOENV_STEP_NATIVE", "1") != "0"   # step() as two library calls when it can
        # device-resident steps issue the next frame's atmosphere before the spots of this frame (see _step_native)
        self.prefetch_early = os.environ.get("AOENV_PREFETCH_EARLY", "1") != "0"
        self._native_key, self._native = None, None

    # ---- configuration ------------------------------------------------------------------------------------
    def set_params_file(self, param_file, oopao_path):
        self.param_file = param_file
        self.oopao_path = oopao_path

    def _load_param(self, args):
        if isinstance(self.param_file, dict):
            return dict(self.param_file)
        name = self.param_file or "rlao_b200.Conf.parameter_file_synthetic_SHWFS"
        try:
            config = importlib.import_module(name)
        except ModuleNotFoundError:
            config = importlib.import_module("rlao_b200." + name)
        return config.initializeParameterFile(args)

    def set_params(self, args=None, wfs_type="shackhartmann", modal_basis="zernike", gainCL=0.5, n_envs=1, device=None,
                   rng="philox", seed=0, env_offset=0, warp_kernel="lagrange018", canvas_slack=96):
        """OOPAOEnvRazor.py:91-339 (SH branch; `wfs_type="pyramid"` builds the Pyramid of OOPAOEnv.py:239-249 instead)."""
        if wfs_type not in ("shackhartmann", "pyramid"):
            raise NotImplementedError(f"wfs_type {wfs_type!r}: only 'shackhartmann' and 'pyramid' are implemented")
        self.wfs_type = wfs_type
        args = args if args is not None else types.SimpleNamespace()
        self.gainCL = gainCL
        self.n_envs = int(n_envs)
        self.env_offset = int(env_offset)
        param = self._load_param(args)
        self.param = param
        self.tel = Telescope(resolution=param["resolution"], diameter=param["diameter"], samplingTime=param["samplingTime"],
                             centralObstruction=param["centralObstruction"], fov=param.get("fov", 0), n_envs=n_envs,
                             device=device)
        self.device = self.tel.device
        self.source = Source(optBand=param["opticalBand"], magnitude=param["magnitude"])
        self.source * self.tel
        self.atm = Atmosphere(telescope=self.tel, r0=param["r0"], L0=param["L0"], windSpeed=param["windSpeed"],
                              fractionalR0=param["fractionalR0"], windDirection=param["windDirection"],
                              altitude=param["altitude"], rng=rng, seed=seed, env_offset=env_offset,
                              warp_kernel=warp_kernel, canvas_slack=canvas_slack)
        self.atm.initializeAtmosphere(self.tel)
        self.atm.update()
        self.tel + self.atm
        # deformable mirror
        nAct = param["nActuator"]
        self.nActuator = nAct
        if param.get("dm_geometry", "razor") == "cartesian":
            self.dm = DeformableMirror(telescope=self.tel, nSubap=param["nSubaperture"], mechCoupling=param["mechanicalCoupling"],
                                       misReg=MisRegistration(param))
            self.dm_mask = np.reshape(self.dm.validAct, (nAct, nAct)).astype(int)
        else:
            # OOPAOEnvRazor.py:167-193: explicit coordinates from the actuator mask, DeformableMirror(nSubap=nActuator)
            x = np.linspace(-self.tel.D / 2, self.tel.D / 2, nAct)
            X, Y = np.meshgrid(x, x)
            keep = np.asarray(param["boolActMask"]).astype(bool).reshape(-1)
            coords = np.stack([X.reshape(-1)[keep], Y.reshape(-1)[keep]], axis=1)
            self.dm = DeformableMirror(telescope=self.tel, nSubap=nAct, mechCoupling=param["mechanicalCoupling"],
                                       M4_param=param, coordinates=coords)
            self.dm_mask = np.asarray(param["boolActMask"]).astype(int)
        self.xvalid, self.yvalid = np.nonzero(self.dm_mask)
        self.tel - self.atm
        if wfs_type == "pyramid":                                                                    # OOPAOEnv.py:239-246
            from ..Pyramid import Pyramid
            self.wfs = Pyramid(nSubap=param["nSubaperture"], telescope=self.tel, lightRatio=param.get("lightThreshold", 0.1),
                               modulation=param.get("modulation", 3), binning=1,
                               n_pix_separation=param.get("n_pix_separation", 4), n_pix_edge=2,
                               postProcessing=param.get("postProcessing", "slopesMaps"))
        else:
            self.wfs = ShackHartmann(telescope=self.tel, nSubap=param["nSubaperture"], lightRatio=param.get("lightRatio", 0.5),
                                     threshold_cog=param.get("threshold_cog", 0.01), is_geometric=param.get("is_geometric", False),
                                     shannon_sampling=param.get("shannon_sampling", True))
        cam = self.wfs.cam
        cam.sensor = param.get("cam_sensor", cam.sensor)
        cam.FWC = param.get("cam_FWC", cam.FWC)
        cam.bits = param.get("cam_bits", cam.bits)
        cam.QE = param.get("cam_QE", cam.QE)
        cam.darkCurrent = param.get("cam_darkCurrent", cam.darkCurrent)
        cam.integrationTime = param["samplingTime"]
        cam.seed = seed
        self.wfs.env_offset = self.env_offset       # every shard draws its own camera noise, also outside step()
        # production mode: atm.update() of frame t+1 runs on a side stream underneath the WFS of frame t (Atmosphere.prefetch)
        pf = os.environ.get("AOENV_ATM_PREFETCH", "1")               # 0 = off, 1 = when the batch is large enough, force = always
        self.atm.pipelined = "force" if pf == "force" else pf != "0"
        # a Shack-Hartmann evaluates the default (separable) mirror's surface inside its frame kernel: step() then computes
        # only T = C gx per command; the [n_envs, R, R] surface is produced on demand (dm.OPD, tel.OPD, PSF)
        if wfs_type != "pyramid" and getattr(self.wfs, "inline_dm", False) and self.dm.fused_tables() is not None \
                and self.wfs._dm_windows(self.dm.fused_tables()) is not None:
            self.dm.lazy_surface = True
        self.tel * self.wfs
        # modal basis and calibration
        nZ = param.get("nZernike", 50)
        if nZ and nZ > 0:
            Z = Zernike(self.tel, nZ)
            Z.computeZernike(self.tel)
            M2C = linalg.pinv(self.dm.modes[self.tel._pupil_idx, :].double()) @ Z.modes              # :261
        else:
            M2C = torch.eye(self.dm.nValidAct, dtype=torch.float64, device=self.device)
        calib_zonal = InteractionMatrix(ngs=self.source, atm=self.atm, tel=self.tel, dm=self.dm, wfs=self.wfs,
                                        M2C=torch.eye(self.dm.nValidAct, dtype=torch.float64, device=self.device),
                                        stroke=1e-9, nMeasurements=param.get("nMeasurements", 25), noise="off")
        self.calib_zonal = calib_zonal
        calib = CalibrationVault(calib_zonal.D @ M2C)                                                # :290
        self.tel.resetOPD()
        self.dm.coefs = 0
        self._dm_prev = torch.zeros((self.n_envs, self.dm._Kp), dtype=torch.float32, device=self.device)
        self._coefs_buf = torch.zeros((2, self.n_envs, self.dm._Kp), dtype=torch.float32, device=self.device)
        self._coefs_slot = 0
        self.source * self.tel * self.dm * self.wfs
        self.tel + self.atm
        self.calib_CL = calib
        self.M2C_CL = M2C
        nLoop = param.get("nLoop", None)
        self.SR = []
        self._nLoop = nLoop
        self.total = torch.zeros((nLoop, self.n_envs), dtype=torch.float32, device=self.device) if nLoop else None
        self.residual = torch.zeros((nLoop, self.n_envs), dtype=torch.float32, device=self.device) if nLoop else None
        cam.photonNoise = param.get("cam_photonNoise", True)                                         # :332-333 (OOPAOEnv.py:379)
        cam.readoutNoise = param.get("cam_readoutNoise", 14 if wfs_type == "shackhartmann" else 0)
        self.set_reconstructor(M2C @ calib.M)                                                        # :336
        self.F = M2C @ linalg.pinv(M2C)                                                              # :337
        nA_, Kp_ = self.dm.nValidAct, self.dm._Kp
        self._F32 = torch.zeros((nA_, Kp_), dtype=torch.float32, device=self.device)      # K-padded operand of F @ z
        self._F32[:, :nA_] = self.F.to(torch.float32)
        self._F_op = gemm.Operator(self._F32, parts=2)
        self.dm.free_float64()
        # device-side index tables and outputs
        B, nA = self.n_envs, self.dm.nValidAct
        self._act_idx = torch.as_tensor((self.xvalid * nAct + self.yvalid).astype(np.int32), device=self.device)
        self._rec = torch.zeros((B, (nA + 3) // 4 * 4), dtype=torch.float32, device=self.device)
        self._obs = torch.zeros((B, nAct, nAct), dtype=torch.float32, device=self.device)
        self._reward = torch.zeros((B,), dtype=torch.float32, device=self.device)
        self._strehl = torch.zeros((B,), dtype=torch.float32, device=self.device)
        self._total_now = torch.zeros((B,), dtype=torch.float32, device=self.device)
        self._residual_now = torch.zeros((B,), dtype=torch.float32, device=self.device)
        self._phase_scale = 2 * math.pi / self.source.wavelength
        self._noise_seed = (seed * 7919 + 5) & 0xFFFFFFFFFFFFFFFF
        self._noise_calls = 0
        self._noise_z = torch.zeros((B, self.dm._Kp), dtype=torch.float32, device=self.device)
        self._noise_planes = torch.zeros((2, B, self.dm._Kp), dtype=torch.bfloat16, device=self.device)
        self._noise_vec = torch.zeros((B, (nA + 3) // 4 * 4), dtype=torch.float32, device=self.device)

    def set_reconstructor(self, R):
        """reconstructor [nValidAct, nSignal] (float64 kept for inspection, padded float32 copy for the step GEMM)."""
        self.reconstructor = torch.as_tensor(R, dtype=torch.float64, device=self.device)
        nA, nSig = self.reconstructor.shape
        self._Rm = torch.zeros((nA, self.wfs._lds), dtype=torch.float32, device=self.device)
        self._Rm[:, :nSig] = self.reconstructor.to(torch.float32)
        self._Rm_op = gemm.Operator(self._Rm, parts=2)

    @property
    def dm_prev(self):
        d = self._dm_prev[:, :self.dm.nValidAct]
        return d[0] if self.n_envs == 1 else d

    @dm_prev.setter
    def dm_prev(self, val):
        t = torch.as_tensor(val, dtype=torch.float32, device=self.device)
        self._dm_prev.zero_()
        self._dm_prev[:, :self.dm.nValidAct] = t

    # ---- helpers ------------------------------------------------------------------------------------------
    def _sq(self, t):
        return t[0] if self.n_envs == 1 else t

    def _observe(self, with_stats):
        """obs = vec_to_img(-reconstructor @ signal) * 1e6 (+ reward, Strehl, rms diagnostics)."""
        lib, st, B, nA = _lib.load(), _lib.stream_ptr(self.device), self.n_envs, self.dm.nValidAct
        sig = self.wfs._signal
        gemm.gemm_tn(sig, self._Rm_op, self._rec, B, nA,
                     x_planes=self.wfs._signal_planes if gemm.uses_tensor_cores(B) else None)
        _lib.check(lib.aoenv_observe(_lib.ptr(self._rec), self._rec.stride(0), _lib.ptr(self._act_idx), B, nA,
                                     self.nActuator ** 2, _lib.ptr(self.wfs._stats) if with_stats else None,
                                     float(self.tel.pixelArea), self._phase_scale, _lib.ptr(self._obs), _lib.ptr(self._reward),
                                     _lib.ptr(self._strehl), _lib.ptr(self._total_now), _lib.ptr(self._residual_now), st),
                   "observe")

    def _action_tensor(self, action):
        a = torch.as_tensor(action, dtype=torch.float32, device=self.device)
        nAct = self.nActuator
        if a.ndim == 2:
            a = a.unsqueeze(0).expand(self.n_envs, -1, -1)
        return a.reshape(self.n_envs, nAct * nAct).contiguous()

    # ---- gym-style API --------------------------------------------------------------------------------------
    def reset_soft(self):
        """OOPAOEnvRazor.py:74-79."""
        self.action_buffer = []
        self._observe(False)
        return self._sq(self._obs).clone()

    def reset(self):
        raise NotImplementedError("reset() rebuilds the whole simulation in the reference (set_params without arguments, "
                                  "OOPAOEnvRazor.py:66-71, which raises there too); use set_params(...) then reset_soft()")

    def reset_envs(self, env_ids, seed):
        """New episode for the environments `env_ids` only (the others continue bit for bit): new phase screens in every
        layer (Atmosphere.reset_envs, which applies them to the frame the next step measures) and a flat mirror — their
        rows of the current commands, of dm_prev, of the current surface's T = C gx rows and, if it is materialised, of
        the surface itself are zeroed.  The next step's sensor sees the new atmosphere with a flat mirror, and its command
        is that step's action alone.  No physical parameter is per environment: the operators, wind, r0, L0, the sub-pixel
        phase of the wind and the window origins stay the batch's (see Atmosphere.reset_envs for the one difference from
        generateNewPhaseScreen).

        env_ids: host list / array of indices, or a bool mask [n_envs]; a mask on the device costs one synchronisation.
        Returns the int32 device tensor of the reset environments."""
        atm, dm = self.atm, self.dm
        atm._check_partial_reset()
        idx = atm.env_index(env_ids)
        if idx.numel() == 0:
            return idx
        if dm._coefs_matrix is not None or dm._multi is not None:
            raise NotImplementedError("reset_envs needs per-environment commands (the mirror holds a calibration command matrix)")
        atm._reset_listed(idx, seed)
        rows = idx.long()
        slot = dm._slot
        self._dm_prev[rows] = 0
        for c in {id(t): t for t in (dm._coefs, dm._coefs_of[slot]) if t is not None}.values():
            c[rows] = 0
        if dm._rows is not None and dm._rows_valid[slot]:
            dm._rows[slot][rows] = 0                      # T = C gx: zero commands give exactly zero rows
        if dm._valid[slot]:
            dm._opd[slot][rows] = 0
        return idx

    def reset_soft_wfs(self):
        self.action_buffer = []
        return self.wfs.cam.frame.clone()

    # ---- the step as two library calls (aoenv_atm_update + aoenv_sh_step) ------------------------------------------
    def _native_cfg(self):
        """aoenv_sh_step_t for the objects as they are now, or None when this step has to go call by call: another sensor
        or mirror model, the fused / materialised WFS modes, a PSF reward, NVTX ranges, a flux change that the sensor has
        not picked up yet.  Rebuilt only when something it depends on has changed."""
        wfs, dm, tel = self.wfs, self.dm, self.tel
        if (not self.native_step or _NVTX or self.psf_reward is not None or type(wfs) is not ShackHartmann or wfs.use_fused
                or not wfs.inline_dm or not dm.lazy_surface or self.atm.user_defined_opd or dm._multi is not None
                or dm._coefs_matrix is not None):
            return None
        src = tel.src
        if wfs._flux_version != getattr(src, "_flux_version", 0) or wfs.current_nPhoton != src.nPhoton:
            return None                                   # wfs._measure_terms re-initialises the flux on the ordinary path
        key = (wfs._flux_version, wfs.is_geometric, id(wfs._amp), id(wfs._ref_xy), wfs.slopes_units, wfs.threshold_cog, float(self.leak),
               id(self._Rm_op), id(dm._sep), src.wavelength, id(self._coefs_buf))
        if self._native_key == key:
            return self._native
        self._native_key, self._native = key, None
        tables = dm.fused_tables()
        win = wfs._dm_windows(tables) if tables is not None else None
        if win is None or 2 * math.pi / src.wavelength != self._phase_scale:
            return None
        tc = gemm.uses_tensor_cores(self.n_envs)
        dm._rows_of(dm._slot)                             # allocates the T buffers, makes the current slot's rows valid
        c = _lib.ShStepStruct()
        c.B, c.nS, c.n, c.nV, c.lds = self.n_envs, wfs.nSubap, wfs.n_pix_subap, wfs.nValidSubaperture, wfs._signal.stride(0)
        c.nA, c.nAct, c.nAct2 = dm.nValidAct, dm.nAct, self.nActuator ** 2
        c.ldc, c.ldr, c.W, c.rec_parts, c.use_tc = self._coefs_buf.stride(1), self._rec.stride(0), tables["W"], self._Rm_op.parts, int(tc)
        c.geometric = int(wfs.is_geometric)
        c.phase_scale, c.inv_units, c.threshold_cog, c.leak = self._phase_scale, 1.0 / wfs.slopes_units, wfs.threshold_cog, self.leak
        c.n_pupil = float(tel.pixelArea)
        keep = [tel._pupil_f, wfs._amp, wfs._valid_u8, wfs._lit_first, wfs._valid_idx, wfs._ref_xy, wfs._frame, wfs._envmax,
                wfs._stats, wfs._signal, wfs._signal_planes, win, self._Rm, self._Rm_op, self._rec, self._act_idx, self._dm_prev,
                tables]
        c.pupil, c.amp, c.valid, c.order = tel._pupil_f.data_ptr(), wfs._amp.data_ptr(), wfs._valid_u8.data_ptr(), wfs._lit_first.data_ptr()
        c.valid_idx, c.ref_xy, c.envmax = wfs._valid_idx.data_ptr(), wfs._ref_xy.data_ptr(), wfs._envmax.data_ptr()
        if wfs.is_geometric:                              # the geometric sensor weighs with the flux and has no frame
            c.amp, c.frame = wfs._flux.data_ptr(), None
            keep.append(wfs._flux)
        else:
            c.frame = wfs._frame.data_ptr()
        c.stats, c.slopes, c.slope_planes = wfs._stats.data_ptr(), wfs._signal.data_ptr(), wfs._signal_planes.data_ptr()
        c.dm.wlr, c.dm.ilr, c.dm.nActP, c.dm.WL = win[2].data_ptr(), win[1].data_ptr(), dm._rows.shape[2], win[0]
        c.rec_planes = self._Rm_op.planes().data_ptr() if tc else None
        c.rec_f32, c.rec, c.act_idx, c.dm_prev = self._Rm.data_ptr(), self._rec.data_ptr(), self._act_idx.data_ptr(), self._dm_prev.data_ptr()
        c.act_pos, c.wx, c.j0x = tables["act_pos"].data_ptr(), tables["wx"].data_ptr(), tables["j0x"].data_ptr()
        self._native = (c, keep)
        return self._native

    def _step_native(self, i, action, native, action_ready=None, after_observe=None):
        """OOPAOEnvRazor.py:474-514 through aoenv_atm_update + aoenv_sh_step; the Python objects are kept in step (slots,
        counters, lazy frames) exactly as the call-by-call path leaves them.  action_ready / after_observe: see
        _step_views."""
        c = native[0]
        dm, wfs, atm, B, dev = self.dm, self.wfs, self.atm, self.n_envs, self.device
        slot = dm._slot
        atm.update()                                                       # :482 (consumes a frame computed ahead)
        self.tel._set_lazy(atm._opd, DMSurfaceRef(dm, slot))               # :488 tel*dm, lazily
        det = None if wfs.is_geometric else wfs.cam.as_struct(self.env_offset)
        nAct = self.nActuator
        obs = torch.empty((B, nAct, nAct), dtype=torch.float32, device=dev)
        reward = torch.empty((B,), dtype=torch.float32, device=dev)
        strehl = torch.empty((B,), dtype=torch.float32, device=dev)
        coefs = self._coefs_buf[self._coefs_slot]
        args = [atm._opd.data_ptr(), dm._rows[slot].data_ptr(), ctypes.byref(det) if det is not None else None, None,
                coefs.data_ptr(), dm._rows[slot ^ 1].data_ptr(), obs.data_ptr(), reward.data_ptr(), strehl.data_ptr(),
                self._total_now.data_ptr(), self._residual_now.data_ptr(), _lib.stream_ptr(dev)]
        step, cref = _lib.load().aoenv_sh_step, ctypes.byref(c)
        if atm.can_prefetch() or after_observe is not None or action_ready is not None:
            # the next frame's atmosphere goes on the side stream right behind the spots and the slopes: it then fills the
            # SMs that the small kernels of the rest (reconstruction, observation, command, T rows) leave idle; a host-facing
            # caller starts its download once the observation is queued and has the command wait for its upload
            # Where the next frame's atmosphere is issued.  Behind the spots and the slopes it fills the SMs that the small
            # kernels of the rest leave idle and never delays the observation — what a caller that waits for the
            # observation on the host needs (issued before the spots, the strict host loop drops from 1.32 M to 0.95 M
            # env-steps/s at cfg3: the observation arrives later by the atmosphere's share of the SMs).  A device-resident
            # loop only sees throughput, and there the earlier issue lets the HBM-bound atmosphere kernels slip into the
            # FP32-bound spots kernel's tail and gaps: 0.748 -> 0.735 ms per step, bit-identical results.
            early = atm.sm_partition is not None or (self.prefetch_early and after_observe is None and action_ready is None)
            if early:
                atm.prefetch()
            _lib.check(step(cref, 1, *args), "sh_step")
            if not early:
                atm.prefetch()
            _lib.check(step(cref, 2, *args), "sh_step")
            if after_observe is not None:
                after_observe(self._sq(obs), self._sq(reward), self._sq(strehl))
            if action_ready is not None:
                torch.cuda.current_stream(dev).wait_event(action_ready)
            args[3] = self._action_tensor(action).data_ptr()               # (after the wait: it may have to make a copy)
            _lib.check(step(cref, 4, *args), "sh_step")
        else:
            act = self._action_tensor(action)
            args[3] = act.data_ptr()
            _lib.check(step(cref, 7, *args), "sh_step")
        self._coefs_slot ^= 1
        dm._coefs, dm._multi, dm._coefs_matrix, dm._slot = coefs, None, None, slot ^ 1
        dm._coefs_of[slot ^ 1], dm._rows_valid[slot ^ 1], dm._valid[slot ^ 1] = coefs, True, False
        if not wfs.is_geometric:
            wfs.cam.frame = wfs._frame[0] if B == 1 else wfs._frame
        wfs._signal_is_multi = False
        self._obs, self._reward, self._strehl = obs, reward, strehl
        if self.total is not None and i is not None and 0 <= i < self._nLoop:
            self.total[i] = self._total_now
            self.residual[i] = self._residual_now
        s = self._sq(strehl)
        self.SR.append(s)
        self.wfsSignal = wfs.signal
        return self._sq(obs), self._sq(reward), s, False, {"strehl": s}

    def step(self, i, action):
        """OOPAOEnvRazor.py:474-514.  Returns fresh tensors (the reference returns fresh arrays)."""
        native = self._native_cfg()
        if native is not None and self.dm._rows_valid[self.dm._slot]:
            return self._step_native(i, action, native)
        obs, reward, strehl, done, info = self._measure_frame(i)
        self._apply_command(action)
        strehl = strehl.clone()
        self.SR[-1] = strehl
        return obs.clone(), reward.clone(), strehl, done, {"strehl": strehl}

    def _step_views(self, i, action, action_ready=None, after_observe=None):
        """The step itself; returns views of the internal output buffers (overwritten by the next step).

        The observation of frame i depends on the slopes only, not on the action applied in this call (one frame of
        DM lag), so it is produced BEFORE the command update: a host-facing caller can start copying it out
        (`after_observe(obs, reward, strehl)` is called at that point of the stream) while the command update and the
        next DM surface are still being computed, and can upload the action on another stream (`action_ready`: CUDA
        event the command update waits for) while the atmosphere and the WFS run."""
        native = self._native_cfg()
        if native is not None and self.dm._rows_valid[self.dm._slot]:
            return self._step_native(i, action, native, action_ready, after_observe)     # fresh tensors rather than views
        out = self._measure_frame(i, after_observe)
        self._apply_command(action, action_ready)
        return out

    def _measure_frame(self, i, after_observe=None, atmosphere_done=False):
        """First half of step (OOPAOEnvRazor.py:482-488, 496-506): atmosphere, WFS on (atmosphere + the DM surface
        commanded at the previous step), reconstruction, reward, Strehl.  `atmosphere_done`: atm.update() for this
        frame has already been issued (it depends on nothing the step computes)."""
        if not atmosphere_done:
            with _range("aoenv.atmosphere"):
                self.atm.update()                                          # :482 -> tel.OPD = atm.OPD (lazy)
        else:
            self.atm._join_prefetch(consume=True)                          # issued ahead on the side stream, if at all
        dm_surface = self.dm.surface_ref()                                 # surface commanded at the previous step
        self.tel._set_lazy(self.atm._opd, dm_surface)                      # :488 tel*dm
        with _range("aoenv.wfs"):
            self.wfs._measure_terms(self.atm._opd, dm_surface, self.env_offset)  # :488 *wfs  (+ stats for :484,502,506)
        if not atmosphere_done:
            with _range("aoenv.atmosphere_next"):
                self.atm.prefetch()          # the next frame's atm.update(), on a side stream underneath this frame's WFS
        with _range("aoenv.reconstruct"):
            self._observe(True)                                            # :496-506
        if self.total is not None and i is not None and 0 <= i < self._nLoop:
            self.total[i] = self._total_now
            self.residual[i] = self._residual_now
        strehl = self._sq(self._strehl)
        if self.psf_reward is not None:
            strehl = self.psf_strehl(*self.psf_reward)
        if after_observe is not None:
            after_observe(self._sq(self._obs), self._sq(self._reward), strehl)
        self.SR.append(strehl if self.psf_reward is not None else strehl.clone())
        self.wfsSignal = self.wfs.signal
        return self._sq(self._obs), self._sq(self._reward), strehl, False, {"strehl": strehl}

    def _apply_command(self, action, action_ready=None):
        """Second half of step (OOPAOEnvRazor.py:479, 492-493): dm.coefs = dm_prev * leak + action, next DM surface."""
        lib, st, B = _lib.load(), _lib.stream_ptr(self.device), self.n_envs
        if action_ready is not None:
            torch.cuda.current_stream(self.device).wait_event(action_ready)
        action = self._action_tensor(action)                               # :479 (img_to_vec * 1e-6 is in the kernel)
        coefs = self._coefs_buf[self._coefs_slot]                         # zero-padded tails, never written
        self._coefs_slot ^= 1
        with _range("aoenv.command"):
            _lib.check(lib.aoenv_command_update(_lib.ptr(action), _lib.ptr(self._act_idx), B, self.dm.nValidAct,
                                                self.nActuator ** 2, ctypes.c_float(self.leak), _lib.ptr(coefs), _lib.ptr(self._dm_prev),
                                                coefs.stride(0), st), "command_update")      # :492-493
            self.dm._set_coefs_batch(coefs)                                # coefs setter side effect: next surface

    # ---- checkpoint / resume (the reference has none: SURVEY.md section 5) -------------------------------------------
    def state_dict(self):
        """Everything that evolves during an episode, as CPU tensors / plain numbers: layer windows with their shift
        bookkeeping and generator counters, DM commands, camera and exploration-noise counters, the per-step records.
        With the counter-based generators a restored environment continues bit for bit."""
        atm = self.atm
        nxt = None
        if atm._prefetched:                  # the layers already hold the next frame: keep its OPD with them
            atm._wait_prefetch()
            nxt = atm._opd_next.detach().cpu().clone()
        layers = []
        for i, ly in enumerate(atm._layers):
            layers.append(dict(map=ly.mapShift.detach().cpu().clone(), buff=ly.buff.copy(), ratio=ly.ratio.copy(),
                               notDoneOnce=ly.notDoneOnce, events=ly.events, philox_seed=getattr(ly, "philox_seed", 0),
                               ext=None))
        return dict(version=1, n_envs=self.n_envs, rng=atm.rng, layers=layers, atm_opd=atm._opd.detach().cpu().clone(),
                    atm_opd_next=nxt,
                    coefs=self.dm._coefs.detach().cpu().clone(), dm_prev=self._dm_prev.detach().cpu().clone(),
                    cam_frame_counter=self.wfs.cam.frame_counter, noise_calls=self._noise_calls,
                    SR=[s.detach().cpu().clone() for s in self.SR],
                    total=None if self.total is None else self.total.detach().cpu().clone(),
                    residual=None if self.residual is None else self.residual.detach().cpu().clone())

    def load_state_dict(self, st):
        """Restores a `state_dict()` of an environment built with the same configuration."""
        if st.get("version") != 1 or st["n_envs"] != self.n_envs or st["rng"] != self.atm.rng:
            raise ValueError("state_dict of another environment (n_envs / rng / version differ)")
        if self.atm.rng != "philox":
            raise NotImplementedError("host MT19937 streams (rng='reference') are not checkpointed; use rng='philox'")
        atm, dev = self.atm, self.device
        atm._join_prefetch(consume=False)
        for i, (ly, s_) in enumerate(zip(atm._layers, st["layers"])):
            atm._cur[i] = 0
            atm._org[i] = atm._fresh_origin(i)
            oy, ox = atm._org[i]
            m = s_["map"].to(dev)
            atm._maps[i, 0, :, oy:oy + atm._M, ox:ox + atm._M] = m if m.ndim == 3 else m.unsqueeze(0)
            ly.buff, ly.ratio, ly.notDoneOnce = s_["buff"].copy(), s_["ratio"].copy(), s_["notDoneOnce"]
            ly.events, ly.philox_seed = s_["events"], s_["philox_seed"]
            atm._rescan_extrema(i)
        atm._opd.copy_(st["atm_opd"].to(dev))
        if st.get("atm_opd_next") is not None:
            if atm._opd_next is None:
                atm._opd_next = torch.empty_like(atm._opd)
                atm._side_stream = torch.cuda.Stream(dev)
            atm._opd_next.copy_(st["atm_opd_next"].to(dev))
            atm._prefetched, atm._prefetch_event = True, torch.cuda.current_stream(dev).record_event()
        coefs = st["coefs"].to(dev)
        self._dm_prev.copy_(st["dm_prev"].to(dev))
        self._coefs_buf[self._coefs_slot].copy_(coefs)
        self.dm._set_coefs_batch(self._coefs_buf[self._coefs_slot])
        self._coefs_slot ^= 1
        self.wfs.cam.frame_counter, self._noise_calls = st["cam_frame_counter"], st["noise_calls"]
        self.SR = [s.to(dev) for s in st["SR"]]
        if st["total"] is not None and self.total is not None:
            self.total.copy_(st["total"].to(dev))
            self.residual.copy_(st["residual"].to(dev))
        self.tel._set_lazy(atm._opd, self.dm.surface_ref())

    def step_wfs(self, i, action):
        """OOPAOEnvRazor.py:553-586 (the definition that is in effect: the second `def step_wfs`): the observation is the
        WFS camera frame, the command accumulates without leak and the action is applied as given (metres)."""
        self._measure_frame(i)
        frame = self.wfs.cam.frame.clone()
        leak, self.leak = self.leak, 1.0
        try:
            self._apply_command(torch.as_tensor(action, dtype=torch.float32, device=self.device) * 1e6)   # the kernel scales by 1e-6
        finally:
            self.leak = leak
        strehl = self.SR[-1]
        reward = self._sq(-torch.linalg.vector_norm(frame.reshape(self.n_envs, -1).float(), dim=1))
        return frame, reward, strehl, False, {"strehl": strehl}

    def _get_reward(self, slopes=None, type="volt"):
        """OOPAOEnvRazor.py:607-614: S2V is never set on this path, so the reward is the Strehl ratio."""
        if getattr(self, "S2V", None) is not None and type != "sh":
            v = torch.as_tensor(slopes, dtype=torch.float64, device=self.device) @ torch.as_tensor(self.S2V, dtype=torch.float64, device=self.device).T
            return -torch.linalg.vector_norm(v, dim=-1)
        return self.get_strehl()

    def compute_dm_proj(self):
        """OOPAOEnvRazor.py:676-680: (modes^T modes)^-1 modes^T, the least-squares projector of an OPD map on the DM."""
        modes = self.dm.modes.double()
        self.dm_proj = torch.linalg.solve(modes.T @ modes, modes.T)
        return self.dm_proj

    def OPD_on_dm(self):
        """OOPAOEnvRazor.py:683-689: the part of tel.OPD the DM can reproduce."""
        if getattr(self, "dm_proj", None) is None:
            self.compute_dm_proj()
        res = self.tel.resolution
        opd = (self.tel._materialise() * self.tel._pupil_f).double().reshape(self.n_envs, res * res)
        out = ((opd @ self.dm_proj.T) @ self.dm.modes.double().T).reshape(self.n_envs, res, res)
        return self._sq(out)

    def set_modalBasis(self, mode="zernike"):
        """OOPAOEnvRazor.py:393-425: recompute the zonal interaction matrix and the modal (50 Zernike) calibration."""
        if mode != "zernike":
            raise NotImplementedError("only the Zernike basis is built by the reference (OOPAOEnvRazor.py:394)")
        paired = self.tel.isPaired
        self.tel - self.atm
        Z = Zernike(self.tel, 50)
        Z.computeZernike(self.tel)
        M2C = linalg.pinv(self.dm.modes[self.tel._pupil_idx, :].double()) @ Z.modes
        eye = torch.eye(self.dm.nValidAct, dtype=torch.float64, device=self.device)
        self.imat = InteractionMatrix(ngs=self.source, atm=self.atm, tel=self.tel, dm=self.dm, wfs=self.wfs, M2C=eye,
                                      stroke=1e-9, nMeasurements=25, noise="off")
        self.calib_CL = CalibrationVault(self.imat.D @ M2C)
        self.M2C_CL = M2C
        self.tel.resetOPD()
        self.dm.coefs = 0
        self.source * self.tel * self.dm * self.wfs
        if paired:
            self.tel + self.atm

    def set_wfs(self, param, type="pyramid"):
        """OOPAOEnvRazor.py:342-391: replace the WFS (the calibration is NOT redone, as in the reference: call
        set_modalBasis / set_reconstructor afterwards)."""
        self.tel - self.atm
        if type == "pyramid":
            from ..Pyramid import Pyramid
            if param.get("psfCentering", True) is not True:
                raise NotImplementedError("Pyramid(psfCentering=False) is out of scope")
            self.wfs = Pyramid(nSubap=param["nSubaperture"], telescope=self.tel, modulation=param["modulation"],
                               lightRatio=param["lightThreshold"], n_pix_separation=param["n_pix_separation"],
                               postProcessing=param["postProcessing"])
        elif type == "shackhartmann":
            self.wfs = ShackHartmann(telescope=self.tel, nSubap=param["nSubaperture"], lightRatio=param.get("lightRatio", 0.5),
                                     threshold_cog=param.get("threshold_cog", 0.01), is_geometric=param.get("is_geometric", False),
                                     shannon_sampling=param.get("shannon_sampling", True))
        else:
            raise NotImplementedError(f"wfs type {type!r}")
        self.wfs_type = type
        self.tel * self.wfs

    def calculate_strehl_AVG(self):
        """OOPAOEnvRazor.py:589-596 (mean over the episode; here also over environments and, when
        torch.distributed is initialised, over ranks)."""
        if len(self.SR) == 0:
            return float("nan")
        s = torch.stack([x.reshape(-1) for x in self.SR]).double()
        tot = torch.stack([s.sum(), torch.tensor(float(s.numel()), dtype=torch.float64, device=s.device)])
        import torch.distributed as dist
        if dist.is_available() and dist.is_initialized():
            dist.all_reduce(tot)
        self.SR = []
        return float(tot[0] / tot[1])

    def integrator(self):
        return -self.gainCL * self.vec_to_img(self.wfs.signal.double() @ self.reconstructor.T)

    def get_slopes(self):
        return self.wfs.signal

    def get_strehl(self):
        """OOPAOEnvRazor.py:604-605."""
        ph = self.tel._materialise() * self.tel._pupil_f * self._phase_scale
        v = ph.reshape(ph.shape[0], -1)[:, self.tel._pupil_idx].double().var(dim=1, unbiased=False)
        return self._sq(torch.exp(-v).float())

    def sample_noise(self, sigma, use_torch=True):
        """OOPAOEnvRazor.py:616-619: F @ (sigma * N(0, I)), as an actuator image per environment."""
        lib, st, B, nA = _lib.load(), _lib.stream_ptr(self.device), self.n_envs, self.dm.nValidAct
        tc = gemm.uses_tensor_cores(B)
        # Philox normals (counter = call number; environments of other shards sit at other rows of the stream) ...
        _lib.check(lib.aoenv_normal_fill(ctypes.c_uint64(self._noise_seed + (self.env_offset << 20)), ctypes.c_uint64(self._noise_calls),
                                         B, nA, self.dm._Kp, ctypes.c_float(float(sigma)), _lib.ptr(self._noise_z),
                                         _lib.ptr(self._noise_planes) if tc else None, 2, st), "normal_fill")
        self._noise_calls += 1
        # ... times F on the tensor cores, scattered to actuator images
        gemm.gemm_tn(self._noise_z, self._F_op, self._noise_vec, B, nA, x_planes=self._noise_planes if tc else None)
        img = torch.empty((B, self.nActuator, self.nActuator), dtype=torch.float32, device=self.device)
        _lib.check(lib.aoenv_vec_to_img(_lib.ptr(self._noise_vec), self._noise_vec.stride(0), _lib.ptr(self._act_idx), B, nA,
                                        self.nActuator ** 2, ctypes.c_float(1.0), _lib.ptr(img), st), "vec_to_img")
        return self._sq(img)

    def vec_to_img(self, action_vec, use_torch=True):
        """OOPAOEnvRazor.py:621-630."""
        v = torch.as_tensor(action_vec, device=self.device)
        lead = v.shape[:-1]
        img = torch.zeros(lead + (self.nActuator, self.nActuator), dtype=v.dtype, device=self.device)
        img[..., torch.as_tensor(self.xvalid, device=self.device), torch.as_tensor(self.yvalid, device=self.device)] = v
        return img

    def img_to_vec(self, action):
        """OOPAOEnvRazor.py:634-641."""
        a = torch.as_tensor(action, device=self.device)
        return a[..., torch.as_tensor(self.xvalid, device=self.device), torch.as_tensor(self.yvalid, device=self.device)]

    def change_mag(self, mag):
        """OOPAOEnvRazor.py:644-647."""
        self.source.nPhoton = self.source.zeroPoint * 10 ** (-0.4 * mag)
        self.source.magnitude = mag
        self.source * self.tel * self.wfs

    def psf_strehl(self, zeroPaddingFactor=4, window=32):
        """Strehl from the science PSF peak (tel.computePSF(zp); PSF.max()/psf_model_max, caller pattern
        MAIN_CODE/closedLoopPlayground.py:25-30), evaluated with the pruned-DFT kernel on the central window."""
        from ..psf import psf_peak
        if not hasattr(self, "_psf_model_max") or self._psf_model_key != (zeroPaddingFactor, window):
            zero = torch.zeros((1, self.tel.resolution, self.tel.resolution), dtype=torch.float32, device=self.device)
            self._psf_model_max = psf_peak(self.tel, zero, None, zeroPaddingFactor, window)[0]
            self._psf_model_key = (zeroPaddingFactor, window)
        a, b = self.tel._terms()
        return self._sq(psf_peak(self.tel, a, b, zeroPaddingFactor, window) / self._psf_model_max)

