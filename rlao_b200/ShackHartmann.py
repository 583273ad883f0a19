"""ShackHartmann — mirror of OOPAO/ShackHartmann.py (diffractive, NGS, binning 1), batched over environments.

`tel*wfs` / `wfs.wfs_measure()` run two kernels (include/aoenv.h): aoenv_shwfs_frame (lenslet fields ->
spots -> detector -> camera frame + per-environment maximum) and aoenv_shwfs_slopes (thresholded centre of
gravity -> slopes).  Results: `wfs.signal` ([nSignal], or [n_envs, nSignal]; [nSignal, k] after a k-frame
calibration push as in ShackHartmann.py:674), `wfs.signal_2D`, `wfs.cam.frame`.

`is_geometric=True` builds the geometric sensor instead (DESIGN.md section 2): the flux-weighted mean phase gradient of
every lenslet, one kernel (aoenv_shwfs_geometric), noise-free; the camera is not used and `wfs.cam.frame` is not written.
"""
import ctypes as C
import math
import os

import numpy as np
import torch

from . import _lib, gemm
from .DeformableMirror import DMSurfaceRef
from .Detector import Detector

_SUPPORTED_N = (4, 6, 8, 10, 12)
_FUSED_N = (4, 6, 8)              # the cluster-fused cross-check kernel (AOENV_WFS=fused) and the alternative frame variants


class ShackHartmann:
    def __init__(self, nSubap, telescope, lightRatio, threshold_cog=0.01, is_geometric=False, binning_factor=1,
                 padding_extension_factor=1, threshold_convolution=0.05, shannon_sampling=False, unit_P2V=False):
        self.tag = "shackHartmann"
        self.telescope = telescope
        if telescope.src is None:
            raise AttributeError("The telescope was not coupled to any source object! Make sure to couple it with an src object using src*tel")
        if binning_factor != 1 or padding_extension_factor > 2:
            raise NotImplementedError("binning_factor != 1 / extended field of view are out of scope")
        if getattr(telescope.src, "type", "NGS") == "LGS":
            raise NotImplementedError("LGS spot elongation is out of scope")
        self.device = telescope.device
        self.n_envs = telescope.n_envs
        self._is_geometric = bool(is_geometric)
        self.nSubap = int(nSubap)
        self._lightRatio = lightRatio
        self.binning_factor = 1
        self.zero_padding = 2
        self.padding_extension_factor = padding_extension_factor
        self.threshold_convolution = threshold_convolution
        self.threshold_cog = threshold_cog
        self.shannon_sampling = shannon_sampling
        self.unit_P2V = unit_P2V
        R = telescope.resolution
        if R % self.nSubap != 0:
            raise ValueError("telescope.resolution must be a multiple of nSubap")
        self.n_pix_subap = R // self.nSubap
        if self.n_pix_subap not in _SUPPORTED_N:
            raise NotImplementedError(f"{self.n_pix_subap} pixels per subaperture: compiled sizes are {_SUPPORTED_N}")
        self.n_pix_subap_init = self.n_pix_subap
        self.n_pix_lenslet_init = self.n_pix_subap * self.zero_padding
        self.n_pix_lenslet = self.n_pix_lenslet_init
        self.is_extended = False
        self.is_LGS = False
        self.cam = Detector(round(self.nSubap * self.n_pix_subap))
        self.cam.photonNoise = 0
        self.cam.readoutNoise = 0
        src = telescope.src
        self.fov_lenslet_arcsec = (self.n_pix_subap * 206265 * self.binning_factor / self.padding_extension_factor
                                   * src.wavelength / (telescope.D / self.nSubap)) / (1 + self.shannon_sampling)
        self.fov_pixel_arcsec = self.fov_lenslet_arcsec / self.n_pix_subap
        self.fov_pixel_binned_arcsec = self.fov_lenslet_arcsec / self.n_pix_subap_init
        self.get_camera_frame_multi = False
        # Production path: the frame kernel (three lanes per lenslet for 6-pixel lenslets) + the slopes kernel.
        # use_fused (opt-in, AOENV_WFS=fused): ONE cluster kernel for DM surface + spots + slopes (aoenv_shwfs_fused), for a
        # uniform flux over a binary pupil; correct and tested, but measured slower on B200 (a third of its time is spent
        # at the cluster barrier that the environment-wide centroiding threshold needs — profiles/r2_*).  With it,
        # keep_frame = False (default) leaves the camera frame unwritten: `wfs.cam.frame` is then produced on demand from
        # the inputs of the last measurement.
        self.env_offset = 0          # global index of this shard's first environment (seeds of the camera streams)
        self.use_fused = os.environ.get("AOENV_WFS", "kernels") == "fused" and not self._is_geometric
        self.keep_frame = False
        self._fused_plans = {}
        # inline_dm (default): a separable mirror's surface that exists only as commands (DMSurfaceRef of a lazy mirror) is
        # evaluated inside the frame kernel (aoenv_shwfs_frame_dm); AOENV_WFS_INLINE_DM=0 reads the materialised surface
        self.inline_dm = os.environ.get("AOENV_WFS_INLINE_DM", "1") != "0"
        self._dm_window_cache = {}
        self._last_inputs = None
        ii, jj = np.meshgrid(np.arange(self.nSubap), np.arange(self.nSubap), indexing="ij")
        self.index_x, self.index_y = ii.reshape(-1), jj.reshape(-1)
        self.initialize_flux()
        self._select_valid()
        B = self.n_envs
        # (the geometric sensor has no camera frame)
        self._frame = None if self._is_geometric else torch.zeros((B, R, R), dtype=torch.float32, device=self.device)
        self._envmax = torch.zeros((B,), dtype=torch.int32, device=self.device)
        self._stats = torch.zeros((B, 4), dtype=torch.float64, device=self.device)
        self._signal = torch.zeros((B, self._lds), dtype=torch.float32, device=self.device)
        self._signal_planes = torch.zeros((2, B, self._lds), dtype=torch.bfloat16, device=self.device)   # GEMM operand form
        self._signal_is_multi = False
        self.initialize_wfs()

    # ---- flux / valid subapertures (ShackHartmann.py:215-240,327-338) -------------------------------------
    def initialize_flux(self, input_flux_map=None):
        src, nS, n = self.telescope.src, self.nSubap, self.n_pix_subap
        flux = np.asarray(src.fluxMap if input_flux_map is None else input_flux_map.T, dtype=np.float64)
        self.photon_per_subaperture = flux.reshape(nS, n, nS, n).sum(axis=(1, 3)).reshape(-1)
        self.photon_per_subaperture_2D = self.photon_per_subaperture.reshape(nS, nS)
        self._amp = torch.as_tensor(np.sqrt(flux), dtype=torch.float32, device=self.device).contiguous()
        if self._is_geometric:                                           # the weights of the geometric sensor
            self._flux = torch.as_tensor(flux, dtype=torch.float32, device=self.device).contiguous()
        self.current_nPhoton = src.nPhoton
        self._flux_version = getattr(src, "_flux_version", 0)
        # fused-kernel form: binary pupil mask + one amplitude (valid only when the flux is uniform over the pupil)
        pup = np.asarray(self.telescope.pupil)
        inside = pup > 0
        vals = flux[inside]
        self._uniform_flux = bool(inside.any() and np.all((pup == 0) | (pup == 1)) and np.all(flux[~inside] == 0)
                                  and np.all(vals == vals[0]))
        self._amp0 = float(np.sqrt(vals[0])) if self._uniform_flux else 0.0
        self._pupil8 = torch.as_tensor(inside.astype(np.uint8), device=self.device).contiguous()

    def _select_valid(self):
        nS = self.nSubap
        pps = self.photon_per_subaperture
        self.valid_subapertures = (pps >= self._lightRatio * pps.max()).reshape(nS, nS)
        self.valid_subapertures_1D = self.valid_subapertures.reshape(-1)
        self.validLenslets_x, self.validLenslets_y = np.where(self.valid_subapertures)
        self.valid_slopes_maps = np.concatenate((self.valid_subapertures, self.valid_subapertures))
        self.nValidSubaperture = int(self.valid_subapertures.sum())
        self.nSignal = 2 * self.nValidSubaperture
        self._lds = (self.nSignal + 15) // 16 * 16
        dev = self.device
        self._valid_u8 = torch.as_tensor(self.valid_subapertures_1D.astype(np.uint8), device=dev).contiguous()
        self._valid_idx = torch.as_tensor(np.nonzero(self.valid_subapertures_1D)[0].astype(np.int32), device=dev).contiguous()
        slot = np.full(nS * nS, -1, dtype=np.int32)
        slot[np.nonzero(self.valid_subapertures_1D)[0]] = np.arange(self.nValidSubaperture, dtype=np.int32)
        self._slot_of = torch.as_tensor(slot, device=dev).contiguous()
        v1 = np.asarray(self.valid_subapertures_1D).astype(bool).reshape(-1)
        self._lit_first = torch.as_tensor(np.concatenate([np.nonzero(v1)[0], np.nonzero(~v1)[0]]).astype(np.int32),
                                          device=dev).contiguous()       # lenslet order of the frame kernel: lit ones first
        self._fused_plans = {}

    @property
    def lightRatio(self):
        return self._lightRatio

    @lightRatio.setter
    def lightRatio(self, val):
        """ShackHartmann.py:737-764."""
        self._lightRatio = val
        self._select_valid()
        self._signal = torch.zeros((self.n_envs, self._lds), dtype=torch.float32, device=self.device)
        self._signal_planes = torch.zeros((2, self.n_envs, self._lds), dtype=torch.bfloat16, device=self.device)
        self.initialize_wfs()

    @property
    def is_geometric(self):
        return self._is_geometric

    @is_geometric.setter
    def is_geometric(self, val):
        if bool(val) != self._is_geometric:
            raise NotImplementedError("the calibration (reference, slope units) belongs to the sensor mode: build a new "
                                      "ShackHartmann(is_geometric=...) instead of switching it")

    # ---- kernels ------------------------------------------------------------------------------------------
    def _dm_windows_host(self, dm_tables):
        """Row-weight windows of a separable DM (aoenv_dm_sep_t): first actuator row of every lenslet row's window, the
        window height WL (14 or 18; 0 = bands too wide) and the weights of every pixel row relative to its window."""
        nS, n = self.nSubap, self.n_pix_subap
        R = nS * n
        by, gy = dm_tables["by_host"], dm_tables["gy_host"]            # [R, 2] band of every pixel row, [nAct, R] weights
        lo = by[:, 0].reshape(nS, n).min(axis=1)
        hi = by[:, 1].reshape(nS, n).max(axis=1)
        need = int((hi - lo + 1).max())
        WL = 14 if need <= 14 else (18 if need <= 18 else 0)
        if WL == 0:
            return 0, None, None
        half = (WL + 1) // 2
        hp = (half + 3) // 4 * 4
        wl = np.zeros((R, 2 * hp), dtype=np.float32)
        for y in range(R):
            i0 = lo[y // n]
            for i in range(by[y, 0], by[y, 1] + 1):
                t = i - i0
                wl[y, (t // half) * hp + t % half] = gy[i, y]
        return WL, lo.astype(np.int32), wl

    def _dm_windows(self, dm_tables):
        """Device copy of _dm_windows_host, cached per mirror geometry; None if the windows do not fit."""
        key = id(dm_tables)
        hit = self._dm_window_cache.get(key)
        if hit is None:
            WL, ilr, wlr = self._dm_windows_host(dm_tables)
            hit = (WL, None, None) if WL == 0 else (
                WL, torch.as_tensor(ilr, dtype=torch.int32, device=self.device).contiguous(),
                torch.as_tensor(wlr, dtype=torch.float32, device=self.device).contiguous())
            self._dm_window_cache[key] = (hit, dm_tables)             # keeps the tables alive: id() stays unique
        else:
            hit = hit[0]
        return hit if hit[0] != 0 else None

    def _fused_plan(self, dm_tables):
        """Launch shape of aoenv_shwfs_fused: CTAs per environment (cluster) and the strip of lenslet rows each owns (cut
        so that rows + lit lenslets are even), warp groups, the lit-first lenslet order of every strip, and — with a
        separable DM — the window tables: first actuator row of every lenslet row's band, row weights relative to it."""
        key = id(dm_tables) if dm_tables is not None else 0
        plan = self._fused_plans.get(key)
        if plan is not None:
            return plan
        lib, nS, n, dev = _lib.load(), self.nSubap, self.n_pix_subap, self.device
        if n not in _FUSED_N:
            raise NotImplementedError(f"the fused WFS kernel (AOENV_WFS=fused) is compiled for {_FUSED_N} pixels per "
                                      f"subaperture, not {n}")
        R = nS * n
        groups = int(os.environ.get("AOENV_WFS_GROUPS", "4"))
        valid = self.valid_subapertures
        lit_row = valid.sum(axis=1).astype(np.float64)
        WL, ilr, wlr = 0, None, None
        if dm_tables is not None:
            WL, ilr, wlr = self._dm_windows_host(dm_tables)
            if WL == 0:
                raise NotImplementedError("DM influence bands are too wide for the fused kernel")

        def t_rows_for(rs):
            if ilr is None:
                return 0
            return int(max(ilr[rs[k + 1] - 1] + WL - ilr[rs[k]] for k in range(len(rs) - 1)))

        # contiguous strips minimising the largest cost: phase D is paid per lenslet row, the transforms per lit lenslet
        # (one row of phase D ~ 0.26 nS lit lenslets); one dynamic programme serves every cluster size
        Cmax = min(16, nS)
        cost = 0.26 * nS + lit_row
        pre = np.concatenate([[0.0], np.cumsum(cost)])
        seg = pre[None, :] - pre[:, None]                                   # seg[s0, e] = cost of rows [s0, e)
        best = np.full((Cmax + 1, nS + 1), np.inf)
        arg = np.zeros((Cmax + 1, nS + 1), dtype=np.int64)
        best[0, 0] = 0.0
        for c in range(1, Cmax + 1):
            for e in range(c, nS + 1):
                v = np.maximum(best[c - 1, c - 1:e], seg[c - 1:e, e])
                k = int(np.argmin(v))
                best[c, e], arg[c, e] = v[k], c - 1 + k

        def partition(C_):
            rs, e = [nS], nS
            for c in range(C_, 0, -1):
                e = int(arg[c, e])
                rs.append(e)
            return rs[::-1]

        def smem_for(rs):
            rows_max = max(rs[k + 1] - rs[k] for k in range(len(rs) - 1))
            return lib.aoenv_shwfs_fused_smem(nS, n, rows_max, groups, t_rows_for(rs), WL)
        forced = os.environ.get("AOENV_WFS_CLUSTER")
        limit = 227 * 1024
        cands = {c: partition(c) for c in range(1, Cmax + 1)}
        if forced:
            cluster = int(forced)
        else:
            # portable cluster sizes first: the largest one that leaves >= 96 lenslets per CTA on average, else a single
            # CTA; configurations whose strips do not fit in shared memory take the largest cluster (<= 16) that does
            fit8 = [c for c in cands if c <= 8 and 0 < smem_for(cands[c]) <= limit]
            good = [c for c in fit8 if nS * nS // c >= 96]
            if good:
                cluster = max(good)
            elif fit8:
                cluster = min(fit8)
            else:
                fit16 = [c for c in cands if 0 < smem_for(cands[c]) <= limit]
                if not fit16:
                    raise NotImplementedError(f"{nS} x {nS} lenslets of {n} px do not fit the fused WFS kernel")
                cluster = max(fit16)
        rs = cands[cluster]
        rows_max = max(rs[k + 1] - rs[k] for k in range(cluster))
        order = np.zeros((cluster, rows_max * nS), dtype=np.int32)
        nlit = np.zeros(cluster, dtype=np.int32)
        for r in range(cluster):
            v = valid[rs[r]:rs[r + 1]].reshape(-1)
            o = np.concatenate([np.nonzero(v)[0], np.nonzero(~v)[0]])
            order[r, :len(o)] = o
            nlit[r] = int(v.sum())
        td = lambda a, dt: torch.as_tensor(np.ascontiguousarray(a), dtype=dt, device=dev).contiguous()
        plan = dict(cluster=cluster, groups=groups, t_rows=t_rows_for(rs), WL=WL, row_start=(C.c_int32 * (cluster + 1))(*rs),
                    rows=rs, order=td(order, torch.int32), nlit=td(nlit, torch.int32),
                    ilr=td(ilr, torch.int32) if ilr is not None else None, wlr=td(wlr, torch.float32) if wlr is not None else None)
        self._fused_plans[key] = plan
        return plan

    def _fused_ok(self, opd_a):
        return (self.use_fused and self._uniform_flux and self.telescope.resolution % 4 == 0 and opd_a.dtype == torch.float32
                and opd_a.is_contiguous())

    def _run_fused(self, opd_a, opd_b, scale, det, frame, envmax, stats, slopes, ref_xy, inv_units, slope_planes, want_frame):
        """aoenv_shwfs_fused (+ the camera pass and the slopes kernel when a noisy detector sits in between).
        opd_b: None, a tensor, or a DMSurfaceRef whose mirror has the separable tables."""
        lib, st = _lib.load(), _lib.stream_ptr(self.device)
        F = opd_a.shape[0]
        dm_struct, tables, b_tensor = None, None, None
        if isinstance(opd_b, DMSurfaceRef):
            tables = opd_b.dm.fused_tables()
            if tables is None:
                b_tensor = opd_b.tensor()
        elif opd_b is not None:
            b_tensor = opd_b
        plan = self._fused_plan(tables)
        if tables is not None:
            rows = opd_b.rows                       # T = C gx of this surface (aoenv_dm_rows, run when it was commanded)
            dm_struct = _lib.DmSepStruct()
            dm_struct.rows, dm_struct.wlr, dm_struct.ilr = rows.data_ptr(), plan["wlr"].data_ptr(), plan["ilr"].data_ptr()
            dm_struct.nActP, dm_struct.WL, dm_struct.t_rows = rows.shape[1], plan["WL"], plan["t_rows"]
        noisy = det is not None
        write_frame = want_frame or noisy
        _lib.check(lib.aoenv_shwfs_fused(
            _lib.ptr(opd_a), _lib.ptr(b_tensor), C.byref(dm_struct) if dm_struct is not None else None, _lib.ptr(self._pupil8),
            C.c_float(self._amp0), plan["row_start"], _lib.ptr(plan["order"]), _lib.ptr(plan["nlit"]), _lib.ptr(self._slot_of), F,
            self.nSubap,
            self.n_pix_subap, plan["cluster"], plan["groups"], C.c_float(scale), _lib.ptr(ref_xy), self.nValidSubaperture,
            C.c_float(inv_units), C.c_float(self.threshold_cog), _lib.ptr(frame) if write_frame else None,
            None if (noisy or slopes is None) else _lib.ptr(slopes), slopes.stride(0) if slopes is not None else 0,
            None if noisy else _lib.ptr(slope_planes), 2, _lib.ptr(envmax), _lib.ptr(stats), st), "shwfs_fused")
        if noisy:
            _lib.check(lib.aoenv_shwfs_camera(_lib.ptr(frame), _lib.ptr(self._valid_u8), F, self.nSubap, self.n_pix_subap,
                                              C.byref(det), 0, _lib.ptr(envmax), st), "shwfs_camera")
            _lib.check(lib.aoenv_shwfs_slopes(_lib.ptr(frame), _lib.ptr(envmax), 0, _lib.ptr(self._valid_idx),
                                              self.nValidSubaperture, _lib.ptr(ref_xy), C.c_float(inv_units),
                                              C.c_float(self.threshold_cog), F, self.nSubap, self.n_pix_subap,
                                              _lib.ptr(slopes), slopes.stride(0), _lib.ptr(slope_planes), 2, st), "shwfs_slopes")

    def _second_term(self, opd_b):
        """(opd_b tensor or None, aoenv_dm_sep_t or None): a separable mirror whose surface exists only as commands is
        passed in factored form (T = C gx + row windows) and evaluated inside the kernel; any other surface as a tensor."""
        if isinstance(opd_b, DMSurfaceRef):
            tables = opd_b.dm.fused_tables() if (self.inline_dm and opd_b.dm.lazy_surface) else None
            win = self._dm_windows(tables) if tables is not None else None
            if win is not None and not opd_b.materialised:
                rows = opd_b.rows
                dm_struct = _lib.DmSepStruct()
                dm_struct.rows, dm_struct.wlr, dm_struct.ilr = rows.data_ptr(), win[2].data_ptr(), win[1].data_ptr()
                dm_struct.nActP, dm_struct.WL, dm_struct.t_rows = rows.shape[1], win[0], 0
                return None, dm_struct
            return opd_b.tensor(), None
        return opd_b, None

    def _run(self, opd_a, opd_b, pupil, scale, shared_max, det, frame, envmax, stats, slopes, ref_xy, inv_units,
             slope_planes=None):
        lib, st = _lib.load(), _lib.stream_ptr(self.device)
        F = opd_a.shape[0]
        opd_b, dm_struct = self._second_term(opd_b)
        _lib.check(lib.aoenv_shwfs_frame_dm(_lib.ptr(opd_a), _lib.ptr(opd_b) if dm_struct is None else None,
                                            C.byref(dm_struct) if dm_struct is not None else None, _lib.ptr(self._lit_first),
                                            _lib.ptr(pupil), _lib.ptr(self._amp), _lib.ptr(self._valid_u8), F, self.nSubap,
                                            self.n_pix_subap, C.c_float(scale), C.byref(det) if det is not None else None,
                                            int(shared_max), _lib.ptr(frame), _lib.ptr(envmax), _lib.ptr(stats), st),
                   "shwfs_frame_dm")
        _lib.check(lib.aoenv_shwfs_slopes(_lib.ptr(frame), _lib.ptr(envmax), int(shared_max), _lib.ptr(self._valid_idx),
                                          self.nValidSubaperture, _lib.ptr(ref_xy), C.c_float(inv_units),
                                          C.c_float(self.threshold_cog), F, self.nSubap, self.n_pix_subap,
                                          _lib.ptr(slopes), slopes.stride(0), _lib.ptr(slope_planes), 2, st), "shwfs_slopes")

    def _run_geometric(self, opd_a, opd_b, slopes, inv_units, slope_planes=None, stats=None):
        """aoenv_shwfs_geometric: slopes [F, lds] of OPD = opd_a + opd_b (pupil-less), + the pupil statistics."""
        opd_b, dm_struct = self._second_term(opd_b)
        _lib.check(_lib.load().aoenv_shwfs_geometric(
            _lib.ptr(opd_a), _lib.ptr(opd_b), C.byref(dm_struct) if dm_struct is not None else None,
            _lib.ptr(self.telescope._pupil_f), _lib.ptr(self._flux), _lib.ptr(self._valid_idx), self.nValidSubaperture,
            opd_a.shape[0], self.nSubap, self.n_pix_subap, C.c_float(2 * math.pi / self.telescope.src.wavelength),
            C.c_float(inv_units), _lib.ptr(slopes), slopes.stride(0), _lib.ptr(slope_planes), 2, _lib.ptr(stats),
            _lib.stream_ptr(self.device)), "shwfs_geometric")

    def _measure_terms(self, opd_a, opd_b, env_offset=None):
        """Per-environment measurement (single-frame branch, ShackHartmann.py:522-601) on OPD = opd_a + opd_b
        (opd_b: tensor, None, or a DMSurfaceRef = a DM surface that exists only as commands)."""
        if self._flux_version != getattr(self.telescope.src, "_flux_version", 0) or self.current_nPhoton != self.telescope.src.nPhoton:
            self.initialize_flux()                                       # ShackHartmann.py:515-517,534
        tel = self.telescope
        if self._is_geometric:
            planes = self._signal_planes if gemm.uses_tensor_cores(opd_a.shape[0]) else None
            self._run_geometric(opd_a, opd_b, self._signal, 1.0 / self.slopes_units, planes, self._stats)
            self._signal_is_multi = False
            return
        env_offset = self.env_offset if env_offset is None else env_offset
        det = self.cam.as_struct(env_offset)
        scale = 2 * math.pi / tel.src.wavelength
        planes = self._signal_planes if gemm.uses_tensor_cores(opd_a.shape[0]) else None
        if self._fused_ok(opd_a):
            keep = self.keep_frame or det is not None
            self._run_fused(opd_a, opd_b, scale, det, self._frame, self._envmax, self._stats, self._signal, self._ref_xy,
                            1.0 / self.slopes_units, planes, keep)
            if keep:
                self.cam.frame = self._frame[0] if self.n_envs == 1 else self._frame
            else:
                self._last_inputs = (opd_a, opd_b, scale)
                self.cam._frame_src = self._frame_on_demand
        else:
            self._run(opd_a, opd_b, tel._pupil_f, scale, False, det, self._frame, self._envmax, self._stats, self._signal,
                      self._ref_xy, 1.0 / self.slopes_units, slope_planes=planes)
            self.cam.frame = self._frame[0] if self.n_envs == 1 else self._frame
        self._signal_is_multi = False

    def _frame_on_demand(self):
        """`wfs.cam.frame` of a measurement that did not write it: the fused kernel again, frame only, on the inputs of
        that measurement (the atmosphere OPD buffer and the DM commands are unchanged until the next step)."""
        opd_a, opd_b, scale = self._last_inputs
        self._run_fused(opd_a, opd_b, scale, None, self._frame, None, None, None, self._ref_xy, 1.0, None, True)
        return self._frame[0] if self.n_envs == 1 else self._frame

    def _measure_f64(self, opd, shared_max, ref_xy64, inv_units):
        """Calibration-grade float64 measurement of F wavefronts [F, R, R] with the ideal detector
        (aoenv_shwfs_measure_f64).  Returns slopes [F, 2*nValid] float64."""
        F, R, dev = opd.shape[0], self.telescope.resolution, self.device
        tel = self.telescope
        frame = torch.empty((F, R, R), dtype=torch.float64, device=dev)
        envmax = torch.zeros((1 if shared_max else F,), dtype=torch.int64, device=dev)
        lds = 2 * self.nValidSubaperture
        slopes = torch.zeros((F, lds), dtype=torch.float64, device=dev)
        opd = opd.to(torch.float32).contiguous()
        _lib.check(_lib.load().aoenv_shwfs_measure_f64(
            _lib.ptr(opd), _lib.ptr(tel._pupil_f), _lib.ptr(self._amp), _lib.ptr(self._valid_u8), _lib.ptr(self._valid_idx),
            self.nValidSubaperture, _lib.ptr(ref_xy64), float(inv_units), float(self.threshold_cog), F, self.nSubap,
            self.n_pix_subap, 2 * math.pi / tel.src.wavelength, int(shared_max), _lib.ptr(frame), _lib.ptr(envmax),
            _lib.ptr(slopes), lds, _lib.stream_ptr(dev)), "shwfs_measure_f64")
        return slopes

    def _measure_geometric_f64(self, opd, inv_units):
        """Calibration-grade geometric measurement of F wavefronts [F, R, R] (aoenv_shwfs_geometric_f64).  Returns slopes
        [F, 2*nValid] float64."""
        F, nV = opd.shape[0], self.nValidSubaperture
        slopes = torch.zeros((F, 2 * nV), dtype=torch.float64, device=self.device)
        opd = opd.to(torch.float32).contiguous()
        _lib.check(_lib.load().aoenv_shwfs_geometric_f64(
            _lib.ptr(opd), _lib.ptr(self._flux), _lib.ptr(self._valid_idx), nV, F, self.nSubap, self.n_pix_subap,
            2 * math.pi / self.telescope.src.wavelength, float(inv_units), _lib.ptr(slopes), 2 * nV,
            _lib.stream_ptr(self.device)), "shwfs_geometric_f64")
        return slopes

    def measure_frames(self, opd):
        """Multi-frame branch (ShackHartmann.py:605-674): k wavefronts [k, R, R] (OPD_no_pupil, metres), no
        detector, ONE centroiding threshold for the whole batch.  Returns signal [k, nSignal] (float64: this is
        the calibration path)."""
        if self._is_geometric:                                           # noise-free: the camera is not used
            return self._measure_geometric_f64(opd, 1.0 / self.slopes_units)
        if self.cam.photonNoise or self.cam.readoutNoise:
            raise NotImplementedError("noisy multi-frame measurements are not supported (calibrate with noise='off')")
        return self._measure_f64(opd, True, self._ref_xy64, 1.0 / self.slopes_units)

    def wfs_measure(self, phase_in=None):
        """ShackHartmann.py:511-695."""
        tel = self.telescope
        if phase_in is not None:
            ph = torch.as_tensor(phase_in, dtype=torch.float32, device=self.device)
            ph = ph.unsqueeze(0) if ph.ndim == 2 else ph
            lam = tel.src.wavelength
            tel.OPD = ph * (lam / (2 * math.pi))
        a, b = tel._terms(resolve=False)
        if a.shape[0] == self.n_envs:
            self._measure_terms(a, b)
        else:
            if isinstance(b, DMSurfaceRef):
                b = b.tensor()
            opd = a if b is None else a + b
            self._multi_signal = self.measure_frames(opd)
            self._signal_is_multi = True

    def sh_measure(self, phase_in):
        self.wfs_measure(phase_in=phase_in)

    # ---- results ------------------------------------------------------------------------------------------
    @property
    def signal(self):
        if self._signal_is_multi:
            return self._multi_signal.T                                   # [nSignal, k] as ShackHartmann.py:674
        s = self._signal[:, :self.nSignal]
        return s[0] if self.n_envs == 1 else s

    @property
    def signal_2D(self):
        s = self._signal[:, :self.nSignal]
        nS, nV = self.nSubap, self.nValidSubaperture
        out = torch.zeros((s.shape[0], 2 * nS, nS), dtype=torch.float32, device=self.device)
        vx = torch.as_tensor(self.validLenslets_x, device=self.device)
        vy = torch.as_tensor(self.validLenslets_y, device=self.device)
        out[:, vx, vy] = s[:, :nV]
        out[:, vx + nS, vy] = s[:, nV:]
        return out[0] if self.n_envs == 1 else out

    # ---- initialisation (ShackHartmann.py:254-312) ----------------------------------------------------------
    def initialize_wfs(self):
        self.isInitialized = False
        tel, dev = self.telescope, self.device
        R, nV, nS = tel.resolution, self.nValidSubaperture, self.nSubap
        zero_ref = torch.zeros((2, nV), dtype=torch.float64, device=dev)
        if self._is_geometric:
            # a flat wavefront has zero gradient: the reference slopes are exactly zero
            def centroids(opd):
                return self._measure_geometric_f64(opd.reshape(1, R, R), 1.0)[0]
            self._ref_xy64 = zero_ref
            self._ref_xy = torch.zeros((2, nV), dtype=torch.float32, device=dev)
            self.reference_slopes_maps = np.zeros((2 * nS, nS))
        else:
            def centroids(opd):
                return self._measure_f64(opd.reshape(1, R, R), False, zero_ref, 1.0)[0]
            self._init_reference(centroids)
        self._init_units(centroids)
        self.isInitialized = True
        tel.resetOPD()

    def _init_reference(self, centroids):
        """Reference slopes of the diffractive sensor: the centroids of a flat wavefront."""
        tel, dev = self.telescope, self.device
        R, nV, nS = tel.resolution, self.nValidSubaperture, self.nSubap
        lam = tel.src.wavelength
        flat = centroids(torch.zeros((R, R), dtype=torch.float32, device=dev))
        self._ref_xy64 = flat.reshape(2, nV).contiguous()
        # the float32 step kernels subtract a reference measured by themselves, so that a flat wavefront gives
        # exactly zero signal as in the reference (same code path for both measurements there)
        f32 = dict(dtype=torch.float32, device=dev)
        fr32, em32 = torch.empty((1, R, R), **f32), torch.zeros((1,), dtype=torch.int32, device=dev)
        raw32 = torch.zeros((1, self._lds), **f32)
        zero32 = torch.zeros((1, R, R), **f32)
        if self._fused_ok(zero32):
            self._run_fused(zero32, None, 2 * math.pi / lam, None, fr32, em32, None, raw32, torch.zeros((2, nV), **f32), 1.0,
                            None, False)
        else:
            self._run(zero32, None, tel._pupil_f, 2 * math.pi / lam, False, None, fr32, em32, None, raw32,
                      torch.zeros((2, nV), **f32), 1.0)
        self._ref_xy = raw32[0, :2 * nV].reshape(2, nV).contiguous()
        ref2d = np.zeros((2 * nS, nS))
        f = flat.cpu().numpy()
        ref2d[self.validLenslets_x, self.validLenslets_y] = f[:nV]
        ref2d[self.validLenslets_x + nS, self.validLenslets_y] = f[nV:]
        self.reference_slopes_maps = ref2d

    def _init_units(self, centroids):
        tel, dev = self.telescope, self.device
        R, nV = tel.resolution, self.nValidSubaperture
        lam = tel.src.wavelength
        # slope units from five tip ramps.  Quirk kept (ShackHartmann.py:288-290): tel.pupil is an int array, so
        # `Tip[tel.pupil]` fancy-indexes rows 0/1 and the ramp is normalised by the std of the FULL ramp.
        ramp = np.linspace(0, np.pi, R, endpoint=False)
        tip = np.tile(ramp[None, :], (R, 1))
        if not self.unit_P2V:
            tip = tip / np.std(tip[np.asarray(tel.pupil).astype(int)])
        amp = 10e-9
        mean_slope = np.zeros(5)
        tip_dev = torch.as_tensor(tip, dtype=torch.float64, device=dev)
        for i in range(5):
            opd = (tip_dev * ((i - 2) * amp)).to(torch.float32)
            c = centroids(opd)
            mean_slope[i] = float((c[:nV] - self._ref_xy64[0]).mean())
        self.p = np.polyfit(np.linspace(-2, 2, 5) * amp, mean_slope, deg=1)
        self.slopes_units = float(np.abs(self.p[0]) * (lam / 2 / np.pi))

    def __mul__(self, obj):
        """wfs*cam (ShackHartmann.py:769-782): the detector already ran inside the frame kernel."""
        if getattr(obj, "tag", None) != "detector":
            print("Error light propagated to the wrong type of object")
        return -1
