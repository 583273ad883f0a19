"""Atmosphere — mirror of OOPAO/Atmosphere.py (on-axis NGS, fov = 0), batched over environments.

Every environment owns its own set of layer maps (independent turbulence realisations); the wind vector,
r0, L0 and the Cn2 profile belong to the Atmosphere object and are therefore shared by all environments, so
the integer-pixel extrusions (`add_row`) fire on the same step for the whole batch and become one GEMM
X[B, nO] = [Z | xi][B, nI+nO] @ [A | B]^T.

HBM layout: canvases[layer][2][B][Mc][pitch] float32 — the reference's (R+6)^2 map is a WINDOW at a movable origin
inside a canvas of side Mc = M + slack: add_row moves the origin by -step and writes only the 4M-4 ring pixels
(the reference copies the whole map); the window is re-centred into the other canvas once every `slack` events.
ext[layer][B][2] uint64 (window extrema with position, for the interpolation clip), opd[B][R][R] (OPD_no_pupil, m).
"""
import ctypes as C
import math
import os
import time

import numpy as np
import torch
from numpy.random import RandomState

from . import _lib, gemm
from .tools import vonkarman as vk


class _LayerView:
    """`atm.layer_k` — the handful of per-layer attributes callers poke at (Atmosphere.py:192-298)."""

    def __init__(self, atm, index):
        self._atm, self._i = atm, index
        # the shift bookkeeping lives in the state block shared with the library (aoenv_atm_state_t): the same numbers
        # whether a frame is sequenced here (_plan_layer / _extrude_group) or by aoenv_atm_update
        self._c = atm._cstate.layer[index]
        self._ratio = np.ctypeslib.as_array(self._c.ratio)
        self._buff = np.ctypeslib.as_array(self._c.buff)
        self.altitude = atm.altitude[index]
        self.windSpeed = atm._windSpeed[index]
        self.direction = atm._windDirection[index]
        self.vY = self.windSpeed * np.cos(np.deg2rad(self.direction))
        self.vX = self.windSpeed * np.sin(np.deg2rad(self.direction))
        self.ratio = np.zeros(2)
        self.buff = np.zeros(2)
        self.notDoneOnce = True
        self.resolution = atm._ops.layer_res
        self.D = atm._ops.layer_D
        self.seed = index
        self.events = 0           # number of add_row calls so far (Philox stream id)
        self.philox_seed = 0

    ratio = property(lambda self: self._ratio, lambda self, v: self._ratio.__setitem__(slice(None), v))
    buff = property(lambda self: self._buff, lambda self, v: self._buff.__setitem__(slice(None), v))
    vX = property(lambda self: self._c.vX, lambda self, v: setattr(self._c, "vX", float(v)))
    vY = property(lambda self: self._c.vY, lambda self, v: setattr(self._c, "vY", float(v)))
    events = property(lambda self: self._c.events, lambda self, v: setattr(self._c, "events", int(v)))
    philox_seed = property(lambda self: self._c.philox_seed, lambda self, v: setattr(self._c, "philox_seed", int(v)))
    notDoneOnce = property(lambda self: bool(self._c.not_done_once), lambda self, v: setattr(self._c, "not_done_once", int(bool(v))))

    @property
    def mapShift(self):
        a = self._atm
        if a._prefetched:                    # a frame computed ahead on the side stream may still be writing the ring
            a._wait_prefetch()
        oy, ox = a._org[self._i]
        m = a._maps[self._i, a._cur[self._i], :, oy:oy + a._M, ox:ox + a._M]
        return m[0] if a.n_envs == 1 else m

    @property
    def A(self):
        return self._atm._ops.A

    @property
    def B(self):
        return self._atm._ops.B


class _CurView:
    """atm._cur[i]: canvas buffer in use, stored in the shared state block."""

    def __init__(self, st):
        self._st = st

    def __getitem__(self, i):
        return self._st.layer[i].cur

    def __setitem__(self, i, v):
        self._st.layer[i].cur = int(v)


class _OrgView:
    """atm._org[i] = [row, col]: window origin inside the canvas, stored in the shared state block."""

    def __init__(self, st):
        self._st = st

    def __getitem__(self, i):
        o = self._st.layer[i].org
        return [o[0], o[1]]

    def __setitem__(self, i, v):
        o = self._st.layer[i].org
        o[0], o[1] = int(v[0]), int(v[1])


class Atmosphere:
    def __init__(self, telescope, r0, L0, windSpeed, fractionalR0, windDirection, altitude, mode=2, param=None,
                 asterism=None, rng="philox", seed=0, warp_kernel="lagrange018", env_offset=0, canvas_slack=96):
        """`rng`: 'philox' — device counter-based streams (production); 'reference' — the reference's MT19937
        streams for environment 0 (RandomState(42 + 1000*layer) etc., Atmosphere.py:201,579), offset by
        104729*env for the others: host-generated, for parity runs and small batches.
        `env_offset`: global index of this shard's first environment (multi-GPU sharding)."""
        if asterism is not None or mode != 2:
            raise NotImplementedError("asterisms / screen modes other than 2 are out of scope")
        if telescope.src is None:
            raise AttributeError("The telescope was not coupled to any source object! Make sure to couple it with an src object using src*tel")
        if rng not in ("philox", "reference"):
            raise ValueError("rng must be 'philox' or 'reference'")
        self.hasNotBeenInitialized = True
        self.telescope = telescope
        self.device = telescope.device
        self.n_envs = telescope.n_envs
        self.r0_def = 0.15
        self._r0 = r0
        self._L0 = L0
        self.fractionalR0 = list(fractionalR0)
        self.altitude = list(altitude)
        self.nLayer = len(self.fractionalR0)
        if self.nLayer > 8:
            raise ValueError("at most 8 layers (AOENV_MAX_LAYERS)")
        self._windSpeed = list(windSpeed)
        self._windDirection = list(windDirection)
        self.tag = "atmosphere"
        self.nExtra = 2
        self.wavelength = 500e-9
        self.user_defined_opd = False
        self.native_update = os.environ.get("AOENV_ATM_NATIVE", "1") != "0"     # frames sequenced by aoenv_atm_update
        self.pipelined = False           # set by the environment: update() of the next frame runs ahead on a side stream
        self._prefetched, self._prefetch_event, self._side_stream, self._opd_next = False, None, None, None
        self.sm_partition = None             # rlao_b200.sm_partition.SMPartition: the side stream runs on its own SMs
        self.mode = mode
        self.seeingArcsec = 206265 * (self.wavelength / r0)
        self.rng = rng
        self.seed = int(seed)
        self.env_offset = int(env_offset)
        self.warp_kernel = warp_kernel
        self.canvas_slack = max(1, int(canvas_slack))   # add_row events between two re-centrings of a layer's canvas
        self.xi_queue = None        # optional iterator of [B, nO] tensors: injected innovations (parity runs)
        self.xi_log = None          # set to [] to record every innovation block used
        self.screen_inject = None   # optional [nLayer][B, 2, N, N] normal draws for the next generateNewPhaseScreen (parity runs)

    # ------------------------------------------------------------------------------------------------
    def initializeAtmosphere(self, telescope):
        """Atmosphere.py:145-190."""
        tel = telescope
        self.fov, self.fov_rad = tel.fov, tel.fov_rad
        if tel.fov != 0 and any(a != 0 for a in self.altitude):
            # layers in altitude grow with the field of view (Atmosphere.py:215-218: one set of operators per layer)
            raise NotImplementedError("fov > 0 with layers in altitude is out of scope (ground layers only)")
        dev, B, R = self.device, self.n_envs, tel.resolution
        if self.hasNotBeenInitialized:
            self.initial_r0 = self._r0
            self._ops = vk.VKOperators(R, tel.D, self._L0, self._r0, self.r0_def, dev)
            ops = self._ops
            self._M = ops.layer_res + self.nExtra
            self._S = (self.canvas_slack + 3) // 4 * 4        # multiple of 4: re-centred windows stay 16-byte aligned
            self._Mc = self._M + self._S
            self._pitch = (self._Mc + 3) // 4 * 4
            self._env_stride = self._Mc * self._pitch
            self._nO, self._nI = ops.outer_rc.shape[0], ops.inner_rc.shape[0]
            self._K = (self._nI + self._nO + 15) // 16 * 16
            self._ldx = (self._nO + 3) // 4 * 4
            self._W = torch.zeros((self._nO, self._K), dtype=torch.float32, device=dev)
            self._W[:, :self._nI] = ops.A.to(torch.float32)
            self._W_op = gemm.Operator(self._W, parts=3)       # the extruded ring is advected across the pupil: 2^-24
            self._upload_B()
            self._inner_rc = torch.as_tensor(ops.inner_rc, dtype=torch.int32, device=dev).contiguous()
            self._maps = torch.zeros((self.nLayer, 2, B, self._Mc, self._pitch), dtype=torch.float32, device=dev)
            self._cstate = _lib.AtmState()
            self._cur = _CurView(self._cstate)
            self._org = _OrgView(self._cstate)                       # window origin (row, col) inside the canvas
            # per layer [3][B][2]: block 0 = extrema of the window, block 1 = of its interior, block 2 = previous origin
            # (csrc/atm.cu)
            self._ext = torch.zeros((self.nLayer, 3, B, 2), dtype=torch.int64, device=dev)
            # add_row workspaces hold one row per (layer of a group, environment): layers that extrude in the same
            # round of a step share the operator [A | B] and go through ONE gather / GEMM / ring sequence
            G = self._group_max = min(self.nLayer, _lib.MAX_LAYERS)
            self._flag = torch.zeros((G * B,), dtype=torch.int32, device=dev)
            self._zx = torch.zeros((G * B, self._K), dtype=torch.float32, device=dev)
            self._zx_planes = torch.zeros((self._W_op.parts * G * B, self._K), dtype=torch.bfloat16, device=dev)
            self._X = torch.zeros((G * B, self._ldx), dtype=torch.float32, device=dev)
            self._opd = torch.zeros((B, R, R), dtype=torch.float32, device=dev)
            self._fp_off = 1 + (ops.layer_res // 2 - R // 2)         # crop [1:-1] + centred footprint (:231-232)
            self.ps_loop = ops.layer_D / ops.layer_res
            st = self._cstate
            st.nLayer, st.B, st.R, st.M, st.Mc, st.pitch, st.S = self.nLayer, B, R, self._M, self._Mc, self._pitch, self._S
            st.nI, st.nO, st.ldz, st.ldx, st.group_max, st.parts = self._nI, self._nO, self._K, self._ldx, G, self._W_op.parts
            st.fp_off, st.use_tc = self._fp_off, int(gemm.uses_tensor_cores())
            st.warp_kernel = {"lagrange018": 0, "catmull_rom": 1}.get(self.warp_kernel, -1)
            st.env_stride, st.env_offset = self._env_stride, self.env_offset
            st.sampling_time, st.ps_loop = float(tel.samplingTime), float(self.ps_loop)
            st.opd_scale = self.wavelength / 2 / math.pi
            for i in range(self.nLayer):
                st.weight[i] = math.sqrt(self.fractionalR0[i])
                st.maps[i][0], st.maps[i][1] = self._maps[i, 0].data_ptr(), self._maps[i, 1].data_ptr()
                st.ext[i] = self._ext[i].data_ptr()
            st.inner_rc, st.zx, st.zx_planes = self._inner_rc.data_ptr(), self._zx.data_ptr(), self._zx_planes.data_ptr()
            st.X, st.flag, st.w_f32 = self._X.data_ptr(), self._flag.data_ptr(), self._W.data_ptr()
            self._layers = [_LayerView(self, i) for i in range(self.nLayer)]
            for i, ly in enumerate(self._layers):
                setattr(self, "layer_" + str(i + 1), ly)
            # first screens (Atmosphere.py:251-293): phase seeded with the layer index, ring from RandomState(42+1000 i)
            self._new_screens(screen_seed=lambda i: i, ring_seed=lambda i: 42 + i * 1000)
        else:
            raise NotImplementedError("re-initialising an Atmosphere is not supported; build a new one")
        self.hasNotBeenInitialized = False
        self.generateNewPhaseScreen(seed=0)        # Atmosphere.py:185
        self.update()                              # :188

    def _upload_B(self):
        self._W[:, self._nI:self._nI + self._nO] = self._ops.B.to(torch.float32)
        self._W_op.invalidate()

    # ---- random streams -----------------------------------------------------------------------------
    def _host_xi(self, layer_index):
        ly = self._layers[layer_index]
        xi = np.stack([rs.normal(size=self._nO) for rs in ly.host_rng])
        return torch.as_tensor(xi, dtype=torch.float32, device=self.device)

    def _new_screens(self, screen_seed, ring_seed):
        ops, B, dev = self._ops, self.n_envs, self.device
        N, delta = ops.layer_res, ops.layer_D / ops.layer_res
        for i, ly in enumerate(self._layers):
            if self.rng == "reference":
                ph = np.stack([vk.screen_reference_rng(self._r0, self._L0, N, delta, screen_seed(i) + 104729 * (self.env_offset + e))
                               for e in range(B)])
                phase = torch.as_tensor(ph, dtype=torch.float32, device=dev)
                ly.host_rng = [RandomState(ring_seed(i) + 104729 * (self.env_offset + e)) for e in range(B)]
            else:
                phase = None                       # synthesised on the device straight into the canvas (below)
                ly.philox_seed = (self.seed * 1000003 + ring_seed(i)) & 0xFFFFFFFFFFFFFFFF
                ly.events = 0
            self._cur[i] = 0
            self._org[i] = self._fresh_origin(i)
            oy, ox = self._org[i]
            if phase is not None:
                self._maps[i, 0, :, oy + 1:oy + self._M - 1, ox + 1:ox + self._M - 1] = phase
            else:
                dst = self._maps[i, 0].data_ptr() + 4 * ((oy + 1) * self._pitch + ox + 1)
                self._screen_synth().generate(self._screen_key(screen_seed(i)), self.env_offset, B, dst, self._pitch,
                                              self._env_stride,
                                              inject=self.screen_inject[i] if self.screen_inject is not None else None)
            self._extrude(i, 0, 0, force_rescan=True)
            ly.notDoneOnce = True

    def _screen_synth(self):
        key = (float(self._r0), float(self._L0))
        if getattr(self, "_synth_key", None) != key:
            ops = self._ops
            self._synth = vk.ScreenSynth(self._r0, self._L0, ops.layer_res, ops.layer_D / ops.layer_res, self.device)
            self._synth_key = key
        return self._synth

    def _screen_key(self, screen_seed):
        """Philox key of a layer's screens (the stream of environment e is env_offset + e)."""
        return (self.seed * 1000003 + screen_seed * 7919 + 12345) & 0xFFFFFFFFFFFFFFFF

    # ---- device steps -------------------------------------------------------------------------------
    def _fresh_origin(self, i):
        """Origin with the most head-room for the layer's drift: the origin moves by -sign(v) per event."""
        ly, S = self._layers[i], self._S

        def pick(v, align):
            o = S if v > 0 else (0 if v < 0 else S // 2)
            return o // align * align
        return [pick(ly.vY, 1), pick(ly.vX, 4)]

    def _win_ptr(self, i, buf=None, org=None):
        buf = self._cur[i] if buf is None else buf
        oy, ox = self._org[i] if org is None else org
        return self._maps[i, buf].data_ptr() + 4 * (oy * self._pitch + ox)

    def _compact(self, i):
        """Re-centres layer i's window into the other canvas buffer."""
        oy, ox = self._org[i]
        foy, fox = self._fresh_origin(i)
        cur = self._cur[i]
        _lib.check(_lib.load().aoenv_atm_compact(self._win_ptr(i, cur, (oy, ox)), self._win_ptr(i, 1 - cur, (foy, fox)),
                                                 self.n_envs, self._M, self._pitch, self._env_stride, _lib.ptr(self._ext[i]),
                                                 (foy - oy) * self._pitch + (fox - ox), _lib.stream_ptr(self.device)),
                   "atm_compact")
        self._cur[i], self._org[i] = 1 - cur, [foy, fox]

    def _rescan_extrema(self, i):
        """Exact window extrema of layer i from the maps (after the maps were written from outside: checkpoint restore).
        The ring kernel with force_rescan recomputes them; writing the ring back in place does not change the map."""
        B, M, pitch = self.n_envs, self._M, self._pitch
        oy, ox = self._org[i]
        win = self._maps[i, self._cur[i], :, oy:oy + M, ox:ox + M]
        ring = torch.cat([win[:, 0, :], torch.stack([win[:, 1:M - 1, 0], win[:, 1:M - 1, M - 1]], dim=2).reshape(B, -1),
                          win[:, M - 1, :]], dim=1)                       # numpy boolean-mask order of the outer ring
        self._X[:B, :self._nO] = ring
        _lib.check(_lib.load().aoenv_atm_ring(self._win_ptr(i), B, M, pitch, self._env_stride, oy * pitch + ox, self._nO,
                                              _lib.ptr(self._X), self._ldx, self._ext[i].data_ptr(), _lib.ptr(self._flag), 1,
                                              _lib.stream_ptr(self.device)), "atm_ring")

    def _extrude(self, i, sx, sy, force_rescan=False):
        """add_row (Atmosphere.py:301-311) for layer i and every environment."""
        self._extrude_group([(i, sx, sy)], force_rescan)

    def _extrude_group(self, group, force_rescan=False):
        """add_row for the layers of `group` = [(layer, sx, sy), ...] (distinct layers) and every environment."""
        lib = _lib.load()
        B, M, pitch, S, G = self.n_envs, self._M, self._pitch, self._S, len(group)
        st = _lib.stream_ptr(self.device)
        tc = gemm.uses_tensor_cores(G * B)
        xi = None
        wins, sxs, sys_, seeds, ids = [], [], [], [], []
        for i, sx, sy in group:
            ly = self._layers[i]
            sx, sy = int(sx), int(sy)
            oy, ox = self._org[i]
            if not (0 <= oy - sy <= S and 0 <= ox - sx <= S):
                self._compact(i)
                oy, ox = self._org[i]
                if not (0 <= oy - sy <= S and 0 <= ox - sx <= S):
                    raise RuntimeError("canvas_slack too small for this wind direction change")
            if self.xi_queue is not None or self.rng == "reference":
                assert G == 1, "injected innovations are consumed in the reference's order, one layer at a time"
                if self.xi_queue is not None:
                    xi = torch.as_tensor(next(self.xi_queue), dtype=torch.float32, device=self.device).reshape(B, self._nO).contiguous()
                else:
                    xi = self._host_xi(i)
            if self.xi_log is not None:
                self.xi_log.append(None if xi is None else xi.clone())
            wins.append(self._win_ptr(i))
            sxs.append(sx)
            sys_.append(sy)
            seeds.append(getattr(ly, "philox_seed", 0))
            ids.append(((ly.events << 8) | i) + (self.env_offset << 40))
            ly.events += 1
        planes = _lib.ptr(self._zx_planes) if tc else None
        zx = None if tc else _lib.ptr(self._zx)        # the tensor-core GEMM reads the bf16 planes only: no float32 copy
        if G == 1:
            _lib.check(lib.aoenv_atm_gather(wins[0], B, M, pitch, self._env_stride, sxs[0], sys_[0], _lib.ptr(self._inner_rc),
                                            self._nI, self._nO, _lib.ptr(xi), C.c_uint64(seeds[0]), C.c_uint64(ids[0]),
                                            zx, self._K, planes, self._W_op.parts, st), "atm_gather")
        else:
            _lib.check(lib.aoenv_atm_gather_multi((C.c_void_p * G)(*[w.value if hasattr(w, "value") else w for w in wins]),
                                                  (C.c_int32 * G)(*sxs), (C.c_int32 * G)(*sys_), (C.c_uint64 * G)(*seeds),
                                                  (C.c_uint64 * G)(*ids), G, B, M, pitch, self._env_stride,
                                                  _lib.ptr(self._inner_rc), self._nI, self._nO, None, zx, self._K,
                                                  planes, self._W_op.parts, st), "atm_gather_multi")
        gemm.gemm_tn(self._zx, self._W_op, self._X, G * B, self._nO, backend="tc" if tc else "simt",
                     x_planes=self._zx_planes if tc else None)
        wins, offs, exts = [], [], []
        for i, sx, sy in group:
            oy, ox = self._org[i]
            self._org[i] = [oy - int(sy), ox - int(sx)]
            noy, nox = self._org[i]
            wins.append(self._win_ptr(i))
            offs.append(noy * pitch + nox)
            exts.append(self._ext[i].data_ptr())
        if G == 1:
            _lib.check(lib.aoenv_atm_ring(wins[0], B, M, pitch, self._env_stride, offs[0], self._nO, _lib.ptr(self._X), self._ldx,
                                          exts[0], _lib.ptr(self._flag), int(force_rescan), st), "atm_ring")
        else:
            _lib.check(lib.aoenv_atm_ring_multi((C.c_void_p * G)(*[w.value if hasattr(w, "value") else w for w in wins]),
                                                (C.c_int64 * G)(*offs), (C.c_void_p * G)(*exts), G, B, M, pitch, self._env_stride,
                                                self._nO, _lib.ptr(self._X), self._ldx, _lib.ptr(self._flag), int(force_rescan), st),
                       "atm_ring_multi")

    def _plan_layer(self, i):
        """Integer part of updateLayer (Atmosphere.py:350-404): the add_row steps (sx, sy) layer i takes this frame, in
        order; leaves ly.buff ready for the sub-pixel shift."""
        ly = self._layers[i]
        steps = []
        if ly.vX == 0 and ly.vY == 0:
            return steps
        if ly.notDoneOnce:
            ly.notDoneOnce = False
            ly.ratio = np.array([ly.vX * self.telescope.samplingTime / self.ps_loop,
                                 ly.vY * self.telescope.samplingTime / self.ps_loop])
            ly.buff = np.zeros(2)
        ratio = ly.ratio
        n = np.abs(ratio)
        n[np.isinf(n)] = 0
        n = n.astype(int)
        sgn = np.sign(ratio)
        for _ in range(n.min()):
            steps.append((sgn[0], sgn[1]))
        for _ in range(n.max() - n.min()):
            step = sgn.copy()
            step[n == n.min()] = 0
            steps.append((step[0], step[1]))
        ly.buff = ly.buff + (np.abs(ratio) % 1) * sgn
        if abs(ly.buff[0]) >= 1 or abs(ly.buff[1]) >= 1:
            step = np.sign(ly.buff)
            step[np.abs(ly.buff) < 1] = 0
            steps.append((step[0], step[1]))
        ly.buff = (np.abs(ly.buff) % 1) * np.sign(ly.buff)
        return steps

    def _update_layer(self, i):
        for sx, sy in self._plan_layer(i):
            self._extrude(i, sx, sy)

    def _update_layers(self):
        """All layers of one frame.  Layers are independent, and with the counter-based generator the innovation of
        an add_row depends only on (layer, event number, environment): the r-th add_row of every layer that has
        one this frame is done together.  Injected / host-generated innovations keep the reference's layer-by-layer
        order."""
        if self.xi_queue is not None or self.rng == "reference" or self.nLayer == 1:
            for i in range(self.nLayer):
                self._update_layer(i)
            return
        plans = [self._plan_layer(i) for i in range(self.nLayer)]
        for r in range(max((len(p_) for p_ in plans), default=0)):
            group = [(i, *plans[i][r]) for i in range(self.nLayer) if len(plans[i]) > r]
            for k in range(0, len(group), self._group_max):
                self._extrude_group(group[k:k + self._group_max])

    def _publish(self, out=None, env_idx=None):
        """Sub-pixel shift of every layer + Cn2-weighted sum -> OPD_no_pupil (Atmosphere.py:406-407,439-478); with
        env_idx (int32 device tensor), the rows of those environments only."""
        out = self._opd if out is None else out
        L = self.nLayer
        maps = (C.c_void_p * L)(*[self._maps[i, self._cur[i]].data_ptr() for i in range(L)])
        exts = (C.c_void_p * L)(*[self._ext[i].data_ptr() for i in range(L)])
        org = (C.c_int32 * (2 * L))(*[v for i in range(L) for v in self._org[i]])
        roff, coff = (C.c_int32 * L)(), (C.c_int32 * L)()
        wr, wc, wt = (C.c_float * (4 * L))(), (C.c_float * (4 * L))(), (C.c_float * L)()
        for i, ly in enumerate(self._layers):
            oc, wcol = vk.cubic_tap_weights(float(ly.buff[0]), self.warp_kernel)      # x -> columns
            orow, wrow = vk.cubic_tap_weights(float(ly.buff[1]), self.warp_kernel)    # y -> rows
            roff[i], coff[i] = orow, oc
            for k in range(4):
                wr[4 * i + k], wc[4 * i + k] = wrow[k], wcol[k]
            wt[i] = math.sqrt(self.fractionalR0[i])
        args = (maps, exts, org, L, self.n_envs, self.telescope.resolution, self._M, self._Mc, self._pitch, self._fp_off, roff,
                coff, wr, wc, wt, C.c_float(self.wavelength / 2 / math.pi))
        if env_idx is None:
            _lib.check(_lib.load().aoenv_atm_phase(*args, _lib.ptr(out), _lib.stream_ptr(self.device)), "atm_phase")
        else:
            _lib.check(_lib.load().aoenv_atm_phase_envs(*args, _lib.ptr(env_idx), env_idx.numel(), _lib.ptr(out),
                                                        _lib.stream_ptr(self.device)), "atm_phase_envs")

    def _advance(self, out):
        """One frame: the add_row steps of every layer, then the sub-pixel shift into `out`.  Sequenced by the library
        (aoenv_atm_update, a few microseconds of host time) in the production mode, by the Python methods above when
        innovations are injected, generated on the host or recorded."""
        if (self.native_update and self.rng == "philox" and self.xi_queue is None and self.xi_log is None
                and self._cstate.warp_kernel >= 0):
            tc = self._cstate.use_tc
            self._cstate.sampling_time, self._cstate.env_offset = float(self.telescope.samplingTime), self.env_offset
            _lib.check(_lib.load().aoenv_atm_update(C.byref(self._cstate), _lib.ptr(self._W_op.planes()) if tc else None,
                                                    _lib.ptr(out), _lib.stream_ptr(self.device)), "atm_update")
        else:
            self._update_layers()
            self._publish(out)

    # ---- the next frame, one step ahead, on a second stream -------------------------------------------------
    # atm.update() depends on nothing the rest of env.step computes, and its kernels are bound by HBM (sub-pixel shift,
    # ring writes) while the wavefront sensor is bound by the FP32 pipe: prefetch() issues the update of the NEXT frame on a
    # side stream, into the other OPD buffer, so that the GPU runs it underneath the WFS / reconstruction of the current
    # frame; the next update() only waits for it and swaps the buffers.  Same kernels, same order, same numbers.
    PREFETCH_MIN_PIXELS = 1 << 25        # below this (n_envs x R x R) a step is launch-bound and the second stream only adds
                                         # host work (measured: cfg2, 1024 x 120^2, 5.07 M -> 4.45 M env-steps/s with it)

    def can_prefetch(self):
        if self.pipelined != "force" and (not self.pipelined or self._opd is None
                                          or self._opd.numel() < self.PREFETCH_MIN_PIXELS):
            return False
        return (self.rng == "philox" and self.xi_queue is None and self.xi_log is None
                and not self.user_defined_opd and self._opd is not None and self._opd.is_cuda)

    def prefetch(self):
        """Returns True if the next frame is (now) computed ahead."""
        if self._prefetched:
            return True
        if not self.can_prefetch():
            return False
        dev = self.device
        if self._side_stream is None:
            if self.sm_partition is not None:
                # a stream of the green context that owns the atmosphere's share of the SMs (rlao_b200/sm_partition.py)
                self._side_stream = self.sm_partition.side
            else:
                # same priority as the main stream (measured: a higher one, -1, lets the atmosphere push the WFS kernel
                # aside and the step gets slower, 0.802 vs 0.779 ms; the host-facing loop drops from 1.29 M to 0.98 M)
                self._side_stream = torch.cuda.Stream(dev, priority=int(os.environ.get("AOENV_ATM_PREFETCH_PRIORITY", "0")))
            self._opd_next = torch.empty_like(self._opd)
        main, side = torch.cuda.current_stream(dev), self._side_stream
        # the other OPD buffer was read by the WFS of the previous frame, the canvases by nothing else: everything already
        # queued on the main stream must be done before the side stream starts
        side.wait_event(main.record_event())
        with torch.cuda.stream(side):
            self._advance(self._opd_next)
            self._prefetch_event = side.record_event()
        self._prefetched = True
        return True

    def _wait_prefetch(self):
        """Makes the current stream wait for the frame computed ahead (and for what reset_envs changed in it)."""
        if self._prefetch_event is not None:
            torch.cuda.current_stream(self.device).wait_event(self._prefetch_event)

    def _join_prefetch(self, consume):
        """Makes the current stream wait for a prefetched frame; consume=True makes it the current frame, False drops it
        (the layers have moved on by one frame nobody saw: only for calls that replace the screens anyway)."""
        if not self._prefetched:
            return False
        self._wait_prefetch()
        self._prefetched = False
        if consume:
            self._opd, self._opd_next = self._opd_next, self._opd
        return True

    # ---- public API -----------------------------------------------------------------------------------
    def update(self, OPD=None):
        """Atmosphere.py:409-428."""
        if OPD is None:
            self.user_defined_opd = False
            if not self._join_prefetch(consume=True):
                self._advance(self._opd)
        else:
            self.user_defined_opd = True
            t = torch.as_tensor(OPD, dtype=torch.float32, device=self.device)
            self._opd = (t if t.ndim == 3 else t.unsqueeze(0).expand(self.n_envs, -1, -1)).contiguous().clone()
        if self.telescope.isPaired:
            self * self.telescope

    def generateNewPhaseScreen(self, seed=None):
        """Atmosphere.py:560-592."""
        if seed is None:
            t = time.localtime()
            seed = t.tm_hour * 3600 + t.tm_min * 60 + t.tm_sec
        self._join_prefetch(consume=False)
        self._new_screens(screen_seed=lambda i: seed + i, ring_seed=lambda i: seed + i * 1000)
        # the reference publishes layer.phase (the un-shifted screen) here; buff is reset by notDoneOnce
        for ly in self._layers:
            ly.buff = np.zeros(2)
        self._publish()
        if self.telescope.isPaired:
            self * self.telescope

    # ---- episode reset of a subset of the environments ------------------------------------------------------------
    RESET_STREAM = 1 << 63          # stream-id bit of the ring innovations of reset_envs: no per-frame add_row sets it

    def env_index(self, env_ids):
        """Environment list of reset_envs -> sorted, distinct int32 device tensor.  `env_ids`: host list / array of
        indices, or a bool mask [n_envs] (on the device: counting it costs one synchronisation)."""
        B = self.n_envs
        if torch.is_tensor(env_ids) and env_ids.dtype == torch.bool:
            if tuple(env_ids.shape) != (B,):
                raise ValueError(f"reset mask of shape {tuple(env_ids.shape)}, expected ({B},)")
            return torch.nonzero(env_ids.to(self.device)).reshape(-1).to(torch.int32)
        ids = np.asarray(env_ids.cpu() if torch.is_tensor(env_ids) else env_ids).reshape(-1)
        if ids.dtype == bool:
            if ids.shape != (B,):
                raise ValueError(f"reset mask of shape {ids.shape}, expected ({B},)")
            ids = np.nonzero(ids)[0]
        if ids.size and (not np.issubdtype(ids.dtype, np.integer) or ids.min() < 0 or ids.max() >= B):
            raise ValueError(f"environment indices must be integers in [0, {B})")
        t = torch.from_numpy(np.unique(ids).astype(np.int32))
        if self.device.type == "cuda":               # pinned, so that the upload does not synchronise the stream
            return t.pin_memory().to(self.device, non_blocking=True)
        return t

    def _check_partial_reset(self):
        if self.rng != "philox":
            raise NotImplementedError("reset_envs draws from the counter-based generator: rng='reference' has one host stream "
                                      "per environment and is not supported")
        if self.xi_queue is not None or self.xi_log is not None or self.screen_inject is not None:
            raise NotImplementedError("reset_envs does not support injected or recorded draws (xi_queue / xi_log / screen_inject)")
        if self.user_defined_opd:
            raise NotImplementedError("reset_envs redraws the layers: the OPD was set by the user (update(OPD))")

    def reset_envs(self, env_ids, seed):
        """New episode for the environments `env_ids` only: their windows in every layer get the screen and the outer ring
        that generateNewPhaseScreen(seed) draws for them, the other environments are untouched bit for bit.

        The reset applies to the frame the next update() returns, whatever the prefetch setting: that frame is computed
        now if it has not been computed ahead, then the listed environments' windows are redrawn at the layers' current
        origins and their rows of it are recomputed.  Screen of environment e: the Philox stream generateNewPhaseScreen
        gives it.  Ring: the zero-shift add_row of a new screen, with innovations keyed by (seed, layer, env_offset + e) in
        a stream domain of their own (RESET_STREAM): the layers' add_row counters do not move, so every other environment
        draws exactly what it would have drawn.  The one difference from generateNewPhaseScreen: the sub-pixel phase of the
        wind (layer.buff) and the window origin belong to the layer, so a reset environment keeps the batch's values, where
        a full reset sets buff = 0.

        env_ids: host list / array of indices, or a bool mask [n_envs]; a mask on the device costs one synchronisation
        (to count it).  Returns the int32 device tensor of the reset environments."""
        self._check_partial_reset()
        return self._reset_listed(self.env_index(env_ids), seed)

    def _reset_listed(self, idx, seed):
        """reset_envs for idx = env_index(...)."""
        k = idx.numel()
        if k == 0:
            return idx
        if self._prefetched:
            self._wait_prefetch()
        else:
            # the frame the next update() returns, through the prefetch machinery (in line on the current stream)
            if self._opd_next is None:
                self._opd_next = torch.empty_like(self._opd)
            self._advance(self._opd_next)
            self._prefetched = True
        lib, st, M, pitch, es = _lib.load(), _lib.stream_ptr(self.device), self._M, self._pitch, self._env_stride
        synth = self._screen_synth()
        for i in range(self.nLayer):
            dst = self._win_ptr(i) + 4 * (pitch + 1)                      # window interior, current canvas and origin
            synth.generate(self._screen_key(seed + i), self.env_offset, k, dst, pitch, es, env_idx=idx)
        for g0 in range(0, self.nLayer, self._group_max):
            layers = list(range(g0, min(self.nLayer, g0 + self._group_max)))
            G = len(layers)
            tc = gemm.uses_tensor_cores(G * k)
            wins = (C.c_void_p * G)(*[self._win_ptr(i) for i in layers])
            seeds = (C.c_uint64 * G)(*[(self.seed * 1000003 + seed + i * 1000) & 0xFFFFFFFFFFFFFFFF for i in layers])
            ids = (C.c_uint64 * G)(*[self.RESET_STREAM | (self.env_offset << 40) | i for i in layers])
            _lib.check(lib.aoenv_atm_gather_envs(wins, seeds, ids, G, _lib.ptr(idx), k, M, pitch, es, _lib.ptr(self._inner_rc),
                                                 self._nI, self._nO, None if tc else _lib.ptr(self._zx), self._K,
                                                 _lib.ptr(self._zx_planes) if tc else None, self._W_op.parts, st),
                       "atm_gather_envs")
            gemm.gemm_tn(self._zx, self._W_op, self._X, G * k, self._nO, backend="tc" if tc else "simt",
                         x_planes=self._zx_planes if tc else None)
            offs = (C.c_int64 * G)(*[self._org[i][0] * pitch + self._org[i][1] for i in layers])
            exts = (C.c_void_p * G)(*[self._ext[i].data_ptr() for i in layers])
            _lib.check(lib.aoenv_atm_ring_envs(wins, offs, exts, G, _lib.ptr(idx), k, self.n_envs, M, pitch, es, self._nO,
                                               _lib.ptr(self._X), self._ldx, _lib.ptr(self._flag), st), "atm_ring_envs")
        self._publish(self._opd_next, env_idx=idx)
        if self._opd.is_cuda:
            self._prefetch_event = torch.cuda.current_stream(self.device).record_event()
        return idx

    def __mul__(self, obj):
        """atm*tel / atm*src (Atmosphere.py:632-668).  atm*src points the paired telescope at `src` (which must lie inside
        the field of view) and returns the telescope, so that atm*src*tel*cam chains as in the reference."""
        tag = getattr(obj, "tag", None)
        if tag == "source":
            if obj.coordinates[0] > self.fov / 2:
                raise ValueError(f"The source object zenith ({obj.coordinates[0]}\") is outside of the telescope fov ({self.fov // 2}\")! "
                                 "You can:\n - Reduce the zenith of the source \n - Re-initialize the atmosphere object using a telescope "
                                 "with a larger fov")
            if obj.coordinates[0] != 0 and any(a != 0 for a in self.altitude):
                raise NotImplementedError("off-axis sources through layers in altitude (anisoplanatism) are out of scope")
            obj * self.telescope                       # tel.src = src (flux, wavelength)
            obj = self.telescope
        elif tag != "telescope":
            raise AttributeError("The atmosphere can be multiplied only with a Telescope or a Source object!")
        self.telescope = obj
        obj._set_lazy(self._opd, None)
        obj.isPaired = True
        return obj

    @property
    def OPD_no_pupil(self):
        return self._opd[0] if self.n_envs == 1 else self._opd

    @property
    def OPD(self):
        o = self._opd * self.telescope._pupil_f
        return o[0] if self.n_envs == 1 else o

    # ---- live parameter changes (Atmosphere.py:792-870) -----------------------------------------------------
    @property
    def r0(self):
        return self._r0

    @r0.setter
    def r0(self, val):
        self._r0 = val
        if not self.hasNotBeenInitialized:
            if self._prefetched:             # a frame computed ahead (with the old value) may still be reading the operator
                self._wait_prefetch()
            self.seeingArcsec = 206265 * (self.wavelength / val)
            self._ops.B = self._ops.innovation_factor(val)
            self._upload_B()

    @property
    def L0(self):
        return self._L0

    @L0.setter
    def L0(self, val):
        if not self.hasNotBeenInitialized and val != self._L0:
            raise NotImplementedError("changing L0 rebuilds every operator: construct a new Atmosphere")
        self._L0 = val

    def _refresh_wind(self):
        for i, ly in enumerate(self._layers):
            ly.windSpeed, ly.direction = self._windSpeed[i], self._windDirection[i]
            ly.vY = ly.windSpeed * np.cos(np.deg2rad(ly.direction))
            ly.vX = ly.windSpeed * np.sin(np.deg2rad(ly.direction))
            ly.ratio[0] = ly.vX * self.telescope.samplingTime / self.ps_loop
            ly.ratio[1] = ly.vY * self.telescope.samplingTime / self.ps_loop

    @property
    def windSpeed(self):
        return self._windSpeed

    @windSpeed.setter
    def windSpeed(self, val):
        if not self.hasNotBeenInitialized and len(val) != self.nLayer:
            print("Error! Wrong value for the wind-speed! Make sure that you inpute a wind-speed for each layer")
            return
        self._windSpeed = list(val)
        if not self.hasNotBeenInitialized:
            self._refresh_wind()

    @property
    def windDirection(self):
        return self._windDirection

    @windDirection.setter
    def windDirection(self, val):
        if not self.hasNotBeenInitialized and len(val) != self.nLayer:
            print("Error! Wrong value for the wind-speed! Make sure that you inpute a wind-speed for each layer")
            return
        self._windDirection = list(val)
        if not self.hasNotBeenInitialized:
            self._refresh_wind()
