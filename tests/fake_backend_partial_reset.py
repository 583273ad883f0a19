"""CPU stand-in for the entry points of the episode reset of a subset of the environments (aoenv_vk_screens_envs,
aoenv_atm_gather_envs, aoenv_atm_ring_envs, aoenv_atm_phase_envs), on top of tests/fake_backend_geometric.py.  Each works
environment by environment on the listed ones only, so that a test can see that nothing else is written.  Test
infrastructure only, like the stand-ins it extends."""
import ctypes as C

import numpy as np

import fake_backend_geometric
from fake_backend import _arr, _val
from fake_backend_geometric import GeometricFakeLib


def _addr(p):
    return p.value if isinstance(p, C.c_void_p) else int(p)


class PartialResetFakeLib(GeometricFakeLib):
    def aoenv_vk_screens_envs(self, seed, screen0, env_idx, S, N, amp, wa, wb, Kp, parts, sh_ex, sh_ey, h_amp, h_mx, h_my, wp,
                              wa_, lda, wb_, ldb, dst, pitch, env_stride, stream):
        """Screen s = the stand-in's screen of stream screen0 + env_idx[s], written into that environment's window."""
        idx = _arr(env_idx, (S,), np.int32)
        for e in idx:
            self.aoenv_vk_screens(seed, int(_val(screen0)) + int(e), 1, N, amp, None, wa, wb, Kp, parts, sh_ex, sh_ey, h_amp, h_mx,
                                  h_my, wp, wa_, lda, wb_, ldb, _addr(dst) + 4 * int(e) * env_stride, pitch, env_stride, stream)
        self.launches -= 5 * S - 5
        return 0

    def aoenv_atm_gather_envs(self, wins, seeds, stream_ids, G, env_idx, k, M, pitch, env_stride, inner_rc, nI, nO, zx, ldz,
                              zx_planes, parts, stream):
        self.launches += 1
        idx = _arr(env_idx, (k,), np.int32)
        rc = _arr(inner_rc, (nI, 2), np.int32)
        z = _arr(zx, (G * k, ldz))
        z[:] = 0
        for g in range(G):
            for j, e in enumerate(idx):
                m = self._window(int(wins[g]) + 4 * int(e) * env_stride, 1, M, pitch, env_stride)[0]
                z[g * k + j, :nI] = m[rc[:, 0], rc[:, 1]]
                key = (int(seeds[g]) * 1000003 + int(stream_ids[g]) * 7 + int(e)) % (2 ** 32)
                z[g * k + j, nI:nI + nO] = np.random.RandomState(key).normal(size=nO)
        return 0

    def aoenv_atm_ring_envs(self, wins, win_offsets, exts, G, env_idx, k, B, M, pitch, env_stride, nO, X, ldx, flag, stream):
        """Ring of the listed environments and all three blocks of their extrema, exact."""
        self.launches += 2
        idx = _arr(env_idx, (k,), np.int32)
        x = _arr(X, (G * k, ldx))
        outer = np.ones((M, M), dtype=bool)
        outer[1:-1, 1:-1] = False
        for g in range(G):
            e3 = _arr(int(exts[g]), (3, B, 2), np.int64)
            off = int(win_offsets[g])
            flatpos = off + np.arange(M)[:, None] * pitch + np.arange(M)[None, :]
            for j, e in enumerate(idx):
                m = self._window(int(wins[g]) + 4 * int(e) * env_stride, 1, M, pitch, env_stride)[0]
                m[outer] = x[g * k + j, :nO]
                keys = (self._key(m).astype(np.uint64) << np.uint64(32)) | flatpos.astype(np.uint64)
                inner = keys[1:-1, 1:-1]
                e3[0, e] = [np.uint64(keys.min()).astype(np.int64), np.uint64(keys.max()).astype(np.int64)]
                e3[1, e] = [np.uint64(inner.min()).astype(np.int64), np.uint64(inner.max()).astype(np.int64)]
                e3[2, e, 0] = (1 << 32) | off
        return 0

    def aoenv_atm_phase_envs(self, h_canvas, h_ext, h_org, L, B, R, M, Mc, pitch, fp_off, roff, coff, wr, wc, wt, opd_scale,
                             env_idx, k, opd_out, stream):
        tmp = np.zeros((B, R, R), dtype=np.float32)
        self.aoenv_atm_phase(h_canvas, h_ext, h_org, L, B, R, M, Mc, pitch, fp_off, roff, coff, wr, wc, wt, opd_scale,
                             tmp.ctypes.data, stream)
        idx = _arr(env_idx, (k,), np.int32)
        _arr(opd_out, (B, R, R))[idx] = tmp[idx]
        return 0


def install(monkeypatch):
    """fake_backend_geometric.install with the partial-reset entry points."""
    geo = fake_backend_geometric.install(monkeypatch)
    lib = PartialResetFakeLib()
    lib.rs = geo.rs
    from rlao_b200 import _lib
    monkeypatch.setattr(_lib, "load", lambda: lib)
    monkeypatch.setattr(_lib, "launch_count", lambda: lib.launches)
    return lib
