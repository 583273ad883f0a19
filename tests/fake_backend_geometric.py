"""CPU stand-in for the geometric Shack-Hartmann entry points of libaoenv_b200.so (aoenv_shwfs_geometric,
aoenv_shwfs_geometric_f64 and the geometric part of aoenv_sh_step), on top of tests/fake_backend.py.  Test infrastructure
only, like the stand-in it extends."""
import numpy as np

import fake_backend
from fake_backend import FakeLib, _arr, _val


def _gradient_means(total, flux, vi, nS, n):
    """np.gradient of each [R, R] map (unit spacing), flux-weighted mean over lenslet k = vi[t] -> [F, 2, nV]."""
    gy, gx = np.gradient(total, axis=(1, 2))
    tiles = lambda img: img.reshape(img.shape[0], nS, n, nS, n).transpose(0, 1, 3, 2, 4).reshape(img.shape[0], nS * nS, n * n)[:, vi]
    w = flux[None].astype(np.float64)
    sw = tiles(w).sum(axis=2)
    return np.stack([tiles(w * gx).sum(axis=2) / sw, tiles(w * gy).sum(axis=2) / sw], axis=1)


class GeometricFakeLib(FakeLib):
    def aoenv_shwfs_geometric(self, opd_a, opd_b, dm, pupil, flux, valid_idx, nV, B, nS, n, phase_scale, inv_units, slopes, lds,
                              slope_planes, parts, stats, stream):
        """Second term from the factored DM like the stand-in's aoenv_shwfs_frame_dm, statistics like its
        aoenv_shwfs_frame."""
        R = nS * n
        d = dm._obj if hasattr(dm, "_obj") else dm
        if d is not None and getattr(d, "rows", None):
            assert not opd_b
            WL, half = d.WL, (d.WL + 1) // 2
            hp = (half + 3) // 4 * 4
            trows = _arr(d.rows, (B, d.nActP, R)).astype(np.float64)
            wlr, ilr = _arr(d.wlr, (R, 2 * hp)).astype(np.float64), _arr(d.ilr, (nS,), np.int32)
            b_ = np.zeros((B, R, R), dtype=np.float32)
            for y in range(R):
                i0 = int(ilr[y // n])
                w = np.array([wlr[y, (t // half) * hp + t % half] for t in range(WL)])
                b_[:, y, :] = np.einsum("t,btx->bx", w, trows[:, i0:i0 + WL, :])
            kt_from_b = False
        else:
            b_ = _arr(opd_b, (B, R, R))
            kt_from_b = b_ is not None
        self.launches += 2 if stats else 1
        a = _arr(opd_a, (B, R, R))
        total = a + b_ if b_ is not None else a.copy()
        st = _arr(stats, (B, 4), np.float64)
        if st is not None:
            m = _arr(pupil, (R, R)) > 0
            for e in range(B):
                ka = a[e][R // 2, R // 2]
                kt = total[e][R // 2, R // 2] if kt_from_b else ka
                da, dt = (a[e] - ka)[m].astype(np.float64), (total[e] - kt)[m].astype(np.float64)
                st[e] = [da.sum(), (da ** 2).sum(), dt.sum(), (dt ** 2).sum()]
        g = _gradient_means(total.astype(np.float64), _arr(flux, (R, R)), _arr(valid_idx, (nV,), np.int32), nS, n)
        _arr(slopes, (B, lds))[:, :2 * nV] = (g.reshape(B, 2 * nV) * float(_val(phase_scale)) * float(_val(inv_units))).astype(np.float32)
        return 0

    def aoenv_shwfs_geometric_f64(self, opd, flux, valid_idx, nV, F, nS, n, phase_scale, inv_units, slopes, lds, stream):
        self.launches += 1
        R = nS * n
        g = _gradient_means(_arr(opd, (F, R, R)).astype(np.float64), _arr(flux, (R, R)), _arr(valid_idx, (nV,), np.int32), nS, n)
        _arr(slopes, (F, lds), np.float64)[:, :2 * nV] = g.reshape(F, 2 * nV) * float(_val(phase_scale)) * float(_val(inv_units))
        return 0

    def aoenv_sh_step(self, c, part, opd_a, rows_cur, det, action, coefs_next, rows_next, obs, reward, strehl, total, residual,
                      stream):
        """With c.geometric, part 1 is aoenv_shwfs_geometric (as csrc/step.cu); the rest as the diffractive stand-in."""
        from rlao_b200 import _lib as L
        s = c._obj if hasattr(c, "_obj") else c
        if (part & 1) and s.geometric:
            dm = L.DmSepStruct()
            dm.rows, dm.wlr, dm.ilr, dm.nActP, dm.WL = rows_cur, s.dm.wlr, s.dm.ilr, s.dm.nActP, s.dm.WL
            self.aoenv_shwfs_geometric(opd_a, None, dm, s.pupil, s.amp, s.valid_idx, s.nV, s.B, s.nS, s.n, s.phase_scale,
                                       s.inv_units, s.slopes, s.lds, None, 2, s.stats, stream)
            part &= ~1
        if part:
            return super().aoenv_sh_step(c, part, opd_a, rows_cur, det, action, coefs_next, rows_next, obs, reward, strehl,
                                         total, residual, stream)
        return 0


def install(monkeypatch):
    """fake_backend.install with the geometric entry points."""
    fake = fake_backend.install(monkeypatch)
    geo = GeometricFakeLib()
    geo.rs = fake.rs
    from rlao_b200 import _lib
    monkeypatch.setattr(_lib, "load", lambda: geo)
    monkeypatch.setattr(_lib, "launch_count", lambda: geo.launches)
    return geo
