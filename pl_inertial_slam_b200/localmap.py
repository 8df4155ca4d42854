"""The local map of MapHandler's local-mapping thread, resident on the device (plm_localmap_*, include/plmatch.h).

The reference keeps map_points / map_lines on the host and, for every new keyframe, projects the local landmarks and
matches their representative descriptors against the keyframe's still unmatched features (matchMap2KFPoints / Lines,
src/mapHandler.cpp:583-803).  drivers.matchMap2KF*Full mirror that call from host arrays, re-uploading the whole map
each time.  LocalMap keeps positions, the active flags, med_desc / med_dir and every observation on the device: a
landmark crosses PCIe once, when it is inserted; later calls send only what changes (new observations, moved
positions, flipped flags, culls), and the per-keyframe match runs from the resident rows with copies that do not grow
with the map.  Results equal drivers.matchMap2KF*Full on the same landmarks bit for bit.

    addKeyFrame           -> insert (new landmarks) + add_observations (landmarks seen again)
    local bundle adjustment -> set_positions
    local-map bookkeeping -> set_active / cull
    matchMap2KF*          -> matchMap2KFPoints / matchMap2KFLines (one plm_localmap_match_kf call)
    lookForCommonMatches  -> match_keyframe: both kinds of one keyframe in one call, grids built on the device

One store holds one kind (points or segments), as the reference keeps map_points and map_lines apart.  A landmark's
index is its slot: slots are handed out in insertion order and never reused.  One host thread at a time per store."""
from __future__ import annotations

import ctypes as C
from typing import Optional

import numpy as np

from . import _lib as L
from . import drivers as D
from . import grid as G
from . import matching as M
from .matching import Context


def _p(a: np.ndarray, t):
    return a.ctypes.data_as(t)


def _idx(idx) -> np.ndarray:
    return np.ascontiguousarray(np.asarray(idx, np.int64).reshape(-1), np.int32)


def _params(nnr: float, min_matches: int, max_epip: float) -> L.LocalMapParams:
    """The config values matchMap2KFPoints / Lines read, as plm_localmap_params."""
    p = L.LocalMapParams()
    p.ratio, p.line_sim_th, p.max_epip = float(M.Config.minRatio12P), float(M.Config.lineSimTh), float(max_epip)
    p.nnr, p.ws = float(np.float32(nnr)), int(M.Config.matchingF2FWs)
    p.best_lr, p.fast_matching = int(bool(M.Config.bestLRMatches)), int(bool(D.SlamConfig.fastMatching))
    p.min_matches = int(min_matches)
    return p


class LocalMap:
    """``is_lines``: False = map_points (X = n x 3), True = map_lines (X = n x 6 segment endpoints).  ``lm_capacity`` /
    ``obs_capacity``: landmarks / observation rows the device arenas are first sized for (0 = a small default; they grow
    as needed)."""

    def __init__(self, is_lines: bool, ctx: Optional[Context] = None, lm_capacity: int = 0, obs_capacity: int = 0):
        self.lib = L.load()
        self.is_lines = bool(is_lines)
        self.ctx = ctx
        self.xw = 6 if self.is_lines else 3
        self._h = C.c_void_p()
        L.check(self.lib.plm_localmap_create(M._h(ctx), int(self.is_lines), int(lm_capacity), int(obs_capacity),
                                             C.byref(self._h)), "plm_localmap_create")

    def __len__(self) -> int:
        return int(self.lib.plm_localmap_size(self._h))

    @property
    def h2d_bytes(self) -> int:
        return int(self.lib.plm_localmap_h2d_bytes(self._h))

    @property
    def d2h_bytes(self) -> int:
        return int(self.lib.plm_localmap_d2h_bytes(self._h))

    def _x(self, X, n) -> np.ndarray:
        X = np.ascontiguousarray(X, np.float64).reshape(-1, self.xw)
        if len(X) != n:
            raise ValueError(f"X needs {n} rows of {self.xw} doubles")
        return X

    @staticmethod
    def _dir(d, n) -> np.ndarray:
        d = np.ascontiguousarray(d, np.float64).reshape(-1, 3)
        if len(d) != n:
            raise ValueError(f"dir needs {n} rows of 3 doubles")
        return d

    def insert(self, X, desc: np.ndarray, dir) -> np.ndarray:
        """New landmarks with one observation each (the MapPoint / MapLine constructors) -> their indices."""
        d, pd, n, step = L.desc_args(np.asarray(desc, np.uint8).reshape(-1, 32))
        X, dr = self._x(X, n), self._dir(dir, n)
        first = C.c_int(0)
        L.check(self.lib.plm_localmap_insert(self._h, n, _p(X, L.f64p), pd, step, _p(dr, L.f64p), C.byref(first)),
                "plm_localmap_insert")
        return np.arange(first.value, first.value + n, dtype=np.int32)

    def add_observations(self, lm_idx, desc: np.ndarray, dir) -> None:
        """Observation i (desc row i, dir row i) appended to landmark lm_idx[i], in order; med_desc / med_dir of every
        touched landmark recomputed (updateAverageDescDir of the final lists)."""
        idx = _idx(lm_idx)
        d, pd, n, step = L.desc_args(np.asarray(desc, np.uint8).reshape(-1, 32))
        if len(idx) != n:
            raise ValueError("one landmark index per observation")
        dr = self._dir(dir, n)
        L.check(self.lib.plm_localmap_add_observations(self._h, n, _p(idx, L.i32p), pd, step, _p(dr, L.f64p)),
                "plm_localmap_add_observations")

    def set_positions(self, idx, X) -> None:
        idx = _idx(idx)
        X = self._x(X, len(idx))
        L.check(self.lib.plm_localmap_set_positions(self._h, len(idx), _p(idx, L.i32p), _p(X, L.f64p)),
                "plm_localmap_set_positions")

    def set_active(self, idx, val) -> None:
        """The selection byte of each landmark: local, and not yet observed from this keyframe."""
        idx = _idx(idx)
        v = np.ascontiguousarray(np.broadcast_to(np.asarray(val, np.uint8), idx.shape))
        L.check(self.lib.plm_localmap_set_active(self._h, len(idx), _p(idx, L.i32p), _p(v, L.u8p)),
                "plm_localmap_set_active")

    def cull(self, idx) -> None:
        """map_points[i] = NULL: never selected again."""
        idx = _idx(idx)
        L.check(self.lib.plm_localmap_cull(self._h, len(idx), _p(idx, L.i32p)), "plm_localmap_cull")

    def landmarks(self, idx) -> dict:
        """Read back -> dict(X, med_desc, med_dir, n_obs) for the given live landmarks."""
        idx = _idx(idx)
        n = len(idx)
        X, md = np.zeros((n, self.xw)), np.zeros((n, 32), np.uint8)
        mdir, no = np.zeros((n, 3)), np.zeros(n, np.int32)
        L.check(self.lib.plm_localmap_read(self._h, n, _p(idx, L.i32p), _p(X, L.f64p), _p(md, L.u8p), _p(mdir, L.f64p),
                                           _p(no, L.i32p)), "plm_localmap_read")
        return dict(X=X, med_desc=md, med_dir=mdir, n_obs=no)

    def _match(self, view: L.MapView, desc2: np.ndarray, cs, ci, dirs2, feat, nnr: float, min_matches: int,
               max_epip: float) -> dict:
        d2, p2, n2, step = L.desc_args(np.asarray(desc2, np.uint8).reshape(-1, 32))
        cs = np.ascontiguousarray(cs, np.int32)
        ci = np.ascontiguousarray(ci if len(ci) else np.zeros(1, np.int32), np.int32)
        feat = np.ascontiguousarray(feat, np.float64)
        kf = L.LocalMapKf()
        kf.desc, kf.step = d2.ctypes.data, step.value
        kf.cell_start, kf.cell_items, kf.feat = cs.ctypes.data, ci.ctypes.data, feat.ctypes.data
        if dirs2 is not None:
            dirs2 = np.ascontiguousarray(dirs2, np.float64).reshape(-1, 2)
            kf.dirs2 = dirs2.ctypes.data
        kf.n2, kf.grid_rows, kf.grid_cols = n2, G.GRID_ROWS, G.GRID_COLS
        p = _params(nnr, min_matches, max_epip)
        cap = max(len(self), 1)
        sel, m12, ok = np.zeros(cap, np.int32), np.zeros(cap, np.int32), np.zeros(cap, np.uint8)
        n_sel, count = C.c_int(0), C.c_int(0)
        L.check(self.lib.plm_localmap_match_kf(self._h, C.byref(view), C.byref(kf), C.byref(p), _p(sel, L.i32p),
                                               _p(m12, L.i32p), _p(ok, L.u8p), C.byref(n_sel), C.byref(count)),
                "plm_localmap_match_kf")
        k = n_sel.value
        return dict(sel=sel[:k].copy(), m12=m12[:k].copy(), ok=ok[:k].copy(), matches=count.value)

    def matchMap2KFPoints(self, view: L.MapView, unmatched_points_px: np.ndarray, unmatched_pt_desc: np.ndarray) -> dict:
        """MapHandler::matchMap2KFPoints (mapHandler.cpp:583-682) from the resident landmarks -> the dict of
        drivers.matchMap2KFPointsFull (sel, m12, ok, matches)."""
        if self.is_lines:
            raise ValueError("matchMap2KFPoints on a store of segments")
        c = np.asarray(unmatched_points_px, np.float64).reshape(-1, 2)
        cs, ci = G.csr_from_points(c[:, 0] * view.inv_width, c[:, 1] * view.inv_height)
        return self._match(view, unmatched_pt_desc, cs, ci, None, c, M.Config.minRatio12P, D.SlamConfig.minPointMatches,
                           D.SlamConfig.maxKFEpipP)

    def matchMap2KFLines(self, view: L.MapView, unmatched_lines_px: np.ndarray, unmatched_le: np.ndarray,
                         unmatched_ls_desc: np.ndarray) -> dict:
        """MapHandler::matchMap2KFLines (mapHandler.cpp:685-803) from the resident landmarks -> the dict of
        drivers.matchMap2KFLinesFull."""
        if not self.is_lines:
            raise ValueError("matchMap2KFLines on a store of points")
        lines = np.asarray(unmatched_lines_px, np.float32).reshape(-1, 4)
        cs, ci, dirs = D.line_grid(lines, view.inv_width, view.inv_height)
        le = np.asarray(unmatched_le, np.float64).reshape(-1, 3)
        return self._match(view, unmatched_ls_desc, cs, ci, dirs, le, M.Config.minRatio12L, D.SlamConfig.minLineMatches,
                           D.SlamConfig.maxKFEpipL)

    def close(self) -> None:
        if self._h:
            self.lib.plm_localmap_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def match_keyframe(points_map: Optional[LocalMap], lines_map: Optional[LocalMap], view: L.MapView, kp_px, pdesc, pl, ln_px,
                   ldesc, le, grid_rows: int = G.GRID_ROWS, grid_cols: int = G.GRID_COLS) -> dict:
    """The map half of MapHandler::lookForCommonMatches for one keyframe (matchMap2KFPoints, then matchMap2KFLines) in one
    plm_localmap_match_kf_pl call, from the keyframe's raw features: the grids are built on the device.

    kp_px: n_p x 2 float32 pixel keypoints, pdesc: n_p x 32, pl: n_p x 2 for the gate (None = kp_px); ln_px: n_l x 4
    float32 pixel segments, ldesc: n_l x 32, le: n_l x 3.  Either map may be None (that kind is skipped).  Returns
    dict(points=..., lines=..., cost=...): per kind the dict of LocalMap.matchMap2KFPoints / Lines (sel, m12, ok,
    matches), None for a skipped kind; cost = dict(h2d_bytes, d2h_bytes, syncs) of the call."""
    if points_map is not None and points_map.is_lines:
        raise ValueError("points_map holds segments")
    if lines_map is not None and not lines_map.is_lines:
        raise ValueError("lines_map holds points")
    lib = L.load()
    kp = np.ascontiguousarray(np.asarray(kp_px if kp_px is not None else np.zeros((0, 2)), np.float32).reshape(-1, 2))
    ln = np.ascontiguousarray(np.asarray(ln_px if ln_px is not None else np.zeros((0, 4)), np.float32).reshape(-1, 4))
    pd, _, n_p, pstep = L.desc_args(np.asarray(pdesc if pdesc is not None else np.zeros((0, 32)), np.uint8).reshape(-1, 32))
    ld, _, n_l, lstep = L.desc_args(np.asarray(ldesc if ldesc is not None else np.zeros((0, 32)), np.uint8).reshape(-1, 32))
    plv = np.ascontiguousarray(kp if pl is None else np.asarray(pl), np.float64).reshape(-1, 2)
    lev = np.ascontiguousarray(np.asarray(le if le is not None else np.zeros((0, 3)), np.float64)).reshape(-1, 3)
    if len(kp) != n_p or len(plv) != n_p:
        raise ValueError("kp_px / pl need one row per point descriptor")
    if len(ln) != n_l or len(lev) != n_l:
        raise ValueError("ln_px / le need one row per segment descriptor")
    kf = L.LocalMapKfRaw()
    kf.kp, kf.pdesc, kf.pstep, kf.pl = kp.ctypes.data, pd.ctypes.data, pstep.value, plv.ctypes.data
    kf.segs, kf.ldesc, kf.lstep, kf.le = ln.ctypes.data, ld.ctypes.data, lstep.value, lev.ctypes.data
    kf.n_p, kf.n_l, kf.grid_rows, kf.grid_cols = n_p, n_l, int(grid_rows), int(grid_cols)
    pp = _params(M.Config.minRatio12P, D.SlamConfig.minPointMatches, D.SlamConfig.maxKFEpipP)
    pln = _params(M.Config.minRatio12L, D.SlamConfig.minLineMatches, D.SlamConfig.maxKFEpipL)
    out = L.LocalMapPlOut()
    bufs = []
    for m, o in ((points_map, out.p), (lines_map, out.l)):
        cap = max(len(m), 1) if m is not None else 1
        b = (np.zeros(cap, np.int32), np.zeros(cap, np.int32), np.zeros(cap, np.uint8))
        o.sel, o.m12, o.ok = b[0].ctypes.data, b[1].ctypes.data, b[2].ctypes.data
        bufs.append(b)
    L.check(lib.plm_localmap_match_kf_pl(points_map._h if points_map is not None else None,
                                         lines_map._h if lines_map is not None else None, C.byref(view), C.byref(kf),
                                         C.byref(pp), C.byref(pln), C.byref(out)), "plm_localmap_match_kf_pl")
    res = {}
    for name, m, o, b in (("points", points_map, out.p, bufs[0]), ("lines", lines_map, out.l, bufs[1])):
        k = o.n_sel
        res[name] = None if m is None else dict(sel=b[0][:k].copy(), m12=b[1][:k].copy(), ok=b[2][:k].copy(), matches=o.count)
    res["cost"] = dict(h2d_bytes=out.h2d_bytes, d2h_bytes=out.d2h_bytes, syncs=out.syncs)
    return res
