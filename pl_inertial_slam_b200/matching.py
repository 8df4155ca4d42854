"""Host-side mirror of the reference's matching interface over the CUDA library.

Same names, argument meaning and error behaviour as stvo-pl/include/matching.h:50-60:

    matchNNR(desc1, desc2, nnr, matches_12) -> int          matching.cpp:41-61
    match(desc1, desc2, nnr, matches_12) -> int             matching.cpp:63-91
    distance(a, b) -> int                                   matching.cpp:93-109
    matchGrid(points1, desc1, grid, desc2, w, matches_12)                       :111-177
    matchGrid(lines1,  desc1, grid, desc2, directions2, w, matches_12)          :179-258

``matches_12`` is the in/out ``std::vector<int>&`` of the reference: pass a Python list (it is
resized to len(desc1) with -1 like ``resize(n, -1)`` and updated in place) or an int32 numpy array of
length n1 (updated in place).  ``Config`` mirrors the static getters the path reads
(stvo-pl/include/config.h:39-105).  All arithmetic runs on the GPU through include/plmatch.h; there
is no CPU fallback.
"""
from __future__ import annotations

import ctypes as C
from typing import List, Optional, Sequence, Tuple, Union

import numpy as np

from . import _lib as L
from .grid import GridStructure, GridWindow


class Config:
    """The Config values the matching path reads, with the defaults of config.cpp:49-51,60,63."""
    bestLRMatches: bool = True   # config.cpp:51
    lrInParallel: bool = True    # config.cpp:49 (no effect here: both directions are one launch)
    minRatio12P: float = 0.9     # config.cpp:60 (EuRoC yaml: 0.9, KITTI: 0.75)
    minRatio12L: float = 0.9     # config.cpp:68
    lineSimTh: float = 0.75      # config.cpp:63
    matchingSWs: int = 10        # config.cpp:91
    matchingF2FWs: int = 3       # config.cpp:92
    maxDistEpip: float = 1.0
    minDisp: float = 1.0
    lineHorizTh: float = 0.1
    stereoOverlapTh: float = 0.75
    lsMinDispRatio: float = 0.7


class Context:
    """A plm_ctx: one CUDA stream + scratch.  ``None`` everywhere means the per-thread default."""

    def __init__(self, device: int = 0):
        self._lib = L.load()
        self._h = C.c_void_p()
        L.check(self._lib.plm_ctx_create(device, C.byref(self._h)), "plm_ctx_create")

    @property
    def handle(self):
        return self._h

    def set_stream(self, cuda_stream: Optional[int]):
        """Launch on an external stream handle (0 = the legacy default stream); None = own stream."""
        ext = cuda_stream is not None
        L.check(self._lib.plm_ctx_set_stream(self._h, C.c_void_p(cuda_stream or 0), int(ext)), "plm_ctx_set_stream")

    def synchronize(self):
        L.check(self._lib.plm_ctx_synchronize(self._h), "plm_ctx_synchronize")

    @property
    def launch_count(self) -> int:
        return int(self._lib.plm_ctx_launch_count(self._h))

    def set_profiling(self, on: bool):
        L.check(self._lib.plm_ctx_set_profiling(self._h, int(bool(on))), "plm_ctx_set_profiling")

    def read_profile(self) -> Tuple[float, int]:
        """(summed device ms of the brute-force slice kernel, launches) since the last read."""
        ms, n = C.c_double(0), C.c_int(0)
        L.check(self._lib.plm_ctx_read_profile(self._h, C.byref(ms), C.byref(n)), "plm_ctx_read_profile")
        return ms.value, n.value

    def measure_int_peaks(self) -> Tuple[float, float]:
        p, l = C.c_double(0), C.c_double(0)
        L.check(self._lib.plm_measure_int_peaks(self._h, C.byref(p), C.byref(l)), "plm_measure_int_peaks")
        return p.value, l.value

    def measure_mma_i8_peak(self) -> float:
        """Int8 tensor-core MMA rate of this device, tera-operations/s (plm_measure_mma_i8_peak)."""
        t = C.c_double(0)
        L.check(self._lib.plm_measure_mma_i8_peak(self._h, C.byref(t)), "plm_measure_mma_i8_peak")
        return t.value

    def measure_mma_i8_rate(self, n: int = 256, with_stores: bool = False) -> float:
        """Int8 MMA rate at 128 x n x 32 (n = 128 or 256), optionally with concurrent shared-memory stores, TOPS
        (plm_measure_mma_i8_rate)."""
        t = C.c_double(0)
        L.check(self._lib.plm_measure_mma_i8_rate(self._h, n, 1 if with_stores else 0, C.byref(t)), "plm_measure_mma_i8_rate")
        return t.value

    def close(self):
        if self._h:
            self._lib.plm_ctx_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def _h(ctx: Optional[Context]):
    return ctx.handle if ctx is not None else None


MatchVec = Union[List[int], np.ndarray]


def _m12_in(matches_12: Optional[MatchVec], n1: int) -> np.ndarray:
    """std::vector<int>::resize(n1, -1) on the caller's vector, as an int32 work buffer."""
    buf = np.full(n1, -1, np.int32)
    if matches_12 is not None:
        k = min(len(matches_12), n1)
        if k:
            buf[:k] = np.asarray(matches_12[:k], np.int32)
    return buf


def _m12_out(matches_12: Optional[MatchVec], buf: np.ndarray) -> None:
    if matches_12 is None:
        return
    if isinstance(matches_12, np.ndarray):
        if len(matches_12) != len(buf):
            raise ValueError("numpy matches_12 must already have len(desc1) entries")
        matches_12[:] = buf
    else:
        matches_12[:] = buf.tolist()


class Pending:
    """Result of a matcher call recorded inside a FrameSession: `.value` (the reference's int return) and the match
    vector are defined once the session has ended."""

    def __init__(self):
        self.value = None

    def __int__(self):
        if self.value is None:
            raise RuntimeError("the frame session has not ended yet")
        return int(self.value)


_sessions = {}


def _session_key(ctx: Optional[Context]):
    import threading
    return ("ctx", id(ctx)) if ctx is not None else ("tls", threading.get_ident())


class FrameSession:
    """plm_frame_begin / plm_frame_end: the matcher calls of one frame (stereo matchGrid for points and lines, temporal
    match for points and lines) recorded and executed as ONE host <-> device round trip.

        with M.FrameSession(ctx) as fs:
            a = M.matchGrid(xy, d1, grid, d2, w, m_stereo, ctx=ctx)    # -> Pending
            b = M.match(prev, curr, 0.9, m_temporal, ctx=ctx)           # -> Pending
        int(a), int(b), m_stereo, m_temporal                           # defined after the `with` block
    """

    def __init__(self, ctx: Optional[Context] = None):
        self.ctx = ctx
        self._fin = []

    def __enter__(self):
        L.check(L.load().plm_frame_begin(_h(self.ctx)), "plm_frame_begin")
        _sessions[_session_key(self.ctx)] = self
        return self

    def _defer(self, n, matches_12, buf, keep):
        p = Pending()

        def fin(keep=keep):
            _m12_out(matches_12, buf)
            p.value = n.value
        self._fin.append(fin)
        return p

    def __exit__(self, exc_type, exc, tb):
        _sessions.pop(_session_key(self.ctx), None)
        st = L.load().plm_frame_end(_h(self.ctx))
        if exc_type is None:
            L.check(st, "plm_frame_end")
            for f in self._fin:
                f()
        self._fin = []
        return False


def distance(a: np.ndarray, b: np.ndarray, ctx: Optional[Context] = None) -> int:
    a = np.ascontiguousarray(a, np.uint8).reshape(1, 32)
    b = np.ascontiguousarray(b, np.uint8).reshape(1, 32)
    out = np.zeros(1, np.int32)
    L.check(L.load().plm_hamming256(_h(ctx), a.ctypes.data_as(L.u8p), 32, b.ctypes.data_as(L.u8p), 32, 1,
                                    out.ctypes.data_as(L.i32p)), "distance")
    return int(out[0])


def distances(a: np.ndarray, b: np.ndarray, ctx: Optional[Context] = None) -> np.ndarray:
    """Row-wise StVO::distance over two n x 32 matrices."""
    a, pa, n, sa = L.desc_args(a)
    b, pb, nb, sb = L.desc_args(b)
    if n != nb:
        raise ValueError("row counts differ")
    out = np.zeros(n, np.int32)
    L.check(L.load().plm_hamming256(_h(ctx), pa, sa, pb, sb, n, out.ctypes.data_as(L.i32p)), "distances")
    return out


def knn2(desc1: np.ndarray, desc2: np.ndarray, idx_base: int = 0, ctx: Optional[Context] = None) -> np.ndarray:
    """cv::BFMatcher::knnMatch(k=2) as packed keys: n1 x 2 uint64, (dist << 32 | idx)."""
    d1, p1, n1, s1 = L.desc_args(desc1)
    d2, p2, n2, s2 = L.desc_args(desc2)
    top2 = np.empty((n1, 2), np.uint64)
    L.check(L.load().plm_knn2(_h(ctx), p1, n1, s1, p2, n2, s2, idx_base, top2.ctypes.data_as(L.u64p)), "knn2")
    return top2


def matchNNR(desc1: np.ndarray, desc2: np.ndarray, nnr: float, matches_12: Optional[MatchVec] = None,
             ctx: Optional[Context] = None) -> int:
    d1, p1, n1, s1 = L.desc_args(desc1)
    d2, p2, n2, s2 = L.desc_args(desc2)
    buf = _m12_in(matches_12, n1)
    n = C.c_int(0)
    st = L.load().plm_match_nnr(_h(ctx), p1, n1, s1, p2, n2, s2, C.c_float(nnr), buf.ctypes.data_as(L.i32p),
                                C.byref(n))
    if st == L.PLM_E_TRAIN:
        # knnMatch yields < 2 neighbours per row (or no rows at all): matching.cpp:50-51 / :54
        raise RuntimeError("[matchNNR] Different size for matches and descriptors!")
    L.check(st, "matchNNR")
    sess = _sessions.get(_session_key(ctx))
    if sess is not None:
        return sess._defer(n, matches_12, buf, (d1, d2))
    _m12_out(matches_12, buf)
    return n.value


def match(desc1: np.ndarray, desc2: np.ndarray, nnr: float, matches_12: Optional[MatchVec] = None,
          ctx: Optional[Context] = None) -> int:
    d1, p1, n1, s1 = L.desc_args(desc1)
    d2, p2, n2, s2 = L.desc_args(desc2)
    buf = _m12_in(matches_12, n1)
    n = C.c_int(0)
    st = L.load().plm_match(_h(ctx), p1, n1, s1, p2, n2, s2, C.c_float(nnr), int(bool(Config.bestLRMatches)),
                            buf.ctypes.data_as(L.i32p), C.byref(n))
    if st == L.PLM_E_TRAIN:
        raise RuntimeError("[matchNNR] Different size for matches and descriptors!")
    L.check(st, "match")
    sess = _sessions.get(_session_key(ctx))
    if sess is not None:
        return sess._defer(n, matches_12, buf, (d1, d2))
    _m12_out(matches_12, buf)
    return n.value


def _grid_csr(grid) -> Tuple[np.ndarray, np.ndarray, int, int]:
    if isinstance(grid, GridStructure):
        cs, ci = grid.to_csr()
        return cs, ci, grid.rows, grid.cols
    cs, ci, rows, cols = grid  # pre-flattened (cell_start, cell_items, rows, cols)
    return np.ascontiguousarray(cs, np.int32), np.ascontiguousarray(ci, np.int32), int(rows), int(cols)


def _win(w) -> np.ndarray:
    return w.as_array() if isinstance(w, GridWindow) else np.ascontiguousarray(w, np.int32)


def matchGrid(features1, desc1: np.ndarray, grid, desc2: np.ndarray, *args, ctx: Optional[Context] = None) -> int:
    """Both overloads of StVO::matchGrid, resolved like C++ does by the argument list:

    points: matchGrid(points1, desc1, grid, desc2, w, matches_12)
    lines:  matchGrid(lines1,  desc1, grid, desc2, directions2, w, matches_12)

    points1 = n1 x 2 (x, y) cell coords; lines1 = n1 x 4 (sx, sy, ex, ey) or n1 x 2 x 2.
    grid = GridStructure or (cell_start, cell_items, rows, cols).
    """
    if len(args) == 2:
        (w, matches_12), directions2 = args, None
    elif len(args) == 3:
        directions2, w, matches_12 = args
    else:
        raise TypeError("matchGrid(features1, desc1, grid, desc2, [directions2,] w, matches_12)")
    d1, p1, n1, s1 = L.desc_args(desc1)
    d2, p2, n2, s2 = L.desc_args(desc2)
    is_lines = directions2 is not None
    coords = np.ascontiguousarray(features1, np.int32).reshape(-1, 4 if is_lines else 2)
    if coords.shape[0] != n1:
        raise RuntimeError("[matchGrid] Each line needs a corresponding descriptor!" if is_lines
                           else "[matchGrid] Each point needs a corresponding descriptor!")
    cs, ci, rows, cols = _grid_csr(grid)
    win = _win(w)
    buf = _m12_in(matches_12, n1)
    n = C.c_int(0)
    lib = L.load()
    ci_p = (ci if len(ci) else np.zeros(1, np.int32)).ctypes.data_as(L.i32p)
    if not is_lines:
        st = lib.plm_match_grid_points(_h(ctx), coords.ctypes.data_as(L.i32p), p1, n1, s1, cs.ctypes.data_as(L.i32p),
                                       ci_p, rows, cols, p2, n2, s2, win.ctypes.data_as(L.i32p),
                                       float(Config.minRatio12P), int(bool(Config.bestLRMatches)),
                                       buf.ctypes.data_as(L.i32p), C.byref(n))
    else:
        dirs = np.ascontiguousarray(directions2, np.float64).reshape(-1, 2)
        if dirs.shape[0] < n2:
            raise ValueError("directions2 needs one entry per row of desc2")
        st = lib.plm_match_grid_lines(_h(ctx), coords.ctypes.data_as(L.i32p), p1, n1, s1, cs.ctypes.data_as(L.i32p),
                                      ci_p, rows, cols, p2, n2, s2, dirs.ctypes.data_as(L.f64p),
                                      float(Config.lineSimTh), win.ctypes.data_as(L.i32p), float(Config.minRatio12P),
                                      int(bool(Config.bestLRMatches)), buf.ctypes.data_as(L.i32p), C.byref(n))
    if st == L.PLM_E_GRID:
        raise RuntimeError("[GridStructure] invalid dimension")
    L.check(st, "matchGrid")
    sess = _sessions.get(_session_key(ctx))
    if sess is not None:
        return sess._defer(n, matches_12, buf, (d1, d2, coords, cs, ci, win, directions2 if not is_lines else dirs))
    _m12_out(matches_12, buf)
    return n.value


def stereo_filter_points(kp_l: np.ndarray, kp_r: np.ndarray, matches_12: Sequence[int],
                         ctx: Optional[Context] = None):
    """Gates of StereoFrame::matchStereoPoints (stereoFrame.cpp:162-171) -> (n_kept, keep, disparity)."""
    kp_l = np.ascontiguousarray(kp_l, np.float32).reshape(-1, 2)
    kp_r = np.ascontiguousarray(kp_r, np.float32).reshape(-1, 2)
    m = np.ascontiguousarray(matches_12, np.int32)
    n1 = len(m)
    keep = np.zeros(n1, np.uint8)
    disp = np.zeros(n1, np.float64)
    n = C.c_int(0)
    L.check(L.load().plm_stereo_filter_points(_h(ctx), kp_l.ctypes.data_as(L.f32p), n1, kp_r.ctypes.data_as(L.f32p),
                                              len(kp_r), m.ctypes.data_as(L.i32p), float(Config.maxDistEpip),
                                              float(Config.minDisp), keep.ctypes.data_as(L.u8p),
                                              disp.ctypes.data_as(L.f64p), C.byref(n)), "stereo_filter_points")
    return n.value, keep, disp


def stereo_filter_lines(ln_l: np.ndarray, ln_r: np.ndarray, matches_12: Sequence[int],
                        ctx: Optional[Context] = None):
    """Gates of StereoFrame::matchStereoLines (stereoFrame.cpp:359-385) -> (n_kept, keep, (disp_s, disp_e))."""
    ln_l = np.ascontiguousarray(ln_l, np.float32).reshape(-1, 4)
    ln_r = np.ascontiguousarray(ln_r, np.float32).reshape(-1, 4)
    m = np.ascontiguousarray(matches_12, np.int32)
    n1 = len(m)
    keep = np.zeros(n1, np.uint8)
    disp = np.zeros((n1, 2), np.float64)
    n = C.c_int(0)
    L.check(L.load().plm_stereo_filter_lines(_h(ctx), ln_l.ctypes.data_as(L.f32p), n1, ln_r.ctypes.data_as(L.f32p),
                                             len(ln_r), m.ctypes.data_as(L.i32p), float(Config.minDisp),
                                             float(Config.lineHorizTh), float(Config.stereoOverlapTh),
                                             float(Config.lsMinDispRatio), keep.ctypes.data_as(L.u8p),
                                             disp.ctypes.data_as(L.f64p), C.byref(n)), "stereo_filter_lines")
    return n.value, keep, disp


def line_pair_filter(lines1: np.ndarray, lines2: np.ndarray, matches_12: Sequence[int], overlap_th: float = 0.75,
                     line_sim_th: Optional[float] = None, ctx: Optional[Context] = None):
    """Opt-in geometric filter for matched line pairs (BASELINE config 2): StereoFrame::lineSegmentOverlap
    (stereoFrame.cpp:521-627) of line1[i1] against line2[m12[i1]] and the direction test of matchGrid (matching.cpp:221)
    -> (n_kept, keep, overlap, sim).  line_sim_th defaults to Config.lineSimTh."""
    ln1 = np.ascontiguousarray(lines1, np.float32).reshape(-1, 4)
    ln2 = np.ascontiguousarray(lines2, np.float32).reshape(-1, 4)
    m = np.ascontiguousarray(matches_12, np.int32)
    n1 = len(m)
    if len(ln1) != n1:
        raise RuntimeError("[line_pair_filter] Each line needs a match entry!")
    keep = np.zeros(n1, np.uint8)
    overlap, sim = np.zeros(n1, np.float64), np.zeros(n1, np.float64)
    n = C.c_int(0)
    th = float(Config.lineSimTh if line_sim_th is None else line_sim_th)
    L.check(L.load().plm_line_pair_filter(_h(ctx), ln1.ctypes.data_as(L.f32p), n1, ln2.ctypes.data_as(L.f32p), len(ln2),
                                          m.ctypes.data_as(L.i32p), float(overlap_th), th, keep.ctypes.data_as(L.u8p),
                                          overlap.ctypes.data_as(L.f64p), sim.ctypes.data_as(L.f64p), C.byref(n)),
            "line_pair_filter")
    return n.value, keep, overlap, sim
