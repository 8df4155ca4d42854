"""Host mirror of the bag-of-words loop-candidate scoring around the reference's vendored DBoW2
(src/mapHandler.cpp:3116-3237; 3rdparty/DBoW2): ``Vocabulary.transform`` / ``Vocabulary.score`` and the
``insertKFBowVectorP / L / PL`` bookkeeping of the confusion matrix.  The arithmetic runs on the GPU through
``plm_voc_*`` / ``plm_bow_*`` (include/plmatch.h) and is bit-identical to DBoW2's (same fp64 summation
order).  There is no CPU fallback.

The reference loads its two vocabularies from YAML blobs that are not part of the mount
(.MISSING_LARGE_BLOBS: vocabulary/voc.tar.gz); here a vocabulary is the same tree as flat arrays
(``Vocabulary.from_flat``) -- what TemplatedVocabulary::load (TemplatedVocabulary.h:1437-1488) builds.
"""
from __future__ import annotations

import ctypes as C
import math
from typing import List, Optional, Sequence, Tuple

import numpy as np

from . import _lib as L
from .drivers import SlamConfig
from .matching import Config, Context

TF_IDF, TF, IDF, BINARY = 0, 1, 2, 3   # DBoW2::WeightingType (BowVector.h:38-44)
L1_NORM = 0                            # DBoW2::ScoringType (BowVector.h:47-55)

BowVector = Tuple[np.ndarray, np.ndarray]   # (word ids uint32 ascending, values float64)


def _p(a, typ):
    return a.ctypes.data_as(typ)


class Vocabulary:
    """DBoW2::TemplatedVocabulary<FORB::TDescriptor, FORB> (include/mapHandler.h:70) on the device."""

    def __init__(self, child_start, child_ids, node_desc, node_weight, node_word, weighting: int = TF_IDF,
                 scoring: int = L1_NORM, ctx: Optional[Context] = None):
        self.lib = L.load()
        self.ctx = ctx
        cs = np.ascontiguousarray(child_start, np.int32)
        ci = np.ascontiguousarray(child_ids if len(child_ids) else np.zeros(1, np.int32), np.int32)
        nd = np.ascontiguousarray(node_desc, np.uint8).reshape(-1, 32)
        nw = np.ascontiguousarray(node_weight, np.float64)
        wd = np.ascontiguousarray(node_word, np.int32)
        if not (len(cs) == len(nd) + 1 == len(nw) + 1 == len(wd) + 1):
            raise ValueError("vocabulary arrays disagree on the number of nodes")
        self._h = C.c_void_p()
        L.check(self.lib.plm_voc_create(ctx.handle if ctx else None, len(nd), _p(cs, L.i32p), _p(ci, L.i32p), _p(nd, L.u8p),
                                        _p(nw, L.f64p), _p(wd, L.i32p), int(weighting), int(scoring), C.byref(self._h)),
                "plm_voc_create")
        self.weighting, self.scoring = int(weighting), int(scoring)

    @classmethod
    def from_flat(cls, fv, ctx: Optional[Context] = None) -> "Vocabulary":
        """From any object with child_start / child_ids / node_desc / node_weight / node_word / weighting / scoring."""
        return cls(fv.child_start, fv.child_ids, fv.node_desc, fv.node_weight, fv.node_word, fv.weighting, fv.scoring, ctx)

    def size(self) -> int:
        return int(self.lib.plm_voc_words(self._h))

    def empty(self) -> bool:
        return self.size() == 0

    def transform(self, features: np.ndarray) -> BowVector:
        """TemplatedVocabulary::transform(features, BowVector) (TemplatedVocabulary.h:1045-1101)."""
        return self.transform_batch(features, [0, len(features)])[0]

    def transform_batch(self, desc: np.ndarray, set_start: Sequence[int]) -> List[BowVector]:
        """One launch for many descriptor sets (set s = rows set_start[s] .. set_start[s+1]-1)."""
        desc, dp, n_rows, step = L.desc_args(np.asarray(desc, np.uint8).reshape(-1, 32) if not isinstance(desc, np.ndarray) else desc)
        ss = np.ascontiguousarray(set_start, np.int32)
        n_sets = len(ss) - 1
        ids = np.zeros(max(n_rows, 1), np.uint32)
        vals = np.zeros(max(n_rows, 1), np.float64)
        lens = np.zeros(max(n_sets, 1), np.int32)
        L.check(self.lib.plm_bow_transform(self._h, dp, n_rows, step, _p(ss, L.i32p), n_sets, _p(ids, C.c_void_p),
                                           _p(vals, L.f64p), _p(lens, L.i32p)), "plm_bow_transform")
        return [(ids[ss[s]:ss[s] + lens[s]].copy(), vals[ss[s]:ss[s] + lens[s]].copy()) for s in range(n_sets)]

    def score(self, v1: BowVector, v2: BowVector) -> float:
        """TemplatedVocabulary::score -> L1Scoring::score (ScoringObject.cpp:25-69)."""
        return float(score_matrix([v1], [v2], ctx=self.ctx)[0, 0])

    def close(self):
        if self._h:
            self.lib.plm_voc_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def _pack(vectors: Sequence[BowVector]):
    lens = np.array([len(v[0]) for v in vectors], np.int32)
    start = np.concatenate([[0], np.cumsum(lens[:-1], dtype=np.int64)]).astype(np.int64) if len(vectors) else np.zeros(0, np.int64)
    ids = np.concatenate([np.asarray(v[0], np.uint32) for v in vectors]) if len(vectors) else np.zeros(0, np.uint32)
    vals = np.concatenate([np.asarray(v[1], np.float64) for v in vectors]) if len(vectors) else np.zeros(0, np.float64)
    return np.ascontiguousarray(ids), np.ascontiguousarray(vals), start, lens


def score_matrix(queries: Sequence[BowVector], database: Sequence[BowVector], ctx: Optional[Context] = None) -> np.ndarray:
    """scores[q, j] = L1Scoring::score(queries[q], database[j]) in one launch (plm_bow_score)."""
    lib = L.load()
    qi, qv, qs, ql = _pack(queries)
    di, dv, ds, dl = _pack(database)
    out = np.zeros((len(queries), len(database)), np.float64)
    if out.size:
        L.check(lib.plm_bow_score(ctx.handle if ctx else None, _p(qi, C.c_void_p), _p(qv, L.f64p), _p(qs, C.c_void_p),
                                  _p(ql, L.i32p), len(queries), _p(di, C.c_void_p), _p(dv, L.f64p), _p(ds, C.c_void_p),
                                  _p(dl, L.i32p), len(database), _p(out, L.f64p)), "plm_bow_score")
    return out


def vector_stdv(v: Sequence[float]) -> float:
    """stvo-pl/src/auxiliar.cpp:504-513, same operation order (host scalar code; nan for an empty vector as
    in the reference's 0/0)."""
    n = len(v)
    mean = 0.0
    for x in v:
        mean += float(x)
    mean = mean / n if n else float("nan")
    e = 0.0
    for x in v:
        e += (float(x) - mean) * (float(x) - mean)
    return math.sqrt(1.0 / n * e) if n else float("nan")


class KeyFrameBow:
    """The per-keyframe state the three insert functions read: descriptors and, for the combined strategy,
    the image coordinates of the stereo points / line midpoints (mapHandler.cpp:3178-3208)."""

    def __init__(self, kf_idx: int, pdesc_l: Optional[np.ndarray] = None, ldesc_l: Optional[np.ndarray] = None,
                 pt_xy: Optional[np.ndarray] = None, ls_mid_xy: Optional[np.ndarray] = None):
        self.kf_idx = kf_idx
        self.pdesc_l = np.zeros((0, 32), np.uint8) if pdesc_l is None else pdesc_l
        self.ldesc_l = np.zeros((0, 32), np.uint8) if ldesc_l is None else ldesc_l
        self.pt_xy = np.zeros((0, 2)) if pt_xy is None else np.asarray(pt_xy, np.float64)
        self.ls_mid_xy = np.zeros((0, 2)) if ls_mid_xy is None else np.asarray(ls_mid_xy, np.float64)
        self.descDBoW_P: Optional[BowVector] = None
        self.descDBoW_L: Optional[BowVector] = None


class BowConfusion:
    """conf_matrix + the keyframe list of MapHandler, restricted to what insertKFBowVectorP / L / PL touch
    (mapHandler.cpp:3116-3237).  map_keyframes[i] may be None (a culled keyframe is skipped, :3131)."""

    def __init__(self, dbow_voc_p: Optional[Vocabulary] = None, dbow_voc_l: Optional[Vocabulary] = None,
                 ctx: Optional[Context] = None):
        self.dbow_voc_p, self.dbow_voc_l, self.ctx = dbow_voc_p, dbow_voc_l, ctx
        self.map_keyframes: List[Optional[KeyFrameBow]] = []
        self.conf_matrix = np.zeros((0, 0), np.float64)

    def _grow(self, idx: int):
        n = idx + 1
        if self.conf_matrix.shape[0] < n:       # expandGraphs (mapHandler.cpp:874-896) keeps it square
            m = np.zeros((n, n), np.float64)
            k = self.conf_matrix.shape[0]
            m[:k, :k] = self.conf_matrix
            self.conf_matrix = m
        while len(self.map_keyframes) < n:
            self.map_keyframes.append(None)

    def _scores(self, kf: KeyFrameBow, which: str) -> Tuple[np.ndarray, np.ndarray, float]:
        """(indices i < idx with a live keyframe, score(kf, kf_i), score(kf, kf)) for the P or L vocabulary."""
        attr = "descDBoW_" + which
        live = [i for i in range(kf.kf_idx) if self.map_keyframes[i] is not None]
        db = [getattr(self.map_keyframes[i], attr) for i in live] + [getattr(kf, attr)]
        s = score_matrix([getattr(kf, attr)], db, ctx=self.ctx)[0]
        return np.array(live, np.int64), s[:-1], float(s[-1])

    def insertKFBowVectorP(self, kf: KeyFrameBow) -> None:
        """mapHandler.cpp:3116-3139."""
        kf.descDBoW_P = self.dbow_voc_p.transform(kf.pdesc_l)
        self._insert_single(kf, "P")

    def insertKFBowVectorL(self, kf: KeyFrameBow) -> None:
        """mapHandler.cpp:3141-3164."""
        kf.descDBoW_L = self.dbow_voc_l.transform(kf.ldesc_l)
        self._insert_single(kf, "L")

    def _insert_single(self, kf: KeyFrameBow, which: str) -> None:
        idx = kf.kf_idx
        self._grow(idx)
        live, s, s_self = self._scores(kf, which)
        self.conf_matrix[idx, live] = s
        self.conf_matrix[live, idx] = s
        self.conf_matrix[idx, idx] = s_self
        self.map_keyframes[idx] = kf

    def insertKFBowVectorPL(self, kf: KeyFrameBow) -> None:
        """mapHandler.cpp:3166-3237: both vocabularies, scores blended by feature counts (strategy #1) and by
        the spatial dispersion of the features (strategy #2)."""
        kf.descDBoW_P = self.dbow_voc_p.transform(kf.pdesc_l)
        std_pt = vector_stdv(kf.pt_xy[:, 0]) + vector_stdv(kf.pt_xy[:, 1])
        n_pt = len(kf.pt_xy)
        kf.descDBoW_L = self.dbow_voc_l.transform(kf.ldesc_l)
        std_ls = vector_stdv(kf.ls_mid_xy[:, 0]) + vector_stdv(kf.ls_mid_xy[:, 1])
        std_pl = std_ls + std_pt
        n_ls = len(kf.ls_mid_xy)
        n_pl = n_pt + n_ls
        idx = kf.kf_idx
        self._grow(idx)
        live, sp, sp_self = self._scores(kf, "P")
        _, sl, sl_self = self._scores(kf, "L")

        def blend(score_p, score_l):  # numpy evaluates every operation separately: no fused multiply-add
            with np.errstate(divide="ignore", invalid="ignore"):
                score = 0.0 + (score_p * np.float64(n_pt) + score_l * np.float64(n_ls)) / np.float64(n_pl)
                return score + (score_p * np.float64(std_pt) + score_l * np.float64(std_ls)) / np.float64(std_pl)

        s = blend(sp, sl)
        self.conf_matrix[idx, live] = s
        self.conf_matrix[live, idx] = s
        self.conf_matrix[idx, idx] = blend(np.float64(sp_self), np.float64(sl_self))
        self.map_keyframes[idx] = kf


class LoopClosureDB:
    """The BowConfusion bookkeeping and isLoopClosure's matching over keyframes resident on the device (plm_loopdb_*,
    include/plmatch.h).  Each keyframe's left point / line descriptors are uploaded once, by its insert; its BowVector(s)
    are computed into the database's arenas on the device, and every later insert and match reads them there, so the
    per-insert cost does not grow with the number of earlier keyframes (BowConfusion re-packs and re-uploads all of them
    on every insert).  Rows of conf_matrix are bit-identical to BowConfusion's for the same insert / cull sequence.

    ``mode``: 0 / "P", 1 / "L" or 2 / "PL" -- the insert strategy, fixed per database (one MapHandler uses one).  The
    database runs on the vocabularies' context; ``capacity``: keyframes the device arenas are first sized for (0 = a
    small default; they grow as needed).  One host thread at a time per database."""

    MODES = {"P": 0, "L": 1, "PL": 2}

    def __init__(self, dbow_voc_p: Optional[Vocabulary], dbow_voc_l: Optional[Vocabulary], mode, ctx: Optional[Context] = None,
                 capacity: int = 0):
        self.lib = L.load()
        self.mode = self.MODES[mode] if isinstance(mode, str) else int(mode)
        self.dbow_voc_p, self.dbow_voc_l = dbow_voc_p, dbow_voc_l
        first = dbow_voc_l if self.mode == 1 else dbow_voc_p
        if ctx is not None and first is not None and first.ctx is not ctx:
            raise ValueError("the database runs on the context of its vocabularies")
        self.ctx = ctx if ctx is not None else (first.ctx if first is not None else None)
        self._h = C.c_void_p()
        L.check(self.lib.plm_loopdb_create(dbow_voc_p._h if dbow_voc_p is not None else None,
                                           dbow_voc_l._h if dbow_voc_l is not None else None, self.mode, int(capacity),
                                           C.byref(self._h)), "plm_loopdb_create")
        self.map_keyframes: List[Optional[KeyFrameBow]] = []
        self._buf = np.zeros((0, 0), np.float64)   # conf_matrix = _buf[:n, :n]; capacity grows geometrically
        self._n = 0
        self._live = np.zeros(0, bool)
        self._sizes = {}                           # kf_idx -> (point rows, line rows)

    @property
    def conf_matrix(self) -> np.ndarray:
        return self._buf[:self._n, :self._n]

    def _grow(self, idx: int):
        n = idx + 1
        if n > self._buf.shape[0]:                 # expandGraphs (mapHandler.cpp:874-896) keeps it square
            cap = max(n, 2 * self._buf.shape[0], 64)
            m = np.zeros((cap, cap), np.float64)
            m[:self._n, :self._n] = self.conf_matrix
            self._buf = m
            live = np.zeros(cap, bool)
            live[:len(self._live)] = self._live
            self._live = live
        self._n = max(self._n, n)
        while len(self.map_keyframes) < n:
            self.map_keyframes.append(None)

    def _insert(self, kf: KeyFrameBow, blend) -> None:
        idx = int(kf.kf_idx)
        pd, pp, n_p, sp = L.desc_args(kf.pdesc_l)
        ld, lp, n_l, sl = L.desc_args(kf.ldesc_l)
        b = None if blend is None else np.ascontiguousarray(blend, np.float64)
        n0, k0 = self._n, len(self.map_keyframes)
        self._grow(idx)
        row = self._buf[idx]
        st = self.lib.plm_loopdb_insert(self._h, idx, pp, n_p, sp, lp, n_l, sl, None if b is None else _p(b, L.f64p),
                                        _p(row, L.f64p))
        if st != L.PLM_OK:                         # the database is unchanged: so is the matrix
            self._n = n0
            del self.map_keyframes[k0:]
            L.check(st, "plm_loopdb_insert")
        live = np.flatnonzero(self._live[:idx])
        self._buf[live, idx] = row[live]
        self._live[idx] = True
        self.map_keyframes[idx] = kf
        self._sizes[idx] = (n_p, n_l)

    def _need(self, mode: int, name: str):
        if self.mode != mode:
            raise ValueError(f"{name} called on a database created for mode {self.mode}")

    def insertKFBowVectorP(self, kf: KeyFrameBow) -> None:
        """mapHandler.cpp:3116-3139."""
        self._need(0, "insertKFBowVectorP")
        self._insert(kf, None)

    def insertKFBowVectorL(self, kf: KeyFrameBow) -> None:
        """mapHandler.cpp:3141-3164."""
        self._need(1, "insertKFBowVectorL")
        self._insert(kf, None)

    def insertKFBowVectorPL(self, kf: KeyFrameBow) -> None:
        """mapHandler.cpp:3166-3237; the dispersion terms are computed on the host as in BowConfusion."""
        self._need(2, "insertKFBowVectorPL")
        std_pt = vector_stdv(kf.pt_xy[:, 0]) + vector_stdv(kf.pt_xy[:, 1])
        std_ls = vector_stdv(kf.ls_mid_xy[:, 0]) + vector_stdv(kf.ls_mid_xy[:, 1])
        self._insert(kf, [float(len(kf.pt_xy)), std_pt, float(len(kf.ls_mid_xy)), std_ls])

    def cull(self, idx: int) -> None:
        """map_keyframes[idx] = NULL: skipped by every later insert and match."""
        L.check(self.lib.plm_loopdb_cull(self._h, int(idx)), "plm_loopdb_cull")
        self.map_keyframes[idx] = None
        self._live[idx] = False

    def bow_vector(self, idx: int, which: str = "P") -> BowVector:
        """descDBoW_P (which = "P") or descDBoW_L ("L") of keyframe idx, read back from the device."""
        w = {"P": 0, "L": 1}[which] if isinstance(which, str) else int(which)
        n = self._sizes.get(int(idx), (0, 0))[w]
        ids, vals, k = np.zeros(max(n, 1), np.uint32), np.zeros(max(n, 1), np.float64), C.c_int32(0)
        L.check(self.lib.plm_loopdb_bow(self._h, int(idx), w, _p(ids, C.c_void_p), _p(vals, L.f64p), C.byref(k)),
                "plm_loopdb_bow")
        return ids[:k.value].copy(), vals[:k.value].copy()

    def match_candidates(self, kf0, kf1_list) -> List[dict]:
        """isLoopClosure's matching + inlier-ratio gate (mapHandler.cpp:3325-3400) of kf0 against every keyframe of
        kf1_list (keyframes or indices), from the resident descriptors; the dicts of drivers.loopClosureMatch."""
        i0 = int(getattr(kf0, "kf_idx", kf0))
        ks = np.ascontiguousarray([int(getattr(k, "kf_idx", k)) for k in kf1_list], np.int32)
        n = len(ks)
        p0, l0 = self._sizes.get(i0, (0, 0))
        cp, cl = np.zeros(max(n, 1), np.int32), np.zeros(max(n, 1), np.int32)
        mp, ml = np.zeros((max(n, 1), p0), np.int32), np.zeros((max(n, 1), l0), np.int32)
        L.check(self.lib.plm_loopdb_match(self._h, i0, _p(ks, L.i32p), n, C.c_float(Config.minRatio12P),
                                          C.c_float(Config.minRatio12L), int(bool(Config.bestLRMatches)), _p(cp, L.i32p),
                                          _p(cl, L.i32p), _p(mp, L.i32p), _p(ml, L.i32p)), "plm_loopdb_match")
        out = []
        for k in range(n):
            p1, l1 = self._sizes[int(ks[k])]
            with_pt, with_ls = bool(p0 and p1), bool(l0 and l1)    # an empty side is not matched (:3333, :3350)
            common_pt, m_pt = (int(cp[k]), mp[k].copy()) if with_pt else (0, np.zeros(0, np.int32))
            common_ls, m_ls = (int(cl[k]), ml[k].copy()) if with_ls else (0, np.zeros(0, np.int32))
            with np.errstate(divide="ignore", invalid="ignore"):
                r_pt = max(np.float64(100.0 * common_pt) / p0, np.float64(100.0 * common_pt) / p1) if with_pt else 0.0
                r_ls = max(np.float64(100.0 * common_ls) / l0, np.float64(100.0 * common_ls) / l1) if with_ls else 0.0
            ok = bool(r_pt > SlamConfig.lcInlierRatio and r_ls > SlamConfig.lcInlierRatio)
            out.append(dict(common_pt=common_pt, common_ls=common_ls, matches_pt=m_pt, matches_ls=m_ls,
                            inl_ratio_pt=float(r_pt), inl_ratio_ls=float(r_ls), inl_ratio_condition=ok))
        return out

    def isLoopClosure(self, kf0, kf1) -> dict:
        """MapHandler::isLoopClosure's matching and gate for one candidate: drivers.loopClosureMatch's dict."""
        return self.match_candidates(kf0, [kf1])[0]

    @property
    def h2d_bytes(self) -> int:
        return int(self.lib.plm_loopdb_h2d_bytes(self._h))

    @property
    def d2h_bytes(self) -> int:
        return int(self.lib.plm_loopdb_d2h_bytes(self._h))

    def __len__(self) -> int:
        return int(self.lib.plm_loopdb_size(self._h))

    def close(self):
        if self._h:
            self.lib.plm_loopdb_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
