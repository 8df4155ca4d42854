"""The resident local map (LocalMap.matchMap2KF*, localmap.match_keyframe) against a CPU chain built only from
oracle.port: selection, grid fill, matchGrid, the brute-force fallback and the reprojection gate of
MapHandler::matchMap2KFPoints / Lines (src/mapHandler.cpp:583-803), fp64 in the oracle's rounding order.

The other local-map tests compare the store with drivers.matchMap2KF*Full, which runs the same device kernels; a
kernel bug shows on both sides there.  Here the expected side never touches the GPU, and the config values the call
reads are varied per kind: ratios, lineSimTh, the window, the gates and the fallback thresholds.

CPU: the chain reproduces the oracle composition of test_gpu_reproj's end-to-end case, and every boundary
construction below lands on the side of its boundary it is built for.
GPU (-m gpu): both entry points equal the chain bit for bit on those constructions, on a keyframe sequence with the
config drawn per kind, at every grid size up to the 8192-cell limit, at the keyframe size limits and at map scale;
calls past the limits are refused before anything is sent."""
import itertools
from dataclasses import dataclass, field, replace
from typing import Callable, List, Optional, Tuple

import numpy as np
import pytest

import oracle
from test_gpu_localmap import Mirror, build_map, config, ctx, keyframe, new_landmarks, unit  # noqa: F401
from test_gpu_localmap_kf import kf_pair, update
from test_reproj import CAM, H, INV_H, INV_W, W, make_scene

port = oracle.port
SEED = 20261024
KF_MAX_FEATS = 32768            # KF_GRID_MAX_FEATS = GRID_N2_MAX: one bitmap bit per keyframe feature
KF_MAX_CELLS = 8192             # KF_GRID_MAX_CELLS


# ------------------------------------------------------------------------------------------------------ the chain
@dataclass(frozen=True)
class Cfg:
    """The config values one map-to-keyframe call reads (matching.Config / drivers.SlamConfig)."""
    ratio_p: float = 0.9        # minRatio12P
    ratio_l: float = 0.9        # minRatio12L
    line_sim_th: float = 0.75   # lineSimTh
    ws: int = 3                 # matchingF2FWs
    epip_p: float = 1.0         # maxKFEpipP
    epip_l: float = 1.0         # maxKFEpipL
    min_p: int = 10             # minPointMatches
    min_l: int = 6              # minLineMatches
    best_lr: bool = True        # bestLRMatches
    fast: bool = True           # fastMatching


@dataclass(frozen=True)
class View:
    """Camera, image and keyframe grid of one call; inv_w / inv_h = cols / width, rows / height."""
    cam: Tuple[float, float, float, float] = CAM
    width: int = W
    height: int = H
    rows: int = 48
    cols: int = 64

    @property
    def inv_w(self):
        return self.cols / self.width

    @property
    def inv_h(self):
        return self.rows / self.height


def _fallback(d1, d2, nnr, best_lr, m12):
    """StVO::match(d1, d2, nnr) on the grid's vector: stale entries are kept (matching.cpp:63-91).  With one keyframe
    feature the reference reads past knnMatch's row (matching.cpp:54, undefined); the library's rule (DESIGN.md 5) is
    that a row without a second neighbour is not accepted, while the mutual check still culls stale entries."""
    if len(d2) >= 2:
        return port.match(d1, d2, nnr, best_lr, m12=m12)
    m12 = m12.copy()
    n = 0
    if best_lr:
        _, m21 = port.match_nnr(d2, d1, nnr)
        for i1, i2 in enumerate(m12):
            if i2 >= 0 and m21[i2] != i1:
                m12[i1] = -1
                n -= 1
    return n, m12


def chain(lines, X, active, med, T, view, kf, cfg):
    """oracle_map2kf with its intermediate stages: dict(sel, coords, pf, grid, m12_grid, fallback, m12, ok, matches)."""
    geo, d2, feat = kf
    sel, coords, pf = port.map_select(X, active, T, view.cam, view.inv_w, view.inv_h, view.width, view.height)
    ns, n2 = len(sel), len(d2)
    st = dict(sel=sel, coords=coords, pf=pf, grid=None, m12_grid=None, fallback=False)
    if ns == 0 or n2 == 0:       # mapHandler.cpp:611 / :716: nothing to match
        st.update(m12=np.full(ns, -1, np.int32), ok=np.zeros(ns, np.uint8), matches=0)
        return st
    d1 = np.ascontiguousarray(med[sel])
    d2 = np.ascontiguousarray(d2)
    nnr, min_m, max_epip = (cfg.ratio_l, cfg.min_l, cfg.epip_l) if lines else (cfg.ratio_p, cfg.min_p, cfg.epip_p)
    matches, m12 = 0, np.full(ns, -1, np.int32)
    if cfg.fast:
        win = np.full(4, cfg.ws, np.int32)
        if lines:
            cs, ci, dirs = port.csr_from_lines(geo, view.inv_w, view.inv_h, view.rows, view.cols)
            matches, m12 = port.match_grid_lines(coords, d1, cs, ci, view.rows, view.cols, d2, dirs, cfg.line_sim_th,
                                                 win, cfg.ratio_p, cfg.best_lr)
        else:
            cs, ci = port.csr_from_points(geo, view.inv_w, view.inv_h, view.rows, view.cols)
            matches, m12 = port.match_grid_points(coords, d1, cs, ci, view.rows, view.cols, d2, win, cfg.ratio_p,
                                                  cfg.best_lr)
        st.update(grid=matches, m12_grid=m12.copy())
    n1_feats = n2_feats = ns                                # _grid_then_fallback's two counts, both n_sel here
    if n2_feats > min_m and n1_feats > min_m and matches < min_m:
        matches, m12 = _fallback(d1, d2, np.float32(nnr), cfg.best_lr, m12)
        st["fallback"] = True
    count, ok = port.map_gate(pf, m12, feat, max_epip, matches)
    st.update(m12=m12, ok=ok, matches=count)
    return st


def oracle_map2kf(lines, X, active, med, T, view, kf, cfg):
    """matchMap2KFPoints (lines = False) / matchMap2KFLines (lines = True) of one keyframe from oracle.port alone ->
    (sel, m12, ok, matches).

    X / active / med: the map (n x 3 points or n x 6 segment endpoints, the selection byte, med_desc);
    T: Twf (3 x 4); view: View; kf = (geo, desc, feat): points (n2 x 2 float32 pixels, n2 x 32, pl n2 x 2 doubles),
    segments (n2 x 4 float32 pixels, n2 x 32, le n2 x 3 doubles).

    1. port.map_select with T, the camera, inv_w, inv_h, width and height -> sel, cell coords, pf.
    2. port.csr_from_points / csr_from_lines over the raw float32 features at the view's rows x cols (+ directions).
    3. fastMatching: port.match_grid_points / lines, window (ws, ws, ws, ws) with ws = matchingF2FWs, ratio =
       minRatio12P for BOTH kinds (matchGrid reads minRatio12P, matching.py:304 / :312), lineSimTh, bestLRMatches.
    4. the fallback when n_sel > min_matches and the grid count < min_matches (0 without fastMatching), min_matches
       = minPointMatches / minLineMatches: port.match(d1, d2, float32(nnr), bestLRMatches) on the grid's vector,
       nnr = minRatio12P for points and minRatio12L for lines (localmap._params).
    5. port.map_gate(pf, m12, pl or le, maxKFEpipP / maxKFEpipL, count)."""
    st = chain(lines, X, active, med, T, view, kf, cfg)
    return st["sel"], st["m12"], st["ok"], st["matches"]


# ------------------------------------------------------------------------------------------------ constructions
# An exact view: Twf = [I | (0, 0, -0)], fx = fy = 512, (cx, cy) = (384, 256).  A landmark X = ((u - 384) / 512,
# (v - 256) / 512, 1) projects to (u, v) with every operation exact for the dyadic pixels used below.
T0 = np.array([[1.0, 0, 0, 0], [0, 1.0, 0, 0], [0, 0, 1.0, -0.0]])
V0 = View(cam=(512.0, 512.0, 384.0, 256.0))
CELL_W, CELL_H = W / 64.0, H / 48.0          # 11.75 px, 10 px


def x_of(uv, z=1.0):
    uv = np.asarray(uv, np.float64).reshape(-1, 2)
    return np.stack([(uv[:, 0] - 384.0) / 512.0 * z, (uv[:, 1] - 256.0) / 512.0 * z, np.full(len(uv), z)], 1)


def le_of(seg):
    s = np.asarray(seg, np.float32).astype(np.float64).reshape(-1, 4)
    a = np.stack([s[:, 0], s[:, 1], np.ones(len(s))], 1)
    b = np.stack([s[:, 2], s[:, 3], np.ones(len(s))], 1)
    le = np.cross(a, b)
    return le / np.hypot(le[:, 0], le[:, 1])[:, None]


@dataclass
class Case:
    """One call: per kind (X, med, kf) or None; sides = (label, predicate over the chain stages of both kinds)."""
    name: str
    cfg: Cfg
    pts: Optional[tuple]
    lns: Optional[tuple]
    sides: List[Tuple[str, Callable]]
    T: np.ndarray = field(default_factory=lambda: T0)
    view: View = V0


def run_chain(case):
    out = {}
    for kind, lines, part in (("points", False, case.pts), ("lines", True, case.lns)):
        if part is not None:
            X, med, kf = part
            out[kind] = chain(lines, X, np.ones(len(X), np.uint8), med, case.T, case.view, kf, case.cfg)
    return out


def planted(rng, lines, n_lm, near, far, fill, twins=0, twin_off=0.0):
    """n_lm landmarks in the left half of the exact view, all selected.  Landmark i < near has a keyframe feature with
    its descriptor where it projects (a grid match); near <= i < near + far has one 400 px to the right, outside every
    window (only the brute-force fallback finds it); the first `twins` near landmarks get a second such far copy, so the
    fallback's ratio test rejects them and their grid entries stay in m12 (stale; the first twin's near feature is
    twin_off px off, in x for a point and in y for a segment, so that the gate rejects it).  `fill` features of random descriptors follow."""
    # on a lattice of cells far enough apart that no window (ws = 1) reaches another landmark's feature: a window
    # with a single candidate is accepted whatever its distance (best_d2 stays INT_MAX)
    lat = np.array([(c, r) for c in range(0, 24, 6 if lines else 3) for r in range(0, 46, 3)])
    pick = lat[rng.choice(len(lat), n_lm, replace=False)]
    u, v = (pick[:, 0] + 0.5) * CELL_W, (pick[:, 1] + 0.5) * CELL_H
    med = rng.integers(0, 256, (n_lm, 32), dtype=np.uint8)
    if not lines:
        X = x_of(np.stack([u, v], 1))
        geo = [np.stack([u[:near], v[:near]], 1), np.stack([u[near:near + far] + 400, v[near:near + far]], 1),
               np.stack([u[:twins] + 400, v[:twins] + 5], 1), rng.uniform([400, 5], [740, 470], (fill, 2))]
        if twins and twin_off:
            geo[0][0, 0] += twin_off
    else:
        s, e = np.stack([u, v], 1), np.stack([u + 40, v + 3], 1)
        X = np.concatenate([x_of(s), x_of(e)], 1)
        seg = np.concatenate([s, e], 1)
        sh = np.array([400.0, 0, 400.0, 0])
        tw = seg[:twins] + sh + [0, 5, 0, 5]
        geo = [seg[:near], seg[near:near + far] + sh, tw,
               np.concatenate([rng.uniform([400, 5], [700, 470], (fill, 2)), rng.uniform([-30, -30], [30, 30], (fill, 2))], 1)]
        geo[3][:, 2:] += geo[3][:, :2]
        if twins and twin_off:
            geo[0][0, [1, 3]] += twin_off
    geo = np.concatenate(geo).astype(np.float32)
    d2 = np.concatenate([med[:near], med[near:near + far], med[:twins], rng.integers(0, 256, (fill, 32), dtype=np.uint8)])
    feat = le_of(geo) if lines else geo.astype(np.float64)
    return X, med, (geo, d2, feat)


def cases_fallback(rng):
    """The fallback thresholds, per kind (min_p = 10, min_l = 6): the grid count at min - 1 and at min, n_sel at min
    and min + 1, min = 0, keyframes of 1 .. min features, and stale grid entries that reach the gate."""
    base = Cfg(ratio_p=0.75, ratio_l=0.9, epip_p=1.0, epip_l=3.0, min_p=10, min_l=6, ws=1)
    out = []

    def both(name, cfg, kp, kl, sides):
        out.append(Case(name, cfg, planted(rng, False, *kp), planted(rng, True, *kl), sides=sides))

    def side(kind, f):
        return lambda r: f(r[kind])

    for best_lr in (True, False):
        cfg = replace(base, best_lr=best_lr)
        both(f"grid=min-1 lr={best_lr}", cfg, (40, 9, 6, 20), (30, 5, 4, 10),
             [(k, side(k, lambda s, m=m: s["grid"] == m - 1 and s["fallback"])) for k, m in (("points", 10), ("lines", 6))])
        both(f"grid=min lr={best_lr}", cfg, (40, 10, 6, 20), (30, 6, 4, 10),
             [(k, side(k, lambda s, m=m: s["grid"] == m and not s["fallback"])) for k, m in (("points", 10), ("lines", 6))])
    both("n_sel=min", base, (10, 3, 5, 20), (6, 2, 3, 10),
         [(k, side(k, lambda s, m=m: len(s["sel"]) == m and s["grid"] < m and not s["fallback"]))
          for k, m in (("points", 10), ("lines", 6))])
    both("n_sel=min+1", base, (11, 3, 6, 20), (7, 2, 4, 10),
         [(k, side(k, lambda s, m=m: len(s["sel"]) == m + 1 and s["grid"] < m and s["fallback"]))
          for k, m in (("points", 10), ("lines", 6))])
    both("min=0", replace(base, min_p=0, min_l=0), (30, 0, 8, 20), (20, 0, 5, 10),
         [(k, side(k, lambda s: s["grid"] <= 0 and not s["fallback"])) for k in ("points", "lines")])
    both("fast off", replace(base, fast=False), (30, 4, 8, 20), (20, 3, 5, 10),
         [(k, side(k, lambda s: s["grid"] is None and s["fallback"])) for k in ("points", "lines")])
    for k in range(1, 11):                                   # keyframes of 1 .. min features, all far copies
        kl = min(k, 6)
        both(f"n2={k}", base, (20, 0, k, 0), (12, 0, kl, 0),
             [(f"{kind} n2={n2}", side(kind, lambda s, n2=n2: s["fallback"] and len(s["ok"]) > 0))
              for kind, n2 in (("points", k), ("lines", kl))])

    def stale(s):
        rows = (s["m12_grid"] >= 0) & (s["m12"] == s["m12_grid"]) & (s["fresh"] < 0)
        return s["fallback"] and rows.any() and (rows & (s["ok"] == 0)).any()

    for best_lr in (True, False):
        both(f"stale lr={best_lr}", replace(base, best_lr=best_lr), (40, 4, 5, 20, 3, 2.5), (30, 3, 4, 10, 2, -4.5),
             [(k, side(k, stale)) for k in ("points", "lines")])
    return out


def cases_selection(rng):
    """Landmarks whose pf is exactly 0, W or H or one ulp inside, at P.z = +0, -0, subnormal and negative, on cell
    borders (u * inv_w an integer), and segments with one endpoint outside.  Planted keyframe features match the
    selected ones."""
    nx = np.nextafter
    pts = [((-0.75, 0.0, 1.0), False), ((nx(-0.75, 0.0), 0.0, 1.0), True),              # u = 0 / one ulp inside
           ((0.71875, 0.0, 1.0), False), (tuple(x_of([nx(752.0, 0.0), 256.0])[0]), True),  # u = W
           ((0.0, -0.5, 1.0), False), ((0.0, nx(-0.5, 0.0), 1.0), True),                # v = 0
           ((0.0, 0.4375, 1.0), False), (tuple(x_of([384.0, nx(480.0, 0.0)])[0]), True),  # v = H
           ((0.0, 0.0, 0.0), False), ((-1e-3, -1e-3, -0.0), False), ((-0.0, -0.0, -0.0), False),
           ((0.0, 0.0, 5e-324), True), ((0.0, 0.0, -1.0), False), ((0.1, 0.1, -2.0), False)]
    X = [p for p, _ in pts]
    want = [w for _, w in pts]
    ub = CELL_W * np.arange(1, 64)                          # cell borders in u, v
    vb = CELL_H * np.arange(1, 48)
    X += [tuple(r) for r in x_of(np.stack([ub, np.full_like(ub, 77.0)], 1))]
    X += [tuple(r) for r in x_of(np.stack([np.full_like(vb, 333.0), vb], 1))]
    want += [True] * (len(ub) + len(vb))
    Xp = np.asarray(X, np.float64)
    medp = rng.integers(0, 256, (len(Xp), 32), dtype=np.uint8)
    # segments: both endpoints inside, one endpoint outside (each side), an endpoint exactly on u = 0 / one ulp inside
    s_in = np.array([[100.0, 100.0, 160.0, 104.0], [500.0, 300.0, 560.0, 310.0]])
    segs = [(s_in[0], True), (s_in[1], True), ([-10.0, 200.0, 50.0, 204.0], False), ([700.0, 50.0, 760.0, 52.0], False),
            ([300.0, 470.0, 320.0, 490.0], False), ([300.0, -5.0, 330.0, 20.0], False)]
    Xl = [np.concatenate([x_of(s[:2])[0], x_of(s[2:])[0]]) for s, _ in segs]
    wl = [w for _, w in segs]
    Xl.append(np.concatenate([[-0.75, 0.0, 1.0], x_of([60.0, 260.0])[0]]))
    Xl.append(np.concatenate([[nx(-0.75, 0.0), 0.0, 1.0], x_of([60.0, 262.0])[0]]))
    wl += [False, True]
    Xl = np.asarray(Xl)
    medl = rng.integers(0, 256, (len(Xl), 32), dtype=np.uint8)
    # keyframe: a copy of every selected landmark's descriptor where it projects, plus filler
    cfg = Cfg(ratio_p=0.9, ratio_l=0.75, min_p=0, min_l=0)
    sp, _, pp = port.map_select(Xp, None, T0, V0.cam, V0.inv_w, V0.inv_h, W, H)
    sl, _, pl = port.map_select(Xl, None, T0, V0.cam, V0.inv_w, V0.inv_h, W, H)
    kp = np.concatenate([pp, rng.uniform([5, 5], [745, 475], (40, 2))]).astype(np.float32)
    dp = np.concatenate([medp[sp], rng.integers(0, 256, (40, 32), dtype=np.uint8)])
    seg = pl.astype(np.float32)
    dl = medl[sl]
    wp, wl = np.asarray(want), np.asarray(wl)

    def picks(s, w):
        got = np.isin(np.arange(len(w)), s["sel"])
        return np.array_equal(got, w) and got.any() and not got.all()

    def border(s):
        u = s["pf"][:, 0]
        on = u * V0.inv_w == np.trunc(u * V0.inv_w)
        k = np.flatnonzero(on & (u > 0))
        return len(k) > 0 and np.array_equal(s["coords"][k, 0], (u[k] * V0.inv_w).astype(np.int32))

    sides = [("points selected as built", lambda r: picks(r["points"], wp)),
             ("segments selected as built", lambda r: picks(r["lines"], wl)),
             ("a landmark on a cell border", lambda r: border(r["points"]))]
    return [Case("selection", cfg, (Xp, medp, (kp, dp, kp.astype(np.float64))), (Xl, medl, (seg, dl, le_of(seg))),
                 sides=sides)]


def cases_gate(rng):
    """Points: distance exactly max_epip (rejected: the test is a strict <) and one ulp below (accepted), pl far from
    kp (the gate reads pl, the grid kp).  Segments: e0 / e1 exactly max_epip, one ulp below, and large negative
    errors (accepted: the test is signed)."""
    out = []
    for ep, el in ((1.0, 3.0), (3.0, 1.0)):
        below = np.nextafter(ep, 0.0)
        pf = np.array([[200.0, 100.0], [ep + 0.5, 150.0], [300.0, 300.0], [500.0, 60.0]])
        kp = pf.copy()
        kp[3] = [650.0, 400.0]                                    # kp far away: no grid match although pl = pf
        pl = pf.copy()
        pl[0, 0] -= ep                                             # distance exactly ep
        pl[1, 0] = pf[1, 0] - below                                # one ulp below
        pl[2, 0] += 5.0                                            # kp on the landmark, pl 5 px off
        medp = rng.integers(0, 256, (4, 32), dtype=np.uint8)
        fill = rng.uniform([5, 5], [745, 475], (30, 2))
        kpf = np.concatenate([kp, fill]).astype(np.float32)
        plf = np.concatenate([pl, fill.astype(np.float32).astype(np.float64)])
        dp = np.concatenate([medp, rng.integers(0, 256, (30, 32), dtype=np.uint8)])
        # segments from y = 0.75 to y = 0.25 (so e0 >= e1 for le = (0, 1, c)); e0 = 0.75 + c, e1 = 0.25 + c
        bl = np.nextafter(el, 0.0)
        segs = np.array([[100.0, 0.75, 220.0, 0.25], [300.0, 0.75, 420.0, 0.25], [500.0, 0.75, 620.0, 0.25],
                         [100.0, 200.0, 220.0, 204.0], [300.0, 0.25, 420.0, 0.75]])
        le = np.array([[0.0, 1.0, el - 0.75], [0.0, 1.0, bl - 0.75], [0.0, 1.0, -1e6], [0.0, 1.0, -5e5],
                       [0.0, 1.0, el - 0.75]])                     # the last: e1 = el exactly, e0 below
        Xl = np.concatenate([x_of(segs[:, :2]), x_of(segs[:, 2:])], 1)
        medl = rng.integers(0, 256, (len(segs), 32), dtype=np.uint8)
        cfg = Cfg(epip_p=ep, epip_l=el, min_p=0, min_l=0, ws=1)

        def pts_side(s, ep=ep, below=below, pf=pf, pl=pl):
            d = np.hypot(*(pf - pl)[:2].T)
            return (d[0] == ep and d[1] == below and np.array_equal(s["pf"], pf)
                    and np.array_equal(s["m12"][:4], [0, 1, 2, -1]) and np.array_equal(s["ok"][:4], [0, 1, 0, 0]))

        def ln_side(s, el=el, bl=bl, le=le):
            p = s["pf"]
            e0 = le[:, 0] * p[:, 0] + le[:, 1] * p[:, 1] + le[:, 2]
            e1 = le[:, 0] * p[:, 2] + le[:, 1] * p[:, 3] + le[:, 2]
            return (e0[0] == el and e0[1] == bl and e1[4] == el and e0[2] < -1e5 and
                    np.array_equal(s["m12"], np.arange(5)) and np.array_equal(s["ok"], [0, 1, 1, 1, 0]))

        out.append(Case(f"gate ep={ep}", cfg, (x_of(pf), medp, (kpf, dp, plf)),
                        (Xl, medl, (segs.astype(np.float32), medl, le)),
                        sides=[("points", lambda r, f=pts_side: f(r["points"])), ("lines", lambda r, f=ln_side: f(r["lines"]))]))
    return out


def cases_window(rng):
    """Keyframe keypoints and vertical segments exactly on cell borders (in u and in v) and one float32 ulp below,
    each with a unique descriptor shared by a landmark in the middle of the cell exactly ws cells away ("in") and one
    ws + 1 cells away ("out")."""
    out = []
    for ws in (1, 3):
        cfg = Cfg(ws=ws, min_p=0, min_l=0, ratio_p=0.9, best_lr=True)
        kp, lmk, pairs = [], [], []                     # pairs: (kp index, in row, out row)
        j = 0
        for axis, n_b, cell in ((0, 64, CELL_W), (1, 48, CELL_H)):
            for k in range(1, n_b):
                for below in (False, True):
                    b = np.float32(k * cell)
                    c = np.nextafter(b, np.float32(0)) if below else b
                    inv = V0.inv_w if axis == 0 else V0.inv_h
                    own = int(np.trunc(np.float64(c) * inv))
                    sgn = 1 if (k + below) % 2 == 0 else -1
                    if not (0 <= own + sgn * (ws + 1) < n_b):
                        sgn = -sgn
                    if not (0 <= own + sgn * (ws + 1) < n_b):
                        continue
                    other = (j * 7) % (48 if axis == 0 else 64)
                    o_mid = (other + 0.5) * (CELL_H if axis == 0 else CELL_W)
                    pt = [c, o_mid] if axis == 0 else [o_mid, c]
                    mids = [(own + sgn * d + 0.5) * cell for d in (ws, ws + 1)]
                    kp.append(pt)
                    for m in mids:
                        lmk.append([m, o_mid] if axis == 0 else [o_mid, m])
                    pairs.append((len(kp) - 1, len(lmk) - 2, len(lmk) - 1))
                    j += 1
        kp = np.asarray(kp, np.float32)
        d = rng.integers(0, 256, (len(kp), 32), dtype=np.uint8)
        medp = np.repeat(d, 2, axis=0)
        pairs = np.asarray(pairs)
        # segments: vertical, 25 px, at u exactly on a column border or one ulp below; landmarks vertical in the middle
        # of the column ws / ws + 1 away
        seg, lseg, lpairs = [], [], []
        for k in range(1, 64):
            for below in (False, True):
                b = np.float32(k * CELL_W)
                c = np.nextafter(b, np.float32(0)) if below else b
                own = int(np.trunc(np.float64(c) * V0.inv_w))
                sgn = 1 if (k + below) % 2 == 0 else -1
                if not (0 <= own + sgn * (ws + 1) < 64):
                    sgn = -sgn
                if not (0 <= own + sgn * (ws + 1) < 64):
                    continue
                y0 = ((len(seg) * 5) % 44 + 0.5) * CELL_H
                seg.append([c, y0, c, y0 + 25])
                for dd in (ws, ws + 1):
                    m = (own + sgn * dd + 0.5) * CELL_W
                    lseg.append([m, y0, m, y0 + 25])
                lpairs.append((len(seg) - 1, len(lseg) - 2, len(lseg) - 1))
        # horizontal, 25 px, at v exactly on a row border or one ulp below; landmarks horizontal in the middle of the
        # row ws / ws + 1 away
        n_vert = len(seg)
        for k in range(1, 48):
            for below in (False, True):
                b = np.float32(k * CELL_H)
                c = np.nextafter(b, np.float32(0)) if below else b
                own = int(np.trunc(np.float64(c) * V0.inv_h))
                sgn = 1 if (k + below) % 2 == 0 else -1
                if not (0 <= own + sgn * (ws + 1) < 48):
                    sgn = -sgn
                if not (0 <= own + sgn * (ws + 1) < 48):
                    continue
                x0 = (((len(seg) - n_vert) * 7) % 58 + 0.5) * CELL_W
                seg.append([x0, c, x0 + 25, c])
                for dd in (ws, ws + 1):
                    m = (own + sgn * dd + 0.5) * CELL_H
                    lseg.append([x0, m, x0 + 25, m])
                lpairs.append((len(seg) - 1, len(lseg) - 2, len(lseg) - 1))
        seg = np.asarray(seg, np.float32)
        lseg = np.asarray(lseg)
        dl = rng.integers(0, 256, (len(seg), 32), dtype=np.uint8)
        Xl = np.concatenate([x_of(lseg[:, :2]), x_of(lseg[:, 2:])], 1)
        lpairs = np.asarray(lpairs)

        def in_out(s, pr, n):
            return (len(s["sel"]) == n and np.array_equal(s["m12"][pr[:, 1]], pr[:, 0])
                    and not (s["m12"][pr[:, 2]] == pr[:, 0]).any())

        def borders(geo, inv):
            v = geo.astype(np.float64) * inv
            return (v == np.round(v)).any() and (np.trunc(v) != np.round(v)).any()

        sides = [("points in / out", lambda r, p=pairs, n=len(medp): in_out(r["points"], p, n)),
                 ("segments in / out", lambda r, p=lpairs, n=len(Xl): in_out(r["lines"], p, n)),
                 ("keypoints on borders and one ulp below", lambda r, g=kp: borders(g[:, 0], V0.inv_w)
                  and borders(g[:, 1], V0.inv_h)),
                 ("segment endpoints on column and row borders and one ulp below",
                  lambda r, g=seg, nv=n_vert: borders(g[:nv, 0], V0.inv_w) and borders(g[nv:, 1], V0.inv_h))]
        out.append(Case(f"window ws={ws}", cfg, (x_of(np.asarray(lmk)), medp, (kp, d, kp.astype(np.float64))),
                        (Xl, np.repeat(dl, 2, axis=0), (seg, dl, le_of(seg))), sides=sides))
    return out


def big_keyframe(rng, related_px, related_d):
    """KF_MAX_FEATS keypoints: the related ones first, random ones, then clusters of 40 .. 300 keypoints in single
    cells; the last 40 indices (the last bitmap word and the one before) go into one cluster."""
    n = KF_MAX_FEATS
    kp = rng.uniform([1, 1], [W - 1, H - 1], (n, 2))
    kp[:len(related_px)] = related_px
    d = rng.integers(0, 256, (n, 32), dtype=np.uint8)
    d[:len(related_d)] = related_d
    centers = rng.uniform([20, 20], [W - 20, H - 20], (12, 2))
    start = len(related_px) + 1000
    for i, c in enumerate(centers):
        m = 40 + 24 * i
        kp[start:start + m] = c + rng.uniform(-1, 1, (m, 2))
        start += m
    kp[n - 40:] = centers[0] + rng.uniform(-1, 1, (40, 2))
    return kp.astype(np.float32), d


def big_keyframe_ok(kp):
    cs, ci = port.csr_from_points(kp, INV_W, INV_H)
    sizes = np.diff(cs)
    big = np.flatnonzero(sizes > 32)
    last = [c for c in big if (ci[cs[c]:cs[c + 1]] >= KF_MAX_FEATS - 32).any()]
    return len(kp) == KF_MAX_FEATS and len(big) >= 4 and len(last) >= 1


def crossing_segments(rng, n):
    """n segments from u = -20 to u = W + 20 at random heights: each walks every column (items = n * max(rows, cols))."""
    y = rng.uniform(20, H - 20, (n, 2))            # two rows from the border: the walk never leaves the grid in y
    return np.stack([np.full(n, -20.0), y[:, 0], np.full(n, W + 20.0), y[:, 1]], 1).astype(np.float32)


CONSTRUCTIONS = {"fallback": cases_fallback, "selection": cases_selection, "gate": cases_gate, "window": cases_window}


def run_chain_sides(case):
    """The chain's stages per kind, plus "fresh": the fallback's own acceptances from an all -1 vector."""
    r = run_chain(case)
    for kind, s in r.items():
        _, med, kf = case.pts if kind == "points" else case.lns
        nnr = case.cfg.ratio_l if kind == "lines" else case.cfg.ratio_p
        s["fresh"] = _fallback(np.ascontiguousarray(med[s["sel"]]), np.ascontiguousarray(kf[1]), np.float32(nnr),
                               case.cfg.best_lr, np.full(len(s["sel"]), -1, np.int32))[1] if len(s["sel"]) and len(kf[1]) else None
    return r


# ---------------------------------------------------------------------------------------------------------------- CPU
def test_chain_reproduces_the_end_to_end_composition():
    """test_gpu_reproj::test_match_map2kf_points_end_to_end's case (keypoints as the float32 pixels a keyframe holds):
    the chain equals that test's composition of port.map_select, the grid, match_grid_points and map_gate."""
    from pl_inertial_slam_b200 import synth
    rng = np.random.default_rng(7)
    n, n2 = 40_000, 500
    T, X, active = make_scene(5, n)
    med = synth.rand_desc(rng, n)
    s_o, c_o, p_o = port.map_select(X, active, T, CAM, INV_W, INV_H, W, H)
    seen = rng.choice(len(s_o), n2, replace=False)
    pl = p_o[seen] + rng.normal(0, 0.8, (n2, 2))
    pl = np.clip(pl, 1.0, [W - 2.0, H - 2.0]).astype(np.float32).astype(np.float64)
    d2 = synth.flip_bits(rng, med[s_o[seen]], 0.06)
    d2[::9] = synth.rand_desc(rng, len(d2[::9]))
    cs, ci = port.csr_from_points(pl.astype(np.float32), INV_W, INV_H)
    n_o, m_o = port.match_grid_points(c_o, np.ascontiguousarray(med[s_o]), cs, ci, 48, 64, d2,
                                      np.array([3, 3, 3, 3], np.int32), 0.9, True)
    assert n_o >= 10
    cnt_o, ok_o = port.map_gate(p_o, m_o, pl, 1.0, n_o)
    sel, m12, ok, cnt = oracle_map2kf(False, X, active, med, T, View(), (pl.astype(np.float32), d2, pl), Cfg())
    assert np.array_equal(sel, s_o) and np.array_equal(m12, m_o) and np.array_equal(ok, ok_o) and cnt == cnt_o
    assert 50 < cnt <= n_o


@pytest.mark.parametrize("name", sorted(CONSTRUCTIONS))
def test_constructions_land_on_their_side(name):
    """Every boundary construction checked through the chain: a construction that degenerates fails here."""
    cases = CONSTRUCTIONS[name](np.random.default_rng(SEED))
    assert cases
    for case in cases:
        r = run_chain_sides(case)
        for label, pred in case.sides:
            assert pred(r), (case.name, label)


def test_size_constructions():
    rng = np.random.default_rng(SEED + 1)
    kp, _ = big_keyframe(rng, np.zeros((0, 2)), np.zeros((0, 32), np.uint8))
    assert big_keyframe_ok(kp)
    seg = crossing_segments(rng, 3000)
    cs, ci, _ = port.csr_from_lines(seg, INV_W, INV_H)
    assert len(ci) == 3000 * 64 and (np.diff(cs) > 32).sum() > 2000


# ---------------------------------------------------------------------------------------------------------------- GPU
@pytest.fixture
def full_config(config):
    """Every config value the local-map calls read; restored afterwards."""
    from pl_inertial_slam_b200 import drivers as D
    from pl_inertial_slam_b200 import matching as M
    names = [(M.Config, "minRatio12P"), (M.Config, "minRatio12L"), (M.Config, "lineSimTh"), (M.Config, "matchingF2FWs"),
             (M.Config, "bestLRMatches"), (D.SlamConfig, "fastMatching"), (D.SlamConfig, "maxKFEpipP"),
             (D.SlamConfig, "maxKFEpipL"), (D.SlamConfig, "minPointMatches"), (D.SlamConfig, "minLineMatches")]
    saved = [getattr(o, a) for o, a in names]
    yield apply_cfg
    for (o, a), v in zip(names, saved):
        setattr(o, a, v)


def apply_cfg(cfg):
    from pl_inertial_slam_b200 import drivers as D
    from pl_inertial_slam_b200 import matching as M
    M.Config.minRatio12P, M.Config.minRatio12L, M.Config.lineSimTh = cfg.ratio_p, cfg.ratio_l, cfg.line_sim_th
    M.Config.matchingF2FWs, M.Config.bestLRMatches = cfg.ws, cfg.best_lr
    D.SlamConfig.fastMatching, D.SlamConfig.maxKFEpipP, D.SlamConfig.maxKFEpipL = cfg.fast, cfg.epip_p, cfg.epip_l
    D.SlamConfig.minPointMatches, D.SlamConfig.minLineMatches = cfg.min_p, cfg.min_l


def dev_view(T, view):
    from pl_inertial_slam_b200 import drivers as D
    return D.map_view(T, view.cam, view.inv_w, view.inv_h, view.width, view.height)


def assert_kind(got, want, what):
    sel, m12, ok, matches = want
    assert np.array_equal(got["sel"], sel), (what, "sel")
    bad = np.flatnonzero(got["m12"] != m12)[:8] if len(got["m12"]) == len(m12) else "length"
    assert np.array_equal(got["m12"], m12), (what, "m12", bad)
    assert np.array_equal(got["ok"], ok), (what, "ok", np.flatnonzero(got["ok"] != ok)[:8])
    assert got["matches"] == matches, (what, "matches", got["matches"], matches)


def check_stores(pm, mir_p, lm, mir_l, T, view, pk, lk, cfg, what="", fallback=None):
    """match_keyframe and (at the 48 x 64 grid) LocalMap.matchMap2KF* per kind, both equal to the chain -> (the
    device's result, the chain's stages per kind).  fallback = True / False: the chain must / must not have taken the
    fallback in both kinds, checked before the device is compared."""
    from pl_inertial_slam_b200 import localmap as LM
    apply_cfg(cfg)
    v = dev_view(T, view)
    got = LM.match_keyframe(pm, lm, v, *pk, *lk, grid_rows=view.rows, grid_cols=view.cols)
    stages = {}
    for kind, store, mir, kf, lines in (("points", pm, mir_p, pk, False), ("lines", lm, mir_l, lk, True)):
        if store is None:
            continue
        st = chain(lines, mir.X, mir.act(), mir.med, T, view, kf, cfg)
        stages[kind] = st
        if fallback is not None:
            assert st["fallback"] == fallback, (what, kind, "fallback", st["grid"], len(st["sel"]))
        want = st["sel"], st["m12"], st["ok"], st["matches"]
        assert_kind(got[kind], want, (what, kind, "match_keyframe"))
        if (view.rows, view.cols) != (48, 64):
            continue
        geo, d2, feat = kf
        if lines:
            assert_kind(store.matchMap2KFLines(v, geo, feat, d2), want, (what, kind, "matchMap2KFLines"))
        elif np.array_equal(feat, np.asarray(geo, np.float32).astype(np.float64)):
            assert_kind(store.matchMap2KFPoints(v, geo, d2), want, (what, kind, "matchMap2KFPoints"))
    return got, stages


def with_fallback(cfg, mir_p, mir_l, T, view, pk, lk):
    """cfg with minPointMatches / minLineMatches between the chain's grid count and n_sel, so that the brute-force
    fallback runs after the grid pass in both kinds (a window with a single candidate is accepted whatever its
    distance, so unrelated descriptors alone leave hundreds of grid matches)."""
    mins = []
    for lines, mir, kf in ((False, mir_p, pk), (True, mir_l, lk)):
        st = chain(lines, mir.X, mir.act(), mir.med, T, view, kf, replace(cfg, fast=True))
        grid, ns = st["grid"], len(st["sel"])
        assert ns >= grid + 2, (lines, grid, ns)
        mins.append((grid + 1 + ns) // 2)
    return replace(cfg, fast=True, min_p=mins[0], min_l=mins[1])


def stores_of(ctx, case, rng):
    """Fresh stores holding the case's landmarks (one observation each: med_desc = the inserted descriptor)."""
    from pl_inertial_slam_b200.localmap import LocalMap
    out = []
    for lines, part in ((False, case.pts), (True, case.lns)):
        X, med, _ = part
        store, mir = LocalMap(lines, ctx), Mirror(lines)
        if len(X):
            dirs = unit(rng, len(X))
            store.insert(X, med, dirs)
            mir.insert(X, med, dirs)
        out += [store, mir]
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(CONSTRUCTIONS))
def test_constructions_bit_for_bit(ctx, full_config, name):
    rng = np.random.default_rng(SEED + 7)
    for case in CONSTRUCTIONS[name](np.random.default_rng(SEED)):
        pm, mir_p, lm, mir_l = stores_of(ctx, case, rng)
        check_stores(pm, mir_p, lm, mir_l, case.T, case.view, case.pts[2], case.lns[2], case.cfg, case.name)
        pm.close()
        lm.close()


def _spread(n_values, salt):
    """16 indices into n_values values, each value as often as 16 allows, in a seeded order of their own."""
    t = np.resize(np.arange(n_values), 16)
    np.random.default_rng(SEED + salt).shuffle(t)
    return t


_RATIOS = list(itertools.permutations((0.6, 0.75, 0.9, 1.0), 2))
_EPIPS = list(itertools.permutations((0.5, 1.0, 3.0), 2))
_MINS = (0, 1, 6, 10, 40)
_DRAW = dict(ratio=_spread(len(_RATIOS), 11), epip=_spread(len(_EPIPS), 12), sim=_spread(3, 13),
             min_p=_spread(len(_MINS), 14), min_l=_spread(len(_MINS), 16))


def drawn_cfg(i):
    """Keyframe i's config.  (matchingF2FWs, fastMatching, bestLRMatches) runs through all 16 combinations; the other
    values are drawn in their own seeded orders, each value at least once; the two kinds always differ in ratio and
    in the gate."""
    (rp, rl), (ep, el) = _RATIOS[_DRAW["ratio"][i]], _EPIPS[_DRAW["epip"][i]]
    return Cfg(ratio_p=rp, ratio_l=rl, line_sim_th=(0.5, 0.75, 0.95)[_DRAW["sim"][i]], ws=(0, 1, 3, 6)[i % 4],
               epip_p=ep, epip_l=el, min_p=_MINS[_DRAW["min_p"][i]], min_l=_MINS[_DRAW["min_l"][i]],
               best_lr=(i + i // 8) % 2 == 0, fast=(i // 4) % 2 == 0)


class NullStore:
    """Takes a store's updates and does nothing: the CPU replay of the sequence needs only the host mirrors."""

    def insert(self, *args):
        pass

    add_observations = set_positions = set_active = cull = insert


def sequence(pm, lm):
    """16 keyframes; before each, inserts, observations, moves, flips and culls on both stores and their mirrors.  A
    keyframe whose config asks for 40 matches of a kind with fast matching on has few features (30 points, 12
    segments), so that the grid pass can fall short and the fallback runs after it.
    Yields (cfg, mir_p, mir_l, T, points keyframe, segments keyframe)."""
    rng = np.random.default_rng(SEED + 2)
    T, _, _ = make_scene(SEED % 991, 1, False)
    mir_p, mir_l = Mirror(False), Mirror(True)
    for store, mir, lines, n in ((pm, mir_p, False, 2500), (lm, mir_l, True, 1000)):
        X, d, r = new_landmarks(rng, T, n, lines)
        store.insert(X, d, r)
        mir.insert(X, d, r)
    for i in range(16):
        cfg = drawn_cfg(i)
        update(rng, pm, mir_p, T, False)
        update(rng, lm, mir_l, T, True)
        small = cfg.fast and 40 in (cfg.min_p, cfg.min_l)
        pk, lk = kf_pair(rng, mir_p, mir_l, T, n_p=30 if small else 300, n_l=12 if small else 120)
        yield cfg, mir_p, mir_l, T, pk, lk


def test_sequence_covers_the_config_combinations():
    """The sequence's configs and, through the chain, what each keyframe runs: every value of every field; ws = 6
    with the grid pass on; the fallback after a grid pass with bestLRMatches on and off; the fallback without fast
    matching with bestLRMatches on and off."""
    cfgs = [drawn_cfg(i) for i in range(16)]
    assert {(c.ws, c.fast, c.best_lr) for c in cfgs} == set(itertools.product((0, 1, 3, 6), (True, False), (True, False)))
    assert {c.line_sim_th for c in cfgs} == {0.5, 0.75, 0.95}
    assert {c.min_p for c in cfgs} == {c.min_l for c in cfgs} == set(_MINS)
    assert {(c.ratio_p, c.ratio_l) for c in cfgs} == set(_RATIOS) and {(c.epip_p, c.epip_l) for c in cfgs} == set(_EPIPS)
    runs = set()
    for cfg, mir_p, mir_l, T, pk, lk in sequence(NullStore(), NullStore()):
        for lines, mir, kf in ((False, mir_p, pk), (True, mir_l, lk)):
            st = chain(lines, mir.X, mir.act(), mir.med, T, View(), kf, cfg)
            if cfg.fast and st["grid"]:
                runs.add(("grid", cfg.ws))
            if st["fallback"]:
                runs.add(("fallback", cfg.fast, cfg.best_lr, lines))
    assert ("grid", 6) in runs
    for fast, best_lr in itertools.product((True, False), (True, False)):
        assert any(("fallback", fast, best_lr, lines) in runs for lines in (False, True)), (fast, best_lr)
    assert any(("fallback", True, b, True) in runs for b in (True, False))


@pytest.mark.gpu
def test_sequence_config_drawn_per_kind(ctx, full_config):
    """The sequence above on two live stores, both entry points against the chain at every keyframe."""
    from pl_inertial_slam_b200.localmap import LocalMap
    pm = LocalMap(False, ctx, lm_capacity=64, obs_capacity=64)
    lm = LocalMap(True, ctx, lm_capacity=64, obs_capacity=64)
    fallbacks = 0
    for i, (cfg, mir_p, mir_l, T, pk, lk) in enumerate(sequence(pm, lm)):
        _, st = check_stores(pm, mir_p, lm, mir_l, T, View(), pk, lk, cfg, f"kf {i}")
        fallbacks += sum(s["fallback"] for s in st.values())
    assert fallbacks >= 4


@pytest.mark.gpu
def test_nonfinite_positions_are_accepted_and_never_selected(ctx, full_config):
    """set_positions takes NaN and infinite coordinates (PLM_OK, read back bit for bit); such a landmark never projects
    inside the image, so neither the chain nor the device selects it."""
    from pl_inertial_slam_b200.localmap import LocalMap
    rng = np.random.default_rng(SEED + 3)
    T, _, _ = make_scene(41, 1, False)
    for lines in (False, True):
        store, mir = LocalMap(lines, ctx), Mirror(lines)
        X, d, r = new_landmarks(rng, T, 600, lines)
        store.insert(X, d, r)
        mir.insert(X, d, r)
        sp, _, _ = port.map_select(mir.X, mir.act(), T, CAM, INV_W, INV_H, W, H)
        bad = sp[:6]
        Xn = mir.X[bad].copy()
        Xn[0, 0], Xn[1, 2], Xn[2, 1], Xn[3, 0], Xn[4, 2], Xn[5, -1] = np.nan, np.inf, -np.inf, np.inf, -np.nan, np.nan
        store.set_positions(bad, Xn)
        mir.X[bad] = Xn
        rb = store.landmarks(bad)
        assert np.array_equal(rb["X"].view(np.uint64), Xn.view(np.uint64))
        kf = keyframe(rng, mir, T, lines)
        if not lines:
            kf = (kf[0].astype(np.float32), kf[1], kf[0].astype(np.float32).astype(np.float64))
        sel = oracle_map2kf(lines, mir.X, mir.act(), mir.med, T, View(), kf, Cfg())[0]
        assert len(sel) > 0 and not np.isin(bad, sel).any()
        pk, lk = (kf, (np.zeros((0, 4), np.float32), np.zeros((0, 32), np.uint8), np.zeros((0, 3)))) if not lines else \
            ((np.zeros((0, 2), np.float32), np.zeros((0, 32), np.uint8), np.zeros((0, 2))), kf)
        check_stores(store if not lines else None, mir, store if lines else None, mir, T, View(), pk, lk, Cfg(),
                     f"non-finite lines={lines}")
        store.close()


@pytest.mark.gpu
@pytest.mark.parametrize("rows,cols", [(48, 64), (1, 1), (30, 40), (64, 128)])
def test_grid_sizes(ctx, full_config, rows, cols):
    """match_keyframe at other keyframe grids (inv_width / inv_height set to match); only the chain is a reference."""
    rng = np.random.default_rng(SEED + rows * 1000 + cols)
    T, _, _ = make_scene(43, 1, False)
    view = View(rows=rows, cols=cols)
    pm, mir_p = build_map(rng, ctx, False, 3000, T)
    lm, mir_l = build_map(rng, ctx, True, 1200, T)
    cfgs = (Cfg(), Cfg(ratio_p=0.75, ratio_l=1.0, ws=1, best_lr=False), Cfg(ws=0), Cfg(ws=1, ratio_l=0.75, best_lr=False))
    for i, cfg in enumerate(cfgs):
        (kp, pd, pl), (ln, ld, le) = kf_pair(rng, mir_p, mir_l, T)
        kp = np.concatenate([kp, (np.arange(1, cols)[:, None] * [W / cols, 0] + [0, 37]).astype(np.float32)])
        pd = np.concatenate([pd, rng.integers(0, 256, (cols - 1, 32), dtype=np.uint8)])
        pk, lk = (kp, pd, kp.astype(np.float64)), (ln, ld, le)
        fb = i >= 2                                       # the last two: the fallback after the grid pass
        if fb:
            cfg = with_fallback(cfg, mir_p, mir_l, T, view, pk, lk)
        _, st = check_stores(pm, mir_p, lm, mir_l, T, view, pk, lk, cfg, f"{rows}x{cols} cfg {i}", fallback=fb)
        assert fb or (st["points"]["matches"] > 0 and st["lines"]["matches"] > 0)


@pytest.mark.gpu
def test_keyframe_size_limits(ctx, full_config):
    """32 768 keypoints with cells past 32 items (the bitmap sort), one holding indices of the last bitmap word; and
    3000 segments crossing the whole grid, alone (they fill the n_l * max(rows, cols) item capacity exactly) and after
    ordinary ones.  The grid pass, then the fallback after it with bestLRMatches on and off."""
    rng = np.random.default_rng(SEED + 4)
    T, _, _ = make_scene(47, 1, False)
    pm, mir_p = build_map(rng, ctx, False, 4000, T)
    lm, mir_l = build_map(rng, ctx, True, 1500, T)
    (kp0, pd0, _), (ln0, ld0, le0) = kf_pair(rng, mir_p, mir_l, T, n_p=600, n_l=200)
    kp, pd = big_keyframe(rng, kp0, pd0)
    assert big_keyframe_ok(kp)
    cross = crossing_segments(rng, 3000)
    assert len(port.csr_from_lines(cross, INV_W, INV_H)[1]) == len(cross) * 64
    cd = rng.integers(0, 256, (3000, 32), dtype=np.uint8)
    pk = (kp, pd, kp.astype(np.float64))
    for lk in ((cross, cd, le_of(cross)), (np.concatenate([ln0, cross]), np.concatenate([ld0, cd]), np.concatenate([le0, le_of(cross)]))):
        check_stores(pm, mir_p, lm, mir_l, T, View(), pk, lk, Cfg(), "limits, grid")
        for best_lr in (True, False):
            cfg = with_fallback(Cfg(ratio_p=0.6, best_lr=best_lr), mir_p, mir_l, T, View(), pk, lk)
            check_stores(pm, mir_p, lm, mir_l, T, View(), pk, lk, cfg, f"limits, fallback lr={best_lr}", fallback=True)


@pytest.mark.gpu
def test_refusals_at_the_limits(ctx, full_config):
    """8193 grid cells, and 32 769 keypoints with fast matching on: PLM_E_UNSUPPORTED, nothing sent."""
    from pl_inertial_slam_b200 import _lib as L
    from pl_inertial_slam_b200 import localmap as LM
    rng = np.random.default_rng(SEED + 5)
    T, _, _ = make_scene(53, 1, False)
    pm, mir_p = build_map(rng, ctx, False, 1000, T)
    lm, mir_l = build_map(rng, ctx, True, 500, T)
    pk, lk = kf_pair(rng, mir_p, mir_l, T)
    apply_cfg(Cfg())
    v = dev_view(T, View())
    sent = (pm.h2d_bytes, lm.h2d_bytes)
    with pytest.raises(L.PlmError) as e:
        LM.match_keyframe(pm, lm, v, *pk, *lk, grid_rows=3, grid_cols=2731)
    assert e.value.status == L.PLM_E_UNSUPPORTED and 3 * 2731 == KF_MAX_CELLS + 1
    kp = rng.uniform([1, 1], [W - 1, H - 1], (KF_MAX_FEATS + 1, 2)).astype(np.float32)
    pd = rng.integers(0, 256, (len(kp), 32), dtype=np.uint8)
    with pytest.raises(L.PlmError) as e:
        LM.match_keyframe(pm, lm, v, kp, pd, None, *lk)
    assert e.value.status == L.PLM_E_UNSUPPORTED
    assert (pm.h2d_bytes, lm.h2d_bytes) == sent
    check_stores(pm, mir_p, lm, mir_l, T, View(), pk, lk, Cfg(), "after the refusals")


@pytest.mark.gpu
def test_map_scale(ctx, full_config):
    """200 000 points and 70 001 segments: the grid pass; the fallback after it on unrelated keyframe descriptors,
    with bestLRMatches on and off; and the fallback without fast matching."""
    rng = np.random.default_rng(SEED + 6)
    T, _, _ = make_scene(59, 1, False)
    pm, mir_p = build_map(rng, ctx, False, 200_000, T)
    lm, mir_l = build_map(rng, ctx, True, 70_001, T)
    (kp, pd, pl), (ln, ld, le) = kf_pair(rng, mir_p, mir_l, T, n_p=600, n_l=200)
    cfg = Cfg(ratio_p=0.9, ratio_l=0.75, epip_p=3.0, epip_l=1.0)
    _, st = check_stores(pm, mir_p, lm, mir_l, T, View(), (kp, pd, pl), (ln, ld, le), cfg, "map scale, grid",
                         fallback=False)
    assert st["points"]["matches"] > 0 and st["lines"]["matches"] > 0
    pk = (kp, rng.integers(0, 256, pd.shape, dtype=np.uint8), pl)
    lk = (ln, rng.integers(0, 256, ld.shape, dtype=np.uint8), le)
    for best_lr in (True, False):
        fb = with_fallback(replace(cfg, best_lr=best_lr), mir_p, mir_l, T, View(), pk, lk)
        check_stores(pm, mir_p, lm, mir_l, T, View(), pk, lk, fb, f"map scale, fallback lr={best_lr}", fallback=True)
    check_stores(pm, mir_p, lm, mir_l, T, View(), pk, lk, replace(cfg, fast=False), "map scale, no fast matching",
                 fallback=True)
