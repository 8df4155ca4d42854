"""One keyframe against both resident stores in one call (plm_localmap_match_kf_pl, localmap.match_keyframe): the map
half of MapHandler::lookForCommonMatches (src/mapHandler.cpp:865-871) from the keyframe's raw features, grids built on
the device.

GPU (-m gpu): bit for bit against LocalMap.matchMap2KFPoints + matchMap2KFLines (host-built grids, one
plm_localmap_match_kf per kind) and against drivers.matchMap2KF*Full on a host mirror, over a sequence of keyframes
with both stores updated between them; grid corner cases; one kind only; per-call bytes, launches and synchronisations
against the header's formulas and independent of the map size; failed calls leave both stores unchanged.
CPU: the ctypes layouts, argument checks made before any CUDA call, and the host grid builders the comparison rests on
(grid.csr_from_points, drivers.line_grid) against the oracle's grid fill."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import oracle
from conftest import ROOT
from test_gpu_localmap import (Mirror, build_map, config, ctx, keyframe, new_landmarks, oracle_flip,  # noqa: F401
                               unit)
from test_reproj import CAM, H, INV_H, INV_W, W, make_scene

SEED = 20261023


# ---------------------------------------------------------------------------------------------------------------- CPU
def test_kf_struct_layouts_match_the_header(tmp_path):
    from pl_inertial_slam_b200 import _lib as L
    pairs = [("plm_localmap_kf_raw", L.LocalMapKfRaw), ("plm_localmap_out", L.LocalMapOut),
             ("plm_localmap_pl_out", L.LocalMapPlOut)]
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "plmatch.h"', 'int main(void) {']
    for cname, cls in pairs:
        lines.append(f'  printf("{cname} %zu", sizeof({cname}));')
        for fname, _ in cls._fields_:
            lines.append(f'  printf(" %zu", offsetof({cname}, {fname}));')
        lines.append('  printf("\\n");')
    lines += ['  return 0;', '}']
    src = tmp_path / "layout.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "layout"
    subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    out = subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.strip().splitlines()
    assert len(out) == len(pairs)
    for (cname, cls), line in zip(pairs, out):
        nums = [int(x) for x in line.split()[1:]]
        assert nums[0] == C.sizeof(cls), cname
        assert nums[1:] == [getattr(cls, f).offset for f, _ in cls._fields_], cname


def test_kf_argument_checks_need_no_gpu(plm_lib):
    """Failures reported before any CUDA call (this runs without a device)."""
    from pl_inertial_slam_b200 import _lib as L
    lib = plm_lib
    v, kf, p, out = L.MapView(), L.LocalMapKfRaw(), L.LocalMapParams(), L.LocalMapPlOut()
    kf.grid_rows, kf.grid_cols = 48, 64
    f = lib.plm_localmap_match_kf_pl
    assert f(None, None, C.byref(v), C.byref(kf), C.byref(p), C.byref(p), C.byref(out)) == L.PLM_E_INVALID   # no store
    assert f(None, None, None, C.byref(kf), C.byref(p), C.byref(p), C.byref(out)) == L.PLM_E_INVALID
    assert f(None, None, C.byref(v), None, C.byref(p), C.byref(p), C.byref(out)) == L.PLM_E_INVALID
    assert f(None, None, C.byref(v), C.byref(kf), C.byref(p), C.byref(p), None) == L.PLM_E_INVALID


def scenario_kp():
    """Keypoints on cell borders (x * inv_width exactly an integer), in the image corners, and outside the image."""
    bx = np.arange(0, 65) * (W / 64.0)               # 11.75 px: exact in float32 and in the double product
    by = np.arange(0, 49) * (H / 48.0)               # 10 px
    kp = [np.stack([bx, np.full_like(bx, 100.0)], 1), np.stack([np.full_like(by, 200.0), by], 1),
          [[0, 0], [W - 1e-3, H - 1e-3], [W, H], [-0.5, 3], [-20, 40], [W + 30, 10], [30, -1], [30, H + 7],
           [np.nextafter(np.float32(11.75), np.float32(0)), 5]]]
    return np.concatenate([np.asarray(k, np.float64) for k in kp]).astype(np.float32)


def scenario_segments(rng):
    """Horizontal, vertical, zero-length, reversed, steep / shallow both ways, and segments longer than the grid."""
    s = [[10, 100, 600, 100], [600, 100, 10, 100], [300, 5, 300, 470], [300, 470, 300, 5], [250, 250, 250, 250],
         [0, 0, 0, 0], [11.75, 10, 11.75, 10], [-300, 240, W + 400, 240], [376, -500, 380, H + 600],
         [-100, -100, W + 100, H + 100], [W + 100, H + 100, -100, -100], [700, 20, 30, 460], [30, 460, 700, 20],
         [5, 5, 700, 9], [5, 5, 9, 470], [W - 1, H - 1, W + 50, H + 50], [-50, -50, -1, -1]]
    r = rng.uniform(-60, [W + 60, H + 60, W + 60, H + 60], (40, 4))
    return np.concatenate([np.asarray(s, np.float64), r]).astype(np.float32)


def test_host_grids_match_the_oracle_fill():
    """The host grids the GPU tests compare against (grid.csr_from_points over kp * inv, drivers.line_grid) equal the
    oracle's restatement of the grid fill of stereoFrame.cpp:146-150 / :336-349, and every segment's cells equal the
    compiled reference's getLineCoords when it is built."""
    from pl_inertial_slam_b200 import drivers as D
    from pl_inertial_slam_b200 import grid as G
    rng = np.random.default_rng(SEED)
    kp = np.concatenate([scenario_kp(), rng.uniform(-30, [W + 30, H + 30], (500, 2)).astype(np.float32)])
    c = kp.astype(np.float64)
    cs, ci = G.csr_from_points(c[:, 0] * INV_W, c[:, 1] * INV_H)
    cs_o, ci_o = oracle.port.csr_from_points(kp, INV_W, INV_H)
    assert np.array_equal(cs, cs_o) and np.array_equal(ci, ci_o)
    seg = scenario_segments(rng)
    cs, ci, dirs = D.line_grid(seg, INV_W, INV_H)
    cs_o, ci_o, dirs_o = oracle.port.csr_from_lines(seg, INV_W, INV_H)
    assert np.array_equal(cs, cs_o) and np.array_equal(ci, ci_o)
    assert np.array_equal(dirs.view(np.uint64), dirs_o.view(np.uint64))             # NaN of zero-length segments too
    assert np.isnan(dirs[4]).all()
    for k in range(len(cs) - 1):                                                     # push order: ascending index
        assert (np.diff(ci[cs[k]:cs[k + 1]]) > 0).all()
    if oracle.ref.available():
        s64 = seg.astype(np.float64) * [INV_W, INV_H, INV_W, INV_H]
        ids, cx, cy = G.line_cells(s64[:, 0], s64[:, 1], s64[:, 2], s64[:, 3])
        for i, s in enumerate(s64):
            want = oracle.ref.line_coords(*s)
            assert np.array_equal(np.stack([cx[ids == i], cy[ids == i]], 1), want)


# ---------------------------------------------------------------------------------------------------------------- GPU
def to_kf(kp_px, d2):
    """Points of a keyframe as the raw call takes them: float32 pixels; pl = the same values in double."""
    kp = np.asarray(kp_px, np.float32).reshape(-1, 2)
    return kp, d2, kp.astype(np.float64)


def run_both(pm, lm, view, pk, lk):
    """match_keyframe and the two host-grid calls on the same stores -> (combined, per kind results)."""
    from pl_inertial_slam_b200 import localmap as LM
    kp, pd, pl = pk
    ln, ld, le = lk
    got = LM.match_keyframe(pm, lm, view, kp, pd, pl, ln, ld, le)
    want = {"points": pm.matchMap2KFPoints(view, kp, pd) if pm is not None else None,
            "lines": lm.matchMap2KFLines(view, ln, le, ld) if lm is not None else None}
    return got, want


def assert_same(a, b):
    for k in ("sel", "m12", "ok"):
        assert np.array_equal(a[k], b[k]), k
    assert a["matches"] == b["matches"]


def check_kf(pm, lm, view, pk, lk, mir_p=None, mir_l=None):
    """match_keyframe == host-grid path == drivers.matchMap2KF*Full (when a mirror is given)."""
    from pl_inertial_slam_b200 import drivers as D
    got, want = run_both(pm, lm, view, pk, lk)
    for kind in ("points", "lines"):
        if want[kind] is None:
            assert got[kind] is None
            continue
        assert_same(got[kind], want[kind])
    if mir_p is not None:
        kp, pd, _ = pk
        assert_same(got["points"], D.matchMap2KFPointsFull(mir_p.X, mir_p.act(), mir_p.med, view, kp.astype(np.float64), pd))
    if mir_l is not None:
        ln, ld, le = lk
        assert_same(got["lines"], D.matchMap2KFLinesFull(mir_l.X, mir_l.act(), mir_l.med, view, ln, le, ld))
    return got


def kf_pair(rng, mir_p, mir_l, T, n_p=300, n_l=120):
    px, pd, _ = keyframe(rng, mir_p, T, False, n2=n_p)
    ln, ld, le = keyframe(rng, mir_l, T, True, n2=n_l)
    return to_kf(px, pd), (ln, ld, le)


def update(rng, store, mir, T, lines):
    X, d, r = new_landmarks(rng, T, 30, lines)
    store.insert(X, d, r)
    mir.insert(X, d, r)
    live = mir.live()
    idx = rng.choice(live, 120)
    od, orr = oracle_flip(rng, mir.med[idx], 0.1), unit(rng, len(idx))
    store.add_observations(idx, od, orr)
    mir.add(idx, od, orr)
    mv = rng.choice(mir.live(), 150, replace=False)
    Xn = mir.X[mv] + rng.normal(0, 0.05, (len(mv), mir.xw))
    store.set_positions(mv, Xn)
    mir.X[mv] = Xn
    fl = rng.choice(mir.live(), 200, replace=False)
    val = (rng.random(len(fl)) < 0.6).astype(np.uint8)
    store.set_active(fl, val)
    mir.active[fl] = val
    cu = rng.choice(mir.live(), 8, replace=False)
    store.cull(cu)
    mir.alive[cu] = False


@pytest.mark.gpu
def test_sequence_parity_both_kinds(ctx, config):
    """24 keyframes; between them inserts, observations, moves, active flips and culls on both stores; best_lr on / off
    and ratios 0.9 / 0.75 in turn."""
    from pl_inertial_slam_b200 import drivers as D
    from pl_inertial_slam_b200.localmap import LocalMap
    Cfg, _ = config
    rng = np.random.default_rng(SEED + 1)
    T, _, _ = make_scene(SEED % 997, 1, False)
    view = D.map_view(T, CAM, INV_W, INV_H, W, H)
    pm, mir_p = LocalMap(False, ctx, lm_capacity=64, obs_capacity=64), Mirror(False)
    lm, mir_l = LocalMap(True, ctx, lm_capacity=64, obs_capacity=64), Mirror(True)
    for store, mir, lines, n in ((pm, mir_p, False, 2500), (lm, mir_l, True, 1000)):
        X, d, r = new_landmarks(rng, T, n, lines)
        store.insert(X, d, r)
        mir.insert(X, d, r)
    total = 0
    for kf_i in range(24):
        Cfg.bestLRMatches = kf_i % 2 == 0
        Cfg.minRatio12P = Cfg.minRatio12L = 0.9 if (kf_i // 2) % 2 == 0 else 0.75
        update(rng, pm, mir_p, T, False)
        update(rng, lm, mir_l, T, True)
        pk, lk = kf_pair(rng, mir_p, mir_l, T)
        got = check_kf(pm, lm, view, pk, lk, mir_p, mir_l)
        total += got["points"]["matches"] + got["lines"]["matches"]
        assert got["cost"]["syncs"] <= 3
    assert total > 0


@pytest.mark.gpu
def test_grid_corner_cases(ctx, config):
    """Keypoints on cell borders and outside the image, tie-stress descriptors, and horizontal, vertical, zero-length
    (NaN direction), reversed and longer-than-the-grid segments: equal to the host-grid path and the drivers."""
    from pl_inertial_slam_b200 import drivers as D
    from pl_inertial_slam_b200 import synth
    Cfg, _ = config
    rng = np.random.default_rng(SEED + 2)
    T, _, _ = make_scene(23, 1, False)
    view = D.map_view(T, CAM, INV_W, INV_H, W, H)
    pm, mir_p = build_map(rng, ctx, False, 3000, T)
    lm, mir_l = build_map(rng, ctx, True, 1500, T)
    kp = scenario_kp()
    seg = scenario_segments(rng)
    (kp0, pd0, _), (ln0, ld0, le0) = kf_pair(rng, mir_p, mir_l, T)
    kp = np.concatenate([kp, kp0])
    seg = np.concatenate([seg, ln0])
    a = np.concatenate([seg[:, :2].astype(np.float64), np.ones((len(seg), 1))], 1)
    b = np.concatenate([seg[:, 2:].astype(np.float64), np.ones((len(seg), 1))], 1)
    le = np.cross(a, b)
    with np.errstate(invalid="ignore", divide="ignore"):
        le /= np.hypot(le[:, 0], le[:, 1])[:, None]
    le[np.isnan(le)] = 0.0
    for desc_kind in ("related", "tie"):
        if desc_kind == "related":
            pd = np.concatenate([rng.integers(0, 256, (len(kp) - len(kp0), 32), dtype=np.uint8), pd0])
            ld = np.concatenate([rng.integers(0, 256, (len(seg) - len(ln0), 32), dtype=np.uint8), ld0])
        else:
            pd, ld = synth.tie_stress_desc(rng, len(kp)), synth.tie_stress_desc(rng, len(seg))
        for best_lr in (True, False):
            Cfg.bestLRMatches = best_lr
            check_kf(pm, lm, view, to_kf(kp, pd), (seg, ld, le), mir_p, mir_l)
    # every keypoint / segment in one or two cells: cells far past the per-thread sort size
    Cfg.bestLRMatches = True
    kp_one = np.tile(np.float32([[100.3, 200.7]]), (300, 1))
    seg_one = np.tile(np.float32([[100.0, 200.0, 130.0, 201.0]]), (150, 1))
    check_kf(pm, lm, view, to_kf(kp_one, synth.tie_stress_desc(rng, 300)),
             (seg_one, synth.tie_stress_desc(rng, 150), np.tile([0.0, 1.0, -200.0], (150, 1))), mir_p, mir_l)


@pytest.mark.gpu
def test_one_kind_and_empty_cases(ctx, config):
    from pl_inertial_slam_b200 import drivers as D
    from pl_inertial_slam_b200.localmap import LocalMap
    _, Slam = config
    rng = np.random.default_rng(SEED + 3)
    T, _, _ = make_scene(29, 1, False)
    view = D.map_view(T, CAM, INV_W, INV_H, W, H)
    pm, mir_p = build_map(rng, ctx, False, 3000, T)
    lm, mir_l = build_map(rng, ctx, True, 1500, T)
    pk, lk = kf_pair(rng, mir_p, mir_l, T)
    e_p = (np.zeros((0, 2), np.float32), np.zeros((0, 32), np.uint8), np.zeros((0, 2)))
    e_l = (np.zeros((0, 4), np.float32), np.zeros((0, 32), np.uint8), np.zeros((0, 3)))
    check_kf(pm, None, view, pk, lk, mir_p)                                  # lines = NULL
    check_kf(None, lm, view, pk, lk, None, mir_l)                            # points = NULL
    check_kf(pm, lm, view, pk, e_l, mir_p, mir_l)                            # n_l = 0
    check_kf(pm, lm, view, e_p, lk, mir_p, mir_l)                            # n_p = 0
    check_kf(pm, lm, view, e_p, e_l, mir_p, mir_l)
    empty_l, mir_e = LocalMap(True, ctx), Mirror(True)                       # an empty map
    got = check_kf(pm, empty_l, view, pk, lk, mir_p, mir_e)
    assert len(got["lines"]["sel"]) == 0
    # the fallback in one kind only (unrelated point descriptors), then in the other; fast matching on and off
    kp, pd, pl = pk
    ln, ld, le = lk
    pk_rand = (kp, rng.integers(0, 256, pd.shape, dtype=np.uint8), pl)
    lk_rand = (ln, rng.integers(0, 256, ld.shape, dtype=np.uint8), le)
    for fast in (True, False):
        Slam.fastMatching = fast
        check_kf(pm, lm, view, pk_rand, lk, mir_p, mir_l)
        check_kf(pm, lm, view, pk, lk_rand, mir_p, mir_l)
        check_kf(pm, lm, view, pk, lk, mir_p, mir_l)
    Slam.fastMatching = True
    # n_sel = 0 in one kind, then in both
    pm.set_active(np.arange(len(mir_p.X))[mir_p.alive], 0)
    mir_p.active[:] = 0
    got = check_kf(pm, lm, view, pk, lk, mir_p, mir_l)
    assert len(got["points"]["sel"]) == 0 and len(got["lines"]["sel"]) > 0
    lm.set_active(np.arange(len(mir_l.X))[mir_l.alive], 0)
    mir_l.active[:] = 0
    got = check_kf(pm, lm, view, pk, lk, mir_p, mir_l)
    assert got["cost"]["syncs"] == 1 and got["cost"]["d2h_bytes"] == 8


@pytest.mark.gpu
def test_cost_formulas_independent_of_map_size(ctx, config):
    """10 000 landmarks per kind, then the same plus 190 000 behind the camera: equal bytes, launches and
    synchronisations per call, equal to the header's formulas; launches = the two match_kf calls' + 1 grid build."""
    from pl_inertial_slam_b200 import drivers as D
    from pl_inertial_slam_b200 import localmap as LM
    T, _, _ = make_scene(31, 1, False)
    view = D.map_view(T, CAM, INV_W, INV_H, W, H)
    costs = []
    for extra in (0, 190_000):
        rng = np.random.default_rng(SEED + 4)
        pm, mir_p = build_map(rng, ctx, False, 10_000, T)
        lm, mir_l = build_map(rng, ctx, True, 10_000, T)
        for store, mir, lines in ((pm, mir_p, False), (lm, mir_l, True)):
            if extra:
                X, d, r = new_landmarks(np.random.default_rng(5), T, extra, lines, behind=True)
                store.insert(X, d, r)
                mir.insert(X, d, r)
        pk, lk = kf_pair(rng, mir_p, mir_l, T, n_p=500, n_l=200)
        kp, pd, pl = pk
        ln, ld, le = lk
        rows = []
        for kind_pk in (pk, (kp, rng.integers(0, 256, pd.shape, dtype=np.uint8), pl)):   # grid only, then a fallback
            LM.match_keyframe(pm, lm, view, *kind_pk, *lk)                                 # warm-up: staging sized
            ctx.synchronize()
            h = (pm.h2d_bytes, pm.d2h_bytes, lm.h2d_bytes, lm.d2h_bytes)
            l0 = ctx.launch_count
            got = LM.match_keyframe(pm, lm, view, *kind_pk, *lk)
            ctx.synchronize()
            l_pl = ctx.launch_count - l0
            dh = (pm.h2d_bytes - h[0], pm.d2h_bytes - h[1], lm.h2d_bytes - h[2], lm.d2h_bytes - h[3])
            l0 = ctx.launch_count
            pm.matchMap2KFPoints(view, kind_pk[0], kind_pk[1])
            l_p = ctx.launch_count - l0
            l0 = ctx.launch_count
            lm.matchMap2KFLines(view, ln, le, ld)
            l_l = ctx.launch_count - l0
            c = got["cost"]
            nsp, nsl = len(got["points"]["sel"]), len(got["lines"]["sel"])
            assert nsp > 0 and nsl > 0
            assert c["h2d_bytes"] == 56 * len(kp) + 72 * len(ln)
            assert c["d2h_bytes"] == 8 + 8 * (c["syncs"] == 3) + 9 * (nsp + nsl) + 8
            assert c["syncs"] == 3                      # both n_sel > min_matches: the grid counts are read
            assert l_pl == l_p + l_l + 1
            assert dh == (56 * len(kp), 4 + 4 + 9 * nsp + 4, 72 * len(ln), 4 + 4 + 9 * nsl + 4)
            rows.append((tuple(c.values()), l_pl, dh, nsp, nsl))
        costs.append(rows)
    assert costs[0] == costs[1]


@pytest.mark.gpu
def test_failed_calls_leave_both_stores_unchanged(ctx, config):
    from pl_inertial_slam_b200 import _lib as L
    from pl_inertial_slam_b200 import drivers as D
    from pl_inertial_slam_b200 import localmap as LM
    from pl_inertial_slam_b200.localmap import LocalMap
    from pl_inertial_slam_b200.matching import Context
    Cfg, _ = config
    rng = np.random.default_rng(SEED + 5)
    T, _, _ = make_scene(37, 1, False)
    view = D.map_view(T, CAM, INV_W, INV_H, W, H)
    pm, mir_p = build_map(rng, ctx, False, 3000, T)
    lm, mir_l = build_map(rng, ctx, True, 1500, T)
    pk, lk = kf_pair(rng, mir_p, mir_l, T)

    def snapshot():
        return pm.landmarks(mir_p.live()), lm.landmarks(mir_l.live()), len(pm), len(lm)

    first = check_kf(pm, lm, view, pk, lk, mir_p, mir_l)
    before = snapshot()
    sent = (pm.h2d_bytes, lm.h2d_bytes)
    other = Context(0)
    lm_other = LocalMap(True, other)
    X, d, r = new_landmarks(rng, T, 50, True)
    lm_other.insert(X, d, r)
    with pytest.raises(L.PlmError) as e:                                      # stores on different contexts
        LM.match_keyframe(pm, lm_other, view, *pk, *lk)
    assert e.value.status == L.PLM_E_INVALID
    Cfg.minRatio12P = 1.5                                                     # ratio > 1
    with pytest.raises(L.PlmError) as e:
        LM.match_keyframe(pm, lm, view, *pk, *lk)
    assert e.value.status == L.PLM_E_RATIO
    Cfg.minRatio12P = 0.9
    bad = np.asarray(lk[0]).copy()
    bad[0, 0] = np.nan                                                        # a segment endpoint that is not finite
    with pytest.raises(L.PlmError) as e:
        LM.match_keyframe(pm, lm, view, *pk, bad, lk[1], lk[2])
    assert e.value.status == L.PLM_E_INVALID
    # null pointers through the C entry point
    lib = L.load()
    kf, p, out = L.LocalMapKfRaw(), L.LocalMapParams(), L.LocalMapPlOut()
    kf.n_p, kf.n_l, kf.grid_rows, kf.grid_cols = 5, 5, 48, 64
    assert lib.plm_localmap_match_kf_pl(pm._h, lm._h, C.byref(view), C.byref(kf), C.byref(p), C.byref(p), C.byref(out)) == L.PLM_E_INVALID
    assert lib.plm_localmap_match_kf_pl(pm._h, lm._h, C.byref(view), C.byref(kf), None, C.byref(p), C.byref(out)) == L.PLM_E_INVALID
    assert lib.plm_localmap_match_kf_pl(lm._h, pm._h, C.byref(view), C.byref(kf), C.byref(p), C.byref(p), C.byref(out)) == L.PLM_E_INVALID
    assert (pm.h2d_bytes, lm.h2d_bytes) == sent                              # nothing was sent
    after = snapshot()
    for x, y in zip(before[:2], after[:2]):
        for k in x:
            assert np.array_equal(np.asarray(x[k]).view(np.uint8), np.asarray(y[k]).view(np.uint8)), k
    assert before[2:] == after[2:]
    again = check_kf(pm, lm, view, pk, lk, mir_p, mir_l)
    for kind in ("points", "lines"):
        assert_same(first[kind], again[kind])
    # a culled-only map: nothing selected, nothing changed
    cu = mir_l.live()
    lm.cull(cu)
    mir_l.alive[cu] = False
    got = check_kf(pm, lm, view, pk, lk, mir_p, mir_l)
    assert len(got["lines"]["sel"]) == 0 and got["lines"]["matches"] == 0
    assert len(lm) == before[3]
    lm_other.close()
