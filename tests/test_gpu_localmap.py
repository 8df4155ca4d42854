"""Resident local map (plm_localmap_*, localmap.LocalMap; src/mapHandler.cpp:583-803, src/mapFeatures.cpp).

GPU (-m gpu), bit for bit (fp64 by bit pattern): sequences of inserts / observation appends / moves / active flips /
culls, each step followed by a match against drivers.matchMap2KF*Full on a host mirror of X, active and med_desc, and
read-backs against oracle.port.med_desc on the mirrored observation lists; edge cases; growth from capacity 1; per-call
copies and launches independent of the map size; failed calls leave the store unchanged.
CPU: argument validation (reported before any CUDA call) and the ctypes layouts of the two new structs."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT
from test_reproj import CAM, H, INV_H, INV_W, W, make_scene

SEED = 20261022


# ---------------------------------------------------------------------------------------------------------------- CPU
def test_localmap_struct_layouts_match_the_header(tmp_path):
    from pl_inertial_slam_b200 import _lib as L
    pairs = [("plm_localmap_kf", L.LocalMapKf), ("plm_localmap_params", L.LocalMapParams)]
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


def test_localmap_argument_validation_needs_no_gpu(plm_lib):
    """Every precondition failure below is reported before any CUDA call (this runs without a device)."""
    from pl_inertial_slam_b200 import _lib as L
    lib = plm_lib
    h = C.c_void_p()
    assert lib.plm_localmap_create(None, 2, 0, 0, C.byref(h)) == L.PLM_E_INVALID
    assert lib.plm_localmap_create(None, 0, -1, 0, C.byref(h)) == L.PLM_E_INVALID
    assert lib.plm_localmap_create(None, 0, 0, -1, C.byref(h)) == L.PLM_E_INVALID
    assert lib.plm_localmap_create(None, 0, 0, 1 << 40, C.byref(h)) == L.PLM_E_UNSUPPORTED
    assert lib.plm_localmap_create(None, 0, 0, 0, None) == L.PLM_E_INVALID
    idx = np.zeros(2, np.int32)
    d = np.zeros((2, 32), np.uint8)
    x = np.zeros((2, 6))
    assert lib.plm_localmap_insert(None, 2, x.ctypes.data_as(L.f64p), d.ctypes.data_as(L.u8p), 32, x.ctypes.data_as(L.f64p), None) == L.PLM_E_INVALID
    assert lib.plm_localmap_add_observations(None, 2, idx.ctypes.data_as(L.i32p), d.ctypes.data_as(L.u8p), 32, x.ctypes.data_as(L.f64p)) == L.PLM_E_INVALID
    assert lib.plm_localmap_set_positions(None, 2, idx.ctypes.data_as(L.i32p), x.ctypes.data_as(L.f64p)) == L.PLM_E_INVALID
    assert lib.plm_localmap_set_active(None, 2, idx.ctypes.data_as(L.i32p), d.ctypes.data_as(L.u8p)) == L.PLM_E_INVALID
    assert lib.plm_localmap_cull(None, 2, idx.ctypes.data_as(L.i32p)) == L.PLM_E_INVALID
    n_sel, cnt = C.c_int(0), C.c_int(0)
    assert lib.plm_localmap_match_kf(None, None, None, None, None, None, None, C.byref(n_sel), C.byref(cnt)) == L.PLM_E_INVALID
    assert lib.plm_localmap_read(None, 0, None, None, None, None, None) == L.PLM_E_INVALID
    assert lib.plm_localmap_size(None) == 0 and lib.plm_localmap_h2d_bytes(None) == 0 and lib.plm_localmap_d2h_bytes(None) == 0
    assert lib.plm_localmap_destroy(None) == L.PLM_OK


# ---------------------------------------------------------------------------------------------------------------- GPU
def bits(a):
    return np.ascontiguousarray(a, np.float64).view(np.uint64)


_CTX = []


@pytest.fixture(scope="module")
def ctx(plm_lib):
    from pl_inertial_slam_b200.matching import Context
    if not _CTX:
        _CTX.append(Context(0))
    return _CTX[0]


@pytest.fixture
def config():
    """Config / SlamConfig as the drivers read them; restored afterwards."""
    from pl_inertial_slam_b200 import drivers as D
    from pl_inertial_slam_b200 import matching as M
    saved = (M.Config.minRatio12P, M.Config.minRatio12L, M.Config.bestLRMatches, D.SlamConfig.fastMatching)
    M.Config.minRatio12P, M.Config.minRatio12L, M.Config.bestLRMatches, D.SlamConfig.fastMatching = 0.9, 0.9, True, True
    yield M.Config, D.SlamConfig
    M.Config.minRatio12P, M.Config.minRatio12L, M.Config.bestLRMatches, D.SlamConfig.fastMatching = saved


def unit(rng, n):
    v = rng.normal(0, 1, (n, 3))
    return v / np.linalg.norm(v, axis=1, keepdims=True)


class Mirror:
    """What MapHandler would hold on the host: X, active, culled slots and the observation lists; med_desc / med_dir
    from oracle.port.med_desc."""

    def __init__(self, lines):
        self.xw = 6 if lines else 3
        self.X = np.zeros((0, self.xw))
        self.active = np.zeros(0, np.uint8)
        self.alive = np.zeros(0, bool)
        self.obs_d, self.obs_r = [], []
        self.med = np.zeros((0, 32), np.uint8)
        self.mdir = np.zeros((0, 3))

    def insert(self, X, d, r):
        self.X = np.concatenate([self.X, X])
        self.active = np.concatenate([self.active, np.ones(len(X), np.uint8)])
        self.alive = np.concatenate([self.alive, np.ones(len(X), bool)])
        self.obs_d += [[row] for row in d]
        self.obs_r += [[row] for row in r]
        self.med = np.concatenate([self.med, d])
        self.mdir = np.concatenate([self.mdir, r])

    def recompute(self, ids):
        import oracle
        ids = np.unique(ids)
        lens = [len(self.obs_d[i]) for i in ids]
        start = np.concatenate([[0], np.cumsum(lens)]).astype(np.int32)
        desc = np.concatenate([np.asarray(self.obs_d[i]) for i in ids])
        dirs = np.concatenate([np.asarray(self.obs_r[i]) for i in ids])
        _, med, mdir = oracle.port.med_desc(desc, dirs, start)
        self.med[ids], self.mdir[ids] = med, mdir

    def add(self, idx, d, r):
        for i, a, b in zip(idx, d, r):
            self.obs_d[i].append(a)
            self.obs_r[i].append(b)
        self.recompute(idx)

    def live(self):
        return np.flatnonzero(self.alive)

    def act(self):
        return (self.active.astype(bool) & self.alive).astype(np.uint8)


def keyframe(rng, mir, T, lines, n2=300, noise=0.7, random_frac=0.1):
    """A keyframe whose unmatched features see some of the selectable landmarks (pixels, descriptors, le for lines)."""
    import oracle
    s_o, _, p_o = oracle.port.map_select(mir.X, mir.act(), T, CAM, INV_W, INV_H, W, H) if len(mir.X) else (np.zeros(0, np.int32), None, np.zeros((0, 4 if lines else 2)))
    k = min(n2, len(s_o))
    seen = rng.choice(len(s_o), k, replace=False) if k else np.zeros(0, np.int64)
    px = p_o[seen] + rng.normal(0, noise, (k, p_o.shape[1]))
    px = np.clip(px, 1.0, np.tile([W - 2.0, H - 2.0], px.shape[1] // 2))
    d2 = oracle_flip(rng, mir.med[s_o[seen]], 0.06)
    nr = int(k * random_frac)
    if nr:
        d2[:nr] = rng.integers(0, 256, (nr, 32), dtype=np.uint8)
    if not lines:
        return px, d2, None
    px = px.astype(np.float32)
    p64 = px.astype(np.float64)
    a = np.stack([p64[:, 0], p64[:, 1], np.ones(k)], 1)
    b = np.stack([p64[:, 2], p64[:, 3], np.ones(k)], 1)
    le = np.cross(a, b)
    le /= np.hypot(le[:, 0], le[:, 1])[:, None]
    return px, d2, le


def oracle_flip(rng, d, p):
    from pl_inertial_slam_b200 import synth
    return synth.flip_bits(rng, np.ascontiguousarray(d), p)


def match_both(lm, mir, view, kf):
    from pl_inertial_slam_b200 import drivers as D
    px, d2, le = kf
    if le is None:
        got = lm.matchMap2KFPoints(view, px, d2)
        want = D.matchMap2KFPointsFull(mir.X, mir.act(), mir.med, view, px, d2)
    else:
        got = lm.matchMap2KFLines(view, px, le, d2)
        want = D.matchMap2KFLinesFull(mir.X, mir.act(), mir.med, view, px, le, d2)
    return got, want


def assert_match(lm, mir, view, kf):
    got, want = match_both(lm, mir, view, kf)
    for k in ("sel", "m12", "ok"):
        assert np.array_equal(got[k], want[k]), k
    assert got["matches"] == want["matches"]
    return got


def assert_readback(lm, mir, ids):
    ids = np.asarray(ids)
    ids = ids[mir.alive[ids]]
    r = lm.landmarks(ids)
    assert np.array_equal(bits(r["X"]), bits(mir.X[ids]))
    assert np.array_equal(r["med_desc"], mir.med[ids])
    assert np.array_equal(bits(r["med_dir"]), bits(mir.mdir[ids]))
    assert np.array_equal(r["n_obs"], [len(mir.obs_d[i]) for i in ids])


def new_landmarks(rng, T, n, lines, behind=False):
    _, X, _ = make_scene(int(rng.integers(1 << 30)), n, lines)
    if behind:                      # behind the camera (Pf2 < 0): never selected; X = R^T (Pf - t)
        P = np.concatenate([rng.uniform(-6, 6, (n, 2)), rng.uniform(-12, -1, (n, 1))], 1)
        ends = [P] + ([P + rng.normal(0, 0.4, (n, 3))] if lines else [])
        X = np.concatenate([(e - T[:, 3]) @ T[:, :3] for e in ends], 1)
    return X, rng.integers(0, 256, (n, 32), dtype=np.uint8), unit(rng, n)


@pytest.mark.gpu
@pytest.mark.parametrize("lines", [False, True])
def test_sequence_parity(ctx, config, lines):
    """30 keyframes: inserts, observation appends (three landmarks driven past 32, 64 and 128 observations through
    several relocations), moves, active flips and culls, each step followed by a match and read-backs."""
    from pl_inertial_slam_b200 import drivers as D
    from pl_inertial_slam_b200.localmap import LocalMap
    rng = np.random.default_rng(SEED + lines)
    T, _, _ = make_scene(SEED % 1000, 1, lines)
    view = D.map_view(T, CAM, INV_W, INV_H, W, H)
    lm, mir = LocalMap(lines, ctx, lm_capacity=64, obs_capacity=64), Mirror(lines)
    X, d, r = new_landmarks(rng, T, 3000 if not lines else 1200, lines)
    assert np.array_equal(lm.insert(X, d, r), np.arange(len(X)))
    mir.insert(X, d, r)
    hot = np.array([5, 17, 29])
    for kf_i in range(30):
        # insert
        X, d, r = new_landmarks(rng, T, 40, lines)
        first = len(mir.X)
        assert np.array_equal(lm.insert(X, d, r), np.arange(first, first + 40))
        mir.insert(X, d, r)
        assert_match(lm, mir, view, keyframe(rng, mir, T, lines))
        # observations: random live landmarks (repeats inside the call) + the hot ones, 2 / 3 / 5 per keyframe
        live = mir.live()
        idx = np.concatenate([rng.choice(live, 150), rng.choice(live, 20), np.repeat(hot, [2, 3, 5])])
        rng.shuffle(idx)
        idx = idx[mir.alive[idx]]
        od = oracle_flip(rng, mir.med[idx], 0.1)
        orr = unit(rng, len(idx))
        lm.add_observations(idx, od, orr)
        mir.add(idx, od, orr)
        assert_match(lm, mir, view, keyframe(rng, mir, T, lines))
        assert_readback(lm, mir, np.concatenate([np.unique(idx), rng.choice(len(mir.X), 50)]))
        # moves (a slot twice: the last entry wins)
        mv = rng.choice(mir.live(), 200, replace=False)
        mv = np.concatenate([mv, mv[:3]])
        Xn = mir.X[mv] + rng.normal(0, 0.05, (len(mv), mir.xw))
        lm.set_positions(mv, Xn)
        mir.X[mv[:-3]] = Xn[:-3]
        mir.X[mv[-3:]] = Xn[-3:]
        assert_match(lm, mir, view, keyframe(rng, mir, T, lines))
        # active flips
        fl = rng.choice(mir.live(), 300, replace=False)
        v = (rng.random(len(fl)) < 0.6).astype(np.uint8)
        lm.set_active(fl, v)
        mir.active[fl] = v
        assert_match(lm, mir, view, keyframe(rng, mir, T, lines))
        # culls (never a hot landmark)
        cands = np.setdiff1d(mir.live(), hot)
        cu = rng.choice(cands, 10, replace=False)
        lm.cull(cu)
        mir.alive[cu] = False
        out = assert_match(lm, mir, view, keyframe(rng, mir, T, lines))
        assert not np.isin(out["sel"], cu).any()
    assert len(lm) == len(mir.X)
    n_obs = [len(mir.obs_d[i]) for i in hot]
    assert n_obs[0] > 32 and n_obs[1] > 64 and n_obs[2] > 128
    assert_readback(lm, mir, np.arange(len(mir.X)))


def build_map(rng, ctx, lines, n, T, **kw):
    from pl_inertial_slam_b200.localmap import LocalMap
    lm, mir = LocalMap(lines, ctx, **kw), Mirror(lines)
    X, d, r = new_landmarks(rng, T, n, lines)
    lm.insert(X, d, r)
    mir.insert(X, d, r)
    idx = rng.choice(n, n // 2)
    od, orr = oracle_flip(rng, mir.med[idx], 0.1), unit(rng, len(idx))
    lm.add_observations(idx, od, orr)
    mir.add(idx, od, orr)
    fl = rng.choice(n, n // 5, replace=False)
    lm.set_active(fl, 0)
    mir.active[fl] = 0
    return lm, mir


@pytest.mark.gpu
@pytest.mark.parametrize("lines", [False, True])
def test_edge_cases(ctx, config, lines):
    from pl_inertial_slam_b200 import drivers as D
    from pl_inertial_slam_b200.localmap import LocalMap
    Cfg, Slam = config
    rng = np.random.default_rng(SEED + 10 + lines)
    T, _, _ = make_scene(7, 1, lines)
    view = D.map_view(T, CAM, INV_W, INV_H, W, H)
    # an empty map
    lm0, mir0 = LocalMap(lines, ctx), Mirror(lines)
    kf_empty = keyframe(rng, mir0, T, lines)
    out = assert_match(lm0, mir0, view, kf_empty)
    assert len(out["sel"]) == 0
    lm, mir = build_map(rng, ctx, lines, 4000, T)
    kf = keyframe(rng, mir, T, lines)
    assert_match(lm, mir, view, kf)
    # keyframes with 0 and 1 features
    for k in (0, 1):
        px, d2, le = kf
        out = assert_match(lm, mir, view, (px[:k], d2[:k], None if le is None else le[:k]))
        assert len(out["sel"]) > 0
    # the fallback: a keyframe of unrelated descriptors leaves matchGrid below min_matches; fast matching on and off
    px, d2, le = kf
    kf_rand = (px, rng.integers(0, 256, d2.shape, dtype=np.uint8), le)
    for fast in (True, False):
        Slam.fastMatching = fast
        assert_match(lm, mir, view, kf_rand)
        assert_match(lm, mir, view, kf)
    Slam.fastMatching = True
    # best_lr 0 / 1, ratios 0.75 / 0.9
    for best_lr in (False, True):
        for ratio in (0.75, 0.9):
            Cfg.bestLRMatches, Cfg.minRatio12P, Cfg.minRatio12L = best_lr, ratio, ratio
            assert_match(lm, mir, view, kf)
            assert_match(lm, mir, view, kf_rand)
    Cfg.bestLRMatches, Cfg.minRatio12P, Cfg.minRatio12L = True, 0.9, 0.9
    # n_sel == 0: every landmark inactive
    lm.set_active(np.arange(len(mir.X)), 0)
    mir.active[:] = 0
    out = assert_match(lm, mir, view, kf)
    assert len(out["sel"]) == 0 and out["matches"] == 0


@pytest.mark.gpu
@pytest.mark.parametrize("lines", [False, True])
@pytest.mark.parametrize("n", [70_001, 200_000])
def test_large_maps(ctx, config, lines, n):
    from pl_inertial_slam_b200 import drivers as D
    rng = np.random.default_rng(SEED + n + lines)
    T, _, _ = make_scene(11, 1, lines)
    view = D.map_view(T, CAM, INV_W, INV_H, W, H)
    lm, mir = build_map(rng, ctx, lines, n, T)
    kf = keyframe(rng, mir, T, lines, n2=600 if not lines else 200)
    out = assert_match(lm, mir, view, kf)
    assert out["matches"] > 0
    px, d2, le = kf
    assert_match(lm, mir, view, (px, rng.integers(0, 256, d2.shape, dtype=np.uint8), le))   # fallback at map scale
    assert_readback(lm, mir, rng.choice(n, 2000, replace=False))


def run_short(rng_seed, ctx, lines, **kw):
    """A short fixed sequence -> (list of match outputs, final read-back)."""
    from pl_inertial_slam_b200 import drivers as D
    from pl_inertial_slam_b200.localmap import LocalMap
    rng = np.random.default_rng(rng_seed)
    T, _, _ = make_scene(13, 1, lines)
    view = D.map_view(T, CAM, INV_W, INV_H, W, H)
    lm, mir = LocalMap(lines, ctx, **kw), Mirror(lines)
    outs = []
    for step in range(6):
        X, d, r = new_landmarks(rng, T, 300, lines)
        lm.insert(X, d, r)
        mir.insert(X, d, r)
        idx = np.concatenate([rng.choice(len(mir.X), 200), np.repeat([3], 12)])
        od, orr = oracle_flip(rng, mir.med[idx], 0.1), unit(rng, len(idx))
        lm.add_observations(idx, od, orr)
        mir.add(idx, od, orr)
        mv = rng.choice(len(mir.X), 50, replace=False)
        mir.X[mv] += 0.01
        lm.set_positions(mv, mir.X[mv])
        outs.append(assert_match(lm, mir, view, keyframe(rng, mir, T, lines)))
    return outs, lm.landmarks(np.arange(len(mir.X)))


@pytest.mark.gpu
@pytest.mark.parametrize("lines", [False, True])
def test_growth_from_capacity_one(ctx, config, lines):
    a_out, a_rb = run_short(SEED + 20, ctx, lines, lm_capacity=1, obs_capacity=1)
    b_out, b_rb = run_short(SEED + 20, ctx, lines, lm_capacity=1 << 16, obs_capacity=1 << 20)
    for x, y in zip(a_out, b_out):
        for k in ("sel", "m12", "ok"):
            assert np.array_equal(x[k], y[k])
        assert x["matches"] == y["matches"]
    for k in a_rb:
        assert np.array_equal(np.asarray(a_rb[k]).view(np.uint8), np.asarray(b_rb[k]).view(np.uint8)), k


@pytest.mark.gpu
@pytest.mark.parametrize("lines", [False, True])
def test_cost_independent_of_map_size(ctx, config, lines):
    """The same calls on a map of 10 000 landmarks and on the same map plus 190 000 landmarks behind the camera: equal
    host <-> device bytes and launches per call, equal to the header's formulas."""
    from pl_inertial_slam_b200 import drivers as D
    from pl_inertial_slam_b200 import grid as G
    T, _, _ = make_scene(17, 1, lines)
    view = D.map_view(T, CAM, INV_W, INV_H, W, H)
    per, costs, n_sels = (2 if lines else 1), [], []
    for extra in (0, 190_000):
        rng = np.random.default_rng(SEED + 30)
        lm, mir = build_map(rng, ctx, lines, 10_000, T)
        if extra:
            X, d, r = new_landmarks(np.random.default_rng(5), T, extra, lines, behind=True)
            lm.insert(X, d, r)
            mir.insert(X, d, r)
        kf = keyframe(rng, mir, T, lines, n2=500 if not lines else 200)
        upd = [("insert", lambda: lm.insert(*new_landmarks(rng, T, 64, lines)[:3])),
               ("add", lambda: lm.add_observations(np.concatenate([np.arange(100), np.arange(50)]),
                                                   rng.integers(0, 256, (150, 32), dtype=np.uint8), unit(rng, 150))),
               ("pos", lambda: lm.set_positions(np.arange(500, 2500), mir.X[500:2500])),
               ("act", lambda: lm.set_active(np.arange(3000, 6000), 1)),
               ("cull", lambda: lm.cull(np.arange(9000, 9010))),
               ("match", lambda: n_sels.append(len(match_both(lm, mir, view, kf)[0]["sel"])))]
        cost = {}
        for name, fn in upd:
            h0, d0, l0 = lm.h2d_bytes, lm.d2h_bytes, ctx.launch_count
            fn()
            ctx.synchronize()
            cost[name] = (lm.h2d_bytes - h0, lm.d2h_bytes - d0, ctx.launch_count - l0)
            if name == "cull":
                mir.alive[9000:9010] = False
        costs.append(cost)
    assert n_sels[0] == n_sels[1] > 0
    assert costs[0] == costs[1]
    c = costs[0]
    xw = 3 * per
    assert c["insert"] == (64 * (56 + 8 * xw), 0, 1)
    assert c["add"] == (60 * 150 + 20 * 100, 0, 3)
    assert c["pos"] == (2000 * (4 + 8 * xw), 0, 1)
    assert c["act"] == (3000 * 5, 0, 1)
    assert c["cull"] == (40, 0, 1)
    px, d2, le = kf
    n2 = len(d2)
    if lines:
        cs, ci, _ = D.line_grid(px, INV_W, INV_H)
    else:
        cs, ci = G.csr_from_points(px[:, 0] * INV_W, px[:, 1] * INV_H)
    assert c["match"][0] == n2 * (48 + 24 * lines) + 4 * (len(cs) + len(ci))
    ns = n_sels[0]
    assert c["match"][1] in (4 + 9 * ns + 4, 4 + 4 + 9 * ns + 4)


@pytest.mark.gpu
@pytest.mark.parametrize("lines", [False, True])
def test_failed_calls_leave_the_store_unchanged(ctx, config, lines):
    from pl_inertial_slam_b200 import _lib as L
    from pl_inertial_slam_b200 import drivers as D
    rng = np.random.default_rng(SEED + 40 + lines)
    T, _, _ = make_scene(19, 1, lines)
    view = D.map_view(T, CAM, INV_W, INV_H, W, H)
    lm, mir = build_map(rng, ctx, lines, 3000, T)
    lm.cull([7, 8])
    mir.alive[[7, 8]] = False
    kf = keyframe(rng, mir, T, lines)
    ids = mir.live()
    before = assert_match(lm, mir, view, kf), lm.landmarks(ids), len(lm)
    h2d = lm.h2d_bytes
    xw = mir.xw
    bad = [lambda: lm.add_observations([1, 7], rng.integers(0, 256, (2, 32), dtype=np.uint8), unit(rng, 2)),   # culled
           lambda: lm.add_observations([1, 3000], rng.integers(0, 256, (2, 32), dtype=np.uint8), unit(rng, 2)),  # out of range
           lambda: lm.set_positions([2, -1], np.zeros((2, xw))),
           lambda: lm.set_active([8], [1]),
           lambda: lm.cull([9, 7]),                                                                                # culled again
           lambda: lm.cull([10, 11, 10]),                                                                          # twice in a call
           lambda: lm.landmarks([7])]
    for fn in bad:
        with pytest.raises(L.PlmError) as e:
            fn()
        assert e.value.status == L.PLM_E_INVALID
    # null pointers through the C entry points
    lib = L.load()
    assert lib.plm_localmap_insert(lm._h, 1, None, None, 32, None, None) == L.PLM_E_INVALID
    assert lib.plm_localmap_add_observations(lm._h, 1, None, None, 32, None) == L.PLM_E_INVALID
    assert lm.h2d_bytes == h2d                      # nothing was sent
    after = assert_match(lm, mir, view, kf), lm.landmarks(ids)
    for k in ("sel", "m12", "ok"):
        assert np.array_equal(before[0][k], after[0][k])
    assert before[0]["matches"] == after[0]["matches"]
    for k in before[1]:
        assert np.array_equal(np.asarray(before[1][k]).view(np.uint8), np.asarray(after[1][k]).view(np.uint8)), k
    assert len(lm) == before[2]
