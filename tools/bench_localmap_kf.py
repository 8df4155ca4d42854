"""Per-keyframe cost of matching one keyframe against both resident stores in one call (localmap.match_keyframe,
plm_localmap_match_kf_pl: grids built on the device) against the two-call path it replaces, at the config 4 shapes:
200 000 point landmarks x 600 keyframe points and 50 000 segment landmarks x 200 keyframe segments, one view.

    python tools/bench_localmap_kf.py --out profiles/r11_localmap_kf_b200.json

The maps and keyframes are built as tools/bench_localmap.py builds them (about three observations per landmark, 80 %
active; keyframe features are noisy projections of selected landmarks with noisy copies of their med_desc, 10 %
unrelated), except that both kinds share one camera pose.  Before anything is timed the three paths are compared (sel,
m12, ok, count of both kinds); a mismatch aborts the run.  Reported, wall time per keyframe with a context synchronise
at the end of each call (median and p90; arms (a) and (b) alternate call by call):
  (a) match_keyframe: one call for both kinds;
  (b) the host grid build (grid.csr_from_points, drivers.line_grid) + LocalMap.matchMap2KFPoints + matchMap2KFLines;
  (c) drivers.matchMap2KFPointsFull + matchMap2KFLinesFull (host arrays, the whole map uploaded per call);
plus bytes, launches and synchronisations per call of (a), and device time per call of (a) and (b) by kernel / copy from
torch.profiler's CUDA activity in a separate run.  Needs a CUDA device; the card's name, power limit and clock are read
in the same run and written next to the numbers."""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import bench_localmap as B  # noqa: E402
from pl_inertial_slam_b200 import drivers as D  # noqa: E402
from pl_inertial_slam_b200 import localmap as LM  # noqa: E402
from pl_inertial_slam_b200 import synth  # noqa: E402
from pl_inertial_slam_b200.localmap import LocalMap  # noqa: E402
from pl_inertial_slam_b200.matching import Context  # noqa: E402


def build_kind(kind, ctx, rng, T):
    """bench_localmap.build with a given pose."""
    lines = kind == "lines"
    n_map, n2 = B.SHAPES[kind]
    X = np.concatenate([rng.uniform(-4, 4, (n_map, 2)), rng.uniform(2, 12, (n_map, 1))], 1)
    if lines:
        X = np.concatenate([X, X + rng.normal(0, 0.4, (n_map, 3))], 1)
    lm = LocalMap(lines, ctx, lm_capacity=n_map, obs_capacity=8 * n_map)
    base = synth.rand_desc(rng, n_map)
    lm.insert(X, base, B.unit(rng, n_map))
    idx = rng.integers(0, n_map, 2 * n_map).astype(np.int32)
    for lo in range(0, len(idx), 100_000):
        part = idx[lo:lo + 100_000]
        lm.add_observations(part, synth.flip_bits(rng, base[part], 0.08), B.unit(rng, len(part)))
    active = (rng.random(n_map) < 0.8).astype(np.uint8)
    lm.set_active(np.flatnonzero(active == 0).astype(np.int32), 0)
    med = lm.landmarks(np.arange(n_map))["med_desc"]
    view = D.map_view(T, B.CAM, B.INV_W, B.INV_H, B.W, B.H)
    sel, _, pf = D.mapSelect(X, active, view, ctx)
    seen = rng.choice(len(sel), n2, replace=False)
    px = np.clip(pf[seen] + rng.normal(0, 0.7, (n2, pf.shape[1])), 1.0, np.tile([B.W - 2.0, B.H - 2.0], pf.shape[1] // 2))
    px = px.astype(np.float32)
    d2 = synth.flip_bits(rng, med[sel[seen]], 0.06)
    d2[: n2 // 10] = synth.rand_desc(rng, n2 // 10)
    p = px.astype(np.float64)
    if lines:
        le = np.cross(np.stack([p[:, 0], p[:, 1], np.ones(n2)], 1), np.stack([p[:, 2], p[:, 3], np.ones(n2)], 1))
        feat = le / np.hypot(le[:, 0], le[:, 1])[:, None]
    else:
        feat = p
    return dict(lm=lm, X=X, active=active, med=med, px=px, d2=d2, feat=feat)


def arm_a(P, L, view):
    return LM.match_keyframe(P["lm"], L["lm"], view, P["px"], P["d2"], P["feat"], L["px"], L["d2"], L["feat"])


def arm_b(P, L, view):
    return dict(points=P["lm"].matchMap2KFPoints(view, P["px"], P["d2"]),
                lines=L["lm"].matchMap2KFLines(view, L["px"], L["feat"], L["d2"]))


def arm_c(P, L, view, ctx):
    return dict(points=D.matchMap2KFPointsFull(P["X"], P["active"], P["med"], view, P["feat"], P["d2"], ctx),
                lines=D.matchMap2KFLinesFull(L["X"], L["active"], L["med"], view, L["px"], L["feat"], L["d2"], ctx))


def same(x, y):
    return all(np.array_equal(x[k], y[k]) for k in ("sel", "m12", "ok")) and x["matches"] == y["matches"]


def profile(fn, n):
    import torch
    from torch.profiler import ProfilerActivity, profile as prof_ctx
    with prof_ctx(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        for _ in range(n):
            fn()
        torch.cuda.synchronize()
    out = {}
    for e in prof.key_averages():
        t = getattr(e, "device_time_total", None)
        if t is None:
            t = getattr(e, "cuda_time_total", 0.0)
        if t and (e.device_type is not None and "CUDA" in str(e.device_type)):
            out[e.key[:80]] = round(float(t) / n, 2)
    out["device_total_us"] = round(sum(out.values()), 2)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=300)
    ap.add_argument("--drivers-reps", type=int, default=30)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    ctx = Context(0)
    rng = np.random.default_rng(20261023)
    T = np.concatenate([np.eye(3), rng.normal(0, 0.2, (3, 1))], 1)
    view = D.map_view(T, B.CAM, B.INV_W, B.INV_H, B.W, B.H)
    P, L = build_kind("points", ctx, rng, T), build_kind("lines", ctx, rng, T)
    res = dict(tool="bench_localmap_kf", card=B.card(), shapes={k: dict(landmarks=v[0], keyframe=v[1]) for k, v in B.SHAPES.items()})
    a, b, c = arm_a(P, L, view), arm_b(P, L, view), arm_c(P, L, view, ctx)
    for kind in ("points", "lines"):      # equality first: nothing is timed on a mismatch
        if not (same(a[kind], b[kind]) and same(a[kind], c[kind])):
            raise SystemExit(f"{kind}: match_keyframe, the two-call path and the drivers disagree -- nothing timed")
        res[kind] = dict(n_sel=int(len(a[kind]["sel"])), matches=int(a[kind]["matches"]))
    l0 = ctx.launch_count
    a = arm_a(P, L, view)
    ctx.synchronize()
    res["a_cost"] = dict(launches=int(ctx.launch_count - l0), **a["cost"])
    l0 = ctx.launch_count
    arm_b(P, L, view)
    ctx.synchronize()
    res["b_launches"] = int(ctx.launch_count - l0)
    for _ in range(30):                   # warm-up of both arms
        arm_a(P, L, view)
        arm_b(P, L, view)
    ctx.synchronize()
    ta, tb = [], []
    for _ in range(args.reps):
        for fn, acc in ((lambda: arm_a(P, L, view), ta), (lambda: arm_b(P, L, view), tb)):
            t0 = time.perf_counter()
            fn()
            ctx.synchronize()
            acc.append((time.perf_counter() - t0) * 1e3)
    res["a_match_keyframe_wall"] = B.stats(ta)
    res["b_host_grid_two_calls_wall"] = B.stats(tb)
    for _ in range(3):
        arm_c(P, L, view, ctx)
    tc = []
    for _ in range(args.drivers_reps):
        t0 = time.perf_counter()
        arm_c(P, L, view, ctx)
        ctx.synchronize()
        tc.append((time.perf_counter() - t0) * 1e3)
    res["c_drivers_wall"] = B.stats(tc)
    res["a_device_us"] = profile(lambda: arm_a(P, L, view), 30)     # profiled separately: tracing slows the host
    res["b_device_us"] = profile(lambda: arm_b(P, L, view), 30)
    res["card_after"] = B.card()
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
