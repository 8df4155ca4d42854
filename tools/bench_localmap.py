"""Per-keyframe cost of the resident local map (localmap.LocalMap, plm_localmap_*) against the host-array drivers
(drivers.matchMap2KFPointsFull / LinesFull, which upload the whole map on every call), at the config 4 shapes:
200 000 point landmarks x 600 keyframe points and 50 000 segment landmarks x 200 keyframe lines.

    python tools/bench_localmap.py --out profiles/r9_localmap_b200.json

Map: landmarks in front of the camera (80 % active), about three observations each; keyframe features are noisy
projections of selected landmarks with noisy copies of their med_desc (10 % unrelated).  Before anything is timed, one
keyframe of each kind is matched both ways and compared (sel, m12, ok, count); a mismatch aborts the run.  Reported:
  * match: wall time per call (each call ends in a device synchronise), median and p90, for LocalMap.matchMap2KF* and
    for the drivers on the same map and keyframe; launches and host <-> device bytes per LocalMap call;
  * device time per LocalMap call by kernel / copy, from torch.profiler's CUDA activity in a separate run;
  * the per-keyframe updates: 600 new observations, 20 000 moved landmarks, 3 000 active flips -- wall time per call
    followed by a context synchronise, launches and bytes.
Needs a CUDA device; the card's name and power limit are read in the same run and written next to the numbers."""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from pl_inertial_slam_b200 import drivers as D  # noqa: E402
from pl_inertial_slam_b200 import synth  # noqa: E402
from pl_inertial_slam_b200.localmap import LocalMap  # noqa: E402
from pl_inertial_slam_b200.matching import Context  # noqa: E402

W, H = 752, 480
CAM = (435.2, 435.2, 367.4, 252.2)
INV_W, INV_H = 64.0 / W, 48.0 / H
SHAPES = {"points": (200_000, 600), "lines": (50_000, 200)}


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        name, power, clock = [x.strip() for x in out[0].split(",")]
        return dict(name=name, power_limit=power, max_sm_clock=clock)
    except Exception as e:  # the numbers are still reported, marked without their card
        return dict(error=str(e))


def stats(ms):
    a = np.asarray(ms, np.float64)
    return dict(n=len(a), median_ms=float(np.median(a)), p90_ms=float(np.percentile(a, 90)))


def scene(rng, n, lines):
    T = np.concatenate([np.eye(3), rng.normal(0, 0.2, (3, 1))], 1)
    X = np.concatenate([rng.uniform(-4, 4, (n, 2)), rng.uniform(2, 12, (n, 1))], 1)
    if lines:
        X = np.concatenate([X, X + rng.normal(0, 0.4, (n, 3))], 1)
    return T, X


def unit(rng, n):
    v = rng.normal(0, 1, (n, 3))
    return v / np.linalg.norm(v, axis=1, keepdims=True)


def build(kind, ctx, seed):
    lines = kind == "lines"
    n_map, n2 = SHAPES[kind]
    rng = np.random.default_rng(seed)
    T, X = scene(rng, n_map, lines)
    lm = LocalMap(lines, ctx, lm_capacity=n_map, obs_capacity=8 * n_map)
    base = synth.rand_desc(rng, n_map)
    lm.insert(X, base, unit(rng, n_map))
    idx = rng.integers(0, n_map, 2 * n_map).astype(np.int32)
    for lo in range(0, len(idx), 100_000):
        part = idx[lo:lo + 100_000]
        lm.add_observations(part, synth.flip_bits(rng, base[part], 0.08), unit(rng, len(part)))
    active = (rng.random(n_map) < 0.8).astype(np.uint8)
    off = np.flatnonzero(active == 0).astype(np.int32)
    lm.set_active(off, 0)
    med = lm.landmarks(np.arange(n_map))["med_desc"]
    view = D.map_view(T, CAM, INV_W, INV_H, W, H)
    sel, _, pf = D.mapSelect(X, active, view, ctx)
    seen = rng.choice(len(sel), n2, replace=False)
    px = np.clip(pf[seen] + rng.normal(0, 0.7, (n2, pf.shape[1])), 1.0, np.tile([W - 2.0, H - 2.0], pf.shape[1] // 2))
    d2 = synth.flip_bits(rng, med[sel[seen]], 0.06)
    d2[: n2 // 10] = synth.rand_desc(rng, n2 // 10)
    kf = dict(px=px, d2=d2)
    if lines:
        px = px.astype(np.float32)
        p = px.astype(np.float64)
        le = np.cross(np.stack([p[:, 0], p[:, 1], np.ones(n2)], 1), np.stack([p[:, 2], p[:, 3], np.ones(n2)], 1))
        kf = dict(px=px, d2=d2, le=le / np.hypot(le[:, 0], le[:, 1])[:, None])
    return dict(lm=lm, X=X, active=active, med=med, view=view, kf=kf, lines=lines, rng=rng, n_map=n_map)


def call_store(m):
    kf = m["kf"]
    if m["lines"]:
        return m["lm"].matchMap2KFLines(m["view"], kf["px"], kf["le"], kf["d2"])
    return m["lm"].matchMap2KFPoints(m["view"], kf["px"], kf["d2"])


def call_drivers(m, ctx):
    kf = m["kf"]
    if m["lines"]:
        return D.matchMap2KFLinesFull(m["X"], m["active"], m["med"], m["view"], kf["px"], kf["le"], kf["d2"], ctx)
    return D.matchMap2KFPointsFull(m["X"], m["active"], m["med"], m["view"], kf["px"], kf["d2"], ctx)


def check(m, ctx, kind):
    a, b = call_store(m), call_drivers(m, ctx)
    same = all(np.array_equal(a[k], b[k]) for k in ("sel", "m12", "ok")) and a["matches"] == b["matches"]
    if not same:
        raise SystemExit(f"{kind}: LocalMap and drivers.matchMap2KF*Full disagree -- nothing timed")
    return dict(n_sel=int(len(a["sel"])), matches=int(a["matches"]))


def timed(fn, reps, warm, sync=None):
    for _ in range(warm):
        fn()
    if sync:
        sync()
    ms = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        if sync:
            sync()
        ms.append((time.perf_counter() - t0) * 1e3)
    return stats(ms)


def per_call(m, ctx, fn):
    lm = m["lm"]
    l0, h0, d0 = ctx.launch_count, lm.h2d_bytes, lm.d2h_bytes
    fn()
    ctx.synchronize()
    return dict(launches=int(ctx.launch_count - l0), h2d_bytes=int(lm.h2d_bytes - h0), d2h_bytes=int(lm.d2h_bytes - d0))


def profile_split(m, ctx, n):
    """Device time per LocalMap call by kernel / copy (microseconds), torch.profiler's CUDA activity."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        for _ in range(n):
            call_store(m)
        torch.cuda.synchronize()
    out = {}
    for e in prof.key_averages():
        t = getattr(e, "device_time_total", None)
        if t is None:
            t = getattr(e, "cuda_time_total", 0.0)
        if t and (e.device_type is not None and "CUDA" in str(e.device_type)):
            out[e.key[:80]] = round(float(t) / n, 2)
    out["device_total_us"] = round(sum(v for k, v in out.items()), 2)
    return out


def updates(m, ctx, reps):
    lm, rng, n_map = m["lm"], m["rng"], m["n_map"]
    live = np.arange(n_map, dtype=np.int32)
    obs_idx = rng.integers(0, n_map, (reps, 600)).astype(np.int32)
    obs_d = synth.rand_desc(rng, 600)
    obs_r = unit(rng, 600)
    mv = [np.sort(rng.choice(live, 20_000, replace=False)).astype(np.int32) for _ in range(4)]
    X = m["X"]
    fl = [rng.choice(live, 3000, replace=False).astype(np.int32) for _ in range(4)]
    it = iter(range(10 ** 9))
    fns = {"add_observations_600": lambda: lm.add_observations(obs_idx[next(it) % reps], obs_d, obs_r),
           "set_positions_20000": lambda: lm.set_positions(mv[next(it) % 4], X[mv[0]]),
           "set_active_3000": lambda: lm.set_active(fl[next(it) % 4], m["active"][fl[0]])}
    out = {}
    for name, fn in fns.items():
        out[name] = dict(wall=timed(fn, reps, 5, ctx.synchronize), **per_call(m, ctx, fn))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=200)
    ap.add_argument("--drivers-reps", type=int, default=30)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    ctx = Context(0)
    res = dict(tool="bench_localmap", card=card(), shapes={k: dict(landmarks=v[0], keyframe=v[1]) for k, v in SHAPES.items()})
    maps = {kind: build(kind, ctx, 20261022 + i) for i, kind in enumerate(SHAPES)}
    for kind, m in maps.items():      # equality first: nothing is timed on a mismatch
        res.setdefault(kind, {})["check"] = check(m, ctx, kind)
    for kind, m in maps.items():
        r = res[kind]
        r["match_wall"] = timed(lambda: call_store(m), args.reps, 20)
        r["drivers_wall"] = timed(lambda: call_drivers(m, ctx), args.drivers_reps, 3)
        r["match_cost"] = per_call(m, ctx, lambda: call_store(m))
        r["updates"] = updates(m, ctx, args.reps)
    for kind, m in maps.items():      # profiled separately: tracing slows the host
        res[kind]["match_device_us"] = profile_split(m, ctx, 20)
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
