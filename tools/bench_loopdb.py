"""Per-insert cost of the loop-closure keyframe database (bow.LoopClosureDB, plm_loopdb_*) against the host-repack path
(bow.BowConfusion), and of its candidate matching against drivers.loopClosureMatch.

    python tools/bench_loopdb.py --out profiles/r3_loopdb.json

Keyframes: 800 point and 200 line descriptors each (noisy copies of vocabulary leaves; a pool of --pool distinct
keyframes, cycled), point vocabulary k = 10 / L = 5 (as bench_extras.bow_scoring), line vocabulary k = 8 / L = 4.
LoopClosureDB: --n-kf inserts in modes P and PL; wall time per insert (the call ends in a device synchronise) as median
and p90 over windows of 100 inserts around database sizes 100 / 2000 / n-kf, launches and bytes per insert, and the
device-time split (transform, score, blend, copies) from torch.profiler's CUDA activity over 50 further inserts at
the largest size.  BowConfusion: map_keyframes pre-filled with vectors to 100 / 2000 / n-kf keyframes, single inserts
timed.  Matching: match_candidates for 1 / 10 / 100 candidates against one drivers.loopClosureMatch per candidate.
Needs a CUDA device; the card's name and power limit are read in the same run."""
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

from pl_inertial_slam_b200 import bow as B  # noqa: E402
from pl_inertial_slam_b200 import drivers as D  # noqa: E402
from pl_inertial_slam_b200 import synth  # noqa: E402
from pl_inertial_slam_b200.matching import Context  # noqa: E402

N_P, N_L = 800, 200


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        name, power, clock = [x.strip() for x in out[0].split(",")]
        return dict(name=name, power_limit=power, max_sm_clock=clock)
    except Exception as e:  # the numbers are still reported, marked without their card
        return dict(error=str(e))


def stats(ms):
    a = np.asarray(ms, np.float64)
    return dict(n=len(a), median_ms=float(np.median(a)), p90_ms=float(np.percentile(a, 90)))


def make_pool(fp, fl, n_pool, seed):
    rng = np.random.default_rng(seed)
    pts = synth.vocabulary_features(seed + 1, fp, n_pool * N_P, flip_p=0.05).reshape(n_pool, N_P, 32)
    lns = synth.vocabulary_features(seed + 2, fl, n_pool * N_L, flip_p=0.05).reshape(n_pool, N_L, 32)
    xy = rng.uniform(0, 700, (n_pool, N_P, 2))
    mid = rng.uniform(0, 450, (n_pool, N_L, 2))
    return pts, lns, xy, mid


def kf_of(pool, i):
    pts, lns, xy, mid = pool
    k = i % len(pts)
    return B.KeyFrameBow(i, pts[k], lns[k], xy[k], mid[k])


def profile_split(db, mode, pool, first, n):
    """Device time per insert by kernel / copy, from torch.profiler's CUDA activity (microseconds)."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        for i in range(first, first + n):
            getattr(db, "insertKFBowVector" + mode)(kf_of(pool, i))
        torch.cuda.synchronize()
    groups = {"transform": "bow_transform_slots_kernel", "score": "bow_score_row_kernel", "blend": "bow_blend_kernel",
              "h2d": "Memcpy HtoD", "d2h": "Memcpy DtoH"}
    out = {k: 0.0 for k in groups}
    for e in prof.key_averages():
        t = getattr(e, "device_time_total", None)
        if t is None:
            t = getattr(e, "cuda_time_total", 0.0)
        for k, pat in groups.items():
            if pat in e.key:
                out[k] += float(t) / n
    out["device_total"] = sum(out.values())
    return out


def bench_db(mode, vp, vl, ctx, pool, n_kf, windows):
    db = B.LoopClosureDB(vp, vl, mode, capacity=1024)
    ins = getattr(db, "insertKFBowVector" + mode)
    times = np.zeros(n_kf)
    l0, h0, d0 = ctx.launch_count, db.h2d_bytes, db.d2h_bytes
    last = {}
    for i in range(n_kf):
        kf = kf_of(pool, i)
        if i == n_kf - 1:
            l0, h0, d0 = ctx.launch_count, db.h2d_bytes, db.d2h_bytes
        t0 = time.perf_counter()
        ins(kf)
        times[i] = (time.perf_counter() - t0) * 1e3
        if i == n_kf - 1:
            last = dict(launches=ctx.launch_count - l0, h2d_bytes=db.h2d_bytes - h0, d2h_bytes=db.d2h_bytes - d0)
    res = dict(windows={str(c): stats(times[max(0, c - 50): c + 50]) for c in windows},
               per_insert_at_largest=last, total_inserts=n_kf)
    res["device_split_us_at_largest"] = profile_split(db, mode, pool, n_kf, 50)
    return db, res


def bench_confusion(mode, vp, vl, ctx, pool, sizes):
    pts, lns, _, _ = pool
    start_p = np.arange(0, (len(pts) + 1) * N_P, N_P, dtype=np.int32)
    start_l = np.arange(0, (len(lns) + 1) * N_L, N_L, dtype=np.int32)
    vec_p = vp.transform_batch(pts.reshape(-1, 32), start_p)
    vec_l = vl.transform_batch(lns.reshape(-1, 32), start_l)
    out = {}
    for n in sizes:
        reps = 50 if n <= 200 else (20 if n <= 4000 else 5)
        conf = B.BowConfusion(vp, vl, ctx)
        conf.conf_matrix = np.zeros((n + reps + 1, n + reps + 1))     # pre-sized: _grow copies nothing in the window
        for i in range(n):
            kf = kf_of(pool, i)
            kf.descDBoW_P, kf.descDBoW_L = vec_p[i % len(pts)], vec_l[i % len(lns)]
            conf.map_keyframes.append(kf)
        ins = getattr(conf, "insertKFBowVector" + mode)
        ms = []
        for r in range(reps + 1):
            kf = kf_of(pool, n + r)
            t0 = time.perf_counter()
            ins(kf)
            ms.append((time.perf_counter() - t0) * 1e3)
        out[str(n)] = stats(ms[1:])
        del conf
    return out


def bench_match(db, pool, n_kf, counts, reps=20):
    pts, lns, _, _ = pool
    out = {}
    rng = np.random.default_rng(7)
    kf0 = n_kf - 1
    for n in counts:
        cands = [int(c) for c in rng.choice(n_kf - 1, n, replace=False)]
        db.match_candidates(kf0, cands)
        t_db = []
        for _ in range(reps):
            t0 = time.perf_counter()
            db.match_candidates(kf0, cands)
            t_db.append((time.perf_counter() - t0) * 1e3)
        k0 = kf0 % len(pts)
        t_ref = []
        for _ in range(max(2, reps // max(1, n // 10))):
            t0 = time.perf_counter()
            for c in cands:
                k1 = c % len(pts)
                D.loopClosureMatch(pts[k0], pts[k1], lns[k0], lns[k1])
            t_ref.append((time.perf_counter() - t0) * 1e3)
        out[str(n)] = dict(loopdb=stats(t_db), loop_closure_match_per_candidate=stats(t_ref))
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--n-kf", type=int, default=20_000)
    ap.add_argument("--pool", type=int, default=2000)
    ap.add_argument("--out", default=None, help="JSON file (default: stdout only)")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_loopdb needs a CUDA device")
    n_kf = args.n_kf
    windows = sorted({100, 2000, n_kf - 50} if n_kf > 2100 else {100, n_kf - 50})
    ctx = Context(0)
    fp = synth.make_vocabulary(synth.SEED0 + 42, k=10, L=5, ragged=0.02)
    fl = synth.make_vocabulary(synth.SEED0 + 44, k=8, L=4, ragged=0.02)
    vp, vl = B.Vocabulary.from_flat(fp, ctx), B.Vocabulary.from_flat(fl, ctx)
    pool = make_pool(fp, fl, args.pool, synth.SEED0 + 45)
    res = dict(card=card(), torch=torch.__version__, n_kf=n_kf, pool=args.pool, points_per_kf=N_P, lines_per_kf=N_L,
               words_p=vp.size(), words_l=vl.size(), loopdb={}, bow_confusion={})
    sizes = [100, 2000, n_kf] if n_kf > 2100 else [100, n_kf]
    for mode in ("P", "PL"):
        db, r = bench_db(mode, vp, vl, ctx, pool, n_kf, windows)
        res["loopdb"][mode] = r
        if mode == "P":
            res["match"] = bench_match(db, pool, n_kf, [1, 10, 100])
        db.close()
        del db
        res["bow_confusion"][mode] = bench_confusion(mode, vp, vl, ctx, pool, sizes)
        print(json.dumps({mode: dict(loopdb=r, bow_confusion=res["bow_confusion"][mode])}), flush=True)
    res["card_after"] = card()
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
