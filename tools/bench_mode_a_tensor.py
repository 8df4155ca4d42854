#!/usr/bin/env python
"""A/B of loop-closure "Mode A" batches: the integer list kernels (option batch_umma = 0) against the tensor-core pairs
kernel (K1c, batch_umma = 1), alternating in one process.

Each shape is one query keyframe of n1 rows against n_kf keyframes of kf_rows rows resident on the device, the batch
KeyframeDB.match_all builds (plm_batch_set_match_dev, every job sharing the query slot).  Per arm a MatchBatch is
prepared once; the timed unit is one plm_batch_run (kernel, merge, mutual check) between CUDA events on the context's
stream, `--reps` runs per round, `--rounds` rounds with the arms alternating.  Reported per shape:
* device ms per run (median, spread), unique pairs/s (n1 x rows) and reference-equivalent pairs/s (x 2 with best_lr:
  StVO::match scans both directions);
* the int8 TOPS the tensor arm issues (256-row query groups x 128-row units x 256 bits) against
  plm_measure_mma_i8_rate(n = 128) measured in the same run;
* whether both arms gave identical counts and match vectors (a mismatch fails the run).
Also: card name, power limit and SM clock (nvidia-smi query, read in this run); the crossover grid over n1 and the
keyframe count, for points (800-row keyframes) and lines (200-row keyframes); with a library built with
PLM_BUILD_DEFINES=-DPLM_UMMA_STAMPS, the per-role cycle stamps of the tensor kernel at the bench-extras shape.

    python tools/bench_mode_a_tensor.py --out profiles/r6_mode_a_tensor_b200.json
"""
from __future__ import annotations

import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from bench_knn_tensor import card_info, role_stamps  # noqa: E402


def make_db(torch, dev, n_kf, kf_rows, nq, seed):
    """Random rows on the device; half of every keyframe are noisy copies of query rows (bits flip with p = 1/8), so
    that both ratio tests and the mutual check accept a realistic share."""
    g = torch.Generator(device=dev).manual_seed(seed)
    q = torch.randint(0, 256, (nq, 32), dtype=torch.uint8, device=dev, generator=g)
    rows = torch.randint(0, 256, (n_kf, kf_rows, 32), dtype=torch.uint8, device=dev, generator=g)
    k = kf_rows // 2
    src = q[torch.randint(0, nq, (n_kf, k), device=dev, generator=g)]
    noise = torch.randint(0, 256, src.shape, dtype=torch.uint8, device=dev, generator=g)
    for _ in range(2):
        noise &= torch.randint(0, 256, src.shape, dtype=torch.uint8, device=dev, generator=g)
    rows[:, :k] = src ^ noise
    return q, rows.reshape(n_kf * kf_rows, 32)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=4)
    ap.add_argument("--reps", type=int, default=20, help="timed runs per arm per round (large shapes: fewer)")
    ap.add_argument("--out", default=None)
    ap.add_argument("--stamps-only", action="store_true", help="only the role stamps (needs a PLM_UMMA_STAMPS build)")
    args = ap.parse_args()

    import torch
    from pl_inertial_slam_b200 import _lib as L
    from pl_inertial_slam_b200.matching import Context
    from pl_inertial_slam_b200.replay import MatchBatch

    if not torch.cuda.is_available():
        raise SystemExit("bench_mode_a_tensor.py needs a CUDA device")
    lib = L.load()
    dev = torch.device("cuda", 0)
    ctx = Context(0)
    stream = torch.cuda.Stream(dev)
    ctx.set_stream(stream.cuda_stream)
    sms = torch.cuda.get_device_properties(0).multi_processor_count

    def prepare(v, arena, n_rows, nq, n_kf, kf_rows, best_lr):
        assert lib.plm_set_option(b"batch_umma", v) == 0
        jobs = np.zeros(n_kf, L.PAIR_JOB_DTYPE)
        jobs["off1"], jobs["n1"] = n_rows, nq
        jobs["off2"], jobs["n2"] = np.arange(n_kf) * kf_rows, kf_rows
        jobs["off_m"] = np.arange(n_kf, dtype=np.int64) * nq
        b = MatchBatch(ctx)
        b.set_match_dev(arena, jobs, 0.9, best_lr, n_kf * nq)
        lib.plm_set_option(b"batch_umma", -1)
        return b

    def timed(b, reps):
        ms = []
        with torch.cuda.stream(stream):
            for _ in range(reps):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream)
                b.run()
                e1.record(stream)
                e1.synchronize()
                ms.append(e0.elapsed_time(e1))
        return ms

    def shape(nq, n_kf, kf_rows, best_lr=True, rounds=None, reps=None, seed=1):
        rounds, reps = rounds or args.rounds, reps or args.reps
        q, rows = make_db(torch, dev, n_kf, kf_rows, nq, seed)
        n_rows = rows.shape[0]
        arena = torch.cat([rows, q]).contiguous()
        torch.cuda.synchronize()
        arms = {"int_list": prepare(0, arena, n_rows, nq, n_kf, kf_rows, best_lr),
                "tensor_pairs": prepare(1, arena, n_rows, nq, n_kf, kf_rows, best_lr)}
        times = {k: [] for k in arms}
        outs = {}
        for k, b in arms.items():  # warm-up
            timed(b, 2)
        for r in range(rounds):
            for k in (list(arms) if r % 2 == 0 else list(reversed(list(arms)))):
                times[k] += timed(arms[k], reps)
        for k, b in arms.items():
            outs[k] = b.fetch()
            b.close()
        same = bool(np.array_equal(outs["int_list"][0], outs["tensor_pairs"][0]) and
                    np.array_equal(outs["int_list"][1], outs["tensor_pairs"][1]))
        pairs = float(nq) * n_rows
        groups, units = -(-nq // 256), n_kf * -(-kf_rows // 128)
        mma_ops = 2.0 * groups * 256 * units * 128 * 256
        res = {"n1": nq, "n_kf": n_kf, "kf_rows": kf_rows, "best_lr": best_lr, "db_mb": n_rows * 32 / 2**20,
               "identical_m12_and_counts": same, "accepted_pairs": int(np.maximum(outs["tensor_pairs"][1], 0).sum())}
        for k, ms in times.items():
            a = np.array(ms)
            med = float(np.median(a))
            res[k] = {"ms_median": med, "ms_min": float(a.min()), "spread_pct": float((a.max() - a.min()) / med * 100),
                      "n": len(ms), "unique_pairs_per_s": pairs / (med * 1e-3),
                      "reference_equiv_pairs_per_s": pairs * (2 if best_lr else 1) / (med * 1e-3)}
        t = res["tensor_pairs"]["ms_median"] * 1e-3
        res["tensor_pairs"]["int8_tops_issued"] = mma_ops / t * 1e-12
        res["tensor_pairs"]["share_of_mma_rate_n128"] = mma_ops / t * 1e-12 / mma_n128
        res["speedup"] = res["int_list"]["ms_median"] / res["tensor_pairs"]["ms_median"]
        del arena, rows, q
        torch.cuda.empty_cache()
        if not same:
            raise SystemExit(f"arms disagree at n1={nq} n_kf={n_kf} kf_rows={kf_rows} best_lr={best_lr}")
        print(json.dumps({k: res[k] for k in ("n1", "n_kf", "kf_rows", "best_lr", "speedup")}), flush=True)
        return res

    if args.stamps_only:
        if not hasattr(lib, "plm_debug_umma_stamps"):
            raise SystemExit("--stamps-only needs a library built with -DPLM_UMMA_STAMPS")
        q, rows = make_db(torch, dev, 2000, 800, 800, 1)
        arena = torch.cat([rows, q]).contiguous()
        b = prepare(1, arena, rows.shape[0], 800, 2000, 800, True)
        timed(b, 3)
        st = role_stamps(lib, lambda: timed(b, 1))
        out = {"card": card_info(), "shape": "800 x 2000 x 800, best_lr", "role_stamps": st}
        print(json.dumps(out, indent=1))
        if args.out:
            with open(args.out, "w") as f:
                json.dump(out, f, indent=1)
        return

    card_before = card_info()
    mma_n128 = ctx.measure_mma_i8_rate(128, False)
    results = {
        # bench-extras shape (extras.loop_closure_per_pair): the 51 MB database stays in the 126 MB L2 between runs
        "points_800_x_2000x800": shape(800, 2000, 800),
        "points_800_x_2000x800_no_best_lr": shape(800, 2000, 800, best_lr=False),
        # 512 MB: does not fit L2
        "points_800_x_20000x800": shape(800, 20000, 800, rounds=3, reps=5),
        "lines_200_x_2000x200": shape(200, 2000, 200),
    }
    grid = []
    for kf_rows in (800, 200):
        for nq in (16, 32, 64, 128, 256):
            for n_kf in (1, 3, 10, 30, 100, 300):
                r = shape(nq, n_kf, kf_rows, rounds=2, reps=10, seed=nq * 1000 + n_kf)
                grid.append({k: r[k] for k in ("n1", "n_kf", "kf_rows", "speedup")} |
                            {"int_ms": r["int_list"]["ms_median"], "tensor_ms": r["tensor_pairs"]["ms_median"],
                             "live_rows": n_kf * kf_rows})
    card_after = card_info()
    out = {"card_before": card_before, "card_after": card_after, "sm_count": sms,
           "mma_i8_rate_n128_tops": mma_n128, "shapes": results, "crossover_grid": grid}
    print(json.dumps(out, indent=1))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
