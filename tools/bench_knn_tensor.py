#!/usr/bin/env python
"""A/B of the brute-force top-2 kernels on the bench shape: the integer kernel (knn2 variant 3, LOP3/POPC) against the
tensor-core kernel (variant 7, int8 tcgen05 MMA), alternating in one process.

* card name, power limit and SM clocks (nvidia-smi, read in this run);
* config 5 on one GPU: 6400 queries x 16 M rows through plm_dev_knn2 (slice kernel + merge), a 256 MiB L2 flush
  between calls, CUDA events around each call; `--rounds` rounds of `--calls` calls per kernel, alternating;
* the keys of both kernels compared on every call of the last round;
* the int8 MMA rate of the card measured in the same run (plm_measure_mma_i8_rate): 128 x 256 x 32 (the peak) and
  128 x 128 x 32 (the shape the tensor kernel issues), each alone and with concurrent shared-memory stores as the
  expansion makes them; and the integer-pipe peaks (plm_measure_int_peaks), so that the tensor kernel's MAC/s can be
  set against a measured rate;
* with a library built with PLM_BUILD_DEFINES=-DPLM_UMMA_STAMPS: the per-role cycle stamps of the tensor kernel at the
  bench shape (SM cycles per unit, and the share of it each role spent waiting), which show the role that bounds it;
* the query count at which the tensor kernel overtakes the integer one (2 M rows, n1 = 256 ... 4096).

    python tools/bench_knn_tensor.py --out profiles/r4_knn_tensor_b200.json
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card_info() -> dict:
    q = "name,power.limit,clocks.sm,clocks.max.sm,driver_version"
    try:
        out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        return dict(zip(q.split(","), [x.strip() for x in out.split(",")]))
    except (OSError, subprocess.SubprocessError) as e:
        return {"error": repr(e)}


def role_stamps(lib, call) -> dict:
    """Per-role SM cycles of knn2_umma_kernel from a PLM_UMMA_STAMPS build: one call at the bench shape, then per role
    the median over CTAs of cycles per unit and of the share of its time spent in mbarrier waits."""
    import ctypes as C
    call()
    buf = (C.c_longlong * (160 * 4 * 3))()
    assert lib.plm_debug_umma_stamps(buf) == 0
    a = np.frombuffer(buf, dtype=np.int64).reshape(160, 4, 3)
    a = a[a[:, 0, 2] > 0]
    out = {}
    for r, name in enumerate(("readout", "expander", "producer", "mma")):
        total, waited, units = a[:, r, 0].astype(float), a[:, r, 1].astype(float), a[:, r, 2].astype(float)
        out[name] = {"cycles_per_unit_median": float(np.median(total / units)),
                     "wait_share_median": float(np.median(waited / total)), "units_median": float(np.median(units))}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=4)
    ap.add_argument("--calls", type=int, default=3, help="timed calls per kernel per round")
    ap.add_argument("--n-kf", type=int, default=20000)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch
    import bench
    from pl_inertial_slam_b200 import _lib
    from pl_inertial_slam_b200.database import DeviceOps

    lib = _lib.load()
    if not torch.cuda.is_available():
        raise SystemExit("bench_knn_tensor.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    ops = DeviceOps(0)
    n_rows = args.n_kf * bench.PER_KF
    db = torch.from_numpy(bench.gen_rows(0, args.n_kf)).to(dev)
    q = torch.from_numpy(bench.gen_queries(0, 8, args.n_kf)).to(dev)
    n_q = q.shape[0]
    flush = torch.empty(bench.L2_FLUSH_BYTES, dtype=torch.uint8, device=dev)
    arms = {"int_t13": 3, "tensor_umma": 7}

    def run(v, queries, rows, calls):
        assert lib.plm_set_option(b"knn_variant", v) == 0
        ops.knn2(queries, rows)  # warm-up (module load, attributes, scratch)
        ms, out = [], None
        for i in range(calls):
            flush.fill_(i & 0xFF)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            out = ops.knn2(queries, rows)
            e1.record()
            torch.cuda.synchronize()
            ms.append(e0.elapsed_time(e1))
        return ms, out

    card_before = card_info()
    mma_tops = ops.ctx.measure_mma_i8_peak()
    mma_rates = {f"n{n}{'_with_stores' if sts else ''}": ops.ctx.measure_mma_i8_rate(n, sts)
                 for n in (256, 128) for sts in (False, True)}
    popc_gops, lop3_gops = ops.ctx.measure_int_peaks()
    times = {k: [] for k in arms}
    equal = None
    for r in range(args.rounds):
        outs = {}
        for name, v in (arms.items() if r % 2 == 0 else reversed(list(arms.items()))):
            ms, outs[name] = run(v, q, db, args.calls)
            times[name] += ms
        equal = bool(torch.equal(outs["int_t13"], outs["tensor_umma"]))
    card_after = card_info()

    pairs = float(n_q) * n_rows
    macs = pairs * 256
    res = {}
    for name, ms in times.items():
        a = np.array(ms)
        res[name] = {"ms_per_call": {"median": float(np.median(a)), "min": float(a.min()), "max": float(a.max()),
                                     "spread_pct": float((a.max() - a.min()) / np.median(a) * 100), "n": len(ms)},
                     "pairs_per_s": pairs / (np.median(a) * 1e-3)}
    t_med = res["tensor_umma"]["ms_per_call"]["median"] * 1e-3
    res["tensor_umma"]["int8_tops_achieved"] = 2 * macs / t_med * 1e-12
    res["tensor_umma"]["share_of_measured_mma_peak"] = 2 * macs / t_med * 1e-12 / mma_tops
    res["speedup_median"] = res["int_t13"]["ms_per_call"]["median"] / res["tensor_umma"]["ms_per_call"]["median"]

    # crossover in the number of queries (automatic mode needs >= 65 536 rows; 2 M rows here)
    sweep = []
    rows2 = db[: 2_000_000]
    for n1 in (256, 512, 1024, 2048, 4096):
        row = {"n1": n1, "n2": int(rows2.shape[0])}
        for name, v in arms.items():
            ms, _ = run(v, q[:n1], rows2, 3)
            row[name + "_ms"] = float(np.median(ms))
        sweep.append(row)
    stamps = role_stamps(lib, lambda: run(7, q, db, 1)) if hasattr(lib, "plm_debug_umma_stamps") else None
    lib.plm_set_option(b"knn_variant", -1)

    out = {"card_before": card_before, "card_after": card_after,
           "shape": {"queries": n_q, "db_rows": n_rows, "K_bits": 256, "pairs_per_call": pairs, "macs_per_call": macs},
           "call": "plm_dev_knn2 (slice kernel + merge kernel), L2 flushed (256 MiB write) before each call",
           "measured_peaks": {"int8_mma_tops": mma_tops, "popc_gops": popc_gops, "lop3_gops": lop3_gops},
           "int8_mma_tops_by_shape": mma_rates,
           "tensor_share_of_n128_rate": res["tensor_umma"]["int8_tops_achieved"] / mma_rates["n128"],
           "tensor_role_stamps": stamps,
           "keys_equal_last_round": equal, "arms": res, "n1_crossover_2m_rows": sweep}
    text = json.dumps(out, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
