#!/usr/bin/env python
"""Benchmark of the descriptor-matching hot path (BASELINE.json: descriptor-pairs/s vs the POPC/HBM
roofline).

Workload (config 5 of BASELINE.json, the one the metric is quoted on): loop-closure all-pairs
keyframe matching.  The keyframe database is 20 000 keyframes x 800 descriptors = 16 M rows of 256
bits (512 MB); it fits one GPU, so N GPUs share the SAME database, row-sharded (strong scaling).
A step matches a batch of --kf-batch query keyframes (x 800 descriptors) against the whole database:
local brute-force top-2 kernel -> all_gather of the packed per-query top-2 (NCCL) -> lexicographic
merge kernel -> matchNNR acceptance.  pairs/step = kf_batch * 800 * 16 M (unique pairs).

`value`      device time of the step with the queries already in HBM (CUDA events, max over ranks)
`e2e`        the same step through the public API with the query batch in pinned HOST memory and the
             match vector + count read back to the host (H2D and D2H inside the timed region)
`roofline`   the brute-force slice kernel alone (timed per launch with CUDA events on the launching
             stream inside the library) against the integer-pipe peak MEASURED in this run
`cpu_baseline` the reference's own matchNNR (matching.cpp compiled unmodified, oracle/_ref) on this
             box's host cores, on a bounded sample of the same workload

`--impl reference` runs only the CPU arm (rank 0) and prints the same JSON shape.
`--dump-outputs DIR` writes the match vector and count of the last timed step (rank 0) as DIR/m12.npy and
DIR/count.npy, so that two builds can be compared output for output on the same seeded inputs.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "descriptor_pairs_per_s"
UNIT = "pairs/s"
N_KF, PER_KF = 20000, 800
POPC_PER_PAIR = 8                 # SURVEY.md 8d: one pair = 8 POPC.32 + 8 LOP(xor) + 7 adds
# instructions per pair on the two integer pipes, counted from the SASS main loop of knn2_slice_kernel<128, V>
# (cuobjdump of the shipped library, DESIGN.md 3): ALU pipe = LOP3 + VIMNMX(3), XU pipe = POPC
ALU_INSTR_PER_PAIR = {"t13": 13.625, "csa4": 16.75, "csa5": 22.0, "popc8": 16.0}
POPC_ISSUED_PER_PAIR = {"t13": 4, "csa4": 4, "csa5": 5, "popc8": 8}
DEFAULT_VARIANT = "t13"
L2_FLUSH_BYTES = 256 << 20


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--kf-batch", type=int, default=8, help="query keyframes per step")
    ap.add_argument("--n-kf", type=int, default=N_KF, help="keyframes in the database")
    ap.add_argument("--nnr", type=float, default=0.9)
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="budget of the CPU baseline sample")
    ap.add_argument("--exchange", default="auto", choices=["auto", "peer", "nccl"],
                    help="multi-GPU top-2 merge: the library's peer-memory kernel (auto falls back to NCCL) or NCCL all_gather")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the per-frame / replay side metrics")
    ap.add_argument("--no-verify", action="store_true", help="skip the untimed verification step / multi-GPU check")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step returned (match vector and accepted "
                         "count, float64) as DIR/<name>.npy; the inputs depend only on the arguments")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs applies to the GPU path (--impl b200): the reference arm sizes its sample by timing")
    return args


# ------------------------------------------------------------------------------------------------
# synthetic data: deterministic in the keyframe index, independent of the number of ranks
def gen_rows(kf_lo: int, kf_hi: int) -> np.ndarray:
    """Descriptor rows of keyframes [kf_lo, kf_hi): 800 random 256-bit rows per keyframe, generated in
    blocks of 250 keyframes with a block-indexed seed."""
    from pl_inertial_slam_b200 import synth
    blk = 250
    out = np.empty(((kf_hi - kf_lo) * PER_KF, 32), np.uint8)
    pos = 0
    b = kf_lo // blk
    while b * blk < kf_hi:
        rng = np.random.default_rng(synth.SEED0 + 5 + 1000 * b)
        rows = rng.integers(0, 256, size=(blk * PER_KF, 32), dtype=np.uint8)
        lo, hi = max(kf_lo, b * blk), min(kf_hi, (b + 1) * blk)
        n = (hi - lo) * PER_KF
        out[pos:pos + n] = rows[(lo - b * blk) * PER_KF:(hi - b * blk) * PER_KF]
        pos += n
        b += 1
    return out


def gen_queries(step: int, kf_batch: int, n_kf: int) -> np.ndarray:
    """Query keyframes of one step: noisy revisits (8 % bit flips) of database keyframes."""
    from pl_inertial_slam_b200 import synth
    rng = np.random.default_rng(synth.SEED0 + 55 + step)
    src = rng.integers(0, n_kf, kf_batch)
    q = np.concatenate([gen_rows(int(k), int(k) + 1) for k in src])
    return synth.flip_bits(rng, q, 0.08)


# ------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.gpu), "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def stop(self, t0: float, t1: float):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for ts, line in self.lines:
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            if t0 - 0.05 <= ts <= t1 + 0.15:
                try:
                    sm.append(float(f[1]))
                    mx.append(float(f[2]))
                except ValueError:
                    continue
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples in the timed region"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                "samples": len(sm)}


# ------------------------------------------------------------------------------------------------
def cpu_reference_arm(sample_rows: int, n_q: int, seconds: float, nnr: float, reps_min: int = 1):
    """The reference's matchNNR (oracle/_ref, matching.cpp compiled unmodified; its knnMatch is the
    OpenCV-semantics stand-in, row-parallel over all host threads) on n_q queries x sample_rows
    database rows.  Falls back to the scalar C port when the reference build is absent."""
    import oracle
    cores = len(os.sched_getaffinity(0))
    q = gen_queries(10_000, max(1, n_q // PER_KF), N_KF)[:n_q]
    kind = "reference" if oracle.ref.available() else "port"
    if kind == "reference":
        oracle.ref.set_threads(cores)
        fn = lambda d: oracle.ref.match_nnr(q, d, nnr)  # noqa: E731
        used = cores
    else:
        fn = lambda d: oracle.port.match_nnr(q, d, nnr)  # noqa: E731
        used = 1
    # calibrate on a small slice, then size the sample for ~`seconds`
    cal_rows = min(sample_rows, 20_000)
    db = gen_rows(0, (cal_rows + PER_KF - 1) // PER_KF)[:cal_rows]
    t = time.perf_counter()
    fn(db)
    dt = max(time.perf_counter() - t, 1e-4)
    rate = n_q * cal_rows / dt
    rows = int(min(sample_rows, max(cal_rows, rate * seconds / n_q / max(reps_min, 1))))
    rows = max(PER_KF, rows // PER_KF * PER_KF)
    db = gen_rows(0, rows // PER_KF)
    times = []
    t_end = time.perf_counter() + seconds
    while len(times) < reps_min or (time.perf_counter() < t_end and len(times) < 20):
        t = time.perf_counter()
        fn(db)
        times.append(time.perf_counter() - t)
    med = float(np.median(times))
    return {"value": n_q * rows / med, "unit": UNIT, "cores": used, "kind": kind,
            "sample": f"matchNNR {n_q} queries x {rows} database rows (of {N_KF * PER_KF}), median of {len(times)} runs",
            "seconds_per_run": med}


def cv2_all_core(n_q: int, rows: int):
    """cv2.BFMatcher.knnMatch(k=2) with all threads: the real OpenCV code family the reference links."""
    try:
        import cv2
    except ImportError:
        return None
    cores = len(os.sched_getaffinity(0))
    cv2.setNumThreads(cores)
    q = gen_queries(10_001, max(1, n_q // PER_KF), N_KF)[:n_q]
    db = gen_rows(0, rows // PER_KF)
    bf = cv2.BFMatcher(cv2.NORM_HAMMING)
    bf.knnMatch(q[:64], db[:1000], k=2)
    t = time.perf_counter()
    bf.knnMatch(q, db, k=2)
    dt = time.perf_counter() - t
    return {"value": n_q * len(db) / dt, "unit": UNIT, "cores": cores, "kind": "cv2.BFMatcher 4.x knnMatch",
            "sample": f"{n_q} x {len(db)}"}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    n_q = args.kf_batch * PER_KF
    per_step = max(0.5, min(8.0, 75.0 / max(1, args.steps + args.warmup)))  # whole run ~1-1.5 min
    import oracle
    cores = len(os.sched_getaffinity(0))
    kind = "reference" if oracle.ref.available() else "port"
    if kind == "reference":
        oracle.ref.set_threads(cores)
    q = gen_queries(0, args.kf_batch, args.n_kf)
    # size the per-step sample once
    # calibrate on a sample that is already larger than the CPU caches (the full-size scan streams the
    # database from DRAM once per query row, like OpenCV's batchDistance loop order)
    cal = gen_rows(0, 250 if kind == "reference" else 5)
    fn0 = oracle.ref.match_nnr if kind == "reference" else oracle.port.match_nnr
    fn0(q[:64], cal[:1000], args.nnr)
    t = time.perf_counter()
    fn0(q, cal, args.nnr)
    rate = n_q * len(cal) / max(time.perf_counter() - t, 1e-4)
    rows = int(max(PER_KF, min(args.n_kf * PER_KF, rate * per_step / n_q) // PER_KF * PER_KF))
    db = gen_rows(0, rows // PER_KF)
    fn = oracle.ref.match_nnr if kind == "reference" else oracle.port.match_nnr
    for _ in range(args.warmup):
        fn(q, db, args.nnr)
    t0 = time.perf_counter()
    for s in range(args.steps):
        fn(q, db, args.nnr)
    dt = time.perf_counter() - t0
    value = n_q * rows * args.steps / dt
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u32 (xor+popcount)",
        "data": "synthetic",
        "config": {"workload": "loop-closure all-pairs matchNNR, bounded sample of config 5",
                   "kf_batch": args.kf_batch, "per_kf": PER_KF, "db_rows_sampled": rows,
                   "db_rows_full": args.n_kf * PER_KF, "nnr": args.nnr},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores if kind == "reference" else 1, "kind": kind,
                         "sample": f"each step = matchNNR of {n_q} queries x {rows} database rows "
                                   f"(of {args.n_kf * PER_KF})"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------
VERIFY_STEP = 777_000          # query seed of the untimed verification step (the same at every N)
VERIFY_SAMPLE = 64             # queries checked against the reference on the WHOLE database


def verify_step(db, args, dev, rank: int) -> dict:
    """One untimed step whose result is (a) summarised as (count, crc32 of the match vector) -- identical at
    N = 1/2/4/8 by construction -- and (b) checked on rank 0, for the first VERIFY_SAMPLE queries, against the
    reference's own matchNNR (oracle/_ref, matching.cpp compiled unmodified) on all 16 M database rows."""
    import zlib
    import torch
    q = gen_queries(VERIFY_STEP, args.kf_batch, args.n_kf)
    count, m12 = db.match_nnr(torch.from_numpy(q).to(dev), args.nnr)
    torch.cuda.synchronize()
    m12_h = m12.cpu().numpy()
    out = {"step_seed": VERIFY_STEP, "count": int(count.item()), "crc32_m12": zlib.crc32(m12_h.tobytes()) & 0xFFFFFFFF}
    if rank == 0:
        import oracle
        full = gen_rows(0, args.n_kf)
        if oracle.ref.available():
            oracle.ref.set_threads(len(os.sched_getaffinity(0)))
            n_s, m_s = oracle.ref.match_nnr(q[:VERIFY_SAMPLE], full, args.nnr)
            out["checker"] = "oracle/_ref matchNNR (reference matching.cpp) on all database rows"
        else:
            n_s, m_s = oracle.port.match_nnr(q[:VERIFY_SAMPLE], full, args.nnr)
            out["checker"] = "oracle port matchNNR on all database rows"
        del full
        out["sampled_queries"] = VERIFY_SAMPLE
        out["sample_matches"] = int(n_s)
        out["oracle_ok"] = bool((m12_h[:VERIFY_SAMPLE] == m_s).all() and int((m12_h[:VERIFY_SAMPLE] >= 0).sum()) == int(n_s))
        out["ok"] = out["oracle_ok"]
    return out


def dist_check(rank: int, world: int, local_rank: int, dev) -> dict:
    """N > 1: every sharded path (flat database through both exchange forms, row-sharded matchGrid + match fallback)
    against the oracle on every rank before anything is timed (tests/dist_gpu_check.py, compact sizes)."""
    import torch
    import torch.distributed as dist
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    ok = torch.ones(1, dtype=torch.int32, device=dev)
    info = {}
    try:
        import dist_gpu_check
        info = dist_gpu_check.run_checks(rank, world, local_rank, dev, compact=True)
    except Exception as e:  # noqa: BLE001 -- reported in the line, the run still fails below
        ok.zero_()
        info = {"ok": False, "error": repr(e)[:300]}
    dist.all_reduce(ok, op=dist.ReduceOp.MIN)
    info["ok"] = bool(ok.item())
    return info


def dump_outputs(out_dir: str, count, m12) -> None:
    """What ShardedDescriptorDB.match_nnr returned in the last timed step: the accepted count and the match vector
    (database row per query, -1 where rejected), both as float64 (row indices < 2^53 stay exact)."""
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "count.npy"), count.cpu().numpy().astype(np.float64))
    np.save(os.path.join(out_dir, "m12.npy"), m12.cpu().numpy().astype(np.float64))


# ------------------------------------------------------------------------------------------------
def run_b200(args):
    import torch
    import torch.distributed as dist
    from pl_inertial_slam_b200 import _lib
    from pl_inertial_slam_b200.database import ShardedDescriptorDB, shard_bounds

    _lib.load()  # fails loudly when the CUDA library is missing -- there is no fallback
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        import datetime
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # a rank that dies in the pre-timing check must take the job down instead of hanging its peers
        dist.init_process_group("nccl", device_id=dev, timeout=datetime.timedelta(seconds=240))

    n_rows = args.n_kf * PER_KF
    lo, hi = shard_bounds(n_rows, world, rank)
    assert lo % PER_KF == 0 and hi % PER_KF == 0, "shards are whole keyframes"
    shard_host = gen_rows(lo // PER_KF, hi // PER_KF)
    shard = torch.from_numpy(shard_host).to(dev)
    del shard_host
    db = ShardedDescriptorDB(n_rows=n_rows, shard=shard, device=local_rank, exchange=args.exchange)
    ctx = db.ops.ctx
    n_q = args.kf_batch * PER_KF
    total_steps = args.warmup + args.steps
    q_host = [torch.from_numpy(gen_queries(s, args.kf_batch, args.n_kf)).pin_memory() for s in range(total_steps)]
    q_dev = [q.to(dev) for q in q_host]
    flush = torch.empty(L2_FLUSH_BYTES, dtype=torch.uint8, device=dev)
    pairs_per_step = float(n_q) * float(n_rows)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def step_device(q):
        count, m12 = db.match_nnr(q, args.nnr)
        return count, m12

    # ---- correctness before anything is timed ------------------------------------------------
    dcheck = dist_check(rank, world, local_rank, dev) if (world > 1 and not args.no_verify) else None
    if dcheck is not None and not dcheck["ok"]:
        raise SystemExit(f"dist_check failed: {dcheck}")
    verify = verify_step(db, args, dev, rank) if not args.no_verify else None
    if rank == 0 and verify is not None and not verify["ok"]:
        raise SystemExit(f"verification against the reference failed: {verify}")

    # ---- live integer-pipe peaks (roofline denominators) -------------------------------------
    popc_gops, lop3_gops = ctx.measure_int_peaks()

    # ---- warm-up -------------------------------------------------------------------------------
    for s in range(args.warmup):
        step_device(q_dev[s])
        flush.fill_(s & 0xFF)
    barrier()
    if db.peer is not None and not db.peer.healthy():
        # a peer-memory exchange timed out on some rank during warm-up (peer stores not visible on this box?):
        # every rank switches to the NCCL form -- bit-identical results -- and warms up again
        if args.exchange == "peer":
            raise SystemExit("peer-memory exchange requested but an exchange timed out")
        db.peer = None
        for s in range(args.warmup):
            step_device(q_dev[s])
            flush.fill_(s & 0xFF)
        barrier()

    # ---- timed: device-resident inputs ---------------------------------------------------------
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        time.sleep(0.25)
    ctx.read_profile()
    ctx.set_profiling(True)
    launches0 = ctx.launch_count
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    barrier()
    t_wall0 = time.time()
    last = None
    for s in range(args.steps):
        ev[s][0].record()
        last = step_device(q_dev[args.warmup + s])
        ev[s][1].record()
        flush.fill_(s & 0xFF)  # L2 flush between timed iterations (outside the event pair)
    barrier()
    t_wall1 = time.time()
    dev_ms = sum(a.elapsed_time(b) for a, b in ev)
    launches = ctx.launch_count - launches0
    ctx.set_profiling(False)
    slice_ms, slice_n = ctx.read_profile()
    clocks = sampler.stop(t_wall0, t_wall1) if rank == 0 else None
    n_matches = int(last[0].item())
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, *last)

    # ---- timed: end to end (host query batch in pinned memory -> host match vector) ------------
    barrier()
    e2e_ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    m12_host = torch.empty(n_q, dtype=torch.int32).pin_memory()
    cnt_host = torch.empty(1, dtype=torch.int32).pin_memory()
    e2e_wall = 0.0
    for s in range(args.steps):
        t0 = time.perf_counter()
        e2e_ev[s][0].record()
        q = q_host[args.warmup + s].to(dev, non_blocking=True)
        count, m12 = step_device(q)
        m12_host.copy_(m12, non_blocking=True)
        cnt_host.copy_(count, non_blocking=True)
        e2e_ev[s][1].record()
        torch.cuda.synchronize()
        e2e_wall += time.perf_counter() - t0
        flush.fill_(s & 0xFF)
    barrier()
    e2e_ms = sum(a.elapsed_time(b) for a, b in e2e_ev)
    if db.peer is not None:
        db.peer.check()  # raises if any peer-memory exchange timed out

    # ---- config 4 (map -> frame, row-sharded map) at this N: collective, every rank takes part -----------
    config4 = None
    if not args.no_extras:
        try:
            import bench_extras
            config4 = bench_extras.map_to_frame(ctx, world, rank)
        except Exception as e:  # noqa: BLE001 -- a side metric must never kill the headline line
            config4 = {"error": repr(e)[:300]}
        barrier()

    # ---- max over ranks ------------------------------------------------------------------------
    t = torch.tensor([dev_ms, e2e_ms, e2e_wall * 1e3, slice_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dev_ms, e2e_ms, e2e_wall_ms, slice_ms_max = [float(x) for x in t.tolist()]

    if rank == 0:
        value = pairs_per_step * args.steps / (dev_ms * 1e-3)
        e2e_value = pairs_per_step * args.steps / (max(e2e_ms, e2e_wall_ms) * 1e-3)
        # roofline of the dominant kernel: per-launch pairs = n_q x local shard rows
        pairs_per_launch = float(n_q) * float(hi - lo)
        launch_ms = slice_ms / max(slice_n, 1)
        popc_equiv = pairs_per_launch * POPC_PER_PAIR / (launch_ms * 1e-3) * 1e-9  # Gop/s
        variant = os.environ.get("PLM_KNN_VARIANT", DEFAULT_VARIANT)
        variant = variant if variant in ALU_INSTR_PER_PAIR else DEFAULT_VARIANT
        pairs_rate = pairs_per_launch / (launch_ms * 1e-3) * 1e-9                   # G pairs/s inside the kernel
        pipes = {
            "xu_popc": {"instr_per_pair": POPC_ISSUED_PER_PAIR[variant], "achieved": pairs_rate * POPC_ISSUED_PER_PAIR[variant],
                        "peak": popc_gops},
            "alu_lop3": {"instr_per_pair": ALU_INSTR_PER_PAIR[variant], "achieved": pairs_rate * ALU_INSTR_PER_PAIR[variant],
                         "peak": lop3_gops},
        }
        for v in pipes.values():
            v["frac"] = v["achieved"] / v["peak"]
            v["unit"] = "Ginstr/s"
        binding = max(pipes, key=lambda k: pipes[k]["frac"])
        algo_bytes = 32.0 * (n_q + (hi - lo)) + 16.0 * n_q
        hbm_peak = 6535.4
        try:
            hbm_peak = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"]
        except Exception:
            pass
        traffic, traffic_src = None, None
        try:
            tj = json.load(open(os.path.join(ROOT, "profiles", "knn2_slice_traffic.json")))
            if tj.get("variant") == variant:     # only a capture of the kernel that actually ran counts
                traffic, traffic_src = tj["dram_bytes_per_launch"], tj.get("source")
        except Exception:
            pass
        roofline = {
            "kernel": f"knn2_slice_kernel<128, {variant}> (brute-force Hamming top-2)",
            "bound": "int",
            "pipe": binding,
            "unit": "Ginstr/s issued on the binding integer pipe (instructions per pair counted from the SASS main loop)",
            "achieved": pipes[binding]["achieved"], "peak": pipes[binding]["peak"], "frac": pipes[binding]["frac"],
            "peak_source": "measured in this run (plm_measure_int_peaks: independent POPC / LOP3 chains on every SM)",
            "pipes": pipes,
            "kernel_ms_per_launch": launch_ms, "launches_timed": slice_n,
            "share_of_step": slice_ms / dev_ms,
            "variant": variant,
            "popc8_equivalent": {"unit": "Gop/s (8 POPC.32 per pair, the unit of work of SURVEY 8d)", "achieved": popc_equiv,
                                 "peak": popc_gops, "frac": popc_equiv / popc_gops,
                                 "note": "secondary figure: the kernel issues 4 POPC + 13 LOP3 per pair (carry-save form in a "
                                         "transformed domain), so it exceeds a roofline that assumes 8 POPC per pair"},
            "hbm": {"unit": "GB/s", "achieved": algo_bytes / (launch_ms * 1e-3) * 1e-9, "peak": hbm_peak,
                    "frac": algo_bytes / (launch_ms * 1e-3) * 1e-9 / hbm_peak, "algorithmic_bytes_per_launch": algo_bytes},
            "traffic": traffic, "traffic_source": traffic_src,
        }
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": dev_ms / args.steps, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "u32 (xor+popcount)", "data": "synthetic",
            "config": {"workload": "config 5: loop-closure all-pairs keyframe matching (matchNNR, flat database)",
                       "keyframes": args.n_kf, "descriptors_per_kf": PER_KF, "db_rows": n_rows,
                       "db_bytes": n_rows * 32, "kf_batch": args.kf_batch, "queries_per_step": n_q, "nnr": args.nnr,
                       "parallelism": f"database row-sharded over {world} GPU(s), " + (
                           "no exchange" if world == 1 else
                           "per-query top-2 pushed into every rank's buffer over NVLink peer memory and merged by one kernel"
                           if db.peer is not None else "NCCL all_gather of packed top-2 + merge kernel"),
                       "l2": f"{L2_FLUSH_BYTES >> 20} MiB flush write between timed iterations"},
            "pairs_per_step": pairs_per_step,
            "reference_equivalent_pairs_per_s": value,
            "matches_last_step": n_matches,
            "verify": verify, "dist_check": dcheck,
            "config4_map_to_frame": config4,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": n_q * 32,
                    "d2h_bytes_per_step": n_q * 4 + 4, "ms_per_step_device": e2e_ms / args.steps,
                    "ms_per_step_wall": e2e_wall_ms / args.steps,
                    "note": "database shard resident in HBM (uploaded once, like the reference's in-RAM keyframe DB)"},
            "gpu_launches": int(launches) * world,
            "clocks": clocks,
            "roofline": roofline,
        }
        if not args.no_extras and world == 1:  # side metrics are single-GPU workloads (configs 1-4 on one GPU)
            try:
                import bench_extras
                line["extras"] = bench_extras.run(ctx, args)
            except Exception as e:  # noqa: BLE001 -- side metrics must never kill the headline line
                line["extras"] = {"error": repr(e)}
        if not args.no_cpu_baseline and world == 1:  # the CPU arm is reported at N=1 only
            base = cpu_reference_arm(sample_rows=400_000, n_q=PER_KF, seconds=args.cpu_seconds, nnr=args.nnr)
            cv = cv2_all_core(PER_KF, 200_000)
            if cv:
                base["cv2_all_core"] = cv
            line["cpu_baseline"] = base
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
