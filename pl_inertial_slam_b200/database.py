"""Device-resident descriptor databases sharded over GPUs (one process per GPU, torch.distributed).

The reference keeps every keyframe's descriptor Mats and the local map in host memory
(include/keyFrame.h:69-96, src/mapHandler.cpp:583-803) and matches on one core.  Here the rows live in
HBM, row-sharded contiguously over the ranks (SURVEY.md 8e); torch is plumbing only (device memory,
streams, the NCCL collective), all arithmetic is in the CUDA library:

* ``ShardedDescriptorDB`` -- flat keyframe database (config 5): queries replicated, per-shard top-2
  with GLOBAL row indices, all_gather of the packed keys, lexicographic merge.  Unsigned min over
  (distance << 32 | global index) is the reference's lowest-index tie-breaking, so any number of
  shards gives bit-identical results.
  The exchange itself is the library's own kernel over NVLink peer memory (``PeerExchange``: push into every
  rank's buffer, flag, wait, merge, ratio test -- csrc/plm_peer.cuh); NCCL's all_gather + a merge kernel is
  the equivalent form used when CUDA IPC peer mapping is unavailable.
* ``ShardedMap`` -- the local map is desc1 (the QUERY side) of matchMap2KF* (config 4): rows
  sharded, the frame (desc2 + its grid) replicated.  ``match`` needs one exchange (the 21 direction's
  top-2), ``match_grid`` needs the per-column running minima of lower-ranked shards before matching
  and the per-column best pairs after it.

The arithmetic backend is injected (``DeviceOps`` = the CUDA library) so the orchestration can be
exercised on CPU tensors with gloo in the test-suite.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import Sequence, Optional, Tuple

import numpy as np
import torch

from . import _lib as L
from .matching import Context

INT64_MIN = -(1 << 63)


def _ptr(t: Optional[torch.Tensor]) -> C.c_void_p:
    return C.c_void_p(t.data_ptr() if t is not None and t.numel() else 0)


def shard_bounds(n_rows: int, world: int, rank: int) -> Tuple[int, int]:
    """Contiguous row ranges [g*ceil(N/G), ...) (SURVEY 8e)."""
    per = (n_rows + world - 1) // world
    lo = min(n_rows, rank * per)
    return lo, min(n_rows, lo + per)


@dataclass
class GridFrame:
    """The replicated (train) side of a matchGrid call, resident on the device."""
    d2: torch.Tensor                 # n2 x 32 uint8
    cell_start: torch.Tensor         # rows*cols+1 int32
    cell_items: torch.Tensor         # int32
    rows: int
    cols: int
    dirs2: Optional[torch.Tensor] = None   # n2 x 2 float64 (lines)


class DeviceOps:
    """The plm_dev_* entry points on torch CUDA tensors, launched on torch's current stream."""

    def __init__(self, device: Optional[int] = None):
        self.device = torch.cuda.current_device() if device is None else device
        self.ctx = Context(self.device)
        self.lib = L.load()

    def _bind_stream(self):
        self.ctx.set_stream(torch.cuda.current_stream(self.device).cuda_stream)

    def knn2(self, q: torch.Tensor, db: torch.Tensor, idx_base: int = 0, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """q: nq x 32 uint8, db: n x 32 uint8 (contiguous) -> nq x 2 int64 packed keys."""
        assert q.is_cuda and db.is_cuda and q.dtype == torch.uint8 and db.dtype == torch.uint8
        assert q.is_contiguous() and db.is_contiguous() and q.shape[-1] == 32 and db.shape[-1] == 32
        nq, n = q.shape[0], db.shape[0]
        if out is None:
            out = torch.empty((nq, 2), dtype=torch.int64, device=q.device)
        self._bind_stream()
        L.check(self.lib.plm_dev_knn2(self.ctx.handle, _ptr(q), nq, _ptr(db), n, idx_base, _ptr(out)), "plm_dev_knn2")
        return out

    def top2_merge(self, parts: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """parts: P x nq x 2 int64 packed keys -> nq x 2 (two smallest keys per query)."""
        assert parts.dtype == torch.int64 and parts.is_contiguous() and parts.dim() == 3
        p, nq = parts.shape[0], parts.shape[1]
        if out is None:
            out = torch.empty((nq, 2), dtype=torch.int64, device=parts.device)
        self._bind_stream()
        L.check(self.lib.plm_dev_top2_merge(self.ctx.handle, _ptr(parts), p, nq, _ptr(out)), "plm_dev_top2_merge")
        return out

    def nnr_accept(self, top2: torch.Tensor, nnr: float, m12: torch.Tensor, count: Optional[torch.Tensor]) -> None:
        assert m12.dtype == torch.int32
        self._bind_stream()
        L.check(self.lib.plm_dev_nnr_accept(self.ctx.handle, _ptr(top2), top2.shape[0], C.c_float(nnr), _ptr(m12),
                                            _ptr(count)), "plm_dev_nnr_accept")

    def cross_check(self, m12: torch.Tensor, i1_base: int, m21: torch.Tensor, count: torch.Tensor) -> None:
        self._bind_stream()
        L.check(self.lib.plm_dev_cross_check(self.ctx.handle, _ptr(m12), m12.shape[0], i1_base, _ptr(m21),
                                             m21.shape[0], _ptr(count)), "plm_dev_cross_check")

    def _grid_args(self, coords, d1, i1_base, frame: GridFrame, win, ratio, line_sim_th, best_lr, m12, count):
        a = L.DevGridArgs()
        a.coords, a.d1 = _ptr(coords), _ptr(d1)
        a.cell_start, a.cell_items = _ptr(frame.cell_start), _ptr(frame.cell_items)
        a.d2, a.dirs2 = _ptr(frame.d2), _ptr(frame.dirs2)
        a.m12_inout, a.count = _ptr(m12), _ptr(count)
        a.i1_base, a.ratio, a.line_sim_th = int(i1_base), float(ratio), float(line_sim_th)
        a.n1, a.n2 = int(d1.shape[0]), int(frame.d2.shape[0])
        a.grid_rows, a.grid_cols = frame.rows, frame.cols
        a.is_lines, a.best_lr = int(frame.dirs2 is not None), int(bool(best_lr))
        for i in range(4):
            a.win[i] = int(win[i])
        return a

    def grid_colmin(self, coords, d1, i1_base, frame, win, ratio, line_sim_th, best_lr) -> torch.Tensor:
        """Per-column minimum distance over this shard's candidate pairs: int16 bits of uint16, n2."""
        n2 = frame.d2.shape[0]
        out = torch.empty(n2, dtype=torch.int16, device=d1.device)
        a = self._grid_args(coords, d1, i1_base, frame, win, ratio, line_sim_th, best_lr, None, None)
        # setup validates m12/count pointers only when n1 > 0; colmin never writes them
        dummy = torch.zeros(max(1, d1.shape[0]) + 1, dtype=torch.int32, device=d1.device)
        a.m12_inout, a.count = _ptr(dummy), C.c_void_p(dummy.data_ptr() + 4 * max(1, d1.shape[0]))
        self._bind_stream()
        L.check(self.lib.plm_dev_grid_colmin(self.ctx.handle, C.byref(a), _ptr(out)), "plm_dev_grid_colmin")
        return out

    def grid_match(self, coords, d1, i1_base, frame, win, ratio, line_sim_th, best_lr, m12, count,
                   seed: Optional[torch.Tensor]) -> torch.Tensor:
        """Match this shard's rows; returns m21key int64 bits of uint64, n2."""
        n2 = frame.d2.shape[0]
        key = torch.empty(n2, dtype=torch.int64, device=d1.device)
        a = self._grid_args(coords, d1, i1_base, frame, win, ratio, line_sim_th, best_lr, m12, count)
        self._bind_stream()
        L.check(self.lib.plm_dev_grid_match(self.ctx.handle, C.byref(a), _ptr(seed), _ptr(key)), "plm_dev_grid_match")
        return key

    def m21_from_keys(self, key: torch.Tensor) -> torch.Tensor:
        m21 = torch.empty(key.shape[0], dtype=torch.int32, device=key.device)
        self._bind_stream()
        L.check(self.lib.plm_dev_m21_from_keys(self.ctx.handle, _ptr(key), key.shape[0], _ptr(m21)), "plm_dev_m21_from_keys")
        return m21


class _Group:
    """The collectives the sharded paths need, on the default (or a given) process group."""

    def __init__(self, group=None):
        import torch.distributed as dist
        self.dist = dist if (dist.is_available() and dist.is_initialized()) else None
        self.group = group
        self.world = self.dist.get_world_size(group) if self.dist else 1
        self.rank = self.dist.get_rank(group) if self.dist else 0

    def all_gather(self, t: torch.Tensor) -> torch.Tensor:
        """-> [world, *t.shape]"""
        if self.world == 1:
            return t.unsqueeze(0)
        t = t.contiguous()
        flat = torch.empty((self.world * t.shape[0],) + tuple(t.shape[1:]), dtype=t.dtype, device=t.device)
        self.dist.all_gather_into_tensor(flat, t, group=self.group)   # concatenation along dim 0
        return flat.view((self.world,) + tuple(t.shape))

    def all_reduce_sum(self, t: torch.Tensor) -> torch.Tensor:
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.SUM, group=self.group)
        return t


class PeerExchange:
    """Top-2 exchange over NVLink peer memory (plm_peer_* / plm_dev_top2_exchange, csrc/plm_peer.cuh): one
    kernel pushes this rank's packed keys into every rank's exchange buffer, waits for the others and merges.
    torch.distributed only carries the 64-byte CUDA IPC handles once, at construction.

    ``PeerExchange.create`` returns None when peer mapping is not possible on some rank (e.g. every process is
    restricted to its own device); the callers then keep using the NCCL all_gather + merge-kernel form, which
    gives bit-identical results."""

    def __init__(self, g: "_Group", ops: "DeviceOps", q_cap: int):
        self.q_cap = int(q_cap)
        self._setup(g, ops, int(ops.lib.plm_peer_buffer_bytes(g.world, self.q_cap)))

    def _setup(self, g: "_Group", ops: "DeviceOps", n_bytes: int) -> None:
        """Allocate this rank's buffer, exchange the CUDA IPC handles, map the other ranks' buffers."""
        self.g, self.ops = g, ops
        self.lib = ops.lib
        self.world, self.rank = g.world, g.rank
        self.epoch = 0
        self._own = C.c_void_p()
        self._opened = []
        dev = torch.device("cuda", ops.device)
        handle = (C.c_uint8 * 64)()
        st = self.lib.plm_peer_alloc_bytes(ops.ctx.handle, n_bytes, C.byref(self._own), handle)
        ok = torch.tensor([1 if st == L.PLM_OK else 0], dtype=torch.int32, device=dev)
        mine = torch.tensor(list(handle), dtype=torch.uint8, device=dev)
        handles = g.all_gather(mine).cpu().numpy()                      # [world, 64]
        ptrs = (C.c_void_p * self.world)()
        if st == L.PLM_OK:
            ptrs[self.rank] = self._own
            for r in range(self.world):
                if r == self.rank:
                    continue
                p = C.c_void_p()
                h = (C.c_uint8 * 64)(*handles[r].tolist())
                if self.lib.plm_peer_open(ops.ctx.handle, h, C.byref(p)) != L.PLM_OK:
                    ok[0] = 0
                    break
                self._opened.append(p)
                ptrs[r] = p
        g.dist.all_reduce(ok, op=g.dist.ReduceOp.MIN, group=g.group)
        self.ok = bool(ok.item())
        self.ptrs = ptrs
        # timeout flag of the peer kernels: pinned host memory that the device writes through its unified address, so
        # the host can look at it on every call without a stream synchronisation
        self.error = torch.zeros(1, dtype=torch.int32).pin_memory()
        self.failed = False
        if not self.ok:
            self.close()

    def _raise_if_failed(self) -> None:
        """A wait that timed out leaves results unwritten and the double-buffer invariant broken: the first call after
        the flag became visible raises, and so does every later one (no silent garbage, no silent fallback)."""
        if self.failed or int(self.error[0]) != 0:
            self.failed = True
            raise RuntimeError("peer-memory exchange: a rank did not arrive within the spin limit "
                               "(option peer_spin_ms); this exchange object is unusable -- rebuild it or use exchange='nccl'")

    @classmethod
    def create(cls, g: "_Group", ops, q_cap: int) -> Optional["PeerExchange"]:
        if g.world <= 1 or g.world > 16 or not isinstance(ops, DeviceOps):
            return None
        x = cls(g, ops, q_cap)
        return x if x.ok else None

    def exchange(self, local: torch.Tensor, out: Optional[torch.Tensor] = None, nnr: float = 0.0,
                 m12: Optional[torch.Tensor] = None, count: Optional[torch.Tensor] = None) -> Optional[torch.Tensor]:
        """local: n1 x 2 int64 packed keys of this rank -> merged keys over all ranks (and / or the matchNNR
        acceptance written to m12 / count).  Every rank must call this with the same n1, in the same order."""
        n1 = int(local.shape[0])
        assert n1 <= self.q_cap and local.dtype == torch.int64 and local.is_contiguous()
        self._raise_if_failed()
        if out is None and m12 is None:
            out = torch.full((n1, 2), -1, dtype=torch.int64, device=local.device)   # absent keys if a wait times out
        self.epoch += 1
        self.ops._bind_stream()
        L.check(self.lib.plm_dev_top2_exchange(self.ops.ctx.handle, self.ptrs, self.rank, self.world, self.q_cap,
                                               self.epoch, _ptr(local), n1, _ptr(out), C.c_float(nnr), _ptr(m12),
                                               _ptr(count), _ptr(self.error)), "plm_dev_top2_exchange")
        return out

    def _reduce(self, op: int, src: torch.Tensor, n_chunks: int) -> torch.Tensor:
        self._raise_if_failed()
        out = torch.full_like(src, -1)                                               # identity of both reductions
        self.epoch += 1
        self.ops._bind_stream()
        L.check(self.lib.plm_dev_peer_reduce(self.ops.ctx.handle, self.ptrs, self.rank, self.world, self.q_cap, self.epoch,
                                             op, _ptr(src), n_chunks, _ptr(out), _ptr(self.error)), "plm_dev_peer_reduce")
        return out

    def min_u64(self, keys: torch.Tensor) -> torch.Tensor:
        """Element-wise unsigned minimum over ALL ranks of an int64-bits-of-uint64 vector (the per-column best pairs)."""
        n = int(keys.shape[0])
        pad = torch.full((n + (n & 1),), -1, dtype=torch.int64, device=keys.device)  # -1 == UINT64_MAX
        pad[:n] = keys
        return self._reduce(0, pad, pad.shape[0] // 2)[:n]

    def prefix_min_u16(self, vals: torch.Tensor) -> torch.Tensor:
        """Element-wise unsigned minimum over the ranks BELOW this one of an int16-bits-of-uint16 vector (0xFFFF where
        there is none): the running column minima that seed this shard's matchGrid thresholds."""
        n = int(vals.shape[0])
        pad = torch.full(((n + 7) // 8 * 8,), -1, dtype=torch.int16, device=vals.device)  # -1 == 0xFFFF
        pad[:n] = vals
        return self._reduce(1, pad, pad.shape[0] // 8)[:n]

    def fits(self, n_bytes: int) -> bool:
        return (n_bytes + 15) // 16 <= self.q_cap

    def healthy(self) -> bool:
        """Host sync + one all_reduce: True when no exchange timed out on ANY rank since construction."""
        torch.cuda.synchronize()
        bad = torch.tensor([1 if (self.failed or int(self.error[0]) != 0) else 0], dtype=torch.int32,
                           device=torch.device("cuda", self.ops.device))
        self.g.dist.all_reduce(bad, op=self.g.dist.ReduceOp.MAX, group=self.g.group)
        return int(bad.item()) == 0

    def check(self) -> None:
        """Host sync: raises if any exchange since the last check timed out waiting for a peer."""
        torch.cuda.synchronize()
        self._raise_if_failed()

    def close(self) -> None:
        for p in self._opened:
            self.lib.plm_peer_close(self.ops.ctx.handle, p)
        self._opened = []
        if self._own:
            if self.g.dist is not None and self.ok:
                torch.cuda.synchronize()
                self.g.dist.barrier(group=self.g.group)   # nobody may still be writing into this buffer
            self.lib.plm_peer_free(self.ops.ctx.handle, self._own)
            self._own = C.c_void_p()


class PeerGather(PeerExchange):
    """All-gather of the per-shard match vectors + sum of the per-shard counts over NVLink peer memory
    (plm_dev_peer_allgather_i32): the last step of the row-sharded match / matchGrid as one kernel."""

    def __init__(self, g: "_Group", ops: "DeviceOps", n_rows_cap: int):
        self.n_rows_cap = int(n_rows_cap)
        self._setup(g, ops, int(ops.lib.plm_peer_gather_bytes(g.world, self.n_rows_cap)))

    @classmethod
    def create(cls, g: "_Group", ops, n_rows_cap: int) -> Optional["PeerGather"]:
        if g.world <= 1 or g.world > 16 or not isinstance(ops, DeviceOps):
            return None
        x = cls(g, ops, n_rows_cap)
        return x if x.ok else None

    def gather(self, local: torch.Tensor, row_lo: int, n_rows: int, count: Optional[torch.Tensor]):
        """-> (global int32 vector [n_rows], summed count [1]) on every rank."""
        assert local.dtype == torch.int32 and local.is_contiguous() and n_rows <= self.n_rows_cap
        self._raise_if_failed()
        out = torch.full((n_rows,), -1, dtype=torch.int32, device=local.device)
        total = torch.full((1,), torch.iinfo(torch.int32).min, dtype=torch.int32, device=local.device)
        self.epoch += 1
        self.ops._bind_stream()
        L.check(self.lib.plm_dev_peer_allgather_i32(self.ops.ctx.handle, self.ptrs, self.rank, self.world, self.n_rows_cap,
                                                    self.epoch, _ptr(local), int(row_lo), int(local.shape[0]), int(n_rows),
                                                    _ptr(count), _ptr(out), _ptr(total), _ptr(self.error)),
                "plm_dev_peer_allgather_i32")
        return out, total


class ShardSet:
    """The keyframe database / local map row-sharded over several GPUs INSIDE ONE PROCESS (plm_shard_* of
    include/plmatch.h): what a single C++ host such as the reference's MapHandler calls; host buffers in and out,
    every index global.  No torch.distributed involved -- the library enables peer access and drives the peer-memory
    kernels itself."""

    def __init__(self, devices: Sequence[int], q_cap: int, rows_cap: int):
        self.lib = L.load()
        devs = (C.c_int * len(devices))(*[int(d) for d in devices])
        h = C.c_void_p()
        L.check(self.lib.plm_shard_create(devs, len(devices), int(q_cap), int(rows_cap), C.byref(h)), "plm_shard_create")
        self._h = h
        self.n_devices = len(devices)

    def upload(self, rows: np.ndarray, coords: Optional[np.ndarray] = None) -> None:
        d, p, n, step = L.desc_args(rows)
        self._keep = (d, None)
        cp, per = None, 0
        if coords is not None:
            c = np.ascontiguousarray(coords, np.int32)
            assert c.shape[0] == n and c.shape[1] in (2, 4)
            cp, per = c.ctypes.data_as(L.i32p), int(c.shape[1])
        L.check(self.lib.plm_shard_upload(self._h, p, n, step, cp, per), "plm_shard_upload")
        self.n_rows = n

    def ranges(self):
        out = []
        for i in range(self.n_devices):
            lo, hi = C.c_int64(), C.c_int64()
            L.check(self.lib.plm_shard_range(self._h, i, C.byref(lo), C.byref(hi)), "plm_shard_range")
            out.append((lo.value, hi.value))
        return out

    @property
    def launch_count(self) -> int:
        return int(self.lib.plm_shard_launch_count(self._h))

    def knn2(self, q: np.ndarray) -> np.ndarray:
        d, p, n1, step = L.desc_args(q)
        top2 = np.empty((n1, 2), np.uint64)
        L.check(self.lib.plm_shard_match_nnr(self._h, p, n1, step, C.c_float(0.0), top2.ctypes.data_as(L.u64p), None, None),
                "plm_shard_match_nnr")
        return top2

    def match_nnr(self, q: np.ndarray, nnr: float, m12: Optional[np.ndarray] = None):
        d, p, n1, step = L.desc_args(q)
        buf = np.full(n1, -1, np.int32) if m12 is None else np.array(m12, np.int32)
        n = C.c_int(0)
        st = self.lib.plm_shard_match_nnr(self._h, p, n1, step, C.c_float(nnr), None, buf.ctypes.data_as(L.i32p), C.byref(n))
        if st == L.PLM_E_TRAIN:
            raise RuntimeError("[matchNNR] Different size for matches and descriptors!")
        L.check(st, "plm_shard_match_nnr")
        return n.value, buf

    def match_grid(self, grid, d2: np.ndarray, win, ratio: float, best_lr: bool = True, dirs2: Optional[np.ndarray] = None,
                   line_sim_th: float = 0.75, m12: Optional[np.ndarray] = None):
        cs, ci, rows, cols = grid
        cs = np.ascontiguousarray(cs, np.int32)
        ci = np.ascontiguousarray(ci, np.int32)
        d, p2, n2, step2 = L.desc_args(d2)
        w = np.ascontiguousarray(win, np.int32)
        dr = None if dirs2 is None else np.ascontiguousarray(dirs2, np.float64)
        buf = np.full(self.n_rows, -1, np.int32) if m12 is None else np.array(m12, np.int32)
        n = C.c_int(0)
        L.check(self.lib.plm_shard_match_grid(self._h, cs.ctypes.data_as(L.i32p), ci.ctypes.data_as(L.i32p), int(rows), int(cols), p2, n2,
                                              step2, None if dr is None else dr.ctypes.data_as(L.f64p), float(line_sim_th),
                                              w.ctypes.data_as(L.i32p), float(ratio), int(bool(best_lr)), buf.ctypes.data_as(L.i32p),
                                              C.byref(n)), "plm_shard_match_grid")
        return n.value, buf

    def match(self, d2: np.ndarray, nnr: float, best_lr: bool = True, m12: Optional[np.ndarray] = None):
        d, p2, n2, step2 = L.desc_args(d2)
        buf = np.full(self.n_rows, -1, np.int32) if m12 is None else np.array(m12, np.int32)
        n = C.c_int(0)
        st = self.lib.plm_shard_match(self._h, p2, n2, step2, C.c_float(nnr), int(bool(best_lr)), buf.ctypes.data_as(L.i32p), C.byref(n))
        if st == L.PLM_E_TRAIN:
            raise RuntimeError("[matchNNR] Different size for matches and descriptors!")
        L.check(st, "plm_shard_match")
        return n.value, buf

    def close(self) -> None:
        if getattr(self, "_h", None):
            self.lib.plm_shard_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:  # noqa: BLE001
            pass


class ShardedDescriptorDB:
    """Flat descriptor database (config 5), row-sharded over the ranks of a process group.

    Pass ``rows`` (host, the WHOLE database; each rank uploads only its shard) or an already resident
    ``shard`` tensor with the global row count ``n_rows``.
    """

    def __init__(self, rows: Optional[np.ndarray] = None, n_rows: Optional[int] = None, device: Optional[int] = None,
                 group=None, shard: Optional[torch.Tensor] = None, ops=None, exchange: str = "auto", q_cap: int = 8192):
        """exchange: "peer" / "auto" = per-query top-2 merged by the peer-memory kernel (falls back to NCCL when
        peer mapping is unavailable; "peer" raises instead), "nccl" = all_gather + merge kernel.  q_cap = the
        largest query batch the peer buffers are sized for (larger batches take the NCCL form)."""
        self.g = _Group(group)
        self.world, self.rank = self.g.world, self.g.rank
        self.ops = ops if ops is not None else DeviceOps(device)
        self.peer = PeerExchange.create(self.g, self.ops, q_cap) if exchange in ("peer", "auto") else None
        if exchange == "peer" and self.world > 1 and self.peer is None:
            raise RuntimeError("peer-memory exchange requested but CUDA IPC peer mapping is unavailable")
        if shard is not None:
            assert n_rows is not None
            self.n_rows = int(n_rows)
            self.lo, self.hi = shard_bounds(self.n_rows, self.world, self.rank)
            assert shard.shape[0] == self.hi - self.lo
            self.shard = shard
        else:
            self.n_rows = int(rows.shape[0])
            self.lo, self.hi = shard_bounds(self.n_rows, self.world, self.rank)
            t = torch.from_numpy(np.ascontiguousarray(rows[self.lo:self.hi]))
            self.shard = t.to(torch.device("cuda", self.ops.device)) if hasattr(self.ops, "device") else t

    def knn2_local(self, q: torch.Tensor) -> torch.Tensor:
        """Packed top-2 of the queries over THIS rank's shard, with global row indices."""
        return self.ops.knn2(q, self.shard, idx_base=self.lo)

    def knn2(self, q: torch.Tensor) -> torch.Tensor:
        """Packed top-2 over the whole database: local kernel -> all_gather -> merge kernel."""
        local = self.knn2_local(q)
        if self.world == 1:
            return local
        if self.peer is not None and q.shape[0] <= self.peer.q_cap:
            return self.peer.exchange(local)
        return self.ops.top2_merge(self.g.all_gather(local))

    def match_nnr(self, q: torch.Tensor, nnr: float):
        """StVO::matchNNR of the queries against the whole (sharded) database -> (count, m12)."""
        m12 = torch.full((q.shape[0],), -1, dtype=torch.int32, device=q.device)
        count = torch.zeros(1, dtype=torch.int32, device=q.device)
        if self.world > 1 and self.peer is not None and q.shape[0] <= self.peer.q_cap:
            # local slices -> ONE kernel: push to the peers, wait, merge, ratio test
            self.peer.exchange(self.knn2_local(q), nnr=nnr, m12=m12, count=count)
            return count, m12
        top2 = self.knn2(q)
        self.ops.nnr_accept(top2, nnr, m12, count)
        return count, m12


class KeyframeDB:
    """Loop-closure matching per keyframe pair against a resident keyframe database (SURVEY 8d "Mode A"):
    MapHandler::isLoopClosure runs StVO::match(kf0.desc, kf1.desc) for ONE candidate pair (mapHandler.cpp:3325-3378,
    each pair with its own ratio tests and mutual check); here one query keyframe is matched against EVERY keyframe of
    the database in one batched launch (plm_batch_set_match_dev over the resident arena).  For several GPUs give every
    rank a contiguous range of keyframes: the pairs are independent, only the per-keyframe counts are gathered.
    Every job of the batch shares the query slot, so with option "batch_umma" = 1 (read when the job tables are built
    for a query size) both directions of every pair come from one int8 tensor-core product (DESIGN K1c); the results
    are identical to the integer list kernels', which the automatic choice keeps (they measured faster).

    ``rows``: all descriptors of the database keyframes back to back (n x 32 uint8), ``kf_start``: n_kf + 1 row offsets;
    ``q_cap``: the largest query keyframe (rows reserved behind the database for the query slot)."""

    def __init__(self, rows, kf_start, device: int = 0, q_cap: int = 2048, ctx: Optional[Context] = None):
        from .replay import MatchBatch
        self.ctx = ctx if ctx is not None else Context(device)
        dev = torch.device("cuda", device)
        rows_t = torch.as_tensor(rows)
        self.n_rows = int(rows_t.shape[0])
        self.q_cap = int(q_cap)
        self.kf_start = np.ascontiguousarray(kf_start, np.int64)
        self.n_kf = len(self.kf_start) - 1
        self.arena = torch.zeros((self.n_rows + self.q_cap, 32), dtype=torch.uint8, device=dev)
        self.arena[: self.n_rows] = rows_t.to(dev)
        self.batch = MatchBatch(self.ctx)
        self._prepared = None      # (nq, nnr, best_lr) the job tables were built for

    def _prepare(self, nq: int, nnr: float, best_lr: bool) -> None:
        if self._prepared == (nq, nnr, best_lr):
            return
        jobs = np.zeros(self.n_kf, L.PAIR_JOB_DTYPE)
        jobs["off1"] = self.n_rows                             # the query slot
        jobs["n1"] = nq
        jobs["off2"] = self.kf_start[:-1]
        jobs["n2"] = np.diff(self.kf_start)
        jobs["off_m"] = np.arange(self.n_kf, dtype=np.int64) * nq
        self.batch.set_match_dev(self.arena, jobs, nnr, best_lr, self.n_kf * nq)
        self._prepared = (nq, nnr, best_lr)

    def match_all(self, query, nnr: float, best_lr: bool = True, want_matches: bool = False):
        """StVO::match(query, keyframe k) for every k -> counts int32[n_kf] (INT32_MIN where the reference would be
        UB: a keyframe with fewer than 2 descriptors) and, with want_matches, the match vectors int32[n_kf, nq]."""
        q = torch.as_tensor(query)
        nq = int(q.shape[0])
        if nq > self.q_cap:
            raise ValueError("query keyframe larger than q_cap")
        self._prepare(nq, float(np.float32(nnr)), bool(best_lr))
        self.ctx.synchronize()                                  # earlier runs have finished reading the slot
        self.arena[self.n_rows: self.n_rows + nq] = q.to(self.arena.device)
        torch.cuda.current_stream(self.arena.device).synchronize()
        self.batch.run()
        if want_matches:
            m12, counts = self.batch.fetch()
            return counts, m12.reshape(self.n_kf, nq)
        return self.batch.fetch_counts(), None


class ShardedMap:
    """The local map as the row-sharded QUERY side (desc1) of matchMap2KF* (config 4).

    ``d1_shard`` / ``coords_shard`` are this rank's rows [lo, hi) of the n_rows map features
    (coords: n x 2 cell coordinates for points, n x 4 for lines).
    """

    def __init__(self, n_rows: int, d1_shard: torch.Tensor, coords_shard: Optional[torch.Tensor] = None, group=None,
                 ops=None, device: Optional[int] = None, exchange: str = "auto", q_cap: int = 4096):
        self.g = _Group(group)
        self.world, self.rank = self.g.world, self.g.rank
        self.ops = ops if ops is not None else DeviceOps(device)
        self.peer = PeerExchange.create(self.g, self.ops, q_cap) if exchange in ("peer", "auto") else None
        if exchange == "peer" and self.world > 1 and self.peer is None:
            raise RuntimeError("peer-memory exchange requested but CUDA IPC peer mapping is unavailable")
        self.gatherer = PeerGather.create(self.g, self.ops, int(n_rows)) if self.peer is not None else None
        self.n_rows = int(n_rows)
        self.lo, self.hi = shard_bounds(self.n_rows, self.world, self.rank)
        assert d1_shard.shape[0] == self.hi - self.lo
        self.d1 = d1_shard
        self.coords = coords_shard
        self.per = (self.n_rows + self.world - 1) // self.world

    # -- helpers ---------------------------------------------------------------------------------
    def _gather_rows(self, m12_local: torch.Tensor) -> torch.Tensor:
        """Concatenate the per-shard match vectors into the global n_rows vector (on every rank)."""
        if self.world == 1:
            return m12_local
        pad = torch.full((self.per,), -1, dtype=m12_local.dtype, device=m12_local.device)
        pad[: m12_local.shape[0]] = m12_local
        return self.g.all_gather(pad).reshape(-1)[: self.n_rows]

    def _peer_group(self, n_xchg_epochs: int) -> "L.PeerGroup":
        """The two sets of peer buffers + the epochs the next fused call consumes."""
        grp = L.PeerGroup()
        grp.xchg, grp.gather = self.peer.ptrs, self.gatherer.ptrs
        grp.rank, grp.world, grp.q_cap = self.rank, self.world, self.peer.q_cap
        grp.n_rows_cap = self.gatherer.n_rows_cap
        grp.xchg_epoch, grp.gather_epoch = self.peer.epoch + 1, self.gatherer.epoch + 1
        self.peer.epoch += n_xchg_epochs
        self.gatherer.epoch += 1
        return grp

    def _finish(self, m12_local: torch.Tensor, count: torch.Tensor):
        """Global match vector + global count on every rank: one peer-memory kernel, or all_reduce + all_gather."""
        if self.gatherer is not None:
            m12, total = self.gatherer.gather(m12_local, self.lo, self.n_rows, count)
            return total, m12
        self.g.all_reduce_sum(count)
        return count, self._gather_rows(m12_local)

    def _local_m12(self, m12_global: Optional[torch.Tensor], device) -> torch.Tensor:
        if m12_global is None:
            return torch.full((self.hi - self.lo,), -1, dtype=torch.int32, device=device)
        return m12_global[self.lo:self.hi].clone()

    # -- StVO::match (brute-force fallback, mapHandler.cpp:645-650) --------------------------------
    def match(self, d2: torch.Tensor, nnr: float, best_lr: bool = True, m12_inout: Optional[torch.Tensor] = None):
        """-> (count tensor [1], m12 global int32[n_rows]); m12_inout is the global in/out vector."""
        dev = d2.device
        m12 = self._local_m12(m12_inout, dev)
        if self.peer is not None and self.gatherer is not None and 2 <= d2.shape[0] <= self.peer.q_cap:
            # one C call: both directions, the peer-memory exchange, mutual check and the all-gather back to back
            self.peer._raise_if_failed()
            self.gatherer._raise_if_failed()
            grp = self._peer_group(1 if best_lr else 0)   # only epochs that are really used are consumed
            out = torch.full((self.n_rows,), -1, dtype=torch.int32, device=dev)
            total = torch.full((1,), torch.iinfo(torch.int32).min, dtype=torch.int32, device=dev)
            self.ops._bind_stream()
            L.check(self.ops.lib.plm_dev_sharded_match(self.ops.ctx.handle, _ptr(self.d1), int(self.d1.shape[0]), self.lo, _ptr(d2),
                                                       int(d2.shape[0]), C.c_float(nnr), int(bool(best_lr)), _ptr(m12), C.byref(grp),
                                                       self.n_rows, _ptr(out), _ptr(total), _ptr(self.peer.error)),
                    "plm_dev_sharded_match")
            return total, out
        count = torch.zeros(1, dtype=torch.int32, device=dev)
        # direction 12: the shard's rows are final locally
        top12 = self.ops.knn2(self.d1, d2, idx_base=0)
        self.ops.nnr_accept(top12, nnr, m12, count)
        if best_lr:
            # direction 21: per-shard top-2 with global map indices -> gather -> merge -> ratio test
            part = self.ops.knn2(d2, self.d1, idx_base=self.lo)
            m21 = torch.full((d2.shape[0],), -1, dtype=torch.int32, device=dev)
            if self.world > 1 and self.peer is not None and d2.shape[0] <= self.peer.q_cap:
                self.peer.exchange(part, nnr=nnr, m12=m21)       # push / wait / merge / ratio test in one kernel
            else:
                top21 = part if self.world == 1 else self.ops.top2_merge(self.g.all_gather(part))
                self.ops.nnr_accept(top21, nnr, m21, None)
            self.ops.cross_check(m12, self.lo, m21, count)
        return self._finish(m12, count)

    # -- StVO::matchGrid (mapHandler.cpp:637-642 / :752-757) --------------------------------------
    def match_grid(self, frame: GridFrame, win, ratio: float, line_sim_th: float = 0.75, best_lr: bool = True,
                   m12_inout: Optional[torch.Tensor] = None):
        dev = frame.d2.device
        n2 = frame.d2.shape[0]
        if self.world == 1:
            # one device: the whole matchGrid is one C call (four launches back to back, the fresh vector and the count
            # are initialised inside the first pass)
            fresh = m12_inout is None
            m12 = torch.empty(self.n_rows, dtype=torch.int32, device=dev) if fresh else m12_inout.clone()
            count = torch.empty(1, dtype=torch.int32, device=dev) if fresh else torch.zeros(1, dtype=torch.int32, device=dev)
            a = self.ops._grid_args(self.coords, self.d1, 0, frame, win, ratio, line_sim_th, best_lr, m12, count)
            self.ops._bind_stream()
            L.check(self.ops.lib.plm_dev_match_grid(self.ops.ctx.handle, C.byref(a), int(fresh)), "plm_dev_match_grid")
            return count, m12
        m12 = self._local_m12(m12_inout, dev)
        count = torch.zeros(1, dtype=torch.int32, device=dev)
        if self.peer is not None and self.gatherer is not None and (n2 == 0 or self.peer.fits(8 * n2)):
            # everything in one C call: the launches go out back to back, the three exchanges are peer-memory kernels
            a = self.ops._grid_args(self.coords, self.d1, self.lo, frame, win, ratio, line_sim_th, best_lr, m12, count)
            self.peer._raise_if_failed()
            self.gatherer._raise_if_failed()
            grp = self._peer_group(2 if (best_lr and n2 > 0) else 0)
            out = torch.full((self.n_rows,), -1, dtype=torch.int32, device=dev)
            total = torch.full((1,), torch.iinfo(torch.int32).min, dtype=torch.int32, device=dev)
            self.ops._bind_stream()
            L.check(self.ops.lib.plm_dev_sharded_match_grid(self.ops.ctx.handle, C.byref(a), C.byref(grp), self.n_rows, _ptr(out),
                                                            _ptr(total), _ptr(self.peer.error)), "plm_dev_sharded_match_grid")
            return total, out
        seed = None
        use_peer = self.peer is not None and n2 > 0 and self.peer.fits(8 * n2)
        if best_lr and self.world > 1:
            # running column minima left behind by the rows of lower-ranked shards
            cm = self.ops.grid_colmin(self.coords, self.d1, self.lo, frame, win, ratio, line_sim_th, best_lr)
            if use_peer:
                seed = self.peer.prefix_min_u16(cm).contiguous()            # one kernel over NVLink peer memory
            else:
                # uint16 bits travel as int32 (neither NCCL nor gloo carries 16-bit integers)
                allcm = self.g.all_gather(cm.to(torch.int32) & 0xFFFF)      # [world, n2], 0xFFFF = none
                if self.rank > 0:
                    seed = allcm[: self.rank].min(dim=0).values.to(torch.int16).contiguous()
        key = self.ops.grid_match(self.coords, self.d1, self.lo, frame, win, ratio, line_sim_th, best_lr, m12, count, seed)
        if best_lr:
            if self.world > 1 and use_peer:
                key = self.peer.min_u64(key).contiguous()                   # unsigned min over the shards, one kernel
            elif self.world > 1:
                # unsigned min over shards of (distance << 32 | global row): flip the sign bit so that
                # signed min orders like unsigned
                allk = self.g.all_gather(key) ^ INT64_MIN
                key = (allk.min(dim=0).values ^ INT64_MIN).contiguous()
            m21 = self.ops.m21_from_keys(key) if n2 else torch.empty(0, dtype=torch.int32, device=dev)
            self.ops.cross_check(m12, self.lo, m21, count)
        return self._finish(m12, count)
