"""Planted-copy detectors for the tcgen05 pipeline (`umma_pipeline`): cells that take another cell's value.

Both tensor-core kernels (K1b `knn2_umma_kernel`, K1c `knn2_umma_pairs_kernel`) stream 128-row train units through an
8-deep packed ring, 3 expanded B tiles and 2 accumulator buffers, and output only a top-2 per query.  With random rows a
cell that reads a wrong value almost never beats the query's top-2, so such a leak stays invisible.  Here the expected
output is known by construction and every leak changes it:
  * K1b: every query appears exactly twice in the train set as an exact copy, all other rows (fillers) equal no query.
    The output is (0 << 32 | idx_base + first copy, 0 << 32 | idx_base + second copy).  A cell that reads another row,
    another query or another accumulator column makes the owner of the displaced copy lose it, or gives a query a false
    distance 0 -- either changes that query's keys.  With no fillers every cell of the distance matrix is watched.
  * K1c: every job's train range is a permutation of the query rows (plus fillers), so each query is in each job once:
    m12 is the inverse permutation and every count is n1 (best 0, second > 0: the ratio test passes for any nnr, and
    under best_lr direction 21 finds the same pairs).
A failure names, for each wrong query, where the lost and the false rows sit in the pipeline (CTA, position c in its
share, ring stage, B tile, accumulator buffer, column) and how far the false row is from the true copy it mirrors.
"""
import numpy as np
import pytest

import oracle
from pl_inertial_slam_b200 import synth

port = oracle.port

RING = 8        # KNN_UMMA_STAGES
B_TILES = 3     # KNN_UMMA_BSTAGES
ROWS = 128      # train rows per unit
GROUP = 256     # queries per group


# ---------------------------------------------------------------------------------------------------------------------
# where a cell sits in the pipeline


class Split:
    """The (query group, unit) work list of one tensor-core launch over its CTAs, as umma_cta_of cuts it: CTA k owns
    items [k * total / ctas, (k + 1) * total / ctas), item x = group * n_units + unit; every ring runs on across the
    segments of a share, so position c = x - first item of the CTA indexes all of them."""

    def __init__(self, n1, n_units, sms):
        self.groups = -(-n1 // GROUP)
        self.n_units = n_units
        self.total = self.groups * n_units
        self.ctas = min(sms, self.total)

    def cta_of(self, x):
        return ((x + 1) * self.ctas - 1) // self.total

    def share(self, cta):
        return cta * self.total // self.ctas, (cta + 1) * self.total // self.ctas

    def cell(self, g, unit, col):
        x = g * self.n_units + unit
        cta = self.cta_of(x)
        c = x - self.share(cta)[0]
        return dict(cta=cta, c=c, stage=c % RING, tile=c % B_TILES, acc=c % 2, unit=unit, col=col)


def describe(cell):
    return ("CTA {cta} c={c} (ring stage {stage}, B tile {tile}, accumulator {acc}) unit {unit} column {col}"
            .format(**cell))


def relate(false, source):
    """How a false cell relates to the true copy whose value it shows (both in one CTA's share)."""
    if false["cta"] != source["cta"]:
        return "copy in another CTA (%s)" % describe(source)
    same = [k for k in ("stage", "tile", "acc") if false[k] == source[k]]
    return "from %s: dc=%+d dcol=%+d, same %s" % (describe(source), source["c"] - false["c"], source["col"] - false["col"],
                                                  "/".join(same) or "nothing")


def _knn2_diagnosis(split, got, want, copies, owner, idx_base):
    """One line per wrong query (the first 8): lost copies and false rows at distance 0, and where they sit."""
    bad = np.flatnonzero((got != want).any(1))
    lines = ["%d of %d queries wrong" % (bad.size, len(got))]
    for i in bad[:8]:
        g = i // GROUP
        d0 = {int(k & 0xFFFFFFFF) - idx_base for k in got[i] if k >> np.uint64(32) == 0}
        true = {int(r) for r in copies[i]}
        msg = ["query %d: got %s want %s" % (i, [hex(int(k)) for k in got[i]], [hex(int(k)) for k in want[i]])]
        for r in sorted(true - d0):
            msg.append("lost row %d at %s" % (r, describe(split.cell(g, r // ROWS, r % ROWS))))
        for r in sorted(d0 - true):
            f = split.cell(g, r // ROWS, r % ROWS)
            rel = [relate(f, split.cell(g, s // ROWS, s % ROWS)) for s in sorted(true)]
            msg.append("false row %d (a copy of query %s) at %s; %s" % (r, owner.get(r), describe(f), "; ".join(rel)))
        lines.append(" | ".join(msg))
    return "\n".join(lines)


def test_diagnosis_of_recorded_tie_stress_failure():
    """tests/test_gpu_knn_tensor.py::test_tie_stress[513-70000] on 148 SMs: query 512 got row 522 at distance 0 (true
    distance 3).  The only distance-0 row at row 522's column in that CTA's share is row 1546: c = 1 against c = 9, the
    same packed-ring stage and column -- the next unit to use the stage."""
    rng = np.random.default_rng(5 + 513)
    d1, d2 = synth.tie_stress_desc(rng, 513), synth.tie_stress_desc(rng, 70_000)
    dist = np.unpackbits(d2 ^ d1[512], axis=1).sum(1)
    assert dist[522] == 3
    split = Split(513, -(-70_000 // ROWS), 148)
    false = split.cell(2, 522 // ROWS, 522 % ROWS)
    lo, hi = split.share(false["cta"])
    share_rows = [r for r in np.flatnonzero(dist == 0) if lo <= 2 * split.n_units + r // ROWS < hi]
    assert share_rows == [617, 1546]
    src = split.cell(2, 1546 // ROWS, 1546 % ROWS)
    assert (false["cta"], false["c"], src["c"]) == (99, 1, 9)
    assert false["stage"] == src["stage"] and false["col"] == src["col"] == 10
    assert false["tile"] != src["tile"]
    assert relate(false, src).endswith("dc=+8 dcol=+0, same stage/acc")


# ---------------------------------------------------------------------------------------------------------------------
# K1b: knn2 with planted copies


@pytest.fixture(scope="module")
def M(plm_lib):
    from pl_inertial_slam_b200 import matching
    return matching


@pytest.fixture(scope="module")
def sms(plm_lib):
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


@pytest.fixture
def variant(plm_lib):
    def force(v):
        assert plm_lib.plm_set_option(b"knn_variant", v) == 0
    yield force
    plm_lib.plm_set_option(b"knn_variant", -1)


def _distinct_queries(rng, n1):
    d1 = synth.rand_desc(rng, n1)
    assert len(np.unique(d1, axis=0)) == n1
    return d1


def _planted(rng, d1, positions, n2):
    """Train set of n2 rows: query i at rows positions[i] (two each), random fillers elsewhere that equal no query."""
    n1 = len(d1)
    d2 = synth.rand_desc(rng, n2)
    pos = np.sort(np.asarray(positions, np.int64), 1)
    assert pos.shape == (n1, 2) and len(np.unique(pos)) == 2 * n1 and pos.max() < n2
    d2[pos[:, 0]] = d1
    d2[pos[:, 1]] = d1
    filler = np.ones(n2, bool)
    filler[pos.ravel()] = False
    qset = {row.tobytes() for row in d1}
    assert not any(row.tobytes() in qset for row in d2[filler])
    return d2, pos


def _expected(pos, idx_base):
    return (pos + idx_base).astype(np.uint64)   # distance 0: the key is the index


def _check_knn2(got, pos, idx_base, n2, sms):
    want = _expected(pos, idx_base)
    if not np.array_equal(got, want):
        owner = {int(r): i for i, p in enumerate(pos) for r in p}
        pytest.fail(_knn2_diagnosis(Split(len(pos), -(-n2 // ROWS), sms), got, want, pos, owner, idx_base))


@pytest.mark.gpu
@pytest.mark.parametrize("n1", [513, 4100, 12_000, 35_000])
def test_knn2_every_cell_watched(M, variant, sms, n1):
    """n2 = 2 n1, no fillers: every (query, row) cell of the product decides a key.  Shares run from 1 unit (513) to
    ~500 (35 000), so the ring, the B tiles and the accumulator pair wrap many times and segments switch; the last
    unit is ragged for every n1."""
    rng = np.random.default_rng(700 + n1)
    d1 = _distinct_queries(rng, n1)
    d2, pos = _planted(rng, d1, rng.permutation(2 * n1).reshape(n1, 2), 2 * n1)
    assert len(d2) % ROWS != 0
    base = 2 ** 32 - 2 * n1 - 5   # keys near the top of the 32-bit index range
    variant(7)
    _check_knn2(M.knn2(d1, d2, idx_base=base), pos, base, len(d2), sms)


@pytest.mark.gpu
def test_knn2_automatic_mode_takes_the_tensor_path(plm_lib, variant, sms):
    """35 000 queries x 70 000 rows (copies at random rows, fillers elsewhere) through plm_dev_knn2 in automatic mode:
    the launches are knn2_umma_kernel and the merge, and every key is the planted one."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    from pl_inertial_slam_b200.database import DeviceOps
    rng = np.random.default_rng(801)
    n1, n2 = 35_000, 70_000
    d1 = _distinct_queries(rng, n1)
    d2, pos = _planted(rng, d1, rng.choice(n2, 2 * n1, replace=False).reshape(n1, 2), n2)
    variant(-1)
    ops = DeviceOps(0)
    q, db = torch.from_numpy(d1).cuda(), torch.from_numpy(d2).cuda()
    ops.knn2(q, db, idx_base=3)   # first call: module load outside the profiled window
    torch.cuda.synchronize()
    n0 = ops.ctx.launch_count
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = ops.knn2(q, db, idx_base=3)
        torch.cuda.synchronize()
    assert ops.ctx.launch_count - n0 == 2
    kernels = [e.key for e in prof.key_averages() if e.device_type == torch.autograd.DeviceType.CUDA]
    assert any("knn2_umma_kernel" in k for k in kernels), kernels
    _check_knn2(out.cpu().numpy().view(np.uint64), pos, 3, n2, sms)


def _alias_positions(rng, n1, n2, sms, deltas=(1, 2, 3, 8)):
    """Copy positions for n1 queries in n2 rows such that, inside every CTA's share, units c and c + d of one query
    group (d in deltas) hold copies of two different queries at the same column.  A unit that reads the row of the
    unit d positions later (a ring stage, B tile or accumulator buffer released too early) then gives the second query
    a false 0 and takes the first query's copy away.  A group of one query cannot pair two queries: its copies go to
    rows 4 * 128 + 10 + 128 d at d = 8 and 2 (1546 is the row of the tie-stress failure), over filler rows in unit 4."""
    n_units = -(-n2 // ROWS)
    split = Split(n1, n_units, sms)
    used, rows = set(), {q: [] for q in range(n1)}

    def put(q, r):
        assert r not in used and len(rows[q]) < 2
        rows[q].append(r)
        used.add(r)

    pools = []
    for g in range(split.groups):
        qs = np.arange(g * GROUP, min(n1, (g + 1) * GROUP))
        if len(qs) == 1:
            put(int(qs[0]), 4 * ROWS + 10 + 8 * ROWS)
            put(int(qs[0]), 4 * ROWS + 20 + 2 * ROWS)
        pools.append([int(q) for q in rng.permutation(np.repeat(qs, 2))] if len(qs) > 1 else [])
    for cta in range(split.ctas):
        lo, hi = split.share(cta)
        for d in deltas:
            starts = [x for x in range(lo, hi - d) if x // n_units == (x + d) // n_units]
            if not starts:
                continue
            g, u = divmod(int(rng.choice(starts)), n_units)
            pool = pools[g]
            cols = [col for col in rng.permutation(ROWS) if (u + d) * ROWS + col < n2
                    and u * ROWS + col not in used and (u + d) * ROWS + col not in used]
            b = pool[-1] if pool else None
            a = next((k for k in range(len(pool) - 2, -1, -1) if pool[k] != b), None)
            if not cols or a is None:
                continue
            put(pool.pop(a), u * ROWS + int(cols[0]))
            put(pool.pop(), (u + d) * ROWS + int(cols[0]))
    free = rng.permutation(np.setdiff1d(np.arange(n2), np.fromiter(used, np.int64)))
    k = 0
    for pool in pools:   # copies no probe took: any free row
        for q in pool:
            put(q, int(free[k]))
            k += 1
    return np.array([rows[q] for q in range(n1)], np.int64)


@pytest.mark.gpu
def test_knn2_alias_probe_at_tie_stress_geometry(M, variant, sms):
    """513 queries x 70 000 rows (the failing tie-stress shape), mostly fillers: in every CTA's share, copies of two
    different queries at the same column of units c and c + d for d = 1, 2, 3 (B tiles, accumulator pair) and 8 (the
    packed ring), so a leak along any of those periods changes two queries' keys."""
    rng = np.random.default_rng(518)
    n1, n2 = 513, 70_000
    d1 = _distinct_queries(rng, n1)
    pos = _alias_positions(rng, n1, n2, sms)
    d2, pos = _planted(rng, d1, pos, n2)
    variant(7)
    _check_knn2(M.knn2(d1, d2, idx_base=3), pos, 3, n2, sms)


# ---------------------------------------------------------------------------------------------------------------------
# K1c: loop-closure batches whose jobs are permutations of the query rows


@pytest.fixture
def umma(plm_lib):
    def force(v):
        assert plm_lib.plm_set_option(b"batch_umma", v) == 0
    yield force
    plm_lib.plm_set_option(b"batch_umma", -1)


def _perm_batch(rng, n1, fillers):
    """Arena = n1 distinct query rows, then one job per entry of `fillers`: a permutation of the query rows with that
    many filler rows (equal to no query) inserted at random places.  Returns the arena, the job table and, per job,
    the job row of each query (the expected m12)."""
    from pl_inertial_slam_b200 import _lib as L
    q = _distinct_queries(rng, n1)
    qset = {row.tobytes() for row in q}
    rows, jobs, want, off = [q], np.zeros(len(fillers), L.PAIR_JOB_DTYPE), [], n1
    for j, nf in enumerate(fillers):
        n2 = n1 + int(nf)
        at = np.sort(rng.choice(n2, n1, replace=False))          # job rows that hold query rows
        perm = rng.permutation(n1)                                # job row at[k] = query perm[k]
        d2 = synth.rand_desc(rng, n2)
        assert not any(d2[r].tobytes() in qset for r in np.setdiff1d(np.arange(n2), at))
        d2[at] = q[perm]
        inv = np.empty(n1, np.int32)
        inv[perm] = at
        rows.append(d2)
        jobs[j] = (0, off, j * n1, n1, n2)
        want.append(inv)
        off += n2
    return np.ascontiguousarray(np.concatenate(rows)), jobs, want


def _run_batch(umma, arena, jobs, best_lr, nnr=0.8):
    from pl_inertial_slam_b200 import replay
    umma(1)
    m_in = np.full(int(jobs["n1"].sum()), -1, np.int32)
    b = replay.MatchBatch()
    b.set_match(arena, jobs, nnr, best_lr, m_in)
    b.run()
    m12, counts = b.fetch()
    b.close()
    return m12, counts


def _check_batch(arena, jobs, want, m12, counts, sms):
    n1 = int(jobs[0]["n1"])
    units = [-(-int(n2) // ROWS) for n2 in jobs["n2"]]
    unit0 = np.concatenate([[0], np.cumsum(units)])
    split = Split(n1, int(unit0[-1]), sms)
    lines = []
    for j, inv in enumerate(want):
        got = m12[j * n1:(j + 1) * n1]
        bad = np.flatnonzero(got != inv)
        if counts[j] == n1 and bad.size == 0:
            continue
        lines.append("job %d: count %d of %d, %d queries wrong" % (j, counts[j], n1, bad.size))
        for i in bad[:4]:
            g = i // GROUP
            cell = lambda jj, r: split.cell(g, int(unit0[jj] + r // ROWS), int(r % ROWS))
            msg = "  query %d: lost row %d at %s" % (i, inv[i], describe(cell(j, inv[i])))
            if got[i] >= 0:
                f = cell(j, got[i])
                lo, hi = split.share(f["cta"])
                src = [cell(jj, want[jj][i]) for jj in range(len(want))
                       if lo <= g * split.n_units + unit0[jj] + want[jj][i] // ROWS < hi and jj != j]
                msg += "; false row %d at %s; %s" % (got[i], describe(f), "; ".join(relate(f, s) for s in src[:3]))
            lines.append(msg)
        if len(lines) > 24:
            break
    if lines:
        pytest.fail("\n".join(lines))


@pytest.mark.gpu
@pytest.mark.parametrize("best_lr", [True, False])
@pytest.mark.parametrize("n1,fillers", [
    (800, [0] * 2000),                                 # the loop-closure shape: 2000 keyframes of 800 rows
    (256, [0] * 300),                                  # one full query group
    (300, list(range(0, 300 * 37, 37))),               # ragged query group and ragged jobs
    (513, list(range(5, 513 * 7, 7)) + [0] * 40),
    (256, [9_000, 12_345, 20_000]),                    # 3 long jobs: each cut into pieces across CTAs
])
def test_pairs_every_query_in_every_job(umma, sms, n1, fillers, best_lr):
    """K1c: every job's m12 is the inverse permutation, every count is n1, in both directions (best_lr)."""
    rng = np.random.default_rng(900 + n1 + len(fillers) + int(best_lr))
    arena, jobs, want = _perm_batch(rng, n1, fillers)
    m12, counts = _run_batch(umma, arena, jobs, best_lr)
    _check_batch(arena, jobs, want, m12, counts, sms)


@pytest.mark.gpu
def test_pairs_construction_matches_oracle(umma, sms):
    """The construction itself, checked at 256 x 300 against oracle.port.match per job, both best_lr settings."""
    rng = np.random.default_rng(950)
    arena, jobs, want = _perm_batch(rng, 256, rng.integers(0, 40, 300))
    for best_lr in (True, False):
        m12, counts = _run_batch(umma, arena, jobs, best_lr)
        _check_batch(arena, jobs, want, m12, counts, sms)
        for j, jb in enumerate(jobs):
            o1, o2, n1, n2 = (int(jb[k]) for k in ("off1", "off2", "n1", "n2"))
            n_o, m_o = port.match(arena[o1:o1 + n1], arena[o2:o2 + n2], np.float32(0.8), best_lr)
            assert n_o == n1 and np.array_equal(m_o, want[j]), j
