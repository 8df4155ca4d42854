"""Loop-closure batches on the tensor cores (K1c, `knn2_umma_pairs_kernel`): both directions of every keyframe pair of a
shared-query batch from one int8 product.

Every live job of such a batch shares one query range (one query keyframe against many keyframes, as
KeyframeDB.match_all and LoopClosureDB.match_candidates build it).  The kernel cuts each job into 128-row units, spreads
the (256-query group, unit) list over one CTA per SM -- so a job can be cut between CTAs (pieces) -- and writes the
partials that the integer list path's merge and mutual check consume.  Every comparison is bit for bit: counts and every
entry of the match arena, against `oracle.port.match` per pair or against the integer list kernels (`batch_umma` = 0).
"""
import numpy as np
import pytest

import oracle
from pl_inertial_slam_b200 import synth

pytestmark = pytest.mark.gpu
port = oracle.port
INT32_MIN = np.iinfo(np.int32).min


@pytest.fixture
def umma(plm_lib):
    def force(v):
        assert plm_lib.plm_set_option(b"batch_umma", v) == 0
    yield force
    plm_lib.plm_set_option(b"batch_umma", -1)


@pytest.fixture(scope="module")
def sms(plm_lib):
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def _noisy(rng, src, n):
    return synth.flip_bits(rng, src[rng.integers(0, len(src), n)], 0.1)


def _shared_batch(rng, q, sizes, stale=True):
    """Arena = query rows, then each job's train rows (half of them noisy copies of query rows); every job matches
    the query range against its own train range."""
    from pl_inertial_slam_b200 import _lib as L
    n1 = len(q)
    rows, jobs, off = [q], np.zeros(len(sizes), L.PAIR_JOB_DTYPE), n1
    for j, n2 in enumerate(sizes):
        d2 = synth.rand_desc(rng, n2)
        if n2 and n1:
            k = n2 // 2
            d2[:k] = _noisy(rng, q, k)
        rows.append(d2)
        jobs[j] = (0, off, j * n1, n1, n2)
        off += n2
    return np.ascontiguousarray(np.concatenate(rows)), jobs, _stale_in(rng, jobs, stale)


def _stale_in(rng, jobs, stale=True):
    n_m = int((jobs["off_m"] + jobs["n1"]).max()) if len(jobs) else 0
    m_in = np.full(n_m, -1, np.int32)
    if stale:
        for jb in jobs:
            sl = m_in[jb["off_m"]:jb["off_m"] + jb["n1"]]
            sl[::3] = rng.integers(0, max(int(jb["n2"]), 1), len(sl[::3]))
    return m_in


def _run(umma, v, arena, jobs, nnr, best_lr, m_in):
    from pl_inertial_slam_b200 import replay
    umma(v)
    b = replay.MatchBatch()
    b.set_match(arena, jobs, nnr, best_lr, m_in)
    b.run()
    out = b.fetch()
    b.close()
    return out


def _check_oracle(arena, jobs, nnr, best_lr, m_in, m12, counts):
    for j, jb in enumerate(jobs):
        o1, o2, om, n1, n2 = (int(jb[k]) for k in ("off1", "off2", "off_m", "n1", "n2"))
        got, mi = m12[om:om + n1], m_in[om:om + n1]
        if n2 < 2 or (best_lr and n1 < 2):
            assert counts[j] == INT32_MIN and np.array_equal(got, mi), j
            continue
        n_o, m_o = port.match(arena[o1:o1 + n1], arena[o2:o2 + n2], np.float32(nnr), best_lr, m12=mi)
        assert counts[j] == n_o, (j, counts[j], n_o)
        assert np.array_equal(got, m_o), (j, np.flatnonzero(got != m_o)[:8])


def _check_both(umma, arena, jobs, nnr, best_lr, m_in):
    m12, counts = _run(umma, 1, arena, jobs, nnr, best_lr, m_in)
    _check_oracle(arena, jobs, nnr, best_lr, m_in, m12, counts)
    m0, c0 = _run(umma, 0, arena, jobs, nnr, best_lr, m_in)
    assert np.array_equal(counts, c0) and np.array_equal(m12, m0)


JOB_SIZES = [0, 1, 2, 3, 127, 128, 129, 800, 5000]


@pytest.mark.parametrize("n1", [2, 3, 255, 256, 257, 800, 1000])
@pytest.mark.parametrize("best_lr", [True, False])
@pytest.mark.parametrize("nnr", [0.9, 0.75])
def test_forced_tensor_path_against_oracle(umma, n1, best_lr, nnr):
    """Ragged query groups and job sizes 0 .. 5000 (empty and 1-row jobs are skipped), stale IN entries."""
    rng = np.random.default_rng(1000 + n1 + (7 if best_lr else 0) + int(nnr * 100))
    q = synth.rand_desc(rng, n1)
    arena, jobs, m_in = _shared_batch(rng, q, JOB_SIZES)
    _check_both(umma, arena, jobs, nnr, best_lr, m_in)


@pytest.mark.parametrize("nq,kf_rows", [(800, 800), (200, 200)])
def test_realistic_size_against_integer_path(umma, nq, kf_rows):
    """800-point query x 2000 keyframes x 800 points, and 200 lines x 2000 x 200: tensor path == integer list path."""
    rng = np.random.default_rng(2000 + nq)
    q = synth.rand_desc(rng, nq)
    arena, jobs, m_in = _shared_batch(rng, q, [kf_rows] * 2000, stale=False)
    for best_lr in (True, False):
        m1, c1 = _run(umma, 1, arena, jobs, 0.9, best_lr, m_in)
        m0, c0 = _run(umma, 0, arena, jobs, 0.9, best_lr, m_in)
        assert np.array_equal(c1, c0) and np.array_equal(m1, m0)
        assert (c1 > 0).mean() > 0.9
    for j in range(0, 2000, 397):  # a few pairs against the oracle as well
        _check_oracle(arena, jobs[j:j + 1], 0.9, True, m_in, *_run(umma, 1, arena, jobs[j:j + 1], 0.9, True, m_in))


def test_ties(umma):
    """Tie-stress descriptors on both sides; duplicate train rows far apart in one job (lowest train index wins);
    duplicate query rows in different groups (lowest query index wins in direction 21); all-zero and all-ones
    descriptors (distance 256 between them)."""
    from pl_inertial_slam_b200 import _lib as L
    rng = np.random.default_rng(3000)
    q = synth.tie_stress_desc(rng, 800)
    q[600:700] = q[0:100]                                      # groups 0 and 2
    q[700] = 0
    q[701] = 255
    parts = [synth.tie_stress_desc(rng, 900), synth.rand_desc(rng, 5000), np.zeros((300, 32), np.uint8),
             np.full((300, 32), 255, np.uint8), q[::-1].copy()]
    parts[1][:200] = _noisy(rng, q, 200)
    parts[1][4800:5000] = parts[1][:200]                       # far apart in one job
    parts[2][::2] = 255
    arena = np.ascontiguousarray(np.concatenate([q] + parts))
    jobs, off = np.zeros(len(parts), L.PAIR_JOB_DTYPE), len(q)
    for j, p in enumerate(parts):
        jobs[j] = (0, off, j * len(q), len(q), len(p))
        off += len(p)
    m_in = _stale_in(rng, jobs)
    for best_lr in (True, False):
        _check_both(umma, arena, jobs, 0.9, best_lr, m_in)


def test_pieces(umma, sms):
    """A job longer than one CTA's share (its 12 task has many slots), and many ragged jobs whose share boundaries fall
    inside jobs and across query groups."""
    rng = np.random.default_rng(4000)
    q = synth.rand_desc(rng, 300)                              # 2 groups
    arena, jobs, m_in = _shared_batch(rng, q, [sms * 3 * 128 + 50])
    _check_both(umma, arena, jobs, 0.9, True, m_in)
    q = synth.rand_desc(rng, 600)                              # 3 groups
    sizes = list(rng.integers(50, 3000, 60)) + [2, 129, 7000]
    arena, jobs, m_in = _shared_batch(rng, q, sizes)
    for best_lr in (True, False):
        _check_both(umma, arena, jobs, 0.75, best_lr, m_in)


def test_job_layout(umma):
    """Unsorted, overlapping and repeated train ranges, and a job whose train range is the query range itself."""
    from pl_inertial_slam_b200 import _lib as L
    rng = np.random.default_rng(5000)
    n1 = 500
    q = synth.rand_desc(rng, n1)
    pool = np.concatenate([_noisy(rng, q, 3000), synth.rand_desc(rng, 3000)])
    rng.shuffle(pool)
    arena = np.ascontiguousarray(np.concatenate([q, pool]))
    ranges = [(4000, 900), (n1, 2000), (1500, 1200), (n1, 2000), (5000, 1500), (0, n1), (200, 700), (n1 + 100, 129)]
    jobs = np.zeros(len(ranges), L.PAIR_JOB_DTYPE)
    for j, (o2, n2) in enumerate(ranges):
        jobs[j] = (0, o2, j * n1, n1, n2)
    m_in = _stale_in(rng, jobs)
    for best_lr in (True, False):
        _check_both(umma, arena, jobs, 0.9, best_lr, m_in)


def test_repeated_match_all_rewrites_the_query(umma):
    """Back-to-back KeyframeDB.match_all calls with different query keyframes (and sizes) in the query slot: each one
    equals the oracle, nothing of an earlier query survives."""
    from pl_inertial_slam_b200.database import KeyframeDB
    rng = np.random.default_rng(6000)
    kf_sizes = rng.integers(100, 900, 40)
    kf_start = np.concatenate([[0], np.cumsum(kf_sizes)])
    base = synth.rand_desc(rng, 900)
    rows = np.concatenate([_noisy(rng, base, int(n)) for n in kf_sizes])
    db = KeyframeDB(rows, kf_start, device=0, q_cap=1024)
    umma(1)
    for i, nq in enumerate([800, 800, 257, 800, 1000]):
        q = _noisy(rng, base, nq)
        counts, m12 = db.match_all(q, 0.9, True, want_matches=True)
        for k in range(len(kf_sizes)):
            n_o, m_o = port.match(q, rows[kf_start[k]:kf_start[k + 1]], np.float32(0.9), True)
            assert counts[k] == n_o and np.array_equal(m12[k], m_o), (i, k)


def test_keyframe_db_automatic_selection(umma):
    """KeyframeDB.match_all with the automatic choice at a loop-closure shape: equal to the integer path."""
    from pl_inertial_slam_b200.database import KeyframeDB
    rng = np.random.default_rng(7000)
    base = synth.rand_desc(rng, 800)
    rows = _noisy(rng, base, 300 * 800)
    kf_start = np.arange(301) * 800
    db = KeyframeDB(rows, kf_start, device=0, q_cap=800)
    q = _noisy(rng, base, 800)
    for best_lr in (True, False):
        umma(-1)
        db._prepared = None                                    # the path is chosen when the job tables are built
        c_auto, m_auto = db.match_all(q, 0.9, best_lr, want_matches=True)
        umma(0)
        db._prepared = None
        c0, m0 = db.match_all(q, 0.9, best_lr, want_matches=True)
        assert np.array_equal(c_auto, c0) and np.array_equal(m_auto, m0)


def test_loopdb_candidates_automatic_selection(umma):
    """LoopClosureDB.match_candidates on the tensor path (one batch per kind) and with the automatic choice: each pair
    equals plm_match."""
    from pl_inertial_slam_b200 import bow as B
    from pl_inertial_slam_b200 import matching as M
    rng = np.random.default_rng(8000)
    vp = B.Vocabulary.from_flat(synth.make_vocabulary(synth.SEED0 + 170, k=10, L=3))
    vl = B.Vocabulary.from_flat(synth.make_vocabulary(synth.SEED0 + 171, k=6, L=3))
    base_p, base_l = synth.rand_desc(rng, 800), synth.rand_desc(rng, 200)
    kfs = [(_noisy(rng, base_p, 800), _noisy(rng, base_l, 200)) for _ in range(61)]
    db = B.LoopClosureDB(vp, vl, "PL")
    for i, (p, l) in enumerate(kfs):
        db.insertKFBowVectorPL(B.KeyFrameBow(i, p, l, rng.random((len(p), 2)) * 640, rng.random((len(l), 2)) * 480))
    for v in (1, -1):
        umma(v)
        got = db.match_candidates(0, list(range(1, 61)))
        for k, g in zip(range(1, 61), got):
            for s, key in ((0, "pt"), (1, "ls")):
                m12 = []
                n = M.match(kfs[0][s], kfs[k][s], M.Config.minRatio12P if s == 0 else M.Config.minRatio12L, m12)
                assert g["common_" + key] == n and np.array_equal(g["matches_" + key], np.array(m12, np.int32)), (v, k, key)


@pytest.mark.parametrize("best_lr", [True, False])
def test_launch_counts(umma, best_lr):
    """A run is the same number of launches on both paths: 3 with best_lr (kernel, merge, mutual check), 2 without."""
    from pl_inertial_slam_b200 import replay
    from pl_inertial_slam_b200.matching import Context
    rng = np.random.default_rng(9000)
    arena, jobs, m_in = _shared_batch(rng, synth.rand_desc(rng, 800), [800] * 50)
    ctx = Context(0)
    for v in (1, 0):
        umma(v)
        b = replay.MatchBatch(ctx)
        b.set_match(arena, jobs, 0.9, best_lr, m_in)
        n0 = ctx.launch_count
        b.run()
        b.fetch_counts()
        assert ctx.launch_count - n0 == (3 if best_lr else 2)
        b.close()
