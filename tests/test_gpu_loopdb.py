"""Loop-closure keyframe database on the device (plm_loopdb_*, bow.LoopClosureDB; src/mapHandler.cpp:3116-3237,
3325-3400).

GPU (-m gpu): insert / cull sequences in modes P, L and PL bit for bit against bow.BowConfusion and the oracle's
DBoW2 restatement; stored vectors; growth of the device arenas; untouched entries of a row; per-insert cost independent
of the database size; isLoopClosure's matching against drivers.loopClosureMatch and the oracle.
CPU: argument validation, reported before any CUDA call."""
import ctypes as C

import numpy as np
import pytest

import oracle
from pl_inertial_slam_b200 import synth

port = oracle.port


def bits(a):
    return np.ascontiguousarray(a, np.float64).view(np.uint64)


def assert_same(got, want):
    """NaN entries as NaN (x86 and the GPU produce different NaN bit patterns), every other entry by bit pattern."""
    got, want = np.asarray(got, np.float64), np.asarray(want, np.float64)
    assert got.shape == want.shape
    nan = np.isnan(want)
    assert np.array_equal(np.isnan(got), nan)
    assert np.array_equal(bits(got)[~nan], bits(want)[~nan])


@pytest.fixture(scope="module")
def vocs():
    fp = synth.make_vocabulary(synth.SEED0 + 170, k=10, L=3)
    fl = synth.make_vocabulary(synth.SEED0 + 171, k=6, L=3)
    return fp, fl


_CTX = []   # the context outlives every vocabulary / database built on it, also when those end up in a reference cycle


@pytest.fixture(scope="module")
def dev(vocs):
    from pl_inertial_slam_b200 import bow as B
    from pl_inertial_slam_b200.matching import Context
    if not _CTX:
        _CTX.append(Context(0))
    ctx = _CTX[0]
    return ctx, B.Vocabulary.from_flat(vocs[0], ctx), B.Vocabulary.from_flat(vocs[1], ctx)


def make_sequence(vocs, n=40, seed=5):
    """(kf_idx, points, lines, point xy, line midpoints) with sizes 0 / 1 / 2 / 300 / 8192 in both sets, a revisit,
    gaps in kf_idx and a keyframe without lines."""
    fp, fl = vocs
    rng = np.random.default_rng(seed)
    sizes_p = {0: 300, 1: 0, 2: 1, 3: 2, 6: 8192, 12: 0}
    sizes_l = {0: 300, 1: 1, 2: 0, 3: 2, 8: 8192, 10: 0, 13: 0}
    seq, idx = [], 0
    for i in range(n):
        n_p = sizes_p.get(i, int(rng.integers(40, 260)))
        n_l = sizes_l.get(i, int(rng.integers(10, 90)))
        p = synth.vocabulary_features(1000 + i, fp, n_p)
        l = synth.vocabulary_features(2000 + i, fl, n_l)
        if i == 15:                                        # a revisit of keyframe 4
            p, l = seq[4][1].copy(), seq[4][2].copy()
        seq.append((idx, p, l, rng.uniform(0, 700, (len(p), 2)), rng.uniform(0, 450, (len(l), 2))))
        idx += 1 + (2 if i in (3, 11, 26) else 0)         # gaps
    return seq


CULL_NOW = {7}          # culled right after its insert
CULL_LATER = {3: 20}    # position -> culled after the insert at this position


def run(db, seq, mode, culls=True):
    from pl_inertial_slam_b200 import bow as B
    for pos, (idx, p, l, pt, ls) in enumerate(seq):
        getattr(db, "insertKFBowVector" + mode)(B.KeyFrameBow(idx, p, l, pt, ls))
        if not culls:
            continue
        for c in [pos] if pos in CULL_NOW else []:
            _cull(db, seq[c][0])
        for c, after in CULL_LATER.items():
            if after == pos:
                _cull(db, seq[c][0])


def _cull(db, idx):
    if hasattr(db, "cull"):
        db.cull(idx)
    else:
        db.map_keyframes[idx] = None


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["P", "L", "PL"])
def test_insert_parity_with_bow_confusion(vocs, dev, mode):
    from pl_inertial_slam_b200 import bow as B
    ctx, vp, vl = dev
    seq = make_sequence(vocs)
    ref = B.BowConfusion(vp, vl, ctx)
    db = B.LoopClosureDB(vp, vl, mode)
    run(ref, seq, mode)
    run(db, seq, mode)
    assert_same(db.conf_matrix, ref.conf_matrix)
    assert [k is None for k in db.map_keyframes] == [k is None for k in ref.map_keyframes]
    if mode == "PL":
        assert np.isnan(db.conf_matrix[seq[10][0]]).any()         # the keyframe without lines blends to NaN
    if mode == "P":
        assert db.conf_matrix[seq[15][0], seq[4][0]] > 0.99       # the revisit scores like the keyframe itself
    assert len(db) == len(seq)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["P", "PL"])
def test_insert_matches_the_oracle(vocs, dev, mode):
    """A short sequence against oracle.port.bow_transform / bow_score and the blend formula."""
    from pl_inertial_slam_b200 import bow as B
    fp, fl = vocs
    ctx, vp, vl = dev
    seq = make_sequence(vocs, n=9, seed=8)
    db = B.LoopClosureDB(vp, vl, mode)
    run(db, seq, mode, culls=False)
    db.cull(seq[2][0])
    idx, p, l, pt, ls = seq[-1]
    seq = seq + [(idx + 2, p[::-1].copy(), l, pt, ls)]
    getattr(db, "insertKFBowVector" + mode)(B.KeyFrameBow(*seq[-1]))
    n = seq[-1][0] + 1
    want = np.zeros((n, n))
    bp = [port.bow_transform(fp, s[1]) for s in seq]
    bl = [port.bow_transform(fl, s[2]) for s in seq]
    for i, (a, _, _, pt, ls) in enumerate(seq):
        for j in range(i + 1):
            if i == len(seq) - 1 and j == 2:               # culled before the last insert
                continue
            sp, sl = port.bow_score(bp[i], bp[j]), port.bow_score(bl[i], bl[j])
            if mode == "P":
                s = sp
            else:
                n_pt, n_ls = len(pt), len(ls)
                std_pt = B.vector_stdv(pt[:, 0]) + B.vector_stdv(pt[:, 1])
                std_ls = B.vector_stdv(ls[:, 0]) + B.vector_stdv(ls[:, 1])
                with np.errstate(divide="ignore", invalid="ignore"):
                    s = 0.0
                    s += (np.float64(sp) * n_pt + np.float64(sl) * n_ls) / np.float64(n_pt + n_ls)
                    s += (np.float64(sp) * std_pt + np.float64(sl) * std_ls) / np.float64(std_ls + std_pt)
            b = seq[j][0]
            want[a, b] = want[b, a] = s
    assert_same(db.conf_matrix, want)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["P", "L", "PL"])
def test_stored_vectors(vocs, dev, mode):
    from pl_inertial_slam_b200 import _lib as L
    from pl_inertial_slam_b200 import bow as B
    fp, fl = vocs
    ctx, vp, vl = dev
    seq = make_sequence(vocs)
    db = B.LoopClosureDB(vp, vl, mode)
    run(db, seq, mode)
    culled = {seq[c][0] for c in list(CULL_NOW) + list(CULL_LATER)}
    for idx, p, l, _, _ in seq:
        for which, voc, d in (("P", fp, p), ("L", fl, l)):
            if which not in mode:
                continue
            if idx in culled:
                with pytest.raises(L.PlmError) as e:
                    db.bow_vector(idx, which)
                assert e.value.status == L.PLM_E_INVALID
                continue
            ids, vals = db.bow_vector(idx, which)
            wi, wv = port.bow_transform(voc, d)
            assert np.array_equal(ids, wi), (idx, which)
            assert np.array_equal(bits(vals), bits(wv)), (idx, which)


@pytest.mark.gpu
def test_growth_gives_the_same_rows_and_vectors(vocs, dev):
    from pl_inertial_slam_b200 import bow as B
    ctx, vp, vl = dev
    seq = make_sequence(vocs, n=30, seed=11)
    tiny = B.LoopClosureDB(vp, vl, "PL", capacity=1)        # 1 slot, 512 rows, 256 entries per vocabulary at first
    roomy = B.LoopClosureDB(vp, vl, "PL", capacity=256)
    run(tiny, seq, "PL")
    run(roomy, seq, "PL")
    assert np.array_equal(bits(tiny.conf_matrix), bits(roomy.conf_matrix))
    for idx, *_ in seq:
        if tiny.map_keyframes[idx] is None:
            continue
        for which in "PL":
            a, b = tiny.bow_vector(idx, which), roomy.bow_vector(idx, which)
            assert np.array_equal(a[0], b[0]) and np.array_equal(bits(a[1]), bits(b[1]))


@pytest.mark.gpu
def test_untouched_entries_keep_their_value(vocs, dev):
    from pl_inertial_slam_b200 import _lib as L
    from pl_inertial_slam_b200 import bow as B
    fp, _ = vocs
    ctx, vp, vl = dev
    db = B.LoopClosureDB(vp, vl, "P")
    present = [0, 1, 3, 4, 7, 8]
    for i in present:
        db.insertKFBowVectorP(B.KeyFrameBow(i, synth.vocabulary_features(300 + i, fp, 120)))
    db.cull(3)
    db.cull(8)
    idx = 11
    d = synth.vocabulary_features(400, fp, 150)
    sentinel = np.float64(-1234.5)
    row = np.full(idx + 3, sentinel)
    st = db.lib.plm_loopdb_insert(db._h, idx, d.ctypes.data_as(L.u8p), len(d), 32, None, 0, 32, None,
                                  row.ctypes.data_as(L.f64p))
    assert st == L.PLM_OK
    live = {0, 1, 4, 7}
    for j in range(len(row)):
        assert (row[j] == sentinel) == (j not in live and j != idx), j
    # an insert with a kf_idx that is not larger than every earlier one, and a cull of an absent keyframe
    assert db.lib.plm_loopdb_insert(db._h, idx, d.ctypes.data_as(L.u8p), len(d), 32, None, 0, 32, None,
                                    row.ctypes.data_as(L.f64p)) == L.PLM_E_INVALID
    assert db.lib.plm_loopdb_cull(db._h, 5) == L.PLM_E_INVALID
    assert db.lib.plm_loopdb_cull(db._h, 3) == L.PLM_E_INVALID            # already culled
    assert db.lib.plm_loopdb_cull(db._h, 40) == L.PLM_E_INVALID
    assert len(db) == len(present) + 1


@pytest.mark.gpu
def test_failed_insert_leaves_the_database_unchanged(vocs, dev):
    from pl_inertial_slam_b200 import _lib as L
    from pl_inertial_slam_b200 import bow as B
    fp, fl = vocs
    ctx, vp, vl = dev
    seq = make_sequence(vocs, n=6, seed=3)
    a, b = B.LoopClosureDB(vp, vl, "PL"), B.LoopClosureDB(vp, vl, "PL")
    run(a, seq[:3], "PL", culls=False)
    run(b, seq[:3], "PL", culls=False)
    h2d, n = a.h2d_bytes, len(a)
    big = synth.vocabulary_features(9, fp, 8193)
    with pytest.raises(L.PlmError) as e:
        a.insertKFBowVectorPL(B.KeyFrameBow(seq[3][0], big, seq[3][2], np.zeros((8193, 2)), seq[3][4]))
    assert e.value.status == L.PLM_E_UNSUPPORTED
    with pytest.raises(L.PlmError) as e:
        a.insertKFBowVectorPL(B.KeyFrameBow(seq[1][0], *seq[3][1:]))
    assert e.value.status == L.PLM_E_INVALID
    with pytest.raises(ValueError):
        a.insertKFBowVectorP(B.KeyFrameBow(seq[3][0], seq[3][1]))
    assert a.h2d_bytes == h2d and len(a) == n and a.conf_matrix.shape == b.conf_matrix.shape
    run(a, seq[3:], "PL", culls=False)
    run(b, seq[3:], "PL", culls=False)
    assert_same(a.conf_matrix, b.conf_matrix)


@pytest.mark.gpu
@pytest.mark.parametrize("mode,launches", [("P", 2), ("L", 2), ("PL", 3)])
def test_per_insert_cost_is_independent_of_the_database_size(vocs, dev, mode, launches):
    """The launches and the host -> device bytes of an insert are the same at the 5th and the 40th keyframe: the
    earlier keyframes never cross PCIe again."""
    from pl_inertial_slam_b200 import bow as B
    ctx, vp, vl = dev
    seq = make_sequence(vocs, seed=21)
    db = B.LoopClosureDB(vp, vl, mode, capacity=1)           # growth on the way must not add copies from the host
    per_launch, per_bytes = [], []
    for pos, (idx, p, l, pt, ls) in enumerate(seq):
        l0, b0 = ctx.launch_count, db.h2d_bytes
        getattr(db, "insertKFBowVector" + mode)(B.KeyFrameBow(idx, p, l, pt, ls))
        if pos >= 4:
            per_launch.append(ctx.launch_count - l0)
            per_bytes.append(db.h2d_bytes - b0 - 32 * (len(p) + len(l)))
        if pos == 7:
            db.cull(idx)
    assert set(per_launch) == {launches}
    assert set(per_bytes) == {0}


def _match_keyframes(n_kf=8, seed=4):
    """Descriptor sets where kf 1.. share noisy copies of kf 0's rows; kf 5 has 1 line, kf 6 no lines, kf 7 one point."""
    rng = np.random.default_rng(seed)
    base_p, base_l = synth.rand_desc(rng, 400), synth.rand_desc(rng, 120)
    kfs = []
    for i in range(n_kf):
        n_p, n_l = int(rng.integers(200, 400)), int(rng.integers(40, 120))
        p = synth.rand_desc(rng, n_p)
        l = synth.rand_desc(rng, n_l)
        k = n_p // 2 if i else n_p
        p[:k] = synth.flip_bits(rng, base_p[rng.choice(400, k, replace=False)], 0.05 * (i % 3))
        kl = n_l // 2 if i else n_l
        l[:kl] = synth.flip_bits(rng, base_l[rng.choice(120, kl, replace=False)], 0.05 * (i % 3))
        kfs.append((p, l))
    kfs[5] = (kfs[5][0], kfs[5][1][:1].copy())
    kfs[6] = (kfs[6][0], np.zeros((0, 32), np.uint8))
    kfs[7] = (kfs[7][0][:1].copy(), kfs[7][1])
    return kfs


def _same_dict(got, want):
    assert got["common_pt"] == want["common_pt"] and got["common_ls"] == want["common_ls"]
    assert np.array_equal(got["matches_pt"], want["matches_pt"])
    assert np.array_equal(got["matches_ls"], want["matches_ls"])
    assert got["inl_ratio_pt"] == want["inl_ratio_pt"] and got["inl_ratio_ls"] == want["inl_ratio_ls"]
    assert got["inl_ratio_condition"] == want["inl_ratio_condition"]


@pytest.mark.gpu
@pytest.mark.parametrize("nnr_l", [0.9, 0.8])
def test_loop_closure_matching(vocs, dev, nnr_l):
    from pl_inertial_slam_b200 import _lib as L
    from pl_inertial_slam_b200 import bow as B
    from pl_inertial_slam_b200 import drivers as D
    from pl_inertial_slam_b200 import matching as M
    ctx, vp, vl = dev
    kfs = _match_keyframes()
    db = B.LoopClosureDB(vp, vl, "P", capacity=2)
    for i, (p, l) in enumerate(kfs):
        db.insertKFBowVectorP(B.KeyFrameBow(2 * i, p, l))
    db.insertKFBowVectorP(B.KeyFrameBow(100, kfs[1][0], kfs[1][1]))
    db.cull(100)
    old = M.Config.minRatio12L
    M.Config.minRatio12L = nnr_l
    try:
        for a in range(len(kfs)):
            cands = [b for b in range(len(kfs)) if b != a]
            got = db.match_candidates(2 * a, [2 * b for b in cands])
            for b, g in zip(cands, got):
                want = D.loopClosureMatch(kfs[a][0], kfs[b][0], kfs[a][1], kfs[b][1])
                _same_dict(g, want)
                _same_dict(db.isLoopClosure(2 * a, 2 * b), want)
                for s, nnr, key in ((0, M.Config.minRatio12P, "pt"), (1, nnr_l, "ls")):
                    d0, d1 = kfs[a][s], kfs[b][s]
                    if len(d0) >= 2 and len(d1) >= 2:
                        n, m12 = port.match(d0, d1, np.float32(nnr), True)
                        assert g["common_" + key] == n and np.array_equal(g["matches_" + key], m12)
        assert any(d["inl_ratio_condition"] for d in db.match_candidates(0, [2, 4, 6]))
    finally:
        M.Config.minRatio12L = old
    with pytest.raises(L.PlmError) as e:
        db.match_candidates(0, [2, 100])                      # a culled candidate
    assert e.value.status == L.PLM_E_INVALID
    assert db.match_candidates(0, []) == []


def test_argument_validation_needs_no_gpu(plm_lib):
    """Precondition failures are reported before any CUDA call (insert / cull with a bad index on a live database:
    test_untouched_entries_keep_their_value)."""
    from pl_inertial_slam_b200 import _lib as L
    h = C.c_void_p()
    assert plm_lib.plm_loopdb_create(None, None, 0, 0, None) == L.PLM_E_INVALID
    assert plm_lib.plm_loopdb_create(None, None, 3, 0, C.byref(h)) == L.PLM_E_INVALID
    assert plm_lib.plm_loopdb_create(None, None, -1, 0, C.byref(h)) == L.PLM_E_INVALID
    for mode in (0, 1, 2):
        assert plm_lib.plm_loopdb_create(None, None, mode, 0, C.byref(h)) == L.PLM_E_INVALID
    assert not h.value
    d = np.zeros((4, 32), np.uint8)
    row = np.zeros(8)
    assert plm_lib.plm_loopdb_insert(None, 0, d.ctypes.data_as(L.u8p), 4, 32, None, 0, 32, None,
                                     row.ctypes.data_as(L.f64p)) == L.PLM_E_INVALID
    assert plm_lib.plm_loopdb_cull(None, 0) == L.PLM_E_INVALID
    n = C.c_int32(0)
    assert plm_lib.plm_loopdb_bow(None, 0, 0, None, None, C.byref(n)) == L.PLM_E_INVALID
    c = np.zeros(1, np.int32)
    k1 = np.zeros(1, np.int32)
    assert plm_lib.plm_loopdb_match(None, 0, k1.ctypes.data_as(L.i32p), 1, 0.9, 0.9, 1, c.ctypes.data_as(L.i32p),
                                    c.ctypes.data_as(L.i32p), None, None) == L.PLM_E_INVALID
    assert plm_lib.plm_loopdb_destroy(None) == L.PLM_OK
    assert plm_lib.plm_loopdb_size(None) == 0
    assert plm_lib.plm_loopdb_h2d_bytes(None) == 0 and plm_lib.plm_loopdb_d2h_bytes(None) == 0
