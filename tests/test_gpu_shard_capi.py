"""plm_shard_*: the keyframe database / local map sharded over the GPUs of one box inside ONE process (the entry
point a C++ host such as the reference's MapHandler calls; include/plmatch.h).  Host buffers in and out, compared with
the oracle: flat-database matchNNR / knnMatch (config 5, mapHandler.cpp:3301-3409), map -> frame matchGrid and the
match fallback on the same vector (config 4, mapHandler.cpp:583-803).  n_devices = 1 runs on any GPU machine; 2 / 4 / 8
devices run where the machine has them (real peer-memory exchanges over NVLink between kernels running on different
GPUs) and skip elsewhere."""
import numpy as np
import pytest
import torch

import oracle
from helpers import oracle_grid, random_grid_case
from pl_inertial_slam_b200 import synth

pytestmark = pytest.mark.gpu
port = oracle.port


@pytest.fixture(scope="module", params=(1, 2, 4, 8), ids=lambda k: f"{k}gpu")
def devices(request, plm_lib):
    """The first k GPUs.  The device counts are fixed parameters, so every machine collects the same test ids; a count
    larger than the machine has is skipped."""
    k = request.param
    if torch.cuda.device_count() < k:
        pytest.skip(f"needs {k} GPUs")
    return list(range(k))


def test_flat_database_match_nnr(devices):
    from pl_inertial_slam_b200.database import ShardSet
    rng = np.random.default_rng(12)
    ss = ShardSet(devices, q_cap=512, rows_cap=70_000)
    for n_rows, tie in ((30_011, True), (70_000, False), (len(devices), True), (3, True)):
        db = synth.tie_stress_desc(rng, n_rows) if tie else synth.rand_desc(rng, n_rows)
        ss.upload(db)
        r = ss.ranges()
        assert r[0][0] == 0 and r[-1][1] == n_rows and all(a[1] == b[0] for a, b in zip(r, r[1:]))
        for n1 in (1, 127, 512, 513, 1300):        # slices of q_cap = 512, ragged tails
            q = synth.tie_stress_desc(rng, n1) if tie else synth.rand_desc(rng, n1)
            if not tie:
                k = n1 // 2
                q[:k] = synth.flip_bits(rng, db[rng.integers(0, n_rows, k)], 0.08)
            assert (ss.knn2(q) == port.knn2_packed(q, db)).all(), (n_rows, n1)
            stale = np.full(n1, -1, np.int32)
            stale[::7] = 5
            n_g, m_g = ss.match_nnr(q, 0.9, m12=stale)
            if n_rows >= 2:
                n_o, m_o = port.match_nnr(q, db, 0.9, m12=stale)
            else:                                   # a single train row: no second neighbour, nothing is accepted
                n_o, m_o = 0, stale
            assert n_g == n_o and (m_g == m_o).all(), (n_rows, n1)
    ss.upload(db[:0])
    with pytest.raises(RuntimeError):
        ss.match_nnr(q, 0.9)                       # empty train set: the reference throws
    assert ss.match_nnr(q[:0], 0.9)[0] == 0
    assert ss.launch_count > 0
    ss.close()


@pytest.mark.parametrize("is_lines", [False, True])
def test_map_to_frame_match_grid_and_fallback(devices, is_lines):
    from pl_inertial_slam_b200.database import ShardSet
    rng = np.random.default_rng(40 + int(is_lines))
    n1, n2 = (24_000, 600) if not is_lines else (9_000, 200)
    ss = ShardSet(devices, q_cap=1024, rows_cap=n1)
    for trial, tie in enumerate((False, True)):
        case = random_grid_case(rng, n1 - 13 * trial, n2, is_lines=is_lines, tie=tie, win=(3, 3, 3, 3), zero_len=3 if is_lines else 0)
        ss.upload(case["d1"], case["coords"])
        grid = (case["cell_start"], case["cell_items"], case["rows"], case["cols"])
        for best_lr in (True, False):
            stale = np.full(len(case["d1"]), -1, np.int32)
            stale[rng.choice(len(stale), 50, replace=False)] = rng.integers(0, n2, 50)
            n_o, m_o = oracle_grid(port, case, 0.9, best_lr, m12=stale)
            n_g, m_g = ss.match_grid(grid, case["d2"], case["win"], 0.9, best_lr, dirs2=case["dirs2"], m12=stale)
            assert n_g == n_o and (m_g == m_o).all(), (tie, best_lr)
            # fallback on the vector matchGrid just filled (mapHandler.cpp:645-650)
            n_o2, m_o2 = port.match(case["d1"], case["d2"], 0.9, best_lr, m12=m_o)
            n_g2, m_g2 = ss.match(case["d2"], 0.9, best_lr, m12=m_g)
            assert n_g2 == n_o2 and (m_g2 == m_o2).all(), (tie, best_lr)
    # sparse frame: one feature on the frame side must not raise
    n_g, m_g = ss.match(case["d2"][:1], 0.9, True)
    assert n_g == 0 and (m_g == -1).all()
    ss.close()


def test_argument_checks(plm_lib):
    import ctypes as C
    from pl_inertial_slam_b200 import _lib as L
    h = C.c_void_p()
    devs = (C.c_int * 2)(0, 0)
    assert plm_lib.plm_shard_create(devs, 2, 128, 1000, C.byref(h)) == L.PLM_E_INVALID     # shards must not share a GPU
    assert plm_lib.plm_shard_create(devs, 0, 128, 1000, C.byref(h)) == L.PLM_E_INVALID
    assert plm_lib.plm_shard_create(devs, 1, 0, 1000, C.byref(h)) == L.PLM_E_INVALID
