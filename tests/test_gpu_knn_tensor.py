"""Parity of the tensor-core brute-force kernel (knn2 variant 7, `knn2_umma_kernel`).

The kernel computes every Hamming distance as |q| + dot(+-1 query bytes, 0/1 train bytes) with int8 tcgen05 MMAs and
keeps the blocked top-2 of the integer kernels, so its keys must equal the oracle's bit for bit: ragged query groups
(256 queries per CTA, two M = 128 tiles) and ragged train units (128 rows), a nonzero idx_base, ties, duplicates far
apart, and the extreme descriptors (all zeros / all ones) that give the largest |q| and dot values.  Variant 7 is forced
so that small shapes take it too; automatic mode picks it for >= 65 536 train rows and >= 256 queries.
"""
import numpy as np
import pytest

import oracle
from pl_inertial_slam_b200 import synth

pytestmark = pytest.mark.gpu
port = oracle.port


@pytest.fixture(scope="module")
def M(plm_lib):
    from pl_inertial_slam_b200 import matching
    return matching


@pytest.fixture
def variant(plm_lib):
    """Force a knn variant for one test, automatic mode afterwards."""
    def force(v):
        assert plm_lib.plm_set_option(b"knn_variant", v) == 0
    yield force
    plm_lib.plm_set_option(b"knn_variant", -1)


def _case(seed, n1, n2, tie=False):
    rng = np.random.default_rng(seed)
    if tie:
        return synth.tie_stress_desc(rng, n1), synth.tie_stress_desc(rng, n2)
    d1, d2 = synth.rand_desc(rng, n1), synth.rand_desc(rng, n2)
    k = n1 * 2 // 3
    rows = rng.choice(n1, k, replace=False)
    d1[rows] = synth.flip_bits(rng, d2[rng.integers(0, n2, k)], 0.08)
    src = rng.integers(0, n2 // 2, min(64, n2 // 2))   # exact duplicates far apart: the lower index must win
    d2[n2 - 1 - np.arange(len(src))] = d2[src]
    return d1, d2


def _check(got, want):
    bad = np.flatnonzero((got != want).any(1))
    assert bad.size == 0, (bad[:8], got[bad[:4]], want[bad[:4]])


@pytest.mark.parametrize("n1", [1, 127, 128, 129, 255, 257, 4100])
def test_ragged_query_groups(M, variant, n1):
    d1, d2 = _case(31 + n1, n1, 70003)
    variant(7)
    _check(M.knn2(d1, d2, idx_base=5), port.knn2_packed(d1, d2, idx_base=5))


@pytest.mark.parametrize("n2", [65535, 65536, 65537, 70003, 140001, 300, 2])
def test_ragged_train_units(M, variant, n2):
    d1, d2 = _case(77 + n2, 300, n2)
    variant(7)
    _check(M.knn2(d1, d2, idx_base=12345), port.knn2_packed(d1, d2, idx_base=12345))


@pytest.mark.parametrize("n1,n2", [(513, 70000), (1024, 65536)])
def test_tie_stress(M, variant, n1, n2):
    d1, d2 = _case(5 + n1, n1, n2, tie=True)
    variant(7)
    _check(M.knn2(d1, d2, idx_base=3), port.knn2_packed(d1, d2, idx_base=3))


def test_extreme_descriptors(M, variant):
    """All-zero and all-ones rows on both sides: |q| = 0 / 256, dot = 0 / -256 / +256."""
    rng = np.random.default_rng(2024)
    d1, d2 = synth.rand_desc(rng, 600), synth.rand_desc(rng, 70000)
    d1[0::4] = 0
    d1[1::4] = 255
    d2[100:110] = 0
    d2[60000:60005] = 0
    d2[200:203] = 255
    d2[69990:] = 255
    variant(7)
    got = M.knn2(d1, d2)
    _check(got, port.knn2_packed(d1, d2))
    assert (got[0::4, 0] == np.uint64(100)).all() and (got[1::4, 0] == np.uint64(200)).all()


def test_match_nnr(M, variant):
    d1, d2 = _case(909, 2000, 90001)
    n_o, m_o = port.match_nnr(d1, d2, 0.8)
    variant(7)
    m_g = np.full(len(d1), -1, np.int32)
    assert M.matchNNR(d1, d2, 0.8, m_g) == n_o
    assert (m_g == m_o).all()


def test_same_keys_as_integer_kernel(M, variant):
    """Forced variant 7 and forced variant 3 on the same inputs: identical keys (beyond what the oracle can check
    quickly: 3000 queries x 400 000 rows)."""
    d1, d2 = _case(4242, 3000, 400_000)
    variant(3)
    k3 = M.knn2(d1, d2, idx_base=77)
    variant(7)
    k7 = M.knn2(d1, d2, idx_base=77)
    _check(k7, k3)


def test_launch_count_unchanged(plm_lib, variant):
    """One plm_dev_knn2 call is the slice kernel and the merge kernel, on either path."""
    import torch
    from pl_inertial_slam_b200.database import DeviceOps
    rng = np.random.default_rng(8)
    ops = DeviceOps(0)
    q = torch.from_numpy(synth.rand_desc(rng, 2048)).cuda()
    db = torch.from_numpy(synth.rand_desc(rng, 100_000)).cuda()
    counts, outs = [], []
    for v in (3, -1):   # the integer kernel, then automatic mode (the tensor-core kernel at this shape)
        variant(v)
        n0 = ops.ctx.launch_count
        outs.append(ops.knn2(q, db, idx_base=9))
        torch.cuda.synchronize()
        counts.append(ops.ctx.launch_count - n0)
    assert counts == [2, 2]
    assert torch.equal(outs[0], outs[1])


def test_full_size_shard_merge_of_halves(M, variant):
    """2 M-row shard: the result equals the merge of the results over two halves (idx_base carries the global index),
    a planted duplicate is found at distance 0 with the lowest index, 64 sampled queries equal the oracle."""
    rng = np.random.default_rng(321)
    n2, n1 = 2_000_000, 1500
    d2 = synth.rand_desc(rng, n2)
    d1 = synth.rand_desc(rng, n1)
    d1[:100] = d2[rng.integers(1000, n2, 100)]
    d2[7] = d1[3]
    d2[900_001] = d1[3]
    variant(7)
    full = M.knn2(d1, d2)
    h = n2 // 2 + 3
    lo, hi = M.knn2(d1, d2[:h]), M.knn2(d1, d2[h:], idx_base=h)
    merged = np.sort(np.concatenate([lo, hi], 1), 1)[:, :2]
    _check(full, merged)
    assert (full[:100, 0] >> np.uint64(32) == 0).all()
    assert full[3, 0] == np.uint64(7) and (full[3, 1] >> np.uint64(32)) == 0 and (full[3, 1] & np.uint64(0xFFFFFFFF)) > 7
    sample = rng.choice(n1, 64, replace=False)
    _check(full[sample], port.knn2_packed(d1[sample], d2))
