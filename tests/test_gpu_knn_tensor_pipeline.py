"""Pipeline edges of the warp-specialised tensor-core brute force (knn2 variant 7, `knn2_umma_kernel`).

The kernel streams packed train units through an 8-deep ring, expands them into 3 B tiles and alternates 2
accumulator buffers, all on mbarrier phases that run on across the segments (query groups) of a CTA's share of the
(group, 128-row unit) work list.  These cases put the ends of shares and segments at every position of those rings:
shares of 1 .. ring depth + 1 units, group boundaries at every ring phase, many short segments per CTA with a ragged
unit inside the share, a bound (`gthr`) that drops early, and back-to-back launches.  Every result is compared bit
for bit with the oracle or with the integer kernel (variant 3).
"""
import numpy as np
import pytest

import oracle
from pl_inertial_slam_b200 import synth

pytestmark = pytest.mark.gpu
port = oracle.port

RING = 8        # KNN_UMMA_STAGES
B_TILES = 3     # KNN_UMMA_BSTAGES
ROWS = 128      # train rows per unit
GROUP = 256     # queries per group


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


def _case(seed, n1, n2):
    rng = np.random.default_rng(seed)
    d1, d2 = synth.rand_desc(rng, n1), synth.rand_desc(rng, n2)
    k = n1 // 2
    d1[:k] = synth.flip_bits(rng, d2[rng.integers(0, n2, k)], 0.1)
    return d1, d2


def _check(got, want):
    bad = np.flatnonzero((got != want).any(1))
    assert bad.size == 0, (bad[:8], got[bad[:4]], want[bad[:4]])


def _switch_positions(n1, n2, ctas):
    """Units a CTA has scanned when it switches query group (same split as umma_cta_of)."""
    groups, units = -(-n1 // GROUP), -(-n2 // ROWS)
    total = groups * units
    ctas = min(ctas, total)
    pos = set()
    for g in range(1, groups):
        x = g * units
        c = ((x + 1) * ctas - 1) // total
        start = c * total // ctas
        if start < x:
            pos.add(x - start)
    return pos


@pytest.mark.parametrize("share", [1, 2, 3, RING - 1, RING, RING + 1])
def test_cta_share_lengths(M, variant, sms, share):
    """One query group, every CTA scans exactly `share` units; the last unit is ragged."""
    n2 = sms * share * ROWS - 37
    d1, d2 = _case(100 + share, 200, n2)
    variant(7)
    _check(M.knn2(d1, d2, idx_base=11), port.knn2_packed(d1, d2, idx_base=11))


def _group_switch_shapes(sms):
    """(queries, train rows) with ragged last groups and units whose group switches, together, fall after every residue
    of the packed ring and of the B tiles (and so of the accumulator pair)."""
    shapes, ring, tiles = [], set(), set()
    for n1, u in ((g * GROUP - 3, u) for u in range(100, 400) for g in (13, 16)):
        pos = _switch_positions(n1, u * ROWS - 9, sms)
        if {p % RING for p in pos} - ring or {p % B_TILES for p in pos} - tiles:
            shapes.append((n1, u * ROWS - 9))
            ring |= {p % RING for p in pos}
            tiles |= {p % B_TILES for p in pos}
        if len(ring) == RING and len(tiles) == B_TILES:
            return shapes
    raise AssertionError("no set of train sizes covers every ring phase")


def test_group_switch_at_every_ring_phase(M, variant, sms):
    """13 or 16 query groups over shares of ~9-40 units: across these shapes a CTA switches group after every residue
    of the packed ring, the B tiles and the accumulator pair."""
    for i, (n1, n2) in enumerate(_group_switch_shapes(sms)):
        d1, d2 = _case(200 + i, n1, n2)
        variant(7)
        _check(M.knn2(d1, d2, idx_base=i), port.knn2_packed(d1, d2, idx_base=i))


def test_many_short_segments(M, variant, sms):
    """20 000 queries x 1 000 rows: 79 groups of 8 units each (the last one 104 rows), so a CTA crosses several groups
    and scans ragged units that are not the last of its share."""
    d1, d2 = _case(300, 20_000, 1_000)
    assert len(_switch_positions(len(d1), len(d2), sms)) > 0
    variant(7)
    _check(M.knn2(d1, d2, idx_base=7), port.knn2_packed(d1, d2, idx_base=7))


def test_bound_drops_early(M, variant):
    """Near duplicates of every query at the start of the train set: the shared second-best bound falls within the
    first units, so nearly every later block is skipped; exact duplicates far apart keep the lowest index."""
    rng = np.random.default_rng(400)
    n1, n2 = 700, 300_000
    d1, d2 = synth.rand_desc(rng, n1), synth.rand_desc(rng, n2)
    d2[: 3 * n1] = synth.flip_bits(rng, np.repeat(d1, 3, axis=0), 0.02)
    d2[n2 - 50:] = d2[:50]
    variant(7)
    _check(M.knn2(d1, d2, idx_base=2), port.knn2_packed(d1, d2, idx_base=2))


def test_back_to_back_launches(M, variant):
    """Launches of different shapes in a row on one context, each equal to the oracle."""
    variant(7)
    for i, (n1, n2) in enumerate([(300, 70_001), (1, 200), (900, 131_072), (300, 70_001), (5000, 9_999)]):
        d1, d2 = _case(500 + i, n1, n2)
        _check(M.knn2(d1, d2, idx_base=i), port.knn2_packed(d1, d2, idx_base=i))


def test_bench_sized_queries_against_integer_kernel(M, variant):
    """6400 queries x 2 M rows (25 groups), the query count of the bench: identical keys to variant 3."""
    d1, d2 = _case(600, 6400, 2_000_000)
    variant(3)
    k3 = M.knn2(d1, d2, idx_base=5)
    variant(7)
    k7 = M.knn2(d1, d2, idx_base=5)
    _check(k7, k3)
