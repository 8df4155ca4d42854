"""The packed readout of the tensor-core scan (K1b, `knn2_umma_kernel`): columns, halves, masks and signs.

K1b loads a unit's 128 accumulator columns as 64 registers of two signed 16-bit halves (column 2i in the low half of
register i, column 2i + 1 in the high half), tests the whole unit with one minimum, and runs the blocked top-2 test only
on a unit that passes.  A wrong idea of which column sits in which half, a mask on the wrong half of a short unit, an
unsigned min or a wrong tie order each change a key here.  Every case plants the true best and second best where the
readout is most likely to get them wrong, checks that the construction gives the keys it was built for (oracle.port on
the host), and compares the kernel's keys with the oracle's bit for bit.
"""
import numpy as np
import pytest

import oracle
from pl_inertial_slam_b200 import synth

port = oracle.port
ROWS = 128   # train rows per unit = accumulator columns


@pytest.fixture(scope="module")
def M(plm_lib):
    from pl_inertial_slam_b200 import matching
    return matching


@pytest.fixture
def variant(plm_lib):
    def force(v):
        assert plm_lib.plm_set_option(b"knn_variant", v) == 0
    yield force
    plm_lib.plm_set_option(b"knn_variant", -1)


def _flip_exactly(rng, row, k):
    """row with exactly k of its 256 bits flipped."""
    bits = np.unpackbits(row)
    bits[rng.choice(256, k, replace=False)] ^= 1
    return np.packbits(bits)


def _plant(rng, n1, n2, rows_best, rows_second, d_best=3, d_second=6):
    """n1 random queries and n2 random train rows; query i's best is row rows_best[i] (d_best bits away) and its second
    best row rows_second[i] (d_second bits away).  Random rows sit at about 128 +- 8 bits, far above both."""
    d1, d2 = synth.rand_desc(rng, n1), synth.rand_desc(rng, n2)
    for i in range(n1):
        d2[rows_best[i]] = _flip_exactly(rng, d1[i], d_best)
        d2[rows_second[i]] = _flip_exactly(rng, d1[i], d_second)
    return d1, d2


def _planted_keys(rows_best, rows_second, d_best, d_second, idx_base):
    b = (np.uint64(d_best) << np.uint64(32)) | (np.asarray(rows_best, np.uint64) + np.uint64(idx_base))
    s = (np.uint64(d_second) << np.uint64(32)) | (np.asarray(rows_second, np.uint64) + np.uint64(idx_base))
    return np.stack([b, s], 1)


def _check(got, want):
    bad = np.flatnonzero((got != want).any(1))
    assert bad.size == 0, ("%d queries wrong" % bad.size, bad[:8], [[hex(int(k)) for k in r] for r in got[bad[:4]]],
                           [[hex(int(k)) for k in r] for r in want[bad[:4]]])


def _run(M, variant, d1, d2, idx_base, want=None):
    oracle_keys = port.knn2_packed(d1, d2, idx_base=idx_base)
    if want is not None:   # the construction gives the keys it was built for
        _check(oracle_keys, want)
    variant(7)
    _check(M.knn2(d1, d2, idx_base=idx_base), oracle_keys)


@pytest.mark.gpu
@pytest.mark.parametrize("col_best,col_second,same_unit", [
    (0, 1, True), (1, 0, True),          # the two halves of register 0
    (126, 127, True), (127, 126, True),  # the two halves of register 63
    (0, 127, True), (127, 0, True),      # the first and last column
    (2, 5, False), (5, 2, False),        # even against odd, in different units
    (1, 126, False), (64, 63, True),     # across the middle of the unit
])
def test_planted_columns(M, variant, col_best, col_second, same_unit):
    """Best and second best of every query at fixed columns of a unit: a swapped half moves the key by one column."""
    rng = np.random.default_rng(4000 + 128 * col_best + col_second + int(same_unit))
    n1, n2 = 300, 140_003
    units = rng.choice(n2 // ROWS, (n1, 2), replace=False)
    rows_best = units[:, 0] * ROWS + col_best
    rows_second = (units[:, 0] if same_unit else units[:, 1]) * ROWS + col_second
    d1, d2 = _plant(rng, n1, n2, rows_best, rows_second)
    _run(M, variant, d1, d2, 11, _planted_keys(rows_best, rows_second, 3, 6, 11))


@pytest.mark.gpu
@pytest.mark.parametrize("tail", [1, 2, 17, 127])
def test_short_last_unit(M, variant, tail):
    """n2 = 128 m + tail: the last unit has `tail` live columns, the rest masked.  The best sits at the last live column
    (the low half next to a masked high half for odd tails), the second best at the one before it or, for tail 1, in
    the unit before.  A short unit's masked columns are computed from the rows its packed ring stage held 8 units
    earlier; the 8 units before the last hold near copies of the queries past column `tail`, so those stale columns
    are small distances."""
    rng = np.random.default_rng(4100 + tail)
    n1, n2 = 300, 547 * ROWS + tail
    last = n2 - tail
    rows_best = np.full(n1, last + tail - 1)
    rows_second = np.full(n1, last + tail - 2) if tail > 1 else np.full(n1, last - ROWS)
    d1 = synth.rand_desc(rng, 1)
    d1 = np.repeat(d1, n1, 0)                 # one query repeated: every lane of the group plants the same rows
    d1[1:] = synth.flip_bits(rng, d1[1:], 0.02)
    d2 = synth.rand_desc(rng, n2)
    d2[rows_best[0]] = _flip_exactly(rng, d1[0], 1)
    d2[rows_second[0]] = _flip_exactly(rng, d1[0], 2)
    for u in range(1, 9):                      # near copies under the masked columns, one ring depth back
        for col in range(tail, ROWS):
            d2[last - u * ROWS + col] = _flip_exactly(rng, d1[0], 20 + (col % 7))
    want0 = _planted_keys(rows_best[:1], rows_second[:1], 1, 2, 3)
    _run(M, variant, d1, d2, 3)
    _check(port.knn2_packed(d1[:1], d2, idx_base=3), want0)


@pytest.mark.gpu
def test_dot_range_ends(M, variant):
    """|q| = 0 and 256 against all-zero and all-ones rows: dot = +256 and -256, the ends of the 16-bit halves.  All-ones
    queries find all-ones rows at distance 0 (dot -256, negative in its half), all-zero queries find all-zero rows."""
    rng = np.random.default_rng(4200)
    n1, n2 = 300, 70_003
    d1 = synth.rand_desc(rng, n1)
    d1[0::3] = 0
    d1[1::3] = 255
    d2 = synth.rand_desc(rng, n2)
    # ones at an odd column and in both halves of one register, zeros in both halves of one register and in the short
    # last unit
    ones, zeros = np.array([777, 40_002, 40_003]), np.array([1_280, 1_281, 69_999])
    d2[ones] = 255
    d2[zeros] = 0
    want = port.knn2_packed(d1, d2, idx_base=0)
    assert np.array_equal(want[1::3], _planted_keys(np.full(100, 777), np.full(100, 40_002), 0, 0, 0))
    assert np.array_equal(want[0::3], _planted_keys(np.full(100, 1_280), np.full(100, 1_281), 0, 0, 0))
    _run(M, variant, d1, d2, 0)


@pytest.mark.gpu
@pytest.mark.parametrize("fill", [0, 255])
def test_uniform_extreme_train_set(M, variant, fill):
    """Every train row all zeros or all ones: every distance of a query is 0 or 256 (dot 0 / +-256 in every half), so
    the top-2 is rows 0 and 1 by the lowest-index rule."""
    rng = np.random.default_rng(4300 + fill)
    n1, n2 = 257, 66_000
    d1 = synth.rand_desc(rng, n1)
    d1[0::2] = 0
    d1[1::2] = 255
    d2 = np.full((n2, 32), fill, np.uint8)
    d = np.where((d1[:, 0] == fill), 0, 256).astype(np.uint64)
    want = np.stack([(d << np.uint64(32)) | np.uint64(5), (d << np.uint64(32)) | np.uint64(6)], 1)
    _run(M, variant, d1, d2, 5, want)


@pytest.mark.gpu
@pytest.mark.parametrize("where", ["best", "second"])
def test_tie_inside_one_register(M, variant, where):
    """Two rows at the same distance in the two halves of one register (columns 2j, 2j + 1) and a third, later one:
    the lower column wins.  'best': the tie is the top-2 itself; 'second': a better row elsewhere, the tie decides the
    second best."""
    rng = np.random.default_rng(4400 + len(where))
    n1, n2 = 300, 140_003
    units = 3 * rng.choice(n2 // ROWS // 3, n1, replace=False)   # query i: units u, u + 1 and u + 2 of its own
    j = rng.integers(0, ROWS // 2, n1)
    lo = units * ROWS + 2 * j
    later = (units + 1) * ROWS + 2 * j            # same distance, a unit later
    d1, d2 = synth.rand_desc(rng, n1), synth.rand_desc(rng, n2)
    for i in range(n1):
        row = _flip_exactly(rng, d1[i], 4)
        d2[lo[i]] = d2[lo[i] + 1] = d2[later[i]] = row
    if where == "best":
        want = _planted_keys(lo, lo + 1, 4, 4, 0)
    else:
        better = (units + 2) * ROWS + rng.integers(0, ROWS, n1)
        for i in range(n1):
            d2[better[i]] = _flip_exactly(rng, d1[i], 1)
        want = _planted_keys(better, lo, 1, 4, 0)
    _run(M, variant, d1, d2, 0, want)
