"""CPU tests of the column layout's host helpers (geonomics_b200.genome_pack): column rows <-> the reference's
use_tskit rows, and the bound that decides when the columns are widened."""
import numpy as np

from geonomics_b200 import genome_pack as gp


def test_rows_and_columns_round_trip_against_numpy():
    rng = np.random.default_rng(1)
    L, n = 700, 9
    col_locus = np.array([5, 40, 300, 2, 699, 128, 31], np.int64)     # starting columns ascending, then appended
    rows = rng.integers(0, 2, (n, len(col_locus), 2)).astype(np.int8)  # ascending locus order
    packed = gp.rows_to_cols(rows, col_locus, gp.words_per_hap(128))
    assert packed.shape == (n, 2, 4)
    bits = np.unpackbits(packed.view(np.uint8), axis=-1, bitorder='little')   # [n, 2, 128]
    order = np.sort(col_locus)
    for j, l in enumerate(col_locus):
        r = int(np.searchsorted(order, l))
        assert np.array_equal(bits[:, :, j], rows[:, r, :])
    assert not bits[:, :, len(col_locus):].any()
    assert np.array_equal(gp.cols_to_rows(packed, col_locus), rows)
    # the by-locus view of the same rows
    by_locus = gp.rows_to_loci(rows, order, L)
    assert np.array_equal(gp.loci_to_rows(by_locus, order), rows)


def test_col_capacity():
    assert [gp.col_capacity(k) for k in (0, 20, 64, 65, 120, 192, 193)] == [128, 128, 128, 256, 256, 256, 384]


def test_column_budget_reads_and_widens_only_when_the_bound_passes():
    reads = []

    def reader(v):
        def f():
            reads.append(v)
            return v
        return f
    b = gp.ColumnBudget(20, 128, 64, 1 << 20)
    assert b.take(1, reader(0)) == (1, 128) and reads == []           # 84 <= 128
    assert b.take(1, reader(30)) == (1, 128) and reads == [30]        # 148 > 128: read 30, one step fits
    assert b.bound == 94
    assert b.take(5, reader(70)) == (2, 256) and reads == [30, 70]    # 70 + 64 > 128: double once, two steps fit
    assert b.bound == 198
    assert b.take(1, reader(100)) == (1, 256) and reads[-1] == 100    # 262 > 256: read again, no widening
    # several steps per call when they fit; never past the capacity that holds every locus
    b = gp.ColumnBudget(10, 512, 64, 1 << 20)
    assert b.take(10, reader(10)) == (7, 512) and reads[-1] == 10
    b = gp.ColumnBudget(100, 128, 64, 128)
    assert b.take(50, reader(0)) == (50, 128)
    # no non-neutral mutation: nothing to bound
    b = gp.ColumnBudget(100, 128, 0, 1 << 20)
    assert b.take(1000, reader(0)) == (1000, 128)
