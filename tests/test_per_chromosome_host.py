"""Host-side checks of FitHiC.fit_transform_arrays(per_chromosome=True): the argument checks and the split of the records and
fragments by chromosome (blueberry_b200.fithic.split_chromosomes) run before any device work, so they need no GPU."""
import numpy as np
import pytest

from blueberry_b200.fithic import FitHiC, split_chromosomes


def _records():
    chrom = np.array([2, 2, 2, 0, 0, 5, 5, 5, 5], dtype=np.int32)
    mid = np.arange(chrom.size, dtype=np.int32) * 1000 + 500
    frag_chrom = np.array([0, 0, 2, 5, 2, 7, 5, 0], dtype=np.int32)
    return chrom, mid, frag_chrom


def test_split_orders_chromosomes_and_finds_their_rows_and_fragments():
    chrom, _, fc = _records()
    plan = split_chromosomes(chrom, chrom, fc)
    assert [x[0] for x in plan] == [0, 2, 5]
    assert [(x[1], x[2]) for x in plan] == [(3, 5), (0, 3), (5, 9)]
    assert [x[3].tolist() for x in plan] == [[0, 1, 7], [2, 4], [3, 6]]
    assert [x[4] for x in plan] == [None, None, None]


def test_split_n_tests_one_value_or_a_mapping():
    chrom, _, fc = _records()
    assert [x[4] for x in split_chromosomes(chrom, chrom, fc, n_tests=40)] == [40, 40, 40]
    plan = split_chromosomes(chrom, chrom, fc, n_tests={np.int64(5): 7, 0: 3})
    assert [x[4] for x in plan] == [3, None, 7]


def test_split_of_no_rows_is_empty():
    e = np.zeros(0, dtype=np.int32)
    assert split_chromosomes(e, e, np.array([0, 1])) == []


def test_a_chromosome_with_a_single_row():
    chrom = np.array([1, 1, 4, 3, 3], dtype=np.int32)
    plan = split_chromosomes(chrom, chrom, np.array([1, 3, 4]))
    assert [(x[0], x[1], x[2]) for x in plan] == [(1, 0, 2), (3, 3, 5), (4, 2, 3)]


def test_inter_chromosomal_rows_raise_value_error():
    chrom, _, fc = _records()
    c2 = chrom.copy()
    c2[4] = 2
    with pytest.raises(ValueError, match="intra-chromosomal"):
        split_chromosomes(chrom, c2, fc)


def test_rows_of_a_chromosome_must_be_contiguous():
    chrom, _, fc = _records()
    c = chrom.copy()
    c[1] = 0                                 # 2 0 2 0 0 5 ...: chromosomes 0 and 2 each in two blocks
    with pytest.raises(ValueError, match="not contiguous"):
        split_chromosomes(c, c, fc)


def test_unsupported_options_and_missing_columns():
    chrom, _, fc = _records()
    with pytest.raises(NotImplementedError):
        split_chromosomes(chrom, chrom, fc, refit=True)
    with pytest.raises(NotImplementedError):
        split_chromosomes(chrom, chrom, fc, group=True)
    with pytest.raises(ValueError):
        split_chromosomes(None, None, fc)
    with pytest.raises(ValueError):
        split_chromosomes(chrom, chrom[:-1], fc)


def test_the_public_call_checks_before_any_device_work():
    """No GPU is needed to reach these errors through FitHiC.fit_transform_arrays."""
    chrom, mid, fc = _records()
    fm = np.arange(fc.size, dtype=np.int32) * 1000 + 500
    model = FitHiC("x", 1000, max_dist=100000)
    cnt = np.ones(chrom.size, dtype=np.int32)
    c2 = chrom.copy()
    c2[0] = 0
    with pytest.raises(ValueError):
        model.fit_transform_arrays(chrom, mid, c2, mid, cnt, fc, fm, per_chromosome=True)
    c = chrom.copy()
    c[1] = 0
    with pytest.raises(ValueError):
        model.fit_transform_arrays(c, mid, c, mid, cnt, fc, fm, per_chromosome=True)
    with pytest.raises(NotImplementedError):
        model.fit_transform_arrays(chrom, mid, chrom, mid, cnt, fc, fm, per_chromosome=True, refit=True)
    with pytest.raises(NotImplementedError):
        model.fit_transform_arrays(chrom, mid, chrom, mid, cnt, fc, fm, per_chromosome=True, group=True)
