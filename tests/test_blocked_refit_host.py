"""Host-side logic of the two-pass workload in row blocks (distributed.BlockedPass(refit=True)): the memory estimate that
routes fit_transform_arrays(refit=True) onto it, the outlier threshold the constructor computes, and the argument checks
that run before any device work.  No GPU needed."""
import numpy as np
import pytest
import torch

from blueberry_b200 import distributed as D
from blueberry_b200 import fithic


class _FakeEngine(object):
    """What BlockedPass(refit=True) reads of a PassEngine before any device work: the conditions of the streaming K4 and the
    possible pairs per distance key (a CPU tensor here)."""
    lib, device = None, "cuda:0"

    def __init__(self, possible, R=1000, min_dist=0, max_dist=2_000_000):
        self.R, self.min_dist, self.max_dist, self.bias = R, min_dist, max_dist, None
        self.possible = torch.as_tensor(np.asarray(possible, dtype=np.int64))


def _shard(n, chrom=0):
    return (chrom, np.zeros(n, np.int32), np.zeros(n, np.int32), np.zeros(n, np.int32))


def test_refit_estimate_adds_pass_one():
    for rows in (4, 1_000_000, 1_000_000_000, 6_030_000_000):
        for q in (True, False):
            one, two = D.resident_pass_bytes(rows, q), D.resident_pass_bytes(rows, q, refit=True)
            # pass 1's p (8 B), deferred list (rows / 4 x 16 B) and candidate list (rows / 16 x 12 B)
            assert abs((two - one) - rows * (8 + 4 + 0.75)) <= 1
    assert D.resident_pass_bytes(1 << 30, True, refit=True) == int((1 << 30) * 69.5)


def test_defaults_give_the_single_pass_values():
    rows = 123_456_789
    assert D.resident_pass_bytes(rows) == D.resident_pass_bytes(rows, True, refit=False) == int(rows * 56.75)
    assert D.resident_pass_bytes(rows, False) == int(rows * 24.75)
    for free in (0, D.resident_pass_bytes(rows) + (1 << 30), D.resident_pass_bytes(rows, refit=True) + (1 << 30)):
        for q in (True, False):
            assert D.needs_blocked_pass(rows, free, q) == D.needs_blocked_pass(rows, free, q, refit=False)


def test_refit_routes_at_2_32_rows_and_by_free_memory():
    big = 1 << 60
    assert not D.needs_blocked_pass((1 << 32) - 4, big, refit=True)
    assert D.needs_blocked_pass(1 << 32, big, refit=True)
    rows, margin = 1_000_000_000, 1 << 30
    one, two = D.resident_pass_bytes(rows, True), D.resident_pass_bytes(rows, True, refit=True)
    assert not D.needs_blocked_pass(rows, two + margin, True, margin, refit=True)
    assert D.needs_blocked_pass(rows, two + margin - 1, True, margin, refit=True)
    # free memory that holds the single pass but not the two-pass: only refit is routed
    free = (one + two) // 2 + margin
    assert not D.needs_blocked_pass(rows, free, True, margin) and D.needs_blocked_pass(rows, free, True, margin, refit=True)
    # about 2.5e9 rows of two-pass on a 180 GB card
    assert D.needs_blocked_pass(2_600_000_000, 180 * 10 ** 9, refit=True)
    assert not D.needs_blocked_pass(2_400_000_000, 180 * 10 ** 9, refit=True)


def test_use_blocked_pass_defaults(monkeypatch):
    rows = 1_000_000_000
    one, two = D.resident_pass_bytes(rows, True), D.resident_pass_bytes(rows, True, refit=True)
    free = (one + two) // 2 + (1 << 30)
    monkeypatch.setattr(torch.cuda, "mem_get_info", lambda dev=None: (free, 2 * free))
    assert fithic.use_blocked_pass(rows, True, "cuda:0") is False
    assert fithic.use_blocked_pass(rows, True, "cuda:0", refit=False) is False
    assert fithic.use_blocked_pass(rows, True, "cuda:0", refit=True) is True
    assert fithic.use_blocked_pass(1 << 32, True, "cuda:0") is True


def test_threshold_from_the_fragments():
    possible = [0, 5, 7, 11, 13]
    bp = D.BlockedPass(_FakeEngine(possible, R=1000, min_dist=0, max_dist=3000), refit=True, block_rows=4096)
    assert bp.p_outlier == 1.0 / fithic._in_range_possible(np.array(possible), 1000, 0, 3000) == 1.0 / 23
    assert D.BlockedPass(_FakeEngine(possible), block_rows=4096).p_outlier is None


def test_no_in_range_pair_raises_in_the_constructor():
    with pytest.raises(ZeroDivisionError):
        D.BlockedPass(_FakeEngine([4, 0, 0], R=1000, min_dist=0, max_dist=2000), refit=True)


def test_without_refit_possible_is_not_read():
    class NoPossible(_FakeEngine):
        @property
        def possible(self):
            raise AssertionError("BlockedPass(refit=False) read engine.possible")

        @possible.setter
        def possible(self, v):
            pass

    D.BlockedPass(NoPossible([1]), block_rows=4096)


@pytest.mark.parametrize("case", ["without_refit", "short", "long", "count", "readonly", "float32", "device_like_2d"])
def test_p_first_out_errors_before_device_work(case):
    refit = case != "without_refit"
    bp = D.BlockedPass(_FakeEngine([0, 9, 9]), refit=refit, block_rows=4096)
    shards = [_shard(10), _shard(7, 1)]
    p, q = [np.empty(10), np.empty(7)], [np.empty(10), np.empty(7)]
    p1 = [np.empty(10), np.empty(7)]
    if case == "short":
        p1[1] = np.empty(6)
    elif case == "long":
        p1[0] = np.empty(11)
    elif case == "count":
        p1 = p1[:1]
    elif case == "readonly":
        p1[0].flags.writeable = False
    elif case == "float32":
        p1[1] = np.empty(7, np.float32)
    elif case == "device_like_2d":
        p1[0] = np.empty((10, 1))
    with pytest.raises(ValueError):
        bp.check(shards, p, q, p_first_out=p1)
    with pytest.raises(ValueError):
        bp.run(shards, p, q, p_first_out=p1)      # the fake engine has no device: reaching device work would fail otherwise


def test_check_keeps_its_three_results():
    bp = D.BlockedPass(_FakeEngine([0, 9, 9]), refit=True, block_rows=4096)
    shards = [_shard(10), _shard(7, 1)]
    p, q, p1 = [np.empty(10), np.empty(7)], [np.empty(10), np.empty(7)], [np.empty(10), np.empty(7)]
    sizes, ps, qs = bp.check(shards, p, q, p_first_out=p1)
    assert sizes == [10, 7] and len(ps) == len(qs) == 2
