"""Host-side logic of the blocked genome-wide pass (distributed.BlockedPass): the block plan, the routing of
fit_transform_arrays onto it, and the argument checks that run before any device work.  No GPU needed."""
import numpy as np
import pytest

from blueberry_b200 import distributed as D
from blueberry_b200 import fithic


def _check_plan(sizes, block_rows):
    blocks = D.plan_blocks(sizes, block_rows)
    seen = [np.zeros(n, dtype=np.int64) for n in sizes]
    for blk in blocks:
        assert blk, "no empty blocks"
        end = 0
        for (s, lo, n, off) in blk:
            assert n > 0
            assert off % D.BLOCK_ALIGN == 0 and off % 4 == 0
            assert off >= end, "pieces do not overlap on the device"
            end = off + n
            seen[s][lo:lo + n] += 1
        assert sum(n for (_, _, n, _) in blk) <= block_rows
        assert D.block_device_rows(blk) <= (block_rows + D.BLOCK_ALIGN - 1) // D.BLOCK_ALIGN * D.BLOCK_ALIGN < (1 << 32)
    for s in seen:
        assert (s == 1).all(), "every row exactly once"
    return blocks


@pytest.mark.parametrize("sizes,block_rows", [
    ([10_000, 3, 0, 1, 50_000, 4096, 8191], 8192),
    ([1], 4096),
    ([0, 0], 4096),
    ([], 4096),
    ([1 << 20], 1 << 16),
    ([123_457, 99_999, 7], 3 * 4096),
    ([123_457, 99_999, 7], 12_345),
    ([70_001, 3, 5], 4097),
    ([5000] * 23, 1 << 27),
])
def test_plan_covers_every_row_once(sizes, block_rows):
    blocks = _check_plan(sizes, block_rows)
    if sum(sizes) == 0:
        assert blocks == []


def test_plan_cuts_a_shard_larger_than_a_block():
    blocks = _check_plan([20_000], 8192)
    assert [len(b) for b in blocks] == [1, 1, 1]
    assert [(lo, n) for b in blocks for (_, lo, n, _) in b] == [(0, 8192), (8192, 8192), (16384, 3616)]


def test_plan_cuts_shards_at_odd_rows():
    blocks = _check_plan([64_320, 40_200, 16_290], 12_345)
    assert any(lo % 4 for b in blocks for (_, lo, _, _) in b)


def test_plan_places_pieces_on_chunks():
    blk = D.plan_blocks([5, 4100, 3], 3 * 4096)
    assert blk == [[(0, 0, 5, 0), (1, 0, 4100, 4096)], [(2, 0, 3, 0)]]


def test_plan_rows_beyond_2_32_in_blocks_below_it():
    sizes = [3_000_000_000, 2_500_000_000, 1_000]
    blocks = D.plan_blocks(sizes, 1 << 27)
    assert sum(n for b in blocks for (_, _, n, _) in b) == sum(sizes)
    assert max(D.block_device_rows(b) for b in blocks) <= 1 << 27


@pytest.mark.parametrize("bad", [0, -4096, 1 << 32, (1 << 32) - 4095])
def test_plan_rejects_bad_block_rows(bad):
    with pytest.raises(ValueError):
        D.plan_blocks([10], bad)


def test_routing_at_2_32_rows():
    big = 1 << 60
    assert not D.needs_blocked_pass((1 << 32) - 4, big)
    assert D.needs_blocked_pass(1 << 32, big)
    assert D.needs_blocked_pass(1 << 33, big)


def test_routing_by_memory_estimate():
    rows = 1_000_000_000
    need = D.resident_pass_bytes(rows, True)
    # 12 B of records, 8 + 8 B of p / q, rows / 4 x 16 B deferred, rows / 16 x 12 B candidates
    assert need >= int(rows * 32.75)
    assert D.resident_pass_bytes(rows, False) < need
    margin = 1 << 30
    assert not D.needs_blocked_pass(rows, need + margin, True, margin)
    assert D.needs_blocked_pass(rows, need + margin - 1, True, margin)
    # config 5 on one B200: 6.03e9 records
    assert D.needs_blocked_pass(6_030_000_000, 180 << 30)


def test_compact_runs():
    c = np.array([0, 0, 0, 2, 2, 5], dtype=np.int32)
    assert fithic.compact_runs(c, c, 6) == [(0, 0, 3), (2, 3, 5), (5, 5, 6)]
    assert fithic.compact_runs(None, None, 7) == [(0, 0, 7)]
    assert fithic.compact_runs(c, c[::-1].copy(), 6) is None
    inter = np.arange(200) % 2
    assert fithic.compact_runs(inter, inter, 200) is None


class _FakeEngine(object):
    """What BlockedPass reads of a PassEngine before any device work."""
    lib, device = None, "cuda:0"

    def __init__(self, R=1000, min_dist=0, max_dist=2_000_000, bias=None):
        self.R, self.min_dist, self.max_dist, self.bias = R, min_dist, max_dist, bias


class _Bias(object):
    def __init__(self, step):
        self.step = step


@pytest.mark.parametrize("kw", [dict(min_dist=-1), dict(max_dist=(1 << 31) - 10), dict(R=1), dict(bias=_Bias(1))])
def test_engine_without_streaming_k4_is_refused(kw):
    with pytest.raises(ValueError):
        D.BlockedPass(_FakeEngine(**kw))


def test_bad_block_rows_refused():
    with pytest.raises(ValueError):
        D.BlockedPass(_FakeEngine(), block_rows=0)


def _shard(n, chrom=0):
    return (chrom, np.zeros(n, np.int32), np.zeros(n, np.int32), np.zeros(n, np.int32))


@pytest.mark.parametrize("case", ["short_p", "no_q", "q_without_q_values", "five_columns", "ragged", "float32_out",
                                  "readonly_out", "2d_column", "float_records", "count_p"])
def test_argument_errors_before_device_work(case):
    bp = D.BlockedPass(_FakeEngine(), q_values=case != "q_without_q_values", block_rows=4096)
    shards = [_shard(10), _shard(7, 1)]
    p = [np.empty(10), np.empty(7)]
    q = [np.empty(10), np.empty(7)]
    if case == "short_p":
        p[1] = np.empty(6)
    elif case == "no_q":
        q = None
    elif case == "five_columns":
        shards[0] = (0, 0) + shards[0][1:]
    elif case == "ragged":
        shards[1] = (1, np.zeros(7, np.int32), np.zeros(6, np.int32), np.zeros(7, np.int32))
    elif case == "float32_out":
        p[0] = np.empty(10, np.float32)
    elif case == "readonly_out":
        p[0].flags.writeable = False
    elif case == "2d_column":
        shards[0] = (0, np.zeros((10, 1), np.int32), np.zeros(10, np.int32), np.zeros(10, np.int32))
    elif case == "float_records":
        shards[0] = (0, np.zeros(10), np.zeros(10), np.zeros(10))
    elif case == "count_p":
        p = p[:1]
    with pytest.raises(ValueError):
        bp.run(shards, p, q)          # the fake engine has no device: reaching device work would fail otherwise


def test_too_many_candidate_places_refused():
    bp = D.BlockedPass(_FakeEngine(), block_rows=4096, cand_capacity=1 << 22)
    n = 4096 * 1100
    with pytest.raises(ValueError):
        bp.check([(0, np.zeros(n, np.int32), np.zeros(n, np.int32), np.zeros(n, np.int32))], [np.empty(n)], [np.empty(n)])
