"""GPU tests of the per-chromosome pass (FitHiC.fit_transform_arrays(per_chromosome=True), distributed.ChromosomePass) and of
its two kernels:

  * bbk_fit_batched against one bbk_fit per problem, bit for bit (mixed table sizes, s given, too many bins, a failed fit,
    a problem with too small a workspace, more problems than SMs);
  * bbk_bh_qvalues_segmented against bbk_bh_qvalues_listed on every segment alone, bit for bit (empty and tiny segments, ties,
    NaN, p == 1.0 groups with q below 1, N given or not, the pass over p, an overflowed candidate list, > 256 segments);
  * the contract: per_chromosome=True against the loop of single-chromosome calls, every field bit for bit;
  * every chromosome against the CPU oracle run on that chromosome alone;
  * three chromosomes of BASELINE config 2's shape with a deferred list that overflows.
"""
import ctypes
import struct

import numpy as np
import pytest

from helpers import log10_close

pytestmark = pytest.mark.gpu

_FIT_COMPARED = [(0, 72), (120, 136), (184, 192)]      # BbkFitResult bytes without the SM cycle counters


def _fit_bytes(raw):
    """The result bytes a fit defines: all but the cycle counters, and for a failed fit (which raises) not min_x / max_x,
    which the kernel does not set before it stops."""
    raw = bytes(raw)
    parts = _FIT_COMPARED if struct.unpack_from("i", raw)[0] == 0 else [(0, 32), (48, 72), (120, 136), (184, 192)]
    return b"".join(raw[a:b] for a, b in parts)


def _bits(a):
    a = np.ascontiguousarray(a)
    return a.view(np.uint8).tobytes() if a.size else b""


def _t32(a, dev):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.int32)).to(dev)


# ------------------------------------------------------------------------------------------------ bbk_fit_batched
def _fit_tables(seed, R, max_dist, dev):
    """possible / observed / totals of one synthetic chromosome, filled by the library's own K2a and K1."""
    from blueberry_b200 import synth
    from blueberry_b200.engine import PassEngine, Shard
    rng = np.random.default_rng(seed)
    nb = int(rng.integers(60, 400))
    c = synth.make_contacts([nb], R, max_dist, float(rng.choice([5.0, 60.0, 400.0])), seed)
    eng = PassEngine(R, 30, 0, max_dist, nb, dev)
    eng.set_fragments([nb], [(nb - 1) * R])
    eng.hist([Shard(_t32(c["mid1"], dev), _t32(c["mid2"], dev), _t32(c["count"], dev), chrom=0)])
    return eng


def _clone_engine(src, dev, max_bins=None):
    from blueberry_b200.engine import PassEngine
    e = PassEngine(src.R, src.n_bins, src.min_dist, src.max_dist, src.nkeys, dev, max_bins=max_bins)
    e.possible.copy_(src.possible)
    e.stats.copy_(src.stats)
    return e


def _fit_outputs(e):
    import torch
    torch.cuda.synchronize()
    return [_fit_bytes(e.fit_result.cpu().numpy().tobytes())] + [_bits(t.cpu().numpy()) for t in
                                                                  (e.x, e.y, e.bin_of_key, e.spline_y, e.spline_raw, e.knots, e.coefs)]


@pytest.mark.parametrize("n_problems", [7, 300])
def test_batched_fit_equals_single_fits(n_problems):
    import torch
    from blueberry_b200 import _lib
    dev = torch.device("cuda", 0)
    lib = _lib.load()
    R, max_dist = 10000, 1_500_000
    tables = [_fit_tables(s, R, max_dist, dev) for s in range(min(n_problems, 24))]
    singles, batched, s_given = [], [], {}
    for i in range(n_problems):
        src = tables[i % len(tables)]
        kind = i % 7
        max_bins = 4 if kind == 3 else None                        # kind 3: more bins than the buffers hold -> TOO_MANY_BINS
        a, b = _clone_engine(src, dev, max_bins), _clone_engine(src, dev, max_bins)
        if kind == 4:                                              # kind 4: no possible pairs -> ZERO_PAIRS_BIN
            a.possible.zero_(); b.possible.zero_()
        if kind == 2:                                              # kind 2: s given (a slightly different s than min(y)**2)
            a.fit()
            s = float(_lib.FitResult.from_buffer_copy(a.fit_result.cpu().numpy().tobytes()).smoothing) * 1.5
            a.fit(smoothing=s)
            req = _lib.FitResult()
            req.status, req.smoothing = _lib.FIT_S_GIVEN, s
            b.fit_result.copy_(torch.frombuffer(bytearray(bytes(req)), dtype=torch.uint8))
            s_given[i] = s
        else:
            a.fit()
        singles.append(a)
        batched.append(b)
    probs = (_lib.FitProblem * n_problems)()
    for i, (pr, e) in enumerate(zip(probs, batched)):
        pr.d_possible, pr.d_obs_sum, pr.d_totals = e.possible.data_ptr(), e.obs_sum.data_ptr(), e.totals.data_ptr()
        pr.d_result, pr.d_x, pr.d_y, pr.d_bin_of_key = e.fit_result.data_ptr(), e.x.data_ptr(), e.y.data_ptr(), e.bin_of_key.data_ptr()
        pr.d_spline_y, pr.d_spline_raw, pr.d_knots, pr.d_coefs = (e.spline_y.data_ptr(), e.spline_raw.data_ptr(), e.knots.data_ptr(),
                                                                  e.coefs.data_ptr())
        pr.d_workspace, pr.workspace_bytes = e.fit_ws.data_ptr(), e.fit_ws.numel()
        pr.nkeys, pr.max_bins = e.nkeys, e.max_bins
        if i % 7 == 5:                                             # kind 5: a workspace one byte too small
            pr.workspace_bytes = int(lib.bbk_fit_workspace_bytes(e.max_bins, e.nkeys)) - 1
    d_probs = torch.frombuffer(bytearray(bytes(probs)), dtype=torch.uint8).to(dev)
    _lib.check(lib.bbk_fit_batched(_lib.ptr(d_probs), n_problems, 30, R, 0, max_dist, _lib.stream_ptr()), "bbk_fit_batched")
    statuses = set()
    for i, (a, b) in enumerate(zip(singles, batched)):
        res = _lib.FitResult.from_buffer_copy(b.fit_result.cpu().numpy().tobytes())
        statuses.add(res.status)
        if i % 7 == 5:
            assert res.status == -17
            assert not b.x.any() and not b.spline_y.any()          # nothing else written
            continue
        assert _fit_outputs(a) == _fit_outputs(b), "problem %d differs" % i
        if i in s_given:
            assert res.smoothing == s_given[i] and res.status == 0
    assert {0, -13, -11, -17} <= statuses
    widths = {e.nkeys for e in batched}
    assert len(widths) > 3


# ------------------------------------------------------------------------------------------------ bbk_bh_qvalues_segmented
def _keys(p):
    return p.view(np.uint64) | np.uint64(1 << 63)


def _phist(p):
    h = np.zeros(4098, dtype=np.int64)
    ok = ~np.isnan(p)
    ones = ok & (p == 1.0)
    rest = p[ok & ~ones]
    np.add.at(h, ((rest.view(np.uint64) >> np.uint64(51)) & np.uint64(4095)).astype(np.int64), 1)
    h[4096] = int(ones.sum())
    h[4097] = int((~ok).sum())
    return h


def _segment_p(rng, n):
    """p as K4 leaves it: mostly uniform, exact 1.0 (zero counts), NaN (not emitted), a tail of tiny p with ties."""
    p = rng.random(n)
    u = rng.random(n)
    p[u < 0.25] = 1.0
    p[(u >= 0.25) & (u < 0.3)] = np.nan
    tiny = (u >= 0.3) & (u < 0.36)
    p[tiny] = 10.0 ** -rng.uniform(2, 14, int(tiny.sum()))
    if n > 10:
        k = rng.choice(np.flatnonzero(tiny | (p < 0.5)), min(6, n // 3), replace=False) if (tiny | (p < 0.5)).sum() >= 6 else []
        for j in k:
            p[j] = p[k[0]]                                          # a tie group
    return p


class _Seg(object):
    pass


def _make_segment(rng, n, n_tests, dev, cand_cap=None):
    import torch
    from blueberry_b200 import _lib
    s = _Seg()
    s.n, s.n_tests = n, n_tests
    s.p = _segment_p(rng, n)
    small = np.flatnonzero(~np.isnan(s.p) & (s.p < 0.03125))
    cap = len(small) if cand_cap is None else cand_cap
    s.overflow = len(small) > cap
    s.keys = _keys(s.p[small[:cap]]).astype(np.uint64)
    s.rows = small[:cap].astype(np.uint32)
    s.hist = torch.from_numpy(_phist(s.p)).to(dev)
    st = _lib.ScoreState()
    st.n_cand, st.cand_overflow = len(small), 1 if s.overflow else 0
    s.state = torch.frombuffer(bytearray(bytes(st)), dtype=torch.uint8).to(dev)
    s.cap = max(cap, 1)
    return s


def _qvalues_alone(s, dev):
    """bbk_bh_qvalues_listed on the segment in buffers of its own."""
    import torch
    from blueberry_b200 import _lib
    lib = _lib.load()
    p = torch.from_numpy(np.concatenate([s.p, np.full(4, np.nan)])).to(dev)
    q = torch.where(torch.isnan(p), p, torch.ones_like(p))
    keys = torch.zeros(s.cap, dtype=torch.int64, device=dev)
    rows = torch.zeros(s.cap, dtype=torch.int32, device=dev)
    if len(s.keys):
        keys[:len(s.keys)] = torch.from_numpy(s.keys.view(np.int64)).to(dev)
        rows[:len(s.rows)] = torch.from_numpy(s.rows.view(np.int32)).to(dev)
    cands = _lib.Candidates(keys.data_ptr(), rows.data_ptr(), s.cap)
    ws = torch.empty(int(lib.bbk_bh_workspace_bytes(max(s.n, 1))), dtype=torch.uint8, device=dev)
    _lib.check(lib.bbk_bh_qvalues_listed(_lib.ptr(p), s.n, s.n_tests, _lib.ptr(s.hist), _lib.ptr(q), ctypes.byref(cands),
                                         _lib.ptr(s.state), _lib.ptr(ws), ws.numel(), _lib.stream_ptr()), "bbk_bh_qvalues_listed")
    return q[:s.n].cpu().numpy()


def _qvalues_segmented(segs, dev):
    import torch
    from blueberry_b200 import _lib
    from blueberry_b200.distributed import layout_rows
    lib = _lib.load()
    starts, rows = layout_rows([s.n for s in segs])
    m = max(rows, 4)
    p = np.full(m, np.nan)
    for s, a in zip(segs, starts):
        p[a:a + s.n] = s.p
    d_p = torch.from_numpy(p).to(dev)
    d_q = torch.where(torch.isnan(d_p), d_p, torch.ones_like(d_p))
    keep = []
    desc = (_lib.BhSegment * len(segs))()
    for d, s, a in zip(desc, segs, starts):
        keys = torch.zeros(s.cap, dtype=torch.int64, device=dev)
        rws = torch.zeros(s.cap, dtype=torch.int32, device=dev)
        if len(s.keys):
            keys[:len(s.keys)] = torch.from_numpy(s.keys.view(np.int64)).to(dev)
            rws[:len(s.rows)] = torch.from_numpy((s.rows + a).astype(np.uint32).view(np.int32)).to(dev)
        keep += [keys, rws]
        d.d_p_hist, d.d_state, d.n_tests = s.hist.data_ptr(), s.state.data_ptr(), s.n_tests
        d.cands = _lib.Candidates(keys.data_ptr(), rws.data_ptr(), s.cap)
    d_desc = torch.frombuffer(bytearray(bytes(desc)), dtype=torch.uint8).to(dev)
    off = torch.tensor(starts + [rows], dtype=torch.int64, device=dev)
    ws = torch.empty(int(lib.bbk_bh_segmented_workspace_bytes(m, len(segs))), dtype=torch.uint8, device=dev)
    _lib.check(lib.bbk_bh_qvalues_segmented(_lib.ptr(d_p), m, _lib.ptr(off), _lib.ptr(d_desc), len(segs), _lib.ptr(d_q),
                                            _lib.ptr(ws), ws.numel(), _lib.stream_ptr()), "bbk_bh_qvalues_segmented")
    q = d_q.cpu().numpy()
    return [q[a:a + s.n] for s, a in zip(segs, starts)], q, starts


@pytest.mark.parametrize("case", ["mixed", "many"])
def test_segmented_qvalues_equal_listed_qvalues_per_segment(case):
    import torch
    dev = torch.device("cuda", 0)
    rng = np.random.default_rng(17 if case == "mixed" else 18)
    segs = []
    if case == "mixed":
        spec = [(0, -1, None), (1, -1, None), (3, -1, None), (20000, -1, None), (15001, 7, None),      # N = 7: q(p == 1) < 1
                (30000, 25, None), (9999, -1, 40), (50003, -1, None), (2, 5, None), (40000, 3000, None)]
        for n, nt, cap in spec:
            segs.append(_make_segment(rng, n, nt, dev, cap))
    else:                                                           # more than 256 segments: two segment digits
        for i in range(300):
            n = int(rng.choice([0, 1, 3, 17, 400, 2500]))
            segs.append(_make_segment(rng, n, int(rng.choice([-1, -1, 9, 2 * n + 1])), dev))
    got, q_all, starts = _qvalues_segmented(segs, dev)
    below_one = 0
    for i, s in enumerate(segs):
        want = _qvalues_alone(s, dev)
        assert _bits(got[i]) == _bits(want), "segment %d (%d rows, N %d) differs" % (i, s.n, s.n_tests)
        if s.n and (s.p == 1.0).any():
            below_one += int((want[s.p == 1.0] < 1.0).any())
    assert below_one >= 1                                          # a p == 1.0 group whose q fell below 1
    if case == "mixed":
        assert any(s.overflow for s in segs)
        pad = np.ones(len(q_all), bool)
        for s, a in zip(segs, starts):
            pad[a:a + s.n] = False
        assert np.isnan(q_all[pad]).all()                          # the rows between segments are left alone


# ------------------------------------------------------------------------------------------------ the contract
def _random_genome(seed):
    from blueberry_b200 import synth
    rng = np.random.default_rng(seed)
    n_chrom = int(rng.integers(1, 6))
    bins = [int(rng.integers(120, 420)) for _ in range(n_chrom)]
    R = int(rng.choice([1000, 5000, 10000]))
    max_dist = int(rng.choice([40, 90, 300])) * R
    min_dist = int(rng.choice([0, 0, 3 * R]))
    with_bias = bool(rng.random() < 0.6)
    bias = synth.make_bias(bins, seed, sigma=0.3) if with_bias else None
    c = synth.make_contacts(bins, R, min(max_dist, max(bins) * R), float(rng.choice([4.0, 40.0, 300.0])), seed, bias,
                            keep_zeros=bool(rng.random() < 0.7))
    fc, fm = synth.make_fragments(bins, R)
    ids = rng.permutation(np.arange(n_chrom) * 2 + 1)               # chromosome ids: not 0..n-1, not in file order
    chrom = ids[c["chrom"]].astype(np.int32)
    fc = ids[fc].astype(np.int32)
    barr = None
    if with_bias:
        bc = np.concatenate([np.full(b, ids[i]) for i, b in enumerate(bins)]).astype(np.int32)
        bm = fm.copy()
        bv = np.concatenate(bias)
        drop = rng.random(bc.size) < 0.1                            # loci without a bias
        if n_chrom > 1:
            drop |= bc == ids[0]                                    # and a chromosome without any
        barr = (bc[~drop], bm[~drop], bv[~drop])
    n_bins = int(rng.choice([30, 100]))
    return dict(R=R, max_dist=max_dist, min_dist=min_dist, n_bins=n_bins, chrom=chrom, mid1=c["mid1"], mid2=c["mid2"],
                count=c["count"], fc=fc, fm=fm, bias=barr, ids=ids)


def _alone(g, c, q_values, n_tests):
    """fit_transform_arrays for chromosome c alone: its rows, its fragments, its bias rows."""
    from blueberry_b200.fithic import FitHiC
    model = FitHiC("x", g["R"], n_bins=g["n_bins"], max_dist=g["max_dist"], min_dist=g["min_dist"])
    rows = np.flatnonzero(g["chrom"] == c)
    fs = g["fc"] == c
    b = None
    if g["bias"] is not None:
        bs = g["bias"][0] == c
        b = tuple(a[bs] for a in g["bias"])
    return model.fit_transform_arrays(g["chrom"][rows], g["mid1"][rows], g["chrom"][rows], g["mid2"][rows], g["count"][rows],
                                      g["fc"][fs], g["fm"][fs], bias=b, q_values=q_values, n_tests=n_tests)


def _assert_same_output(a, b):
    for f in ("p", "q", "keep", "x", "y", "spline_y", "spline_y_raw", "possible", "observed", "bin_of_key"):
        va, vb = getattr(a, f), getattr(b, f)
        assert (va is None) == (vb is None), f
        if va is not None:
            assert va.dtype == vb.dtype and va.shape == vb.shape and _bits(va) == _bits(vb), f
    assert struct.pack("d", a.residual) == struct.pack("d", b.residual)
    assert a.totals == b.totals
    assert _fit_bytes(a.fit) == _fit_bytes(b.fit)


def _check_against_loop(g, q_values, n_tests):
    """per_chromosome=True against the single calls in ascending id order: every field bit for bit, or, when a single call
    raises, the same exception type naming the lowest failing chromosome.  Returns the output (None when it raised)."""
    from blueberry_b200.fithic import FitHiC
    model = FitHiC("x", g["R"], n_bins=g["n_bins"], max_dist=g["max_dist"], min_dist=g["min_dist"])
    alone, first_error = {}, None
    for c in sorted(int(x) for x in g["ids"]):
        try:
            alone[c] = _alone(g, c, q_values, n_tests.get(c) if n_tests else None)
        except Exception as e:
            first_error = (c, e)
            break
    call = lambda: model.fit_transform_arrays(g["chrom"], g["mid1"], g["chrom"], g["mid2"], g["count"], g["fc"], g["fm"],
                                              bias=g["bias"], q_values=q_values, n_tests=n_tests, per_chromosome=True)
    if first_error is not None:
        with pytest.raises(type(first_error[1]), match="chromosome %d:" % first_error[0]):
            call()
        return None
    out = call()
    assert sorted(out) == sorted(alone)
    for c in sorted(out):
        rows = np.flatnonzero(g["chrom"] == c)
        assert out[c].rows == (int(rows[0]), int(rows[-1]) + 1)
        _assert_same_output(out[c], alone[c])
    return out


@pytest.mark.parametrize("seed", range(8))
def test_per_chromosome_equals_the_loop_of_single_calls(seed):
    g = _random_genome(seed)
    rng = np.random.default_rng(1000 + seed)
    n_tests = None
    if seed in (2, 6):
        n_tests = {int(c): int(rng.integers(5, 5000)) for c in g["ids"][::2]}
    assert _check_against_loop(g, seed != 3, n_tests) is not None


def test_per_chromosome_tiny_and_failed_chromosomes():
    """A chromosome cut to three in-range rows and one cut to a single in-range row, against their single calls.  Then
    chromosomes whose counts are all zero (S == 0): the call raises what their single call raises (ZeroDivisionError),
    naming the LOWEST such id."""
    g = next(x for x in (_random_genome(s) for s in range(4, 60)) if len(x["ids"]) >= 4)
    ids = sorted(int(c) for c in g["ids"])
    d = g["mid2"].astype(np.int64) - g["mid1"].astype(np.int64)
    in_range = (d > g["min_dist"]) & (d <= g["max_dist"])
    keepm = np.ones(len(g["chrom"]), bool)
    for c, n in ((ids[1], 3), (ids[2], 1)):
        rows = np.flatnonzero(g["chrom"] == c)
        keepm[rows] = False
        keepm[rows[in_range[rows]][:n]] = True
    for k in ("chrom", "mid1", "mid2", "count"):
        g[k] = g[k][keepm]
    g["count"] = g["count"].copy()
    g["count"][np.isin(g["chrom"], ids[1:3])] = 5
    assert [int((g["chrom"] == c).sum()) for c in ids[1:3]] == [3, 1]
    _check_against_loop(g, True, None)
    for zeros in ([ids[-1]], [ids[0], ids[-1]]):
        g["count"] = g["count"].copy()
        g["count"][np.isin(g["chrom"], zeros)] = 0
        with pytest.raises(ZeroDivisionError):
            _alone(g, zeros[0], True, None)
        _check_against_loop(g, True, None)


# ------------------------------------------------------------------------------------------------ against the oracle
def test_per_chromosome_against_oracle_on_each_chromosome():
    from blueberry_b200 import synth
    from blueberry_b200.fithic import FitHiC
    from oracle import fithic_oracle as fo
    R, bins, max_dist = 10000, [420, 300, 180], 2_000_000
    fc, fm = synth.make_fragments(bins, R)
    bias = synth.make_bias(bins, 11)
    c = synth.make_contacts(bins, R, max_dist, 150.0, 31, bias)
    bc = np.concatenate([np.full(b, i) for i, b in enumerate(bins)]).astype(np.int32)
    bv = np.concatenate(bias)
    model = FitHiC("x", R, n_bins=100, max_dist=max_dist, min_dist=0)
    out = model.fit_transform_arrays(c["chrom"], c["mid1"], c["chrom"], c["mid2"], c["count"], fc, fm, bias=(bc, fm, bv),
                                     q_values=True, per_chromosome=True)
    for ci in range(len(bins)):
        o = out[ci]
        r = c["chrom"] == ci
        f = fc == ci
        bd, _ = fo.read_bias_arrays(bc[f], fm[f], bv[f])
        ref = fo.fithic_arrays(fc[f], fm[f], c["chrom"][r], c["mid1"][r], c["chrom"][r], c["mid2"][r], c["count"][r], R, 100, 0,
                               max_dist, bias=bd)
        assert np.array_equal(o.observed, ref.contacts.observed) and o.totals["observedIntraInRangeSum"] == ref.contacts.S
        assert np.array_equal(o.x, np.array(ref.x)) and np.array_equal(o.y, np.array(ref.y))
        assert np.array_equal(o.spline_y, ref.spline_y)
        assert np.array_equal(o.keep, ref.keep)
        sel = ref.keep & (ref.p > 0)
        ok, nbad = log10_close(o.p[sel], ref.p[sel], 1e-6)
        assert ok, nbad
        keep = ref.keep
        assert np.array_equal(o.q[keep], fo.benjamini_hochberg_correction(o.p[keep], int(keep.sum())))
        q_ref = fo.benjamini_hochberg_correction(ref.p[keep], int(keep.sum()))
        ok, nbad = log10_close(o.q[keep], q_ref, 1e-6)
        assert ok, "chromosome %d: %d q-values differ from BH(reference p) by more than 1e-6 in log10" % (ci, nbad)
        # ranks outside declared near-ties (the rule of test_several_shards_against_oracle_and_reference_q)
        pr, pg = ref.p[keep], o.p[keep]
        order = np.argsort(pr, kind="stable")
        srt = pr[order]
        with np.errstate(divide="ignore"):
            gap = np.diff(np.log10(np.maximum(srt, 1e-320)))
        near = np.zeros(len(srt), bool)
        close = gap < 2e-6
        near[1:] |= close
        near[:-1] |= close
        rank_ref = np.searchsorted(srt, pr, side="left")
        rank_gpu = np.searchsorted(np.sort(pg), pg, side="left")
        tied_ref = np.zeros(len(pr), bool)
        tied_ref[order] = near
        assert not ((rank_ref != rank_gpu) & ~tied_ref).any()


# ------------------------------------------------------------------------------------------------ scale
def test_config2_shape_chromosomes_with_an_overflowing_deferred_list():
    """Three chromosomes of BASELINE config 2's shape (5 kb, 10 Mb cap), a deferred list too small for at least one of them:
    ChromosomePass repairs it and every chromosome equals its pass alone (GenomePass), bit for bit."""
    import torch
    from blueberry_b200 import synth
    from blueberry_b200.distributed import ChromosomePass, GenomePass
    from blueberry_b200.engine import BiasTables, PassEngine, Shard
    dev = torch.device("cuda", 0)
    R, bins, max_dist = 5000, [3000, 2400, 1500], 10_000_000
    bias = synth.make_bias(bins, 3)
    c = synth.make_contacts(bins, R, max_dist, 600.0, 77, bias)
    tabs = BiasTables([np.where((b < 0.5) | (b > 2), -1.0, b) for b in bias], [R // 2] * len(bins), dev)

    def engine(i):
        e = PassEngine(R, 100, 0, max_dist, bins[i], dev)
        e.set_fragments([bins[i]], [(bins[i] - 1) * R])
        e.set_bias(tabs)
        return e

    shards = []
    for i in range(len(bins)):
        sel = np.flatnonzero(c["chrom"] == i)
        shards.append(Shard(_t32(c["mid1"][sel], dev), _t32(c["mid2"][sel], dev), _t32(c["count"][sel], dev), chrom=i))
    cap = 1 << 14
    cp = ChromosomePass([engine(i) for i in range(len(bins))], shards, q_values=True, list_capacity=cap)
    fits = cp.run()
    grown = [i for i in range(len(bins)) if cp.lists[i][3].capacity > cap]
    assert grown                                                   # at least one chromosome overflowed and was repaired
    for i in range(len(bins)):
        assert cp.last_state[i][1].overflow == 0
        gp = GenomePass(engine(i), group=False, q_values=True)
        gp.attach([shards[i]])
        fit = gp.run()
        assert _fit_bytes(bytes(fit)) == _fit_bytes(bytes(fits[i]))
        assert _bits(gp.shard_p(0).cpu().numpy()) == _bits(cp.chrom_p(i).cpu().numpy())
        assert _bits(gp.shard_q(0).cpu().numpy()) == _bits(cp.chrom_q(i).cpu().numpy())
