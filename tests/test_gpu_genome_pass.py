"""GPU tests of the multi-shard / multi-GPU pass (blueberry_b200.distributed.GenomePass) and of the streaming K4 it runs
(bbk_score_guard -> bbk_score_pairs -> bbk_score_deferred -> bbk_bh_qvalues_listed):

  * the streaming path against the direct kernel (bbk_pvalues + bbk_bh_qvalues): same NaN rows, same rows at exactly 1.0,
    every other p within 1e-9 (relative), q bit for bit the reference's BH of the p beside it - whatever the shard
    sizes, tails, biases, zero rows (shards with chromosome columns take the direct kernel inside GenomePass);
  * the exact mode the guard falls back to (every in-range row through its prior) and the guard's own decision;
  * several shards on one GPU against the CPU oracle on the concatenated records (genome-wide S, spline and q);
  * q end to end against BH over the REFERENCE's p (log10 tolerance; identical ranks outside declared near-ties);
  * BASELINE config 2's shape on a 1e7-record sample against the oracle;
  * N > 1 GPUs (skipped on a one-GPU box): tests/multi_gpu_check.py under torchrun for world 2, 4, 8.
"""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest

from helpers import log10_close

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _engine(bins, R, min_dist, max_dist, bias, dev, n_bins=100):
    from blueberry_b200.engine import BiasTables, PassEngine
    nkeys = max(bins)
    eng = PassEngine(R, n_bins, min_dist, max_dist, nkeys, dev)
    eng.set_fragments(bins, [(b - 1) * R for b in bins])
    if bias is not None:
        tabs = [np.where((b < 0.5) | (b > 2), -1.0, b) for b in bias]
        eng.set_bias(BiasTables(tabs, [R // 2] * len(bins), dev))
    return eng


def _t32(a, dev):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.int32)).to(dev)


def _direct(eng, shards, dev, n_tests=-1):
    """The direct kernels on the same shards: p per shard, q over the concatenation (one ranking)."""
    import torch
    from blueberry_b200 import _lib
    from blueberry_b200.distributed import layout_rows
    starts, rows = layout_rows([s.n for s in shards])
    rows = max(rows, 4)
    p = torch.full((rows,), float("nan"), dtype=torch.float64, device=dev)
    q = torch.full((rows,), float("nan"), dtype=torch.float64, device=dev)
    for s, a in zip(shards, starts):
        if s.n:
            eng.pvalues(s, p[a:a + s.n])
    ws = torch.empty(int(eng.lib.bbk_bh_workspace_bytes(rows)), dtype=torch.uint8, device=dev)
    _lib.check(eng.lib.bbk_bh_qvalues(_lib.ptr(p), rows, n_tests, _lib.BH_UNSORTED, None, _lib.ptr(q), None, _lib.ptr(ws), ws.numel(),
                                      _lib.stream_ptr()), "bbk_bh_qvalues")
    torch.cuda.synchronize()
    return p.cpu().numpy(), q.cpu().numpy(), starts


def _same(a, b):
    return np.array_equal(np.isnan(a), np.isnan(b)) and np.array_equal(a[~np.isnan(a)], b[~np.isnan(b)])


def _close(a, b, rel=1e-9):
    """Same NaN pattern, the same rows at exactly 0.0, everything else within `rel` (relative).  The streaming path and the
    general kernel evaluate the same tail with different but equivalent sums (lower tail for small counts; the general kernel's
    upper sum for a count far below the mean adds ~lambda rising terms and lands within ~1e-12 of 1.0 where the lower tail gives
    1.0 exactly; its serial general form on a shard's last n % 4 records), so they agree to rounding, not to the bit."""
    if not np.array_equal(np.isnan(a), np.isnan(b)):
        return False
    ok = ~np.isnan(a)
    a, b = a[ok], b[ok]
    if not np.array_equal(a == 0.0, b == 0.0):
        return False
    pos = (a > 0) & (b > 0)
    return bool((np.abs(a[pos] / b[pos] - 1.0) <= rel).all())


def _bh_of(p):
    """The reference's BH over the non-NaN rows of p, N = their number (the oracle's restatement of fithic.py:466-487)."""
    from oracle import fithic_oracle as fo
    q = np.full(len(p), np.nan)
    ok = ~np.isnan(p)
    q[ok] = fo.benjamini_hochberg_correction(p[ok], int(ok.sum()))
    return q


def _random_shards(seed, dev, with_chr=False):
    """Shards with awkward sizes (tails of 0..3 records, a one-record shard, an empty one), off-grid / negative / out-of-range
    distances, zero and negative counts."""
    import torch
    from blueberry_b200 import synth
    from blueberry_b200.engine import Shard
    rng = np.random.default_rng(seed)
    bins = [int(rng.integers(150, 500)) for _ in range(3)]
    R = int(rng.choice([1000, 5000, 10000]))
    max_dist = int(rng.choice([40, 90, 10 ** 5])) * R
    min_dist = int(rng.choice([0, 0, 3 * R]))
    with_bias = bool(rng.random() < 0.75)
    bias = synth.make_bias(bins, seed, sigma=0.3) if with_bias else None
    c = synth.make_contacts(bins, R, min(max_dist, max(bins) * R), float(rng.choice([2.0, 40.0, 600.0])), seed, bias, keep_zeros=bool(rng.random() < 0.7))
    chrom, m1, m2, cn = c["chrom"].copy(), c["mid1"].copy(), c["mid2"].copy(), c["count"].copy()
    n = len(cn)
    k = rng.choice(n, max(n // 60, 1), replace=False); m2[k] += 333                    # off-grid
    k = rng.choice(n, max(n // 90, 1), replace=False); m1[k], m2[k] = m2[k].copy(), m1[k].copy()   # negative distances
    k = rng.choice(n, max(n // 200, 1), replace=False); cn[k] = -2                      # negative counts score like zeros
    k = rng.choice(n, max(n // 300, 1), replace=False); cn[k] = 700                     # far above any mean
    shards, parts = [], []
    for ci in range(len(bins)):
        sel = np.flatnonzero(chrom == ci)
        cut = int(rng.integers(1, max(len(sel) - 1, 2)))
        for piece in (sel[:cut], sel[cut:cut + 1], sel[cut + 1:]):                      # three pieces, one of them a single record
            parts.append((ci, piece))
    parts.insert(2, (0, np.zeros(0, dtype=np.int64)))                                   # an empty shard
    for ci, piece in parts:
        if with_chr:
            c2 = np.full(len(piece), ci, dtype=np.int32)
            if len(piece) > 10:
                c2[rng.choice(len(piece), 3, replace=False)] = (ci + 1) % len(bins)      # inter-chromosomal rows
            shards.append(Shard(_t32(m1[piece], dev), _t32(m2[piece], dev), _t32(cn[piece], dev),
                                _t32(np.full(len(piece), ci), dev), _t32(c2, dev)))
        else:
            shards.append(Shard(_t32(m1[piece], dev), _t32(m2[piece], dev), _t32(cn[piece], dev), chrom=ci))
    eng = _engine(bins, R, min_dist, max_dist, bias, dev, n_bins=int(rng.choice([30, 100])))
    return eng, shards


@pytest.mark.parametrize("seed,with_chr", [(s, False) for s in range(8)] + [(s, True) for s in range(8, 12)])
def test_split_k4_matches_the_direct_kernel(seed, with_chr):
    import torch
    from blueberry_b200.distributed import GenomePass
    dev = torch.device("cuda", 0)
    eng, shards = _random_shards(seed, dev, with_chr)
    gp = GenomePass(eng, group=False, q_values=True)
    gp.attach(shards)
    assert gp.listed == (not with_chr)
    try:
        gp.run()
    except (ZeroDivisionError, ValueError):
        pytest.skip("degenerate random case (the fit raises, as the reference would)")
    p_new, q_new = gp.p.cpu().numpy(), gp.q.cpu().numpy()
    score = gp.last_score
    assert score.overflow == 0 and score.cand_overflow == 0
    p_old, q_old, starts = _direct(eng, shards, dev)
    assert gp.offsets == starts
    assert _close(p_new[:gp.rows], p_old[:gp.rows]), "p differs between the split and the direct kernel"
    assert _same(q_new[:gp.rows], _bh_of(p_new[:gp.rows])), "q is not the reference's BH of the p beside it"
    assert _close(q_new[:gp.rows], q_old[:gp.rows], 1e-8), "q differs between the listed and the full Benjamini-Hochberg step"


@pytest.mark.parametrize("case", ["sizes", "negative", "wide_bias", "no_bias_row", "all_zero", "all_out_of_range", "dense_hits"])
def test_streaming_k4_edge_shapes(case):
    """The corners of bbk_score_pairs against the general kernel: shard sizes around the 4-row group and the 256-row warp tile,
    negative coordinates (the wrapped subtraction is not the distance), a bias table the 32-bit path cannot index (wide path),
    a chromosome without bias entries, shards of zero counts only / out-of-range rows only, and tiles in which nearly every row
    is deferred and a q-value candidate (the warp buffers flush many times per tile)."""
    import torch
    from blueberry_b200 import synth
    from blueberry_b200.distributed import GenomePass
    from blueberry_b200.engine import BiasTables, PassEngine, Shard
    dev = torch.device("cuda", 0)
    rng = np.random.default_rng(hash(case) % 1000)
    R, bins, max_dist = 5000, [700, 400], 600 * 5000
    bias = synth.make_bias(bins, 8, sigma=0.3)
    c = synth.make_contacts(bins, R, max_dist, 300.0 if case == "dense_hits" else 30.0, 3, bias)
    chrom, m1, m2, cn = c["chrom"], c["mid1"].copy(), c["mid2"].copy(), c["count"].copy()
    eng = PassEngine(R, 100, 0, max_dist, max(bins), dev)
    eng.set_fragments(bins, [(b - 1) * R for b in bins])
    tabs = [np.where((b < 0.5) | (b > 2), -1.0, b) for b in bias]
    mid0 = [R // 2, R // 2]
    if case == "wide_bias":
        tabs[0] = np.concatenate([np.full(3, np.nan), tabs[0]])
        mid0 = [R // 2 - 3 * R, R // 2]                       # a table that starts below zero: the 64-bit lookup
    if case == "no_bias_row":
        tabs = tabs[:1]
        mid0 = mid0[:1]                                        # chromosome 1 has no table at all
    eng.set_bias(BiasTables(tabs, mid0, dev))
    sel0, sel1 = np.flatnonzero(chrom == 0), np.flatnonzero(chrom == 1)
    if case == "negative":
        k = rng.choice(len(sel0), 300, replace=False)
        m1[sel0[k]] = -m1[sel0[k]] - 1                         # mid1 < 0: in range as a number, never a table hit
        k = rng.choice(len(sel0), 300, replace=False)
        m1[sel0[k]], m2[sel0[k]] = m2[sel0[k]].copy(), -m1[sel0[k]].copy() - 7   # mid2 < mid1 with a huge wrapped difference
    if case == "all_zero":
        cn[sel0] = 0
    if case == "all_out_of_range":
        m2[sel1] = m1[sel1] + max_dist + R
    if case == "dense_hits":
        cn[sel0[:5000]] += 900                                 # a run of rows far above any mean: deferred and significant
    pieces = []
    if case == "sizes":
        at = 0
        for n in (1, 2, 3, 4, 5, 255, 256, 257, 260, 511, 513, 1023, 1025, 4099):
            pieces.append((0, sel0[at:at + n])); at += n
        pieces.append((1, sel1))
    else:
        pieces = [(0, sel0), (1, sel1)]
    shards = [Shard(_t32(m1[ix], dev), _t32(m2[ix], dev), _t32(cn[ix], dev), chrom=ci) for ci, ix in pieces]
    gp = GenomePass(eng, group=False, q_values=True)
    gp.attach(shards)
    assert gp.listed
    gp.run()
    p_old, q_old, _ = _direct(eng, shards, dev)
    p_new, q_new = gp.p.cpu().numpy()[:gp.rows], gp.q.cpu().numpy()[:gp.rows]
    assert _close(p_new, p_old[:gp.rows]), case
    assert _same(q_new, _bh_of(p_new)), case
    if case == "dense_hits":
        assert gp.last_score.n_list > 4000 and gp.last_score.n_cand > 4000


@pytest.mark.parametrize("seed", [1, 5])
def test_exact_mode_equals_speculative_mode(seed):
    """What the guard falls back to: every in-range row through its prior.  Forced here by raising BbkScoreState.exact
    right after the guard (the guard itself is tested below)."""
    import torch
    from blueberry_b200.distributed import GenomePass
    dev = torch.device("cuda", 0)
    eng, shards = _random_shards(seed, dev)
    gp = GenomePass(eng, group=False, q_values=True)
    gp.attach(shards)
    gp.run()
    assert gp.last_score.exact == 0
    p_spec, q_spec = gp.p.clone(), gp.q.clone()
    gp.p.fill_(7.0); gp.q.fill_(7.0)
    gp.force_exact = True
    gp.run()
    assert gp.last_score.exact == 1
    rows = gp.rows
    real = np.ones(rows, bool)                                                          # (padding rows are rewritten too: NaN)
    assert _same(gp.p.cpu().numpy()[:rows][real], p_spec.cpu().numpy()[:rows][real])
    assert _same(gp.q.cpu().numpy()[:rows][real], q_spec.cpu().numpy()[:rows][real])


def test_guard_decision():
    import torch
    from blueberry_b200 import _lib
    dev = torch.device("cuda", 0)
    lib = _lib.load()

    def run(values, status=0):
        fit = _lib.FitResult()
        fit.status, fit.L = status, len(values)
        d_fit = torch.frombuffer(bytearray(bytes(fit)), dtype=torch.uint8).to(dev)
        sy = torch.tensor(values, dtype=torch.float64, device=dev)
        state = torch.zeros(ctypes.sizeof(_lib.ScoreState), dtype=torch.uint8, device=dev)
        _lib.check(lib.bbk_score_guard(_lib.ptr(d_fit), _lib.ptr(sy), _lib.ptr(state), _lib.stream_ptr()), "guard")
        return _lib.ScoreState.from_buffer_copy(state.cpu().numpy().tobytes()).exact

    assert run([1e-3, 1e-5, 1e-9]) == 0
    assert run([0.0625] * 2000) == 0                   # 16 * max == 1: still inside [0, 1]
    assert run([0.07, 1e-5]) == 1                      # a bias product of 16 could push the prior above 1
    assert run([1e-3, 0.0]) == 0                       # prior 0 (or -0.0 with a negative bias, which bdtrc accepts) gives p = 1.0 for count <= 0
    assert run([1e-3, -1e-12]) == 1
    assert run([1e-3, float("nan")]) == 1
    assert run([0.5], status=-12) == 0                 # failed fit: nothing is scored, the host raises


def test_several_shards_against_oracle_and_reference_q():
    """Three chromosomes as five shards on one GPU, scored with ONE genome-wide table / S / spline, q ranked over all of them:
    against the CPU oracle on the concatenated records.  q is also compared with BH over the ORACLE's p (the reference's
    p): ranks identical outside near-ties, log10 q within the p tolerance."""
    import torch
    from blueberry_b200 import synth
    from blueberry_b200.distributed import GenomePass
    from blueberry_b200.engine import Shard
    from oracle import fithic_oracle as fo
    dev = torch.device("cuda", 0)
    R, bins, max_dist = 10000, [420, 300, 180], 2_000_000
    fc, fm = synth.make_fragments(bins, R)
    bias = synth.make_bias(bins, 11)
    c = synth.make_contacts(bins, R, max_dist, 150.0, 31, bias)
    eng = _engine(bins, R, 0, max_dist, bias, dev)
    cuts = [0, 30000, int((c["chrom"] == 0).sum()), int((c["chrom"] <= 1).sum()) - 17, int((c["chrom"] <= 1).sum()), len(c["count"])]
    shards = []
    for a, b in zip(cuts[:-1], cuts[1:]):
        shards.append(Shard(_t32(c["mid1"][a:b], dev), _t32(c["mid2"][a:b], dev), _t32(c["count"][a:b], dev), chrom=int(c["chrom"][a])))
    gp = GenomePass(eng, group=False, q_values=True)
    gp.attach(shards)
    fit = gp.run()
    p = np.concatenate([gp.shard_p(i).cpu().numpy() for i in range(len(shards))])
    q = np.concatenate([gp.shard_q(i).cpu().numpy() for i in range(len(shards))])
    bc = np.concatenate([np.full(b, i) for i, b in enumerate(bins)])
    bd, _ = fo.read_bias_arrays(bc, fm, np.concatenate(bias))
    ref = fo.fithic_arrays(fc, fm, c["chrom"], c["mid1"], c["chrom"], c["mid2"], c["count"], R, 100, 0, max_dist, bias=bd)
    assert np.array_equal(eng.obs_sum.cpu().numpy(), ref.contacts.observed) and int(fit.S) == ref.contacts.S
    assert np.array_equal(eng.spline_y[:fit.L].cpu().numpy(), ref.spline_y)
    assert np.array_equal(p <= 1, ref.keep)
    sel = ref.keep & (ref.p > 0)
    ok, nbad = log10_close(p[sel], ref.p[sel], 1e-6)
    assert ok, nbad
    # q on the device's own p: bit-exact BH
    keep = ref.keep
    assert np.array_equal(q[keep], fo.benjamini_hochberg_correction(p[keep], int(keep.sum())))
    # q against BH of the REFERENCE's p
    q_ref = fo.benjamini_hochberg_correction(ref.p[keep], int(keep.sum()))
    ok, nbad = log10_close(q[keep], q_ref, 1e-6)
    assert ok, "%d q-values differ from BH(reference p) by more than 1e-6 in log10" % nbad
    # ranks: 1 + number of strictly smaller p.  Declared near-ties: pairs of DISTINCT reference p-values closer than 1e-6 in log10
    pr, pg = ref.p[keep], p[keep]
    order = np.argsort(pr, kind="stable")
    srt = pr[order]
    with np.errstate(divide="ignore"):
        gap = np.diff(np.log10(np.maximum(srt, 1e-320)))
    near = np.zeros(len(srt), bool)
    close = gap < 2e-6                                  # neighbours in the reference's order that the tolerance cannot separate
    near[1:] |= close; near[:-1] |= close
    rank_ref = np.searchsorted(srt, pr, side="left")
    rank_gpu = np.searchsorted(np.sort(pg), pg, side="left")
    tied_ref = np.zeros(len(pr), bool)
    tied_ref[order] = near
    bad = (rank_ref != rank_gpu) & ~tied_ref
    # (rows inside a cluster may swap or merge; that never changes how many rows lie strictly below a row OUTSIDE it)
    assert not bad.any(), "%d rows outside declared near-ties changed rank" % int(bad.sum())


def test_config2_shape_sample_against_oracle():
    """BASELINE config 2's shape (5 kb, 10 Mb cap, D = 2001, deep counts near the diagonal) on a 5000-bin chromosome =
    8.0e6 records, against the oracle."""
    import torch
    from blueberry_b200 import synth
    from blueberry_b200.distributed import GenomePass
    from blueberry_b200.engine import Shard
    from oracle import fithic_oracle as fo
    dev = torch.device("cuda", 0)
    R, bins, max_dist = 5000, [5000], 10_000_000
    fc, fm = synth.make_fragments(bins, R)
    bias = synth.make_bias(bins, 3)
    c = synth.make_contacts(bins, R, max_dist, 600.0, 77, bias)
    eng = _engine(bins, R, 0, max_dist, bias, dev)
    sh = Shard(_t32(c["mid1"], dev), _t32(c["mid2"], dev), _t32(c["count"], dev), chrom=0)
    gp = GenomePass(eng, group=False, q_values=True)
    gp.attach([sh])
    fit = gp.run()
    p, q = gp.shard_p(0).cpu().numpy(), gp.shard_q(0).cpu().numpy()
    bd, _ = fo.read_bias_arrays(np.zeros(bins[0], dtype=np.int64), fm, bias[0])
    ref = fo.fithic_arrays(fc, fm, None, c["mid1"], None, c["mid2"], c["count"], R, 100, 0, max_dist, bias=bd)
    assert np.array_equal(eng.obs_sum.cpu().numpy(), ref.contacts.observed) and int(fit.S) == ref.contacts.S
    assert np.array_equal(eng.x[:fit.n_out].cpu().numpy(), np.array(ref.x)) and np.array_equal(eng.y[:fit.n_out].cpu().numpy(), np.array(ref.y))
    assert np.array_equal(eng.spline_y[:fit.L].cpu().numpy(), ref.spline_y)
    assert np.array_equal(p <= 1, ref.keep)
    sel = ref.keep & (ref.p >= 1e-300)
    ok, nbad = log10_close(p[sel], ref.p[sel], 1e-5)
    assert ok, nbad
    keep = ref.keep
    assert np.array_equal(q[keep], fo.benjamini_hochberg_correction(p[keep], int(keep.sum())))
    assert gp.last_score.exact == 0


def test_config4_shape_sample_two_pass_against_oracle():
    """BASELINE config 4's shape (1 kb, 2 Mb cap, D = 2001, depth 60: ~93 % of the records have count 0), both passes -
    the fit, the outlier cut at 1 / possibleIntraInRangeCount, the refit over the remaining records, every record scored
    again - on a 4000-bin chromosome = 6.0e6 records, through the drop-in entry point, against the oracle's composition of
    the reference's functions (SURVEY.md 8c)."""
    import warnings
    from blueberry_b200 import synth
    from blueberry_b200.fithic import FitHiC
    from oracle import fithic_oracle as fo
    R, bins, max_dist = 1000, [4000], 2_000_000
    fc, fm = synth.make_fragments(bins, R)
    bias = synth.make_bias(bins, 4)
    c = synth.make_contacts(bins, R, max_dist, 60.0, 404, bias)
    assert 0.85 < float((c["count"] == 0).mean()) < 0.97
    bd, _ = fo.read_bias_arrays(np.zeros(bins[0], dtype=np.int64), fm, bias[0])
    model = FitHiC("unused", R, n_bins=100, max_dist=max_dist, min_dist=0)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        r1, r2, outlier, thr = fo.fithic_two_pass_arrays(fc, fm, c["chrom"], c["mid1"], c["chrom"], c["mid2"], c["count"], R, 100,
                                                         model.min_dist, model.max_dist, bias=bd)
    with np.errstate(invalid="ignore", divide="ignore"):
        assert not (r1.keep & (np.abs(r1.p / thr - 1.0) < 1e-9)).any()          # no record sits on the outlier threshold
    assert int(outlier.sum()) > 0
    barr = (np.zeros(bins[0], dtype=np.int32), fm.copy(), bias[0])
    out = model.fit_transform_arrays(c["chrom"], c["mid1"], c["chrom"], c["mid2"], c["count"], fc, fm, bias=barr, refit=True, q_values=True)
    assert np.array_equal(out.observed, r2.contacts.observed)
    assert out.totals["observedIntraInRangeSum"] == r2.contacts.S
    assert np.array_equal(out.x, np.array(r2.x)) and np.array_equal(out.y, np.array(r2.y))
    assert np.array_equal(out.spline_y, r2.spline_y)
    assert np.array_equal(out.keep, r2.keep)
    sel = r2.keep & (r2.p >= 1e-300)
    ok, nbad = log10_close(out.p[sel], r2.p[sel], 1e-5)
    assert ok, "%d p-values differ by more than 1e-5 in log10" % nbad
    assert np.array_equal(out.q[out.keep], fo.benjamini_hochberg_correction(out.p[out.keep], int(out.keep.sum())))


def test_two_passes_in_flight_equal_serial_passes():
    """Independent passes on two streams, each with its own engine and GenomePass (bench.py's two_passes_in_flight): the same
    records through both lanes, and different records through the two lanes at once, against each lane run alone."""
    import torch
    from blueberry_b200 import synth
    from blueberry_b200.distributed import GenomePass
    from blueberry_b200.engine import Shard
    dev = torch.device("cuda", 0)
    R, bins, max_dist = 5000, [900, 700], 2_000_000
    bias = synth.make_bias(bins, 5)
    lanes = []
    for seed, depth in ((11, 80.0), (12, 9.0)):
        c = synth.make_contacts(bins, R, max_dist, depth, seed, bias)
        shards = []
        for ci in range(len(bins)):
            sel = np.flatnonzero(c["chrom"] == ci)
            shards.append(Shard(_t32(c["mid1"][sel], dev), _t32(c["mid2"][sel], dev), _t32(c["count"][sel], dev), chrom=ci))
        gp = GenomePass(_engine(bins, R, 0, max_dist, bias, dev), group=False, q_values=True)
        gp.attach(shards)
        gp.run()
        lanes.append((gp, gp.p.clone(), gp.q.clone(), torch.cuda.Stream(dev)))
    torch.cuda.synchronize()
    main = torch.cuda.current_stream(dev)
    for gp, _, _, st in lanes:
        gp.p.fill_(7.0); gp.q.fill_(7.0)
        st.wait_stream(main)
    for _ in range(3):
        for gp, _, _, st in lanes:
            with torch.cuda.stream(st):
                gp.enqueue()
    for gp, p_alone, q_alone, st in lanes:
        with torch.cuda.stream(st):
            gp.finish()
        assert _same(gp.p.cpu().numpy()[:gp.rows], p_alone.cpu().numpy()[:gp.rows])
        assert _same(gp.q.cpu().numpy()[:gp.rows], q_alone.cpu().numpy()[:gp.rows])


def test_list_overflow_is_detected_and_repaired():
    import torch
    from blueberry_b200.distributed import GenomePass
    dev = torch.device("cuda", 0)
    eng, shards = _random_shards(3, dev)
    gp = GenomePass(eng, group=False, q_values=True)
    gp.attach(shards, list_capacity=64, cand_capacity=8)            # far too small
    gp.run()                                                        # finish() sees the flag and repeats with a full-size list
    assert gp.last_score.overflow == 0
    p_old, q_old, _ = _direct(eng, shards, dev)
    assert _close(gp.p.cpu().numpy()[:gp.rows], p_old[:gp.rows])
    assert _same(gp.q.cpu().numpy()[:gp.rows], _bh_of(gp.p.cpu().numpy()[:gp.rows]))     # the candidate overflow falls back to the full pass: still exact


@pytest.mark.parametrize("n_tests", [-1, 25])
def test_k4_handover_matches_two_pass_qvalues(n_tests):
    """The streaming K4's hand-over to K5 (q pre-filled, the small p listed, bbk_bh_qvalues_listed) against bbk_bh_qvalues on
    the pass's own p, bit for bit.  n_tests = 25 pushes the saturation bucket above 2^-5, so the listed call has to fall back
    to the full pass on its own (and q of the p == 1.0 rows drops below 1)."""
    import torch
    from blueberry_b200 import _lib
    from blueberry_b200.distributed import GenomePass
    from blueberry_b200.engine import BiasTables, PassEngine, Shard
    lib = _lib.load()
    dev = torch.device("cuda:0")
    R, nb, K = 5000, 7001, 300
    P = int(lib.bbk_synth_n_pairs(nb, K))
    assert P % 4 != 0                                 # the shard ends inside a group of four rows
    rng = np.random.default_rng(9)
    bias_host = np.exp(rng.normal(0.0, 0.25, size=nb))
    bias_dev = torch.from_numpy(bias_host).to(dev)
    cols = [torch.empty(P, dtype=torch.int32, device=dev) for _ in range(3)]
    _lib.check(lib.bbk_synth_contacts(nb, K, R, 120.0, 1.08, 77, _lib.ptr(bias_dev), _lib.ptr(cols[0]), _lib.ptr(cols[1]),
                                      _lib.ptr(cols[2]), _lib.stream_ptr()), "synth")
    eng = PassEngine(R, 100, 0, K * R, nb, dev)
    eng.set_fragments([nb], [(nb - 1) * R])
    eng.set_bias(BiasTables([np.where((bias_host < 0.5) | (bias_host > 2), -1.0, bias_host)], [R // 2], dev))
    gp = GenomePass(eng, group=False, q_values=True)
    gp.attach([Shard(*cols)])
    assert gp.listed
    gp.run(n_tests=n_tests)
    use_list = int(gp.bh_ws[100:104].view(torch.int32)[0])          # BhState::use_list of the q-value step
    p1, q1 = gp.shard_p(0), gp.shard_q(0)
    q0 = torch.full((P + 3,), -7.0, dtype=torch.float64, device=dev)[:P]
    ws = torch.empty(int(lib.bbk_bh_workspace_bytes(P)), dtype=torch.uint8, device=dev)
    _lib.check(lib.bbk_bh_qvalues(_lib.ptr(p1), P, n_tests, _lib.BH_UNSORTED, None, _lib.ptr(q0), None, _lib.ptr(ws), ws.numel(),
                                  _lib.stream_ptr()), "bbk_bh_qvalues")
    torch.cuda.synchronize()
    assert torch.equal(q0.view(torch.int64), q1.view(torch.int64))
    assert use_list == (1 if n_tests < 0 else 0)
    if n_tests > 0:
        assert float(q1[p1 == 1.0][0]) < 1.0
    assert int((q1 < 1.0).sum()) > 1000


def test_fit_transform_arrays_pinned_and_wide_inputs():
    """The drop-in array call: pinned int32 torch columns, int64 numpy columns and a value beyond int32 (OverflowError)."""
    import torch
    from blueberry_b200 import synth
    from blueberry_b200.fithic import FitHiC
    R, bins, max_dist = 10000, [300, 200], 1_500_000
    fc, fm = synth.make_fragments(bins, R)
    c = synth.make_contacts(bins, R, max_dist, 80.0, 5)
    model = FitHiC("x", R, max_dist=max_dist)
    a = model.fit_transform_arrays(c["chrom"], c["mid1"], c["chrom"], c["mid2"], c["count"], fc, fm, q_values=True)
    pin = lambda v: torch.from_numpy(np.ascontiguousarray(v, dtype=np.int32)).pin_memory()
    b = model.fit_transform_arrays(c["chrom"], pin(c["mid1"]), c["chrom"], pin(c["mid2"]), pin(c["count"]), fc, fm, q_values=True)
    w = model.fit_transform_arrays(c["chrom"].astype(np.int64), c["mid1"].astype(np.int64), c["chrom"].astype(np.int64),
                                   c["mid2"].astype(np.int64), c["count"].astype(np.int64), fc, fm, q_values=True)
    for o in (b, w):
        assert _same(a.p, o.p) and _same(a.q, o.q)
    big = c["mid2"].astype(np.int64)
    big[7] = 2 ** 31 + 5
    with pytest.raises(OverflowError):
        model.fit_transform_arrays(c["chrom"], c["mid1"], c["chrom"], big, c["count"], fc, fm)


def _pack_roundtrip(p, q, dev, cap_p=None, cap_q=None):
    """bbk_pack_scores on the device, bbkio_unpack_scores on the host."""
    import torch
    from blueberry_b200 import _io, _lib
    lib = _lib.load()
    m = len(p)
    dp = torch.from_numpy(p).to(dev)
    dq = torch.from_numpy(q).to(dev) if q is not None else None
    cap_p = m if cap_p is None else cap_p
    cap_q = (m if cap_q is None else cap_q) if q is not None else 0
    codes = torch.zeros(max(int(lib.bbk_pack_code_words(m)), 1), dtype=torch.int32, device=dev)
    chunks = torch.zeros(max(int(lib.bbk_pack_chunks(m)), 1) * 24, dtype=torch.uint8, device=dev)
    vp = torch.zeros(max(cap_p, 1), dtype=torch.float64, device=dev)
    vq = torch.zeros(max(cap_q, 1), dtype=torch.float64, device=dev)
    state = torch.zeros(ctypes.sizeof(_lib.PackState), dtype=torch.uint8, device=dev)
    _lib.check(lib.bbk_pack_scores(_lib.ptr(dp), _lib.ptr(dq), m, _lib.ptr(codes), _lib.ptr(chunks), _lib.ptr(vp), cap_p,
                                   _lib.ptr(vq) if q is not None else None, cap_q, _lib.ptr(state), _lib.stream_ptr()), "bbk_pack_scores")
    torch.cuda.synchronize()
    st = _lib.PackState.from_buffer_copy(state.cpu().numpy().tobytes())
    if st.overflow:
        return st, None, None
    po, qo = _io.unpack_scores(codes.cpu().numpy(), chunks.cpu().numpy(), vp.cpu().numpy(), vq.cpu().numpy() if q is not None else None,
                               m, want_q=q is not None)
    return st, po, qo


@pytest.mark.parametrize("m", [0, 1, 15, 16, 17, 4095, 4096, 4097, 70001, 1 << 20])
def test_pack_scores_roundtrip_is_lossless(m):
    import torch
    dev = torch.device("cuda", 0)
    rng = np.random.default_rng(m + 1)
    p = rng.random(m)
    kind = rng.integers(0, 10, m)
    p[kind < 5] = 1.0
    p[kind == 5] = np.nan
    p[kind == 6] = 0.0
    p[kind == 7] = 5e-324 * rng.integers(1, 100, int((kind == 7).sum()))          # denormals
    q = np.where(np.isnan(p), np.nan, 1.0)
    sig = (kind >= 8) & ~np.isnan(p)
    q[sig] = np.minimum(p[sig] * 3.0, 1.0)
    q[(kind == 4)] = 0.25                                                         # p == 1.0 with q < 1 (the ones fix)
    st, po, qo = _pack_roundtrip(p, q, dev)
    assert st.overflow == 0 and int(st.n_p) == int(((p != 1.0) | (q != 1.0))[~(np.isnan(p) & np.isnan(q))].sum())
    assert np.array_equal(po.view(np.uint64), p.view(np.uint64)) and np.array_equal(qo.view(np.uint64), q.view(np.uint64))
    st, po, qo = _pack_roundtrip(p, None, dev)                                    # without q-values
    assert np.array_equal(po.view(np.uint64), p.view(np.uint64)) and qo is None
    if m >= 4096:
        st, po, qo = _pack_roundtrip(p, q, dev, cap_p=10, cap_q=10)               # too small: flagged, nothing written out of bounds
        assert st.overflow == 1


def test_host_stream_packed_results_equal_dense():
    """The end-to-end stream with packed results (two bits per row + the values that are not 1.0 / NaN over the host link)
    gives the same p / q, bit for bit, as the dense columns; a pass that overflows the value lists comes back dense."""
    import torch
    from blueberry_b200.distributed import GenomePass, HostStream, layout_rows
    dev = torch.device("cuda", 0)
    eng, shards = _random_shards(2, dev)
    shards = [s for s in shards if s.chr1 is None]
    gp = GenomePass(eng, group=False, q_values=True)
    gp.attach(shards)
    gp.run()
    p_ref, q_ref = gp.p.cpu().numpy().copy(), gp.q.cpu().numpy().copy()
    sizes, chroms = [s.n for s in shards], [s.chrom for s in shards]
    starts, rows = layout_rows(sizes)
    rows = max(rows, 4)
    h = [torch.zeros(rows, dtype=torch.int32).pin_memory() for _ in range(3)]
    for s, a in zip(shards, starts):
        h[0][a:a + s.n] = s.mid1.cpu(); h[1][a:a + s.n] = s.mid2.cpu(); h[2][a:a + s.n] = s.count.cpu()
    real = np.zeros(rows, bool)
    for s, a in zip(shards, starts):
        real[a:a + s.n] = True
    for caps in ((rows, rows), (8, 8)):
        gp2 = GenomePass(eng, group=False, q_values=True)
        pipe = HostStream(gp2, sizes, chroms, slots=2, packed=True, cap_p=caps[0], cap_q=caps[1])
        outs = [pipe.packed_buffers() for _ in range(3)]
        for o in outs:
            pipe.submit_packed(h[0], h[1], h[2], o)
        pipe.drain()
        for o in outs:
            assert o.overflow == (caps[0] == 8)
            p, q = o.dense()
            assert _same(p[real], p_ref[:rows][real]) and _same(q[real], q_ref[:rows][real])
            assert np.isnan(p[~real]).all()
        if caps[0] != 8:
            assert outs[0].nbytes() < 16 * rows + 4096


def test_host_stream_matches_serial_genome_passes():
    """distributed.HostStream: five different libraries (different sizes and seeds) streamed through two device slots
    give bit-for-bit the p and q of the same libraries run one at a time on the default stream."""
    import torch
    from blueberry_b200 import _lib
    from blueberry_b200.distributed import GenomePass, HostStream
    from blueberry_b200.engine import BiasTables, PassEngine, Shard
    lib = _lib.load()
    dev = torch.device("cuda:0")
    R, nb, K = 5000, 6000, 400
    P = int(lib.bbk_synth_n_pairs(nb, K))
    rng = np.random.default_rng(5)
    bias_host = np.exp(rng.normal(0.0, 0.25, size=nb))
    bias_dev = torch.from_numpy(bias_host).to(dev)
    eng = PassEngine(R, 100, 0, K * R, nb, dev)
    eng.set_fragments([nb], [(nb - 1) * R])
    eng.set_bias(BiasTables([np.where((bias_host < 0.5) | (bias_host > 2), -1.0, bias_host)], [R // 2], dev))
    libs, want = [], []
    for i in range(5):
        cols = [torch.empty(P, dtype=torch.int32, device=dev) for _ in range(3)]
        _lib.check(lib.bbk_synth_contacts(nb, K, R, 40.0 + 25 * i, 1.08, 100 + i, _lib.ptr(bias_dev), _lib.ptr(cols[0]),
                                          _lib.ptr(cols[1]), _lib.ptr(cols[2]), _lib.stream_ptr()), "synth")
        n = P - 1000 * i - (i & 1)                    # ragged sizes, odd and even
        cols = [c[:n].contiguous() for c in cols]
        gp = GenomePass(eng, group=False)
        gp.attach([Shard(*cols)])
        gp.run()
        fit = eng.read_fit()
        want.append((gp.shard_p(0).cpu(), gp.shard_q(0).cpu(), (fit.S, fit.n_knots, fit.smoothing, fit.y_min)))
        libs.append([c.cpu().pin_memory() for c in cols])
    torch.cuda.synchronize()
    pipe = HostStream(GenomePass(eng, group=False), [P], [0], slots=2)
    outs = []
    for cols in libs:
        n = cols[0].numel()
        h_p, h_q = torch.empty(n, dtype=torch.float64).pin_memory(), torch.empty(n, dtype=torch.float64).pin_memory()
        outs.append((h_p, h_q, pipe.submit(cols[0], cols[1], cols[2], h_p, h_q, sizes=[n])))
    outs[0][2].synchronize()                          # the event of the first library alone makes its outputs readable
    assert torch.equal(outs[0][0].view(torch.int64), want[0][0].view(torch.int64))
    pipe.drain()
    for (h_p, h_q, _), (p, q, _fit) in zip(outs, want):
        assert torch.equal(h_p.view(torch.int64), p.view(torch.int64))
        assert torch.equal(h_q.view(torch.int64), q.view(torch.int64))
    assert (want[0][0][:100000] != want[1][0][:100000]).any()
    # every pass leaves its own fit result (the engine's is overwritten by the next pass); the last `slots` are held
    for k in (3, 4):
        fit = pipe.fit_of(k)
        assert (fit.S, fit.n_knots, fit.smoothing, fit.y_min) == want[k][2]
        assert fit.y_min > 0 and PassEngine.reference_smoothing(fit) in (None, fit.y_min ** 2)
    with pytest.raises(KeyError):
        pipe.fit_of(0)
    # a library without a single contact: the reference divides by S == 0 (fithic.py:216); the stream reports it per pass
    zero = torch.zeros(libs[0][2].numel(), dtype=torch.int32).pin_memory()
    h_p = torch.empty(zero.numel(), dtype=torch.float64).pin_memory()
    pipe.submit(libs[0][0], libs[0][1], zero, h_p, sizes=[zero.numel()])           # without h_q: no q-value step
    assert pipe.gp.q_values
    with pytest.raises(ZeroDivisionError):
        pipe.fit_of(5)
    pipe.submit(libs[1][0], libs[1][1], libs[1][2], outs[1][0], outs[1][1], sizes=[libs[1][0].numel()])     # and the next pass is not affected
    assert pipe.fit_of(6).S == want[1][2][0]
    assert torch.equal(outs[1][0].view(torch.int64), want[1][0].view(torch.int64))
    with pytest.raises(ValueError):
        pipe.submit(libs[0][0], libs[0][1], libs[0][2], torch.empty(libs[0][0].numel(), dtype=torch.float64), sizes=[libs[0][0].numel()])


def test_host_stream_deferred_list_holds_every_row():
    """A slot of more than 2^20 rows, nearly all of them deferred by the streaming K4 (counts above 64 go to its patch pass).
    Nothing in the stream synchronises, so nothing would see a deferred-list overflow: the stream's list has a place for every
    row of a slot, and p and q equal those of GenomePass.run (which repeats a pass whose list overflowed) bit for bit."""
    import torch
    from blueberry_b200 import _lib
    from blueberry_b200.distributed import GenomePass, HostStream
    from blueberry_b200.engine import PassEngine, Shard
    lib = _lib.load()
    dev = torch.device("cuda:0")
    R, nb, K = 5000, 20050, 100
    n = int(lib.bbk_synth_n_pairs(nb, K))
    assert n > 1 << 20 and n % 4 == 0
    cols = [torch.empty(n, dtype=torch.int32, device=dev) for _ in range(3)]
    _lib.check(lib.bbk_synth_contacts(nb, K, R, 20000.0, 1.08, 3, None, _lib.ptr(cols[0]), _lib.ptr(cols[1]), _lib.ptr(cols[2]),
                                      _lib.stream_ptr()), "synth")
    eng = PassEngine(R, 100, 0, K * R, nb, dev)
    eng.set_fragments([nb], [(nb - 1) * R])
    gp = GenomePass(eng, group=False)
    gp.attach([Shard(*cols)])
    assert gp.listed
    fit = gp.run()
    assert gp.last_score.n_list > max(1 << 20, n // 4)            # more rows deferred than a default-size list holds
    want_p, want_q = gp.shard_p(0).cpu(), gp.shard_q(0).cpu()
    h = [c.cpu().pin_memory() for c in cols]
    h_p, h_q = (torch.empty(n, dtype=torch.float64).pin_memory() for _ in range(2))
    pipe = HostStream(GenomePass(eng, group=False), [n], [0], slots=2)
    pipe.submit(h[0], h[1], h[2], h_p, h_q)
    pipe.drain()
    assert (pipe.fit_of(0).S, pipe.fit_of(0).smoothing) == (fit.S, fit.smoothing)
    assert torch.equal(h_p.view(torch.int64), want_p.view(torch.int64))
    assert torch.equal(h_q.view(torch.int64), want_q.view(torch.int64))


def _torchrun(world, script, timeout=900):
    env = dict(os.environ)
    env["MASTER_ADDR"] = "127.0.0.1"
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(world), "--master-addr", "127.0.0.1",
           "--master-port", str(29600 + world), os.path.join(ROOT, "tests", script)]
    return subprocess.run(cmd, env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, timeout=timeout, cwd=ROOT)


@pytest.mark.parametrize("world", [2, 4, 8])
def test_multi_gpu_pass_against_single_process_oracle(world):
    import torch
    if torch.cuda.device_count() < world:
        pytest.skip("needs %d GPUs" % world)
    r = _torchrun(world, "multi_gpu_check.py")
    assert r.returncode == 0, r.stdout.decode(errors="replace")[-4000:]
