"""GPU tests of the two-pass workload in row blocks from host memory (distributed.BlockedPass(refit=True)): every case equals
the resident two-pass that fit_transform_arrays(refit=True) runs - GenomePass(q_values=False).run(), then
GenomePass.run(n_tests, exclude=(p_first, 1 / possibleIntraInRangeCount)) on the same engine - bit for bit: p_first, p and q
of every row, the tables after pass 2, bins, spline and spline_raw, and both passes' BbkFitResult without the SM cycle
counters; plus the config-4 shape against the oracle and fit_transform_arrays(refit=True) on the blocked path."""
import numpy as np
import pytest

from helpers import log10_close

pytestmark = pytest.mark.gpu


def _fit_cmp(raw):
    raw = bytes(raw)
    return raw[:72] + raw[184:]


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.uint64)


def _genome(bins, R=10000, max_dist=2_000_000, depth=150.0, seed=31, bias_on=(0,), loop_rate=1e-3):
    from blueberry_b200 import synth
    bias = synth.make_bias(bins, seed)
    for c in range(len(bins)):
        if c not in bias_on:
            bias[c] = np.ones(bins[c])
    c = synth.make_contacts(bins, R, max_dist, depth, seed, bias, loop_rate=loop_rate)
    shards = []
    for k in range(len(bins)):
        sel = c["chrom"] == k
        shards.append((k, c["mid1"][sel].copy(), c["mid2"][sel].copy(), c["count"][sel].copy()))
    return dict(bins=bins, R=R, max_dist=max_dist, bias=bias, shards=shards, contacts=c)


def _engine(g, dev, n_bins=100, max_bins=None):
    from blueberry_b200.engine import BiasTables, PassEngine
    bins, R = g["bins"], g["R"]
    eng = PassEngine(R, n_bins, 0, g["max_dist"], max(bins), dev, max_bins=max_bins)
    eng.set_fragments(bins, [(b - 1) * R for b in bins])
    tabs = [np.where((b < 0.5) | (b > 2), -1.0, b) for b in g["bias"]]
    eng.set_bias(BiasTables(tabs, [R // 2] * len(bins), dev))
    return eng


def _threshold(eng):
    from blueberry_b200.fithic import _in_range_possible
    return 1.0 / _in_range_possible(eng.possible.cpu().numpy(), eng.R, eng.min_dist, eng.max_dist)


def _tables(eng):
    return eng.obs_sum.cpu().numpy(), eng.totals.cpu().numpy()


def _state(eng, fit):
    obs, totals = _tables(eng)
    return dict(obs=obs, totals=totals, x=eng.x[:fit.n_out].cpu().numpy(), y=eng.y[:fit.n_out].cpu().numpy(),
                sy=eng.spline_y[:fit.L].cpu().numpy(), sr=eng.spline_raw[:fit.L].cpu().numpy(),
                fit=_fit_cmp(eng.fit_result.cpu().numpy().tobytes()))


def _resident(g, dev, q_values=True, n_tests=-1, force_exact=False, **ekw):
    """The resident two-pass of fit_transform_arrays(refit=True) over the genome's shards."""
    import torch
    from blueberry_b200.distributed import GenomePass
    from blueberry_b200.engine import Shard
    eng = _engine(g, dev, **ekw)
    shards = [Shard(*(torch.from_numpy(np.ascontiguousarray(a, dtype=np.int32)).to(dev) for a in sh[1:]), chrom=sh[0]) for sh in g["shards"]]
    gp1 = GenomePass(eng, group=False, q_values=False)
    gp1.force_exact = force_exact
    gp1.attach(shards)
    fit1 = gp1.run()
    table1 = _tables(eng)
    thr = _threshold(eng)
    gp2 = GenomePass(eng, group=False, q_values=q_values)
    gp2.force_exact = force_exact
    gp2.attach(shards)
    fit2 = gp2.run(n_tests, exclude=(gp1.p, thr))
    n = len(g["shards"])
    return dict(fit1=fit1, fit2=fit2, thr=thr, table1=table1, p1=[gp1.shard_p(i).cpu().numpy() for i in range(n)],
                p=[gp2.shard_p(i).cpu().numpy() for i in range(n)],
                q=[gp2.shard_q(i).cpu().numpy() for i in range(n)] if q_values else None, state=_state(eng, fit2))


def _blocked(g, dev, q_values=True, n_tests=-1, force_exact=False, block_rows=1 << 27, resident_bytes=None, cand_capacity=None,
             with_first=True, **ekw):
    from blueberry_b200.distributed import BlockedPass
    eng = _engine(g, dev, **ekw)
    bp = BlockedPass(eng, q_values=q_values, block_rows=block_rows, resident_bytes=resident_bytes, cand_capacity=cand_capacity,
                     refit=True)
    bp.force_exact = force_exact
    shards = g["shards"]
    p = [np.full(len(sh[1]), -7.0) for sh in shards]
    q = [np.full(len(sh[1]), -7.0) for sh in shards] if q_values else None
    p1 = [np.full(len(sh[1]), -7.0) for sh in shards] if with_first else None
    fit2 = bp.run(shards, p, q, n_tests=n_tests, p_first_out=p1)
    return dict(fit1=bp.fit_first, fit2=fit2, thr=bp.p_outlier, p1=p1, p=p, q=q, state=_state(eng, fit2), bp=bp)


def _assert_same(ref, got, q_values=True):
    assert ref["thr"] == got["thr"]
    st_r, st_b = ref["state"], got["state"]
    for k in st_r:
        if k == "fit":
            assert st_r[k] == st_b[k], "fit results differ"
        else:
            assert np.array_equal(_bits(st_r[k]) if st_r[k].dtype == np.float64 else st_r[k],
                                  _bits(st_b[k]) if st_b[k].dtype == np.float64 else st_b[k]), k
    assert _fit_cmp(bytes(ref["fit2"])) == _fit_cmp(bytes(got["fit2"])), "pass 2's FitResult"
    assert _fit_cmp(bytes(ref["fit1"])) == _fit_cmp(bytes(got["fit1"])), "pass 1's FitResult"
    for i in range(len(ref["p"])):
        if got["p1"] is not None:
            assert np.array_equal(_bits(ref["p1"][i]), _bits(got["p1"][i])), "p_first of shard %d" % i
        assert np.array_equal(_bits(ref["p"][i]), _bits(got["p"][i])), "p of shard %d" % i
        if q_values:
            assert np.array_equal(_bits(ref["q"][i]), _bits(got["q"][i])), "q of shard %d" % i


def _outlier_blocks(ref, bp):
    """Blocks of bp's plan that hold at least one pass-1 outlier."""
    return [k for k, blk in enumerate(bp.blocks) if any((ref["p1"][s][lo:lo + n] <= ref["thr"]).any() for (s, lo, n, _) in blk)]


@pytest.fixture(scope="module")
def dev():
    import torch
    return torch.device("cuda", 0)


@pytest.fixture(scope="module")
def g3():
    return _genome([420, 300, 180], bias_on=(0, 2))


@pytest.fixture(scope="module")
def ref3(g3, dev):
    return _resident(g3, dev)


@pytest.mark.parametrize("block_rows", [1 << 27, 4096, 3 * 4096, 12_345, 5_003])
def test_block_sizes(g3, ref3, dev, block_rows):
    got = _blocked(g3, dev, block_rows=block_rows)
    _assert_same(ref3, got)
    bp = got["bp"]
    nb = len(bp.blocks)
    assert nb == 1 if block_rows == 1 << 27 else nb > 1
    assert sum(int((p <= ref3["thr"]).sum()) for p in ref3["p1"]) > 0
    if nb > 1:
        assert len(_outlier_blocks(ref3, bp)) > 1
    if block_rows in (12_345, 5_003):     # chromosomes cut inside, at rows that are not multiples of 4
        assert any(lo % 4 for b in bp.blocks for (_, lo, _, _) in b)


@pytest.mark.parametrize("budget", ["all", "none", "half"])
def test_residency_budgets(g3, ref3, dev, budget):
    total = sum(len(sh[1]) for sh in g3["shards"]) * 12
    rb = {"all": None, "none": 0, "half": total // 2}[budget]
    got = _blocked(g3, dev, block_rows=8 * 4096, resident_bytes=rb)
    _assert_same(ref3, got)
    res = got["bp"].resident
    assert all(res) if budget == "all" else (not any(res) if budget == "none" else (any(res) and not all(res)))


def test_without_q_values(g3, dev):
    ref = _resident(g3, dev, q_values=False)
    _assert_same(ref, _blocked(g3, dev, q_values=False, block_rows=5 * 4096, resident_bytes=0), q_values=False)


@pytest.mark.parametrize("n_tests", [25, 40_000])
def test_n_tests(g3, dev, n_tests):
    ref = _resident(g3, dev, n_tests=n_tests)
    _assert_same(ref, _blocked(g3, dev, n_tests=n_tests, block_rows=9 * 4096, resident_bytes=50_000))


@pytest.mark.parametrize("budget", [None, 0])
def test_without_p_first_out(g3, ref3, dev, budget):
    got = _blocked(g3, dev, block_rows=6 * 4096, resident_bytes=budget, with_first=False)
    _assert_same(ref3, got)


def test_genome_without_outliers(dev):
    """No pass-1 outlier: table 2 equals table 1 (and everything equals the resident two-pass)."""
    for seed in range(40, 46):             # the first seed whose pass 1 has no outlier (fixed: the genomes are seeded)
        g = _genome([260, 140], depth=0.5, seed=seed, bias_on=(), loop_rate=0.0)
        ref = _resident(g, dev)
        if not any((p <= ref["thr"]).any() for p in ref["p1"]):
            break
    else:
        pytest.fail("every candidate genome has a pass-1 outlier")
    for k, t in enumerate(ref["table1"]):
        assert np.array_equal(t, (ref["state"]["obs"], ref["state"]["totals"])[k])
    got = _blocked(g, dev, block_rows=4096, resident_bytes=0)
    _assert_same(ref, got)


def test_candidate_lists_overflow(g3, ref3, dev):
    got = _blocked(g3, dev, block_rows=6 * 4096, cand_capacity=16)
    assert any(s.cand_overflow for s in got["bp"].last_states)
    _assert_same(ref3, got)


def test_exact_mode(g3, dev):
    ref = _resident(g3, dev, force_exact=True)
    _assert_same(ref, _blocked(g3, dev, force_exact=True, block_rows=7 * 4096, resident_bytes=0))


def test_pass_one_wants_more_bins(g3, dev):
    ref = _resident(g3, dev, max_bins=4)
    got = _blocked(g3, dev, max_bins=4, block_rows=7 * 4096)
    assert ref["fit1"].n_out > 4
    _assert_same(ref, got)


@pytest.mark.parametrize("which", [0, 1])
def test_fit_settled_on_reference_s(g3, dev, monkeypatch, which):
    """A reference s that differs from the kernel's once, in pass 1 only (which = 0) or in pass 2 only (which = 1); the
    passes are told apart by their S (pass 2's table leaves the outliers out)."""
    from blueberry_b200.engine import PassEngine

    def patch():
        seen, given = [], set()

        def ref_s(fit):
            if fit.n_out <= 0:
                return None
            if int(fit.S) not in seen:
                seen.append(int(fit.S))
            if seen.index(int(fit.S)) != which or fit.smoothing in given:
                return None
            s = fit.smoothing * 1.25
            given.add(s)
            return s
        monkeypatch.setattr(PassEngine, "reference_smoothing", staticmethod(ref_s))
        return given

    given = patch()
    ref = _resident(g3, dev)
    assert (ref["fit1"], ref["fit2"])[which].smoothing in given
    assert (ref["fit1"], ref["fit2"])[1 - which].smoothing not in given
    patch()
    _assert_same(ref, _blocked(g3, dev, block_rows=7 * 4096, resident_bytes=0))


def test_all_zero_counts_raise_and_leave_outputs(dev):
    g = _genome([200, 150], bias_on=())
    g["shards"] = [(c, m1, m2, np.zeros_like(cn)) for c, m1, m2, cn in g["shards"]]
    with pytest.raises(ZeroDivisionError):
        _resident(g, dev)
    from blueberry_b200.distributed import BlockedPass
    bp = BlockedPass(_engine(g, dev), block_rows=4096, refit=True)
    p, q, p1 = ([np.full(len(sh[1]), -7.0) for sh in g["shards"]] for _ in range(3))
    with pytest.raises(ZeroDivisionError):
        bp.run(g["shards"], p, q, p_first_out=p1)
    assert all((x == -7.0).all() for x in p + q + p1)
    assert bp.fit_first is None


def test_fragments_without_an_in_range_pair(dev):
    from blueberry_b200.distributed import BlockedPass
    from blueberry_b200.engine import PassEngine
    lone = PassEngine(10000, 100, 0, 100_000, 1, dev)
    lone.set_fragments([1, 1], [0, 0])
    with pytest.raises(ZeroDivisionError):
        BlockedPass(lone, refit=True)


def test_config4_shape_against_resident_and_oracle(dev):
    """BASELINE config 4's shape (1 kb, 2 Mb cap, ~93 % zero counts, a 4000-bin chromosome = 6.0e6 records) in blocks of 2^20
    rows, some of them resident: equal to the resident two-pass, and to the oracle's two passes under the bars of the
    resident pass' oracle test."""
    import warnings
    from blueberry_b200 import synth
    from oracle import fithic_oracle as fo
    g = _genome([4000], R=1000, max_dist=2_000_000, depth=60.0, seed=404, bias_on=(0,))
    c = g["contacts"]
    assert 0.85 < float((c["count"] == 0).mean()) < 0.97
    ref = _resident(g, dev)
    got = _blocked(g, dev, block_rows=1 << 20, resident_bytes=30 << 20)
    bp = got["bp"]
    assert len(bp.blocks) == 6 and any(bp.resident) and not all(bp.resident)
    _assert_same(ref, got)
    assert len(_outlier_blocks(ref, bp)) > 1

    R, bins = g["R"], g["bins"]
    fc, fm = synth.make_fragments(bins, R)
    bd, _ = fo.read_bias_arrays(np.zeros(bins[0], dtype=np.int64), fm, g["bias"][0])
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        r1, r2, outlier, thr = fo.fithic_two_pass_arrays(fc, fm, c["chrom"], c["mid1"], c["chrom"], c["mid2"], c["count"], R, 100,
                                                         0, g["max_dist"], bias=bd)
    assert int(outlier.sum()) > 0 and thr == got["thr"]
    st = got["state"]
    p1, p, q = got["p1"][0], got["p"][0], got["q"][0]
    assert np.array_equal(p1 <= 1, r1.keep)
    assert int((p1 <= thr).sum()) == int(outlier.sum())
    assert np.array_equal(st["obs"], r2.contacts.observed)
    assert int(st["totals"][0]) == r2.contacts.S
    assert np.array_equal(st["x"], np.array(r2.x)) and np.array_equal(st["y"], np.array(r2.y))
    assert np.array_equal(st["sy"], r2.spline_y)
    keep = p <= 1
    assert np.array_equal(keep, r2.keep)
    sel = r2.keep & (r2.p >= 1e-300)
    ok, nbad = log10_close(p[sel], r2.p[sel], 1e-5)
    assert ok, "%d p-values differ by more than 1e-5 in log10" % nbad
    assert np.array_equal(q[keep], fo.benjamini_hochberg_correction(p[keep], int(keep.sum())))


def _close(a, b, rel):
    """Same NaN pattern, the same rows at exactly 0.0, everything else within `rel` (relative)."""
    if not np.array_equal(np.isnan(a), np.isnan(b)):
        return False
    ok = ~np.isnan(a)
    a, b = a[ok], b[ok]
    if not np.array_equal(a == 0.0, b == 0.0):
        return False
    pos = (a > 0) & (b > 0)
    return bool((np.abs(a[pos] / b[pos] - 1.0) <= rel).all())


def _dropin(monkeypatch, bins, seed):
    """fit_transform_arrays(refit=True) on a synthetic genome, resident and routed to the blocked path."""
    from blueberry_b200 import fithic, synth
    R, max_dist = 10000, 1_500_000
    bias = synth.make_bias(bins, seed)
    fc, fm = synth.make_fragments(bins, R)
    c = synth.make_contacts(bins, R, max_dist, 120.0, seed + 10, bias)
    bc = np.concatenate([np.full(b, i, dtype=np.int32) for i, b in enumerate(bins)])
    model = fithic.FitHiC("blocked", R, n_bins=100, max_dist=max_dist, min_dist=0)

    def call(blocked, **kw):
        seen = []

        def route(rows, want_q, d, refit=False):
            seen.append(refit)
            return blocked and refit
        monkeypatch.setattr(fithic, "use_blocked_pass", route)
        out = model.fit_transform_arrays(c["chrom"], c["mid1"], c["chrom"], c["mid2"], c["count"], fc, fm,
                                         bias=(bc, fm, np.concatenate(bias)), refit=True, **kw)
        assert seen == [True]
        return out
    return call


def test_fit_transform_arrays_refit_on_the_blocked_path(dev, monkeypatch):
    """One chromosome: the resident two-pass scores with the streaming K4 as the blocked one does, so every PassOutput field
    but gpu_launches is the same, p_first included."""
    call = _dropin(monkeypatch, [700], 1)
    for kw in (dict(q_values=True), dict(q_values=False), dict(q_values=True, n_tests=25)):
        a, b = call(False, **kw), call(True, **kw)
        assert a.p_first is not None and b.p_first is not None
        for f in type(a).__slots__:
            if f == "gpu_launches":
                continue
            va, vb = getattr(a, f, None), getattr(b, f, None)
            if f == "fit":
                assert _fit_cmp(bytes(va)) == _fit_cmp(bytes(vb))
            elif isinstance(va, np.ndarray):
                assert va.dtype == vb.dtype and np.array_equal(va.view(np.uint8), vb.view(np.uint8)), f
            elif f == "frag":
                assert type(va) is type(vb)
            else:
                assert va == vb, f


def test_fit_transform_arrays_refit_on_the_blocked_path_several_chromosomes(dev, monkeypatch):
    """Several chromosomes: the resident two-pass of the drop-in call holds them in one shard with chromosome columns and scores
    with the general kernel, which agrees with the streaming K4 to rounding, not to the bit (test_split_k4_matches_the_direct_kernel).
    The tables, bins, spline and fits are the same; p_first, p and q agree within that test's bounds."""
    call = _dropin(monkeypatch, [300, 200, 120], 1)
    a, b = call(False, q_values=True), call(True, q_values=True)
    assert _fit_cmp(bytes(a.fit)) == _fit_cmp(bytes(b.fit))
    for f in ("x", "y", "spline_y", "spline_y_raw", "observed", "possible", "bin_of_key", "keep"):
        assert np.array_equal(getattr(a, f), getattr(b, f)), f
    assert a.totals == b.totals
    assert _close(a.p_first, b.p_first, 1e-9) and _close(a.p, b.p, 1e-9) and _close(a.q, b.q, 1e-8)
