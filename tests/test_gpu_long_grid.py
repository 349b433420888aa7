"""The fit kernel (K2/K3, csrc/fit_stage.cu) and the histogram (K1, csrc/hist.cu) on the long distance tables of the
reference's default call on a human chromosome (49,851 keys for chr1 at 5 kb), against the CPU oracle:

  a. bbk_fit on synthetic tables, every output bit for bit against calculate_probabilities / UnivariateSpline /
     IsotonicRegression.  The fit runs each phase in a 200 KB shared pool when it fits and from the global workspace
     otherwise; the pool-or-global decisions are restated here (and checked against bbk_fit_workspace_bytes), and every case
     asserts which phases it runs from global memory, so that the global branches cannot go untested unnoticed;
  b. bbk_fit_batched mixing pool and global problems (and one bad problem) against one bbk_fit per problem;
  c. K1 at table sizes on both sides of the 40,960 keys it keeps in shared memory, and a run long enough that every CTA
     flushes its shared table;
  d. the whole pass on 49,851 bins (direct and streaming K4, per chromosome, refit) against fithic_arrays.

Bars (DESIGN "Parity contract"): integers, bins, bin_of_key, x, y, knots, coefficients, spline_raw and spline_y bit for bit;
the residual within 1e-12 relative; p within 1e-5 in log10; q bit for bit on the device's own p.
"""
import warnings

import numpy as np
import pytest

from helpers import log10_close
from test_long_grid_host import synthetic_table

pytestmark = pytest.mark.gpu

R = 5000

# ------------------------------------------------------------------------------------------------ the fit's memory plan
POOL_DOUBLES = 200 * 1024 // 8                                 # fit_pool_bytes()


def need_binning(nk_eff, max_bins):                             # 3 int64 tables + 2 int32 bound arrays
    return 3 * nk_eff + max_bins + 2


def coop_ws_doubles(m):                                         # bbk_coop_ws_doubles (fit_coop.h)
    nest = m + 4
    spline = nest * 4 + nest * 4 + nest * 5 + nest * 5 + m * 4 + (nest + 1) // 2 + 8
    return spline + nest * 5 + nest + m + 3 * ((m + 1) // 2 + 1) + 8


def need_spline(m):
    return coop_ws_doubles(m) + 2 * m


def need_eval(m, L):                                            # knots, coefficients, residual terms, 3 grids + flags
    return 3 * (m + 4) + 4 * L + 8


def workspace_bytes(max_bins, nkeys):
    m = max(max_bins, 4)
    return (max(need_binning(nkeys, m), need_spline(m), need_eval(m, nkeys)) + 16) * 8


def global_phases(nk_eff, max_bins, m, L):
    g = set()
    if need_binning(nk_eff, max_bins) > POOL_DOUBLES:
        g.add("binning")
    if m >= 4 and need_spline(m) > POOL_DOUBLES:
        g.add("spline")
    if L > 0 and need_eval(m, L) > POOL_DOUBLES:
        g.add("eval")
    return g


def test_memory_plan_restatement():
    from blueberry_b200 import _lib
    lib = _lib.load()
    assert need_binning(8362, 512) <= POOL_DOUBLES < need_binning(8363, 512)
    assert need_spline(772) <= POOL_DOUBLES < need_spline(773)
    assert need_eval(100, 6320) <= POOL_DOUBLES < need_eval(100, 6321)
    for max_bins in (4, 5, 100, 255, 256, 257, 512, 771, 772, 773, 1000, 4000, 8362, 49851):
        for nkeys in (1, 7, 2001, 6320, 8362, 8363, 25000, 40960, 49851, 100000):
            assert int(lib.bbk_fit_workspace_bytes(max_bins, nkeys)) == workspace_bytes(max_bins, nkeys), (max_bins, nkeys)


# ------------------------------------------------------------------------------------------------ a. bbk_fit
def _oracle_fit(possible, observed, S, n_bins, min_dist, max_dist, s=None):
    """calculate_probabilities and fit_spline_tables (fithic.py:160-227, :340-374) with s = min(y)**2 or the given s."""
    from scipy.interpolate import UnivariateSpline
    from sklearn.isotonic import IsotonicRegression
    from oracle import fithic_oracle as fo
    x, y, _, bok = fo.calculate_probabilities(possible, observed, S, n_bins, R, min_dist, max_dist)
    out = dict(x=np.array(x), y=np.array(y), bin_of_key=bok, m=len(x))
    if len(x) < 4:
        return out
    s = min(y) ** 2 if s is None else s
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        ius = UnivariateSpline(x, y, s=s)
    keys = [k * R for k in range(len(possible))]
    spline_x = [i for i in keys if min(x) <= i <= max(x)]
    raw = ius(spline_x)
    new_y = IsotonicRegression(increasing=False).fit_transform(spline_x, raw)
    d = ius._data
    out.update(s=s, k0=spline_x[0] // R, L=len(spline_x), spline_raw=np.asarray(raw), spline_y=np.asarray(new_y),
               residual=sum([i * i for i in (y - ius(x))]), n_knots=d[7], knots=d[8][:d[7]], coefs=d[9][:d[7]], ier=d[13])
    return out


def _engine(possible, observed, S, n_bins, min_dist, max_dist, sizes, max_bins=None):
    import torch
    from blueberry_b200.engine import PassEngine
    dev = torch.device("cuda", 0)
    eng = PassEngine(R, n_bins, min_dist, max_dist, len(possible), dev, max_bins=max_bins)
    eng.set_fragments(sizes, [(nf - 1) * R for nf in sizes])
    eng.obs_sum.copy_(torch.from_numpy(observed))
    eng.totals.zero_()
    eng.totals[0] = S
    torch.cuda.synchronize()
    assert np.array_equal(eng.possible.cpu().numpy(), possible)
    return eng


def _read(eng):
    import torch
    from blueberry_b200 import _lib
    torch.cuda.synchronize()
    return _lib.FitResult.from_buffer_copy(eng.fit_result.cpu().numpy().tobytes())


def _device_fit(eng, s=None):
    """bbk_fit as the product runs it: min(y)**2 as the reference computes it (libm pow) when it differs from the kernel's
    ymin * ymin, or the given s."""
    from blueberry_b200.engine import PassEngine
    eng.fit(smoothing=s)
    fr = _read(eng)
    if s is None and fr.status == 0:
        s_ref = PassEngine.reference_smoothing(fr)
        if s_ref is not None:
            eng.fit(smoothing=s_ref)
            fr = _read(eng)
    return fr


def _check_fit(eng, fr, ref, nk_eff):
    assert fr.status == 0 and fr.n_out == ref["m"]
    m, L = fr.n_out, fr.L
    assert np.array_equal(eng.x[:m].cpu().numpy(), ref["x"]) and np.array_equal(eng.y[:m].cpu().numpy(), ref["y"])
    assert np.array_equal(eng.bin_of_key.cpu().numpy(), ref["bin_of_key"])
    assert fr.smoothing == ref["s"] and fr.ier == ref["ier"]
    assert fr.n_knots == ref["n_knots"]
    assert np.array_equal(eng.knots[:fr.n_knots].cpu().numpy(), ref["knots"])
    assert np.array_equal(eng.coefs[:fr.n_knots].cpu().numpy(), ref["coefs"])        # with scipy's zeros in the last four
    assert (fr.k0, L) == (ref["k0"], ref["L"])
    raw, sy = eng.spline_raw.cpu().numpy(), eng.spline_y.cpu().numpy()
    assert np.array_equal(raw[:L], ref["spline_raw"])
    assert np.array_equal(sy[:L], ref["spline_y"])
    assert not raw[L:].any() and not sy[L:].any()
    assert abs(fr.residual - ref["residual"]) <= 1e-12 * abs(ref["residual"])
    g = global_phases(nk_eff, eng.max_bins, m, L)
    print("m=%d nk_eff=%d L=%d max_bins=%d global: %s" % (m, nk_eff, L, eng.max_bins, ",".join(sorted(g)) or "none"))
    return g


def _nk_eff(nkeys, max_dist):
    return nkeys if max_dist < 0 else min(nkeys, max_dist // R + 1)


def _fit_case(nkeys, seed, n_bins, min_dist=-1, max_dist=-1, chroms=1, s_factor=None):
    possible, observed, _ = synthetic_table(nkeys, seed, chroms=chroms)
    k = np.arange(nkeys)
    rng_ = (k * R > min_dist) if min_dist > -1 else np.ones(nkeys, bool)
    if max_dist > -1:
        rng_ &= k * R <= max_dist
    observed = np.where(rng_, observed, 0)                      # K1 counts in-range distances only
    S = int(observed.sum()) + 77                                # and S also counts in-range records off the grid
    sizes = [nkeys] + [int(nkeys * f) for f in np.random.default_rng(seed).uniform(0.2, 0.8, chroms - 1)]
    eng = _engine(possible, observed, S, n_bins, min_dist, max_dist, sizes)
    s = None
    if s_factor is not None:
        s = min(_oracle_fit(possible, observed, S, n_bins, min_dist, max_dist)["y"]) ** 2 * s_factor
    ref = _oracle_fit(possible, observed, S, n_bins, min_dist, max_dist, s)
    fr = _device_fit(eng, s)
    return _check_fit(eng, fr, ref, _nk_eff(nkeys, max_dist)), eng, fr


def test_fit_binning_pool_boundary():
    """nk_eff 8,362 is the last table whose binning fits the pool at max_bins 512; 8,363 runs it from global memory."""
    g1, e1, _ = _fit_case(8362, 1, 100)
    g2, e2, _ = _fit_case(8363, 2, 100, chroms=2)
    assert e1.max_bins == e2.max_bins == 512
    assert "binning" not in g1 and "binning" in g2


def test_fit_evaluation_pool_boundary():
    """Grids on both sides of the last L whose evaluation and antitonic regression fit the pool (6,320 at m = 100)."""
    seen = set()
    for nk_eff in (6900, 6950, 7000, 7050, 7100):
        g, _, fr = _fit_case(20000, 5, 100, max_dist=(nk_eff - 1) * R + 3)
        seen.add("eval" in g)
    assert seen == {True, False}


@pytest.mark.parametrize("n_bins", [256, 257, 258, 300])
def test_fit_more_bins_than_threads(n_bins):
    """m = 255, 256, 257 and 299 bins against the fit's 256 threads."""
    g, _, fr = _fit_case(3000, 0, n_bins, chroms=2)
    assert fr.n_out == n_bins - 1 and not g


@pytest.mark.parametrize("n_bins", [800, 900, 1000])
def test_fit_spline_from_global_memory(n_bins):
    g, _, fr = _fit_case(20000, 7 + n_bins, n_bins, chroms=2)
    assert fr.n_out > 772 and "spline" in g


@pytest.mark.parametrize("n_bins", [100, 1000])
def test_fit_full_chromosome_table(n_bins):
    g, _, fr = _fit_case(49851, 11, n_bins, chroms=3)
    assert {"binning", "eval"} <= g
    assert ("spline" in g) == (n_bins == 1000)


@pytest.mark.parametrize("nk_eff", [8362, 8363])
def test_fit_table_cut_by_max_dist(nk_eff):
    g, eng, fr = _fit_case(49851, 13, 100, max_dist=(nk_eff - 1) * R + 3)
    assert ("binning" in g) == (nk_eff == 8363)
    bok = eng.bin_of_key.cpu().numpy()
    assert (bok[nk_eff:] == -1).all()


def test_fit_with_min_dist():
    g, eng, fr = _fit_case(20000, 17, 300, min_dist=40 * R + 3, chroms=2)
    bok = eng.bin_of_key.cpu().numpy()
    assert (bok[:41] == -1).all() and bok[41] == 0
    assert "binning" in g


def test_fit_given_smoothing_on_the_full_table():
    g, _, fr = _fit_case(49851, 19, 100, chroms=1, s_factor=1.7)
    assert {"binning", "eval"} <= g


def test_fit_every_key_a_bin_then_more_bins():
    """desired == 0 from the start: every key closes a bin.  The default max_bins is too small (-13); after grow_bins()
    the fit of several thousand bins (zero y: the interpolating spline) runs from global memory."""
    nkeys = 8000
    possible, _, _ = synthetic_table(nkeys, 23)
    observed = np.zeros(nkeys, np.int64)
    observed[[3, 50, 2000]] = [20, 9, 4]
    S = 33
    eng = _engine(possible, observed, S, 100, -1, -1, [nkeys])
    fr = _device_fit(eng)
    assert fr.status == -13
    assert eng.grow_bins()
    ref = _oracle_fit(possible, observed, S, 100, -1, -1)
    fr = _device_fit(eng)
    g = _check_fit(eng, fr, ref, nkeys)
    assert fr.n_out > 5000 and g == {"binning", "spline", "eval"}


def test_fit_failures_in_the_global_regime():
    from oracle import fithic_oracle as fo
    nkeys = 49851
    possible, observed, S = synthetic_table(nkeys, 29)
    eng = _engine(possible, np.zeros(nkeys, np.int64), 0, 100, -1, -1, [nkeys])
    assert _device_fit(eng).status == -14                       # S == 0
    with pytest.raises(ZeroDivisionError):
        fo.calculate_probabilities(possible, np.zeros(nkeys, np.int64), 0, 100, R, -1, -1)
    ref_bins = fo.calculate_probabilities(possible, observed, S, 100, R, -1, -1)[3]
    zero = np.flatnonzero(ref_bins == 40)                       # a whole bin without possible pairs
    possible = possible.copy()
    possible[zero] = 0
    with pytest.raises(ZeroDivisionError):
        fo.calculate_probabilities(possible, observed, S, 100, R, -1, -1)
    import torch
    from blueberry_b200.engine import PassEngine
    eng = PassEngine(R, 100, -1, -1, nkeys, torch.device("cuda", 0))
    eng.possible.copy_(torch.from_numpy(possible))
    eng.obs_sum.copy_(torch.from_numpy(observed))
    eng.totals.zero_()
    eng.totals[0] = S
    assert _device_fit(eng).status == -11
    assert "binning" in global_phases(nkeys, eng.max_bins, 0, 0)


# ------------------------------------------------------------------------------------------------ b. bbk_fit_batched
def _fit_fields(fr):
    """Every field of a fit result but the SM cycle counters."""
    return tuple(getattr(fr, f) for f, _ in fr._fields_ if f not in ("phase_cycles", "spline_diag"))


def _outputs(e):
    import torch
    torch.cuda.synchronize()
    return [t.cpu().numpy().tobytes() for t in (e.x, e.y, e.bin_of_key, e.spline_y, e.spline_raw, e.knots, e.coefs)]


def test_batched_fit_mixing_pool_and_global_problems():
    import torch
    from blueberry_b200 import _lib
    lib = _lib.load()
    dev = torch.device("cuda", 0)
    n_bins = 100
    problems = []                                               # (nkeys, seed, chroms, s_factor)
    for nkeys, seed, chroms, sf in [(3000, 31, 1, None), (8362, 1, 1, None), (8363, 2, 2, None), (20000, 37, 2, None),
                                    (49851, 11, 3, None), (49851, 19, 1, 1.7), (6000, 41, 1, None)]:
        possible, observed, S = synthetic_table(nkeys, seed, chroms=chroms)
        S += 77
        sizes = [nkeys] + [int(nkeys * f) for f in np.random.default_rng(seed).uniform(0.2, 0.8, chroms - 1)]
        a = _engine(possible, observed, S, n_bins, -1, -1, sizes)
        b = _engine(possible, observed, S, n_bins, -1, -1, sizes)
        s = None
        if sf is not None:
            a.fit()
            s = _read(a).smoothing * sf
        fa = _device_fit(a, s)
        ref = _oracle_fit(possible, observed, S, n_bins, -1, -1, s if s is not None else (fa.smoothing if fa.status == 0 else None))
        _check_fit(a, fa, ref, nkeys)
        if s is not None:
            req = _lib.FitResult()
            req.status, req.smoothing = _lib.FIT_S_GIVEN, s
            b.fit_result.copy_(torch.frombuffer(bytearray(bytes(req)), dtype=torch.uint8))
        elif fa.smoothing != fa.y_min * fa.y_min:               # the reference's s, given as the product gives it
            req = _lib.FitResult()
            req.status, req.smoothing = _lib.FIT_S_GIVEN, fa.smoothing
            b.fit_result.copy_(torch.frombuffer(bytearray(bytes(req)), dtype=torch.uint8))
        problems.append((a, b, fa))
    bad = _engine(*synthetic_table(6000, 43)[:2], 1000, n_bins, -1, -1, [6000])
    probs = (_lib.FitProblem * (len(problems) + 1))()
    for pr, e in zip(probs, [b for _, b, _ in problems] + [bad]):
        pr.d_possible, pr.d_obs_sum, pr.d_totals = e.possible.data_ptr(), e.obs_sum.data_ptr(), e.totals.data_ptr()
        pr.d_result, pr.d_x, pr.d_y, pr.d_bin_of_key = e.fit_result.data_ptr(), e.x.data_ptr(), e.y.data_ptr(), e.bin_of_key.data_ptr()
        pr.d_spline_y, pr.d_spline_raw, pr.d_knots, pr.d_coefs = (e.spline_y.data_ptr(), e.spline_raw.data_ptr(), e.knots.data_ptr(),
                                                                  e.coefs.data_ptr())
        pr.d_workspace, pr.workspace_bytes = e.fit_ws.data_ptr(), e.fit_ws.numel()
        pr.nkeys, pr.max_bins = e.nkeys, e.max_bins
    probs[len(problems)].workspace_bytes = workspace_bytes(bad.max_bins, bad.nkeys) - 1
    d_probs = torch.frombuffer(bytearray(bytes(probs)), dtype=torch.uint8).to(dev)
    bad_before = _outputs(bad)
    _lib.check(lib.bbk_fit_batched(_lib.ptr(d_probs), len(probs), n_bins, R, -1, -1, _lib.stream_ptr()), "bbk_fit_batched")
    regimes = set()
    for i, (a, b, fa) in enumerate(problems):
        fb = _read(b)
        assert _fit_fields(fb) == _fit_fields(fa), "problem %d" % i
        assert _outputs(b) == _outputs(a), "problem %d" % i
        regimes.add(frozenset(global_phases(a.nkeys, a.max_bins, fa.n_out, fa.L)))
    assert frozenset() in regimes and frozenset({"binning", "eval"}) in regimes and len(regimes) >= 3
    fbad = _read(bad)
    assert fbad.status == -17 and fbad.n_out == 0 and fbad.residual == 0.0
    assert _outputs(bad) == bad_before


# ------------------------------------------------------------------------------------------------ c. K1 across MAX_SMEM_KEYS
MAX_SMEM_KEYS = 40960


def _hist_records(nkeys, seed):
    rng = np.random.default_rng(seed)
    n = 3 * 4096 * 50 + 1234                                    # a partial last tile
    keys = rng.integers(0, nkeys + 40, n)                       # and a few distances past the table
    edge = rng.choice(n, n // 5, replace=False)
    keys[edge] = np.clip(MAX_SMEM_KEYS + rng.integers(-6, 6, len(edge)), 0, nkeys + 39)
    mid1 = rng.integers(0, 10 ** 8, n).astype(np.int64) * 2 + 1
    mid2 = mid1 + keys * R
    k = rng.choice(n, n // 40, replace=False)
    mid2[k] += rng.integers(1, R, len(k))                       # off the grid
    k = rng.choice(n, n // 60, replace=False)
    mid1[k], mid2[k] = mid2[k].copy(), mid1[k].copy()           # negative distances
    count = rng.poisson(1.5, n).astype(np.int64)
    count[rng.choice(n, n // 20, replace=False)] = 0
    k = rng.choice(n, n // 30, replace=False)
    count[k] = rng.choice([4095, 4096, 2 ** 31 - 1], len(k))
    for i in range(21):                                         # the big counts on the keys around the shared table's end
        mid2[i] = mid1[i] + (MAX_SMEM_KEYS - 3 + i % 7) * R
        count[i] = (4095, 4096, 2 ** 31 - 1)[i // 7]
    assert (mid2 < 2 ** 31).all()
    chr1 = rng.integers(0, 3, n).astype(np.int32)
    chr2 = np.where(rng.random(n) < 0.9, chr1, (chr1 + 1) % 3).astype(np.int32)
    return mid1, mid2, count, chr1, chr2


@pytest.mark.parametrize("nkeys", [25600, 40959, 40960, 40961, 49851, 100000])
@pytest.mark.parametrize("variant", ["general", "fast", "chrom"])
def test_hist_across_the_shared_table_size(nkeys, variant):
    import torch
    from blueberry_b200.engine import PassEngine, Shard
    from oracle import fithic_oracle as fo
    mid1, mid2, count, chr1, chr2 = _hist_records(nkeys, nkeys + len(variant))
    span = (nkeys - 1) * R
    min_dist, max_dist = {"general": (-1, -1), "fast": (0, span), "chrom": (R, span)}[variant]
    if variant != "chrom":
        chr1 = chr2 = None
    dev = torch.device("cuda", 0)
    to = lambda a: None if a is None else torch.from_numpy(np.ascontiguousarray(a, dtype=np.int32)).to(dev)
    sh = Shard(to(mid1), to(mid2), to(count), to(chr1), to(chr2))
    eng = PassEngine(R, 100, min_dist, max_dist, nkeys, device=dev)
    for excl in (False, True):
        keep = np.ones(len(count), bool)
        if excl:
            p = np.random.default_rng(nkeys).random(len(count))
            p[::9] = 0.25
            keep = ~(p <= 0.25)
            eng.hist_excluding([sh], [torch.from_numpy(p).to(dev)], 0.25)
        else:
            eng.hist([sh])
        ref = fo.read_interactions(nkeys, R, None if chr1 is None else chr1[keep], mid1[keep], None if chr2 is None else chr2[keep],
                                   mid2[keep], count[keep], min_dist, max_dist)
        torch.cuda.synchronize()
        obs = eng.obs_sum.cpu().numpy()
        assert np.array_equal(obs, ref.observed), (excl, np.flatnonzero(obs != ref.observed)[:10])
        assert [int(v) for v in eng.totals.cpu().numpy()] == [ref.S, ref.intra_in_range_count, ref.intra_all_sum, ref.intra_all_count,
                                                             ref.inter_all_sum, ref.inter_all_count, ref.min_obs_dist, ref.max_obs_dist]
        if not excl:
            assert (ref.observed[MAX_SMEM_KEYS - 3:min(MAX_SMEM_KEYS + 4, nkeys)] > 2 ** 31).all()


def test_hist_flushes_the_shared_table_in_every_cta():
    """More than 2^20 records per CTA, most of them count 4095 on one key below 40,960: without the flush at FLUSH_PAIRS a
    u32 shared bin would overflow.  The reference table is an int64 index_add_ on the device."""
    import torch
    from blueberry_b200.engine import PassEngine, Shard
    dev = torch.device("cuda", 0)
    nkeys = 49851
    sms = torch.cuda.get_device_properties(dev).multi_processor_count
    # at this table size K1 runs one CTA per SM: 2^21 records per CTA, two flushes each
    n = 2 * sms * (1 << 20) + 1234 * 3 + 1
    heavy_key = 1000
    g = torch.Generator(device=dev).manual_seed(5)
    heavy = torch.rand(n, device=dev, generator=g) < 0.9
    assert 0.9 * n / sms * 4095 > 2 ** 32
    keys = torch.where(heavy, torch.full((n,), heavy_key, dtype=torch.int64, device=dev),
                       torch.randint(0, nkeys + 10, (n,), device=dev, generator=g))
    mid1 = torch.randint(0, 10 ** 8, (n,), device=dev, generator=g, dtype=torch.int64)
    mid2 = mid1 + keys * R
    count = torch.where(heavy, torch.full((n,), 4095, dtype=torch.int64, device=dev),
                        torch.randint(0, 6, (n,), device=dev, generator=g))
    del keys, heavy
    for min_dist, max_dist in ((0, (nkeys - 1) * R), (-1, -1)):
        d = mid2 - mid1
        inr = torch.ones_like(d, dtype=torch.bool)
        if min_dist > -1:
            inr &= d > min_dist
        if max_dist > -1:
            inr &= d <= max_dist
        ongrid = inr & (d % R == 0) & (d // R < nkeys) & (d >= 0)
        ref = torch.zeros(nkeys, dtype=torch.int64, device=dev).index_add_(0, (d[ongrid] // R), count[ongrid])
        S = int(count[inr].sum())
        n_in = int(inr.sum())
        del d, inr, ongrid
        eng = PassEngine(R, 100, min_dist, max_dist, nkeys, device=dev)
        sh = Shard(mid1.to(torch.int32), mid2.to(torch.int32), count.to(torch.int32))
        eng.hist([sh])
        torch.cuda.synchronize()
        assert torch.equal(eng.obs_sum, ref)
        t = eng.totals.cpu().numpy()
        assert int(t[0]) == S and int(t[1]) == n_in
        assert int(ref[heavy_key]) > 2 ** 32
        del sh, eng, ref
        torch.cuda.empty_cache()


# ------------------------------------------------------------------------------------------------ d. end to end
def _sparse_records(bins, seed, rows_per_key=50):
    """About rows_per_key rows per key of each chromosome, log-uniform distances over its whole span, zero rows; each
    chromosome's rows one contiguous block."""
    from blueberry_b200 import synth
    rng = np.random.default_rng(seed)
    chr_, m1, m2, cnt = [], [], [], []
    for c, nb in enumerate(bins):
        n = rows_per_key * nb
        dk = np.floor(np.exp(rng.uniform(0, np.log(nb), n))).astype(np.int64) - 1
        dk[rng.random(n) < 0.02] = 0
        i = (rng.random(n) * (nb - dk)).astype(np.int64)
        lam = 40.0 * (dk + 1.0) ** -0.8
        count = rng.poisson(lam).astype(np.int64)
        count[rng.random(n) < 0.05] = 0
        count[rng.random(n) < 0.5 * (count == 0)] += 1
        count[rng.random(n) < 1e-3] += 300                     # outliers for the refit pass
        order = np.lexsort((i + dk, i))
        chr_.append(np.full(n, c, np.int32))
        m1.append((i[order] * R + R // 2).astype(np.int32))
        m2.append(((i + dk)[order] * R + R // 2).astype(np.int32))
        cnt.append(count[order].astype(np.int32))
    fc, fm = synth.make_fragments(bins, R)
    bias = synth.make_bias(bins, seed, sigma=0.25)
    barr = (np.concatenate([np.full(b, i, dtype=np.int32) for i, b in enumerate(bins)]), fm.copy(), np.concatenate(bias))
    return dict(fc=fc, fm=fm, chr=np.concatenate(chr_), mid1=np.concatenate(m1), mid2=np.concatenate(m2), count=np.concatenate(cnt),
                bias=barr)


def _compare_pass(out, ref):
    from oracle import fithic_oracle as fo
    assert np.array_equal(out.possible, ref.frag.possible)
    assert np.array_equal(out.observed, ref.contacts.observed)
    assert out.totals["observedIntraInRangeSum"] == ref.contacts.S
    assert np.array_equal(out.bin_of_key, ref.bin_of_key)
    assert np.array_equal(out.x, np.array(ref.x)) and np.array_equal(out.y, np.array(ref.y))
    assert out.spline_x[0] == ref.k0 * R and len(out.spline_y) == len(ref.spline_y)
    assert np.array_equal(out.spline_y, ref.spline_y)
    assert abs(out.residual - ref.residual) <= 1e-12 * abs(ref.residual)
    assert np.array_equal(out.keep, ref.keep)
    sel = ref.keep & (ref.p >= 1e-300)
    ok, nbad = log10_close(out.p[sel], ref.p[sel], 1e-5)
    assert ok, "%d p-values differ by more than 1e-5 in log10" % nbad
    assert (out.p[ref.keep & (ref.p < 1e-300)] <= 1e-299).all()
    qref = fo.benjamini_hochberg_correction(out.p[out.keep], int(out.keep.sum()))
    assert np.array_equal(out.q[out.keep], qref)
    m, L = len(out.x), len(out.spline_y)
    print("m=%d nkeys=%d L=%d" % (m, len(out.possible), L))
    return m, L


def _oracle_pass(k, chrom, min_dist, max_dist):
    from oracle import fithic_oracle as fo
    rows = k["chr"] == chrom
    fsel = k["fc"] == chrom
    bsel = k["bias"][0] == chrom
    bd = fo.read_bias_arrays(k["bias"][0][bsel], k["bias"][1][bsel], k["bias"][2][bsel])[0]
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        return fo.fithic_arrays(k["fc"][fsel], k["fm"][fsel], k["chr"][rows], k["mid1"][rows], k["chr"][rows], k["mid2"][rows],
                                k["count"][rows], R, 100, min_dist, max_dist, bias=bd)


@pytest.fixture(scope="module")
def chr1_5kb():
    return _sparse_records([49851], 101)


def test_end_to_end_reference_defaults(chr1_5kb):
    from blueberry_b200.fithic import FitHiC
    k = chr1_5kb
    model = FitHiC("unused", R)                                 # max_dist = min_dist = -1: the reference's defaults
    out = model.fit_transform_arrays(None, k["mid1"], None, k["mid2"], k["count"], k["fc"], k["fm"], bias=k["bias"], q_values=True)
    _compare_pass(out, _oracle_pass(k, 0, model.min_dist, model.max_dist))


def test_end_to_end_whole_span(chr1_5kb):
    from blueberry_b200.fithic import FitHiC
    k = chr1_5kb
    span = (49851 - 1) * R
    model = FitHiC("unused", R, min_dist=0, max_dist=span)
    out = model.fit_transform_arrays(None, k["mid1"], None, k["mid2"], k["count"], k["fc"], k["fm"], bias=k["bias"], q_values=True)
    m, L = _compare_pass(out, _oracle_pass(k, 0, 0, span))
    assert need_eval(m, L) > POOL_DOUBLES and L > 6320


def test_end_to_end_per_chromosome_mixes_regimes():
    from blueberry_b200.fithic import FitHiC
    bins = [49851, 3000, 800]
    k = _sparse_records(bins, 103, rows_per_key=30)
    span = (bins[0] - 1) * R
    model = FitHiC("unused", R, min_dist=0, max_dist=span)
    out = model.fit_transform_arrays(k["chr"], k["mid1"], k["chr"], k["mid2"], k["count"], k["fc"], k["fm"], bias=k["bias"],
                                     q_values=True, per_chromosome=True)
    regimes = set()
    for c in range(3):
        m, L = _compare_pass(out[c], _oracle_pass(k, c, 0, span))
        regimes.add(frozenset(global_phases(len(out[c].possible), max(4, min(bins[c], 512)), m, L)))
    assert frozenset() in regimes and any("binning" in r for r in regimes)


def test_end_to_end_refit_on_the_long_chromosome(chr1_5kb):
    from blueberry_b200.fithic import FitHiC
    from oracle import fithic_oracle as fo
    k = chr1_5kb
    span = (49851 - 1) * R
    model = FitHiC("unused", R, min_dist=0, max_dist=span)
    bd = fo.read_bias_arrays(*k["bias"])[0]
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        r1, r2, outlier, thr = fo.fithic_two_pass_arrays(k["fc"], k["fm"], None, k["mid1"], None, k["mid2"], k["count"], R, 100,
                                                         0, span, bias=bd)
    with np.errstate(invalid="ignore", divide="ignore"):
        assert not (r1.keep & (np.abs(r1.p / thr - 1.0) < 1e-9)).any()
    out = model.fit_transform_arrays(None, k["mid1"], None, k["mid2"], k["count"], k["fc"], k["fm"], bias=k["bias"], refit=True,
                                     q_values=True)
    assert int(outlier.sum()) > 0
    assert np.array_equal(out.observed, r2.contacts.observed)
    assert out.totals["observedIntraInRangeSum"] == r2.contacts.S
    assert np.array_equal(out.x, np.array(r2.x)) and np.array_equal(out.y, np.array(r2.y))
    assert np.array_equal(out.spline_y, r2.spline_y)
    assert np.array_equal(out.keep, r2.keep)
    sel = r2.keep & (r2.p >= 1e-300)
    ok, nbad = log10_close(out.p[sel], r2.p[sel], 1e-5)
    assert ok, "%d p-values differ by more than 1e-5 in log10" % nbad
    qref = fo.benjamini_hochberg_correction(out.p[out.keep], int(out.keep.sum()))
    assert np.array_equal(out.q[out.keep], qref)
