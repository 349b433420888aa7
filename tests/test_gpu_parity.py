"""GPU parity tests: the CUDA path (through the C ABI of libbbk.so) against the CPU oracle and the
golden vectors minted from the reference.  Run on the B200 box with `pytest -m gpu`.

Bars (BASELINE.md section 4, DESIGN.md "Parity contract"):
  * bit-exact: possible pairs, per-distance sums, all totals, bin membership, bin x / y, spline knots,
    BH q-values given the same p, BH ranks, count_band_regions;
  * |delta log10 p| <= 1e-6 against the reference's own output (golden files, S up to 2e5);
  * |delta log10 p| <= 1e-5 against scipy.special.bdtrc at S up to 2^31 (cephes' own error there is
    3e-6, measured against 60-digit arithmetic) and <= 1e-9 against the 60-digit value.
"""
import ctypes

import os

import numpy as np
import pytest

from helpers import PASS_CASES, golden_bias_dict, load_golden, log10_close

pytestmark = pytest.mark.gpu

P_TOL_GOLDEN = 1e-6
P_TOL_SCIPY = 1e-5
P_TOL_TRUTH = 1e-9


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    assert torch.cuda.is_available()
    return torch


def _bias_arg(g):
    if not bool(g["has_bias"]):
        return None
    return (g["bias_chrom"], g["bias_mid"], g["bias_val"])


def _run_case(g, q_values=False):
    from blueberry_b200.fithic import FitHiC
    model = FitHiC("unused", int(g["resolution"]), n_bins=int(g["n_bins"]),
                   max_dist=int(g["max_dist_arg"]), min_dist=int(g["min_dist_arg"]))
    return model.fit_transform_arrays(g["chr1"], g["mid1"], g["chr2"], g["mid2"], g["count"],
                                      g["frag_chrom"], g["frag_mid"], bias=_bias_arg(g), q_values=q_values)


@pytest.mark.parametrize("name", PASS_CASES)
def test_pass_against_reference_golden(name, torch_cuda):
    g = load_golden(name)
    out = _run_case(g)
    # K2a / K1: integers, bit exact
    assert np.array_equal(out.possible, g["ref_possible"])
    assert np.array_equal(out.observed, g["ref_observed"])
    t = out.totals
    assert t["observedIntraInRangeSum"] == int(g["ref_S"])
    assert t["observedIntraInRangeCount"] == int(g["ref_intra_in_range_count"])
    assert t["observedIntraAllSum"] == int(g["ref_intra_all_sum"])
    assert t["observedIntraAllCount"] == int(g["ref_intra_all_count"])
    assert t["observedInterAllSum"] == int(g["ref_inter_all_sum"])
    assert t["observedInterAllCount"] == int(g["ref_inter_all_count"])
    assert t["minObservedGenomicDist"] == int(g["ref_min_obs_dist"])
    assert t["maxObservedGenomicDist"] == int(g["ref_max_obs_dist"])
    assert t["maxPossibleGenomicDist"] == int(g["ref_max_possible_dist"])
    assert t["possibleIntraInRangeCount"] == int(g["ref_possible_intra_in_range"])
    assert t["possibleIntraAllCount"] == int(g["ref_possible_intra_all"])
    assert t["possibleInterAllCount"] == int(g["ref_possible_inter_all"])
    # K2b: bins, bit exact (same float64 operation order as the reference loop)
    assert np.array_equal(out.x, g["ref_x"])
    assert np.array_equal(out.y, g["ref_y"])
    # K3: spline grid and antitonic values
    assert np.array_equal(out.spline_x, g["ref_spline_x"])
    assert np.allclose(out.spline_y, g["ref_spline_y"], rtol=1e-12, atol=0)
    n_exact = int((out.spline_y == g["ref_spline_y"]).sum())
    print("%s: spline_y bit-exact on %d of %d grid points; residual %r vs %r" %
          (name, n_exact, len(out.spline_y), out.residual, float(g["ref_residual"])))
    assert abs(out.residual - float(g["ref_residual"])) <= 1e-12 * abs(float(g["ref_residual"]))
    # K4: the rows the reference emitted, in order, with its p-values
    keep = out.keep
    assert int(keep.sum()) == len(g["ref_out_p"])
    assert np.array_equal(g["mid1"][keep], g["ref_out_mid1"])
    assert np.array_equal(g["mid2"][keep], g["ref_out_mid2"])
    assert np.array_equal(g["count"][keep], g["ref_out_count"])
    ok, nbad = log10_close(out.p[keep], g["ref_out_p"], P_TOL_GOLDEN)
    assert ok, "%d p-values differ by more than %g in log10" % (nbad, P_TOL_GOLDEN)


@pytest.mark.parametrize("name", PASS_CASES)
def test_bin_membership_bit_exact(name, torch_cuda):
    from oracle import fithic_oracle as fo
    g = load_golden(name)
    out = _run_case(g)
    _, _, _, bok = fo.calculate_probabilities(g["ref_possible"], g["ref_observed"], int(g["ref_S"]), int(g["n_bins"]),
                                              int(g["resolution"]), int(g["ref_min_dist"]), int(g["ref_max_dist"]))
    assert np.array_equal(out.bin_of_key, bok)


def _score_table(torch, priors, counts, S, bias=None):
    """Drive K4 directly: record i looks up priors[i] (mid1 = 0, mid2 = i, resolution 1)."""
    from blueberry_b200 import _lib
    from blueberry_b200.engine import PassEngine, Shard
    n = len(priors)
    eng = PassEngine(1, 100, 0, n, n, torch.device("cuda:0"))
    eng.spline_y[:n] = torch.from_numpy(np.asarray(priors, dtype=np.float64)).cuda()
    fr = _lib.FitResult(status=0, n_out=100, k0=0, L=n, n_knots=8, ier=0, S=int(S), min_x=0.0, max_x=float(n - 1),
                        residual=0.0, fp=0.0, smoothing=0.0)
    eng.fit_result.copy_(torch.frombuffer(bytearray(bytes(fr)), dtype=torch.uint8))
    z = torch.zeros(n, dtype=torch.int32, device="cuda:0")
    mid2 = torch.arange(n, dtype=torch.int32, device="cuda:0")
    cnt = torch.from_numpy(np.asarray(counts, dtype=np.int32)).cuda()
    p = torch.empty((n + 1) & ~1, dtype=torch.float64, device="cuda:0")[:n]
    eng.pvalues(Shard(z, mid2, cnt), p)
    torch.cuda.synchronize()
    return p.cpu().numpy()


def _random_tail_cases(rng, n, S):
    mu = 10 ** rng.uniform(-4, 3.3, n)
    mu = np.minimum(mu, S * 0.4)
    q = mu / S
    sd = np.sqrt(mu)
    c = np.maximum(0, mu + rng.uniform(-6, 12, n) * sd + rng.integers(0, 4, n)).astype(np.int64)
    small = rng.random(n) < 0.3
    c[small] = rng.integers(0, 12, int(small.sum()))
    c = np.minimum(c, min(S, 2**31 - 1))
    return q, c


@pytest.mark.parametrize("S", [1000, 213498, 50_000_000, 1_500_000_000, 2**31 - 1])
def test_pvalue_kernel_against_scipy(S, torch_cuda):
    import scipy.special as sc
    rng = np.random.default_rng(S % 9973)
    q, c = _random_tail_cases(rng, 200_001, S)      # odd length: exercises the scalar tail of the kernel
    got = _score_table(torch_cuda, q, c, S)
    with np.errstate(all="ignore"):
        ref = sc.bdtrc((c - 1).astype(np.float64), np.int64(S), q)
    assert not np.isnan(got).any() and not np.isnan(ref).any()
    big = ref >= 1e-300                              # below that cephes is in its denormal / underflow regime
    ok, nbad = log10_close(got[big], ref[big], P_TOL_SCIPY)
    assert ok, "%d of %d differ by more than %g in log10" % (nbad, int(big.sum()), P_TOL_SCIPY)
    assert (got[~big] <= 1e-299).all()
    assert (got[c == 0] == 1.0).all()
    err = np.abs(np.log10(got[big & (ref < 1)]) - np.log10(ref[big & (ref < 1)]))
    print("S=%d: max |dlog10 p| vs scipy %.3g, p99 %.3g" % (S, err.max(), np.percentile(err, 99)))


def test_pvalue_kernel_against_60_digit_truth(torch_cuda):
    import mpmath as mp
    mp.mp.dps = 60
    rng = np.random.default_rng(77)
    S = 1_234_567_891
    q, c = _random_tail_cases(rng, 600, S)
    c = np.maximum(c, 2)
    got = _score_table(torch_cuda, q, c, S)

    def truth(cc, n, qq):
        qq = mp.mpf(float(qq))
        lp = mp.loggamma(n + 1) - mp.loggamma(cc + 1) - mp.loggamma(n - cc + 1) + cc * mp.log(qq) + (n - cc) * mp.log(1 - qq)
        qr = qq / (1 - qq)
        if cc >= (n + 1) * qq:
            term = mp.mpf(1); s = mp.mpf(1); j = cc
            while j < n:
                term *= mp.mpf(n - j) / (j + 1) * qr; s += term; j += 1
                if term < mp.mpf(10) ** -45 * s:
                    break
            return mp.exp(lp) * s
        term = mp.mpf(cc) / ((n - cc + 1) * qr); s = term; j = cc - 1
        while j > 0:
            term *= mp.mpf(j) / ((n - j + 1) * qr); s += term; j -= 1
            if term < mp.mpf(10) ** -45 * s:
                break
        return 1 - mp.exp(lp) * s

    worst = 0.0
    for i in range(len(c)):
        tv = truth(int(c[i]), S, q[i])
        if tv < mp.mpf(10) ** -290:
            continue
        worst = max(worst, abs(float(mp.log10(tv)) - np.log10(got[i])))
    print("max |dlog10 p| vs 60-digit truth: %.3g" % worst)
    assert worst <= P_TOL_TRUTH


def test_pvalue_edge_semantics_match_bdtrc(torch_cuda):
    import scipy.special as sc
    S = 100
    priors = np.array([-0.5, 1.5, 0.5, 0.5, 0.5, 0.0, 1.0, 0.0, 1.0, np.nan, 0.02, 0.005, 0.3, 0.3, -0.1, 0.5])
    counts = np.array([0, 0, 0, -3, 102, 1, 1, 2, 2, 3, 1, 1, 101, 100, 5, 7])
    got = _score_table(torch_cuda, priors, counts, S)
    with np.errstate(all="ignore"):
        ref = sc.bdtrc((counts - 1).astype(np.float64), np.int64(S), priors)
    ref = np.where(ref <= 1, ref, np.nan)             # fithic.py:434 drops the row
    assert np.array_equal(np.isnan(got), np.isnan(ref))
    m = ~np.isnan(ref)
    assert np.allclose(got[m], ref[m], rtol=1e-12, atol=0)
    assert got[2] == 1.0 and got[3] == 1.0 and got[5] == 0.0 and got[6] == 1.0 and got[12] == 0.0


def _bh_device(torch, p, n_tests, positional=False, want_rank=False):
    from blueberry_b200 import _lib
    lib = _lib.load()
    m = len(p)
    dp = torch.empty((m + 1) & ~1, dtype=torch.float64, device="cuda:0")[:m].copy_(torch.from_numpy(np.asarray(p, np.float64)))
    dq = torch.full(((m + 1) & ~1,), -7.0, dtype=torch.float64, device="cuda:0")[:m]
    dr = torch.full((m,), -7, dtype=torch.int64, device="cuda:0") if want_rank else None
    ws = torch.empty(int(lib.bbk_bh_workspace_bytes(m)), dtype=torch.uint8, device="cuda:0")
    _lib.check(lib.bbk_bh_qvalues(_lib.ptr(dp), m, int(n_tests), _lib.BH_POSITIONAL if positional else _lib.BH_UNSORTED,
                                  None, _lib.ptr(dq), _lib.ptr(dr), _lib.ptr(ws), ws.numel(), _lib.stream_ptr()), "bh")
    torch.cuda.synchronize()
    return dq.cpu().numpy(), (dr.cpu().numpy() if want_rank else None)


def test_bh_against_reference_golden(torch_cuda):
    from blueberry_b200.blueberry import benjamini_hochberg, count_band_regions
    from blueberry_b200.fithic import benjamini_hochberg_correction
    g = load_golden("bh_band")
    for tag in ("a", "b", "c", "doc"):
        p, n = g["p_" + tag], int(g["n_" + tag])
        q = benjamini_hochberg_correction(list(p), n)
        assert isinstance(q, list)
        assert np.array_equal(np.array(q), g["q_py_" + tag]), tag
        qs = benjamini_hochberg(np.sort(p), n)
        assert isinstance(qs, np.ndarray) and qs.dtype == np.float64
        assert np.array_equal(qs, g["q_cy_sorted_" + tag]), tag
    assert count_band_regions(g["regions_sorted"]) == int(g["band_sorted"])
    assert count_band_regions(g["regions_shuffled"]) == int(g["band_shuffled"])


@pytest.mark.parametrize("m,frac_ones,n_scale", [(1, 0.0, 1.0), (2, 0.5, 1.0), (4097, 0.0, 1.0), (300_001, 0.6, 1.0),
                                                  (300_001, 0.0, 50.0), (300_001, 0.3, 0.01), (2_000_003, 0.8, 1.0)])
def test_bh_random_bit_exact(m, frac_ones, n_scale, torch_cuda):
    from oracle import fithic_oracle as fo
    rng = np.random.default_rng(m + int(frac_ones * 10))
    p = rng.random(m) ** 3
    p[rng.random(m) < frac_ones] = 1.0
    if m > 100:
        p[rng.integers(0, m, m // 10)] = p[rng.integers(0, m, m // 10)]      # ties
        p[rng.integers(0, m, 5)] = 0.0
        p[rng.integers(0, m, 5)] = 5e-324
        p[rng.integers(0, m, 50)] = 10.0 ** rng.uniform(-300, -5, 50)
    n_tests = max(1, int(m * n_scale))
    q, _ = _bh_device(torch_cuda, p, n_tests)
    ref = fo.benjamini_hochberg_correction(p, n_tests)
    assert np.array_equal(q, ref)
    # with NaN rows (dropped by fithic.py:434): not ranked, q = NaN, others unchanged
    if m > 100:
        p2 = p.copy()
        nan_at = rng.integers(0, m, m // 20)
        p2[nan_at] = np.nan
        q2, rk = _bh_device(torch_cuda, p2, n_tests, want_rank=True)
        valid = ~np.isnan(p2)
        ref2 = fo.benjamini_hochberg_correction(p2[valid], n_tests)
        assert np.isnan(q2[~valid]).all() and np.array_equal(q2[valid], ref2)
        srt = np.sort(p2[valid])
        assert np.array_equal(rk[valid], 1 + np.searchsorted(srt, p2[valid], side="left"))
        assert (rk[~valid] == 0).all()


def test_bh_positional_matches_cython_semantics(torch_cuda):
    from oracle import fithic_oracle as fo
    rng = np.random.default_rng(4)
    for m in (1, 7, 100_003):
        p = np.sort(rng.random(m) ** 2)
        q, _ = _bh_device(torch_cuda, p, 3 * m, positional=True)
        assert np.array_equal(q, fo.benjamini_hochberg_sorted(p, 3 * m))
        # not actually sorted: the reference does not care, it scans in the given order (blueberry.pyx:67-73)
        p = rng.random(m)
        q, _ = _bh_device(torch_cuda, p, m, positional=True)
        assert np.array_equal(q, fo.benjamini_hochberg_sorted(p, m))


@pytest.mark.parametrize("n", [0, 1, 2, 257, 5000])
def test_count_band_regions(n, torch_cuda):
    from blueberry_b200.blueberry import count_band_regions
    from oracle import fithic_oracle as fo
    rng = np.random.default_rng(n)
    reg = np.sort(rng.choice(60000, n, replace=False)).astype(np.float64) * 1000 + 500
    assert count_band_regions(reg) == fo.count_band_regions(reg)
    if n > 2:
        shuf = reg[rng.permutation(n)]
        assert count_band_regions(shuf) == fo.count_band_regions(shuf)
        dup = np.sort(np.concatenate([reg, reg[: n // 3]]))
        assert count_band_regions(dup) == fo.count_band_regions(dup)
    with pytest.raises(TypeError):
        count_band_regions(reg.astype(np.float32))


def test_fit_stage_injection_against_scipy(torch_cuda):
    """K3 alone on given (x, y): knots bit-exact against scipy's FITPACK, antitonic values against sklearn."""
    import warnings
    from scipy.interpolate import UnivariateSpline
    from sklearn.isotonic import IsotonicRegression
    from blueberry_b200 import _lib
    torch = torch_cuda
    lib = _lib.load()
    rng = np.random.default_rng(12)
    R, nkeys = 5000, 2001
    exact_knots = 0
    trials = 25
    for trial in range(trials):
        m = int(rng.integers(8, 140))
        x = np.sort(rng.choice(np.arange(1, nkeys - 1), m, replace=False)).astype(np.float64) * R + rng.random(m) * 100
        y = 1e-3 * (x / R + 1) ** -1.08 * np.exp(rng.normal(0, 0.08 if trial % 2 else 0.3, m))
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            ius = UnivariateSpline(x, y, s=float(min(y) ** 2))
        keys = np.arange(nkeys) * R
        sx = keys[(keys >= x.min()) & (keys <= x.max())]
        raw = ius(sx)
        ref = IsotonicRegression(increasing=False).fit_transform(sx, raw)
        dx, dy = torch.from_numpy(x).cuda(), torch.from_numpy(y).cuda()
        res = torch.zeros(ctypes.sizeof(_lib.FitResult), dtype=torch.uint8, device="cuda:0")
        sy = torch.zeros(nkeys, dtype=torch.float64, device="cuda:0")
        sraw = torch.zeros(nkeys, dtype=torch.float64, device="cuda:0")
        kn = torch.zeros(m + 8, dtype=torch.float64, device="cuda:0")
        co = torch.zeros(m + 8, dtype=torch.float64, device="cuda:0")
        nb = int(lib.bbk_fit_workspace_bytes(max(m, 4), nkeys)) + 16 * m + 64
        ws = torch.zeros(nb, dtype=torch.uint8, device="cuda:0")
        _lib.check(lib.bbk_fit_from_bins(_lib.ptr(dx), _lib.ptr(dy), m, nkeys, R, _lib.ptr(res), _lib.ptr(sy), _lib.ptr(sraw),
                                         _lib.ptr(kn), _lib.ptr(co), _lib.ptr(ws), nb, _lib.stream_ptr()), "fit_from_bins")
        torch.cuda.synchronize()
        fr = _lib.FitResult.from_buffer_copy(res.cpu().numpy().tobytes())
        assert fr.status == 0
        t_ref = ius._data[8][:ius._data[7]]
        assert fr.n_knots == len(t_ref)
        assert np.array_equal(kn.cpu().numpy()[:fr.n_knots], t_ref)
        exact_knots += 1
        assert fr.L == len(sx) and fr.k0 * R == sx[0]
        assert np.array_equal(co.cpu().numpy()[:fr.n_knots - 4], ius._data[9][:fr.n_knots - 4])
        assert np.array_equal(sraw.cpu().numpy()[:fr.L], raw)
        assert np.array_equal(sy.cpu().numpy()[:fr.L], ref)
    assert exact_knots == trials


def test_error_behaviour_matches_reference(torch_cuda):
    from blueberry_b200.fithic import FitHiC
    from blueberry_b200 import synth
    R = 10000
    fc, fm = synth.make_fragments([50], R)
    c = synth.make_contacts([50], R, 200000, 5.0, 3)
    model = FitHiC("x", R, n_bins=20, max_dist=200000)
    # no in-range contacts at all -> the reference divides by observedIntraInRangeSum == 0 (fithic.py:216)
    with pytest.raises(ZeroDivisionError):
        model.fit_transform_arrays(None, c["mid1"], None, c["mid2"], np.zeros_like(c["count"]), fc, fm)
    # too few bins for a cubic spline -> scipy's "m > k must hold"
    with pytest.raises(ValueError):
        FitHiC("x", R, n_bins=2, max_dist=200000).fit_transform_arrays(None, c["mid1"], None, c["mid2"], c["count"], fc, fm)


@pytest.mark.parametrize("m,frac_ones,n_scale", [(300_001, 0.6, 1.0), (300_001, 0.3, 0.01), (50_000, 0.0, 40.0)])
def test_bh_fixed_capacity_gather_single_rank_equals_local(m, frac_ones, n_scale, torch_cuda):
    """The select / fixed-capacity gather / rank / scatter pipeline used across GPUs, run with one rank (the all-gather then
    delivers the send block itself), against the oracle; then with a capacity below the candidate count, which must be
    reported."""
    import ctypes
    from blueberry_b200 import _lib
    from oracle import fithic_oracle as fo
    torch = torch_cuda
    lib = _lib.load()
    dev = torch.device("cuda:0")
    rng = np.random.default_rng(m + 3)
    p = rng.random(m) ** 3
    p[rng.random(m) < frac_ones] = 1.0
    p[rng.integers(0, m, m // 10)] = p[rng.integers(0, m, m // 10)]
    p[rng.integers(0, m, m // 50)] = np.nan
    n_tests = max(1, int(m * n_scale))
    dp = torch.empty((m + 1) & ~1, dtype=torch.float64, device=dev)[:m].copy_(torch.from_numpy(p))
    dq = torch.full(((m + 1) & ~1,), -7.0, dtype=torch.float64, device=dev)[:m]
    # K4's coarse histogram: bucket (bits >> 51) & 4095 of a p in [0, 1), p == 1.0 in slot 4096, NaN in slot 4097
    nan, one = torch.isnan(dp), dp == 1.0
    hist = torch.zeros(_lib.PHIST_LEN, dtype=torch.int64, device=dev)
    hist[:_lib.PHIST_BINS] = torch.bincount(((dp.view(torch.int64) >> 51) & 4095)[~nan & ~one], minlength=_lib.PHIST_BINS)
    hist[_lib.PHIST_BINS] = one.sum()
    hist[_lib.PHIST_BINS + 1] = nan.sum()
    st = _lib.stream_ptr()

    def gathered(cap):
        send = torch.zeros(cap + 1, dtype=torch.int64, device=dev)
        idx = torch.empty(max(cap, 1), dtype=torch.int32, device=dev)
        state = torch.zeros(4, dtype=torch.int64, device=dev)
        q_ones = torch.zeros(2, dtype=torch.float64, device=dev)
        overflow = torch.zeros(1, dtype=torch.int32, device=dev)
        sel_ws = torch.empty(int(lib.bbk_bh_workspace_bytes(0)), dtype=torch.uint8, device=dev)
        gat_ws = torch.empty(int(lib.bbk_bh_gathered_workspace_bytes(1, cap)), dtype=torch.uint8, device=dev)
        _lib.check(lib.bbk_bh_select(_lib.ptr(dp), m, n_tests, _lib.ptr(hist), _lib.ptr(dq), ctypes.c_void_p(send.data_ptr() + 8),
                                     _lib.ptr(idx), cap, _lib.ptr(state), _lib.ptr(sel_ws), sel_ws.numel(), st), "bbk_bh_select")
        _lib.check(lib.bbk_bh_pack_count(_lib.ptr(state), _lib.ptr(send), st), "bbk_bh_pack_count")
        recv = send
        _lib.check(lib.bbk_bh_rank_gathered_padded(_lib.ptr(recv), 1, cap, 0, _lib.ptr(state), _lib.ptr(idx), _lib.ptr(dq), _lib.ptr(q_ones),
                                                   _lib.ptr(overflow), _lib.ptr(gat_ws), gat_ws.numel(), st), "bbk_bh_rank_gathered_padded")
        _lib.check(lib.bbk_bh_fix_ones_dev(_lib.ptr(dp), m, _lib.ptr(q_ones), _lib.ptr(dq), st), "bbk_bh_fix_ones_dev")
        torch.cuda.synchronize()
        return int(state[0].item()), int(overflow.item())

    n_cand, ov = gathered(m)
    q = dq.cpu().numpy()
    valid = ~np.isnan(p)
    assert np.isnan(q[~valid]).all()
    assert np.array_equal(q[valid], fo.benjamini_hochberg_correction(p[valid], n_tests))
    assert ov == 0 and n_cand > 0
    assert gathered(n_cand - 1) == (n_cand, n_cand)


def test_second_pass_against_composed_reference_golden(torch_cuda):
    """BASELINE config 4's refit after outlier removal, against the golden output of the reference's own functions
    composed as in SURVEY 8c (tests/golden/pass2_bias_dense.npz)."""
    from blueberry_b200.fithic import FitHiC
    g = load_golden("pass_bias_dense")
    g2 = load_golden("pass2_bias_dense")
    model = FitHiC("unused", int(g["resolution"]), n_bins=int(g["n_bins"]), max_dist=int(g["max_dist_arg"]), min_dist=int(g["min_dist_arg"]))
    out = model.fit_transform_arrays(g["chr1"], g["mid1"], g["chr2"], g["mid2"], g["count"], g["frag_chrom"], g["frag_mid"],
                                     bias=_bias_arg(g), refit=True, q_values=True)
    assert np.array_equal(out.observed, g2["ref2_observed"])
    assert out.totals["observedIntraInRangeSum"] == int(g2["ref2_S"])
    with np.errstate(invalid="ignore"):
        assert int((out.p_first <= float(g2["threshold"])).sum()) == int(g2["n_outliers"])
    assert np.array_equal(out.x, g2["ref2_x"]) and np.array_equal(out.y, g2["ref2_y"])
    assert np.array_equal(out.spline_x, g2["ref2_spline_x"])
    assert np.array_equal(out.spline_y, g2["ref2_spline_y"])
    keep = out.keep
    assert np.array_equal(g["mid1"][keep], g2["ref2_out_mid1"]) and np.array_equal(g["count"][keep], g2["ref2_out_count"])
    ok, nbad = log10_close(out.p[keep], g2["ref2_out_p"], P_TOL_GOLDEN)
    assert ok, nbad


# K1 works on tiles of 4096 records (two groups of four per thread, 512 threads); sizes on either side of the tile and
# group boundaries, all five kernel variants (32-bit fast path with the records staged through shared memory / the same with a
# table too large for the stages ("fast_wide") / general, fast and general with chromosome columns), coordinates that
# wrap a 32-bit subtraction, off-grid and negative distances, counts above the shared-histogram limit and below zero.
@pytest.mark.parametrize("n", [1, 3, 4, 5, 4093, 4095, 4096, 4097, 4099, 8192, 8195, 12288 + 7, 100003, 1_300_001])
@pytest.mark.parametrize("variant", ["fast", "fast_wide", "general", "chrom", "chrom_general"])
def test_hist_kernel_edge_sizes_against_oracle(n, variant, torch_cuda):
    torch = torch_cuda
    from blueberry_b200.engine import PassEngine, Shard
    from oracle import fithic_oracle as fo
    rng = np.random.default_rng(n * 3 + len(variant))
    R, nkeys = 5000, 700
    bins = rng.integers(0, 900, size=(2, n))
    mid1 = (2500 + R * bins.min(axis=0)).astype(np.int64)
    mid2 = (2500 + R * bins.max(axis=0)).astype(np.int64)
    k = rng.choice(n, max(n // 40, 1), replace=False)
    mid2[k] += rng.integers(1, R, size=len(k))                       # off the grid
    k = rng.choice(n, max(n // 60, 1), replace=False)
    mid1[k], mid2[k] = mid2[k].copy(), mid1[k].copy()                # negative distances
    k = rng.choice(n, max(n // 90, 1), replace=False)
    mid1[k] = rng.choice([-2**31, -2**31 + 1, -5, 2**31 - 1], size=len(k))
    k = rng.choice(n, max(n // 90, 1), replace=False)
    mid2[k] = rng.choice([-2**31, 2**31 - 1, 2**31 - 2, -1], size=len(k))
    count = rng.poisson(0.7, size=n).astype(np.int64)
    k = rng.choice(n, max(n // 70, 1), replace=False)
    count[k] = rng.choice([4095, 4096, 4097, 2**31 - 1, -3, 100000], size=len(k))
    chr1 = chr2 = None
    if variant.startswith("chrom"):
        chr1 = rng.integers(0, 3, size=n).astype(np.int32)
        chr2 = np.where(rng.random(n) < 0.9, chr1, (chr1 + 1) % 3).astype(np.int32)
    if variant == "fast_wide":
        nkeys = 6000                                                 # 2 x (table + stages) does not fit an SM: streaming loads
    min_dist, max_dist = {"fast": (2 * R, 600 * R), "fast_wide": (2 * R, 5900 * R), "general": (-1, -1), "chrom": (R, 800 * R),
                          "chrom_general": (-1, 650 * R)}[variant]
    ref = fo.read_interactions(nkeys, R, chr1, mid1, chr2, mid2, count, min_dist, max_dist)

    dev = torch.device("cuda:0")
    to = lambda a: None if a is None else torch.from_numpy(np.ascontiguousarray(a, dtype=np.int32)).to(dev)
    sh = Shard(to(mid1), to(mid2), to(count), to(chr1), to(chr2))
    eng = PassEngine(R, 100, min_dist, max_dist, nkeys, device=dev)
    eng.hist([sh])
    torch.cuda.synchronize()
    t = eng.totals.cpu().numpy()
    assert np.array_equal(eng.obs_sum.cpu().numpy(), ref.observed)
    assert [int(v) for v in t] == [ref.S, ref.intra_in_range_count, ref.intra_all_sum, ref.intra_all_count,
                                   ref.inter_all_sum, ref.inter_all_count, ref.min_obs_dist, ref.max_obs_dist]

    # the second pass' histogram: the records with p <= threshold left out (fithic.py:413-435 feeding :229-270)
    p = rng.random(n)
    p[rng.choice(n, max(n // 10, 1), replace=False)] = 0.25
    keep = ~(p <= 0.25)
    ref2 = fo.read_interactions(nkeys, R, None if chr1 is None else chr1[keep], mid1[keep], None if chr2 is None else chr2[keep],
                                mid2[keep], count[keep], min_dist, max_dist)
    eng.hist_excluding([sh], [torch.from_numpy(p).to(dev)], 0.25)
    torch.cuda.synchronize()
    t = eng.totals.cpu().numpy()
    assert np.array_equal(eng.obs_sum.cpu().numpy(), ref2.observed)
    assert [int(v) for v in t] == [ref2.S, ref2.intra_in_range_count, ref2.intra_all_sum, ref2.intra_all_count,
                                   ref2.inter_all_sum, ref2.inter_all_count, ref2.min_obs_dist, ref2.max_obs_dist]


def test_extract_contacts_and_genome_qvalues_on_the_device():
    """bbk_extract_contacts (the order-preserving compaction behind utils.extract_contacts) and utils.genome_qvalues against
    the reference golden (bit for bit: rows, band counts, q) and, on a larger random table, against the oracle."""
    from blueberry_b200 import utils
    from blueberry_b200.datatypes import FithicContactMap
    from oracle import datatypes_oracle as do
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "extract_contacts.npz"))
    alpha = float(g["alpha"])
    maps = {int(c): g["map_%d" % c] for c in g["chroms"]}
    for c, m in maps.items():
        out, band = utils.extract_contacts_from_map(m, c, alpha, regions=do.regions(m))
        assert np.array_equal(out, g["ref_contacts_%d" % c]) and band == int(g["ref_band_%d" % c])
        assert np.array_equal(utils.extract_contacts_from_map(m, c), g["ref_contacts_noalpha_%d" % c])
    contacts, q, n = utils.genome_qvalues(maps, alpha)
    assert n == int(g["ref_n"])
    assert np.array_equal(contacts, np.concatenate([g["ref_contacts_%d" % c] for c in g["chroms"]]))
    assert np.array_equal(q, g["ref_q"])
    # maps given as FithicContactMap objects, no alpha, sizes that are not multiples of the chunk, an empty chromosome
    rng = np.random.default_rng(123)
    big = {}
    for c, n_rows in ((1, 70001), (2, 0), (9, 1025)):
        m1 = rng.integers(0, 4000, n_rows) * 5000 + 2500
        m2 = m1 + rng.integers(0, 2300, n_rows) * 5000
        p = rng.random(n_rows) ** 8
        if n_rows:
            p[rng.choice(n_rows, max(n_rows // 50, 1), replace=False)] = np.nan
        big[c] = np.stack([m1, m2, rng.integers(1, 40, n_rows), p, np.full(n_rows, -1.0)], axis=1).astype(np.float64).reshape(-1, 5)
    for a in (0.05, None):
        want_c, want_q, want_n = do.genome_qvalues(big, a)
        got_c, got_q, got_n = utils.genome_qvalues({c: FithicContactMap.from_arrays(m) for c, m in big.items()}, a)
        assert got_n == want_n and np.array_equal(got_c, want_c, equal_nan=True)
        assert np.array_equal(got_q, want_q, equal_nan=True)


def test_extract_contacts_reads_the_result_file_like_the_reference(tmp_path):
    """utils.extract_contacts(celltype, chromosome, resolution, alpha, n_regions) - the reference's signature: the chromosome's
    significances file is found through the DATA_DIR template (datatypes.pyx:26), read like FithicContactMap reads it, filtered
    on the device; a chromosome without a file gives (zeros((0, 5)), 0) and a message, like utils.py:65-67."""
    from blueberry_b200 import _io, utils
    from blueberry_b200.datatypes import FithicContactMap
    from oracle import datatypes_oracle as do
    rng = np.random.default_rng(8)
    n = 3000
    m1 = rng.integers(0, 2500, n) * 5000 + 2500
    m2 = m1 + rng.integers(0, 2300, n) * 5000
    p = rng.random(n) ** 5
    path = str(tmp_path / "{0}.chr{1}.res{2}.sig.txt.gz")
    _io.write_significances(path.format("cellX", 7, 5000), ["chr7"], None, m1, None, m2, rng.integers(1, 30, n), p, None)
    old = utils.DATA_DIR
    utils.DATA_DIR = path
    try:
        got, band = utils.extract_contacts("cellX", 7, 5000, alpha=0.2, n_regions=True)
        held = FithicContactMap(path.format("cellX", 7, 5000), 5000).map
        assert np.array_equal(got, do.extract_contacts(held, 7, 0.2))
        assert band == do.count_band_regions(do.regions(held))
        assert np.array_equal(utils.extract_contacts("cellX", 7, 5000), do.extract_contacts(held, 7))
        empty, zero = utils.extract_contacts("cellX", 8, 5000, alpha=0.2, n_regions=True)
        assert empty.shape == (0, 5) and zero == 0
    finally:
        utils.DATA_DIR = old

