"""The fit stage's arithmetic at the sizes of the reference's default call on a human chromosome (max_dist = min_dist = -1:
one distance key per resolution step, 49,851 keys for chr1 at 5 kb), compiled for the HOST by tests/host_harness (the
same source as the sm_100a kernel, 13 emulated threads) and compared with scipy / sklearn / the oracle bit for bit:

  * the smoothing spline at m on either side of 256 (the device's thread count) and of 772 (the last m whose spline
    workspace fits the fit kernel's shared pool), and up to 3000 bins, including searches that cross scipy's
    cap = max(m/2, 8) retry;
  * the segmented antitonic regression at grid lengths up to 50,000 with 128, 7 and 1 workers;
  * equal-occupancy binning on distance tables of 8,362 / 8,363 (the binning phase's pool boundary at max_bins 512),
    25,000 and 49,851 keys.
"""
import ctypes
import os
import warnings

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _p(a, t=ctypes.c_double):
    return a.ctypes.data_as(ctypes.POINTER(t))


@pytest.fixture(scope="module")
def harness():
    import __graft_entry__
    __graft_entry__.build()
    return ctypes.CDLL(os.path.join(ROOT, "tests", "host_harness", "libfit_harness.so"))


def synthetic_table(nkeys, seed, chroms=1, S_extra=0, zero_tail=0.15, spike=True, depth=1.0):
    """possible / observed of a distance table with nkeys keys: possible pairs of `chroms` chromosomes (the longest has
    nkeys fragments, fithic.py:302-311), a power-law decay with Poisson noise, runs of zero keys at far distances, one spike
    key whose count reaches `desired` for any n_bins >= 40, and S = the table sum + S_extra (off-grid records count in S, fithic.py:262)."""
    rng = np.random.default_rng(seed)
    sizes = [nkeys] + [int(nkeys * f) for f in rng.uniform(0.2, 0.8, chroms - 1)]
    k = np.arange(nkeys, dtype=np.int64)
    possible = np.zeros(nkeys, np.int64)
    for nf in sizes:
        possible += np.where(k <= nf - 1, nf - k, 0)
    lam = depth * 2e4 * (k + 1.0) ** -0.9 * possible / possible[0]
    observed = rng.poisson(lam).astype(np.int64)
    far = int(nkeys * (1 - zero_tail))
    for start in rng.integers(far, nkeys, 6):                   # zero runs at far keys
        observed[start:start + int(rng.integers(20, 400))] = 0
    if spike:
        observed[int(rng.integers(nkeys // 3, far))] += int(observed.sum()) // 40
    S = int(observed.sum()) + int(S_extra)
    return possible, observed, S


# ------------------------------------------------------------------------------------------------ smoothing spline
def _fit(fn, x, y, s):
    m = len(x)
    n = ctypes.c_int()
    fp = ctypes.c_double()
    t = np.zeros(m + 4)
    c = np.zeros(m + 4)
    ier = fn(_p(x), _p(y), m, ctypes.c_double(s), ctypes.byref(n), ctypes.byref(fp), _p(t), _p(c))
    return ier, n.value, t[:n.value].copy(), c[:n.value].copy()


def _spline_cases(m, seed):
    """The shapes of test_fit_stage_host._datasets at a fixed m: smooth, oscillating, noisy and flat decays, one with a zero
    y (s = 0: the interpolating spline), and s / 100."""
    rng = np.random.default_rng(seed)
    x = np.cumsum(rng.random(m) * 1e5 + 1)
    for kind in range(4):
        if kind == 0:
            y = 1e-3 * (x / 5000 + 1) ** -1.08 * np.exp(rng.normal(0, 0.05, m))
        elif kind == 1:
            y = 1e-4 * (1.5 + np.sin(x / 3e5 * rng.random())) + rng.random(m) * 3e-5
        elif kind == 2:
            y = 1e-3 * (x / 5000 + 1) ** -1.0 * np.exp(rng.normal(0, 0.3, m))
        else:
            y = 1e-5 * (x / 5000 + 1) ** -0.5 * (1 + 0.01 * rng.normal(0, 1, m))
        s = float(min(y) ** 2)
        yield "kind%d" % kind, x, y, s
        if kind in (0, 2):
            yield "kind%d/100" % kind, x, y, s * 1e-2
    y = 1e-3 * (x / 5000 + 1) ** -1.08 * np.exp(rng.normal(0, 0.1, m))
    y[int(rng.integers(0, m))] = 0.0
    yield "zero", x, y, 0.0


@pytest.mark.parametrize("m", [255, 256, 257, 772, 773, 1500, 3000])
def test_smoothing_spline_on_long_grids_is_bit_identical_to_scipy(m, harness):
    from scipy.interpolate import UnivariateSpline
    cap = max(m // 2, 8)
    iers, crossed = set(), 0
    for name, x, y, s in _spline_cases(m, m):
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            u = UnivariateSpline(x, y, s=s)
        d = u._data
        n_s, t_s, c_s, ier_s = d[7], d[8][:d[7]], d[9][:d[7]], d[13]
        fns = (harness.th_univariate_spline, harness.th_coop_univariate_spline) if m <= 1500 else (harness.th_coop_univariate_spline,)
        for fn in fns:
            ier, n, t, c = _fit(fn, x, y, s)
            assert (ier, n) == (ier_s, n_s), (name, fn.__name__)
            assert np.array_equal(t, t_s), (name, fn.__name__)
            assert np.array_equal(c[:n - 4], c_s[:n - 4]), (name, fn.__name__)
        iers.add(int(ier_s))
        crossed += n_s > cap + 4 and s > 0              # the capped first search gave up (ier 1): scipy's retry with m + 4
    assert -1 in iers and (0 in iers or 3 in iers or 2 in iers), iers
    assert crossed >= 1, "no case needed more knots than scipy's first search has room for"


# ------------------------------------------------------------------------------------------------ antitonic regression
def _antitonic_cases(L, rng):
    base = 1e-3 * (np.arange(L) + 1.0) ** -1.08
    yield "decreasing", base
    yield "wiggles", base * (1 + 0.2 * rng.normal(0, 1, L) * (rng.random(L) < 0.3))
    yield "oscillation", base * (1 + 0.02 * np.sin(np.arange(L) / 7.0))
    v = base.copy()
    v[rng.integers(0, L, L // 3 + 1)] = v[0]
    yield "ties", v
    yield "plateaus", np.repeat(base[:max(L // 5, 1)], 5)[:L]
    v = base.copy()
    k = rng.integers(0, L, L // 4 + 1)
    v[k] = np.nextafter(v[np.maximum(k - 1, 0)], rng.choice([0.0, 1.0], len(k)))
    yield "ulp", v
    v = base * (1 + 0.3 * np.sin(np.arange(L) / 900.0))          # long rises: pieces that span many workers' chunks
    yield "long_rises", v


@pytest.mark.parametrize("L", [6319, 6320, 6321, 20000, 49851, 50000])
def test_segmented_antitonic_regression_on_long_grids(L, harness):
    from sklearn.isotonic import IsotonicRegression
    rng = np.random.default_rng(L)
    for name, v in _antitonic_cases(L, rng):
        v = np.ascontiguousarray(v, dtype=np.float64)
        ref = IsotonicRegression(increasing=False).fit_transform(np.arange(len(v)), v)
        for nt in (128, 7, 1):
            out = np.full(len(v), -1.0)
            harness.th_antitonic_segmented(_p(v), len(v), nt, _p(out))
            assert np.array_equal(out, ref), (name, nt)


# ------------------------------------------------------------------------------------------------ equal-occupancy binning
def _equal_occupancy(harness, poss, obs, S, n_bins, R, min_dist, max_dist, max_out):
    nk = len(poss)
    x = np.zeros(max_out)
    y = np.zeros(max_out)
    bok = np.zeros(nk, np.int32)
    n = ctypes.c_int()
    st = harness.th_equal_occupancy(_p(poss, ctypes.c_int64), _p(obs, ctypes.c_int64), nk, ctypes.c_int64(S), n_bins,
                                    ctypes.c_int64(R), ctypes.c_int64(min_dist), ctypes.c_int64(max_dist), _p(x), _p(y),
                                    max_out, _p(bok, ctypes.c_int32), ctypes.byref(n))
    return st, x[:n.value], y[:n.value], bok


@pytest.mark.parametrize("nkeys", [8362, 8363, 25000, 49851])
@pytest.mark.parametrize("limits", ["default", "min_dist", "max_dist", "tiny_S"])
def test_equal_occupancy_on_long_tables_is_bit_identical_to_the_oracle(nkeys, limits, harness):
    from oracle import fithic_oracle as fo
    R, n_bins = 5000, 100
    min_dist, max_dist, S_extra = -1, -1, 77
    if limits == "min_dist":
        min_dist = 37 * R + 1
    elif limits == "max_dist":
        max_dist = (nkeys // 3) * R - 7
    poss, obs, S = synthetic_table(nkeys, nkeys + len(limits), chroms=3, S_extra=S_extra)
    if limits == "tiny_S":                                      # desired == 0: every in-range key closes a bin
        obs = np.zeros(nkeys, np.int64)
        obs[[3, 50]] = [20, 9]
        S = 29
    st, x, y, bok = _equal_occupancy(harness, poss, obs, S, n_bins, R, min_dist, max_dist, nkeys)
    assert st == 0
    ox, oy, _, obk = fo.calculate_probabilities(poss, obs, S, n_bins, R, min_dist, max_dist)
    assert len(x) == len(ox) and np.array_equal(x, ox) and np.array_equal(y, oy)
    assert np.array_equal(bok, obk)
    if limits == "tiny_S":
        assert len(x) == nkeys - 48                             # keys 1..3 and 4..50 close one bin each, the rest one per key
    else:
        assert 85 <= len(x) <= 100
    if limits == "max_dist":
        assert (bok[max_dist // R + 1:] == -1).all()
    if limits == "min_dist":
        assert (bok[:38] == -1).all() and bok[38] == 0
