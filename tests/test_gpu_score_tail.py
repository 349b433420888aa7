"""The streaming K4 (bbk_score_pairs + the patch pass bbk_score_deferred) against 60-digit binomial tails at chosen
(count, prior, S), called through the C ABI without K1 or the fit: a hand-built BbkFitResult and a prior table in place of
the spline, so that every row scores exactly the (count, prior, S) the test picked.

include/bbk.h promises p = bdtrc(count-1, S, prior) for every row, and pvalue_tiles.inl that p is a function of
(count, prior, S) whatever the tiling.  The synthetic Hi-C workloads of the pass-level tests never come near the streaming
kernel's own thresholds (the lean lower-tail form up to count 64, priors below 2^-10, the 1e-4 floor of the lower tail, the
count-1 series, the -708 clamp of its exponential, the all-deferred path below S = 64), so the grids here are built around
them.  Run on the B200 box with `pytest -m gpu`.
"""
import ctypes

import numpy as np
import pytest

from helpers import score_table, truth

pytestmark = pytest.mark.gpu

P_TOL_TRUTH = 1e-9                 # |delta log10 p| against the 60-digit value (as in test_gpu_parity.py)
DEEP = 1e-290                      # below this the truth only bounds p: 0 <= p <= 1e-280
R = 2                              # resolution of the harness: row i of a table reads entry idx[i] (mid2 = idx * R)
LOW_C_MAX = 64                     # pvalue_tiles.inl: counts the lean lower-tail form takes
LEAN_MAX_PRIOR = 2.0 ** -10        # ... and priors (0, 2^-10)
LOWER_MIN_P = 1e-4                 # ... and lower-tail results from here up
SMALL_P = 2.0 ** -5                # BBK_SMALL_P: rows below it are q-value candidates
EXACT_OFFSET = 24                  # byte offset of BbkScoreState.exact

S_GRID = [64, 65, 100, 1000, 213498, 5 * 10**7, 1234567891, 2**31 - 1, 2**31, 4 * 10**9, 10**10]
COUNTS = [1, 2, 3, 7, 8, 9, 10, 31, 32, 33, 63, 64, 65, 66]
BIG_COUNTS = [100, 257, 1000, 4000]
FAR_S = [2**31 - 1, 4 * 10**9, 10**10]
# rows where the lean form's clamped exponential, e^-708 times a lower-tail sum of ~(Sq)^(c-1)/(c-1)!, is no longer
# negligible: the true p is 1.0
FAR_KNOWN = [(2**31 - 1, 64, 8.5819e-4), (4 * 10**9, 63, 5.4457e-4), (10**10, 64, 1.8458e-4), (2**31 - 1, 64, 7.5e-4)]


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    assert torch.cuda.is_available()
    return torch


# ---------------------------------------------------------------------------------------------------------- the harness
class Scored(object):
    """What one streaming run leaves.  p / q: per input row; p_rows / q_rows: every rank-local row (padding included);
    row_of: the rank-local row of each input row."""


def bias_tables(torch, L, first=1.0, rest=1.0):
    """One chromosome's bias table over loci 0, R, .., (L-1) R: `first` at locus 0 (every row's mid1), `rest` elsewhere.
    Powers of two with first * rest == 1 keep every prior (but entry 0's) exactly the table value."""
    from blueberry_b200.engine import BiasTables
    v = np.full(L, float(rest))
    v[0] = first
    return BiasTables([v], [0], torch.device("cuda:0"), step=0)


def stream_score(torch, table, idx, counts, S, sizes=None, exact=False, bias=None):
    """Score rows (idx[i], counts[i]) through bbk_score_begin / bbk_score_guard / bbk_score_pairs (once per shard) /
    bbk_score_deferred, as GenomePass._score does: row i has mid1 = 0, mid2 = idx[i] * R, so it reads table[idx[i]]
    (idx < 0: mid2 < mid1, idx >= len(table): past max_dist - both out of range).  sizes: shard sizes (default one shard),
    laid out by distributed.layout_rows.  exact: raise BbkScoreState.exact after the guard, as GenomePass.force_exact."""
    from blueberry_b200 import _lib
    from blueberry_b200.distributed import layout_rows
    lib = _lib.load()
    dev = torch.device("cuda:0")
    table = np.asarray(table, dtype=np.float64)
    idx = np.asarray(idx, dtype=np.int64)
    counts = np.asarray(counts, dtype=np.int64)
    n, L = len(idx), len(table)
    sizes = [n] if sizes is None else list(sizes)
    assert sum(sizes) == n
    starts, rows = layout_rows(sizes)
    m = max(rows, 4)
    row_of = np.concatenate([s + np.arange(k) for s, k in zip(starts, sizes)]).astype(np.int64) if n else np.zeros(0, np.int64)
    mid1 = np.zeros(m, np.int32)
    mid2 = np.zeros(m, np.int32)
    cnt = np.zeros(m, np.int32)
    mid1[row_of] = np.where(idx < 0, R, 0)
    mid2[row_of] = np.where(idx < 0, 0, idx * R)
    cnt[row_of] = counts
    d_mid1, d_mid2, d_cnt = (torch.from_numpy(a).to(dev) for a in (mid1, mid2, cnt))
    fr = _lib.FitResult(status=0, n_out=100, k0=0, L=L, n_knots=8, ier=0, S=int(S), min_x=0.0, max_x=float((L - 1) * R),
                        residual=0.0, fp=0.0, smoothing=0.0)
    fit = torch.frombuffer(bytearray(bytes(fr)), dtype=torch.uint8).to(dev)
    spline = torch.from_numpy(table).to(dev)
    # every real row starts as a sentinel that no result can be; the padding rows hold NaN, as GenomePass.attach leaves them
    p0 = np.full(m, np.nan)
    p0[row_of] = -7.0
    p = torch.from_numpy(p0).to(dev)
    q = torch.from_numpy(p0.copy()).to(dev)
    hist = torch.full((_lib.PHIST_LEN,), -1, dtype=torch.int64, device=dev)
    state = torch.full((ctypes.sizeof(_lib.ScoreState),), 0xAB, dtype=torch.uint8, device=dev)
    cap = max(n, 1)
    l_row = torch.full((cap,), -1, dtype=torch.int32, device=dev)
    l_cnt = torch.full((cap,), -1, dtype=torch.int32, device=dev)
    l_prior = torch.full((cap,), -7.0, dtype=torch.float64, device=dev)
    deferred = _lib.DeferredList(l_row.data_ptr(), l_cnt.data_ptr(), l_prior.data_ptr(), cap)
    c_keys = torch.full((cap,), -1, dtype=torch.int64, device=dev)
    c_rows = torch.full((cap,), -1, dtype=torch.int32, device=dev)
    cands = _lib.Candidates(c_keys.data_ptr(), c_rows.data_ptr(), cap)
    b_struct = ctypes.byref(bias.struct) if bias is not None else None
    b_flags = _lib.ptr(bias.flags) if bias is not None else None
    st = _lib.stream_ptr()
    _lib.check(lib.bbk_score_begin(_lib.ptr(state), _lib.ptr(hist), st), "bbk_score_begin")
    _lib.check(lib.bbk_score_guard(_lib.ptr(fit), _lib.ptr(spline), _lib.ptr(state), st), "bbk_score_guard")
    if exact:
        state[EXACT_OFFSET:EXACT_OFFSET + 4] = torch.tensor([1, 0, 0, 0], dtype=torch.uint8, device=dev)
    for s, k in zip(starts, sizes):
        if k == 0:
            continue
        _lib.check(lib.bbk_score_pairs(_lib.ptr(d_mid1[s:]), _lib.ptr(d_mid2[s:]), _lib.ptr(d_cnt[s:]), k, 0, R, 0, (L - 1) * R,
                                       _lib.ptr(fit), _lib.ptr(spline), b_struct, b_flags, s, _lib.ptr(p), _lib.ptr(q),
                                       _lib.ptr(hist), ctypes.byref(cands), ctypes.byref(deferred), _lib.ptr(state), st),
                   "bbk_score_pairs")
    _lib.check(lib.bbk_score_deferred(ctypes.byref(deferred), _lib.ptr(fit), _lib.ptr(p), _lib.ptr(q), _lib.ptr(hist),
                                      ctypes.byref(cands), _lib.ptr(state), st), "bbk_score_deferred")
    torch.cuda.synchronize()
    out = Scored()
    out.S, out.n, out.rows, out.row_of = int(S), n, rows, row_of
    out.p_rows = p.cpu().numpy()[:rows]
    out.q_rows = q.cpu().numpy()[:rows]
    out.p, out.q = out.p_rows[row_of], out.q_rows[row_of]
    out.hist = hist.cpu().numpy()
    out.state = _lib.ScoreState.from_buffer_copy(state.cpu().numpy().tobytes())
    nl = min(int(out.state.n_list), cap)
    out.d_row, out.d_cnt, out.d_prior = l_row.cpu().numpy()[:nl], l_cnt.cpu().numpy()[:nl], l_prior.cpu().numpy()[:nl]
    nc = min(int(out.state.n_cand), cap)
    out.c_key, out.c_row = c_keys.cpu().numpy()[:nc], c_rows.cpu().numpy()[:nc]
    # the prior each in-range row must see: table value times the two bias values (NaN / absent locus = 1.0)
    inr = (idx >= 0) & (idx < L)
    prior = np.full(n, np.nan)
    prior[inr] = table[idx[inr]]
    if bias is not None:
        bv = bias.bias.cpu().numpy()
        look = lambda loc: np.where((loc < len(bv)) & ~np.isnan(bv[np.minimum(loc, len(bv) - 1)]), bv[np.minimum(loc, len(bv) - 1)], 1.0)
        prior[inr] = prior[inr] * (look(np.zeros(int(inr.sum()), np.int64)) * look(idx[inr]))
    out.counts, out.prior, out.in_range = counts, prior, inr
    out.exact_asked = bool(exact)
    return out


# ------------------------------------------------------------------------------------------------------- the reference
def lean_u(q, S):
    """u = S ln(1 - q) as the lean form computes it (the same series for ln(1 - q)), in float64."""
    q = np.asarray(q, dtype=np.float64)
    return float(S) * (-q * (1.0 + q * (0.5 + q * (1.0 / 3.0 + q * (0.25 + q * (0.2 + q * (1.0 / 6.0)))))))


def reference(counts, priors, S):
    """bdtrc(count-1, S, prior)'s case analysis, 60-digit arithmetic where it computes.  Returns (want, arith, lg, deep):
    want the exact result of the decided rows (NaN / 0.0 / 1.0), arith the rows with a tail, lg their log10 truth, deep
    the rows whose truth is below DEEP."""
    import mpmath as mp
    n = len(counts)
    want = np.full(n, np.nan)
    arith = np.zeros(n, bool)
    deep = np.zeros(n, bool)
    lg = np.zeros(n)
    tv_f = np.full(n, np.nan)
    floor = mp.mpf(DEEP)
    for i in range(n):
        c, q = int(counts[i]), float(priors[i])
        if not (0.0 <= q <= 1.0):
            continue                                   # NaN, checked before the count
        if c <= 0:
            want[i] = 1.0
        elif c - 1 > S:
            continue                                   # NaN (fithic.py:434 drops the row)
        elif c - 1 == S:
            want[i] = 0.0
        elif q == 0.0:
            want[i] = -0.0 if c == 1 and np.signbit(q) else 0.0     # count 1: -expm1(S log1p(-q)), the sign of -q
        elif q == 1.0:
            want[i] = 1.0
        else:
            tv = truth(c, S, q)
            arith[i] = True
            tv_f[i] = float(tv)
            if tv < floor:
                deep[i] = True
            else:
                lg[i] = float(mp.log10(tv))
    return want, arith, lg, deep, tv_f


def mismatches(got, ref):
    """Indices of rows where `got` misses the reference: decided rows bit for bit, the rest within P_TOL_TRUTH in log10."""
    want, arith, lg, deep, _ = ref
    got = np.asarray(got, dtype=np.float64)
    bad = np.zeros(len(got), bool)
    dec = ~arith
    bad[dec] = got[dec].view(np.int64) != want[dec].view(np.int64)
    ok = arith & ~deep
    with np.errstate(divide="ignore", invalid="ignore"):
        err = np.abs(np.log10(got[ok]) - lg[ok])
    bad[ok] = ~(err <= P_TOL_TRUTH)
    bad[deep] = ~((got[deep] >= 0.0) & (got[deep] <= 1e-280))
    return np.flatnonzero(bad)


def describe(which, idx, counts, priors, S, got, ref, limit=12):
    tv = ref[4]
    lines = ["%s, S = %d: %d rows off the 60-digit truth" % (which, S, len(idx))]
    for i in idx[:limit]:
        lines.append("  count %d prior %.17g: p = %.17g, truth %.17g" % (counts[i], priors[i], got[i], tv[i]))
    return "\n".join(lines)


# ------------------------------------------------------------------------------------------------- side-output checks
def check_side_outputs(run, p_ref=None):
    """Everything a streaming run leaves besides p must follow from the final p and the documented deferral rule.
    p_ref (optional): a reference p per input row, to bound which lean rows may have been deferred for a lower tail below
    LOWER_MIN_P; without it the run's own final p serves."""
    from blueberry_b200 import _lib
    p_rows, q_rows = run.p_rows, run.q_rows
    real = run.row_of
    pad = np.setdiff1d(np.arange(run.rows), real)
    p = p_rows[real]
    assert not (p == -7.0).any() and not (run.q == -7.0).any(), "rows left unwritten"
    assert np.isnan(p_rows[pad]).all() and np.isnan(q_rows[pad]).all(), "padding rows must stay NaN"
    st = run.state
    assert st.overflow == 0 and st.cand_overflow == 0
    assert st.exact in (0, 1) and (not run.exact_asked or st.exact == 1)
    nan, one = np.isnan(p), p == 1.0
    # q: NaN with p, 1.0 elsewhere (the q-value step fills in the candidates later)
    assert np.array_equal(np.isnan(run.q), nan) and (run.q[~nan] == 1.0).all()
    # the coarse histogram: bucket (bits >> 51) & 4095 of a p in [0, 1), p == 1.0 in slot 4096, NaN in slot 4097
    assert ((p[~nan] >= 0.0) & (p[~nan] <= 1.0)).all()
    bits = p.view(np.int64)
    h = np.zeros(_lib.PHIST_LEN, np.int64)
    h[:_lib.PHIST_BINS] = np.bincount(((bits >> 51) & 4095)[~nan & ~one], minlength=_lib.PHIST_BINS)
    h[_lib.PHIST_BINS], h[_lib.PHIST_BINS + 1] = one.sum(), nan.sum()
    assert np.array_equal(run.hist, h), "p histogram differs from the one the final p implies"
    # candidates: exactly the rows with p < 2^-5, each once, under the order-preserving key of p: IEEE bits | 2^63, or ~bits
    # for the one negative p there is (-0.0: count 1 at a prior of -0.0, as bdtrc gives it)
    with np.errstate(invalid="ignore"):
        want_c = np.sort(real[p < SMALL_P])
    assert int(st.n_cand) == len(want_c) == len(run.c_row)
    assert np.array_equal(np.sort(run.c_row.astype(np.int64)), want_c)
    cb = p_rows[run.c_row].view(np.uint64)
    key_want = np.where(cb >> np.uint64(63) != 0, ~cb, cb | np.uint64(1 << 63))
    assert np.array_equal(run.c_key.view(np.uint64), key_want)
    # the deferred list
    inv = np.full(run.rows, -1, np.int64)
    inv[real] = np.arange(run.n)
    d_in = inv[run.d_row.astype(np.int64)]
    assert (d_in >= 0).all(), "a padding row was deferred"
    assert len(np.unique(d_in)) == len(d_in) == int(st.n_list), "a row deferred twice"
    c, prior, inr, S = run.counts, run.prior, run.in_range, run.S
    assert np.array_equal(run.d_cnt.astype(np.int64), c[d_in])
    assert np.array_equal(run.d_prior.view(np.int64), prior[d_in].view(np.int64)), "stored prior is not the row's prior"
    with np.errstate(invalid="ignore"):
        valid = inr & (prior >= 0.0) & (prior <= 1.0)
        lean_prior = (prior > 0.0) & (prior < LEAN_MAX_PRIOR)
        u = lean_u(np.where(valid, prior, 0.0), S)
    must = valid & (c >= 1) & ((c > LOW_C_MAX) | ~lean_prior | (S < 64))
    lean2 = valid & (c >= 2) & (c <= LOW_C_MAX) & lean_prior & (S >= 64)
    pr = run.p if p_ref is None else np.asarray(p_ref, dtype=np.float64)
    with np.errstate(invalid="ignore"):
        must |= lean2 & ((pr < LOWER_MIN_P * (1 - 1e-6)) | (u < -708.0 * (1 + 1e-12)))
        may = must | (lean2 & ((pr < LOWER_MIN_P * (1 + 1e-6)) | (u < -708.0 * (1 - 1e-12))))
    listed = np.zeros(run.n, bool)
    listed[d_in] = True
    miss = np.flatnonzero(must & ~listed)
    extra = np.flatnonzero(listed & ~may)
    assert not len(miss), "rows the rule defers were not deferred: %s" % [(int(c[i]), prior[i]) for i in miss[:8]]
    assert not len(extra), "rows deferred against the rule: %s" % [(int(c[i]), prior[i]) for i in extra[:8]]


# ------------------------------------------------------------------------------------------------------------ grids
def _ulps(q, k):
    """q moved by k ulps."""
    out = np.float64(q)
    for _ in range(abs(k)):
        out = np.nextafter(out, np.inf if k > 0 else -np.inf)
    return float(out)


def _crossing(S, target):
    """The prior at which lean_u(prior, S) crosses `target` (< 0), to the ulp."""
    lo, hi = 0.0, 0.5
    for _ in range(2000):
        mid = 0.5 * (lo + hi)
        if mid in (lo, hi):
            break
        if lean_u(mid, S) > target:
            lo = mid
        else:
            hi = mid
    return hi


def _prior_for_p(c, S, p):
    """The prior at which P(X >= c) = p (scipy.stats.binom, double-precision n)."""
    from scipy.optimize import brentq
    from scipy.stats import binom
    f = lambda lq: np.log(binom.sf(c - 1, S, np.exp(lq))) - np.log(p)
    return float(np.exp(brentq(f, np.log(1e-3 * c / S), np.log1p(-1e-9), xtol=1e-15, rtol=1e-15)))


def grid(S):
    """(counts, priors) around every threshold of the lean form at one S."""
    base = list(np.geomspace(1e-12, LEAN_MAX_PRIOR, 13)[:-1])
    base += [_ulps(LEAN_MAX_PRIOR, k) for k in (-2, -1, 0, 1, 2)]
    tiny = [_ulps(_crossing(S, -0.0078125), k) for k in range(-3, 4)]          # the count-1 series switch
    rows = [(c, q) for c in COUNTS for q in base]
    rows += [(c, q) for c in (1, 2, 3) for q in tiny]
    q708 = _crossing(S, -708.0)
    if q708 < 0.25:
        rows += [(c, _ulps(q708, k)) for c in COUNTS for k in range(-3, 4)]   # the clamp of the exponential
    for c in COUNTS:                                                              # the lower tail's 1e-4 floor, both sides
        if 2 <= c <= S:
            q1 = _prior_for_p(c, S, LOWER_MIN_P)
            rows += [(c, q1 * (1 + f)) for f in (-1e-6, -1e-9, 0.0, 1e-9, 1e-6)]
    for c in BIG_COUNTS:                                                          # the patch pass' upper sum
        rows += [(c, min(c * f / S, 0.75)) for f in (0.25, 0.8, 1.0, 1.25, 3.0)]
        rows.append((c, 2.0 ** -11))
    counts = np.array([r[0] for r in rows], np.int64)
    priors = np.array([r[1] for r in rows], np.float64)
    return counts, priors


def far_grid(S):
    """counts 50..64 at priors [1e-5, 2^-10): far below the mean, where the clamped e^-708 shows."""
    qs = list(np.geomspace(1e-5, LEAN_MAX_PRIOR, 25)[:-1]) + [_ulps(LEAN_MAX_PRIOR, -1)]
    rows = [(c, q) for c in range(50, 65) for q in qs] + [(c, q) for s, c, q in FAR_KNOWN if s == S]
    return np.array([r[0] for r in rows], np.int64), np.array([r[1] for r in rows], np.float64)


def _against_truth(torch, S, counts, priors):
    n = len(counts)
    ref = reference(counts, priors, S)
    # with a bias table: locus 0 (every row's mid1) carries 2.0, the others 0.5, so b1 * b2 == 1 and row i (table entry
    # i + 1) still scores priors[i]
    runs = [("streaming", stream_score(torch, priors, np.arange(n), counts, S)),
            ("streaming with bias", stream_score(torch, np.concatenate([[0.0], priors]), np.arange(1, n + 1), counts, S,
                                                 bias=bias_tables(torch, n + 1, 2.0, 0.5)))]
    general = score_table(torch, priors, counts, S)
    failures = []
    bad = mismatches(general, ref)
    if len(bad):
        failures.append(describe("general kernel", bad, counts, priors, S, general, ref))
    for name, run in runs:
        bad = mismatches(run.p, ref)
        if len(bad):
            failures.append(describe(name, bad, counts, priors, S, run.p, ref))
    assert not failures, "\n".join(failures)
    for name, run in runs:
        assert np.array_equal(run.prior.view(np.int64), priors.view(np.int64))
        check_side_outputs(run, p_ref=np.where(ref[1], ref[4], run.p))
        # what bdtrc decides without arithmetic (NaN, 0.0) comes out the same from both kernels
        assert np.array_equal(np.isnan(run.p), np.isnan(general)), name
        assert np.array_equal(run.p == 0.0, general == 0.0), name
        # a deferred row goes through the general kernel's own tail code: the same bits
        d = np.zeros(n, bool)
        d[np.searchsorted(run.row_of, run.d_row.astype(np.int64))] = True
        assert np.array_equal(run.p[d].view(np.int64), general[d].view(np.int64)), name + ": deferred rows differ from bbk_pvalues"
    lean = (counts <= LOW_C_MAX) & (priors > 0) & (priors < LEAN_MAX_PRIOR)
    worst = np.abs(np.log10(runs[0][1].p[ref[1] & ~ref[3] & lean]) - ref[2][ref[1] & ~ref[3] & lean]).max() if (ref[1] & ~ref[3] & lean).any() else 0.0
    print("S=%d: %d rows, %d lean; worst lean |dlog10 p| %.3g" % (S, n, int(lean.sum()), worst))


# ------------------------------------------------------------------------------------------------------------ tests
@pytest.mark.parametrize("S", S_GRID)
def test_stream_against_60_digit_truth(S, torch_cuda):
    """Every threshold of the lean form and the patch pass at one S: the streaming path (with and without a bias table)
    and the general kernel against the 60-digit tail."""
    counts, priors = grid(S)
    _against_truth(torch_cuda, S, counts, priors)


@pytest.mark.parametrize("S", FAR_S)
def test_stream_far_below_the_mean(S, torch_cuda):
    """Counts 50..64 with means S q up to 10^7: the true p is 1.0; a lean form that let the clamped e^-708 decide
    returned p ~ 1e-3 here."""
    counts, priors = far_grid(S)
    _against_truth(torch_cuda, S, counts, priors)


EDGE_PRIORS = [-0.5, 1.5, 0.5, 0.0, 1.0, np.nan, 0.02, 0.005, 0.3, -0.1, -0.0, 1e-3, LEAN_MAX_PRIOR, _ulps(LEAN_MAX_PRIOR, -1),
               1e-7, 0.0625, np.inf, -np.inf, 5e-324]


@pytest.mark.parametrize("S", [1, 2, 63, 64, 100])
@pytest.mark.parametrize("mode", ["speculative", "exact"])
def test_stream_edge_semantics_match_bdtrc(S, mode, torch_cuda):
    """bdtrc's edge cases through the streaming path: NaN for a prior outside [0, 1] (before the count), 1.0 for
    count <= 0, NaN for count-1 > S, 0.0 for count-1 == S, 0 / 1 at prior 0 / 1; S < 64 defers every row.  Speculative
    mode needs a table the guard passes (priors in [0, 1/16]); exact mode takes every prior.  Out-of-range rows are NaN."""
    import scipy.special as sc
    pri = [q for q in EDGE_PRIORS if mode == "exact" or 0.0 <= q <= 0.0625]
    cnts = sorted({-3, 0, 1, 2, 3, 5, 7, 64, 65, 102, max(S - 1, 1), S, S + 1, S + 2})
    counts = np.array([c for q in pri for c in cnts] + [0, 3, 0, 3], np.int64)
    idx = np.array([i for i in range(len(pri)) for _ in cnts] + [-1, -1, len(pri), len(pri) + 5], np.int64)
    run = stream_score(torch_cuda, pri, idx, counts, S, exact=mode == "exact")
    assert run.state.exact == (1 if mode == "exact" else 0)
    check_side_outputs(run)
    inr = run.in_range
    assert np.isnan(run.p[~inr]).all()
    prior = run.prior[inr]
    with np.errstate(all="ignore"):
        want = sc.bdtrc((counts[inr] - 1).astype(np.float64), np.int64(S), prior)
    want = np.where(want <= 1, want, np.nan)                        # fithic.py:434 drops the row
    got = run.p[inr]
    assert np.array_equal(np.isnan(got), np.isnan(want))
    ref = reference(counts[inr], prior, S)
    bad = mismatches(got, ref)
    assert not len(bad), describe("streaming (%s)" % mode, bad, counts[inr], prior, S, got, ref)
    big = ~np.isnan(want) & (want >= DEEP) & (got > 0)
    assert np.abs(np.log10(got[big]) - np.log10(want[big])).max() <= P_TOL_TRUTH


def _layout_rows(rng):
    """A mixed table: count 0 rows, every lean class, deferred counts, priors up to the guard's 1/16, the far-below block,
    and out-of-range rows."""
    n_tab = 3000
    table = np.concatenate([10 ** rng.uniform(-12, np.log10(LEAN_MAX_PRIOR), n_tab - 300),
                            rng.uniform(LEAN_MAX_PRIOR, 0.0625, 200), rng.uniform(1e-5, LEAN_MAX_PRIOR, 100)])
    n = 20000
    idx = rng.integers(0, n_tab, n)
    kind = rng.random(n)
    counts = np.where(kind < 0.3, 0, np.where(kind < 0.6, rng.integers(1, 9, n), np.where(kind < 0.85, rng.integers(9, 65, n),
                      rng.integers(65, 3000, n))))
    far = rng.random(n) < 0.05
    idx[far] = rng.integers(n_tab - 100, n_tab, int(far.sum()))
    counts[far] = rng.integers(50, 65, int(far.sum()))
    oor = rng.random(n) < 0.01
    idx[oor] = np.where(rng.random(int(oor.sum())) < 0.5, -1, n_tab + 3)
    counts[rng.random(n) < 0.01] = -2
    return table, idx, counts


@pytest.mark.parametrize("S", [1000, 1234567891, 10**10])
def test_stream_p_depends_on_count_prior_and_S_only(S, torch_cuda):
    """The same rows in grid order, permuted, sorted by count, and cut into shards of 1, 3, 5, 255, 256, 257, 4099 and
    the rest, each with and without a bias table of ones: every row gets the same p bits (the explicit roundings of the
    term loop and the warp-uniform cmax_s / cmax_l switch must not make a row's p depend on its neighbours)."""
    torch = torch_cuda
    rng = np.random.default_rng(S % 10007)
    table, idx, counts = _layout_rows(rng)
    n = len(idx)
    perm = rng.permutation(n)
    srt = np.argsort(counts, kind="stable")
    cut = [1, 3, 5, 255, 256, 257, 4099]
    layouts = {"grid": (np.arange(n), None), "permuted": (perm, None), "by count": (srt, None),
               "shards": (np.arange(n), cut + [n - sum(cut)])}
    ones = bias_tables(torch, len(table) + 8)
    base = None
    for name, (order, sizes) in layouts.items():
        for b in (None, ones):
            run = stream_score(torch, table, idx[order], counts[order], S, sizes=sizes, bias=b)
            check_side_outputs(run)
            p = np.empty(n)
            p[order] = run.p
            if base is None:
                base = p
                continue
            diff = np.flatnonzero(p.view(np.int64) != base.view(np.int64))
            assert not len(diff), "%s%s: %d rows differ from grid order, e.g. count %d table entry %d: %r vs %r" % (
                name, " with bias" if b is not None else "", len(diff), counts[diff[0]], idx[diff[0]], p[diff[0]], base[diff[0]])
