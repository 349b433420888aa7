"""Shared helpers for the parity tests (tests only)."""
import os

import numpy as np

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
PASS_CASES = ["pass_bias_dense", "pass_nobias_sparse", "pass_messy"]


def load_golden(name):
    g = np.load(os.path.join(GOLDEN, name + ".npz"))
    return {k: g[k] for k in g.files}


def golden_bias_dict(g):
    from oracle import fithic_oracle as fo
    if not bool(g["has_bias"]):
        return None
    return fo.read_bias_arrays(g["bias_chrom"], g["bias_mid"], g["bias_val"])[0]


def log10_close(a, b, tol):
    """|log10 a - log10 b| <= tol where both > 0; exact match where either is 0 or 1."""
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    pos = (a > 0) & (b > 0)
    bad = np.zeros(a.shape, bool)
    with np.errstate(divide="ignore", invalid="ignore"):
        bad[pos] = np.abs(np.log10(a[pos]) - np.log10(b[pos])) > tol
    bad[~pos] = a[~pos] != b[~pos]
    return not bad.any(), int(bad.sum())


def truth(c, n, q):
    """P(X >= c), X ~ Binomial(n, q), in 60-digit arithmetic (mpmath): the value bdtrc(c-1, n, q) approximates.
    For 1 <= c <= n and 0 < q < 1; returns an mpmath number."""
    import mpmath as mp
    with mp.workdps(60):
        qq = mp.mpf(float(q))
        lp = mp.loggamma(n + 1) - mp.loggamma(c + 1) - mp.loggamma(n - c + 1) + c * mp.log(qq) + (n - c) * mp.log(1 - qq)
        qr = qq / (1 - qq)
        if c >= (n + 1) * qq:
            term = mp.mpf(1); s = mp.mpf(1); j = c
            while j < n:
                term *= mp.mpf(n - j) / (j + 1) * qr; s += term; j += 1
                if term < mp.mpf(10) ** -45 * s:
                    break
            return mp.exp(lp) * s
        term = mp.mpf(c) / ((n - c + 1) * qr); s = term; j = c - 1
        while j > 0:
            term *= mp.mpf(j) / ((n - j + 1) * qr); s += term; j -= 1
            if term < mp.mpf(10) ** -45 * s:
                break
        return 1 - mp.exp(lp) * s


def score_table(torch, priors, counts, S):
    """Drive the general K4 kernel (bbk_pvalues) directly: record i looks up priors[i] (mid1 = 0, mid2 = i, resolution 1)."""
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
