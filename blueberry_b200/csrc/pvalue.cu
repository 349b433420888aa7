// pvalue.cu - K4: per-pair binomial survival p-values (reference: fit_spline scoring loop,
// fithic.py:413-435):   p = scipy.special.bdtrc(count-1, S, newSplineY[i] * (bias1*bias2)).
//
// Fused elementwise kernel, 12 B/pair in (int32 mid1, mid2, count), 8 B/pair out (float64 p):
//   load (128-bit, streaming) -> distance -> spline index (closed form of the reference's bisect)
//   -> bias gathers (L2-resident tables) -> prior -> log-space binomial tail -> store (128-bit).
//
// The FP64 special-function work is what threatens the HBM roofline here, and it is very uneven:
// most records have count 0 (p = 1, no arithmetic), some have count 1 (closed form), the rest need a
// tail sum whose length grows towards the diagonal (hundreds of terms at d ~ 0).  Evaluated in place,
// every warp would pay for the union of all branches.  So every WARP works on tiles of 256 records
// in phases, with no CTA barrier:
//   1. classify: each lane resolves the priors of its records; trivial results go straight to the
//      tile's result slots in shared memory, records that need arithmetic are appended to two dense
//      warp-private work lists (count == 1 from the front, count >= 2 from the back; ballot + popc);
//   2. solve: the warp runs down each list with all lanes on the same branch.  A tail sum is a small
//      resumable state: every lane advances its own sum 16 terms between two convergence checks
//      until the whole round of 32 records is done (neighbouring records have similar lengths, so
//      rounds are homogeneous);
//   3. each lane reads its 8 results back and issues coalesced 128-bit streaming stores.
// The hot loop is kept small (tables and rare branches live in separate functions/kernels): with
// autonomous warps the instruction cache is the first thing to overflow.
//
// The tail P(X >= c), X ~ Binomial(S, q), is the regularised incomplete beta I_q(c, S-c+1) that
// cephes' bdtrc evaluates.  Here: pmf(c) * (1 + r_{c+1} + r_{c+1} r_{c+2} + ...), always the upper tail
// (a count more than 9 sigma below the mean gives p = 1.0 directly).  ln pmf(c) = c ln(Sq) - ln c! + sum_{i<c} ln(1-i/S)
// + (S-c) ln(1-q), with the two small logarithms expanded in series (exact to < 1e-12 for the c/S the
// fast path admits) and ln c!, 1/j from shared-memory tables; outside that range the saddle-point
// form (Stirling error + deviance terms; C. Loader, "Fast and accurate computation of binomial
// probabilities", 2000) takes over.  Against 60-digit arithmetic this is good to ~1e-12 in log10 p;
// cephes itself is only good to ~3e-6 at S ~ 1e9 (DESIGN.md), which is what bounds the parity tolerance.
// bdtrc's edge semantics are kept exactly: NaN for a prior outside [0,1] or NaN (checked BEFORE the
// count, so a count of 0 with a negative prior is dropped too), 1.0 for count <= 0, NaN for
// count-1 > S, 0.0 for count-1 == S, the count == 1 closed form, 0 / 1 at q == 0 / 1.
#include <mutex>
#include "common.cuh"

namespace {

constexpr int PV_THREADS = 256;
constexpr int PV_WARPS = PV_THREADS / 32;
constexpr int RCP_TAB = 1024;        // 1/j for j < RCP_TAB
constexpr int LF_TAB = 256;          // ln j! for j < LF_TAB
constexpr double TAIL_EPS = 2e-12;
constexpr int TERM_BLOCK = 16;       // terms summed between two convergence checks (cfg2: 8 -> 1.69 ms, 16 -> 1.64 ms, 32 -> 1.67 ms)
constexpr double LN_2PI = 1.8378770664093454836;

// mathematical constants, filled once per device (pv_tables_kernel): 1/j and ln j!
__device__ double g_rcp[RCP_TAB];
__device__ double g_lfact[LF_TAB];

__global__ void pv_tables_kernel() {
    int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j < RCP_TAB) g_rcp[j] = j ? 1.0 / (double)j : 0.0;
    if (j < LF_TAB) g_lfact[j] = lgamma((double)j + 1.0);
}

__device__ __constant__ double c_stirl[16] = {
    0.0, 0.08106146679532726, 0.04134069595540929, 0.02767792568499834, 0.02079067210376509,
    0.01664469118982119, 0.01387612882307075, 0.01189670994589177, 0.01041126526197209,
    0.009255462182712733, 0.008330563433362871, 0.007573675487951841, 0.006942840107209530,
    0.006408994188004207, 0.005951370112758848, 0.005554733551962801};

// ln(n!) - [n ln n - n + 0.5 ln(2 pi n)]
__device__ __forceinline__ double stirlerr(double n) {
    if (n <= 15.0) return c_stirl[(int)n];
    const double S0 = 1.0 / 12.0, S1 = 1.0 / 360.0, S2 = 1.0 / 1260.0, S3 = 1.0 / 1680.0, S4 = 1.0 / 1188.0;
    double rn = 1.0 / n, rnn = rn * rn;
    if (n > 500.0) return (S0 - S1 * rnn) * rn;
    if (n > 80.0) return (S0 - (S1 - S2 * rnn) * rnn) * rn;
    if (n > 35.0) return (S0 - (S1 - (S2 - S3 * rnn) * rnn) * rnn) * rn;
    return (S0 - (S1 - (S2 - (S3 - S4 * rnn) * rnn) * rnn) * rnn) * rn;
}

// x ln(x/M) + M - x, without cancellation when x ~ M
__device__ __forceinline__ double bd0(double x, double M) {
    double diff = x - M;
    if (fabs(diff) < 0.1 * (x + M)) {
        double v = diff / (x + M);
        double s = diff * v;
        double ej = 2.0 * x * v;
        double v2 = v * v;
        for (int j = 1; j < 1000; ++j) {
            ej *= v2;
            double s1 = s + ej / (double)(2 * j + 1);
            if (s1 == s) return s1;
            s = s1;
        }
        return s;
    }
    return x * log(x / M) + M - x;
}

// General path (any S, any 2 <= c <= S, 0 < q < 1): saddle-point pmf + serial tail sum.  Rare: counts
// beyond the fast path's range, or small S.  Kept out of line so it costs the hot loop one call.
__device__ __noinline__ double tail_general(int c, long long S, double q) {
    const double dn = (double)S, dc = (double)c;
    if ((long long)c == S) return exp(dn * log(q));              // I_q(S, 1) = q^S
    const double mu = dn * q, nmc = dn - dc;
    double lc = stirlerr(dn) - stirlerr(dc) - stirlerr(nmc) - bd0(dc, mu) - bd0(nmc, dn * (1.0 - q));
    double lf = LN_2PI + log(dc) + log1p(-dc / dn);
    double lp = lc - 0.5 * lf;                                   // ln pmf(c)
    const double qr = q / (1.0 - q);
    const double eps = 5.7e-14;
    if (dc >= (dn + 1.0) * q) {
        double term = 1.0, sum = 1.0, dj = dc, rem = nmc;
        while (rem > 0.0) {
            term *= rem * qr / (dj + 1.0);
            sum += term;
            dj += 1.0;
            rem -= 1.0;
            if (term < eps * sum) break;
        }
        if (lp < -690.0) return exp(lp + log(sum));              // keep the denormal range reachable
        return exp(lp) * sum;
    }
    const double iqr = (1.0 - q) / q;
    double term = dc * iqr / (nmc + 1.0), sum = term, dj = dc - 1.0;
    while (dj > 0.0) {
        term *= dj * iqr / (dn - dj + 1.0);
        sum += term;
        dj -= 1.0;
        if (term < eps * sum) break;
    }
    return 1.0 - exp(lp) * sum;
}

// rare branches of the fast path, out of line
__device__ __noinline__ double log1m_big(double q) { return log1p(-q); }
__device__ __noinline__ double lnfact_big(double dc) { return dc * log(dc) - dc + 0.5 * (LN_2PI + log(dc)) + stirlerr(dc); }
__device__ __noinline__ double exp_deep(double lp, double sum) { return exp(lp + log(sum)); }

// ln(1 - q)
__device__ __forceinline__ double log1m(double q) {
    if (q < 9.765625e-4)
        return -q * (1.0 + q * (0.5 + q * (1.0 / 3.0 + q * (0.25 + q * (0.2 + q * (1.0 / 6.0))))));
    return log1m_big(q);
}

struct TailConst {      // per-launch constants (functions of S only)
    double dn;          // (double) S
    double inv_n;       // 1 / S
    double c_max;       // the series form of ln pmf needs c < c_max (= 1e-4 S: 1/(S-j) expands) ...
    double c5_max;      // ... and c^5 < c5_max (= 2e-11 S^4: sum ln(1-i/S) truncated after the cubic term)
};

// The tail sum as a resumable state.  Always the UPPER tail, P(X >= c) = pmf(c) (1 + r(c+1) + r(c+1) r(c+2) + ...) with
// r(j) = pmf(j)/pmf(j-1) = (S - j + 1) q / (j (1 - q)): below the mode the terms first rise (by at most pmf(mode)/pmf(c)),
// the sum comes out as ~1/pmf(c) and p as ~1.  (An earlier version summed the lower tail for c below the mode and returned
// 1 - sum; the two kinds of lanes then ran two different loops one after the other in every round - 8 % of K4's
// instructions at 4 of 32 lanes.  One loop for every lane: 1.87 -> 1.70 ms on cfg2.)
struct TailState {
    double lp;      // ln pmf(c)
    double term;    // last term added, relative to pmf(c)
    double sum;     // sum of the terms so far, relative to pmf(c)
    double a;       // (S - j + 1) q/(1-q) for the next index j
    double step;    // q/(1-q)          (a moves by -step per term)
    int j;          // next index: c+1, c+2, ...
};

__device__ __forceinline__ bool fast_ok(int c, const TailConst& K) {
    double dc = (double)c, c2 = dc * dc;
    return dc < K.c_max && c2 * c2 * dc < K.c5_max;
}

__device__ __forceinline__ void tail_setup(int c, double q, const TailConst& K, const double* __restrict__ lfact, TailState& T) {
    const double dc = (double)c, dn = K.dn, inv_n = K.inv_n;
    const double mu = dn * q;
    const double s1 = 0.5 * dc * (dc - 1.0) * inv_n;
    const double A = -s1 * (1.0 + inv_n * ((2.0 * dc - 1.0) * (1.0 / 6.0) + s1 * (1.0 / 3.0)));   // sum_{i<c} ln(1 - i/S)
    const double lnfact = c < LF_TAB ? lfact[c] : lnfact_big(dc);
    T.lp = dc * log(mu) - lnfact + A + (dn - dc) * log1m(q);
    // More than nine standard deviations below the mean 1 - p is under 1e-19 (the left tail of a binomial is lighter than
    // the normal's): p rounds to 1.0, which is what the degenerate state produces - and the terms, which would rise by
    // pmf(mode)/pmf(c), cannot overflow for the rest.
    const double gap = mu - dc - 2.0;
    const bool far_below = gap > 0.0 && gap * gap > 81.0 * mu;
    const double qr = q / (1.0 - q);
    T.term = 1.0;
    T.sum = 1.0;
    T.j = c + 1;
    T.step = qr;
    T.a = (dn - dc) * qr;
    if (far_below) { T.lp = 0.0; T.a = 0.0; }                    // exhausted at once: exp(0) * 1
}

// Up to 16 terms of the state's own series; returns true when the support is exhausted (nothing left to add).
// The per-term work is kept to the recurrence itself: the table bound and the end of the support are checked
// once per block (the slow variants handle the blocks that cross them, and stop at the end of the support).
__device__ __forceinline__ bool tail_terms16(TailState& T, const TailConst& K, const double* __restrict__ rcp) {
    if (T.j + TERM_BLOCK <= RCP_TAB && T.a > (double)TERM_BLOCK * T.step) {
        const double* r = rcp + T.j;
#pragma unroll 4
        for (int u = 0; u < TERM_BLOCK; ++u) {
            T.term *= T.a * r[u];
            T.sum += T.term;
            T.a -= T.step;
        }
        T.j += TERM_BLOCK;
        return false;
    }
#pragma unroll 1
    for (int u = 0; u < TERM_BLOCK; ++u) {
        if (!(T.a > 0.0)) return true;                           // j > S: pmf is zero from here on
        double r = T.j < RCP_TAB ? rcp[T.j] : 1.0 / (double)T.j;
        T.term *= T.a * r;
        T.sum += T.term;
        T.a -= T.step;
        T.j += 1;
    }
    return false;
}

__device__ __forceinline__ double tail_finish(double lp, double sum) {
    if (lp < -690.0) return exp_deep(lp, sum);                   // keep the denormal range reachable
    const double v = exp(lp) * sum;
    return v > 1.0 ? 1.0 : v;                                    // c far below the mode: the sum of the whole support, up to rounding
}

// Everything bdtrc decides without arithmetic.  Returns 0 when *out is final, 1 for count == 1
// (closed form), 2 for a tail sum (then 0 < q < 1 and 2 <= c <= S).  s_cap = min(S, INT_MAX).
__device__ __forceinline__ int bdtrc_class(int c, int s_cap, bool s_fits, double q, double* out) {
    // bdtrc's decisions in ITS order of precedence: !(0 <= q <= 1) -> NaN; k < 0 -> 1; n < k -> NaN; k == n -> 0; k == 0 -> the
    // closed form; q == 0 -> 0; q == 1 -> 1.  Written as selects, lowest precedence first (a later line overrides an earlier
    // one): the lanes of a warp hold every mix of these cases, and as a chain of early returns the tests ran one after the
    // other on ever fewer lanes (13 % of the kernel's instructions).
    const double qnan = __longlong_as_double(0x7ff8000000000000ll);
    const int k = c - 1;
    int cls = 2;
    double o = qnan;
    if (q == 1.0) { cls = 0; o = 1.0; }
    if (q == 0.0) { cls = 0; o = 0.0; }
    if (k == 0) cls = 1;
    if (s_fits && k == s_cap) { cls = 0; o = 0.0; }
    if (s_fits && k > s_cap) { cls = 0; o = qnan; }
    if (c <= 0) { cls = 0; o = 1.0; }
    if (!(q >= 0.0 && q <= 1.0)) { cls = 0; o = qnan; }
    *out = o;
    return cls;
}

struct PvParams {
    const int32_t* chr1;
    const int32_t* chr2;
    const int32_t* mid1;
    const int32_t* mid2;
    const int32_t* count;
    long long n_pairs;
    int shard_chrom;
    long long R, min_dist, max_dist;
    FastDiv div;
    FastDiv bdiv;        // the bias tables' grid step (the resolution unless BbkBiasTable.step says otherwise)
    const BbkFitResult* fit;
    const double* spline_y;
    const double* bias;
    const long long* chrom_base;
    const long long* mid0;
    int n_chrom;
    double* p;
    long long* p_hist;
};

struct BiasRow { long long base, nloc, mid0; unsigned long long span; };     // span = nloc * R

__device__ __forceinline__ BiasRow bias_row(const PvParams& P, int chrom) {
    BiasRow r = {0, 0, 0, 0};
    if (chrom < 0 || chrom >= P.n_chrom) return r;
    r.base = __ldg(&P.chrom_base[chrom]);
    r.nloc = __ldg(&P.chrom_base[chrom + 1]) - r.base;
    r.mid0 = __ldg(&P.mid0[chrom]);
    r.span = (unsigned long long)r.nloc * (unsigned long long)P.bdiv.R;
    return r;
}

// biasDic[chr][mid] with default 1.0 (fithic.py:418-425) on a dense per-chromosome grid
template <bool FAST>
__device__ __forceinline__ double bias_lookup(const PvParams& P, const BiasRow& row, int mid) {
    const long long off = (long long)mid - row.mid0;
    if ((unsigned long long)off >= row.span) return 1.0;          // before the table, or past its end
    unsigned idx;
    if (FAST) {
        if (off >= (1ll << 31)) return 1.0;                      // (cannot happen with int32 coordinates >= 0)
        idx = fastdiv31((unsigned)off, P.bdiv);
    } else {
        if (off >= (1ll << 32)) return 1.0;
        idx = fastdiv((unsigned)off, P.bdiv);
    }
    if (idx * P.bdiv.R != (unsigned)off) return 1.0;
    double v = __ldg(&P.bias[row.base + idx]);
    return isnan(v) ? 1.0 : v;
}

// The same lookup in two steps, so that the loads of several records can be issued together: where the entry is (and
// whether there is one), then what the loaded value means.  The load itself is unconditional (entry 0 stands in when there
// is no entry) so that nothing but arithmetic separates the loads of a group.
template <bool FAST>
__device__ __forceinline__ bool bias_index(const PvParams& P, const BiasRow& row, int mid, long long* at) {
    const long long off = (long long)mid - row.mid0;
    bool ok = (unsigned long long)off < row.span;
    unsigned idx;
    if (FAST) {
        ok = ok && off < (1ll << 31);
        idx = fastdiv31((unsigned)off, P.bdiv);
    } else {
        ok = ok && off < (1ll << 32);
        idx = fastdiv((unsigned)off, P.bdiv);
    }
    ok = ok && idx * P.bdiv.R == (unsigned)off;
    *at = ok ? row.base + (long long)idx : 0ll;
    return ok;
}
__device__ __forceinline__ double bias_value(double v, bool ok) { return (ok && !isnan(v)) ? v : 1.0; }

// i = min(bisect_left(splineX, clamp(d, min_x, max_x)), L-1) == clamp(ceil((d - splineX[0]) / R), 0, L-1), for an in-range d
template <bool FAST>
__device__ __forceinline__ int spline_index(const PvParams& P, long long d, int k0, int L) {
    int i = 0;
    if (FAST) {
        const int t = (int)d - k0 * (int)P.div.R;                        // k0 * R <= max_dist
        if (t > 0) {
            unsigned qd = fastdiv31((unsigned)t + P.div.R - 1u, P.div);
            i = qd > (unsigned)(L - 1) ? L - 1 : (int)qd;
        }
    } else {
        const long long t = d - (long long)k0 * P.R;
        if (t > 0) {
            long long tt = t + P.R - 1;
            long long qd = tt < (1ll << 32) ? (long long)fastdiv((unsigned)tt, P.div) : tt / P.R;
            i = qd > (long long)(L - 1) ? L - 1 : (int)qd;
        }
    }
    return i;
}

// prior of one record; returns false when the reference does not score it (fithic.py:427).
// FAST: 0 <= min_dist, max_dist + R < 2^31, so every in-range quantity fits 31 bits.
template <bool HAS_CHR, bool HAS_BIAS, bool FAST>
__device__ __forceinline__ bool record_prior(const PvParams& P, int m1, int m2, int c1, int c2, int k0, int L,
                                             const BiasRow& shard_row, bool have_b1, double b1_pre, double* prior_out) {
    const long long d = (long long)m2 - (long long)m1;                   // fithic.py:416
    if (!(P.min_dist <= d && d <= P.max_dist)) return false;
    // i = min(bisect_left(splineX, clamp(d, min_x, max_x)), L-1) == clamp(ceil((d - splineX[0]) / R), 0, L-1)
    int i = 0;
    if (FAST) {
        const int t = (int)d - k0 * (int)P.div.R;                        // k0 * R <= max_dist
        if (t > 0) {
            unsigned qd = fastdiv31((unsigned)t + P.div.R - 1u, P.div);
            i = qd > (unsigned)(L - 1) ? L - 1 : (int)qd;
        }
    } else {
        const long long t = d - (long long)k0 * P.R;
        if (t > 0) {
            long long tt = t + P.R - 1;
            long long qd = tt < (1ll << 32) ? (long long)fastdiv((unsigned)tt, P.div) : tt / P.R;
            i = qd > (long long)(L - 1) ? L - 1 : (int)qd;
        }
    }
    double prior = __ldg(&P.spline_y[i]);
    if (HAS_BIAS) {
        double b1, b2;
        if (HAS_CHR) {
            b1 = bias_lookup<FAST>(P, bias_row(P, c1), m1);
            b2 = bias_lookup<FAST>(P, bias_row(P, c2), m2);
        } else {
            b1 = have_b1 ? b1_pre : bias_lookup<FAST>(P, shard_row, m1);
            b2 = bias_lookup<FAST>(P, shard_row, m2);
        }
        prior = prior * (b1 * b2);                                        // :431
    }
    *prior_out = prior;
    return true;
}

__device__ __forceinline__ double finish_p(double pv) {                  // fithic.py:434: rows with !(p <= 1) are dropped
    return (pv <= 1.0) ? pv : __longlong_as_double(0x7ff8000000000000ll);
}

__device__ __forceinline__ void hist_p(unsigned* sh_hist, double pv, unsigned& ones, unsigned& nans) {
    if (isnan(pv)) { nans += 1; return; }
    if (pv == 1.0) { ones += 1; return; }
    atomicAdd(&sh_hist[(unsigned)((unsigned long long)__double_as_longlong(pv) >> 51) & (BBK_PHIST_BINS - 1)], 1u);
}

constexpr int WT_ITERS = 2;                         // int4 groups per lane per warp tile
constexpr int WT_PAIRS = 32 * 4 * WT_ITERS;         // 256 records per warp tile

struct WarpTile {                                   // warp-private
    double res[WT_PAIRS];                           // result slot of every record of the tile (slot = it*128 + lane*4 + e)
    double q[WT_PAIRS];                             // work lists: prior (count == 1 from the front, tails from the back)
    int c[WT_PAIRS];
    unsigned char slot[WT_PAIRS];
};

struct PvShared {
    double rcp[RCP_TAB];
    double lfact[LF_TAB];
    WarpTile w[PV_WARPS];
};

template <bool HAS_CHR, bool HAS_BIAS, bool HIST, bool FAST>
__global__ void __launch_bounds__(PV_THREADS, 3) pvalues_kernel(PvParams P) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    PvShared& sh = *reinterpret_cast<PvShared*>(smem_raw);
    unsigned* sh_hist = reinterpret_cast<unsigned*>(smem_raw + sizeof(PvShared));
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const long long S = P.fit->S;
    const int k0 = P.fit->k0, L = P.fit->L;
    const bool fit_ok = P.fit->status == BBK_FIT_OK && L > 0;

    for (int j = tid; j < RCP_TAB; j += PV_THREADS) sh.rcp[j] = g_rcp[j];
    for (int j = tid; j < LF_TAB; j += PV_THREADS) sh.lfact[j] = g_lfact[j];
    if (HIST) for (int i = tid; i < BBK_PHIST_BINS; i += PV_THREADS) sh_hist[i] = 0;
    __syncthreads();
    TailConst K;
    K.dn = (double)S;
    K.inv_n = S > 0 ? 1.0 / K.dn : 0.0;
    K.c_max = 1e-4 * K.dn;
    K.c5_max = 2e-11 * (K.dn * K.dn) * (K.dn * K.dn);
    WarpTile& W = sh.w[warp];
    BiasRow shard_row = {0, 0, 0, 0};
    if (HAS_BIAS && !HAS_CHR) shard_row = bias_row(P, P.shard_chrom);
    unsigned ones = 0, nans = 0;
    const bool s_fits = S <= 0x7fffffffll;
    const int s_cap = s_fits ? (int)S : 0x7fffffff;

    const long long n_groups = P.n_pairs >> 2;
    const long long groups_per_tile = 32 * WT_ITERS;
    const long long n_wtiles = (n_groups + groups_per_tile - 1) / groups_per_tile;
    const int4* m1v = reinterpret_cast<const int4*>(P.mid1);
    const int4* m2v = reinterpret_cast<const int4*>(P.mid2);
    const int4* cv = reinterpret_cast<const int4*>(P.count);
    const int4* c1v = reinterpret_cast<const int4*>(P.chr1);
    const int4* c2v = reinterpret_cast<const int4*>(P.chr2);
    double2* pv2 = reinterpret_cast<double2*>(P.p);
    const unsigned lt = (1u << lane) - 1;

    // warps are autonomous: no CTA barrier inside the loop
    for (long long wt = (long long)blockIdx.x * PV_WARPS + warp; wt < n_wtiles; wt += (long long)gridDim.x * PV_WARPS) {
        int n1 = 0, n2 = 0;                          // warp-uniform list lengths
        {   // the records this warp will classify next: pull them into L2 now (their first use stalls on DRAM otherwise)
            const long long wn = wt + (long long)gridDim.x * PV_WARPS;
            if (wn < n_wtiles) {
#pragma unroll
                for (int it = 0; it < WT_ITERS; ++it) {
                    const long long g = wn * groups_per_tile + it * 32 + lane;
                    if (g < n_groups) {
                        asm volatile("prefetch.global.L2 [%0];" :: "l"(m1v + g));
                        asm volatile("prefetch.global.L2 [%0];" :: "l"(m2v + g));
                        asm volatile("prefetch.global.L2 [%0];" :: "l"(cv + g));
                    }
                }
            }
        }
        if (HAS_CHR) {
            // ---- phase 1: classify; trivial results to their slots, the rest into the two dense lists
    #pragma unroll 1
            for (int it = 0; it < WT_ITERS; ++it) {
                const long long g = wt * groups_per_tile + it * 32 + lane;
                const bool live = g < n_groups;
                int4 z4 = make_int4(0, 0, 0, 0);
                int4 a1 = z4, a2 = z4, ac = z4, x1 = z4, x2 = z4;
                if (live) {
                    a1 = ld_stream_int4(m1v + g); a2 = ld_stream_int4(m2v + g); ac = ld_stream_int4(cv + g);
                    if (HAS_CHR) { x1 = ld_stream_int4(c1v + g); x2 = ld_stream_int4(c2v + g); }
                }
                const int m1s[4] = {a1.x, a1.y, a1.z, a1.w}, m2s[4] = {a2.x, a2.y, a2.z, a2.w}, cs[4] = {ac.x, ac.y, ac.z, ac.w};
                const int c1s[4] = {x1.x, x1.y, x1.z, x1.w}, c2s[4] = {x2.x, x2.y, x2.z, x2.w};
                // records that are neighbours in memory usually share their first locus (row-major input): one bias
                // gather serves the group then (any other order just takes the per-record path)
                bool same1 = false;
                double b1g = 1.0;
                if (HAS_BIAS && !HAS_CHR) {
                    same1 = (a1.x == a1.y) & (a1.y == a1.z) & (a1.z == a1.w);
                    if (same1 && live && fit_ok) b1g = bias_lookup<FAST>(P, shard_row, a1.x);
                }
    #pragma unroll
                for (int e = 0; e < 4; ++e) {
                    int cls = 0;                               // 0 final, 1 count == 1, 2 tail sum
                    double prior = 0.0, out = __longlong_as_double(0x7ff8000000000000ll);
                    if (live && fit_ok && record_prior<HAS_CHR, HAS_BIAS, FAST>(P, m1s[e], m2s[e], c1s[e], c2s[e], k0, L, shard_row, same1, b1g, &prior))
                        cls = bdtrc_class(cs[e], s_cap, s_fits, prior, &out);
                    const int slot = it * 128 + lane * 4 + e;
                    unsigned b1 = __ballot_sync(0xffffffffu, cls == 1), b2 = __ballot_sync(0xffffffffu, cls == 2);
                    if (cls) {
                        int pos = cls == 1 ? n1 + __popc(b1 & lt) : WT_PAIRS - 1 - (n2 + __popc(b2 & lt));
                        W.q[pos] = prior;
                        W.c[pos] = cs[e];
                        W.slot[pos] = (unsigned char)slot;
                    } else {
                        W.res[slot] = out;
                    }
                    n1 += __popc(b1);
                    n2 += __popc(b2);
                }
            }
        } else {
            // ---- phase 1: classify; trivial results to their slots, the rest into the two dense lists.  The four records of
            // a lane's group go through the steps together - where their spline and bias entries are, then all the loads,
            // unconditionally, then the products - so that the gathers of a group are in flight at once: as four lookups,
            // each behind its own early returns, they were four L2 latencies in a row (a quarter of the stall samples on the
            // 1 kb workload sat on the first use of a bias value).
#pragma unroll 1
            for (int it = 0; it < WT_ITERS; ++it) {
                const long long g = wt * groups_per_tile + it * 32 + lane;
                const bool live = g < n_groups && fit_ok;
                int4 z4 = make_int4(0, 0, 0, 0);
                int4 a1 = z4, a2 = z4, ac = z4;
                if (g < n_groups) { a1 = ld_stream_int4(m1v + g); a2 = ld_stream_int4(m2v + g); ac = ld_stream_int4(cv + g); }
                const int m1s[4] = {a1.x, a1.y, a1.z, a1.w}, m2s[4] = {a2.x, a2.y, a2.z, a2.w}, cs[4] = {ac.x, ac.y, ac.z, ac.w};
                const bool same1 = (a1.x == a1.y) & (a1.y == a1.z) & (a1.z == a1.w);
                bool inr[4], ok1[4], ok2[4];
                long long at1[4], at2[4];
                int si[4];
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    const long long d = (long long)m2s[e] - (long long)m1s[e];               // fithic.py:416
                    inr[e] = live && P.min_dist <= d && d <= P.max_dist;                      // fithic.py:427
                    si[e] = inr[e] ? spline_index<FAST>(P, d, k0, L) : 0;
                    ok1[e] = false; ok2[e] = false; at1[e] = 0; at2[e] = 0;
                    if (HAS_BIAS) {
                        if (e == 0 || !same1) ok1[e] = bias_index<FAST>(P, shard_row, m1s[e], &at1[e]);
                        ok2[e] = bias_index<FAST>(P, shard_row, m2s[e], &at2[e]);
                    }
                }
                double sv[4], v1[4], v2[4];
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    sv[e] = live ? __ldg(&P.spline_y[si[e]]) : 0.0;
                    v1[e] = 1.0; v2[e] = 1.0;
                    if (HAS_BIAS) {
                        if (e == 0 || !same1) v1[e] = __ldg(&P.bias[at1[e]]);
                        v2[e] = __ldg(&P.bias[at2[e]]);
                    }
                }
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    int cls = 0;                               // 0 final, 1 count == 1, 2 tail sum
                    double prior = sv[e], out = __longlong_as_double(0x7ff8000000000000ll);
                    if (HAS_BIAS) {
                        const double b1 = same1 ? bias_value(v1[0], ok1[0]) : bias_value(v1[e], ok1[e]);
                        prior = prior * (b1 * bias_value(v2[e], ok2[e]));                     // :431
                    }
                    if (inr[e]) cls = bdtrc_class(cs[e], s_cap, s_fits, prior, &out);
                    const int slot = it * 128 + lane * 4 + e;
                    unsigned b1m = __ballot_sync(0xffffffffu, cls == 1), b2m = __ballot_sync(0xffffffffu, cls == 2);
                    if (cls) {
                        int pos = cls == 1 ? n1 + __popc(b1m & lt) : WT_PAIRS - 1 - (n2 + __popc(b2m & lt));
                        W.q[pos] = prior;
                        W.c[pos] = cs[e];
                        W.slot[pos] = (unsigned char)slot;
                    } else {
                        W.res[slot] = out;
                    }
                    n1 += __popc(b1m);
                    n2 += __popc(b2m);
                }
            }
        }
        __syncwarp();
        // ---- phase 2a: count == 1 (bdtrc's closed form; -expm1(S ln(1-q)) also covers its q >= 0.01 branch)
        for (int k = lane; k < n1; k += 32) W.res[W.slot[k]] = -expm1(K.dn * log1m(W.q[k]));
        // ---- phase 2b: tail sums
        for (int kb = 0; kb < n2; kb += 32) {
            const int k = kb + lane;
            const bool active = k < n2;
            const int pos = WT_PAIRS - 1 - (active ? k : 0);
            TailState T;
            T.lp = 0.0; T.term = 0.0; T.sum = 1.0; T.a = 0.0; T.step = 0.0; T.j = 0;
            bool running = false;                    // this lane's sum is set up and not yet converged
            bool fast = false;
            if (active) {
                const int c = W.c[pos];
                const double q = W.q[pos];
                fast = fast_ok(c, K);
                if (fast) { tail_setup(c, q, K, sh.lfact, T); running = true; }
                else W.res[W.slot[pos]] = tail_general(c, S, q);
            }
            // every lane advances its own sum, 16 terms between two convergence checks, until the round is done.  (Handing
            // the last few running sums to 8-lane groups paid while upper- and lower-tail lanes ran separate loops; with
            // one loop for all lanes it no longer does: 1.72 ms with the groups, 1.64 ms without.)
            unsigned rmask = __ballot_sync(0xffffffffu, running);
            while (rmask) {
                if (running) {
                    const bool exhausted = tail_terms16(T, K, sh.rcp);
                    running = !(exhausted || T.term < TAIL_EPS * T.sum);
                }
                rmask = __ballot_sync(0xffffffffu, running);
            }
            if (active && fast) W.res[W.slot[pos]] = tail_finish(T.lp, T.sum);
        }
        __syncwarp();
        // ---- results back to their owners, coalesced 128-bit stores
#pragma unroll 1
        for (int it = 0; it < WT_ITERS; ++it) {
            const long long g = wt * groups_per_tile + it * 32 + lane;
            const double2* rs = reinterpret_cast<const double2*>(&W.res[it * 128 + lane * 4]);
            double2 r01 = rs[0], r23 = rs[1];
            r01.x = finish_p(r01.x); r01.y = finish_p(r01.y); r23.x = finish_p(r23.x); r23.y = finish_p(r23.y);
            if (g < n_groups) {
                st_stream_double2(pv2 + 2 * g, r01);
                st_stream_double2(pv2 + 2 * g + 1, r23);
                if (HIST) { hist_p(sh_hist, r01.x, ones, nans); hist_p(sh_hist, r01.y, ones, nans);
                            hist_p(sh_hist, r23.x, ones, nans); hist_p(sh_hist, r23.y, ones, nans); }
            }
        }
        __syncwarp();      // the tile buffers are reused by the next warp tile
    }
    if (HIST) {
        __syncthreads();
        for (int i = tid; i < BBK_PHIST_BINS; i += PV_THREADS) {
            unsigned v = sh_hist[i];
            if (v) atomicAdd((unsigned long long*)&P.p_hist[i], (unsigned long long)v);
        }
        unsigned o = __reduce_add_sync(0xffffffffu, ones), zn = __reduce_add_sync(0xffffffffu, nans);
        if (lane == 0) {
            if (o) atomicAdd((unsigned long long*)&P.p_hist[BBK_PHIST_BINS], (unsigned long long)o);
            if (zn) atomicAdd((unsigned long long*)&P.p_hist[BBK_PHIST_BINS + 1], (unsigned long long)zn);
        }
    }
}

// the last n_pairs % 4 records (at most 3): one thread each, evaluated in place
template <bool HAS_CHR, bool HAS_BIAS>
__global__ void pvalues_tail_kernel(PvParams P) {
    const long long i = ((P.n_pairs >> 2) << 2) + threadIdx.x;
    if (i >= P.n_pairs) return;
    const double qnan = __longlong_as_double(0x7ff8000000000000ll);
    const long long S = P.fit->S;
    const int k0 = P.fit->k0, L = P.fit->L;
    const bool fit_ok = P.fit->status == BBK_FIT_OK && L > 0;
    BiasRow shard_row = {0, 0, 0, 0};
    if (HAS_BIAS && !HAS_CHR) shard_row = bias_row(P, P.shard_chrom);
    const bool s_fits = S <= 0x7fffffffll;
    const int s_cap = s_fits ? (int)S : 0x7fffffff;
    int c1 = 0, c2 = 0;
    if (HAS_CHR) { c1 = P.chr1[i]; c2 = P.chr2[i]; }
    double pv = qnan, prior = 0.0;
    const int c = P.count[i];
    if (fit_ok && record_prior<HAS_CHR, HAS_BIAS, false>(P, P.mid1[i], P.mid2[i], c1, c2, k0, L, shard_row, false, 1.0, &prior)) {
        double out;
        int cls = bdtrc_class(c, s_cap, s_fits, prior, &out);
        if (cls == 0) pv = out;
        else if (cls == 1) pv = -expm1((double)S * log1m(prior));
        else pv = tail_general(c, S, prior);
    }
    pv = finish_p(pv);
    P.p[i] = pv;
    if (P.p_hist) {
        if (isnan(pv)) atomicAdd((unsigned long long*)&P.p_hist[BBK_PHIST_BINS + 1], 1ull);
        else if (pv == 1.0) atomicAdd((unsigned long long*)&P.p_hist[BBK_PHIST_BINS], 1ull);
        else atomicAdd((unsigned long long*)&P.p_hist[(unsigned)((unsigned long long)__double_as_longlong(pv) >> 51) & (BBK_PHIST_BINS - 1)], 1ull);
    }
}

#include "pvalue_tiles.inl"

int ensure_tables(cudaStream_t st) {
    // 1/j and ln j! are constants; fill them once per device (same values whoever wins a race)
    static std::mutex mu;
    static bool done[64] = {false};
    int dev = 0;
    BBK_CHECK_CUDA(cudaGetDevice(&dev));
    std::lock_guard<std::mutex> lock(mu);
    if (dev >= 0 && dev < 64 && done[dev]) return BBK_OK;
    pv_tables_kernel<<<(RCP_TAB + 255) / 256, 256, 0, st>>>();
    BBK_CHECK_LAUNCH("pv_tables_kernel");
    BBK_CHECK_CUDA(cudaStreamSynchronize(st));
    if (dev >= 0 && dev < 64) done[dev] = true;
    return BBK_OK;
}

template <bool HAS_CHR, bool HAS_BIAS, bool HIST, bool FAST>
int launch_pv(const PvParams& P, cudaStream_t st) {
    long long groups = P.n_pairs >> 2;
    if (groups > 0) {
        long long need = (groups + PV_WARPS * 32 * WT_ITERS - 1) / (PV_WARPS * 32 * WT_ITERS);
        long long grid = (long long)bbk_num_sms() * 3;
        if (need < grid) grid = need;
        size_t smem = sizeof(PvShared) + (HIST ? BBK_PHIST_BINS * sizeof(unsigned) : 0);
        BBK_CHECK_CUDA(cudaFuncSetAttribute(pvalues_kernel<HAS_CHR, HAS_BIAS, HIST, FAST>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        pvalues_kernel<HAS_CHR, HAS_BIAS, HIST, FAST><<<(unsigned)grid, PV_THREADS, smem, st>>>(P);
        BBK_CHECK_LAUNCH("pvalues_kernel");
    }
    if (P.n_pairs & 3) {
        pvalues_tail_kernel<HAS_CHR, HAS_BIAS><<<1, 32, 0, st>>>(P);
        BBK_CHECK_LAUNCH("pvalues_tail_kernel");
    }
    return BBK_OK;
}

}  // namespace

extern "C" int bbk_pvalues(const int32_t* d_chr1, const int32_t* d_chr2, const int32_t* d_mid1, const int32_t* d_mid2,
                           const int32_t* d_count, int64_t n_pairs, int32_t shard_chrom, int64_t resolution, int64_t min_dist,
                           int64_t max_dist, const BbkFitResult* d_fit, const double* d_spline_y, const BbkBiasTable* bias,
                           double* d_p, int64_t* d_p_hist, void* stream) {
    BBK_REQUIRE(n_pairs >= 0, "bbk_pvalues: negative size");
    BBK_REQUIRE(resolution > 0 && resolution < (1ll << 32), "bbk_pvalues: resolution must be in [1, 2^32)");
    BBK_REQUIRE((d_chr1 == nullptr) == (d_chr2 == nullptr), "bbk_pvalues: chr1/chr2 must both be given or both NULL");
    BBK_REQUIRE(d_fit && d_spline_y, "bbk_pvalues: null fit");
    if (n_pairs == 0) return BBK_OK;
    BBK_REQUIRE(d_mid1 && d_mid2 && d_count && d_p, "bbk_pvalues: null column");
    uintptr_t align = (uintptr_t)d_mid1 | (uintptr_t)d_mid2 | (uintptr_t)d_count | (uintptr_t)d_chr1 | (uintptr_t)d_chr2 | (uintptr_t)d_p;
    BBK_REQUIRE((align & 15) == 0, "bbk_pvalues: columns must be 16-byte aligned");
    PvParams P = {};
    P.chr1 = d_chr1; P.chr2 = d_chr2; P.mid1 = d_mid1; P.mid2 = d_mid2; P.count = d_count;
    P.n_pairs = n_pairs; P.shard_chrom = shard_chrom; P.R = resolution; P.min_dist = min_dist; P.max_dist = max_dist;
    P.div = make_fastdiv((uint64_t)resolution);
    P.fit = d_fit; P.spline_y = d_spline_y; P.p = d_p; P.p_hist = (long long*)d_p_hist;
    bool has_bias = bias && bias->d_bias;
    if (has_bias) {
        BBK_REQUIRE(bias->d_chrom_base && bias->d_mid0 && bias->n_chrom > 0, "bbk_pvalues: incomplete bias table");
        BBK_REQUIRE(bias->step >= 0 && bias->step < (1ll << 32), "bbk_pvalues: the bias tables' step must be in [0, 2^32)");
        P.bias = bias->d_bias; P.chrom_base = (const long long*)bias->d_chrom_base; P.mid0 = (const long long*)bias->d_mid0;
        P.n_chrom = bias->n_chrom;
    }
    P.bdiv = (has_bias && bias->step > 0) ? make_fastdiv((uint64_t)bias->step) : P.div;
    cudaStream_t st = (cudaStream_t)stream;
    int rc = ensure_tables(st);
    if (rc != BBK_OK) return rc;
    bool chr = d_chr1 != nullptr, hist = d_p_hist != nullptr;
    // 31-bit fast path: every in-range distance, and distance + resolution, fits 31 bits
    const bool fast = min_dist >= 0 && max_dist >= 0 && max_dist + resolution < (1ll << 31);
#define BBK_PV_CASE(C, B, H) if (chr == C && has_bias == B && hist == H) \
        return fast ? launch_pv<C, B, H, true>(P, st) : launch_pv<C, B, H, false>(P, st);
    BBK_PV_CASE(false, false, false) BBK_PV_CASE(false, false, true)
    BBK_PV_CASE(false, true, false)  BBK_PV_CASE(false, true, true)
    BBK_PV_CASE(true, false, false)  BBK_PV_CASE(true, false, true)
    BBK_PV_CASE(true, true, false)   BBK_PV_CASE(true, true, true)
#undef BBK_PV_CASE
    return BBK_E_INVALID;
}

// ---------------------------------------------------------------------------------------------------
// K4 as one streaming kernel over bulk-staged tiles + a patch kernel for the deferred rows (pvalue_tiles.inl)
// ---------------------------------------------------------------------------------------------------
extern "C" int bbk_score_begin(BbkScoreState* d_state, int64_t* d_p_hist, void* stream) {
    BBK_REQUIRE(d_state, "bbk_score_begin: null state");
    score_begin_kernel<<<(BBK_PHIST_LEN + 255) / 256, 256, 0, (cudaStream_t)stream>>>(d_state, (long long*)d_p_hist);
    BBK_CHECK_LAUNCH("score_begin_kernel");
    return BBK_OK;
}

extern "C" size_t bbk_bias_flags_bytes(int64_t n_entries) { return n_entries <= 0 ? 8 : (size_t)((n_entries + 31) / 32 + 1) * 4; }   // one spare (zero) word

extern "C" int bbk_bias_flags(const double* d_bias, int64_t n_entries, uint32_t* d_flags, void* stream) {
    BBK_REQUIRE(n_entries >= 0, "bbk_bias_flags: negative size");
    if (n_entries == 0) return BBK_OK;
    BBK_REQUIRE(d_bias && d_flags, "bbk_bias_flags: null pointer");
    bias_flags_kernel<<<(unsigned)((n_entries + 255) / 256), 256, 0, (cudaStream_t)stream>>>(d_bias, n_entries, d_flags);
    BBK_CHECK_LAUNCH("bias_flags_kernel");
    return BBK_OK;
}

extern "C" int bbk_score_guard(const BbkFitResult* d_fit, const double* d_spline_y, BbkScoreState* d_state, void* stream) {
    BBK_REQUIRE(d_fit && d_spline_y && d_state, "bbk_score_guard: null pointer");
    score_guard_kernel<<<1, 1024, 0, (cudaStream_t)stream>>>(d_fit, d_spline_y, d_state);
    BBK_CHECK_LAUNCH("score_guard_kernel");
    return BBK_OK;
}

static int check_deferred(const BbkDeferredList* list, const char* who) {
    if (!list || list->capacity < 0) { bbk_set_error("invalid argument: %s: null deferred list / negative capacity", who); return BBK_E_INVALID; }
    if (list->capacity > 0 && !(list->d_row && list->d_count && list->d_prior)) {
        bbk_set_error("invalid argument: %s: incomplete deferred list", who); return BBK_E_INVALID; }
    return BBK_OK;
}

extern "C" int bbk_score_pairs(const int32_t* d_mid1, const int32_t* d_mid2, const int32_t* d_count, int64_t n_pairs,
                               int32_t shard_chrom, int64_t resolution, int64_t min_dist, int64_t max_dist,
                               const BbkFitResult* d_fit, const double* d_spline_y, const BbkBiasTable* bias,
                               const uint32_t* d_bias_flags, int64_t out_base, double* d_p, double* d_q, int64_t* d_p_hist,
                               const BbkCandidates* cands, const BbkDeferredList* deferred, BbkScoreState* d_state, void* stream) {
    BBK_REQUIRE(n_pairs >= 0 && out_base >= 0 && (out_base & 3) == 0, "bbk_score_pairs: out_base must be a non-negative multiple of 4");
    BBK_REQUIRE(out_base + n_pairs < (1ll << 32), "bbk_score_pairs: rank-local rows must be below 2^32");
    BBK_REQUIRE(resolution > 1 && resolution < (1ll << 31), "bbk_score_pairs: resolution must be in [2, 2^31) (use bbk_pvalues otherwise)");
    BBK_REQUIRE(min_dist >= 0 && max_dist >= min_dist && max_dist + resolution < (1ll << 31),
                "bbk_score_pairs: needs 0 <= min_dist <= max_dist and max_dist + resolution < 2^31 (use bbk_pvalues otherwise)");
    BBK_REQUIRE(d_fit && d_spline_y && d_state, "bbk_score_pairs: null pointer");
    int rc = check_deferred(deferred, "bbk_score_pairs");
    if (rc != BBK_OK) return rc;
    if (n_pairs == 0) return BBK_OK;
    BBK_REQUIRE(d_mid1 && d_mid2 && d_count && d_p, "bbk_score_pairs: null column");
    uintptr_t align = (uintptr_t)d_mid1 | (uintptr_t)d_mid2 | (uintptr_t)d_count | (uintptr_t)d_p | (uintptr_t)d_q;
    BBK_REQUIRE((align & 15) == 0, "bbk_score_pairs: columns must be 16-byte aligned");
    BBK_REQUIRE(!cands || (d_q && d_p_hist), "bbk_score_pairs: the candidate list goes with q and the p histogram");
    StParams Q = {};
    Q.mid1 = d_mid1; Q.mid2 = d_mid2; Q.count = d_count; Q.n_pairs = n_pairs;
    Q.shard_chrom = shard_chrom; Q.min_dist = min_dist; Q.max_dist = max_dist;
    Q.div = make_fastdiv((uint64_t)resolution);
    Q.fit = d_fit; Q.spline_y = d_spline_y;
    const bool has_bias = bias && bias->d_bias;
    if (has_bias) {
        BBK_REQUIRE(bias->d_chrom_base && bias->d_mid0 && bias->n_chrom > 0, "bbk_score_pairs: incomplete bias table");
        BBK_REQUIRE(d_bias_flags, "bbk_score_pairs: a bias table needs its flag bits (bbk_bias_flags)");
        BBK_REQUIRE(bias->step == 0 || (bias->step > 1 && bias->step < (1ll << 31)), "bbk_score_pairs: the bias tables' step must be 0 or in [2, 2^31)");
        Q.bias = bias->d_bias; Q.chrom_base = (const long long*)bias->d_chrom_base; Q.mid0 = (const long long*)bias->d_mid0;
        Q.n_chrom = bias->n_chrom; Q.flags = d_bias_flags;
    }
    Q.bdiv = (has_bias && bias->step > 0) ? make_fastdiv((uint64_t)bias->step) : Q.div;
    Q.out_base = out_base; Q.p = d_p; Q.q = d_q; Q.p_hist = (long long*)d_p_hist;
    if (cands && cands->capacity > 0) {
        BBK_REQUIRE(cands->d_keys && cands->d_rows, "bbk_score_pairs: incomplete candidate list");
        Q.c_keys = (unsigned long long*)cands->d_keys; Q.c_idx = cands->d_rows; Q.c_cap = cands->capacity;
    }
    Q.d_row = deferred->d_row; Q.d_cnt = deferred->d_count; Q.d_prior = deferred->d_prior; Q.d_cap = deferred->capacity;
    Q.st = d_state;
    const long long tile_rows = (long long)ST_WARPS * ST_WROWS;
    const long long need = (n_pairs + tile_rows - 1) / tile_rows;
    long long grid = (long long)bbk_num_sms() * ST_CTAS_PER_SM;
    if (need < grid) grid = need;
    cudaStream_t st = (cudaStream_t)stream;
    static std::mutex mu;
    static bool attr_done[64] = {false};
    int dev = 0;
    BBK_CHECK_CUDA(cudaGetDevice(&dev));
    {
        std::lock_guard<std::mutex> lock(mu);
        if (!(dev >= 0 && dev < 64 && attr_done[dev])) {
            BBK_CHECK_CUDA(cudaFuncSetAttribute(score_tiles_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(StShared)));
            BBK_CHECK_CUDA(cudaFuncSetAttribute(score_tiles_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(StShared)));
            BBK_CHECK_CUDA(cudaFuncSetAttribute(score_tiles_kernel<true>, cudaFuncAttributePreferredSharedMemoryCarveout, 100));
            BBK_CHECK_CUDA(cudaFuncSetAttribute(score_tiles_kernel<false>, cudaFuncAttributePreferredSharedMemoryCarveout, 100));
            if (dev >= 0 && dev < 64) attr_done[dev] = true;
        }
    }
    if (has_bias) score_tiles_kernel<true><<<(unsigned)grid, ST_THREADS, sizeof(StShared), st>>>(Q);
    else score_tiles_kernel<false><<<(unsigned)grid, ST_THREADS, sizeof(StShared), st>>>(Q);
    BBK_CHECK_LAUNCH("score_tiles_kernel");
    return BBK_OK;
}

extern "C" int bbk_score_deferred(const BbkDeferredList* deferred, const BbkFitResult* d_fit, double* d_p, double* d_q,
                                  int64_t* d_p_hist, const BbkCandidates* cands, BbkScoreState* d_state, void* stream) {
    BBK_REQUIRE(d_fit && d_p && d_state, "bbk_score_deferred: null pointer");
    int rc = check_deferred(deferred, "bbk_score_deferred");
    if (rc != BBK_OK) return rc;
    if (deferred->capacity == 0) return BBK_OK;
    BBK_REQUIRE(!cands || (d_q && d_p_hist), "bbk_score_deferred: the candidate list goes with q and the p histogram");
    cudaStream_t st = (cudaStream_t)stream;
    rc = ensure_tables(st);
    if (rc != BBK_OK) return rc;
    DfParams D = {};
    D.d_row = deferred->d_row; D.d_cnt = deferred->d_count; D.d_prior = deferred->d_prior; D.d_cap = deferred->capacity;
    D.fit = d_fit; D.p = d_p; D.q = d_q; D.p_hist = (long long*)d_p_hist;
    if (cands && cands->capacity > 0) {
        BBK_REQUIRE(cands->d_keys && cands->d_rows, "bbk_score_deferred: incomplete candidate list");
        D.c_keys = (unsigned long long*)cands->d_keys; D.c_idx = cands->d_rows; D.c_cap = cands->capacity;
    }
    D.st = d_state;
    static std::mutex mu;
    static bool attr_done[64] = {false};
    int dev = 0;
    BBK_CHECK_CUDA(cudaGetDevice(&dev));
    {
        std::lock_guard<std::mutex> lock(mu);
        if (!(dev >= 0 && dev < 64 && attr_done[dev])) {
            BBK_CHECK_CUDA(cudaFuncSetAttribute(score_deferred_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(DfShared)));
            if (dev >= 0 && dev < 64) attr_done[dev] = true;
        }
    }
    // the list length is only known on the device: a grid that covers the device, rounds handed out by stride
    score_deferred_kernel<<<(unsigned)(bbk_num_sms() * 3), PV_THREADS, sizeof(DfShared), st>>>(D);
    BBK_CHECK_LAUNCH("score_deferred_kernel");
    return BBK_OK;
}
