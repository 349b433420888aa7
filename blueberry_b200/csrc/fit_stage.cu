// fit_stage.cu - K2 + K3: possible pairs per distance, equal-occupancy binning, smoothing spline,
// spline evaluation on the distance grid and antitonic regression, in ONE single-CTA kernel so the
// pass never leaves the device between the histogram (K1) and the p-value kernel (K4).
//
// Reference: generate_FragPairs fithic.py:302-311, calculate_probabilities fithic.py:160-227,
// fit_spline fithic.py:340-374.  All of this is O(D) FP64 work (D ~ 2-5 thousand distances,
// ~100 bins): latency-bound, not bandwidth-bound.  The arithmetic lives in fit_stage.h /
// fit_coop.h, which are also compiled on the host by tests/host_harness and checked there against
// scipy/sklearn; this file only stages data in shared memory and runs the phases.
//
// Compiled with -fmad=false: the knot search makes discrete decisions on FP64 values, and the
// CPU libraries it must agree with do not contract a*b+c.
#include "common.cuh"
#include "fit_coop.h"

namespace {

constexpr int FIT_THREADS = 256;

struct FitParams {
    const long long* possible;
    const long long* observed;
    const long long* totals;
    const double* x_in;      // stage-injection: bins given (possible/observed unused)
    const double* y_in;
    int m_in;
    int nkeys;
    int n_bins;
    long long R, min_dist, max_dist;
    int max_bins;
    BbkFitResult* result;
    double* x;
    double* y;
    int* bin_of_key;
    double* spline_y;
    double* spline_raw;
    double* knots;
    double* coefs;
    double* gws;             // global workspace (fallback when a phase does not fit in shared memory)
    size_t pool_doubles;     // dynamic shared memory pool, in doubles
};

struct FitShared {
    BbkCoopState st;
    int status, n_out, k0, L, nk_eff;
    long long S;
    double s, min_x, max_x;
    long long t[7];
    long long slice_tot[FIT_THREADS];
    int s_given;
    double s_in;
    double y_min;
    double cmax[FIT_THREADS], cmin[FIT_THREADS];      // antitonic regression: extrema of each thread's chunk
};

__device__ __forceinline__ double* pick(double* pool, size_t pool_doubles, size_t need, double* global_fallback) {
    return need <= pool_doubles ? pool : global_fallback;
}

// bytes of scratch one fit needs (bbk_fit_workspace_bytes); the batched kernel checks every problem's workspace with it
BBK_HD size_t fit_workspace_bytes(int max_bins, int nkeys) {
    size_t m = max_bins > 4 ? (size_t)max_bins : 4;
    size_t a = (size_t)3 * nkeys + m + 2;
    size_t b = bbk_coop_ws_doubles((int)m) + 2 * m;
    size_t c = 3 * (m + 4) + (size_t)4 * nkeys + 8;
    size_t mx = a > b ? a : b;
    mx = mx > c ? mx : c;
    return (mx + 16) * sizeof(double);
}

// the whole fit of one problem by one CTA of FIT_THREADS threads
__device__ __forceinline__ void fit_body(const FitParams& P) {
    extern __shared__ double pool[];
    __shared__ FitShared sh;
    const int tid = threadIdx.x;
    const bool injected = P.x_in != nullptr;

    if (tid == 0) {
        for (int i = 0; i < 7; ++i) sh.t[i] = 0;
        sh.t[0] = clock64();
        sh.s_given = P.result->status == BBK_FIT_S_GIVEN;      // the caller supplies s (include/bbk.h: BbkFitResult.smoothing)
        sh.s_in = P.result->smoothing;
        sh.status = BBK_FIT_OK;
        sh.n_out = 0; sh.k0 = 0; sh.L = 0; sh.y_min = 0.0; sh.s = 0.0;
        sh.S = injected ? 0 : P.totals[0];
        long long eff = P.nkeys;
        if (P.max_dist > -1) { long long lim = P.max_dist / P.R + 1; if (lim < eff) eff = lim; }
        sh.nk_eff = (int)eff;
        sh.st.n = 0; sh.st.fp = 0.0; sh.st.ier = 0;
        for (int i = 0; i < 8; ++i) sh.st.diag[i] = 0;
    }
    for (int k = tid; k < P.nkeys; k += FIT_THREADS) if (P.bin_of_key) P.bin_of_key[k] = -1;
    __syncthreads();

    int m = 0;
    if (!injected) {
        // ---------------- equal-occupancy binning (fithic.py:160-227)
        const int nk = sh.nk_eff;
        const long long S = sh.S;
        // stage observed[0..nk) (and possible) in shared memory when they fit; bin bounds after them
        size_t need = (size_t)3 * nk + (size_t)P.max_bins + 2;    // 3 int64 tables + 2 int32 bound arrays
        double* base = pick(pool, P.pool_doubles, need, P.gws);
        long long* obs_s = (long long*)base;
        long long* pos_s = obs_s + nk;
        long long* pre_s = pos_s + nk;
        int* bstart = (int*)(pre_s + nk);
        int* bend = bstart + P.max_bins;
        for (int k0 = tid; k0 < nk; k0 += 4 * FIT_THREADS) {     // eight loads in flight per thread: one round trip per 512 keys
            long long o[4], q[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int k = k0 + u * FIT_THREADS;
                o[u] = k < nk ? __ldg(P.observed + k) : 0;
                q[u] = k < nk ? __ldg(P.possible + k) : 0;
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int k = k0 + u * FIT_THREADS;
                if (k < nk) { obs_s[k] = o[u]; pos_s[k] = q[u]; }
            }
        }
        __syncthreads();
        // inclusive prefix sums of observed (the reference's totalInteractionCountSoFar, fithic.py:183): FIT_THREADS keys at
        // a time, a shuffle scan per warp, the warp totals and the running carry through shared memory
        {
            const int lane = tid & 31, warp = tid >> 5;
            long long carry = 0;
            for (int c0 = 0; c0 < nk; c0 += FIT_THREADS) {
                const int k = c0 + tid;
                long long v = k < nk ? obs_s[k] : 0;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    const long long u = __shfl_up_sync(0xffffffffu, v, o);
                    if (lane >= o) v += u;
                }
                if (lane == 31) sh.slice_tot[warp] = v;
                __syncthreads();
                long long add = carry, tot = 0;
#pragma unroll
                for (int w = 0; w < FIT_THREADS / 32; ++w) {
                    const long long wt = sh.slice_tot[w];
                    add += w < warp ? wt : 0;
                    tot += wt;
                }
                if (k < nk) pre_s[k] = v + add;
                carry += tot;
                __syncthreads();
            }
        }
        if (tid < 32) {
            // Bin boundaries by warp 0.  A bin that starts at key s closes at the first key k >= s with
            //   observed[k] >= desired  or  (sum of observed[s..k]) >= desired        (fithic.py:188-197)
            // which 32 lanes test for 32 consecutive keys at a time.  `desired` is an int floor for the first
            // bin (:167) and a double afterwards (:209); for an integer v, v >= d  <=>  v >= ceil(d).
            const int lane = tid;
            int stc = BBK_FIT_OK, nout = 0;
            if (S == 0) {
                bool any = false;
                for (int k = lane; k < nk; k += 32) any |= bbk_in_range((long long)k * P.R, P.min_dist, P.max_dist);
                stc = __any_sync(0xffffffffu, any) ? BBK_FIT_S_ZERO : BBK_FIT_OK;
            } else {
                // the in-range keys form one interval [klo, khi]
                int klo = nk, khi = -1;
                for (int k = lane; k < nk; k += 32)
                    if (bbk_in_range((long long)k * P.R, P.min_dist, P.max_dist)) { klo = min(klo, k); khi = max(khi, k); }
                for (int o = 16; o > 0; o >>= 1) {
                    klo = min(klo, __shfl_xor_sync(0xffffffffu, klo, o));
                    khi = max(khi, __shfl_xor_sync(0xffffffffu, khi, o));
                }
                long long D = 0;
                if (P.n_bins != 0) D = (S >= 0 || S % P.n_bins == 0) ? S / P.n_bins : S / P.n_bins - 1;   // floor (:167)
                // The serial chain per bin is: threshold test -> ballot -> next `desired` (an FP64 division).  The prefix sum at
                // the closing key serves both the division and, as `base`, the next bin, and the next bin's first 32 keys are
                // loaded before the division is started, so nothing but the division and the test is left on that chain.
                int n = 0, s0 = klo;
                long long base = (s0 > 0 && s0 <= khi) ? pre_s[s0 - 1] : 0;
                long long po = 0, pp = 0;                            // first chunk of the current bin
                if (s0 + lane <= khi) { po = obs_s[s0 + lane]; pp = pre_s[s0 + lane]; }
                while (s0 <= khi) {
                    int kk = -1;
                    long long pk = 0;                                // prefix sum at the closing key
                    for (int k0w = s0; k0w <= khi; k0w += 32) {
                        const int k = k0w + lane;
                        long long o = po, q = pp;
                        if (k0w != s0) { o = 0; q = 0; if (k <= khi) { o = obs_s[k]; q = pre_s[k]; } }
                        bool hit = k <= khi && (o >= D || q - base >= D);
                        unsigned bal = __ballot_sync(0xffffffffu, hit);
                        if (bal) {
                            const int src = __ffs(bal) - 1;
                            kk = k0w + src;
                            pk = __shfl_sync(0xffffffffu, q, src);
                            break;
                        }
                    }
                    if (kk < 0) break;                               // the trailing, unfilled bin is dropped
                    if (nout >= P.max_bins) { stc = BBK_FIT_TOO_MANY_BINS; break; }
                    if (lane == 0) { bstart[nout] = s0; bend[nout] = kk; }
                    nout += 1;
                    n += 1;                                          // :206
                    s0 = kk + 1;
                    po = 0; pp = 0;
                    if (s0 + lane <= khi) { po = obs_s[s0 + lane]; pp = pre_s[s0 + lane]; }
                    if (n < P.n_bins) {                              // :208-209
                        double dd = 1.0 * (double)(S - pk) / (double)(P.n_bins - n);
                        double cd = ceil(dd);
                        D = cd >= 9.2e18 ? 0x7fffffffffffffffll : (cd <= -9.2e18 ? -0x7fffffffffffffffll : (long long)cd);
                    }
                    base = pk;
                }
            }
            if (lane == 0) { sh.status = stc; sh.n_out = stc == BBK_FIT_OK ? nout : 0; }
        }
        __syncthreads();
        m = sh.n_out;
        if (tid == 0) sh.t[1] = clock64();
        if (sh.status == BBK_FIT_OK) {
            // bin statistics (fithic.py:211-217): the per-key operands - two int64 -> double conversions and the distance
            // term with its division - are formed by all threads in place (the integer tables and the prefix sums are not
            // needed any more), so that the serial part, one thread per bin adding its keys in the reference's order, is
            // three additions per key
            double* dpos = (double*)pos_s;
            double* dobs = (double*)obs_s;
            double* term = (double*)pre_s;
            for (int k = tid; k < nk; k += FIT_THREADS) {
                const double pv = (double)pos_s[k], ov = (double)obs_s[k];
                term[k] = 1.0 * pv * ((double)((long long)k * P.R) / 10000.0);
                dpos[k] = pv;
                dobs[k] = ov;
            }
            __syncthreads();
            for (int j = tid; j < m; j += FIT_THREADS) {
                double n_pairs = 0.0, n_inter = 0.0, avg = 0.0;
                for (int b = bstart[j]; b <= bend[j]; ++b) {
                    n_pairs += dpos[b];
                    n_inter += dobs[b];
                    avg += term[b];
                }
                if (n_pairs == 0.0 || S == 0) {
                    atomicMin(&sh.status, n_pairs == 0.0 ? BBK_FIT_ZERO_PAIRS_BIN : BBK_FIT_S_ZERO);
                    P.x[j] = 0.0;
                    P.y[j] = 0.0;
                } else {
                    P.y[j] = (n_inter / n_pairs) / (double)S;        // :216
                    P.x[j] = 10000.0 * (avg / n_pairs);              // :217
                }
                if (P.bin_of_key) for (int k = bstart[j]; k <= bend[j]; ++k) P.bin_of_key[k] = j;
            }
        }
        __syncthreads();
    } else {
        m = P.m_in;
        for (int j = tid; j < m; j += FIT_THREADS) { P.x[j] = P.x_in[j]; P.y[j] = P.y_in[j]; }
        if (tid == 0) sh.n_out = m;
        __syncthreads();
    }

    // ---------------- smoothing spline UnivariateSpline(x, y, s=min(y)**2)   (fithic.py:340-343)
    if (tid == 0) sh.t[2] = clock64();
    if (sh.status == BBK_FIT_OK && m < 4 && tid == 0) sh.status = BBK_FIT_TOO_FEW_BINS;
    __syncthreads();
    if (sh.status == BBK_FIT_OK) {
        size_t need = bbk_coop_ws_doubles(m) + (size_t)2 * m;
        double* base = pick(pool, P.pool_doubles, need, P.gws);
        double* xs = base;
        double* ys = base + m;
        for (int j = tid; j < m; j += FIT_THREADS) { xs[j] = P.x[j]; ys[j] = P.y[j]; }
        __syncthreads();
        if (tid == 0) {
            double ymin = ys[0], xmin = xs[0], xmax = xs[0];
            bool nondecr = true, strict = true;
            for (int j = 1; j < m; ++j) {
                ymin = ys[j] < ymin ? ys[j] : ymin;
                xmin = xs[j] < xmin ? xs[j] : xmin;
                xmax = xs[j] > xmax ? xs[j] : xmax;
                nondecr = nondecr && (xs[j] - xs[j - 1] >= 0.0);
                strict = strict && (xs[j] - xs[j - 1] > 0.0);
            }
            sh.y_min = ymin;
            sh.s = sh.s_given ? sh.s_in : ymin * ymin;       // fithic.py:340
            sh.min_x = xmin;                                 // fithic.py:350
            sh.max_x = xmax;
            if (!(sh.s > 0.0 ? nondecr : strict)) sh.status = BBK_FIT_X_NOT_INCREASING;
        }
        __syncthreads();
        if (sh.status == BBK_FIT_OK) {
            BbkCoopWs cw;
            if (base == pool) {                              // everything in shared memory
                bbk_coop_ws_carve(pool + 2 * m, m, &cw);
                bbk_coop_univariate_spline_t<true>(pool, pool + m, m, sh.s, &sh.st, &cw);
            } else {                                         // large m: global workspace
                bbk_coop_ws_carve(base + 2 * m, m, &cw);
                bbk_coop_univariate_spline_t<false>(xs, ys, m, sh.s, &sh.st, &cw);
            }
            __syncthreads();
            const int n = sh.st.n;
            // the search solves for n - 4 coefficients and never writes c[n-4 .. n): that is stale pool or workspace memory,
            // where scipy's array (ius._data[9]) holds zeros
            for (int i = tid; i < m + 4; i += FIT_THREADS) {
                P.knots[i] = i < n ? cw.w.t[i] : 0.0;
                P.coefs[i] = i < n - 4 ? cw.w.c[i] : 0.0;
            }
            __syncthreads();
        }
    }

    // ---------------- splineX = keys within [min(x), max(x)], splineY = ius(splineX)   (fithic.py:350-359)
    if (tid == 0) sh.t[3] = clock64();
    if (sh.status == BBK_FIT_OK) {
        if (tid == 0) {
            // first key k with k*R >= min_x and last key with k*R <= max_x (keys are ints, x are doubles)
            long long k0 = (long long)ceil(sh.min_x / (double)P.R);
            if (k0 < 0) k0 = 0;
            while (k0 > 0 && (double)((k0 - 1) * P.R) >= sh.min_x) --k0;
            while ((double)(k0 * P.R) < sh.min_x) ++k0;
            long long k1 = (long long)floor(sh.max_x / (double)P.R);
            while ((double)((k1 + 1) * P.R) <= sh.max_x) ++k1;
            while (k1 >= 0 && (double)(k1 * P.R) > sh.max_x) --k1;
            if (k1 > P.nkeys - 1) k1 = P.nkeys - 1;
            long long L = k1 - k0 + 1;
            if (L <= 0) { sh.status = BBK_FIT_EMPTY_GRID; L = 0; }
            sh.k0 = (int)k0;
            sh.L = (int)L;
        }
        __syncthreads();
    }
    if (sh.status == BBK_FIT_OK) {
        const int L = sh.L, n = sh.st.n;
        // knots / coefficients back into shared memory for the evaluation
        size_t need = (size_t)3 * (m + 4) + (size_t)4 * L + 8;
        double* base = pick(pool, P.pool_doubles, need, P.gws);
        double* tk = base;
        double* ck = base + (m + 4);
        double* rterm = ck + (m + 4);
        double* vraw = rterm + (m + 4);
        double* wmean = vraw + L;
        double* wcount = wmean + L;
        int* wstart = (int*)(wcount + L);
        for (int i = tid; i < n; i += FIT_THREADS) { tk[i] = P.knots[i]; ck[i] = P.coefs[i]; }
        __syncthreads();
        for (int i = tid; i < L; i += FIT_THREADS) {
            int cur = 4;
            double arg = (double)((long long)(sh.k0 + i) * P.R);
            P.spline_raw[i] = bbk_spline_eval(tk, n, ck, arg, &cur);
        }
        __syncthreads();
        // ---------------- antitonic regression (fithic.py:361-362) and the residual (fithic.py:374)
        // residual terms in parallel (summed in order by thread 0 below)
        for (int j = tid; j < m; j += FIT_THREADS) {
            int cur = 4;
            double dv = P.y[j] - bbk_spline_eval(tk, n, ck, P.x[j], &cur);
            rterm[j] = dv * dv;
        }
        for (int i = tid; i < L; i += FIT_THREADS) vraw[i] = P.spline_raw[i];
        __syncthreads();
        // pool-adjacent-violators, cut into the pieces between safe cuts (fit_stage.h): chunk extrema, piece starts, then
        // every thread runs the pieces that start in its chunk and writes their block means straight to spline_y
        if (tid == 0) sh.t[4] = clock64();
        bbk_pava_phase1(vraw, L, FIT_THREADS, tid, sh.cmax, sh.cmin);
        if (tid == FIT_THREADS - 1) {
            double res = 0.0;
            for (int j = 0; j < m; ++j) res = res + rterm[j];
            P.result->residual = res;
        }
        __syncthreads();
        bbk_pava_phase2(vraw, L, FIT_THREADS, tid, sh.cmax, sh.cmin, wcount, wstart);
        __syncthreads();
        bbk_pava_phase3(vraw, L, FIT_THREADS, tid, wstart, wmean, wcount, P.spline_y);
        for (int i = L + tid; i < P.nkeys; i += FIT_THREADS) { P.spline_y[i] = 0.0; P.spline_raw[i] = 0.0; }
    }
    __syncthreads();
    if (tid == 0) {
        BbkFitResult* r = P.result;
        r->status = sh.status;
        r->n_out = sh.n_out;
        r->k0 = sh.k0;
        r->L = sh.L;
        r->n_knots = sh.st.n;
        r->ier = sh.st.ier;
        r->S = sh.S;
        r->min_x = sh.min_x;
        r->max_x = sh.max_x;
        r->fp = sh.st.fp;
        r->smoothing = sh.s;
        r->y_min = sh.y_min;
        sh.t[5] = clock64();
        for (int i = 0; i < 5; ++i) r->phase_cycles[i] = (sh.t[i + 1] && sh.t[i]) ? sh.t[i + 1] - sh.t[i] : 0;
        r->phase_cycles[5] = sh.t[5] - sh.t[0];
        for (int i = 0; i < 8; ++i) r->spline_diag[i] = sh.st.diag[i];
        if (sh.status != BBK_FIT_OK) r->residual = 0.0;
    }
}

__global__ void __launch_bounds__(FIT_THREADS, 1) fit_kernel(FitParams P) { fit_body(P); }

// bbk_fit_batched: CTA b runs problem b with the shared n_bins / R / distance limits.  A problem that cannot run (sizes, null
// pointers, workspace below fit_workspace_bytes) gets BBK_FIT_BAD_PROBLEM in its own result and touches nothing else.
__global__ void __launch_bounds__(FIT_THREADS, 1) fit_batched_kernel(const BbkFitProblem* problems, int n_bins, long long R,
                                                                     long long min_dist, long long max_dist, size_t pool_doubles) {
    const BbkFitProblem pr = problems[blockIdx.x];
    if (!pr.d_result) return;
    const bool ok = pr.d_possible && pr.d_obs_sum && pr.d_totals && pr.d_x && pr.d_y && pr.d_spline_y && pr.d_spline_raw &&
                    pr.d_knots && pr.d_coefs && pr.d_workspace && pr.nkeys > 0 && pr.max_bins >= 4 &&
                    pr.workspace_bytes >= fit_workspace_bytes(pr.max_bins, pr.nkeys);
    if (!ok) {
        if (threadIdx.x == 0) {
            BbkFitResult* r = pr.d_result;
            r->status = BBK_FIT_BAD_PROBLEM;
            r->n_out = 0; r->k0 = 0; r->L = 0; r->n_knots = 0; r->ier = 0; r->S = 0;
            r->residual = 0.0;
        }
        return;
    }
    FitParams P;
    P.possible = (const long long*)pr.d_possible; P.observed = (const long long*)pr.d_obs_sum; P.totals = (const long long*)pr.d_totals;
    P.x_in = nullptr; P.y_in = nullptr; P.m_in = 0;
    P.nkeys = pr.nkeys; P.n_bins = n_bins; P.R = R; P.min_dist = min_dist; P.max_dist = max_dist; P.max_bins = pr.max_bins;
    P.result = pr.d_result; P.x = pr.d_x; P.y = pr.d_y; P.bin_of_key = pr.d_bin_of_key; P.spline_y = pr.d_spline_y;
    P.spline_raw = pr.d_spline_raw; P.knots = pr.d_knots; P.coefs = pr.d_coefs; P.gws = (double*)pr.d_workspace;
    P.pool_doubles = pool_doubles;
    fit_body(P);
}

__global__ void possible_pairs_kernel(const long long* n_frags, const long long* max_frag, int n_chrom, long long R,
                                      int nkeys, long long* possible) {
    int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= nkeys) return;
    long long d = (long long)k * R, tot = 0;
    for (int c = 0; c < n_chrom; ++c)
        if (d <= max_frag[c]) tot += n_frags[c] - k;          // fithic.py:309-311
    possible[k] = tot;
}

size_t fit_pool_bytes() { return 200 * 1024; }

int launch_fit(FitParams& P, size_t workspace_bytes, cudaStream_t st) {
    size_t need = bbk_fit_workspace_bytes(P.max_bins, P.nkeys);
    if (workspace_bytes < need || !P.gws) {
        bbk_set_error("bbk_fit: workspace too small (%zu < %zu bytes)", workspace_bytes, need);
        return BBK_E_WORKSPACE;
    }
    size_t pool = fit_pool_bytes();
    P.pool_doubles = pool / sizeof(double);
    BBK_CHECK_CUDA(cudaFuncSetAttribute(fit_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pool));
    fit_kernel<<<1, FIT_THREADS, pool, st>>>(P);
    BBK_CHECK_LAUNCH("fit_kernel");
    return BBK_OK;
}

}  // namespace

extern "C" size_t bbk_fit_workspace_bytes(int32_t max_bins, int32_t nkeys) { return fit_workspace_bytes(max_bins, nkeys); }

extern "C" int bbk_possible_pairs(const int64_t* d_n_frags, const int64_t* d_max_frag, int32_t n_chrom, int64_t resolution,
                                  int32_t nkeys, int64_t* d_possible, void* stream) {
    BBK_REQUIRE(d_n_frags && d_max_frag && d_possible, "bbk_possible_pairs: null pointer");
    BBK_REQUIRE(n_chrom >= 0 && nkeys >= 0 && resolution > 0, "bbk_possible_pairs: bad sizes");
    if (nkeys == 0) return BBK_OK;
    possible_pairs_kernel<<<(nkeys + 255) / 256, 256, 0, (cudaStream_t)stream>>>(
        (const long long*)d_n_frags, (const long long*)d_max_frag, n_chrom, resolution, nkeys, (long long*)d_possible);
    BBK_CHECK_LAUNCH("possible_pairs_kernel");
    return BBK_OK;
}

extern "C" int bbk_fit(const int64_t* d_possible, const int64_t* d_obs_sum, int32_t nkeys, const int64_t* d_totals,
                       int32_t n_bins, int64_t resolution, int64_t min_dist, int64_t max_dist, int32_t max_bins,
                       BbkFitResult* d_result, double* d_x, double* d_y, int32_t* d_bin_of_key, double* d_spline_y,
                       double* d_spline_raw, double* d_knots, double* d_coefs, void* d_workspace, size_t workspace_bytes,
                       void* stream) {
    BBK_REQUIRE(d_possible && d_obs_sum && d_totals && d_result && d_x && d_y && d_spline_y && d_spline_raw && d_knots && d_coefs,
                "bbk_fit: null pointer");
    BBK_REQUIRE(nkeys > 0 && max_bins >= 4 && resolution > 0, "bbk_fit: bad sizes");
    FitParams P = {};
    P.possible = (const long long*)d_possible; P.observed = (const long long*)d_obs_sum; P.totals = (const long long*)d_totals;
    P.x_in = nullptr; P.y_in = nullptr; P.m_in = 0;
    P.nkeys = nkeys; P.n_bins = n_bins; P.R = resolution; P.min_dist = min_dist; P.max_dist = max_dist; P.max_bins = max_bins;
    P.result = d_result; P.x = d_x; P.y = d_y; P.bin_of_key = d_bin_of_key; P.spline_y = d_spline_y; P.spline_raw = d_spline_raw;
    P.knots = d_knots; P.coefs = d_coefs; P.gws = (double*)d_workspace;
    return launch_fit(P, workspace_bytes, (cudaStream_t)stream);
}

extern "C" int bbk_fit_from_bins(const double* d_x_in, const double* d_y_in, int32_t m, int32_t nkeys, int64_t resolution,
                                 BbkFitResult* d_result, double* d_spline_y, double* d_spline_raw, double* d_knots,
                                 double* d_coefs, void* d_workspace, size_t workspace_bytes, void* stream) {
    BBK_REQUIRE(d_x_in && d_y_in && d_result && d_spline_y && d_spline_raw && d_knots && d_coefs, "bbk_fit_from_bins: null pointer");
    BBK_REQUIRE(m >= 1 && nkeys > 0 && resolution > 0, "bbk_fit_from_bins: bad sizes");
    // x / y scratch copies live at the end of the caller's workspace
    size_t need = bbk_fit_workspace_bytes(m, nkeys) + (size_t)2 * m * sizeof(double);
    if (workspace_bytes < need) {
        bbk_set_error("bbk_fit_from_bins: workspace too small (%zu < %zu bytes)", workspace_bytes, need);
        return BBK_E_WORKSPACE;
    }
    FitParams P = {};
    P.x_in = d_x_in; P.y_in = d_y_in; P.m_in = m;
    P.nkeys = nkeys; P.n_bins = 0; P.R = resolution; P.min_dist = 0; P.max_dist = -1; P.max_bins = m > 4 ? m : 4;
    P.result = d_result;
    P.x = (double*)((char*)d_workspace + bbk_fit_workspace_bytes(m, nkeys));
    P.y = P.x + m;
    P.bin_of_key = nullptr; P.spline_y = d_spline_y; P.spline_raw = d_spline_raw; P.knots = d_knots; P.coefs = d_coefs;
    P.gws = (double*)d_workspace;
    return launch_fit(P, bbk_fit_workspace_bytes(m, nkeys), (cudaStream_t)stream);
}

extern "C" int bbk_fit_batched(const BbkFitProblem* d_problems, int32_t n_problems, int32_t n_bins, int64_t resolution,
                               int64_t min_dist, int64_t max_dist, void* stream) {
    BBK_REQUIRE(n_problems >= 0 && resolution > 0, "bbk_fit_batched: bad sizes");
    if (n_problems == 0) return BBK_OK;
    BBK_REQUIRE(d_problems, "bbk_fit_batched: null pointer");
    const size_t pool = fit_pool_bytes();
    BBK_CHECK_CUDA(cudaFuncSetAttribute(fit_batched_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pool));
    fit_batched_kernel<<<n_problems, FIT_THREADS, pool, (cudaStream_t)stream>>>(d_problems, n_bins, resolution, min_dist, max_dist,
                                                                               pool / sizeof(double));
    BBK_CHECK_LAUNCH("fit_batched_kernel");
    return BBK_OK;
}
