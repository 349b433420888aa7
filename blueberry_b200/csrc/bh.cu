// bh.cu - K5: Benjamini-Hochberg q-values the way the reference computes them
// (benjamini_hochberg_correction fithic.py:466-487, benjamini_hochberg blueberry.pyx:40-75):
//     sort p ascending; q_(i) = max(q_(i-1), min(p_(i) * N / i, 1))     - a FORWARD running max.
//
// Consequences used here (all exact, no approximation):
//   * tied p share the q of the first of them, so only "1 + number of strictly smaller p" matters;
//   * once some sorted position reaches p*N/i >= 1 every later q is exactly 1.0.  A coarse
//     histogram of p (4096 buckets = exponent + top mantissa bit, filled by K4 or by a pass here)
//     gives the first bucket whose FIRST element is guaranteed to have p*N/rank >= 1; everything
//     from that bucket on (and every p == 1.0 row, i.e. every zero-count pair) gets q = 1.0 without
//     being sorted.  Only the "candidates" below it are radix-sorted - typically a few percent.
//   * the q formula keeps the reference's two roundings: (p * N) / rank.
// Device pipeline (no host synchronisation; candidate count lives on the device):
//   [coarse hist] -> threshold (1 CTA) -> compact + write q=1/NaN (the 16 B/pair pass)
//   -> ONE cooperative launch (one CTA per SM, grid-wide barriers between phases) that ranks the candidates:
//      LSD radix sort of (key, index), 8 x 8 bits, passes with a uniform digit skipped, then head flags +
//      running max and the scatter of q (and rank) to input order.
//      The candidate set is usually small (1e5 of 1e8 rows on BASELINE config 2), so this step is bound by
//      dependent launches, not by bytes: 27 launches became 1 launch with 17 grid barriers.
// BBK_BH_POSITIONAL (blueberry.pyx:40: input already sorted) skips everything but the scan (three small kernels).
#include <cooperative_groups.h>

#include "common.cuh"

namespace cg = cooperative_groups;

namespace {

constexpr int BH_THREADS = 256;
constexpr int SORT_IPT = 8;                         // items per thread per tile in the scatter
constexpr int SORT_WARPS = BH_THREADS / 32;
constexpr int SORT_TILE = BH_THREADS * SORT_IPT;
constexpr int NPASS = 8;

struct BhState {                    // device-resident control block (first bytes of the workspace)
    unsigned long long n_cand;      // candidates appended so far / total after compaction
    unsigned long long n_ones, n_nan, n_valid;
    unsigned long long tau_key;     // keys >= tau_key are saturated (q = 1.0)
    long long n_tests;              // N
    double q_ones;                  // q of the p == 1.0 group
    double total_max;               // running max over all candidates
    int need_ones_fix;              // q_ones != 1.0 -> rewrite the ones
    int skip[NPASS];
    int use_list;                   // listed mode: K4's candidate list holds every candidate (saturation below BBK_SMALL_P)
};

struct BhLayout {
    BhState* st;
    long long* phist;               // [BBK_PHIST_BINS + 2]
    unsigned* block_hist;           // [256 * G]
    double* part_max;               // [G]
    long long* part_head;           // [G]
    unsigned long long* keys[2];    // [m] each
    unsigned* idx[2];               // [m] each
    int G;
};

size_t align256(size_t x) { return (x + 255) & ~(size_t)255; }

size_t bh_layout(void* base, long long m, int G, BhLayout* L) {
    size_t off = 0;
    char* b = (char*)base;
    auto take = [&](size_t bytes) { size_t o = off; off = align256(off + bytes); return b ? b + o : nullptr; };
    BhState* st = (BhState*)take(sizeof(BhState));
    long long* ph = (long long*)take(sizeof(long long) * (BBK_PHIST_BINS + 2));
    unsigned* bhist = (unsigned*)take(sizeof(unsigned) * 256 * (size_t)G);
    double* pm = (double*)take(sizeof(double) * (size_t)G);
    long long* phd = (long long*)take(sizeof(long long) * (size_t)G);
    unsigned long long* k0 = (unsigned long long*)take(sizeof(unsigned long long) * (size_t)m);
    unsigned long long* k1 = (unsigned long long*)take(sizeof(unsigned long long) * (size_t)m);
    unsigned* i0 = (unsigned*)take(sizeof(unsigned) * (size_t)m);
    unsigned* i1 = (unsigned*)take(sizeof(unsigned) * (size_t)m);
    if (L) { L->st = st; L->phist = ph; L->block_hist = bhist; L->part_max = pm; L->part_head = phd;
             L->keys[0] = k0; L->keys[1] = k1; L->idx[0] = i0; L->idx[1] = i1; L->G = G; }
    return off;
}

__device__ __forceinline__ unsigned long long key_of(double v) { return bbk_key_of(v); }
__device__ __forceinline__ double value_of(unsigned long long k) {
    unsigned long long b = (k >> 63) ? (k & 0x7fffffffffffffffull) : ~k;
    return __longlong_as_double((long long)b);
}
__device__ __forceinline__ int bucket_of(double v) {      // v >= 0, not NaN, != 1.0
    return (int)(((unsigned long long)__double_as_longlong(v) >> 51) & (BBK_PHIST_BINS - 1));
}

__global__ void bh_init_kernel(BhState* st, long long* phist, const long long* phist_in, long long n_tests) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < BBK_PHIST_BINS + 2) phist[i] = phist_in ? phist_in[i] : 0;
    if (i == 0) {
        st->n_cand = 0; st->n_ones = 0; st->n_nan = 0; st->n_valid = 0; st->tau_key = ~0ull;
        st->n_tests = n_tests; st->q_ones = 1.0; st->total_max = 0.0; st->need_ones_fix = 0;
        for (int p = 0; p < NPASS; ++p) st->skip[p] = 0;
        st->use_list = 0;
    }
}

// coarse histogram of p (only when K4 did not provide it): 8 B/pair read
__global__ void __launch_bounds__(BH_THREADS) bh_hist_kernel(const double* p, long long m, long long* phist) {
    __shared__ unsigned sh[BBK_PHIST_BINS];
    for (int i = threadIdx.x; i < BBK_PHIST_BINS; i += blockDim.x) sh[i] = 0;
    __syncthreads();
    unsigned ones = 0, nans = 0;
    long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < m; i += stride) {
        double v = ld_stream_double(p + i);
        if (isnan(v)) nans++;
        else if (v == 1.0) ones++;
        else if (v >= 0.0) atomicAdd(&sh[bucket_of(v)], 1u);
        else atomicAdd(&sh[0], 1u);                         // negative "p": smallest bucket (never saturates early)
    }
    __syncthreads();
    for (int i = threadIdx.x; i < BBK_PHIST_BINS; i += blockDim.x)
        if (sh[i]) atomicAdd((unsigned long long*)&phist[i], (unsigned long long)sh[i]);
    unsigned o = __reduce_add_sync(0xffffffffu, ones), z = __reduce_add_sync(0xffffffffu, nans);
    if ((threadIdx.x & 31) == 0) {
        if (o) atomicAdd((unsigned long long*)&phist[BBK_PHIST_BINS], (unsigned long long)o);
        if (z) atomicAdd((unsigned long long*)&phist[BBK_PHIST_BINS + 1], (unsigned long long)z);
    }
}

// one CTA of 1024 threads (4 buckets each): totals, N, and the saturation bucket
__device__ __forceinline__ void bh_threshold_body(BhState* st, const long long* phist, int prune, int listed, const BbkScoreState* ss) {
    __shared__ long long part[1024];
    __shared__ int first_bucket;
    const int t = threadIdx.x;
    long long h[4], loc = 0;
#pragma unroll
    for (int i = 0; i < 4; ++i) { h[i] = phist[4 * t + i]; loc += h[i]; }
    part[t] = loc;
    if (t == 0) first_bucket = BBK_PHIST_BINS;
    __syncthreads();
    for (int o = 1; o < 1024; o <<= 1) {
        long long v = t >= o ? part[t - o] : 0;
        __syncthreads();
        part[t] += v;
        __syncthreads();
    }
    const long long total = part[1023];
    const long long ones = phist[BBK_PHIST_BINS];
    long long n_tests = st->n_tests;
    if (n_tests < 0) n_tests = total + ones;                 // default N: the number of ranked p-values
    if (prune) {
        const double N = (double)n_tests;
        long long cum = part[t] - loc;                       // elements in buckets below 4t
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            int b = 4 * t + i;
            if (b > 0 && h[i] != 0) {                        // bucket 0 also holds negatives: never a threshold
                double v_lo = __longlong_as_double((long long)b << 51);
                // first element of the bucket: p >= v_lo, rank <= cum + 1.  Margin 2^-40 covers both roundings.
                if (v_lo * N >= (double)(cum + 1) * (1.0 + 9.1e-13)) atomicMin(&first_bucket, b);
            }
            cum += h[i];
        }
    }
    __syncthreads();
    if (t == 0) {
        st->n_ones = (unsigned long long)ones;
        st->n_nan = (unsigned long long)phist[BBK_PHIST_BINS + 1];
        st->n_valid = (unsigned long long)(total + ones);
        st->n_tests = n_tests;
        const unsigned long long tau = first_bucket < BBK_PHIST_BINS ? (((unsigned long long)first_bucket << 51) | 0x8000000000000000ull) : ~0ull;
        st->tau_key = tau;
        // listed mode: K4's list of the rows with p < BBK_SMALL_P stands in for the pass over p when it covers every candidate
        // (a candidate list that overflowed is no list: the full pass over p takes over)
        st->use_list = (listed && tau <= bbk_key_of(BBK_SMALL_P) && !(ss && ss->cand_overflow)) ? 1 : 0;
    }
}

__global__ void __launch_bounds__(1024) bh_threshold_kernel(BhState* st, const long long* phist, int prune, int listed,
                                                            const BbkScoreState* ss = nullptr) {
    bh_threshold_body(st, phist, prune, listed, ss);
}

// the 16 B/pair pass: q = 1.0 for saturated / p == 1.0 rows, NaN for NaN rows, candidates appended.  A CTA takes chunks of
// 1024 consecutive rows and reserves the places of a chunk's candidates with ONE global atomic (a warp-aggregated atomic
// per 32 rows was 2.3e7 same-address atomics on a 7.5e8-row shard with many candidates: 11 ms for a 2.5 ms pass).
__global__ void __launch_bounds__(BH_THREADS) bh_compact_kernel(const double* p, long long m, double* q, BhState* st,
                                                                unsigned long long* keys, unsigned* idx, int keep_ones,
                                                                long long* rank, long long key_cap = -1) {
    if (st->use_list) return;                                // K4 pre-filled q and listed every candidate
    __shared__ unsigned s_w[2][BH_THREADS / 32];
    __shared__ unsigned long long s_base[2];
    const unsigned long long tau = st->tau_key;
    const double qnan = __longlong_as_double(0x7ff8000000000000ll);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const long long chunk = (long long)BH_THREADS * 4;
    const long long n_chunks = (m + chunk - 1) / chunk;
    int par = 0;
    for (long long ch = blockIdx.x; ch < n_chunks; ch += gridDim.x, par ^= 1) {
        bool cand[4];
        unsigned long long k[4];
        unsigned cnt = 0;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const long long i = ch * chunk + (long long)j * BH_THREADS + tid;
            const bool live = i < m;
            const double v = live ? ld_stream_double(p + i) : qnan;
            const bool isn = isnan(v);
            k[j] = key_of(v);
            cand[j] = live && !isn && k[j] < tau && (keep_ones || v != 1.0);
            if (live && !cand[j]) { st_stream_double(q + i, isn ? qnan : 1.0); if (rank) rank[i] = 0; }
            cnt += cand[j];
        }
        unsigned inc = cnt;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned y = __shfl_up_sync(0xffffffffu, inc, o);
            if (lane >= o) inc += y;
        }
        if (lane == 31) s_w[par][warp] = inc;
        __syncthreads();
        if (tid == 0) {
            unsigned total = 0;
#pragma unroll
            for (int w = 0; w < BH_THREADS / 32; ++w) total += s_w[par][w];
            s_base[par] = total ? atomicAdd(&st->n_cand, (unsigned long long)total) : 0ull;
        }
        __syncthreads();
        unsigned woff = 0;
#pragma unroll
        for (int w = 0; w < BH_THREADS / 32; ++w) woff += w < warp ? s_w[par][w] : 0u;
        unsigned long long pos = s_base[par] + woff + inc - cnt;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            if (cand[j]) {
                if (key_cap < 0 || (long long)pos < key_cap) {       // a fixed-capacity send block: the count still says how many there were
                    keys[pos] = k[j];
                    idx[pos] = (unsigned)(ch * chunk + (long long)j * BH_THREADS + tid);
                }
                pos += 1;
            }
        }
    }
}

// listed mode (bbk_score_pairs): the rows with p < BBK_SMALL_P are already a list of (key, row); keep those below tau.
// One global atomic per CTA step of 1024 entries (a warp-aggregated one per 32 was 1.5e5 same-address atomics on BASELINE
// config 3: 0.27 ms for a 0.05 ms pass).
__global__ void __launch_bounds__(BH_THREADS) bh_cand_filter_kernel(BhState* st, const BbkScoreState* ss, const unsigned long long* ckeys,
                                                                    const unsigned* crows, unsigned long long* keys, unsigned* idx,
                                                                    long long key_cap = -1) {
    if (!st->use_list) return;
    __shared__ unsigned s_w[2][BH_THREADS / 32];
    __shared__ unsigned long long s_base[2];
    const unsigned long long tau = st->tau_key;
    const long long n = (long long)ss->n_cand;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const long long chunk = (long long)BH_THREADS * 4;
    const long long n_chunks = (n + chunk - 1) / chunk;
    int par = 0;
    for (long long ch = blockIdx.x; ch < n_chunks; ch += gridDim.x, par ^= 1) {
        unsigned long long k[4];
        bool cand[4];
        unsigned cnt = 0;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const long long i = ch * chunk + (long long)j * BH_THREADS + tid;
            k[j] = i < n ? ckeys[i] : ~0ull;
            cand[j] = i < n && k[j] < tau;
            cnt += cand[j];
        }
        unsigned inc = cnt;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned y = __shfl_up_sync(0xffffffffu, inc, o);
            if (lane >= o) inc += y;
        }
        if (lane == 31) s_w[par][warp] = inc;
        __syncthreads();
        if (tid == 0) {
            unsigned total = 0;
#pragma unroll
            for (int w = 0; w < BH_THREADS / 32; ++w) total += s_w[par][w];
            s_base[par] = total ? atomicAdd(&st->n_cand, (unsigned long long)total) : 0ull;
        }
        __syncthreads();
        unsigned woff = 0;
#pragma unroll
        for (int w = 0; w < BH_THREADS / 32; ++w) woff += w < warp ? s_w[par][w] : 0u;
        unsigned long long pos = s_base[par] + woff + inc - cnt;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            if (cand[j]) {
                if (key_cap < 0 || (long long)pos < key_cap) { keys[pos] = k[j]; idx[pos] = crows[ch * chunk + (long long)j * BH_THREADS + tid]; }
                pos += 1;
            }
        }
    }
}

__device__ __forceinline__ int sort_parity(const BhState* st, int pass) {
    int par = 0;
    for (int p = 0; p < pass; ++p) par ^= (st->skip[p] ? 0 : 1);
    return par;
}

struct Chunk { long long lo, hi; };
// block columns actually used for n elements: at least one tile per block, at most G
__device__ __forceinline__ int eff_blocks(long long n, int G) {
    long long g = (n + SORT_TILE - 1) / SORT_TILE;
    if (g < 1) g = 1;
    return g < G ? (int)g : G;
}
__device__ __forceinline__ Chunk chunk_of(long long n, int G, int b) {
    G = eff_blocks(n, G);
    if (b >= G) { Chunk e; e.lo = e.hi = n; return e; }
    long long per = (n + G - 1) / G;
    per = (per + SORT_TILE - 1) / SORT_TILE * SORT_TILE;     // whole tiles per block
    Chunk c;
    c.lo = (long long)b * per;
    c.hi = c.lo + per;
    if (c.lo > n) c.lo = n;
    if (c.hi > n) c.hi = n;
    return c;
}

// ---- running max over the sorted candidates --------------------------------------------------
// element i contributes (value, head): value = head ? min((p*N)/(i+1), 1) : -inf ; head index = i or -1
struct ScanParams {
    BhLayout L;
    const double* p_in;      // positional mode: the input p (no keys)
    long long m;             // positional mode length
    double* q;               // output (input order)
    long long* rank;         // optional
    int positional;
};

__device__ __forceinline__ void scan_elem(const ScanParams& S, const unsigned long long* keys, long long i, double N,
                                          double& val, long long& head, bool& reset) {
    reset = false;
    if (S.positional) {
        double pv = S.p_in[i];
        double bh = (pv * N) / (double)(i + 1);              // two roundings, as fithic.py:474 / blueberry.pyx:68
        bh = (1.0 < bh) ? 1.0 : bh;                          // min(bh, 1): NaN stays NaN
        val = bh;
        head = i;
        reset = isnan(bh);                                   // max(nan, prev) = nan, and the chain restarts after it
        return;
    }
    unsigned long long k = keys[i];
    bool is_head = (i == 0) || (keys[i - 1] != k);
    if (is_head) {
        double bh = (value_of(k) * N) / (double)(i + 1);
        val = (1.0 < bh) ? 1.0 : bh;
        head = i;
    } else {
        val = -INFINITY;
        head = -1;
    }
}

// combine for the (segmented) running max: right operand wins a reset
struct MaxSeg { double v; long long h; int reset; };
__device__ __forceinline__ MaxSeg seg_combine(const MaxSeg& a, const MaxSeg& b) {
    MaxSeg r;
    if (b.reset) { r = b; return r; }
    r.reset = a.reset;
    r.v = (a.v > b.v) ? a.v : b.v;                           // prev wins only when strictly greater (reference's max)
    r.h = a.h > b.h ? a.h : b.h;
    return r;
}

__global__ void __launch_bounds__(BH_THREADS) scan_partial_kernel(ScanParams S) {
    __shared__ MaxSeg red[BH_THREADS];
    const BhState* st = S.L.st;
    const long long n = S.positional ? S.m : (long long)st->n_cand;
    const double N = (double)st->n_tests;
    const unsigned long long* keys = S.positional ? nullptr : S.L.keys[sort_parity(st, NPASS)];
    Chunk c = chunk_of(n, S.L.G, blockIdx.x);
    // thread t scans a contiguous slice of the chunk so that order is preserved
    long long len = c.hi - c.lo, per = (len + blockDim.x - 1) / blockDim.x;
    long long lo = c.lo + (long long)threadIdx.x * per, hi = lo + per;
    if (lo > c.hi) lo = c.hi;
    if (hi > c.hi) hi = c.hi;
    MaxSeg acc = {-INFINITY, -1, 0};
    for (long long i = lo; i < hi; ++i) {
        MaxSeg e; bool rs;
        scan_elem(S, keys, i, N, e.v, e.h, rs);
        e.reset = rs ? 1 : 0;
        if (rs) e.v = -INFINITY;                             // after a NaN the chain restarts from nothing
        acc = seg_combine(acc, e);
    }
    red[threadIdx.x] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        MaxSeg r = red[0];
        for (int t = 1; t < BH_THREADS; ++t) r = seg_combine(r, red[t]);
        S.L.part_max[blockIdx.x] = r.v;
        S.L.part_head[blockIdx.x] = r.h * 2 + r.reset;       // pack reset flag in the low bit
    }
}

__device__ __forceinline__ MaxSeg seg_shfl_up(const MaxSeg& a, int o) {
    MaxSeg r;
    r.v = __shfl_up_sync(0xffffffffu, a.v, o);
    r.h = __shfl_up_sync(0xffffffffu, a.h, o);
    r.reset = __shfl_up_sync(0xffffffffu, a.reset, o);
    return r;
}

__global__ void scan_prefix_kernel(ScanParams S) {           // one warp: exclusive prefix over the G block partials
    if (blockIdx.x != 0 || threadIdx.x >= 32) return;
    BhState* st = S.L.st;
    const int lane = threadIdx.x, G = S.L.G;
    const int per = (G + 31) / 32, lo = lane * per, hi = min(lo + per, G);
    const MaxSeg ident = {-INFINITY, -1, 0};
    MaxSeg loc = ident;
    for (int b = lo; b < hi; ++b) {
        MaxSeg e = {S.L.part_max[b], S.L.part_head[b] >> 1, (int)(S.L.part_head[b] & 1)};
        loc = seg_combine(loc, e);
    }
    MaxSeg inc = loc;                                        // inclusive scan over lanes
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        MaxSeg up = seg_shfl_up(inc, o);
        if (lane >= o) inc = seg_combine(up, inc);
    }
    MaxSeg run = seg_shfl_up(inc, 1);
    if (lane == 0) run = ident;
    for (int b = lo; b < hi; ++b) {
        MaxSeg e = {S.L.part_max[b], S.L.part_head[b] >> 1, (int)(S.L.part_head[b] & 1)};
        S.L.part_max[b] = run.v;                             // exclusive prefix
        S.L.part_head[b] = run.h;
        run = seg_combine(run, e);
    }
    MaxSeg all;
    all.v = __shfl_sync(0xffffffffu, inc.v, 31);
    all.h = __shfl_sync(0xffffffffu, inc.h, 31);
    all.reset = __shfl_sync(0xffffffffu, inc.reset, 31);
    if (lane == 0 && !S.positional) {
        st->total_max = all.v;
        // the p == 1.0 group: one tie group after every candidate (when nothing saturated before it)
        double N = (double)st->n_tests;
        double bh = (1.0 * N) / (double)(st->n_cand + 1);
        bh = (1.0 < bh) ? 1.0 : bh;
        double qo = (all.v > bh) ? all.v : bh;
        if (st->tau_key != ~0ull) qo = 1.0;                  // saturated before the ones
        st->q_ones = qo;
        st->need_ones_fix = (qo != 1.0 && st->n_ones > 0) ? 1 : 0;
    }
}

__global__ void __launch_bounds__(BH_THREADS) scan_apply_kernel(ScanParams S) {
    __shared__ MaxSeg red[BH_THREADS];
    const BhState* st = S.L.st;
    const long long n = S.positional ? S.m : (long long)st->n_cand;
    const double N = (double)st->n_tests;
    const int par = S.positional ? 0 : sort_parity(st, NPASS);
    const unsigned long long* keys = S.positional ? nullptr : S.L.keys[par];
    const unsigned* idx = S.positional ? nullptr : S.L.idx[par];
    Chunk c = chunk_of(n, S.L.G, blockIdx.x);
    long long len = c.hi - c.lo, per = (len + blockDim.x - 1) / blockDim.x;
    long long lo = c.lo + (long long)threadIdx.x * per, hi = lo + per;
    if (lo > c.hi) lo = c.hi;
    if (hi > c.hi) hi = c.hi;
    MaxSeg acc = {-INFINITY, -1, 0};
    for (long long i = lo; i < hi; ++i) {
        MaxSeg e; bool rs;
        scan_elem(S, keys, i, N, e.v, e.h, rs);
        e.reset = rs ? 1 : 0;
        if (rs) e.v = -INFINITY;
        acc = seg_combine(acc, e);
    }
    red[threadIdx.x] = acc;
    __syncthreads();
    // exclusive prefix over threads (sequential by thread 0: 256 combines), seeded with the block prefix
    if (threadIdx.x == 0) {
        MaxSeg run = {S.L.part_max[blockIdx.x], S.L.part_head[blockIdx.x], 0};
        for (int t = 0; t < BH_THREADS; ++t) { MaxSeg e = red[t]; red[t] = run; run = seg_combine(run, e); }
    }
    __syncthreads();
    MaxSeg run = red[threadIdx.x];
    const double qnan = __longlong_as_double(0x7ff8000000000000ll);
    for (long long i = lo; i < hi; ++i) {
        MaxSeg e; bool rs;
        scan_elem(S, keys, i, N, e.v, e.h, rs);
        e.reset = rs ? 1 : 0;
        if (rs) e.v = -INFINITY;
        run = seg_combine(run, e);
        double qv = rs ? qnan : run.v;
        if (S.positional) {
            S.q[i] = qv;
            if (S.rank) S.rank[i] = i + 1;
        } else {
            unsigned o = idx[i];
            S.q[o] = qv;
            if (S.rank) S.rank[o] = run.h + 1;
        }
    }
}

// ---- the candidates' ranking in one cooperative launch ---------------------------------------------
// One CTA of 1024 threads per SM; CTA b owns a contiguous chunk of whole tiles.  Per radix pass:
//   count the chunk's digits -> table[b][256] | grid barrier | every active CTA sums the table's columns itself
//   (its own prefix over earlier CTAs + the digit totals: no scan CTA, no extra barrier), then scatters its tiles
//   in order, ranking equal digits inside a warp with match_any (stable) | grid barrier.
// Then the forward running max over the sorted keys: chunk partials | grid barrier | prefix over earlier CTAs + apply.
constexpr int RK_THREADS = 1024;
constexpr int RK_WARPS = RK_THREADS / 32;
constexpr int RK_IPT = 4;
constexpr int RK_TILE = RK_THREADS * RK_IPT;
constexpr size_t RK_DYN_SMEM = (size_t)RK_TILE * (sizeof(unsigned long long) + sizeof(unsigned));   // the staged tile

struct RankParams {
    BhLayout L;
    double* q;               // output (input order, or gathered order for bbk_bh_rank_gathered_padded)
    long long* rank;         // optional
    long long n_host;        // >= 0: number of (key, index) pairs, known to the host; < 0: BhState::n_cand
    int src;                 // buffer (0 / 1) the pairs start in; a sort-only launch leaves the result there
    // segmented ranking (bbk_bh_qvalues_segmented): the index is a row, row r belongs to the segment s with
    // seg_off[s] <= r < seg_off[s + 1]; seg[s] is that segment's state, seg_start[s] where its candidates start once sorted
    const long long* seg_off;
    BhState* seg;
    unsigned long long* seg_start;
    int n_seg;
    int seg_passes;          // extra stable digit passes keyed on the segment: 1 up to 256 segments, 2 above
};

__device__ __forceinline__ int seg_of(const long long* off, int n_seg, unsigned row) {     // last s with off[s] <= row
    int lo = 0, hi = n_seg - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (__ldg(off + mid) <= (long long)row) lo = mid; else hi = mid - 1;
    }
    return lo;
}

// radix digit of pass `pass`: the 8 bytes of the key, then (segmented) the bytes of the row's segment
template <bool SEG>
__device__ __forceinline__ unsigned rk_digit(const RankParams& R, unsigned long long key, unsigned val, int pass) {
    if (SEG && pass >= NPASS) return ((unsigned)seg_of(R.seg_off, R.n_seg, val) >> (8 * (pass - NPASS))) & 255u;
    return (unsigned)(key >> (8 * pass)) & 255u;
}

__device__ __forceinline__ int rk_eff_blocks(long long n, int G) {
    long long g = (n + RK_TILE - 1) / RK_TILE;
    if (g < 1) g = 1;
    return g < G ? (int)g : G;
}
__device__ __forceinline__ Chunk rk_chunk(long long n, int Ge, int b) {
    Chunk c;
    if (b >= Ge) { c.lo = c.hi = n; return c; }
    long long per = (n + Ge - 1) / Ge;
    per = (per + RK_TILE - 1) / RK_TILE * RK_TILE;
    c.lo = (long long)b * per;
    c.hi = c.lo + per;
    if (c.lo > n) c.lo = n;
    if (c.hi > n) c.hi = n;
    return c;
}

// (running max, index of the last tie-group head): max in both fields, identity (-inf, -1)
struct MaxHead { double v; long long h; };
__device__ __forceinline__ MaxHead mh_combine(const MaxHead& a, const MaxHead& b) {
    MaxHead r;
    r.v = (a.v > b.v) ? a.v : b.v;
    r.h = a.h > b.h ? a.h : b.h;
    return r;
}
// segmented: h = where the element's segment starts; a later segment discards what came before it
__device__ __forceinline__ MaxHead mh_combine_seg(const MaxHead& a, const MaxHead& b) {
    if (b.h > a.h) return b;
    MaxHead r;
    r.v = (a.v > b.v) ? a.v : b.v;
    r.h = a.h;
    return r;
}
template <bool SEG>
__device__ __forceinline__ MaxHead mh_comb(const MaxHead& a, const MaxHead& b) { return SEG ? mh_combine_seg(a, b) : mh_combine(a, b); }
// element i of the sorted candidates of a segmented ranking: rank and N are its segment's, and a tie group never spans a segment
// boundary (fithic.py:473-485 inside every segment)
__device__ __forceinline__ MaxHead mh_elem_seg(const RankParams& R, const unsigned long long* keys, const unsigned* idx, long long i) {
    const int s = seg_of(R.seg_off, R.n_seg, idx[i]);
    const long long start = (long long)R.seg_start[s];
    const unsigned long long k = keys[i];
    MaxHead e;
    e.h = start;
    if (i == start || keys[i - 1] != k) {
        double bh = (value_of(k) * (double)R.seg[s].n_tests) / (double)(i - start + 1);
        e.v = (1.0 < bh) ? 1.0 : bh;
    } else e.v = -INFINITY;
    return e;
}
__device__ __forceinline__ MaxHead mh_elem(const unsigned long long* keys, long long i, double N) {
    MaxHead e;
    const unsigned long long k = keys[i];
    if (i == 0 || keys[i - 1] != k) {
        double bh = (value_of(k) * N) / (double)(i + 1);     // two roundings, as fithic.py:474 / blueberry.pyx:68
        e.v = (1.0 < bh) ? 1.0 : bh;
        e.h = i;
    } else { e.v = -INFINITY; e.h = -1; }
    return e;
}

template <bool SCAN, bool SEG>
__global__ void __launch_bounds__(RK_THREADS, 1) bh_rank_kernel(RankParams R) {
    cg::grid_group grid = cg::this_grid();
    __shared__ unsigned base[256];                   // digit counts of the chunk, then the running output cursor per digit
    __shared__ unsigned col_pre[4][256], col_tot[4][256];
    __shared__ unsigned wsum[8];
    __shared__ unsigned whist[RK_WARPS][256];
    __shared__ int sh_skip;
    __shared__ double wv[RK_WARPS];
    __shared__ long long wh[RK_WARPS];
    __shared__ unsigned gstart[256], tstart[256];    // per digit: global position / staged position of the tile's run
    extern __shared__ __align__(16) unsigned char rk_dyn[];
    unsigned long long* skeys = reinterpret_cast<unsigned long long*>(rk_dyn);               // [RK_TILE] the tile in digit order
    unsigned* svals = reinterpret_cast<unsigned*>(rk_dyn + (size_t)RK_TILE * sizeof(unsigned long long));
    BhState* st = R.L.st;
    const long long n = R.n_host >= 0 ? R.n_host : (long long)st->n_cand;
    const int b = blockIdx.x, Ge = rk_eff_blocks(n, gridDim.x);
    const bool active = b < Ge;
    const Chunk c = rk_chunk(n, Ge, b);
    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
    unsigned* table = R.L.block_hist;                // [Ge][256]
    int par = R.src;
    if (SEG && b == 0 && t == 0) {                   // where every segment's candidates start once sorted (published by the first grid.sync)
        unsigned long long run = 0;
        for (int s = 0; s < R.n_seg; ++s) { R.seg_start[s] = run; run += R.seg[s].n_cand; }
    }
    for (int pass = 0; pass < NPASS + (SEG ? R.seg_passes : 0); ++pass) {
        const unsigned long long* kin = R.L.keys[par];
        if (active) {
            if (t < 256) base[t] = 0;
            if (t == 0) sh_skip = 0;
            __syncthreads();
            for (long long i = c.lo + t; i < c.hi; i += RK_THREADS)
                atomicAdd(&base[rk_digit<SEG>(R, kin[i], SEG ? R.L.idx[par][i] : 0u, pass)], 1u);
            __syncthreads();
            if (t < 256) table[(size_t)b * 256 + t] = base[t];
        }
        grid.sync();
        if (active) {
            {   // column sums of the table: thread (part, d) takes every 4th CTA row
                const int d = t & 255, part = t >> 8;
                unsigned pre = 0, tot = 0;
                for (int bb = part; bb < Ge; bb += 4) {
                    unsigned v = table[(size_t)bb * 256 + d];
                    tot += v;
                    if (bb < b) pre += v;
                }
                col_pre[part][d] = pre; col_tot[part][d] = tot;
            }
            __syncthreads();
            unsigned pre = 0, tot = 0, x = 0;
            if (t < 256) {
                pre = col_pre[0][t] + col_pre[1][t] + col_pre[2][t] + col_pre[3][t];
                tot = col_tot[0][t] + col_tot[1][t] + col_tot[2][t] + col_tot[3][t];
                if ((long long)tot == n) sh_skip = 1;                    // every key has this digit: nothing moves
                x = tot;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) { unsigned y = __shfl_up_sync(0xffffffffu, x, o); if (lane >= o) x += y; }
                if (lane == 31) wsum[warp] = x;
            }
            __syncthreads();
            if (t < 256) {
                unsigned before = 0;
                for (int w = 0; w < warp; ++w) before += wsum[w];
                base[t] = before + x - tot + pre;                        // digits below + same digit in earlier CTAs
            }
            __syncthreads();
            const bool skip = sh_skip != 0;
            if (t == 0 && b == 0 && (!SEG || pass < NPASS)) st->skip[pass] = skip ? 1 : 0;
            if (!skip) {
                const unsigned* iin = R.L.idx[par];
                unsigned long long* kout = R.L.keys[par ^ 1];
                unsigned* iout = R.L.idx[par ^ 1];
                for (long long tile = c.lo; tile < c.hi; tile += RK_TILE) {
                    for (int d = lane; d < 256; d += 32) whist[warp][d] = 0;
                    __syncwarp();
                    unsigned long long key[RK_IPT];
                    unsigned val[RK_IPT], loc[RK_IPT];
                    const long long wbase = tile + (long long)warp * (32 * RK_IPT);
#pragma unroll
                    for (int it = 0; it < RK_IPT; ++it) {
                        const long long i = wbase + it * 32 + lane;
                        const bool live = i < c.hi;
                        key[it] = live ? kin[i] : 0;
                        val[it] = live ? iin[i] : 0;
                    }
#pragma unroll
                    for (int it = 0; it < RK_IPT; ++it) {
                        const bool live = wbase + it * 32 + lane < c.hi;
                        const unsigned dg = live ? rk_digit<SEG>(R, key[it], val[it], pass) : 256u;
                        const unsigned peers = __match_any_sync(0xffffffffu, dg);
                        const unsigned rk = __popc(peers & ((1u << lane) - 1));
                        const unsigned before = live ? whist[warp][dg] : 0;
                        __syncwarp();
                        if (live && rk == 0) whist[warp][dg] = before + __popc(peers);
                        __syncwarp();
                        loc[it] = before + rk;
                    }
                    __syncthreads();
                    // The tile leaves through shared memory in digit order: a digit's elements of this tile are one contiguous run
                    // in the output, so consecutive threads write consecutive addresses (scattering straight from registers
                    // touched up to 32 sectors per warp store for 8-byte elements).
                    unsigned cnt = 0, x = 0;
                    if (t < 256) {   // per digit: the warps' shares become offsets inside the tile's run; advance the CTA's cursor
                        const unsigned run = base[t];
                        gstart[t] = run;
#pragma unroll 8
                        for (int w = 0; w < RK_WARPS; ++w) { unsigned v = whist[w][t]; whist[w][t] = cnt; cnt += v; }
                        base[t] = run + cnt;
                        x = cnt;
#pragma unroll
                        for (int o = 1; o < 32; o <<= 1) { unsigned y = __shfl_up_sync(0xffffffffu, x, o); if (lane >= o) x += y; }
                        if (lane == 31) wsum[warp] = x;
                    }
                    __syncthreads();
                    if (t < 256) {
                        unsigned before = 0;
                        for (int w = 0; w < warp; ++w) before += wsum[w];
                        tstart[t] = before + x - cnt;                    // where the digit's run starts inside the staged tile
                    }
                    __syncthreads();
#pragma unroll
                    for (int it = 0; it < RK_IPT; ++it) {
                        if (wbase + it * 32 + lane < c.hi) {
                            const unsigned dg = rk_digit<SEG>(R, key[it], val[it], pass);
                            const unsigned lp = tstart[dg] + whist[warp][dg] + loc[it];
                            skeys[lp] = key[it];
                            svals[lp] = val[it];
                        }
                    }
                    __syncthreads();
                    const long long left = c.hi - tile;
                    const int n_tile = left < RK_TILE ? (int)left : RK_TILE;
                    for (int k = t; k < n_tile; k += RK_THREADS) {
                        const unsigned long long kk = skeys[k];
                        const unsigned vv = svals[k];
                        const unsigned dg = rk_digit<SEG>(R, kk, vv, pass);
                        const unsigned pos = gstart[dg] + ((unsigned)k - tstart[dg]);
                        kout[pos] = kk;
                        iout[pos] = vv;
                    }
                    __syncthreads();
                }
                par ^= 1;
            }
        }
        grid.sync();
    }

    if (!SCAN) {
        // sort only (bbk_decimate): the caller finds the sorted pairs where it put the unsorted ones
        int fin = R.src;
        for (int ps = 0; ps < NPASS; ++ps) fin ^= (st->skip[ps] ? 0 : 1);      // inactive CTAs did not follow the flips
        par = fin;
        if (par != R.src) {
            const long long stride = (long long)gridDim.x * RK_THREADS;
            for (long long i = (long long)b * RK_THREADS + t; i < n; i += stride) { R.L.keys[R.src][i] = R.L.keys[par][i]; R.L.idx[R.src][i] = R.L.idx[par][i]; }
        }
        return;
    }
    // ---- forward running max over the sorted keys; thread t scans a contiguous slice of the chunk
    const unsigned long long* keys = R.L.keys[par];
    const unsigned* idx = R.L.idx[par];
    const double N = (double)st->n_tests;
    const MaxHead ident = {-INFINITY, -1};
    long long lo = c.lo, hi = c.lo;
    MaxHead excl = ident;                            // everything before this thread's slice, inside the chunk
    if (active) {
        const long long len = c.hi - c.lo, per = (len + RK_THREADS - 1) / RK_THREADS;
        lo = c.lo + (long long)t * per; hi = lo + per;
        if (lo > c.hi) lo = c.hi;
        if (hi > c.hi) hi = c.hi;
        MaxHead acc = ident;
        for (long long i = lo; i < hi; ++i) acc = mh_comb<SEG>(acc, SEG ? mh_elem_seg(R, keys, idx, i) : mh_elem(keys, i, N));
        MaxHead inc = acc;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            MaxHead up;
            up.v = __shfl_up_sync(0xffffffffu, inc.v, o);
            up.h = __shfl_up_sync(0xffffffffu, inc.h, o);
            if (lane >= o) inc = mh_comb<SEG>(up, inc);
        }
        if (lane == 31) { wv[warp] = inc.v; wh[warp] = inc.h; }
        excl.v = __shfl_up_sync(0xffffffffu, inc.v, 1);
        excl.h = __shfl_up_sync(0xffffffffu, inc.h, 1);
        if (lane == 0) excl = ident;
        __syncthreads();
        MaxHead wpre = ident;
        for (int w = 0; w < warp; ++w) { MaxHead e = {wv[w], wh[w]}; wpre = mh_comb<SEG>(wpre, e); }
        excl = mh_comb<SEG>(wpre, excl);
        if (t == RK_THREADS - 1) {
            MaxHead all = mh_comb<SEG>(excl, acc);
            R.L.part_max[b] = all.v;
            R.L.part_head[b] = all.h;
        }
    }
    grid.sync();
    if (active) {
        MaxHead run = ident;                         // chunks of the earlier CTAs
        if (SEG) {      // CTAs in order: the lanes' strided partials are combined in CTA order below
            MaxHead ordered = ident;
            if (lane == 0)
                for (int bb = 0; bb < b; ++bb) { MaxHead e = {R.L.part_max[bb], R.L.part_head[bb]}; ordered = mh_combine_seg(ordered, e); }
            run.v = __shfl_sync(0xffffffffu, ordered.v, 0);
            run.h = __shfl_sync(0xffffffffu, ordered.h, 0);
        } else {
            for (int bb = lane; bb < b; bb += 32) { MaxHead e = {R.L.part_max[bb], R.L.part_head[bb]}; run = mh_combine(run, e); }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                MaxHead other;
                other.v = __shfl_xor_sync(0xffffffffu, run.v, o);
                other.h = __shfl_xor_sync(0xffffffffu, run.h, o);
                run = mh_combine(run, other);
            }
        }
        run = mh_comb<SEG>(run, excl);
        for (long long i = lo; i < hi; ++i) {
            if (SEG) {
                run = mh_combine_seg(run, mh_elem_seg(R, keys, idx, i));
                const unsigned o = idx[i];
                R.q[o] = run.v;
                const int s = seg_of(R.seg_off, R.n_seg, o);
                if ((unsigned long long)i + 1 == R.seg_start[s] + R.seg[s].n_cand) R.seg[s].total_max = run.v;   // the segment's last candidate
            } else {
                run = mh_combine(run, mh_elem(keys, i, N));
                const unsigned o = idx[i];
                R.q[o] = run.v;
                if (R.rank) R.rank[o] = run.h + 1;
            }
        }
    }
    if (!SEG && b == 0 && warp == 0) {                       // the p == 1.0 group: one tie group after every candidate
        MaxHead all = ident;
        for (int bb = lane; bb < Ge; bb += 32) { MaxHead e = {R.L.part_max[bb], R.L.part_head[bb]}; all = mh_combine(all, e); }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            MaxHead other;
            other.v = __shfl_xor_sync(0xffffffffu, all.v, o);
            other.h = __shfl_xor_sync(0xffffffffu, all.h, o);
            all = mh_combine(all, other);
        }
        if (lane == 0) {
            st->total_max = all.v;
            double bh = (1.0 * N) / (double)(st->n_cand + 1);
            bh = (1.0 < bh) ? 1.0 : bh;
            double qo = (all.v > bh) ? all.v : bh;
            if (st->tau_key != ~0ull) qo = 1.0;      // saturated before the ones
            st->q_ones = qo;
            st->need_ones_fix = (qo != 1.0 && st->n_ones > 0) ? 1 : 0;
        }
    }
}

int rank_grid() {            // CTAs of bh_rank_kernel that are resident together (cooperative launch): one per SM
    static int g = 0;
    if (g == 0) {
        int per_sm = 0;
        if (cudaFuncSetAttribute(bh_rank_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)RK_DYN_SMEM) != cudaSuccess) return 0;
        if (cudaFuncSetAttribute(bh_rank_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)RK_DYN_SMEM) != cudaSuccess) return 0;
        if (cudaFuncSetAttribute(bh_rank_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)RK_DYN_SMEM) != cudaSuccess) return 0;
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, bh_rank_kernel<true, false>, RK_THREADS, RK_DYN_SMEM) != cudaSuccess || per_sm < 1) return 0;
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, bh_rank_kernel<true, true>, RK_THREADS, RK_DYN_SMEM) != cudaSuccess || per_sm < 1) return 0;
        g = bbk_num_sms();
    }
    return g;
}

int launch_rank(const BhLayout& L, double* q, long long* rank, cudaStream_t st) {
    int g = rank_grid();
    if (g <= 0 || g > L.G) { bbk_set_error("bh_rank_kernel: cooperative launch not possible on this device"); return BBK_E_CUDA; }
    RankParams R = {};
    R.L = L; R.q = q; R.rank = rank; R.n_host = -1; R.src = 0;
    void* args[] = {&R};
    cudaError_t e = cudaLaunchCooperativeKernel((const void*)bh_rank_kernel<true, false>, dim3(g), dim3(RK_THREADS), args, RK_DYN_SMEM, st);
    if (e != cudaSuccess) { bbk_set_error("bh_rank_kernel: %s", cudaGetErrorString(e)); return BBK_E_CUDA; }
    return BBK_OK;
}

}  // namespace

// ---- the radix sort alone, for the other kernels of the library (decimate.cu): stable LSD sort of n (u64 key, u32 value)
// pairs that sit in buffer `src` of a workspace laid out by bbk_bh_workspace_bytes(capacity); the result is left in the
// same buffer.  n_host < 0: the count is BhState::n_cand (device), see bbk_sort_count_ptr.
void bbk_sort_buffers(void* workspace, long long capacity, int which, unsigned long long** keys, unsigned** idx) {
    BhLayout L;
    bh_layout(workspace, capacity, bbk_num_sms() * 4 > 1024 ? 1024 : bbk_num_sms() * 4, &L);
    *keys = L.keys[which];
    *idx = L.idx[which];
}
unsigned long long* bbk_sort_count_ptr(void* workspace) { return &((BhState*)workspace)->n_cand; }
int bbk_sort_pairs(void* workspace, long long capacity, long long n_host, int src, cudaStream_t st) {
    int g = rank_grid();
    BhLayout L;
    bh_layout(workspace, capacity, bbk_num_sms() * 4 > 1024 ? 1024 : bbk_num_sms() * 4, &L);
    if (g <= 0 || g > L.G) { bbk_set_error("bbk_sort_pairs: cooperative launch not possible on this device"); return BBK_E_CUDA; }
    RankParams R = {};
    R.L = L; R.q = nullptr; R.rank = nullptr; R.n_host = n_host; R.src = src;
    void* args[] = {&R};
    cudaError_t e = cudaLaunchCooperativeKernel((const void*)bh_rank_kernel<false, false>, dim3(g), dim3(RK_THREADS), args, RK_DYN_SMEM, st);
    if (e != cudaSuccess) { bbk_set_error("bbk_sort_pairs: %s", cudaGetErrorString(e)); return BBK_E_CUDA; }
    return BBK_OK;
}

namespace {

// rare: q of the p == 1.0 group is below 1 (N smaller than the number of candidates)
__global__ void __launch_bounds__(BH_THREADS) ones_fix_kernel(const double* p, long long m, double* q, const BhState* st) {
    if (!st->need_ones_fix) return;
    const double qo = st->q_ones;
    long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < m; i += stride)
        if (p[i] == 1.0) q[i] = qo;
}

// ---- genome-wide (multi-GPU) variant: select locally, rank the gathered candidates, scatter back -----
__global__ void export_state_kernel(const BhState* st, unsigned long long* out) {
    out[0] = st->n_cand; out[1] = st->tau_key; out[2] = (unsigned long long)st->n_tests; out[3] = st->n_ones;
}

__global__ void export_ones_kernel(const BhState* st, double* out) { out[0] = st->q_ones; out[1] = st->need_ones_fix ? 1.0 : 0.0; }

__global__ void __launch_bounds__(BH_THREADS) fix_ones_dev_kernel(const double* p, long long m, double* q, const double* q_ones) {
    if (q_ones[1] == 0.0) return;                           // q(p == 1) is 1.0: nothing to do
    const double qo = q_ones[0];
    long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < m; i += stride)
        if (p[i] == 1.0) q[i] = qo;
}

int sort_blocks() { int g = bbk_num_sms() * 4; return g > 1024 ? 1024 : g; }

}  // namespace

extern "C" size_t bbk_bh_workspace_bytes(int64_t m) {
    if (m < 0) return 0;
    return bh_layout(nullptr, m, sort_blocks(), nullptr) + 256;
}

extern "C" int bbk_bh_qvalues(const double* d_p, int64_t m, int64_t n_tests, int32_t mode, const int64_t* d_p_hist,
                              double* d_q, int64_t* d_rank, void* d_workspace, size_t workspace_bytes, void* stream) {
    BBK_REQUIRE(m >= 0 && m < (1ll << 32), "bbk_bh_qvalues: m must be in [0, 2^32)");
    BBK_REQUIRE(mode == BBK_BH_UNSORTED || mode == BBK_BH_POSITIONAL, "bbk_bh_qvalues: unknown mode");
    if (m == 0) return BBK_OK;
    BBK_REQUIRE(d_p && d_q && d_workspace, "bbk_bh_qvalues: null pointer");
    BBK_REQUIRE(((uintptr_t)d_workspace & 255) == 0, "bbk_bh_qvalues: workspace must be 256-byte aligned");
    const int G = sort_blocks();
    BhLayout L;
    size_t need = bh_layout(d_workspace, m, G, &L);
    if (workspace_bytes < need) {
        bbk_set_error("bbk_bh_qvalues: workspace too small (%zu < %zu bytes)", workspace_bytes, need);
        return BBK_E_WORKSPACE;
    }
    cudaStream_t st = (cudaStream_t)stream;
    const int sms = bbk_num_sms();
    bh_init_kernel<<<(BBK_PHIST_BINS + 2 + 255) / 256, 256, 0, st>>>(L.st, L.phist, (const long long*)d_p_hist,
                                                                     mode == BBK_BH_POSITIONAL && n_tests < 0 ? m : n_tests);
    BBK_CHECK_LAUNCH("bh_init_kernel");
    ScanParams S;
    S.L = L; S.p_in = d_p; S.m = m; S.q = d_q; S.rank = (long long*)d_rank; S.positional = mode == BBK_BH_POSITIONAL;
    if (mode == BBK_BH_UNSORTED) {
        long long want = (m + BH_THREADS - 1) / BH_THREADS;
        int grid = (int)(want < (long long)sms * 8 ? want : (long long)sms * 8);
        if (!d_p_hist) {
            bh_hist_kernel<<<grid, BH_THREADS, 0, st>>>(d_p, m, L.phist);
            BBK_CHECK_LAUNCH("bh_hist_kernel");
        }
        const int want_rank = d_rank != nullptr;
        bh_threshold_kernel<<<1, 1024, 0, st>>>(L.st, L.phist, want_rank ? 0 : 1, 0);
        BBK_CHECK_LAUNCH("bh_threshold_kernel");
        bh_compact_kernel<<<grid, BH_THREADS, 0, st>>>(d_p, m, d_q, L.st, L.keys[0], L.idx[0], want_rank, (long long*)d_rank);
        BBK_CHECK_LAUNCH("bh_compact_kernel");
        int rc = launch_rank(L, d_q, (long long*)d_rank, st);
        if (rc != BBK_OK) return rc;
    } else {
        scan_partial_kernel<<<G, BH_THREADS, 0, st>>>(S);
        BBK_CHECK_LAUNCH("scan_partial_kernel");
        scan_prefix_kernel<<<1, 32, 0, st>>>(S);
        BBK_CHECK_LAUNCH("scan_prefix_kernel");
        scan_apply_kernel<<<G, BH_THREADS, 0, st>>>(S);
        BBK_CHECK_LAUNCH("scan_apply_kernel");
    }
    if (mode == BBK_BH_UNSORTED && !d_rank) {
        long long want = (m + BH_THREADS - 1) / BH_THREADS;
        int grid = (int)(want < (long long)sms * 8 ? want : (long long)sms * 8);
        ones_fix_kernel<<<grid, BH_THREADS, 0, st>>>(d_p, m, d_q, L.st);
        BBK_CHECK_LAUNCH("ones_fix_kernel");
    }
    return BBK_OK;
}

// after bbk_score_pairs / bbk_score_deferred: q is pre-filled (1.0 / NaN) for every row and the rows with p < BBK_SMALL_P are listed in `cands`
extern "C" int bbk_bh_qvalues_listed(const double* d_p, int64_t m, int64_t n_tests, const int64_t* d_p_hist, double* d_q,
                                     const BbkCandidates* cands, const BbkScoreState* d_state, void* d_workspace,
                                     size_t workspace_bytes, void* stream) {
    BBK_REQUIRE(m >= 0 && m < (1ll << 32), "bbk_bh_qvalues_listed: m must be in [0, 2^32)");
    if (m == 0) return BBK_OK;
    BBK_REQUIRE(d_p && d_q && d_p_hist && d_workspace && cands && d_state, "bbk_bh_qvalues_listed: null pointer");
    BBK_REQUIRE(cands->capacity >= 0 && (cands->capacity == 0 || (cands->d_keys && cands->d_rows)), "bbk_bh_qvalues_listed: incomplete candidate list");
    BBK_REQUIRE(((uintptr_t)d_workspace & 255) == 0, "bbk_bh_qvalues_listed: workspace must be 256-byte aligned");
    const int G = sort_blocks();
    BhLayout L;
    size_t need = bh_layout(d_workspace, m, G, &L);
    if (workspace_bytes < need) {
        bbk_set_error("bbk_bh_qvalues_listed: workspace too small (%zu < %zu bytes)", workspace_bytes, need);
        return BBK_E_WORKSPACE;
    }
    cudaStream_t st = (cudaStream_t)stream;
    const int sms = bbk_num_sms();
    bh_init_kernel<<<(BBK_PHIST_BINS + 2 + 255) / 256, 256, 0, st>>>(L.st, L.phist, (const long long*)d_p_hist, n_tests);
    BBK_CHECK_LAUNCH("bh_init_kernel");
    bh_threshold_kernel<<<1, 1024, 0, st>>>(L.st, L.phist, 1, 1, d_state);
    BBK_CHECK_LAUNCH("bh_threshold_kernel");
    if (cands->capacity > 0) {
        bh_cand_filter_kernel<<<sms * 2, BH_THREADS, 0, st>>>(L.st, d_state, (const unsigned long long*)cands->d_keys, cands->d_rows, L.keys[0], L.idx[0]);
        BBK_CHECK_LAUNCH("bh_cand_filter_kernel");
    }
    long long want = (m + BH_THREADS - 1) / BH_THREADS;
    int grid = (int)(want < (long long)sms * 8 ? want : (long long)sms * 8);
    // saturation above BBK_SMALL_P, or an overflowed list: the 16 B/pair pass after all; otherwise returns at once
    bh_compact_kernel<<<grid, BH_THREADS, 0, st>>>(d_p, m, d_q, L.st, L.keys[0], L.idx[0], 0, nullptr);
    BBK_CHECK_LAUNCH("bh_compact_kernel");
    int rc = launch_rank(L, d_q, nullptr, st);
    if (rc != BBK_OK) return rc;
    ones_fix_kernel<<<grid, BH_THREADS, 0, st>>>(d_p, m, d_q, L.st);
    BBK_CHECK_LAUNCH("ones_fix_kernel");
    return BBK_OK;
}

// ---------------------------------------------------------------------------------------------------
// Per-segment q-values in one step (bbk_bh_qvalues_segmented): segment s = rows [off[s], off[s+1]) of one p / q pair, each with
// its own histogram, candidate list, score state and N.  Five launches whatever the number of segments:
//   threshold (one CTA per segment, the body of bh_threshold_kernel on the segment's histogram)
//   -> candidate filter over every list (segments whose list holds every candidate)
//   -> the 16 B/row pass over the rows of the other segments only
//   -> one cooperative rank launch: the key passes plus stable digit passes keyed on the row's segment, so the candidates end
//      up ordered by (segment, p); the forward running max restarts at every segment with that segment's N
//   -> ones fix, with a q_ones per segment
// ---------------------------------------------------------------------------------------------------
namespace {

constexpr int BH_SEG_MAX = 1 << 16;      // two segment digits

__device__ void bh_state_init(BhState* st, long long n_tests) {
    st->n_cand = 0; st->n_ones = 0; st->n_nan = 0; st->n_valid = 0; st->tau_key = ~0ull;
    st->n_tests = n_tests; st->q_ones = 1.0; st->total_max = -INFINITY; st->need_ones_fix = 0;
    for (int p = 0; p < NPASS; ++p) st->skip[p] = 0;
    st->use_list = 0;
}

__global__ void __launch_bounds__(1024) bh_threshold_seg_kernel(const BbkBhSegment* segs, BhState* seg_st, BhState* st) {
    const BbkBhSegment& sg = segs[blockIdx.x];
    BhState* ss = seg_st + blockIdx.x;
    if (threadIdx.x == 0) {
        bh_state_init(ss, sg.n_tests);
        if (blockIdx.x == 0) bh_state_init(st, -1);
    }
    __syncthreads();
    bh_threshold_body(ss, (const long long*)sg.d_p_hist, 1, 1, sg.d_state);
}

// appends the lanes' candidates of one warp step: one atomic on the shared count, one on the segment's
__device__ __forceinline__ void seg_append(bool cand, unsigned long long k, unsigned row, BhState* st, BhState* ss,
                                           unsigned long long* keys, unsigned* idx) {
    const unsigned bal = __ballot_sync(0xffffffffu, cand);
    if (!bal) return;
    const int lane = threadIdx.x & 31, leader = __ffs(bal) - 1;
    unsigned long long base = 0;
    if (lane == leader) {
        base = atomicAdd(&st->n_cand, (unsigned long long)__popc(bal));
        atomicAdd(&ss->n_cand, (unsigned long long)__popc(bal));
    }
    base = __shfl_sync(0xffffffffu, base, leader);
    if (cand) {
        const unsigned long long pos = base + __popc(bal & ((1u << lane) - 1));
        keys[pos] = k;
        idx[pos] = row;
    }
}

__global__ void __launch_bounds__(BH_THREADS) bh_cand_filter_seg_kernel(const BbkBhSegment* segs, int n_seg, BhState* seg_st, BhState* st,
                                                                        unsigned long long* keys, unsigned* idx) {
    const long long stride = (long long)gridDim.x * BH_THREADS;
    for (int s = 0; s < n_seg; ++s) {
        BhState* ss = seg_st + s;
        if (!ss->use_list) continue;
        const unsigned long long tau = ss->tau_key;
        const unsigned long long* ck = (const unsigned long long*)segs[s].cands.d_keys;
        const unsigned* cr = segs[s].cands.d_rows;
        const long long n = (long long)segs[s].d_state->n_cand;
        for (long long i0 = (long long)blockIdx.x * BH_THREADS; i0 < n; i0 += stride) {
            const long long i = i0 + threadIdx.x;
            const unsigned long long k = i < n ? ck[i] : ~0ull;
            const bool cand = i < n && k < tau;
            seg_append(cand, k, cand ? cr[i] : 0u, st, ss, keys, idx);
        }
    }
}

// bh_compact_kernel (keep_ones = 0, no rank) over the rows of the segments whose candidate list does not cover every candidate
__global__ void __launch_bounds__(BH_THREADS) bh_compact_seg_kernel(const double* p, double* q, const long long* off, int n_seg,
                                                                    BhState* seg_st, BhState* st, unsigned long long* keys, unsigned* idx) {
    const double qnan = __longlong_as_double(0x7ff8000000000000ll);
    const long long stride = (long long)gridDim.x * BH_THREADS;
    for (int s = 0; s < n_seg; ++s) {
        BhState* ss = seg_st + s;
        if (ss->use_list) continue;
        const unsigned long long tau = ss->tau_key;
        const long long hi = off[s + 1];
        for (long long i0 = off[s] + (long long)blockIdx.x * BH_THREADS; i0 < hi; i0 += stride) {
            const long long i = i0 + threadIdx.x;
            const bool live = i < hi;
            const double v = live ? ld_stream_double(p + i) : qnan;
            const bool isn = isnan(v);
            const unsigned long long k = key_of(v);
            const bool cand = live && !isn && k < tau && v != 1.0;
            if (live && !cand) st_stream_double(q + i, isn ? qnan : 1.0);
            seg_append(cand, k, (unsigned)i, st, ss, keys, idx);
        }
    }
}

// q of every segment's p == 1.0 group: one tie group after the segment's candidates (the end of bh_rank_kernel, per segment)
__global__ void __launch_bounds__(BH_THREADS) ones_fix_seg_kernel(const double* p, double* q, const long long* off, int n_seg, BhState* seg_st) {
    const long long stride = (long long)gridDim.x * BH_THREADS;
    for (int s = 0; s < n_seg; ++s) {
        BhState* ss = seg_st + s;
        if (ss->n_ones == 0) continue;
        double bh = (1.0 * (double)ss->n_tests) / (double)(ss->n_cand + 1);
        bh = (1.0 < bh) ? 1.0 : bh;
        double qo = (ss->total_max > bh) ? ss->total_max : bh;
        if (ss->tau_key != ~0ull) qo = 1.0;
        if (qo == 1.0) continue;
        if (blockIdx.x == 0 && threadIdx.x == 0) { ss->q_ones = qo; ss->need_ones_fix = 1; }
        for (long long i = off[s] + (long long)blockIdx.x * BH_THREADS + threadIdx.x; i < off[s + 1]; i += stride)
            if (p[i] == 1.0) q[i] = qo;
    }
}

size_t bh_seg_layout(void* base, long long m, int n_seg, BhLayout* L, BhState** seg_st, unsigned long long** seg_start) {
    size_t off = bh_layout(base, m, sort_blocks(), L);
    char* b = (char*)base;
    if (seg_st) *seg_st = b ? (BhState*)(b + off) : nullptr;
    off = align256(off + sizeof(BhState) * (size_t)n_seg);
    if (seg_start) *seg_start = b ? (unsigned long long*)(b + off) : nullptr;
    off = align256(off + sizeof(unsigned long long) * (size_t)n_seg);
    return off;
}

}  // namespace

extern "C" size_t bbk_bh_segmented_workspace_bytes(int64_t m, int32_t n_segments) {
    if (m < 0 || n_segments < 0) return 0;
    return bh_seg_layout(nullptr, m, n_segments, nullptr, nullptr, nullptr) + 256;
}

extern "C" int bbk_bh_qvalues_segmented(const double* d_p, int64_t m, const int64_t* d_offsets, const BbkBhSegment* d_segments,
                                        int32_t n_segments, double* d_q, void* d_workspace, size_t workspace_bytes, void* stream) {
    BBK_REQUIRE(m >= 0 && m < (1ll << 32), "bbk_bh_qvalues_segmented: m must be in [0, 2^32)");
    BBK_REQUIRE(n_segments >= 0 && n_segments <= BH_SEG_MAX, "bbk_bh_qvalues_segmented: n_segments must be in [0, 65536]");
    if (n_segments == 0 || m == 0) return BBK_OK;
    BBK_REQUIRE(d_p && d_q && d_offsets && d_segments && d_workspace, "bbk_bh_qvalues_segmented: null pointer");
    BBK_REQUIRE(((uintptr_t)d_workspace & 255) == 0, "bbk_bh_qvalues_segmented: workspace must be 256-byte aligned");
    BhLayout L;
    BhState* seg_st;
    unsigned long long* seg_start;
    size_t need = bh_seg_layout(d_workspace, m, n_segments, &L, &seg_st, &seg_start);
    if (workspace_bytes < need) {
        bbk_set_error("bbk_bh_qvalues_segmented: workspace too small (%zu < %zu bytes)", workspace_bytes, need);
        return BBK_E_WORKSPACE;
    }
    cudaStream_t st = (cudaStream_t)stream;
    const int sms = bbk_num_sms();
    const long long* off = (const long long*)d_offsets;
    bh_threshold_seg_kernel<<<n_segments, 1024, 0, st>>>(d_segments, seg_st, L.st);
    BBK_CHECK_LAUNCH("bh_threshold_seg_kernel");
    bh_cand_filter_seg_kernel<<<sms * 2, BH_THREADS, 0, st>>>(d_segments, n_segments, seg_st, L.st, L.keys[0], L.idx[0]);
    BBK_CHECK_LAUNCH("bh_cand_filter_seg_kernel");
    long long want = (m + BH_THREADS - 1) / BH_THREADS;
    const int grid = (int)(want < (long long)sms * 8 ? want : (long long)sms * 8);
    bh_compact_seg_kernel<<<grid, BH_THREADS, 0, st>>>(d_p, d_q, off, n_segments, seg_st, L.st, L.keys[0], L.idx[0]);
    BBK_CHECK_LAUNCH("bh_compact_seg_kernel");
    const int g = rank_grid();
    if (g <= 0 || g > L.G) { bbk_set_error("bh_rank_kernel: cooperative launch not possible on this device"); return BBK_E_CUDA; }
    RankParams R = {};
    R.L = L; R.q = d_q; R.rank = nullptr; R.n_host = -1; R.src = 0;
    R.seg_off = off; R.seg = seg_st; R.seg_start = seg_start; R.n_seg = n_segments;
    R.seg_passes = n_segments <= 1 ? 0 : (n_segments <= 256 ? 1 : 2);
    void* args[] = {&R};
    cudaError_t e = cudaLaunchCooperativeKernel((const void*)bh_rank_kernel<true, true>, dim3(g), dim3(RK_THREADS), args, RK_DYN_SMEM, st);
    if (e != cudaSuccess) { bbk_set_error("bh_rank_kernel: %s", cudaGetErrorString(e)); return BBK_E_CUDA; }
    ones_fix_seg_kernel<<<grid, BH_THREADS, 0, st>>>(d_p, d_q, off, n_segments, seg_st);
    BBK_CHECK_LAUNCH("ones_fix_seg_kernel");
    return BBK_OK;
}

// ---------------------------------------------------------------------------------------------------
// Genome-wide q-values across ranks (SURVEY.md section 8e, collective 2), in local steps around two host-side collectives:
//   all-reduce(p_hist)  ->  bbk_bh_select[_listed]  ->  bbk_bh_pack_count  ->  all-gather(fixed-capacity key blocks)
//   ->  bbk_bh_rank_gathered_padded  ->  bbk_bh_fix_ones_dev (the rare case q(p == 1) < 1)
// ---------------------------------------------------------------------------------------------------
// cands / d_score: the candidate list of bbk_score_pairs (listed mode), or NULL for a pass over p
static int bh_select_impl(const double* d_p, int64_t m, int64_t n_tests, const int64_t* d_p_hist_global, double* d_q,
                          const BbkCandidates* cands, const BbkScoreState* d_score, uint64_t* d_keys, uint32_t* d_idx,
                          int64_t keys_capacity, uint64_t* d_state, void* d_workspace, size_t workspace_bytes, void* stream) {
    BBK_REQUIRE(m >= 0 && m < (1ll << 32), "bbk_bh_select: m must be in [0, 2^32)");
    BBK_REQUIRE(keys_capacity >= 0, "bbk_bh_select: negative key capacity");
    BBK_REQUIRE(d_p_hist_global && d_state && d_workspace, "bbk_bh_select: null pointer");
    BBK_REQUIRE(m == 0 || (d_p && d_q && d_keys && d_idx), "bbk_bh_select: null array");
    BBK_REQUIRE(((uintptr_t)d_workspace & 255) == 0, "bbk_bh_select: workspace must be 256-byte aligned");
    const int G = sort_blocks();
    BhLayout L;
    size_t need = bh_layout(d_workspace, 0, G, &L);
    if (workspace_bytes < need) { bbk_set_error("bbk_bh_select: workspace too small (%zu < %zu bytes)", workspace_bytes, need); return BBK_E_WORKSPACE; }
    cudaStream_t st = (cudaStream_t)stream;
    const int sms = bbk_num_sms();
    bh_init_kernel<<<(BBK_PHIST_BINS + 2 + 255) / 256, 256, 0, st>>>(L.st, L.phist, (const long long*)d_p_hist_global, n_tests);
    BBK_CHECK_LAUNCH("bh_init_kernel");
    bh_threshold_kernel<<<1, 1024, 0, st>>>(L.st, L.phist, 1, cands ? 1 : 0, d_score);
    BBK_CHECK_LAUNCH("bh_threshold_kernel");
    if (m > 0) {
        if (cands && cands->capacity > 0) {
            bh_cand_filter_kernel<<<sms * 2, BH_THREADS, 0, st>>>(L.st, d_score, (const unsigned long long*)cands->d_keys, cands->d_rows,
                                                                  (unsigned long long*)d_keys, d_idx, keys_capacity);
            BBK_CHECK_LAUNCH("bh_cand_filter_kernel");
        }
        long long want = (m + BH_THREADS - 1) / BH_THREADS;
        int grid = (int)(want < (long long)sms * 8 ? want : (long long)sms * 8);
        // listed mode with the saturation above BBK_SMALL_P, or an overflowed list: the 16 B/pair pass; otherwise returns at once
        bh_compact_kernel<<<grid, BH_THREADS, 0, st>>>(d_p, m, d_q, L.st, (unsigned long long*)d_keys, d_idx, 0, nullptr, keys_capacity);
        BBK_CHECK_LAUNCH("bh_compact_kernel");
    }
    export_state_kernel<<<1, 1, 0, st>>>(L.st, (unsigned long long*)d_state);
    BBK_CHECK_LAUNCH("export_state_kernel");
    return BBK_OK;
}

extern "C" int bbk_bh_select(const double* d_p, int64_t m, int64_t n_tests, const int64_t* d_p_hist_global, double* d_q,
                             uint64_t* d_keys, uint32_t* d_idx, int64_t keys_capacity, uint64_t* d_state, void* d_workspace,
                             size_t workspace_bytes, void* stream) {
    return bh_select_impl(d_p, m, n_tests, d_p_hist_global, d_q, nullptr, nullptr, d_keys, d_idx, keys_capacity, d_state, d_workspace,
                          workspace_bytes, stream);
}

/* bbk_bh_select after bbk_score_pairs / bbk_score_deferred (q pre-filled, candidates listed) */
extern "C" int bbk_bh_select_listed(const double* d_p, int64_t m, int64_t n_tests, const int64_t* d_p_hist_global, double* d_q,
                                    const BbkCandidates* cands, const BbkScoreState* d_score, uint64_t* d_keys, uint32_t* d_idx,
                                    int64_t keys_capacity, uint64_t* d_state, void* d_workspace, size_t workspace_bytes, void* stream) {
    BBK_REQUIRE(cands && d_score, "bbk_bh_select_listed: null candidate list / score state");
    BBK_REQUIRE(cands->capacity >= 0 && (cands->capacity == 0 || (cands->d_keys && cands->d_rows)), "bbk_bh_select_listed: incomplete candidate list");
    return bh_select_impl(d_p, m, n_tests, d_p_hist_global, d_q, cands, d_score, d_keys, d_idx, keys_capacity, d_state, d_workspace,
                          workspace_bytes, stream);
}

// ---- the same with the gather left on the device: no candidate count ever travels to the host -------------------------
// Every rank sends a fixed-capacity block [count | keys[0 .. cap)] (d_keys of bbk_bh_select with its count in front); the
// all-gather delivers `world` such blocks.  Here: prefix the counts, compact the blocks into one key array, rank it, and
// scatter this rank's slice of the q-values back to its rows.  A count above cap puts the largest count into *d_overflow (the host looks
// at it when it reads the results and repeats the step with a capacity that fits).
namespace {

__global__ void gathered_prepare_kernel(const unsigned long long* recv, int world, long long cap, const unsigned long long* state_in,
                                        BhState* st, unsigned long long* offsets, int* overflow) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    unsigned long long run = 0, most = 0;
    int ov = 0;
    for (int r = 0; r < world; ++r) {
        unsigned long long c = recv[(size_t)r * (size_t)(cap + 1)];
        if (c > most) most = c;
        if (c > (unsigned long long)cap) { ov = 1; c = (unsigned long long)cap; }
        offsets[r] = run;
        run += c;
    }
    offsets[world] = run;
    if (ov) *overflow = most < 0x7fffffffull ? (int)most : 0x7fffffff;      // the capacity that would have sufficed
    st->n_cand = run; st->tau_key = state_in[1]; st->n_tests = (long long)state_in[2]; st->n_ones = state_in[3];
    st->n_nan = 0; st->n_valid = 0; st->q_ones = 1.0; st->total_max = 0.0; st->need_ones_fix = 0;
    for (int p = 0; p < NPASS; ++p) st->skip[p] = 0;
    st->use_list = 0;
}

__global__ void __launch_bounds__(BH_THREADS) gathered_compact_kernel(const unsigned long long* recv, int world, long long cap,
                                                                      const unsigned long long* offsets, unsigned long long* keys, unsigned* idx) {
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (int r = 0; r < world; ++r) {
        const unsigned long long off = offsets[r], n = offsets[r + 1] - off;
        const unsigned long long* src = recv + (size_t)r * (size_t)(cap + 1) + 1;
        for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < (long long)n; i += stride) {
            keys[off + i] = src[i];
            idx[off + i] = (unsigned)(off + i);
        }
    }
}

__global__ void __launch_bounds__(BH_THREADS) scatter_slice_kernel(const double* q_all, const unsigned long long* offsets, int rank,
                                                                   const unsigned* idx_local, double* dst) {
    const unsigned long long off = offsets[rank], n = offsets[rank + 1] - off;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < (long long)n; i += stride) dst[idx_local[i]] = q_all[off + i];
}

__global__ void pack_count_kernel(const unsigned long long* state, unsigned long long* send) { send[0] = state[0]; }

}  // namespace

extern "C" size_t bbk_bh_gathered_workspace_bytes(int32_t world, int64_t cap) {
    if (world <= 0 || cap < 0) return 0;
    const long long n = (long long)world * cap;
    return bh_layout(nullptr, n, sort_blocks(), nullptr) + align256(sizeof(double) * (size_t)(n + 1)) + align256(8 * (size_t)(world + 1)) + 512;
}

extern "C" int bbk_bh_pack_count(const uint64_t* d_state, uint64_t* d_send, void* stream) {
    BBK_REQUIRE(d_state && d_send, "bbk_bh_pack_count: null pointer");
    pack_count_kernel<<<1, 1, 0, (cudaStream_t)stream>>>((const unsigned long long*)d_state, (unsigned long long*)d_send);
    BBK_CHECK_LAUNCH("pack_count_kernel");
    return BBK_OK;
}

extern "C" int bbk_bh_rank_gathered_padded(const uint64_t* d_recv, int32_t world, int64_t cap, int32_t rank, const uint64_t* d_state,
                                           const uint32_t* d_idx_local, double* d_q_dst, double* d_q_ones, int32_t* d_overflow,
                                           void* d_workspace, size_t workspace_bytes, void* stream) {
    BBK_REQUIRE(world > 0 && rank >= 0 && rank < world && cap >= 0, "bbk_bh_rank_gathered_padded: bad world / rank / capacity");
    BBK_REQUIRE((long long)world * cap < (1ll << 32), "bbk_bh_rank_gathered_padded: world * cap must be below 2^32");
    BBK_REQUIRE(d_recv && d_state && d_q_ones && d_overflow && d_workspace, "bbk_bh_rank_gathered_padded: null pointer");
    BBK_REQUIRE(((uintptr_t)d_workspace & 255) == 0, "bbk_bh_rank_gathered_padded: workspace must be 256-byte aligned");
    const long long n_max = (long long)world * cap;
    const int G = sort_blocks();
    BhLayout L;
    size_t used = bh_layout(d_workspace, n_max, G, &L);
    double* q_all = (double*)((char*)d_workspace + used);
    used += align256(sizeof(double) * (size_t)(n_max + 1));
    unsigned long long* offsets = (unsigned long long*)((char*)d_workspace + used);
    used += align256(8 * (size_t)(world + 1));
    if (workspace_bytes < used) { bbk_set_error("bbk_bh_rank_gathered_padded: workspace too small (%zu < %zu bytes)", workspace_bytes, used); return BBK_E_WORKSPACE; }
    cudaStream_t st = (cudaStream_t)stream;
    gathered_prepare_kernel<<<1, 32, 0, st>>>((const unsigned long long*)d_recv, world, cap, (const unsigned long long*)d_state, L.st, offsets, d_overflow);
    BBK_CHECK_LAUNCH("gathered_prepare_kernel");
    if (n_max > 0) {
        long long want = (cap + BH_THREADS - 1) / BH_THREADS;
        int grid = (int)(want < (long long)bbk_num_sms() * 4 ? (want > 0 ? want : 1) : (long long)bbk_num_sms() * 4);
        gathered_compact_kernel<<<grid, BH_THREADS, 0, st>>>((const unsigned long long*)d_recv, world, cap, offsets, L.keys[0], L.idx[0]);
        BBK_CHECK_LAUNCH("gathered_compact_kernel");
    }
    int rc = launch_rank(L, q_all, nullptr, st);
    if (rc != BBK_OK) return rc;
    export_ones_kernel<<<1, 1, 0, st>>>(L.st, d_q_ones);
    BBK_CHECK_LAUNCH("export_ones_kernel");
    if (cap > 0 && d_idx_local && d_q_dst) {
        long long want = (cap + BH_THREADS - 1) / BH_THREADS;
        int grid = (int)(want < (long long)bbk_num_sms() * 4 ? want : (long long)bbk_num_sms() * 4);
        scatter_slice_kernel<<<grid, BH_THREADS, 0, st>>>(q_all, offsets, rank, d_idx_local, d_q_dst);
        BBK_CHECK_LAUNCH("scatter_slice_kernel");
    }
    return BBK_OK;
}

extern "C" int bbk_bh_fix_ones_dev(const double* d_p, int64_t m, const double* d_q_ones, double* d_q, void* stream) {
    BBK_REQUIRE(m >= 0, "bbk_bh_fix_ones_dev: negative size");
    if (m == 0) return BBK_OK;
    BBK_REQUIRE(d_p && d_q && d_q_ones, "bbk_bh_fix_ones_dev: null pointer");
    long long want = (m + BH_THREADS - 1) / BH_THREADS;
    int grid = (int)(want < (long long)bbk_num_sms() * 8 ? want : (long long)bbk_num_sms() * 8);
    fix_ones_dev_kernel<<<grid, BH_THREADS, 0, (cudaStream_t)stream>>>(d_p, m, d_q, d_q_ones);
    BBK_CHECK_LAUNCH("fix_ones_dev_kernel");
    return BBK_OK;
}
