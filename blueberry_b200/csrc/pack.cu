// pack.cu - the p / q columns of a pass in the form that leaves the device (the output side of fithic.py:410-435).
//
// Most rows of a Fit-Hi-C pass carry no information in their numbers: a zero-count pair has p = 1.0 and q = 1.0, a row
// the reference does not emit (fithic.py:427, :434) has NaN, and q is 1.0 for all but the few significant rows.  The
// host link (PCIe) is the bottleneck of the end-to-end call, so what crosses it is two bits per row plus the values that
// are not implied:
//     code 0   p = 1.0, q = 1.0
//     code 1   p = NaN, q = NaN            (row not emitted)
//     code 2   p packed,   q = 1.0
//     code 3   p packed,   q packed
// A CTA packs chunks of BBK_PACK_CHUNK consecutive rows: a thread reads 16 rows of p and q, forms their code word,
// a block scan gives every thread its place, ONE atomic per chunk and list reserves the chunk's block of packed values,
// and the chunk table records where it is (chunks land in the lists in no particular order; rows inside a chunk keep
// theirs).  Lossless: bbkio_unpack_scores (host) rebuilds the dense columns bit for bit.
#include "common.cuh"

namespace {

constexpr int PK_THREADS = BBK_PACK_CHUNK / 16;
static_assert(PK_THREADS == 256, "a thread packs 16 rows = one code word");

__global__ void __launch_bounds__(PK_THREADS) pack_scores_kernel(const double* __restrict__ p, const double* __restrict__ q, long long m,
                                                                 unsigned* __restrict__ codes, BbkPackChunk* __restrict__ chunks,
                                                                 double* __restrict__ vals_p, long long cap_p, double* __restrict__ vals_q,
                                                                 long long cap_q, BbkPackState* st) {
    __shared__ unsigned s_w[2][PK_THREADS / 32];
    __shared__ unsigned long long s_base[2][2];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const long long n_chunks = (m + BBK_PACK_CHUNK - 1) / BBK_PACK_CHUNK;
    const double qnan = __longlong_as_double(0x7ff8000000000000ll);
    int par = 0;
    for (long long ch = blockIdx.x; ch < n_chunks; ch += gridDim.x, par ^= 1) {
        const long long r0 = ch * BBK_PACK_CHUNK + (long long)tid * 16;
        double pv[16], qv[16];
        if (r0 + 16 <= m) {
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const double2 a = *reinterpret_cast<const double2*>(p + r0 + 2 * j);
                pv[2 * j] = a.x; pv[2 * j + 1] = a.y;
                if (q) { const double2 b = *reinterpret_cast<const double2*>(q + r0 + 2 * j); qv[2 * j] = b.x; qv[2 * j + 1] = b.y; }
                else { qv[2 * j] = 1.0; qv[2 * j + 1] = 1.0; }
            }
        } else {
#pragma unroll
            for (int j = 0; j < 16; ++j) {
                const bool live = r0 + j < m;
                pv[j] = live ? p[r0 + j] : qnan;
                qv[j] = live ? (q ? q[r0 + j] : 1.0) : qnan;
            }
        }
        unsigned word = 0, np = 0, nq = 0;
#pragma unroll
        for (int j = 0; j < 16; ++j) {
            const bool pn = isnan(pv[j]), qn = isnan(qv[j]);
            unsigned cd;
            if (pn && (qn || !q)) cd = 1u;
            else if (pv[j] == 1.0 && qv[j] == 1.0) cd = 0u;
            else cd = (qv[j] == 1.0) ? 2u : 3u;
            word |= cd << (2 * j);
            np += cd >= 2u; nq += cd == 3u;
        }
        if (r0 < m) codes[r0 >> 4] = word;
        // places inside the chunk: both counts in one scan
        const unsigned packed = np | (nq << 16);
        unsigned inc = packed;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned y = __shfl_up_sync(0xffffffffu, inc, o);
            if (lane >= o) inc += y;
        }
        if (lane == 31) s_w[par][warp] = inc;
        __syncthreads();
        if (tid == 0) {
            unsigned tot = 0;
#pragma unroll
            for (int w = 0; w < PK_THREADS / 32; ++w) tot += s_w[par][w];
            const unsigned tp = tot & 0xffffu, tq = tot >> 16;
            const unsigned long long bp = tp ? atomicAdd((unsigned long long*)&st->n_p, (unsigned long long)tp) : 0ull;
            const unsigned long long bq = tq ? atomicAdd((unsigned long long*)&st->n_q, (unsigned long long)tq) : 0ull;
            s_base[par][0] = bp; s_base[par][1] = bq;
            BbkPackChunk c;
            c.base_p = bp; c.base_q = bq; c.n_p = tp; c.n_q = tq;
            chunks[ch] = c;
            if ((long long)(bp + tp) > cap_p || (long long)(bq + tq) > cap_q) st->overflow = 1;
        }
        __syncthreads();
        unsigned woff = 0;
#pragma unroll
        for (int w = 0; w < PK_THREADS / 32; ++w) woff += w < warp ? s_w[par][w] : 0u;
        const unsigned exc = woff + inc - packed;                       // (fields cannot carry: a chunk has 4096 rows)
        unsigned long long at_p = s_base[par][0] + (exc & 0xffffu), at_q = s_base[par][1] + (exc >> 16);
#pragma unroll
        for (int j = 0; j < 16; ++j) {
            const unsigned cd = (word >> (2 * j)) & 3u;
            if (cd >= 2u) { if ((long long)at_p < cap_p) vals_p[at_p] = pv[j]; at_p += 1; }
            if (cd == 3u) { if ((long long)at_q < cap_q) vals_q[at_q] = qv[j]; at_q += 1; }
        }
    }
}

__global__ void pack_begin_kernel(BbkPackState* st) { st->n_p = 0; st->n_q = 0; st->overflow = 0; st->reserved = 0; }

}  // namespace

extern "C" int64_t bbk_pack_chunks(int64_t m) { return m <= 0 ? 0 : (m + BBK_PACK_CHUNK - 1) / BBK_PACK_CHUNK; }
extern "C" int64_t bbk_pack_code_words(int64_t m) { return m <= 0 ? 0 : (m + 15) / 16; }

extern "C" int bbk_pack_scores(const double* d_p, const double* d_q, int64_t m, uint32_t* d_codes, BbkPackChunk* d_chunks,
                               double* d_values_p, int64_t capacity_p, double* d_values_q, int64_t capacity_q,
                               BbkPackState* d_state, void* stream) {
    BBK_REQUIRE(m >= 0 && capacity_p >= 0 && capacity_q >= 0, "bbk_pack_scores: negative size");
    BBK_REQUIRE(d_state, "bbk_pack_scores: null state");
    cudaStream_t st = (cudaStream_t)stream;
    pack_begin_kernel<<<1, 1, 0, st>>>(d_state);
    BBK_CHECK_LAUNCH("pack_begin_kernel");
    if (m == 0) return BBK_OK;
    BBK_REQUIRE(d_p && d_codes && d_chunks, "bbk_pack_scores: null pointer");
    BBK_REQUIRE((capacity_p == 0 || d_values_p) && (capacity_q == 0 || d_values_q), "bbk_pack_scores: null value list");
    BBK_REQUIRE((((uintptr_t)d_p | (uintptr_t)d_q) & 15) == 0, "bbk_pack_scores: p / q must be 16-byte aligned");
    const long long n_chunks = bbk_pack_chunks(m);
    long long grid = (long long)bbk_num_sms() * 8;
    if (n_chunks < grid) grid = n_chunks;
    pack_scores_kernel<<<(unsigned)grid, PK_THREADS, 0, st>>>(d_p, d_q, m, d_codes, d_chunks, d_values_p, capacity_p, d_values_q,
                                                             capacity_q, d_state);
    BBK_CHECK_LAUNCH("pack_scores_kernel");
    return BBK_OK;
}

// ---- bbk_unpack_records: packed contact records (bbk.h, BbkRecHeader) back into the int32 columns of a pass ------------
// One CTA per chunk (grid-stride).  Thread t decodes the 4-row groups t, t + 256, ... of its chunk, so every 128-bit store of a
// warp covers 512 contiguous bytes.  Row i of a column of b bits is bits [i b, i b + b) of its words: one 64-bit funnel shift
// over the word holding bit i b and the next one, which is read only when the value reaches into it (it then lies inside the
// column's block, so a buffer bbkio_check_records accepted is never read past its payload).
namespace {

constexpr int RU_THREADS = 256;
static_assert(BBK_REC_CHUNK == RU_THREADS * 16, "a thread decodes 16 rows of a chunk");

__device__ __forceinline__ long long rec_get(const unsigned long long* __restrict__ w, int b, long long base, unsigned long long step,
                                             int i) {
    if (b == 0) return base;                             // an empty block: nothing to read
    const unsigned long long bit = (unsigned long long)i * (unsigned)b;
    const unsigned off = (unsigned)(bit & 63u);
    const unsigned long long* p = w + (bit >> 6);
    const unsigned long long lo = __ldg(p), hi = off + (unsigned)b > 64u ? __ldg(p + 1) : 0ull;
    const unsigned long long u = ((lo >> off) | ((hi << 1) << (63u - off))) & ((1ull << b) - 1ull);
    return base + (long long)(step * u);
}

__global__ void __launch_bounds__(RU_THREADS) unpack_records_kernel(const unsigned char* __restrict__ buf, long long rows,
                                                                    int* __restrict__ mid1, int* __restrict__ mid2,
                                                                    int* __restrict__ count) {
    const long long n_chunks = (rows + BBK_REC_CHUNK - 1) / BBK_REC_CHUNK;
    const BbkRecChunk* table = reinterpret_cast<const BbkRecChunk*>(buf + sizeof(BbkRecHeader));
    for (long long ch = blockIdx.x; ch < n_chunks; ch += gridDim.x) {
        const BbkRecChunk C = table[ch];
        const long long r0 = ch * BBK_REC_CHUNK;
        const int n = (int)min((long long)BBK_REC_CHUNK, rows - r0);
        const unsigned long long* w0 = reinterpret_cast<const unsigned long long*>(buf + C.offset);
        const unsigned long long* w1 = w0 + BBK_REC_COL_BYTES(n, C.bits[0]) / 8;
        const unsigned long long* w2 = w1 + BBK_REC_COL_BYTES(n, C.bits[1]) / 8;
        const int b0 = C.bits[0], b1 = C.bits[1], b2 = C.bits[2];
#pragma unroll
        for (int g = 0; g < 4; ++g) {
            const int i0 = (g * RU_THREADS + (int)threadIdx.x) * 4;
            if (i0 >= n) break;
            int m1[4], m2[4], ct[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const int i = min(i0 + k, n - 1);              // rows past the end are decoded again, never stored
                const long long a = rec_get(w0, b0, C.base[0], C.step[0], i);
                m1[k] = (int)a;
                m2[k] = (int)(a + rec_get(w1, b1, C.base[1], C.step[1], i));
                ct[k] = (int)rec_get(w2, b2, C.base[2], C.step[2], i);
            }
            const long long r = r0 + i0;
            if (i0 + 4 <= n) {
                *reinterpret_cast<int4*>(mid1 + r) = make_int4(m1[0], m1[1], m1[2], m1[3]);
                *reinterpret_cast<int4*>(mid2 + r) = make_int4(m2[0], m2[1], m2[2], m2[3]);
                *reinterpret_cast<int4*>(count + r) = make_int4(ct[0], ct[1], ct[2], ct[3]);
            } else {
#pragma unroll
                for (int k = 0; k < 4; ++k)
                    if (i0 + k < n) { mid1[r + k] = m1[k]; mid2[r + k] = m2[k]; count[r + k] = ct[k]; }
            }
        }
    }
}

}  // namespace

extern "C" int bbk_unpack_records(const void* d_buf, int64_t bytes, int64_t rows, int32_t* d_mid1, int32_t* d_mid2, int32_t* d_count,
                                  void* stream) {
    BBK_REQUIRE(rows >= 0 && bytes >= (int64_t)sizeof(BbkRecHeader), "bbk_unpack_records: negative rows or a buffer shorter than its header");
    if (rows == 0) return BBK_OK;
    BBK_REQUIRE(d_buf && d_mid1 && d_mid2 && d_count, "bbk_unpack_records: null pointer");
    BBK_REQUIRE((((uintptr_t)d_buf | (uintptr_t)d_mid1 | (uintptr_t)d_mid2 | (uintptr_t)d_count) & 15) == 0,
                "bbk_unpack_records: buffer and columns must be 16-byte aligned");
    const long long n_chunks = (rows + BBK_REC_CHUNK - 1) / BBK_REC_CHUNK;
    BBK_REQUIRE((uint64_t)bytes >= sizeof(BbkRecHeader) + (uint64_t)n_chunks * sizeof(BbkRecChunk), "bbk_unpack_records: buffer shorter than its chunk table");
    long long grid = (long long)bbk_num_sms() * 8;
    if (n_chunks < grid) grid = n_chunks;
    unpack_records_kernel<<<(unsigned)grid, RU_THREADS, 0, (cudaStream_t)stream>>>(static_cast<const unsigned char*>(d_buf), rows, d_mid1,
                                                                                     d_mid2, d_count);
    BBK_CHECK_LAUNCH("unpack_records_kernel");
    return BBK_OK;
}
