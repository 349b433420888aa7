// common.cuh - shared helpers for the libbbk kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include "../../include/bbk.h"

#ifndef __CUDA_ARCH_LIST__
#endif

void bbk_set_error(const char* fmt, ...);
int bbk_num_sms();

// K4 -> K5 hand-over (bbk_score_pairs / bbk_score_deferred -> bbk_bh_*_listed): K4 lists (key, row) of every p < BBK_SMALL_P,
// so that the q-value step finds its candidates in that list instead of another pass over p.  Exact whatever the bound: when
// the saturation bucket lies above it, K5 falls back to its own pass.
#define BBK_SMALL_P 0.03125
// the library's radix sort on its own (bh.cu): n (u64 key, u32 value) pairs in buffer `src` (0 / 1) of a workspace of
// bbk_bh_workspace_bytes(capacity) bytes, stable, result left in the same buffer; n_host < 0: count at bbk_sort_count_ptr
void bbk_sort_buffers(void* workspace, long long capacity, int which, unsigned long long** keys, unsigned** idx);
unsigned long long* bbk_sort_count_ptr(void* workspace);
int bbk_sort_pairs(void* workspace, long long capacity, long long n_host, int src, cudaStream_t st);

#define BBK_CHECK_CUDA(expr)                                                                  \
    do {                                                                                      \
        cudaError_t _e = (expr);                                                              \
        if (_e != cudaSuccess) {                                                              \
            bbk_set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
            return BBK_E_CUDA;                                                                \
        }                                                                                     \
    } while (0)

#define BBK_CHECK_LAUNCH(name)                                                                \
    do {                                                                                      \
        cudaError_t _e = cudaGetLastError();                                                  \
        if (_e != cudaSuccess) {                                                              \
            bbk_set_error("launch of %s failed: %s", name, cudaGetErrorString(_e));           \
            return BBK_E_CUDA;                                                                \
        }                                                                                     \
    } while (0)

#define BBK_REQUIRE(cond, msg)                                                                \
    do {                                                                                      \
        if (!(cond)) {                                                                        \
            bbk_set_error("invalid argument: %s", msg);                                       \
            return BBK_E_INVALID;                                                             \
        }                                                                                     \
    } while (0)

// order-preserving map double -> u64 (total order of IEEE values; -0 < +0)
__device__ __forceinline__ unsigned long long bbk_key_of(double v) {
    unsigned long long b = (unsigned long long)__double_as_longlong(v);
    return (b >> 63) ? ~b : (b | 0x8000000000000000ull);
}

// streaming 128-bit load that does not allocate in L1 (each record is read exactly once)
__device__ __forceinline__ int4 ld_stream_int4(const int4* p) {
    int4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.s32 {%0, %1, %2, %3}, [%4];"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
    return r;
}
__device__ __forceinline__ int ld_stream_int(const int* p) {
    int r;
    asm volatile("ld.global.nc.L1::no_allocate.s32 %0, [%1];" : "=r"(r) : "l"(p));
    return r;
}
__device__ __forceinline__ double2 ld_stream_double2(const double2* p) {
    double2 r;
    asm volatile("ld.global.nc.L1::no_allocate.v2.f64 {%0, %1}, [%2];" : "=d"(r.x), "=d"(r.y) : "l"(p));
    return r;
}
__device__ __forceinline__ double ld_stream_double(const double* p) {
    double r;
    asm volatile("ld.global.nc.L1::no_allocate.f64 %0, [%1];" : "=d"(r) : "l"(p));
    return r;
}
__device__ __forceinline__ void st_stream_double2(double2* p, double2 v) {
    asm volatile("st.global.L1::no_allocate.v2.f64 [%0], {%1, %2};" :: "l"(p), "d"(v.x), "d"(v.y) : "memory");
}
__device__ __forceinline__ void st_stream_double(double* p, double v) {
    asm volatile("st.global.L1::no_allocate.f64 [%0], %1;" :: "l"(p), "d"(v) : "memory");
}

// exact unsigned division by an invariant divisor R < 2^32:
//   fastdiv   : any a < 2^32        q = hi64(a * ceil(2^64 / R))
//   fastdiv31 : a < 2^31 (cheaper)  q = hi32(a * ceil(2^(31+l) / R)) >> (l-1),  l = ceil(log2 R)
struct FastDiv {
    uint64_t magic;   // ceil(2^64 / R), 0 when R == 1
    uint32_t R;
    uint32_t mul31;   // ceil(2^(31+l) / R), 0 when R == 1
    uint32_t sh31;    // l - 1
};
static inline FastDiv make_fastdiv(uint64_t R) {
    FastDiv f;
    f.R = (uint32_t)R;
    f.magic = (R <= 1) ? 0 : (~0ull / R + 1);   // floor((2^64-1)/R)+1 == ceil(2^64/R) for R not a power of two; exact otherwise too
    f.mul31 = 0;
    f.sh31 = 0;
    if (R > 1) {
        uint32_t l = 0;
        while ((1ull << l) < R) ++l;
        unsigned __int128 num = (unsigned __int128)1 << (31 + l);
        f.mul31 = (uint32_t)((num + R - 1) / R);
        f.sh31 = l - 1;
    }
    return f;
}
__device__ __forceinline__ uint32_t fastdiv(uint32_t a, const FastDiv& f) {
    return f.magic ? (uint32_t)__umul64hi((uint64_t)a, f.magic) : a;
}
__device__ __forceinline__ uint32_t fastdiv31(uint32_t a, const FastDiv& f) {
    return f.mul31 ? (__umulhi(a, f.mul31) >> f.sh31) : a;
}

__device__ __forceinline__ long long warp_sum_ll(long long v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ long long warp_min_ll(long long v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) { long long w = __shfl_xor_sync(0xffffffffu, v, o); v = w < v ? w : v; }
    return v;
}
__device__ __forceinline__ long long warp_max_ll(long long v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) { long long w = __shfl_xor_sync(0xffffffffu, v, o); v = w > v ? w : v; }
    return v;
}
