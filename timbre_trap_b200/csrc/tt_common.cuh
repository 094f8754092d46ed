// Shared device helpers for the timbre-trap B200 kernels (sm_100a only).
#pragma once

#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>

#define TT_OK 0
#define TT_ERR_INVALID 1
#define TT_ERR_CUDA 2
#define TT_ERR_UNSUPPORTED 3
#define TT_ERR_ALLOC 4

void tt_set_error(const char* fmt, ...);
void tt_count_launches(int n);   // bookkeeping for tt_launch_count()

#define TT_CUDA_CHECK(expr)                                                                  \
    do {                                                                                     \
        cudaError_t _e = (expr);                                                             \
        if (_e != cudaSuccess) {                                                             \
            tt_set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
            return TT_ERR_CUDA;                                                              \
        }                                                                                    \
    } while (0)

#define TT_REQUIRE(cond, ...)                                                                \
    do {                                                                                     \
        if (!(cond)) {                                                                       \
            tt_set_error(__VA_ARGS__);                                                       \
            return TT_ERR_INVALID;                                                           \
        }                                                                                    \
    } while (0)

namespace tt {

__device__ __forceinline__ float2 cmul(float2 a, float2 b) {
    return make_float2(a.x * b.x - a.y * b.y, a.x * b.y + a.y * b.x);
}
__device__ __forceinline__ float2 cmulc(float2 a, float2 b) {   // a * conj(b)
    return make_float2(a.x * b.x + a.y * b.y, a.y * b.x - a.x * b.y);
}
__device__ __forceinline__ float2 cadd(float2 a, float2 b) { return make_float2(a.x + b.x, a.y + b.y); }
__device__ __forceinline__ float2 csub(float2 a, float2 b) { return make_float2(a.x - b.x, a.y - b.y); }
__device__ __forceinline__ float2 cscale(float2 a, float s) { return make_float2(a.x * s, a.y * s); }
__device__ __forceinline__ float2 cconj(float2 a) { return make_float2(a.x, -a.y); }
// packed f32x2 forms (sm_100: one FADD2 / FFMA2 per complex add / subtract instead of two scalar FADDs) - bit-identical results
__device__ __forceinline__ float2 cadd2(float2 a, float2 b) { return __fadd2_rn(a, b); }
__device__ __forceinline__ float2 csub2(float2 a, float2 b) { return __ffma2_rn(b, make_float2(-1.f, -1.f), a); }
// multiply by +i / -i
__device__ __forceinline__ float2 cmul_i(float2 a) { return make_float2(-a.y, a.x); }
__device__ __forceinline__ float2 cmul_mi(float2 a) { return make_float2(a.y, -a.x); }

// streaming (evict-first) vector accesses for data touched exactly once
__device__ __forceinline__ void st_stream(float2* p, float2 v) { __stcs(p, v); }
__device__ __forceinline__ void st_stream(float4* p, float4 v) { __stcs(p, v); }
__device__ __forceinline__ float2 ld_stream(const float2* p) { return __ldcs(p); }
__device__ __forceinline__ float4 ld_stream(const float4* p) { return __ldcs(p); }

// Clip tables of the many-clip calls: prefix[c] is the first block (or chunk) of clip c and prefix[n] the end, all relative to
// prefix[0] (a slice of a longer table works unchanged).  Every clip holds at least one entry.  Returns the clip holding x.
__device__ __forceinline__ int find_clip(const int* __restrict__ prefix, int n, int x) {
    const int base = __ldg(prefix);
    int lo = 0, hi = n - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (__ldg(prefix + mid) - base <= x) lo = mid;
        else hi = mid - 1;
    }
    return lo;
}

}  // namespace tt
