// Small element-wise kernels of the model variants (reference: timbre_trap/framework/modules.py:780-1075) and of the skip
// connections (modules.py:95-117, 568-589).  All are single-pass, HBM-bound, 16-byte vectorised.
#include <algorithm>

#include "../../include/timbre_trap_b200.h"
#include "tt_common.cuh"

namespace tt {

// out = x + scale * e on bf16 tensors of identical layout (the decoder's skip connection, Decoder.forward modules.py:568-589, with
// TimbreTrap.apply_skip_connections' learnable weight, modules.py:110-112, read from device memory: no host sync); fp32 math,
// one rounding
__global__ void add_scaled_bf16_kernel(const uint4* __restrict__ x, const uint4* __restrict__ e, const float* __restrict__ scale,
                                       uint4* __restrict__ out, long long n8) {
    const float s = *scale;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n8; i += stride) {
        const uint4 a = __ldcs(x + i), b = __ldcs(e + i);
        const __nv_bfloat162* ah = reinterpret_cast<const __nv_bfloat162*>(&a);
        const __nv_bfloat162* bh = reinterpret_cast<const __nv_bfloat162*>(&b);
        uint4 r;
        uint32_t* rw = reinterpret_cast<uint32_t*>(&r);
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const float2 fa = __bfloat1622float2(ah[k]), fb = __bfloat1622float2(bh[k]);
            __nv_bfloat162 h = __floats2bfloat162_rn(fmaf(s, fb.x, fa.x), fmaf(s, fb.y, fa.y));
            rw[k] = *reinterpret_cast<uint32_t*>(&h);
        }
        out[i] = r;
    }
}

// (x) -> (x, 0) pairs: a one-channel feature map (magnitude / decibels, TimbreTrapMag.encode modules.py:927-950) in the interleaved
// two-channel layout conv_in reads; its second input channel meets zero weights
__global__ void widen_pairs_kernel(const float* __restrict__ x, long long n, float2* __restrict__ out) {
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) out[i] = make_float2(__ldcs(x + i), 0.f);
}

// channel 0 of interleaved pairs through the variant's output non-linearity:
//   0 identity, 1 relu (TimbreTrapMag.decode :976), 2 sigmoid (TimbreTrapMagDB.decode :1052), 3 tanh(relu) (Mag.decode + to_activations :996)
__global__ void channel0_activation_kernel(const float2* __restrict__ pairs, long long n, int mode, float* __restrict__ out) {
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        float v = ld_stream(pairs + i).x;
        if (mode == 1) v = fmaxf(v, 0.f);
        else if (mode == 2) v = 1.f / (1.f + expf(-v));
        else if (mode == 3) v = tanhf(fmaxf(v, 0.f));
        out[i] = v;
    }
}

// backward of channel0_activation seen as pairs -> pairs (f(v0), 0) (the loss step keeps one-channel tensors as such pairs):
// gin = (gout.x * f'(v0), 0), with relu'(0) = 0 as in torch; gout's channel 1 meets a constant and gets no gradient through
__global__ void channel0_activation_bwd_kernel(const float2* __restrict__ pairs, const float2* __restrict__ gout, long long n, int mode,
                                               float2* __restrict__ gin) {
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const float v = ld_stream(pairs + i).x;
        float g = ld_stream(gout + i).x;
        if (mode == 1) {
            g = v > 0.f ? g : 0.f;
        } else if (mode == 2) {
            const float s = 1.f / (1.f + expf(-v));
            g *= (1.f - s) * s;
        } else if (mode == 3) {
            const float t = tanhf(v);
            g = v > 0.f ? g * (1.f - t * t) : 0.f;
        }
        st_stream(gin + i, make_float2(g, 0.f));
    }
}

// fp32 interleaved pairs (coefficients or their gradient, (B, F, T, 2)) -> C8 planar bf16 with one channel group (B, 1, F, T, 8),
// channels 2..7 zero: the layout the tensor-core weight-gradient kernel reads
__global__ void pairs_to_c8_kernel(const float2* __restrict__ pairs, long long n, uint4* __restrict__ c8) {
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const float2 v = ld_stream(pairs + i);
        __nv_bfloat162 h = __floats2bfloat162_rn(v.x, v.y);
        c8[i] = make_uint4(*reinterpret_cast<uint32_t*>(&h), 0u, 0u, 0u);
    }
}

// sum of a[i] * b[i] over two bf16 tensors of one layout (the gradient of a skip connection's scalar weight): per-CTA partials in fp32,
// fixed-order finish in fp64 (bit-reproducible)
__global__ void __launch_bounds__(256) dot_bf16_partial_kernel(const uint4* __restrict__ a, const uint4* __restrict__ b, long long n8,
                                                               float* __restrict__ partial) {
    float acc = 0.f;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n8; i += (long long)gridDim.x * blockDim.x) {
        const uint4 av = __ldcs(a + i), bv = __ldcs(b + i);
        const __nv_bfloat162* ah = reinterpret_cast<const __nv_bfloat162*>(&av);
        const __nv_bfloat162* bh = reinterpret_cast<const __nv_bfloat162*>(&bv);
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const float2 fa = __bfloat1622float2(ah[k]), fb = __bfloat1622float2(bh[k]);
            acc = fmaf(fa.x, fb.x, acc);
            acc = fmaf(fa.y, fb.y, acc);
        }
    }
    __shared__ float red[8];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        float v = 0.f;
        for (int w = 0; w < 8; ++w) v += red[w];
        partial[blockIdx.x] = v;
    }
}
__global__ void dot_finish_kernel(const float* __restrict__ partial, int n, float* __restrict__ out) {
    double acc = 0.0;
    for (int i = 0; i < n; ++i) acc += (double)partial[i];
    *out = (float)acc;
}

}  // namespace tt

using namespace tt;

static int grid_for(long long n) { return (int)std::min<long long>((n + 255) / 256, 148 * 16); }

extern "C" int tt_add_scaled_bf16(const void* x, const void* e, const float* scale, void* out, int64_t n, void* stream) {
    TT_REQUIRE(x && e && scale && out, "null argument");
    TT_REQUIRE(n % 8 == 0, "add_scaled_bf16: element count must be a multiple of 8 (got %lld)", (long long)n);
    if (n <= 0) return TT_OK;
    add_scaled_bf16_kernel<<<grid_for(n / 8), 256, 0, (cudaStream_t)stream>>>((const uint4*)x, (const uint4*)e, scale, (uint4*)out, n / 8);
    tt_count_launches(1);
    TT_CUDA_CHECK(cudaGetLastError());
    return TT_OK;
}

extern "C" int tt_widen_pairs(const float* x, int64_t n, float* out, void* stream) {
    TT_REQUIRE(x && out, "null argument");
    if (n <= 0) return TT_OK;
    widen_pairs_kernel<<<grid_for(n), 256, 0, (cudaStream_t)stream>>>(x, n, (float2*)out);
    tt_count_launches(1);
    TT_CUDA_CHECK(cudaGetLastError());
    return TT_OK;
}

extern "C" int tt_channel0_activation(const float* pairs, int64_t n, int mode, float* out, void* stream) {
    TT_REQUIRE(pairs && out, "null argument");
    TT_REQUIRE(mode >= 0 && mode <= 3, "channel0_activation: mode must be 0..3");
    if (n <= 0) return TT_OK;
    channel0_activation_kernel<<<grid_for(n), 256, 0, (cudaStream_t)stream>>>((const float2*)pairs, n, mode, out);
    tt_count_launches(1);
    TT_CUDA_CHECK(cudaGetLastError());
    return TT_OK;
}

extern "C" int tt_channel0_activation_bwd(const float* pairs_in, const float* gpairs_out, int64_t n, int mode, float* gpairs_in,
                                          void* stream) {
    TT_REQUIRE(pairs_in && gpairs_out && gpairs_in, "null argument");
    TT_REQUIRE(mode >= 0 && mode <= 3, "channel0_activation_bwd: mode must be 0..3");
    if (n <= 0) return TT_OK;
    channel0_activation_bwd_kernel<<<grid_for(n), 256, 0, (cudaStream_t)stream>>>((const float2*)pairs_in, (const float2*)gpairs_out, n,
                                                                                   mode, (float2*)gpairs_in);
    tt_count_launches(1);
    TT_CUDA_CHECK(cudaGetLastError());
    return TT_OK;
}

extern "C" int tt_pairs_to_c8(const float* pairs, int64_t n, void* c8, void* stream) {
    TT_REQUIRE(pairs && c8, "null argument");
    if (n <= 0) return TT_OK;
    pairs_to_c8_kernel<<<grid_for(n), 256, 0, (cudaStream_t)stream>>>((const float2*)pairs, n, (uint4*)c8);
    tt_count_launches(1);
    TT_CUDA_CHECK(cudaGetLastError());
    return TT_OK;
}

extern "C" int tt_dot_scratch_floats(void) { return 148 * 8; }

extern "C" int tt_dot_bf16(const void* a, const void* b, int64_t n, float* out, float* scratch, void* stream) {
    TT_REQUIRE(a && b && out && scratch, "null argument");
    TT_REQUIRE(n % 8 == 0, "dot_bf16: element count must be a multiple of 8");
    cudaStream_t s = (cudaStream_t)stream;
    if (n <= 0) {
        TT_CUDA_CHECK(cudaMemsetAsync(out, 0, sizeof(float), s));
        return TT_OK;
    }
    const int blocks = (int)std::min<long long>((n / 8 + 255) / 256, 148 * 8);
    dot_bf16_partial_kernel<<<blocks, 256, 0, s>>>((const uint4*)a, (const uint4*)b, n / 8, scratch);
    dot_finish_kernel<<<1, 1, 0, s>>>(scratch, blocks, out);
    tt_count_launches(2);
    TT_CUDA_CHECK(cudaGetLastError());
    return TT_OK;
}
