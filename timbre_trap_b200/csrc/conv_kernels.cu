// Encoder / decoder convolutions of Timbre-Trap (reference: timbre_trap/framework/modules.py:396-777) as bf16
// implicit GEMMs on the sm_100a tensor cores (tcgen05.mma, fp32 accumulators in TMEM).
//
// Activation layout ("C8 planar"):  [B][CG][H][T][8] bf16, CG = ceil(C / 8); the 8 channels of one pixel are 16
// contiguous bytes and T is the contiguous pixel axis.  A run of 8 consecutive pixels of one channel group is therefore
// exactly one UMMA core matrix (8 rows x 16 B, SWIZZLE_NONE, K-major), 128 consecutive pixels are the M = 128 rows of
// one MMA (SBO = 128 B), and a convolution tap is nothing but a different start address into the same shared-memory
// tile: the im2col matrix is never materialised.  Two core matrices along K (one MMA, K = 16) are either two channel
// groups of one tap (LBO = plane stride) or, for 8-channel layers, two taps (LBO = their address difference).
//
// conv_rows_kernel is the generic tile kernel: a CTA owns R "row groups" x 128 pixels; for every row group it issues a
// list of MMAs (tap table from the host) into its own TMEM columns, then an epilogue (bias, ELU, bf16 pack, coalesced
// 16 B stores).  It serves the layers below; the residual blocks and the strided / transposed convs of the model run in the
// row-pipelined kernels of res_rs.cu / updown_strip.cu.
//
//   layer (modules.py)                       row group      MMAs / group            N
//   Decoder.convin      :533-536             1 output row   latent/16               C0       (weights depend on the row)
//   single 3x3 / 1x1 conv (backward pass)    1 output row   9*C/16 (+1 if C = 8)    C
//
// Weights arrive pre-packed in the B-operand canonical layout [K/8][N][8] bf16 (timbre_trap_b200/framework/packing.py).

#include <stdlib.h>
#include <string.h>

#include <algorithm>

#include "../../include/timbre_trap_b200.h"
#include "tt_common.cuh"
#include "umma.cuh"

namespace tt {

constexpr int kMaxTaps = 40;
constexpr int kMaxRows = 16;
constexpr int kTileT = 128;
constexpr int kHeaderBytes = 2048;

struct ConvRowsParams {
    const __nv_bfloat16* x;
    __nv_bfloat16* y;
    const __nv_bfloat16* w1;
    const float* b1;
    int B, CGin, Hin, T, CGout, Hout;
    int groups;            // row groups in total (Hout, or ceil(Hout/2) for out_mode 1)
    int R;                 // row groups per CTA (<= kMaxRows)
    int sh;                // input rows advanced per row group
    int row_lo;            // input row held by tile row 0 = g0 * sh + row_lo
    int in_rows;           // tile rows
    int padT;              // T halo on each side
    int n_mma1, kg1;       // MMAs per group, K groups of 8 in the packed weights
    int out_mode;          // 0: N channels -> one output row;  1: two output rows of N/2 channels
    int act;               // ELU on the output
    int post;              // after that, with the tensor `e` (layout of y): 1 = times ELU'(e) as a function of the ACTIVATED value e
                           // (e > 0 ? 1 : e + 1), 2 = plus e  - the element-wise passes of the residual blocks' backward, fused
    const __nv_bfloat16* e;
    int w_group_stride;    // bytes between the packed weights of consecutive row groups (0: shared)
    int b_group_stride;    // floats between the biases of consecutive row groups (0: shared)
    uint32_t tap_off[kMaxTaps];
    uint32_t tap_lbo[kMaxTaps];
};

__device__ __forceinline__ float elu(float v) { return v > 0.f ? v : __expf(v) - 1.f; }

__device__ __forceinline__ uint4 pack8(const float* v) {
    __nv_bfloat162 a = __floats2bfloat162_rn(v[0], v[1]);
    __nv_bfloat162 b = __floats2bfloat162_rn(v[2], v[3]);
    __nv_bfloat162 c = __floats2bfloat162_rn(v[4], v[5]);
    __nv_bfloat162 d = __floats2bfloat162_rn(v[6], v[7]);
    uint4 r;
    r.x = *reinterpret_cast<uint32_t*>(&a);
    r.y = *reinterpret_cast<uint32_t*>(&b);
    r.z = *reinterpret_cast<uint32_t*>(&c);
    r.w = *reinterpret_cast<uint32_t*>(&d);
    return r;
}

__device__ __forceinline__ void unpack8(uint4 r, float* v) {
    const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&r);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        float2 f = __bfloat1622float2(h[i]);
        v[2 * i] = f.x;
        v[2 * i + 1] = f.y;
    }
}

constexpr int kConvThreads = 512;   // 16 warps: warp w owns TMEM lane quadrant w % 4 and row groups (w / 4) mod 4

template <int N1>
__global__ void __launch_bounds__(kConvThreads) conv_rows_kernel(const __grid_constant__ ConvRowsParams p) {
    extern __shared__ __align__(1024) uint8_t smem[];
    constexpr int NC = N1;                          // TMEM columns per row group
    uint64_t* bar1 = reinterpret_cast<uint64_t*>(smem);
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + 256);
    float* sB1 = reinterpret_cast<float*>(smem + 512);

    constexpr int NT = kConvThreads, NW = NT / 32, NWG = NW / 4;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int quad = warp & 3, wg = warp >> 2;
    const int t0 = blockIdx.x * kTileT;
    const int g0 = blockIdx.y * p.R;
    const int b = blockIdx.z;
    const int rows = min(p.R, p.groups - g0);
    const int wrows = p.w_group_stride ? p.R : 1;

    const int TW = kTileT + 2 * p.padT;
    const uint32_t row_bytes = (uint32_t)TW * 16u;
    const uint32_t plane_bytes = (uint32_t)p.in_rows * row_bytes;
    const uint32_t w1_bytes = (uint32_t)p.kg1 * N1 * 16u;
    uint8_t* sW1 = smem + kHeaderBytes;
    uint8_t* sIn = sW1 + (size_t)w1_bytes * wrows;

    // ---- setup --------------------------------------------------------------------------------------
    uint32_t ncols = 32;
    while (ncols < (uint32_t)(p.R * NC)) ncols <<= 1;
    if (warp == 0) umma::tmem_alloc(tmem_slot, ncols);
    if (tid == 0) {
        for (int i = 0; i < kMaxRows; ++i) umma::mbar_init(&bar1[i], 1);
        umma::mbar_fence_init();
    }
    // weights and biases
    for (int r = 0; r < wrows; ++r) {
        const uint4* src = reinterpret_cast<const uint4*>(reinterpret_cast<const uint8_t*>(p.w1) +
                                                          (size_t)(g0 + r) * p.w_group_stride);
        if (r < rows)
            for (int i = tid; i < (int)(w1_bytes / 16); i += NT)
                umma::cp_async16(reinterpret_cast<uint4*>(sW1 + (size_t)r * w1_bytes) + i, src + i, 16u);
    }
    if (p.b_group_stride == 0 && tid < N1) sB1[tid] = p.b1[tid];

    // input tile, zero-filled outside the image ('same' padding, transposed-conv borders)
    {
        const int h_base = g0 * p.sh + p.row_lo;
        const int n_rows_all = p.CGin * p.in_rows;
        for (int rr = warp; rr < n_rows_all; rr += NW) {
            const int cg = rr / p.in_rows, r = rr - cg * p.in_rows;
            const int hi = h_base + r;
            const bool row_ok = hi >= 0 && hi < p.Hin;
            const uint4* src = reinterpret_cast<const uint4*>(p.x) + (((size_t)b * p.CGin + cg) * p.Hin + (row_ok ? hi : 0)) * p.T;
            uint4* dst = reinterpret_cast<uint4*>(sIn + (size_t)cg * plane_bytes + (size_t)r * row_bytes);
            for (int c = lane; c < TW; c += 32) {
                const int t = t0 - p.padT + c;
                const bool ok = row_ok && t >= 0 && t < p.T;
                umma::cp_async16(dst + c, ok ? src + t : reinterpret_cast<const uint4*>(p.x), ok ? 16u : 0u);
            }
        }
        if (tid < 16) reinterpret_cast<uint4*>(sIn + (size_t)p.CGin * plane_bytes)[tid] = make_uint4(0u, 0u, 0u, 0u);
    }
    umma::cp_async_wait_all();
    umma::fence_proxy_async();
    umma::fence_before_sync();
    __syncthreads();
    umma::fence_after_sync();
    const uint32_t tmem = *tmem_slot;

    // ---- all MMAs of all row groups, one commit per group -------------------------------------
    if (tid == 0) {
        const uint32_t idesc = umma::make_idesc_bf16(128, N1);
        const uint32_t in0 = umma::smem_u32(sIn), w0 = umma::smem_u32(sW1);
        for (int i = 0; i < rows; ++i) {
            const uint32_t base = in0 + (uint32_t)(i * p.sh) * row_bytes;
            const uint32_t wb = w0 + (p.w_group_stride ? (uint32_t)i * w1_bytes : 0u);
            for (int m = 0; m < p.n_mma1; ++m) {
                const uint64_t da = umma::make_desc(base + p.tap_off[m], p.tap_lbo[m], 128u);
                const uint64_t db = umma::make_desc(wb + (uint32_t)m * 2u * N1 * 16u, N1 * 16u, 128u);
                umma::mma_bf16(tmem + (uint32_t)(i * NC), da, db, idesc, m > 0);
            }
            umma::commit(&bar1[i]);
        }
    }

    const int j = quad * 32 + lane;                 // pixel within the tile = TMEM lane
    const uint32_t lane_addr = tmem + ((uint32_t)(quad * 32) << 16);
    const bool t_ok = t0 + j < p.T;

    // ---- epilogue ------------------------------------------------------------------------------------
    for (int i = wg; i < rows; i += NWG) {
        umma::mbar_wait(&bar1[i], 0);
        umma::fence_after_sync();
        const float* bias = p.b_group_stride ? p.b1 + (size_t)(g0 + i) * p.b_group_stride : sB1;
#pragma unroll
        for (int c0 = 0; c0 < N1; c0 += 16) {
            float v[16];
            umma::tmem_ld16(lane_addr + (uint32_t)(i * NC + c0), v);
            umma::tmem_ld_wait();
#pragma unroll
            for (int k = 0; k < 16; ++k) v[k] += bias[c0 + k];
            if (p.act) {
#pragma unroll
                for (int k = 0; k < 16; ++k) v[k] = elu(v[k]);
            }
            if (t_ok) {
#pragma unroll
                for (int hh = 0; hh < 2; ++hh) {
                    const int c = c0 + 8 * hh;          // first of 8 channels
                    int ho, cg;
                    if (p.out_mode == 0) { ho = g0 + i; cg = c >> 3; }
                    else { ho = 2 * (g0 + i) + (c >= N1 / 2 ? 1 : 0); cg = (c % (N1 / 2)) >> 3; }
                    if (cg < p.CGout && ho < p.Hout) {
                        const size_t at = (((size_t)b * p.CGout + cg) * p.Hout + ho) * p.T + t0 + j;
                        if (p.post) {
                            float ev[8];
                            unpack8(__ldg(reinterpret_cast<const uint4*>(p.e) + at), ev);
#pragma unroll
                            for (int k = 0; k < 8; ++k) {
                                if (p.post == 1) v[8 * hh + k] *= ev[k] > 0.f ? 1.f : ev[k] + 1.f;
                                else v[8 * hh + k] += ev[k];
                            }
                        }
                        reinterpret_cast<uint4*>(p.y)[at] = pack8(v + 8 * hh);
                    }
                }
            }
        }
    }

    umma::fence_before_sync();
    __syncthreads();
    if (warp == 0) umma::tmem_dealloc(tmem, ncols);
}

// ---------------------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------------------
static size_t conv_rows_smem(const ConvRowsParams& p, int n1) {
    const size_t TW = kTileT + 2 * p.padT;
    const size_t plane = (size_t)p.in_rows * TW * 16;
    return kHeaderBytes + (size_t)p.kg1 * n1 * 16 * (p.w_group_stride ? p.R : 1) + (size_t)p.CGin * plane + 256;
}

template <int N1>
static int launch_conv_rows(const ConvRowsParams& p, cudaStream_t stream) {
    const size_t smem = conv_rows_smem(p, N1);
    TT_REQUIRE(smem <= 227 * 1024, "conv tile needs %zu bytes of shared memory", smem);
    static size_t configured = 0;
    if (smem > configured) {
        TT_CUDA_CHECK(cudaFuncSetAttribute(conv_rows_kernel<N1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        configured = smem;
    }
    dim3 grid((p.T + kTileT - 1) / kTileT, (p.groups + p.R - 1) / p.R, p.B);
    conv_rows_kernel<N1><<<grid, kConvThreads, smem, stream>>>(p);
    tt_count_launches(1);
    TT_CUDA_CHECK(cudaGetLastError());
    return TT_OK;
}

}  // namespace tt

using namespace tt;

static void fill_common(ConvRowsParams& p, const void* x, void* y, const void* w1, const float* b1, int B, int CGin, int Hin,
                        int T, int CGout, int Hout) {
    memset(&p, 0, sizeof(p));
    p.x = (const __nv_bfloat16*)x; p.y = (__nv_bfloat16*)y;
    p.w1 = (const __nv_bfloat16*)w1; p.b1 = b1;
    p.B = B; p.CGin = CGin; p.Hin = Hin; p.T = T; p.CGout = CGout; p.Hout = Hout;
}

static int dispatch_n1(const ConvRowsParams& p, int n1, cudaStream_t s) {
    switch (n1) {
        case 16: return launch_conv_rows<16>(p, s);
        case 32: return launch_conv_rows<32>(p, s);
        case 64: return launch_conv_rows<64>(p, s);
        case 128: return launch_conv_rows<128>(p, s);
        default: tt_set_error("unsupported GEMM N = %d", n1); return TT_ERR_UNSUPPORTED;
    }
}

// A single 3x3 dilated 'same' conv (optionally + ELU) or 1x1 conv on C8 planar tensors through the generic tile kernel: used by
// the backward pass (recompute of the residual block's inner activation; data gradients = convs with transformed weights).
//   k = 3: weights from packing.pack_res3x3 (K order tap-major);  k = 1: packing.pack_res1x1.  bias may be NULL (zeros).
extern "C" int tt_conv_same(const void* x, void* y, const void* w, const float* bias, int B, int C, int H, int T, int k, int dilation,
                            int act_elu, void* stream) {
    return tt_conv_same_post(x, y, w, bias, B, C, H, T, k, dilation, act_elu, 0, nullptr, stream);
}

extern "C" int tt_conv_same_post(const void* x, void* y, const void* w, const float* bias, int B, int C, int H, int T, int k, int dilation,
                                 int act_elu, int post, const void* e, void* stream) {
    TT_REQUIRE(x && y && w, "null argument");
    TT_REQUIRE(post >= 0 && post <= 2 && (post == 0 || e != nullptr), "conv_same: post-op 0, 1 (times ELU'(e)) or 2 (plus e) with its tensor");
    TT_REQUIRE(C == 8 || C == 16 || C == 32, "conv_same: padded channel count must be 8, 16 or 32 (got %d)", C);
    TT_REQUIRE((k == 3 && dilation >= 1 && dilation <= 4) || k == 1, "conv_same: 3x3 (dilation 1..4) or 1x1");
    if (B <= 0 || H <= 0 || T <= 0) return TT_OK;
    static float* zero_bias = nullptr;
    if (!bias) {
        if (!zero_bias) {
            TT_CUDA_CHECK(cudaMalloc((void**)&zero_bias, 256 * sizeof(float)));
            TT_CUDA_CHECK(cudaMemset(zero_bias, 0, 256 * sizeof(float)));
        }
        bias = zero_bias;
    }
    ConvRowsParams p;
    const int d = k == 3 ? dilation : 0, CG = C / 8;
    fill_common(p, x, y, w, bias, B, CG, H, T, CG, H);
    p.groups = H;
    p.R = std::min(C == 8 ? 16 : (C == 16 ? 8 : 4), kMaxRows);
    p.sh = 1; p.row_lo = -d; p.in_rows = p.R + 2 * d; p.padT = d;
    p.out_mode = 0; p.act = act_elu; p.post = post; p.e = (const __nv_bfloat16*)e;
    const uint32_t TW = kTileT + 2 * d, row_bytes = TW * 16, plane = (uint32_t)p.in_rows * row_bytes;
    int m = 0;
    if (k == 3) {
        auto tap_addr = [&](int tap) { return (uint32_t)(((tap / 3) * d) * TW + (tap % 3) * d) * 16u; };
        if (CG == 1) {
            for (int t = 0; t < 10; t += 2) {
                p.tap_off[m] = tap_addr(t);
                p.tap_lbo[m] = t + 1 < 9 ? tap_addr(t + 1) - tap_addr(t) : 16u;
                ++m;
            }
            p.kg1 = 10;
        } else {
            for (int t = 0; t < 9; ++t)
                for (int q = 0; q < CG / 2; ++q) { p.tap_off[m] = tap_addr(t) + (uint32_t)(2 * q) * plane; p.tap_lbo[m] = plane; ++m; }
            p.kg1 = 9 * CG;
        }
    } else {
        if (CG == 1) { p.tap_off[m] = 0; p.tap_lbo[m] = 16u; ++m; p.kg1 = 2; }
        else { for (int q = 0; q < CG / 2; ++q) { p.tap_off[m] = (uint32_t)(2 * q) * plane; p.tap_lbo[m] = plane; ++m; } p.kg1 = CG; }
    }
    p.n_mma1 = m;
    return dispatch_n1(p, std::max(16, C), (cudaStream_t)stream);
}

// Decoder.convin (+ELU): ConvTranspose2d(latent+1, C0, (H0,1)) on a height-1 input = one GEMM per output row h with
// its own weight slice W[:, :, h]; the indicator channel (modules.py:139-142) is folded into a per-row bias table.
//   lat (B, Clat/8, 1, T, 8) -> y (B, C0/8, H0, T, 8);  w packed [H0][Clat/8][C0][8];  bias [H0][C0]
extern "C" int tt_deconv_in(const void* lat, void* y, const void* w, const float* bias, int B, int Clat, int C0, int H0, int T,
                            int act_elu, void* stream) {
    TT_REQUIRE(lat && y && w && bias, "null argument");
    TT_REQUIRE(Clat % 16 == 0 && Clat <= 256 && (C0 == 16 || C0 == 32 || C0 == 64 || C0 == 128), "deconv_in: unsupported sizes");
    if (B <= 0 || T <= 0) return TT_OK;
    ConvRowsParams p;
    const int CG = Clat / 8;
    fill_common(p, lat, y, w, bias, B, CG, 1, T, C0 / 8, H0);
    p.groups = H0;
    p.R = 4;
    p.sh = 0; p.row_lo = 0; p.in_rows = 1; p.padT = 0;
    p.out_mode = 0; p.act = act_elu;
    const uint32_t plane = kTileT * 16;
    int m = 0;
    for (int q = 0; q < CG / 2; ++q) { p.tap_off[m] = 2 * q * plane; p.tap_lbo[m] = plane; ++m; }
    p.n_mma1 = m; p.kg1 = CG;
    p.w_group_stride = CG * C0 * 16;
    p.b_group_stride = C0;
    return dispatch_n1(p, C0, (cudaStream_t)stream);
}

// =========================================================================================================
// Encoder.convlat (modules.py:446,478): Conv2d(C4, latent, (H4,1)) over the full height -> one GEMM over T with
// K = H4 * C4 streamed through a two-stage shared-memory ring (A = input row kh, B = weight slice kh).
//   x (B, C4/8, H4, T, 8) -> lat (B, NL/8, 1, T, 8);  w packed [H4 * C4/8][NL][8];  no activation
// =========================================================================================================
namespace tt {

// barriers, TMEM slot and the bias (NL floats) ahead of the two stages; 1024 B would hold only 224 bias values
constexpr int kLatHeader = 2048;

template <int NL>
__global__ void __launch_bounds__(128) conv_lat_kernel(const __nv_bfloat16* __restrict__ x, __nv_bfloat16* __restrict__ lat,
                                                       const __nv_bfloat16* __restrict__ w, const float* __restrict__ bias,
                                                       int CG, int H, int T) {
    extern __shared__ __align__(1024) uint8_t smem[];
    uint64_t* bar_free = reinterpret_cast<uint64_t*>(smem);          // [2] stage consumed by the tensor core
    uint64_t* bar_done = bar_free + 2;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + 64);
    float* sBias = reinterpret_cast<float*>(smem + 128);                 // NL <= 256 floats: up to smem + 1152
    const uint32_t a_bytes = (uint32_t)CG * kTileT * 16u, b_bytes = (uint32_t)CG * NL * 16u;
    uint8_t* stage0 = smem + kLatHeader;
    const uint32_t stage_bytes = a_bytes + b_bytes;

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int t0 = blockIdx.x * kTileT, b = blockIdx.y;
    constexpr uint32_t ncols = NL < 32 ? 32 : NL;
    if (warp == 0) umma::tmem_alloc(tmem_slot, ncols);
    if (tid == 0) {
        umma::mbar_init(&bar_free[0], 1);
        umma::mbar_init(&bar_free[1], 1);
        umma::mbar_init(bar_done, 1);
        umma::mbar_fence_init();
    }
    for (int i = tid; i < NL; i += 128) sBias[i] = bias[i];
    umma::fence_before_sync();
    __syncthreads();
    umma::fence_after_sync();
    const uint32_t tmem = *tmem_slot;
    const uint32_t idesc = umma::make_idesc_bf16(128, NL);

    for (int kh = 0; kh < H; ++kh) {
        const int s = kh & 1;
        uint8_t* sA = stage0 + (size_t)s * stage_bytes;
        uint8_t* sB = sA + a_bytes;
        if (kh >= 2) {
            umma::mbar_wait(&bar_free[s], (uint32_t)(((kh >> 1) - 1) & 1));
            umma::fence_after_sync();
        }
        for (int i = tid; i < CG * kTileT; i += 128) {
            const int cg = i / kTileT, c = i - cg * kTileT;
            uint4 v = make_uint4(0u, 0u, 0u, 0u);
            if (t0 + c < T) v = __ldg(reinterpret_cast<const uint4*>(x) + (((size_t)b * CG + cg) * H + kh) * T + t0 + c);
            reinterpret_cast<uint4*>(sA)[i] = v;
        }
        const uint4* wsrc = reinterpret_cast<const uint4*>(w) + (size_t)kh * CG * NL;
        for (int i = tid; i < CG * NL; i += 128) reinterpret_cast<uint4*>(sB)[i] = __ldg(wsrc + i);
        umma::fence_proxy_async();
        umma::fence_before_sync();
        __syncthreads();
        umma::fence_after_sync();
        if (tid == 0) {
            const uint32_t a0 = umma::smem_u32(sA), b0 = umma::smem_u32(sB);
            for (int m = 0; m < CG / 2; ++m) {
                const uint64_t da = umma::make_desc(a0 + (uint32_t)m * 2u * kTileT * 16u, kTileT * 16u, 128u);
                const uint64_t db = umma::make_desc(b0 + (uint32_t)m * 2u * NL * 16u, NL * 16u, 128u);
                umma::mma_bf16(tmem, da, db, idesc, kh > 0 || m > 0);
            }
            umma::commit(&bar_free[s]);
            if (kh == H - 1) umma::commit(bar_done);
        }
    }
    umma::mbar_wait(bar_done, 0);
    umma::fence_after_sync();
    const int j = warp * 32 + lane;
    const uint32_t lane_addr = tmem + ((uint32_t)(warp * 32) << 16);
#pragma unroll
    for (int c0 = 0; c0 < NL; c0 += 16) {
        float v[16];
        umma::tmem_ld16(lane_addr + (uint32_t)c0, v);
        umma::tmem_ld_wait();
#pragma unroll
        for (int k = 0; k < 16; ++k) v[k] += sBias[c0 + k];
        if (t0 + j < T) {
            reinterpret_cast<uint4*>(lat)[((size_t)b * (NL / 8) + (c0 >> 3)) * T + t0 + j] = pack8(v);
            reinterpret_cast<uint4*>(lat)[((size_t)b * (NL / 8) + (c0 >> 3) + 1) * T + t0 + j] = pack8(v + 8);
        }
    }
    umma::fence_before_sync();
    __syncthreads();
    if (warp == 0) umma::tmem_dealloc(tmem, ncols);
}

// =========================================================================================================
// Encoder.convin (modules.py:430-433): Conv2d(2, C0, 3, 'same') + ELU, reading the CQT's fp32 interleaved
// (B, F, T, 2) buffer directly and writing C8 planar bf16.  K = 18: CUDA cores, one thread per pixel.
// Decoder.convout (modules.py:543): Conv2d(C, 2, 3, 'same'), C8 planar bf16 -> fp32 interleaved (B, F, T, 2),
// optionally scaled by a per-frame window and accumulated (chunk cross-fade of modules.py:259-263).
// =========================================================================================================
// Each thread produces 4 consecutive frames of one row: the 3 x 6 input window is loaded once and reused by the 4 outputs.
template <int NC>   // output channels computed (4 or 8)
__global__ void __launch_bounds__(128) conv_in_kernel(const float2* __restrict__ x, __nv_bfloat16* __restrict__ y,
                                                      const float* __restrict__ w /* [C0][2][3][3] */,
                                                      const float* __restrict__ bias, int C0, int H, int T, int packed4) {
    __shared__ float sw[NC * 18 + NC];
    for (int i = threadIdx.x; i < NC * 18 + NC; i += 128) {
        float v = 0.f;
        if (i < NC * 18) { if (i < C0 * 18) v = w[i]; }
        else if (i - NC * 18 < C0) v = bias[i - NC * 18];
        sw[i] = v;
    }
    __syncthreads();
    const int t0 = (blockIdx.x * 128 + threadIdx.x) * 4;
    const int h = blockIdx.y, b = blockIdx.z;
    if (t0 >= T) return;
    float acc[4][NC];
#pragma unroll
    for (int o = 0; o < 4; ++o)
#pragma unroll
        for (int c = 0; c < NC; ++c) acc[o][c] = sw[NC * 18 + c];
    const float2* xb = x + (size_t)b * H * T;
#pragma unroll
    for (int ky = 0; ky < 3; ++ky) {
        const int hh = h + ky - 1;
        if (hh < 0 || hh >= H) continue;
        float2 v[6];
#pragma unroll
        for (int i = 0; i < 6; ++i) {
            const int tt_ = t0 - 1 + i;
            v[i] = (tt_ >= 0 && tt_ < T) ? __ldg(xb + (size_t)hh * T + tt_) : make_float2(0.f, 0.f);
        }
#pragma unroll
        for (int kx = 0; kx < 3; ++kx)
#pragma unroll
            for (int c = 0; c < NC; ++c) {
                const float wr = sw[c * 18 + ky * 3 + kx], wi = sw[c * 18 + 9 + ky * 3 + kx];
#pragma unroll
                for (int o = 0; o < 4; ++o) acc[o][c] = fmaf(wi, v[o + kx].y, fmaf(wr, v[o + kx].x, acc[o][c]));
            }
    }
    if (packed4) {
        // (B, H, T, 4) bf16: 4 frames x 4 channels = 32 contiguous bytes per thread (T % 4 == 0)
        float r[16];
#pragma unroll
        for (int o = 0; o < 4; ++o)
#pragma unroll
            for (int c = 0; c < 4; ++c) r[4 * o + c] = (c < NC && c < C0) ? elu(acc[o][c < NC ? c : 0]) : 0.f;
        uint4* dst4 = reinterpret_cast<uint4*>(reinterpret_cast<uint2*>(y) + ((size_t)b * H + h) * T + t0);
        dst4[0] = pack8(r);
        dst4[1] = pack8(r + 8);
        return;
    }
    uint4* dst = reinterpret_cast<uint4*>(y) + ((size_t)b * H + h) * T + t0;
#pragma unroll
    for (int o = 0; o < 4; ++o) {
        if (t0 + o >= T) break;
        float r[8];
#pragma unroll
        for (int c = 0; c < 8; ++c) r[c] = (c < NC && c < C0) ? elu(acc[o][c < NC ? c : 0]) : 0.f;
        dst[o] = pack8(r);
    }
}

template <int NC>   // input channels read (4 or 8)
__global__ void __launch_bounds__(128) conv_out_kernel(const __nv_bfloat16* __restrict__ x, float2* __restrict__ y,
                                                       const float* __restrict__ w /* [2][C][3][3] */,
                                                       const float* __restrict__ bias, int C, int H, int T, int packed4) {
    __shared__ float sw[2 * NC * 9 + 2];
    for (int i = threadIdx.x; i < 2 * NC * 9 + 2; i += 128) {
        float v = 0.f;
        if (i < 2 * NC * 9) {
            const int o = i / (NC * 9), c = (i % (NC * 9)) / 9, k = i % 9;
            if (c < C) v = w[(o * C + c) * 9 + k];
        } else v = bias[i - 2 * NC * 9];
        sw[i] = v;
    }
    __syncthreads();
    const int t0 = (blockIdx.x * 128 + threadIdx.x) * 4;
    const int h = blockIdx.y, b = blockIdx.z;
    if (t0 >= T) return;
    float a0[4], a1[4];
#pragma unroll
    for (int o = 0; o < 4; ++o) { a0[o] = sw[2 * NC * 9]; a1[o] = sw[2 * NC * 9 + 1]; }
    const uint4* xb = reinterpret_cast<const uint4*>(x) + (size_t)b * H * T;
#pragma unroll
    for (int ky = 0; ky < 3; ++ky) {
        const int hh = h + ky - 1;
        if (hh < 0 || hh >= H) continue;
        float v[6][NC];
#pragma unroll
        for (int i = 0; i < 6; ++i) {
            const int tt_ = t0 - 1 + i;
            const bool ok = tt_ >= 0 && tt_ < T;
            if constexpr (NC == 4) {
                const uint2* src = packed4 ? reinterpret_cast<const uint2*>(x) + ((size_t)b * H + hh) * T + tt_
                                           : reinterpret_cast<const uint2*>(xb + (size_t)hh * T + tt_);
                const uint2 raw = ok ? __ldg(src) : make_uint2(0u, 0u);
                const float2 f0 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&raw.x));
                const float2 f1 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&raw.y));
                v[i][0] = f0.x; v[i][1] = f0.y; v[i][2] = f1.x; v[i][3] = f1.y;
            } else {
                float tmp[8];
                unpack8(ok ? __ldg(xb + (size_t)hh * T + tt_) : make_uint4(0u, 0u, 0u, 0u), tmp);
#pragma unroll
                for (int c = 0; c < NC; ++c) v[i][c] = tmp[c];
            }
        }
#pragma unroll
        for (int kx = 0; kx < 3; ++kx)
#pragma unroll
            for (int c = 0; c < NC; ++c) {
                const float w0 = sw[c * 9 + ky * 3 + kx], w1 = sw[NC * 9 + c * 9 + ky * 3 + kx];
#pragma unroll
                for (int o = 0; o < 4; ++o) {
                    a0[o] = fmaf(w0, v[o + kx][c], a0[o]);
                    a1[o] = fmaf(w1, v[o + kx][c], a1[o]);
                }
            }
    }
    float2* dst = y + ((size_t)b * H + h) * T + t0;
    if (t0 + 3 < T) {
        reinterpret_cast<float4*>(dst)[0] = make_float4(a0[0], a1[0], a0[1], a1[1]);
        reinterpret_cast<float4*>(dst)[1] = make_float4(a0[2], a1[2], a0[3], a1[3]);
    } else {
        for (int o = 0; o < 4 && t0 + o < T; ++o) dst[o] = make_float2(a0[o], a1[o]);
    }
}


// ---------------------------------------------------------------------------------------------------------
// Row-walking variants for the packed 4-channel layout (the model's first / last layer: the largest tensors).
// A thread owns 4 consecutive frames and walks down a strip of rows: every input row is loaded ONCE and its contributions to the
// three output rows it touches are accumulated in registers (three rotating accumulator sets: when input row r has been added,
// output row r-1 is complete and is stored).  Output-channel pairs are packed f32x2 accumulators (FFMA2: half the FMA instructions).
// ---------------------------------------------------------------------------------------------------------
__device__ __forceinline__ float2 dup2(float v) { return make_float2(v, v); }

// Decoder.convout, packed4 input (B, H, T, 4) bf16 -> fp32 interleaved (B, H, T, 2)
__global__ void __launch_bounds__(128) conv_out_p4_kernel(const uint2* __restrict__ x, float2* __restrict__ y, const float* __restrict__ w /* [2][C][3][3] */,
                                                          const float* __restrict__ bias, int C, int H, int T, int rows) {
    __shared__ __align__(16) float2 sw[3][3][4];     // [ky][kx][c] -> (w for output 0, w for output 1)
    __shared__ float2 sb;
    for (int i = threadIdx.x; i < 36; i += 128) {
        const int ky = i / 12, kx = (i / 4) % 3, c = i % 4;
        sw[ky][kx][c] = c < C ? make_float2(w[(0 * C + c) * 9 + ky * 3 + kx], w[(1 * C + c) * 9 + ky * 3 + kx]) : make_float2(0.f, 0.f);
    }
    if (threadIdx.x == 0) sb = make_float2(bias[0], bias[1]);
    __syncthreads();
    const int t0 = (blockIdx.x * 128 + threadIdx.x) * 4;
    if (t0 >= T) return;
    const int b = blockIdx.z, h0 = blockIdx.y * rows, h1 = min(H, h0 + rows);
    const float2 bias2 = sb;
    float2 P[4], Q[4], R[4];
#pragma unroll
    for (int f = 0; f < 4; ++f) P[f] = Q[f] = R[f] = bias2;
    const uint2* xb = x + (size_t)b * H * T + t0;
    float2* yb = y + (size_t)b * H * T + t0;
    // the six frames t0-1 .. t0+4 of input row hh (zeros outside the image); issued one row ahead of their use
    auto load = [&](int hh, uint2 (&raw)[6]) {
        if (hh >= 0 && hh < H) {
            const uint2* xr = xb + (size_t)hh * T;
            const uint4 m0 = __ldg(reinterpret_cast<const uint4*>(xr)), m1 = __ldg(reinterpret_cast<const uint4*>(xr) + 1);
            raw[0] = t0 > 0 ? __ldg(xr - 1) : make_uint2(0u, 0u);
            raw[1] = make_uint2(m0.x, m0.y); raw[2] = make_uint2(m0.z, m0.w);
            raw[3] = make_uint2(m1.x, m1.y); raw[4] = make_uint2(m1.z, m1.w);
            raw[5] = t0 + 4 < T ? __ldg(xr + 4) : make_uint2(0u, 0u);
        }
    };
    uint2 raw[6], nxt[6];
    // input row hh: += into A (output row hh-1, ky = 2), Bq (row hh, ky = 1), Cq (row hh+1, ky = 0); then A is complete
    auto step = [&](int hh, float2 (&A)[4], float2 (&Bq)[4], float2 (&Cq)[4]) {
        if (hh < h1) load(hh + 1, nxt);
        if (hh >= 0 && hh < H) {
#pragma unroll
            for (int i = 0; i < 6; ++i) {
                const float v[4] = {__uint_as_float(raw[i].x << 16), __uint_as_float(raw[i].x & 0xFFFF0000u),
                                    __uint_as_float(raw[i].y << 16), __uint_as_float(raw[i].y & 0xFFFF0000u)};
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    const float2 vv = dup2(v[c]);
#pragma unroll
                    for (int kx = 0; kx < 3; ++kx) {
                        const int f = i - kx;
                        if (f >= 0 && f < 4) {
                            Cq[f] = __ffma2_rn(vv, sw[0][kx][c], Cq[f]);
                            Bq[f] = __ffma2_rn(vv, sw[1][kx][c], Bq[f]);
                            A[f] = __ffma2_rn(vv, sw[2][kx][c], A[f]);
                        }
                    }
                }
            }
        }
        const int ho = hh - 1;
        if (ho >= h0 && ho < h1) {
            float4* dst = reinterpret_cast<float4*>(yb + (size_t)ho * T);
            dst[0] = make_float4(A[0].x, A[0].y, A[1].x, A[1].y);
            dst[1] = make_float4(A[2].x, A[2].y, A[3].x, A[3].y);
        }
#pragma unroll
        for (int f = 0; f < 4; ++f) A[f] = bias2;
#pragma unroll
        for (int i = 0; i < 6; ++i) raw[i] = nxt[i];
    };
    int hh = h0 - 1;
    load(hh, raw);
    while (true) {
        step(hh, P, Q, R); if (++hh > h1) break;
        step(hh, Q, R, P); if (++hh > h1) break;
        step(hh, R, P, Q); if (++hh > h1) break;
    }
}

// Decoder.convout FUSED with the Hann cross-fade of 50 %-overlapped chunks and the trim (TimbreTrap.chunked_inference,
// modules.py:237-267), optionally with tanh|.| (TimbreTrap.to_activations, modules.py:271-289): output frame t of item b (after
// the M/2 trim) is  window[p + M/2] * convout(chunk i-1)[p + M/2] + window[p] * convout(chunk i)[p]  with i = t / (M/2) + 1,
// p = t mod (M/2).  A thread owns 4 output frames and walks down the rows of BOTH source chunks (two accumulator sets), so the
// per-chunk fp32 coefficients (2 x 8.8 MB per block) never exist in HBM: read 2 x 4 channels bf16, write one fp32 pair (or one
// fp32 activation) per output frame.  Products are rounded separately and added in chunk order, like the reference's
// `coefficients[...] += window * chunk` (and like crossfade_kernel, which remains for the un-fused API path).
//   x (batch * n_chunks, H, M, 4) bf16 packed4;  coeffs_out (batch, H, (n_chunks-1) M/2, 2) and / or act_out (batch, H, (n_chunks-1) M/2)
// blockIdx.z is the item.  With clip_chunk0 (the many-clip calls) it is clip z of the chunk prefix table instead (find_clip): its
// n = clip_chunk0[z + 1] - clip_chunk0[z] chunks and its (H, (n - 1) M/2) outputs follow those of the clips before it, and the grid
// covers the longest clip (a CTA never straddles two clips; the CTAs past a shorter clip's end do nothing).
__global__ void __launch_bounds__(128) conv_out_xfade_p4_kernel(const uint2* __restrict__ x, const float* __restrict__ window,
                                                                const float* __restrict__ w /* [2][C][3][3] */, const float* __restrict__ bias,
                                                                int C, int H, int M, int n_chunks, int rows, float2* __restrict__ coeffs_out,
                                                                float* __restrict__ act_out, const int* __restrict__ clip_chunk0) {
    __shared__ __align__(16) float2 sw[3][3][4];     // [ky][kx][c] -> (w for output 0, w for output 1)
    __shared__ float2 sb;
    for (int i = threadIdx.x; i < 36; i += 128) {
        const int ky = i / 12, kx = (i / 4) % 3, c = i % 4;
        sw[ky][kx][c] = c < C ? make_float2(w[(0 * C + c) * 9 + ky * 3 + kx], w[(1 * C + c) * 9 + ky * 3 + kx]) : make_float2(0.f, 0.f);
    }
    if (threadIdx.x == 0) sb = make_float2(bias[0], bias[1]);
    __syncthreads();
    const int half = M / 2;
    const int b = blockIdx.z, h0 = blockIdx.y * rows, h1 = min(H, h0 + rows);
    size_t chunk0 = (size_t)b * n_chunks;                        // the item's first chunk
    if (clip_chunk0) {
        chunk0 = (size_t)(__ldg(clip_chunk0 + b) - __ldg(clip_chunk0));
        n_chunks = __ldg(clip_chunk0 + b + 1) - __ldg(clip_chunk0 + b);
    }
    const long long n_out = (long long)(n_chunks - 1) * half;
    const long long t0 = ((long long)blockIdx.x * 128 + threadIdx.x) * 4;
    if (t0 >= n_out) return;
    // the item's outputs: after those of its predecessors, (n_c - 1) M/2 frames of H rows each, i.e. chunk0 - b times H * half
    const size_t out0 = (size_t)H * half * (chunk0 - b);
    const int i1 = (int)(t0 / half) + 1;                         // the later chunk; the earlier one is i1 - 1
    const int p1 = (int)(t0 - (long long)(i1 - 1) * half);       // position in the later chunk; + half in the earlier one
    // source s = 0: earlier chunk at frames p1 + half .., s = 1: later chunk at frames p1 ..
    const int pos[2] = {p1 + half, p1};
    const uint2* xs[2] = {x + (chunk0 + i1 - 1) * H * M + pos[0], x + (chunk0 + i1) * H * M + pos[1]};
    const float4 wv0 = __ldg(reinterpret_cast<const float4*>(window + pos[0])), wv1 = __ldg(reinterpret_cast<const float4*>(window + pos[1]));
    const float win[2][4] = {{wv0.x, wv0.y, wv0.z, wv0.w}, {wv1.x, wv1.y, wv1.z, wv1.w}};
    const float2 bias2 = sb;
    float2 P[2][4], Q[2][4], R[2][4];
#pragma unroll
    for (int s = 0; s < 2; ++s)
#pragma unroll
        for (int f = 0; f < 4; ++f) P[s][f] = Q[s][f] = R[s][f] = bias2;
    auto load = [&](int hh, uint2 (&raw)[2][6]) {
        if (hh >= 0 && hh < H) {
#pragma unroll
            for (int s = 0; s < 2; ++s) {
                const uint2* xr = xs[s] + (size_t)hh * M;
                const uint4 m0 = __ldg(reinterpret_cast<const uint4*>(xr)), m1 = __ldg(reinterpret_cast<const uint4*>(xr) + 1);
                raw[s][0] = pos[s] > 0 ? __ldg(xr - 1) : make_uint2(0u, 0u);          // 'same' padding at the chunk's own borders
                raw[s][1] = make_uint2(m0.x, m0.y); raw[s][2] = make_uint2(m0.z, m0.w);
                raw[s][3] = make_uint2(m1.x, m1.y); raw[s][4] = make_uint2(m1.z, m1.w);
                raw[s][5] = pos[s] + 4 < M ? __ldg(xr + 4) : make_uint2(0u, 0u);
            }
        }
    };
    uint2 raw[2][6], nxt[2][6];
    auto step = [&](int hh, float2 (&A)[2][4], float2 (&Bq)[2][4], float2 (&Cq)[2][4]) {
        if (hh < h1) load(hh + 1, nxt);
        if (hh >= 0 && hh < H) {
#pragma unroll
            for (int s = 0; s < 2; ++s) {
#pragma unroll
                for (int i = 0; i < 6; ++i) {
                    const float v[4] = {__uint_as_float(raw[s][i].x << 16), __uint_as_float(raw[s][i].x & 0xFFFF0000u),
                                        __uint_as_float(raw[s][i].y << 16), __uint_as_float(raw[s][i].y & 0xFFFF0000u)};
#pragma unroll
                    for (int c = 0; c < 4; ++c) {
                        const float2 vv = dup2(v[c]);
#pragma unroll
                        for (int kx = 0; kx < 3; ++kx) {
                            const int f = i - kx;
                            if (f >= 0 && f < 4) {
                                Cq[s][f] = __ffma2_rn(vv, sw[0][kx][c], Cq[s][f]);
                                Bq[s][f] = __ffma2_rn(vv, sw[1][kx][c], Bq[s][f]);
                                A[s][f] = __ffma2_rn(vv, sw[2][kx][c], A[s][f]);
                            }
                        }
                    }
                }
            }
        }
        const int ho = hh - 1;
        if (ho >= h0 && ho < h1) {
            float2 r[4];
#pragma unroll
            for (int f = 0; f < 4; ++f) {
                r[f].x = __fadd_rn(__fmul_rn(win[0][f], A[0][f].x), __fmul_rn(win[1][f], A[1][f].x));
                r[f].y = __fadd_rn(__fmul_rn(win[0][f], A[0][f].y), __fmul_rn(win[1][f], A[1][f].y));
            }
            const size_t o = out0 + (size_t)ho * n_out + t0;
            if (coeffs_out) {
                float4* dst = reinterpret_cast<float4*>(coeffs_out + o);
                __stcs(dst, make_float4(r[0].x, r[0].y, r[1].x, r[1].y));
                __stcs(dst + 1, make_float4(r[2].x, r[2].y, r[3].x, r[3].y));
            }
            if (act_out) {
                float a[4];
#pragma unroll
                for (int f = 0; f < 4; ++f) a[f] = tanhf(sqrtf(r[f].x * r[f].x + r[f].y * r[f].y));
                __stcs(reinterpret_cast<float4*>(act_out + o), make_float4(a[0], a[1], a[2], a[3]));
            }
        }
#pragma unroll
        for (int s = 0; s < 2; ++s) {
#pragma unroll
            for (int f = 0; f < 4; ++f) A[s][f] = bias2;
#pragma unroll
            for (int i = 0; i < 6; ++i) raw[s][i] = nxt[s][i];
        }
    };
    int hh = h0 - 1;
    load(hh, raw);
    while (true) {
        step(hh, P, Q, R); if (++hh > h1) break;
        step(hh, Q, R, P); if (++hh > h1) break;
        step(hh, R, P, Q); if (++hh > h1) break;
    }
}

// Encoder.convin, fp32 interleaved (B, H, T, 2) -> packed4 (B, H, T, 4) bf16, + ELU
__global__ void __launch_bounds__(128) conv_in_p4_kernel(const float2* __restrict__ x, uint2* __restrict__ y, const float* __restrict__ w /* [C0][2][3][3] */,
                                                         const float* __restrict__ bias, int C0, int H, int T, int rows, int act) {
    __shared__ __align__(16) float2 sw[3][3][2][2];  // [ky][kx][re/im][channel pair] -> (w for channel 2p, 2p+1)
    __shared__ float2 sb[2];
    for (int i = threadIdx.x; i < 36; i += 128) {
        const int ky = i / 12, kx = (i / 4) % 3, comp = (i / 2) % 2, pr = i % 2;
        const int c0 = 2 * pr, c1 = 2 * pr + 1;
        sw[ky][kx][comp][pr] = make_float2(c0 < C0 ? w[(c0 * 2 + comp) * 9 + ky * 3 + kx] : 0.f, c1 < C0 ? w[(c1 * 2 + comp) * 9 + ky * 3 + kx] : 0.f);
    }
    if (threadIdx.x < 2) sb[threadIdx.x] = make_float2(2 * threadIdx.x < C0 ? bias[2 * threadIdx.x] : 0.f, 2 * threadIdx.x + 1 < C0 ? bias[2 * threadIdx.x + 1] : 0.f);
    __syncthreads();
    const int t0 = (blockIdx.x * 128 + threadIdx.x) * 4;
    if (t0 >= T) return;
    const int b = blockIdx.z, h0 = blockIdx.y * rows, h1 = min(H, h0 + rows);
    const float2 b01 = sb[0], b23 = sb[1];
    float2 P[4][2], Q[4][2], R[4][2];
#pragma unroll
    for (int f = 0; f < 4; ++f) { P[f][0] = Q[f][0] = R[f][0] = b01; P[f][1] = Q[f][1] = R[f][1] = b23; }
    const float2* xb = x + (size_t)b * H * T + t0;
    uint2* yb = y + (size_t)b * H * T + t0;
    auto load = [&](int hh, float2 (&v)[6]) {
        if (hh >= 0 && hh < H) {
            const float2* xr = xb + (size_t)hh * T;
            const float4 m0 = __ldg(reinterpret_cast<const float4*>(xr)), m1 = __ldg(reinterpret_cast<const float4*>(xr) + 1);
            v[0] = t0 > 0 ? __ldg(xr - 1) : make_float2(0.f, 0.f);
            v[1] = make_float2(m0.x, m0.y); v[2] = make_float2(m0.z, m0.w);
            v[3] = make_float2(m1.x, m1.y); v[4] = make_float2(m1.z, m1.w);
            v[5] = t0 + 4 < T ? __ldg(xr + 4) : make_float2(0.f, 0.f);
        }
    };
    float2 v[6], nxt[6];
    auto step = [&](int hh, float2 (&A)[4][2], float2 (&Bq)[4][2], float2 (&Cq)[4][2]) {
        if (hh < h1) load(hh + 1, nxt);
        if (hh >= 0 && hh < H) {
#pragma unroll
            for (int i = 0; i < 6; ++i) {
#pragma unroll
                for (int comp = 0; comp < 2; ++comp) {
                    const float2 vv = dup2(comp ? v[i].y : v[i].x);
#pragma unroll
                    for (int kx = 0; kx < 3; ++kx) {
                        const int f = i - kx;
                        if (f >= 0 && f < 4) {
#pragma unroll
                            for (int pr = 0; pr < 2; ++pr) {
                                Cq[f][pr] = __ffma2_rn(vv, sw[0][kx][comp][pr], Cq[f][pr]);
                                Bq[f][pr] = __ffma2_rn(vv, sw[1][kx][comp][pr], Bq[f][pr]);
                                A[f][pr] = __ffma2_rn(vv, sw[2][kx][comp][pr], A[f][pr]);
                            }
                        }
                    }
                }
            }
        }
        const int ho = hh - 1;
        if (ho >= h0 && ho < h1) {
            float r[16];
#pragma unroll
            for (int f = 0; f < 4; ++f) {
                r[4 * f] = A[f][0].x; r[4 * f + 1] = A[f][0].y; r[4 * f + 2] = A[f][1].x; r[4 * f + 3] = A[f][1].y;
            }
            if (act) {
#pragma unroll
                for (int e = 0; e < 16; ++e) r[e] = elu(r[e]);
            }
            uint4* dst = reinterpret_cast<uint4*>(yb + (size_t)ho * T);
            dst[0] = pack8(r);
            dst[1] = pack8(r + 8);
        }
#pragma unroll
        for (int f = 0; f < 4; ++f) { A[f][0] = b01; A[f][1] = b23; }
#pragma unroll
        for (int i = 0; i < 6; ++i) v[i] = nxt[i];
    };
    int hh = h0 - 1;
    load(hh, v);
    while (true) {
        step(hh, P, Q, R); if (++hh > h1) break;
        step(hh, Q, R, P); if (++hh > h1) break;
        step(hh, R, P, Q); if (++hh > h1) break;
    }
}

// rows per CTA of the row-walking kernels: long strips amortise the two halo rows, short ones keep small batches parallel
static inline int walk_rows(int B, int H, int T) {
    const long long ctas_per_row_strip = (long long)B * ((T / 4 + 127) / 128);
    int rows = 36;
    while (rows > 6 && ctas_per_row_strip * ((H + rows - 1) / rows) < 4 * 148) rows /= 2;
    return rows;
}

}  // namespace tt

extern "C" int tt_conv_lat(const void* x, void* lat, const void* w, const float* bias, int B, int C4, int H4, int NL, int T,
                           void* stream) {
    TT_REQUIRE(x && lat && w && bias, "null argument");
    TT_REQUIRE(C4 % 16 == 0 && C4 <= 128, "conv_lat: input channels must be a multiple of 16 (<= 128), got %d", C4);
    if (B <= 0 || T <= 0) return TT_OK;
    const int CG = C4 / 8;
    dim3 grid((T + kTileT - 1) / kTileT, B);
    const size_t smem = kLatHeader + 2 * ((size_t)CG * kTileT * 16 + (size_t)CG * NL * 16);
    cudaStream_t s = (cudaStream_t)stream;
#define TT_LAT_CASE(N)                                                                                               \
    case N:                                                                                                          \
        TT_CUDA_CHECK(cudaFuncSetAttribute(conv_lat_kernel<N>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
        conv_lat_kernel<N><<<grid, 128, smem, s>>>((const __nv_bfloat16*)x, (__nv_bfloat16*)lat, (const __nv_bfloat16*)w, bias, CG, H4, T); \
        break;
    switch (NL) {
        TT_LAT_CASE(16) TT_LAT_CASE(32) TT_LAT_CASE(64) TT_LAT_CASE(128) TT_LAT_CASE(256)
        default: tt_set_error("conv_lat: padded latent size must be 16, 32, 64, 128 or 256 (got %d)", NL); return TT_ERR_UNSUPPORTED;
    }
#undef TT_LAT_CASE
    tt_count_launches(1);
    TT_CUDA_CHECK(cudaGetLastError());
    return TT_OK;
}

// packed4: 0 = C8 planar output, 1 = packed 4-channel output, 2 = packed 4-channel output WITHOUT the ELU (the data gradient of
// Decoder.convout in the loss step: a 2 -> 4 channel 3x3 conv of the fp32 coefficient gradient with transposed, flipped weights)
extern "C" int tt_conv_in(const float* coeffs, void* y, const float* w, const float* bias, int B, int C0, int H, int T, int packed4,
                          void* stream) {
    TT_REQUIRE(coeffs && y && w && bias, "null argument");
    TT_REQUIRE(C0 >= 1 && C0 <= 8, "conv_in: at most 8 output channels");
    if (B <= 0 || H <= 0 || T <= 0) return TT_OK;
    TT_REQUIRE(T % 4 == 0, "conv_in: the frame count must be a multiple of 4 (got %d)", T);
    dim3 grid((T / 4 + 127) / 128, H, B);
    TT_REQUIRE(!packed4 || C0 <= 4, "conv_in: the packed layout holds at most 4 channels");
    if (packed4) {
        const int rows = walk_rows(B, H, T);
        conv_in_p4_kernel<<<dim3((T / 4 + 127) / 128, (H + rows - 1) / rows, B), 128, 0, (cudaStream_t)stream>>>((const float2*)coeffs, (uint2*)y, w, bias, C0,
                                                                                                            H, T, rows, packed4 != 2);
    } else if (C0 <= 4) conv_in_kernel<4><<<grid, 128, 0, (cudaStream_t)stream>>>((const float2*)coeffs, (__nv_bfloat16*)y, w, bias, C0, H, T, packed4);
    else conv_in_kernel<8><<<grid, 128, 0, (cudaStream_t)stream>>>((const float2*)coeffs, (__nv_bfloat16*)y, w, bias, C0, H, T, 0);
    tt_count_launches(1);
    TT_CUDA_CHECK(cudaGetLastError());
    return TT_OK;
}

extern "C" int tt_conv_out(const void* x, float* coeffs, const float* w, const float* bias, int B, int C, int H, int T, int packed4,
                           void* stream) {
    TT_REQUIRE(x && coeffs && w && bias, "null argument");
    TT_REQUIRE(C >= 1 && C <= 8, "conv_out: at most 8 input channels");
    if (B <= 0 || H <= 0 || T <= 0) return TT_OK;
    TT_REQUIRE(T % 4 == 0, "conv_out: the frame count must be a multiple of 4 (got %d)", T);
    dim3 grid((T / 4 + 127) / 128, H, B);
    TT_REQUIRE(!packed4 || C <= 4, "conv_out: the packed layout holds at most 4 channels");
    if (packed4) {
        const int rows = walk_rows(B, H, T);
        conv_out_p4_kernel<<<dim3((T / 4 + 127) / 128, (H + rows - 1) / rows, B), 128, 0, (cudaStream_t)stream>>>((const uint2*)x, (float2*)coeffs, w, bias, C, H,
                                                                                                             T, rows);
    } else if (C <= 4) conv_out_kernel<4><<<grid, 128, 0, (cudaStream_t)stream>>>((const __nv_bfloat16*)x, (float2*)coeffs, w, bias, C, H, T, packed4);
    else conv_out_kernel<8><<<grid, 128, 0, (cudaStream_t)stream>>>((const __nv_bfloat16*)x, (float2*)coeffs, w, bias, C, H, T, 0);
    tt_count_launches(1);
    TT_CUDA_CHECK(cudaGetLastError());
    return TT_OK;
}

extern "C" int tt_conv_out_crossfade(const void* x, const float* window, const float* w, const float* bias, int batch, int n_chunks, int C,
                                     int H, int M, float* coeffs_out, float* act_out, void* stream) {
    TT_REQUIRE(x && window && w && bias && (coeffs_out || act_out), "null argument");
    TT_REQUIRE(C >= 1 && C <= 4, "conv_out_crossfade: the packed layout holds at most 4 channels");
    TT_REQUIRE(n_chunks >= 2 && M >= 8 && M % 8 == 0, "conv_out_crossfade: at least two chunks, chunk length a multiple of 8 (got %d, %d)", n_chunks, M);
    if (batch <= 0 || H <= 0) return TT_OK;
    const long long n_out = (long long)(n_chunks - 1) * (M / 2);
    const long long col_ctas = (n_out / 4 + 127) / 128;
    int rows = 36;
    while (rows > 6 && (long long)batch * col_ctas * ((H + rows - 1) / rows) < 4 * 148) rows /= 2;
    TT_REQUIRE(col_ctas < (1ll << 31), "conv_out_crossfade: clip too long for one launch");
    conv_out_xfade_p4_kernel<<<dim3((unsigned)col_ctas, (H + rows - 1) / rows, batch), 128, 0, (cudaStream_t)stream>>>(
        (const uint2*)x, window, w, bias, C, H, M, n_chunks, rows, (float2*)coeffs_out, act_out, nullptr);
    tt_count_launches(1);
    TT_CUDA_CHECK(cudaGetLastError());
    return TT_OK;
}

extern "C" int tt_conv_out_crossfade_clips(const void* x, const float* window, const float* w, const float* bias, const int* clip_chunk0,
                                           int n_clips, int total_chunks, int max_chunks, int C, int H, int M, float* coeffs_out,
                                           float* act_out, void* stream) {
    TT_REQUIRE(x && window && w && bias && clip_chunk0 && (coeffs_out || act_out), "null argument");
    TT_REQUIRE(C >= 1 && C <= 4, "conv_out_crossfade: the packed layout holds at most 4 channels");
    TT_REQUIRE(max_chunks >= 2 && M >= 8 && M % 8 == 0, "conv_out_crossfade: at least two chunks, chunk length a multiple of 8 (got %d, %d)", max_chunks, M);
    TT_REQUIRE(n_clips <= 65535, "conv_out_crossfade: at most 65535 clips per call (got %d)", n_clips);
    if (n_clips <= 0 || H <= 0) return TT_OK;
    const long long col_ctas = ((long long)(max_chunks - 1) * (M / 2) / 4 + 127) / 128;
    // strip height from the CTAs that do work (as if the chunks were one uniform batch), not from the padded grid
    const long long busy_ctas = ((long long)(total_chunks - n_clips) * (M / 2) / 4 + 127) / 128;
    int rows = 36;
    while (rows > 6 && busy_ctas * ((H + rows - 1) / rows) < 4 * 148) rows /= 2;
    TT_REQUIRE(col_ctas < (1ll << 31), "conv_out_crossfade: clip too long for one launch");
    conv_out_xfade_p4_kernel<<<dim3((unsigned)col_ctas, (H + rows - 1) / rows, n_clips), 128, 0, (cudaStream_t)stream>>>(
        (const uint2*)x, window, w, bias, C, H, M, 0, rows, (float2*)coeffs_out, act_out, clip_chunk0);
    tt_count_launches(1);
    TT_CUDA_CHECK(cudaGetLastError());
    return TT_OK;
}
