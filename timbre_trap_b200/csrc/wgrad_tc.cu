// Weight gradients of the 'same' convolutions of the residual blocks (reference: the autograd of timbre_trap/framework/modules.py:743-777
// inside the loss step, experiments/train.py:470-472) on the tensor cores.
//
//     dW[ky][kx][co][ci] = sum over (b, h, t) of  dZ[b, co, h, t] * X[b, ci, h + (ky-1) d, t + (kx-1) d]        (3x3 dilated, zero padding)
//     db[co]             = sum over (b, h, t) of  dZ[b, co, h, t]
//
// is a GEMM whose K axis is the PIXEL axis.  In the C8 planar activation layout (B, CG, H, T, 8) sixteen contiguous bytes hold 8
// channels of one pixel and consecutive pixels are 16 bytes apart: exactly the tcgen05 canonical layout of an MN-major operand
// (a core matrix = 8 k-rows of 16 bytes, SWIZZLE_NONE; LBO = 128 B between 8-pixel groups, SBO = plane stride between channel groups).
// So both operands are the rows the TMA brings in, untouched:
//     A = dZ row   (M = co, 128 lanes of which the first 8 CGo are real)             K = 16 pixels per tcgen05.mma
//     B = X row of the tap, started (kx-1) d pixels further along K (an address offset), N = ci
// A CTA walks a strip of image rows of one 128-pixel column tile (out-of-image rows arrive as zeros from the TMA), accumulates in TMEM
// for the whole life of the CTA, then writes its accumulators to a partial buffer; a second kernel sums the partials in a fixed order
// (deterministic) into the PyTorch weight layout (co, ci, kh, kw).  The 3x3 and (4,1) stride-(2,1) layers have row-stationary kernels
// (wgrad3_kernel, wgrad_ud_kernel); the 1x1 and (H, 1) layers a ring kernel (wgrad_kernel) in which every tap owns NPAD accumulator
// columns and one more "tap" multiplies dZ with a constant ones operand to yield db (the 1x1 layers sum db in otherwise idle warps).
#include <algorithm>

#include "../../include/timbre_trap_b200.h"
#include "strip_common.cuh"

namespace tt {

constexpr int kWgThreads = 128;        // warp 0: TMA producer, warp 1: MMA issuer; after the row loop warps 0-1 drain the accumulators
constexpr int kWgZSlots = 8;           // A-side row ring (upper bound; the launch picks the depth that fits)
constexpr int kWgMaxTaps = 10;         // taps + the bias "tap" a partial block of wgrad_kernel has room for (the (H, 1) layers use 7 + 1)
constexpr int kWgMaxM = 64;            // A-side channels a CTA of the row-walking geometries writes out (TMEM lanes 0..63)

struct WgradParams {
    float* partial;                    // (n_ctas, kWgMaxTaps, kWgMaxM, NPAD) fp32
    int B, T;
    int Hz, Hx;                        // rows of the A-side (dZ) and B-side (X) tensors
    int CGi, CGo;                      // channel groups of the B side (X) and the A side (dZ)
    int rows_per_strip;
    int z_slots;                       // A-side ring depth (<= kWgZSlots)
    int xring;                         // B-side ring depth (<= 16): the rows one A-side row reaches + the prefetch distance
    int tap_group;                     // 0: blockIdx.y walks strips of A-side rows; > 0: the A side has ONE row and blockIdx.y selects a
                                       // group of `tap_group` consecutive B-side rows = vertical taps (the (31,1) layers)
};

// Geometry (compile time): KH vertical taps of width 1; the B-side row of tap ky for A-side row q is  q + ky  (relative to the first
// B-side row of the CTA)
//   1x1 (KH = 1): A-side row q meets B-side row q
//   (H, 1) layers (KH = kLatTapGroup, tap_group > 0): the A side has one row, blockIdx.y selects the group of KH B-side rows
// shared memory plan (bytes): [barriers 1 KB][ones 4 KB][A ring][B ring]; the A operand reads 16 channel groups = 32 KB from its slot, the
// B operand NPAD/8 groups: both stay inside the allocation because the B ring follows and the allocation is padded (see wgrad_smem)
template <int NPAD, int KH, int MW>
__global__ void __launch_bounds__(kWgThreads, 1) wgrad_kernel(const __grid_constant__ CUtensorMap tmap_x, const __grid_constant__ CUtensorMap tmap_z,
                                                              const WgradParams p) {
    // 1x1 layers: the "ones" MMA would be every second MMA; instead warps 2-3 (idle otherwise) sum the A-side rows from shared memory
    constexpr bool BIASW = KH == 1;
    constexpr uint32_t need = (KH + 1) * NPAD;
    constexpr uint32_t ncols = need <= 32 ? 32 : (need <= 64 ? 64 : (need <= 128 ? 128 : (need <= 256 ? 256 : 512)));
    static_assert(need <= 512, "TMEM columns");
    extern __shared__ __align__(1024) uint8_t smem[];
    const int xring = p.xring;
    const uint32_t z_slot = (uint32_t)p.CGo * kStripTileT * 16u;
    const uint32_t x_plane = (uint32_t)kStripTileT * 16u;
    const uint32_t x_slot = (uint32_t)p.CGi * x_plane;
    uint64_t* z_full = reinterpret_cast<uint64_t*>(smem);            // [kWgZSlots]
    uint64_t* z_empty = z_full + kWgZSlots;                           // [kWgZSlots]
    uint64_t* x_full = z_empty + kWgZSlots;                           // [xring <= 16]
    uint64_t* x_empty = x_full + 16;                                  // [xring]
    uint64_t* done = x_empty + 16;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + 512);
    uint8_t* sOnes = smem + 1024;                                      // [2 groups][128 px][8] bf16 ones (group 1 only pads N to 16)
    uint8_t* sZ = smem + 1024 + 4096;
    uint8_t* sX = sZ + p.z_slots * z_slot;
    const int zslots = p.z_slots;

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int t0 = blockIdx.x * kStripTileT;
    const int h0 = p.tap_group ? 0 : blockIdx.y * p.rows_per_strip;
    const int h1 = p.tap_group ? p.Hz : min(p.Hz, h0 + p.rows_per_strip);
    const int b = blockIdx.z;
    const int n_rows = h1 - h0;                         // A-side rows of this strip
    const int n_xrows = n_rows + KH - 1;                // B-side rows, relative index 0 <-> image row x_row0
    const int x_row0 = p.tap_group ? blockIdx.y * p.tap_group : h0;

    if (warp == 0) umma::tmem_alloc(tmem_slot, ncols);
    if (tid == 32) {
        for (int i = 0; i < kWgZSlots; ++i) { umma::mbar_init(&z_full[i], 1); umma::mbar_init(&z_empty[i], BIASW ? 2 : 1); }
        for (int i = 0; i < xring; ++i) { umma::mbar_init(&x_full[i], 1); umma::mbar_init(&x_empty[i], 1); }
        umma::mbar_init(done, 1);
        umma::mbar_fence_init();
    }
    for (int i = tid; i < 2 * kStripTileT * 4; i += kWgThreads) reinterpret_cast<uint32_t*>(sOnes)[i] = 0x3F803F80u;   // bf16 1.0 pairs
    umma::fence_proxy_async();
    umma::fence_before_sync();
    __syncthreads();
    umma::fence_after_sync();
    const uint32_t tmem = *tmem_slot;

    if (warp == 0 && lane == 0) {
        // ================= producer: the B-side rows run ahead of the A-side rows =================
        int xr = 0;                                                    // next B-side row (relative)
        auto load_x = [&]() {
            const int slot = xr % xring;
            if (xr >= xring) umma::mbar_wait(&x_empty[slot], (uint32_t)((xr / xring - 1) & 1));
            mbar_expect_tx(&x_full[slot], (uint32_t)p.CGi * x_plane);
            tma_load_5d(sX + (size_t)slot * x_slot, &tmap_x, &x_full[slot], 0, t0, x_row0 + xr, 0, b);
            ++xr;
        };
        for (int r = 0; r < n_rows; ++r) {
            // as far ahead as the ring allows without waiting for a release that needs THIS iteration's A-side row (deadlock): the
            // slot of row xr is freed by A-side row xr - xring, which must lie before r
            while (xr < n_xrows && xr <= r + xring - 2) load_x();
            const int slot = r % zslots;
            if (r >= zslots) umma::mbar_wait(&z_empty[slot], (uint32_t)((r / zslots - 1) & 1));
            mbar_expect_tx(&z_full[slot], z_slot);
            tma_load_5d(sZ + (size_t)slot * z_slot, &tmap_z, &z_full[slot], 0, t0, h0 + r, 0, b);
        }
    } else if (warp == 1 && lane == 0) {
        // ================= MMA issuer =================
        constexpr uint32_t idesc = umma::make_idesc_bf16(128, NPAD) | (1u << 15) | (1u << 16);     // both operands MN-major
        const uint32_t z0 = umma::smem_u32(sZ), x0 = umma::smem_u32(sX), ones0 = umma::smem_u32(sOnes);
        bool first = true;                                             // the very first MMA of every accumulator overwrites
        for (int r = 0; r < n_rows; ++r) {
            const int zs = r % zslots;
            umma::mbar_wait(&z_full[zs], (uint32_t)((r / zslots) & 1));
            // B-side rows r .. r + KH - 1; those beyond what row r - 1 already waited for may still be in flight
            for (int xr = (r == 0 ? 0 : r + KH - 1); xr <= r + KH - 1; ++xr)
                umma::mbar_wait(&x_full[xr % xring], (uint32_t)((xr / xring) & 1));
            umma::fence_after_sync();
            const uint32_t za = z0 + (uint32_t)zs * z_slot;
            // Descriptors: the high word (group stride, version bit) is constant per operand kind, the low word is (address >> 4) with
            // the k-group stride 128 B in bits 16-29; a K step of 16 pixels advances the address field by 256 B >> 4 = 16.  Everything
            // below is 32-bit adds in the one issuing thread (its instruction stream, not the tensor pipe, bounds this kernel).
            constexpr uint32_t lbo_field = (128u >> 4) << 16;
            const uint32_t hi_a = ((uint32_t)(kStripTileT * 16) >> 4) | (1u << 14);
            const uint32_t hi_b = (x_plane >> 4) | (1u << 14);
            const uint32_t lo_a = ((za >> 4) & 0x3FFFu) | lbo_field, lo_ones = ((ones0 >> 4) & 0x3FFFu) | lbo_field;
            uint32_t lo_b[KH];
#pragma unroll
            for (int ky = 0; ky < KH; ++ky) lo_b[ky] = (((x0 + (uint32_t)((r + ky) % xring) * x_slot) >> 4) & 0x3FFFu) | lbo_field;
            auto d64 = [](uint32_t hi, uint32_t lo) { return ((uint64_t)hi << 32) | lo; };
#pragma unroll
            for (int s = 0; s < kStripTileT / 16; ++s) {
                const bool acc = !(first && s == 0);
                const uint64_t da = d64(hi_a, lo_a + (uint32_t)s * 16u);
#pragma unroll
                for (int ky = 0; ky < KH; ++ky)
                    umma::mma_bf16(tmem + (uint32_t)(ky * NPAD), da, d64(hi_b, lo_b[ky] + (uint32_t)s * 16u), idesc, acc);
                if constexpr (!BIASW) umma::mma_bf16(tmem + (uint32_t)(KH * NPAD), da, d64(hi_a, lo_ones + (uint32_t)s * 16u), idesc, acc);
            }
            first = false;
            umma::commit(&z_empty[zs]);
            umma::commit(&x_empty[r % xring]);                         // the first B-side row of this A-side row: not needed by later rows
        }
        umma::commit(done);
    } else if (BIASW && warp >= 2) {
        // ================= bias gradient of the 1x1 layers: pixel sums of the A-side rows, from the ring =================
        float bsum[32];
#pragma unroll
        for (int k = 0; k < 32; ++k) bsum[k] = 0.f;
        for (int r = warp - 2; r < n_rows; r += 2) {
            const int zs = r % zslots;
            umma::mbar_wait(&z_full[zs], (uint32_t)((r / zslots) & 1));
            const uint8_t* row = sZ + (size_t)zs * z_slot;
#pragma unroll
            for (int cg = 0; cg < 4; ++cg) {
                if (cg < p.CGo) {
#pragma unroll
                    for (int q = 0; q < kStripTileT / 32; ++q) {
                        const uint4 v = *reinterpret_cast<const uint4*>(row + ((size_t)cg * kStripTileT + q * 32 + lane) * 16u);
                        const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&v);
#pragma unroll
                        for (int e = 0; e < 4; ++e) {
                            const float2 f = __bfloat1622float2(h[e]);
                            bsum[cg * 8 + 2 * e] += f.x;
                            bsum[cg * 8 + 2 * e + 1] += f.y;
                        }
                    }
                }
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(&z_empty[zs]);
        }
        float* sB = reinterpret_cast<float*>(smem + 640);               // [2 warps][32]
#pragma unroll
        for (int k = 0; k < 32; ++k) {
            float v = bsum[k];
#pragma unroll
            for (int sft = 16; sft > 0; sft >>= 1) v += __shfl_xor_sync(0xffffffffu, v, sft);
            if (lane == 0) sB[(warp - 2) * 32 + k] = v;
        }
    }
    if constexpr (BIASW) __syncthreads();
    __syncwarp();
    // ================= epilogue: accumulators -> partial buffer (TMEM lane = A-side channel; NPAD columns per tap) =================
    if (warp < MW) {
        constexpr int MROWS = MW * 32;
        umma::mbar_wait_warp(done, 0);
        umma::fence_after_sync();
        const size_t cta = ((size_t)blockIdx.z * gridDim.y + blockIdx.y) * gridDim.x + blockIdx.x;
        float* dst = p.partial + (cta * kWgMaxTaps * MROWS + warp * 32 + lane) * NPAD;
        const uint32_t lane_addr = tmem + ((uint32_t)(warp * 32) << 16);
        if constexpr (BIASW) {
            // the reduction reads the bias of channel o at [KH][o][0]
            const float* sB = reinterpret_cast<const float*>(smem + 640);
            const int o = warp * 32 + lane;
            if (o < 32) dst[(size_t)KH * MROWS * NPAD] = sB[o] + sB[32 + o];       // dst already points at this thread's channel row
        }
#pragma unroll 1
        for (int tap = 0; tap < KH + (BIASW ? 0 : 1); ++tap) {
#pragma unroll
            for (int c0 = 0; c0 < NPAD; c0 += 16) {
                float v[16];
                umma::tmem_ld16(lane_addr + (uint32_t)(tap * NPAD + c0), v);
                umma::tmem_ld_wait();
                float4* o = reinterpret_cast<float4*>(dst + (size_t)tap * MROWS * NPAD + c0);
                o[0] = make_float4(v[0], v[1], v[2], v[3]);
                o[1] = make_float4(v[4], v[5], v[6], v[7]);
                o[2] = make_float4(v[8], v[9], v[10], v[11]);
                o[3] = make_float4(v[12], v[13], v[14], v[15]);
            }
        }
    }
    umma::fence_before_sync();
    __syncthreads();
    if (warp == 0) umma::tmem_dealloc(tmem, ncols);
}

// ------------------------------------------------------------------------------------------------------------------------------------
// 3x3 'same' layers, row-stationary form.  One MMA per tap and K step (9 + 1 for the bias) would leave the kernel bound by its single
// issuing thread - ~45 cycles per tcgen05.mma whatever its size.  Here a B-side (X) row rho meets ALL THREE
// vertical taps at once: the A operand spans the dZ rows rho - d, rho, rho + d, which lie next to each other in shared memory (a
// strip's dZ rows are all resident, stored residue class by residue class mod d), i.e. the TMEM lanes are (j, co) with j = 0, 1, 2
// <-> ky = 2, 1, 0; the horizontal taps are the N groups of the same MMA (one B-side channel group: column kx * 8 + ci) or three
// MMAs (more groups: columns kx * NK + ci).  1 or 3 MMAs per K step instead of 4 or 10; the bias gradient is summed from the
// resident dZ rows by the two otherwise idle warps.  Partials: per CTA (3 CGO 8 lanes) x NCOL columns + CGO 8 bias sums.
// ------------------------------------------------------------------------------------------------------------------------------------
constexpr int kWg3MaxRows = 112;       // dZ rows a strip may hold (its own + 2 d halo rows): one mbarrier each

struct Wgrad3Params {
    float* partial;
    int B, T, H;
    int d;
    int rows_per_strip;
    int xring;
    int per_cta;                       // floats of one CTA's partial block
};

template <int CGO, int CGI>
__global__ void __launch_bounds__(kWgThreads, 1) wgrad3_kernel(const __grid_constant__ CUtensorMap tmap_x, const __grid_constant__ CUtensorMap tmap_z,
                                                               const Wgrad3Params p) {
    constexpr int KH = 3;
    constexpr int NK = CGI == 1 ? 32 : (CGI == 2 ? 16 : 32);          // N of one MMA
    constexpr int NMMA = CGI == 1 ? 1 : 3;                             // MMAs per K step
    constexpr int NCOL = NK * NMMA;                                    // accumulator columns
    constexpr uint32_t ncols = NCOL <= 32 ? 32 : (NCOL <= 64 ? 64 : 128);
    constexpr int MREAL = KH * CGO * 8;                                // lanes (j, co)
    constexpr uint32_t z_slot = (uint32_t)CGO * kStripTileT * 16u;
    extern __shared__ __align__(1024) uint8_t smem[];
    const int d = p.d;                                                 // row distance of the vertical taps
    const int hz = d;                                                  // dZ halo rows on either side / column halo of the X rows
    const int TW = kStripTileT + 2 * hz;
    const uint32_t x_plane = (uint32_t)TW * 16u;
    const uint32_t x_slot = ((uint32_t)CGI * x_plane + 127u) & ~127u;
    const int xring = p.xring;
    uint64_t* z_full = reinterpret_cast<uint64_t*>(smem);             // [kWg3MaxRows]
    uint64_t* x_full = z_full + kWg3MaxRows;                           // [xring <= 8]
    uint64_t* x_empty = x_full + 8;
    uint64_t* done = x_empty + 8;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(done + 1);
    float* sBias = reinterpret_cast<float*>(smem + 1280);              // [2 warps][CGO * 8]
    uint8_t* sX = smem + 2048;
    uint8_t* sZ = sX + (size_t)xring * x_slot;

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int t0 = blockIdx.x * kStripTileT;
    const int h0 = blockIdx.y * p.rows_per_strip, h1 = min(p.H, h0 + p.rows_per_strip);
    const int b = blockIdx.z;
    const int n_rows = h1 - h0;                                        // X rows of the strip
    const int nz = n_rows + 2 * hz;                                    // dZ rows h0 - d .. h1 + d - 1 (out-of-image rows arrive as zeros)
    const int sd = (nz + d - 1) / d;                                   // positions per residue class
    auto zpos = [&](int i) { return (i % d) * sd + i / d; };           // i = dZ row - (h0 - d)

    if (warp == 0) umma::tmem_alloc(tmem_slot, ncols);
    if (tid == 32) {
        for (int i = 0; i < nz; ++i) umma::mbar_init(&z_full[i], 1);
        for (int i = 0; i < xring; ++i) { umma::mbar_init(&x_full[i], 1); umma::mbar_init(&x_empty[i], 1); }
        umma::mbar_init(done, 1);
        umma::mbar_fence_init();
    }
    umma::fence_before_sync();
    __syncthreads();
    umma::fence_after_sync();
    const uint32_t tmem = *tmem_slot;

    if (warp == 0 && lane == 0) {
        // ================= producer: dZ rows in the order the X rows need them, X rows through a small ring =================
        auto load_z = [&](int i) {
            mbar_expect_tx(&z_full[i], z_slot);
            tma_load_5d(sZ + (size_t)zpos(i) * z_slot, &tmap_z, &z_full[i], 0, t0, h0 - hz + i, 0, b);
        };
        for (int i = 0; i < min(nz, 2 * hz + 1); ++i) load_z(i);
        for (int r = 0; r < n_rows; ++r) {
            const int slot = r % xring;
            if (r >= xring) umma::mbar_wait(&x_empty[slot], (uint32_t)((r / xring - 1) & 1));
            mbar_expect_tx(&x_full[slot], (uint32_t)CGI * x_plane);
            tma_load_5d(sX + (size_t)slot * x_slot, &tmap_x, &x_full[slot], 0, t0 - hz, h0 + r, 0, b);
            if (r + 2 * hz + 1 < nz) load_z(r + 2 * hz + 1);
        }
    } else if (warp == 1 && lane == 0) {
        // ================= MMA issuer =================
        constexpr uint32_t idesc = umma::make_idesc_bf16(128, NK) | (1u << 15) | (1u << 16);       // both operands MN-major
        constexpr uint32_t lbo_field = (128u >> 4) << 16;
        const uint32_t hi_a = ((uint32_t)(kStripTileT * 16) >> 4) | (1u << 14);
        const uint32_t hi_b = ((CGI == 1 ? (uint32_t)d * 16u : x_plane) >> 4) | (1u << 14);
        const uint32_t z0 = umma::smem_u32(sZ), x0 = umma::smem_u32(sX);
        auto d64 = [](uint32_t hi, uint32_t lo) { return ((uint64_t)hi << 32) | lo; };
        for (int r = 0; r < n_rows; ++r) {
            // dZ rows r, r + d, r + 2 d (relative to h0 - d): the first two were awaited with earlier X rows once r >= d
            if (r < d) {
                umma::mbar_wait(&z_full[r], 0);
                umma::mbar_wait(&z_full[r + d], 0);
            }
            umma::mbar_wait(&z_full[r + 2 * hz], 0);
            umma::mbar_wait(&x_full[r % xring], (uint32_t)((r / xring) & 1));
            umma::fence_after_sync();
            const uint32_t lo_a = (((z0 + (uint32_t)zpos(r) * z_slot) >> 4) & 0x3FFFu) | lbo_field;
            const uint32_t lo_b = (((x0 + (uint32_t)(r % xring) * x_slot) >> 4) & 0x3FFFu) | lbo_field;
#pragma unroll
            for (int s = 0; s < kStripTileT / 16; ++s) {
                const bool acc = !(r == 0 && s == 0);
                const uint64_t da = d64(hi_a, lo_a + (uint32_t)s * 16u);
#pragma unroll
                for (int kx = 0; kx < NMMA; ++kx)
                    umma::mma_bf16(tmem + (uint32_t)(kx * NK), da, d64(hi_b, lo_b + (uint32_t)(kx * d) + (uint32_t)s * 16u), idesc, acc);
            }
            umma::commit(&x_empty[r % xring]);
        }
        umma::commit(done);
    } else if (warp >= 2) {
        // ================= bias gradient: pixel sums of the strip's OWN dZ rows, from shared memory =================
        float acc[CGO * 8];
#pragma unroll
        for (int k = 0; k < CGO * 8; ++k) acc[k] = 0.f;
        for (int r = warp - 2; r < n_rows; r += 2) {
            const int i = r + hz;                                       // dZ row h0 + r
            umma::mbar_wait(&z_full[i], 0);
            const uint8_t* row = sZ + (size_t)zpos(i) * z_slot;
#pragma unroll
            for (int q = 0; q < kStripTileT / 32; ++q) {
#pragma unroll
                for (int cg = 0; cg < CGO; ++cg) {
                    const uint4 v = *reinterpret_cast<const uint4*>(row + ((size_t)cg * kStripTileT + q * 32 + lane) * 16u);
                    const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&v);
#pragma unroll
                    for (int e = 0; e < 4; ++e) {
                        const float2 f = __bfloat1622float2(h[e]);
                        acc[cg * 8 + 2 * e] += f.x;
                        acc[cg * 8 + 2 * e + 1] += f.y;
                    }
                }
            }
        }
#pragma unroll
        for (int k = 0; k < CGO * 8; ++k) {
            float v = acc[k];
#pragma unroll
            for (int s = 16; s > 0; s >>= 1) v += __shfl_xor_sync(0xffffffffu, v, s);
            if (lane == 0) sBias[(warp - 2) * CGO * 8 + k] = v;
        }
    }
    __syncthreads();
    // ================= epilogue: accumulators and bias sums -> the CTA's partial block =================
    const size_t cta = ((size_t)blockIdx.z * gridDim.y + blockIdx.y) * gridDim.x + blockIdx.x;
    float* dst = p.partial + cta * (size_t)p.per_cta;
    if (tid < CGO * 8) dst[(size_t)MREAL * NCOL + tid] = sBias[tid] + sBias[CGO * 8 + tid];
    if (warp * 32 < MREAL) {
        umma::mbar_wait_warp(done, 0);
        umma::fence_after_sync();
        const uint32_t lane_addr = tmem + ((uint32_t)(warp * 32) << 16);
        const int m = warp * 32 + lane;
#pragma unroll
        for (int c0 = 0; c0 < NCOL; c0 += 16) {
            float v[16];
            umma::tmem_ld16(lane_addr + (uint32_t)c0, v);
            umma::tmem_ld_wait();
            if (m < MREAL) {
                float4* o = reinterpret_cast<float4*>(dst + (size_t)m * NCOL + c0);
                o[0] = make_float4(v[0], v[1], v[2], v[3]);
                o[1] = make_float4(v[4], v[5], v[6], v[7]);
                o[2] = make_float4(v[8], v[9], v[10], v[11]);
                o[3] = make_float4(v[12], v[13], v[14], v[15]);
            }
        }
    }
    umma::fence_before_sync();
    __syncthreads();
    if (warp == 0) umma::tmem_dealloc(tmem, ncols);
}

// dw (co, ci, kh, kh) and db (co) += fixed-order sums over the CTAs' partial blocks of wgrad3_kernel.  A block owns 32 consecutive output
// elements x 8 segments of the CTA range: the lanes of a warp read 32 neighbouring floats of one partial block (neighbouring input
// channels are neighbouring columns), each thread sums its segment front to back, the segments are added in order - bit-reproducible,
// and the reads are coalesced (one warp per element striding over the blocks was 5 % of the loss step).
constexpr int kWg3RedSeg = 8;

__global__ void __launch_bounds__(32 * kWg3RedSeg) wgrad3_reduce_kernel(const float* __restrict__ partial, int n_ctas, int per_cta, int cgo, int ncol,
                                                                       int nk, int kx_in_n, int kh, int m_real, int n_real,
                                                                       float* __restrict__ dw, float* __restrict__ db) {
    __shared__ float part[kWg3RedSeg][32];
    const int lane = threadIdx.x & 31, seg = threadIdx.x >> 5;
    const int i = blockIdx.x * 32 + lane;                                  // over (tap in [0, taps], co, ci); tap == taps: bias
    const int taps = kh * kh;
    const int total = (taps + 1) * m_real * n_real;
    const int tap = i / (m_real * n_real), rem = i - tap * m_real * n_real;
    const int o = rem / n_real, c = rem - o * n_real;
    const bool live = i < total && !(tap == taps && (c != 0 || db == nullptr));
    float acc = 0.f;
    if (live) {
        size_t off;
        if (tap == taps) {
            off = (size_t)kh * cgo * 8 * ncol + o;
        } else {
            const int ky = tap / kh, kx = tap - kh * ky;
            const int m = (kh - 1 - ky) * cgo * 8 + o;
            const int col = kx_in_n ? kx * 8 + c : kx * nk + c;
            off = (size_t)m * ncol + col;
        }
        const int per_seg = (n_ctas + kWg3RedSeg - 1) / kWg3RedSeg;
        const int k0 = seg * per_seg, k1 = min(n_ctas, k0 + per_seg);
        const float* src = partial + off;
        int k = k0;
        for (; k + 4 <= k1; k += 4) {
            const float a0 = src[(size_t)k * per_cta], a1 = src[(size_t)(k + 1) * per_cta], a2 = src[(size_t)(k + 2) * per_cta],
                        a3 = src[(size_t)(k + 3) * per_cta];
            acc += a0; acc += a1; acc += a2; acc += a3;
        }
        for (; k < k1; ++k) acc += src[(size_t)k * per_cta];
    }
    part[seg][lane] = acc;
    __syncthreads();
    if (seg == 0 && live) {
        float v = part[0][lane];
#pragma unroll
        for (int q = 1; q < kWg3RedSeg; ++q) v += part[q][lane];
        if (tap == taps) db[o] += v;
        else dw[((size_t)o * n_real + c) * taps + tap] += v;
    }
}

// ------------------------------------------------------------------------------------------------------------------------------------
// (4,1) stride-(2,1) layers (EncoderBlock.sconv; DecoderBlock.tconv with the sides swapped), row-stationary form.
//     dW[cc][cf][kh] = sum over (b, q, t) of  coarse[b, cc, q, t] * fine[b, cf, 2 q + kh, t]
// A fine row rho meets the coarse rows q0 - 1 and q0 = rho / 2 (taps kh = rho % 2 + 2 and rho % 2): the strip's coarse rows are
// resident and consecutive, so the two are stacked in the MMA's M (TMEM lanes (j, cc), j = 0 <-> q0 - 1), and the row parity selects
// the accumulator columns: ONE MMA per fine row and K step - two per coarse row instead of 4 + 1 with one MMA per tap.  The bias
// gradient of the strided layer (pixel sums of the coarse tensor) comes from the resident rows through the idle warps.
// ------------------------------------------------------------------------------------------------------------------------------------
struct WgradUdParams {
    float* partial;
    int B, T, Hc;                      // coarse rows; fine rows 0 .. 2 Hc + 1 are used
    int rows_per_strip;                // values of q0 per strip (q0 in [0, Hc]: the last one pairs the zero row Hc with row Hc - 1)
    int xring;
    int per_cta;
};

template <int CGC, int CGF>
__global__ void __launch_bounds__(kWgThreads, 1) wgrad_ud_kernel(const __grid_constant__ CUtensorMap tmap_f, const __grid_constant__ CUtensorMap tmap_c,
                                                                 const WgradUdParams p) {
    constexpr int NK = CGF <= 2 ? 16 : 32;                             // N of one MMA (fine-side channels, padded)
    constexpr int NCOL = 2 * NK;                                       // accumulator columns: (row parity, cf)
    constexpr uint32_t ncols = NCOL <= 32 ? 32 : 64;
    constexpr int MREAL = 2 * CGC * 8;                                 // lanes (j, cc)
    static_assert(MREAL <= 128, "two coarse rows of up to 64 channels");
    constexpr uint32_t c_slot = (uint32_t)CGC * kStripTileT * 16u;
    constexpr uint32_t f_plane = (uint32_t)kStripTileT * 16u;
    constexpr uint32_t f_slot = (uint32_t)CGF * f_plane;
    extern __shared__ __align__(1024) uint8_t smem[];
    const int xring = p.xring;
    uint64_t* c_full = reinterpret_cast<uint64_t*>(smem);             // [kWg3MaxRows]
    uint64_t* f_full = c_full + kWg3MaxRows;                           // [xring <= 8]
    uint64_t* f_empty = f_full + 8;
    uint64_t* done = f_empty + 8;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(done + 1);
    float* sBias = reinterpret_cast<float*>(smem + 1280);              // [2 warps][CGC * 8]
    uint8_t* sF = smem + 2048;
    uint8_t* sC = sF + (size_t)xring * f_slot;

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int t0 = blockIdx.x * kStripTileT;
    const int q_lo = blockIdx.y * p.rows_per_strip, q_hi = min(p.Hc + 1, q_lo + p.rows_per_strip);     // values of q0
    const int b = blockIdx.z;
    const int n_q = q_hi - q_lo;
    const int n_frows = 2 * n_q;                                       // fine rows 2 q_lo .. 2 q_hi - 1
    const int nc = n_q + 1;                                            // coarse rows q_lo - 1 .. q_hi - 1 (rows -1 and Hc arrive as zeros)

    if (warp == 0) umma::tmem_alloc(tmem_slot, ncols);
    if (tid == 32) {
        for (int i = 0; i < nc; ++i) umma::mbar_init(&c_full[i], 1);
        for (int i = 0; i < xring; ++i) { umma::mbar_init(&f_full[i], 1); umma::mbar_init(&f_empty[i], 1); }
        umma::mbar_init(done, 1);
        umma::mbar_fence_init();
    }
    umma::fence_before_sync();
    __syncthreads();
    umma::fence_after_sync();
    const uint32_t tmem = *tmem_slot;

    if (warp == 0 && lane == 0) {
        // ================= producer =================
        auto load_c = [&](int i) {
            mbar_expect_tx(&c_full[i], c_slot);
            tma_load_5d(sC + (size_t)i * c_slot, &tmap_c, &c_full[i], 0, t0, q_lo - 1 + i, 0, b);
        };
        load_c(0);
        if (nc > 1) load_c(1);
        for (int r = 0; r < n_frows; ++r) {
            const int slot = r % xring;
            if (r >= xring) umma::mbar_wait(&f_empty[slot], (uint32_t)((r / xring - 1) & 1));
            mbar_expect_tx(&f_full[slot], f_slot);
            tma_load_5d(sF + (size_t)slot * f_slot, &tmap_f, &f_full[slot], 0, t0, 2 * q_lo + r, 0, b);
            if ((r & 1) && (r >> 1) + 2 < nc) load_c((r >> 1) + 2);
        }
    } else if (warp == 1 && lane == 0) {
        // ================= MMA issuer =================
        constexpr uint32_t idesc = umma::make_idesc_bf16(128, NK) | (1u << 15) | (1u << 16);       // both operands MN-major
        constexpr uint32_t lbo_field = (128u >> 4) << 16;
        const uint32_t hi_a = ((uint32_t)(kStripTileT * 16) >> 4) | (1u << 14);
        const uint32_t hi_b = (f_plane >> 4) | (1u << 14);
        const uint32_t c0 = umma::smem_u32(sC), f0 = umma::smem_u32(sF);
        auto d64 = [](uint32_t hi, uint32_t lo) { return ((uint64_t)hi << 32) | lo; };
        for (int r = 0; r < n_frows; ++r) {
            const int qi = r >> 1;                                     // coarse rows qi (= q0 - 1) and qi + 1 (= q0) of the strip's buffer
            if (r == 0) umma::mbar_wait(&c_full[0], 0);
            if ((r & 1) == 0) umma::mbar_wait(&c_full[qi + 1], 0);
            umma::mbar_wait(&f_full[r % xring], (uint32_t)((r / xring) & 1));
            umma::fence_after_sync();
            const uint32_t lo_a = (((c0 + (uint32_t)qi * c_slot) >> 4) & 0x3FFFu) | lbo_field;
            const uint32_t lo_b = (((f0 + (uint32_t)(r % xring) * f_slot) >> 4) & 0x3FFFu) | lbo_field;
            const uint32_t acc_col = tmem + (uint32_t)((r & 1) * NK);
#pragma unroll
            for (int s = 0; s < kStripTileT / 16; ++s)
                umma::mma_bf16(acc_col, d64(hi_a, lo_a + (uint32_t)s * 16u), d64(hi_b, lo_b + (uint32_t)s * 16u), idesc, !(r < 2 && s == 0));
            umma::commit(&f_empty[r % xring]);
        }
        umma::commit(done);
    } else if (warp >= 2) {
        // ================= pixel sums of the strip's own coarse rows q_lo .. min(q_hi, Hc) - 1 (the strided layer's bias gradient) =================
        float acc[CGC * 8];
#pragma unroll
        for (int k = 0; k < CGC * 8; ++k) acc[k] = 0.f;
        const int own = min(q_hi, p.Hc) - q_lo;
        for (int r = warp - 2; r < own; r += 2) {
            const int i = r + 1;                                        // buffer row of coarse row q_lo + r
            umma::mbar_wait(&c_full[i], 0);
            const uint8_t* row = sC + (size_t)i * c_slot;
#pragma unroll
            for (int q = 0; q < kStripTileT / 32; ++q) {
#pragma unroll
                for (int cg = 0; cg < CGC; ++cg) {
                    const uint4 v = *reinterpret_cast<const uint4*>(row + ((size_t)cg * kStripTileT + q * 32 + lane) * 16u);
                    const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&v);
#pragma unroll
                    for (int e = 0; e < 4; ++e) {
                        const float2 f = __bfloat1622float2(h[e]);
                        acc[cg * 8 + 2 * e] += f.x;
                        acc[cg * 8 + 2 * e + 1] += f.y;
                    }
                }
            }
        }
#pragma unroll
        for (int k = 0; k < CGC * 8; ++k) {
            float v = acc[k];
#pragma unroll
            for (int sft = 16; sft > 0; sft >>= 1) v += __shfl_xor_sync(0xffffffffu, v, sft);
            if (lane == 0) sBias[(warp - 2) * CGC * 8 + k] = v;
        }
    }
    __syncthreads();
    const size_t cta = ((size_t)blockIdx.z * gridDim.y + blockIdx.y) * gridDim.x + blockIdx.x;
    float* dst = p.partial + cta * (size_t)p.per_cta;
    if (tid < CGC * 8) dst[(size_t)MREAL * NCOL + tid] = sBias[tid] + sBias[CGC * 8 + tid];
    if (warp * 32 < MREAL) {
        umma::mbar_wait_warp(done, 0);
        umma::fence_after_sync();
        const uint32_t lane_addr = tmem + ((uint32_t)(warp * 32) << 16);
        const int m = warp * 32 + lane;
#pragma unroll
        for (int c0 = 0; c0 < NCOL; c0 += 16) {
            float v[16];
            umma::tmem_ld16(lane_addr + (uint32_t)c0, v);
            umma::tmem_ld_wait();
            if (m < MREAL) {
                float4* o = reinterpret_cast<float4*>(dst + (size_t)m * NCOL + c0);
                o[0] = make_float4(v[0], v[1], v[2], v[3]);
                o[1] = make_float4(v[4], v[5], v[6], v[7]);
                o[2] = make_float4(v[8], v[9], v[10], v[11]);
                o[3] = make_float4(v[12], v[13], v[14], v[15]);
            }
        }
    }
    umma::fence_before_sync();
    __syncthreads();
    if (warp == 0) umma::tmem_dealloc(tmem, ncols);
}

// dw (cc, cf, 4, 1) and db (cc) += fixed-order sums over the partial blocks of wgrad_ud_kernel (same scheme as wgrad3_reduce_kernel)
__global__ void __launch_bounds__(32 * kWg3RedSeg) wgrad_ud_reduce_kernel(const float* __restrict__ partial, int n_ctas, int per_cta, int cgc, int nk,
                                                                         int m_real, int n_real, float* __restrict__ dw, float* __restrict__ db) {
    __shared__ float part[kWg3RedSeg][32];
    const int lane = threadIdx.x & 31, seg = threadIdx.x >> 5;
    const int i = blockIdx.x * 32 + lane;                                  // over (kh in [0, 4], cc, cf); kh == 4: bias
    const int total = 5 * m_real * n_real;
    const int kh = i / (m_real * n_real), rem = i - kh * m_real * n_real;
    const int o = rem / n_real, c = rem - o * n_real;
    const bool live = i < total && !(kh == 4 && (c != 0 || db == nullptr));
    float acc = 0.f;
    if (live) {
        const int ncol = 2 * nk;
        size_t off;
        if (kh == 4) off = (size_t)2 * cgc * 8 * ncol + o;
        else off = (size_t)((kh < 2 ? 1 : 0) * cgc * 8 + o) * ncol + (size_t)(kh & 1) * nk + c;      // kh = parity + 2 (1 - j)
        const int per_seg = (n_ctas + kWg3RedSeg - 1) / kWg3RedSeg;
        const int k0 = seg * per_seg, k1 = min(n_ctas, k0 + per_seg);
        const float* src = partial + off;
        for (int k = k0; k < k1; ++k) acc += src[(size_t)k * per_cta];
    }
    part[seg][lane] = acc;
    __syncthreads();
    if (seg == 0 && live) {
        float v = part[0][lane];
#pragma unroll
        for (int q = 1; q < kWg3RedSeg; ++q) v += part[q][lane];
        if (kh == 4) db[o] += v;
        else dw[((size_t)o * n_real + c) * 4 + kh] += v;
    }
}

// dW (m, n, taps) and db (m) += fixed-order sums of the per-CTA partials (m = A-side channel = co, n = B-side channel = ci)
// One WARP per output element: the lanes stride over the CTAs' partials, then a shuffle tree - a fixed order, so still bit-reproducible.
__global__ void __launch_bounds__(256) wgrad_reduce_kernel(const float* __restrict__ partial, int n_ctas, int npad, int taps, int m_real, int n_real,
                                                           float* __restrict__ dw, float* __restrict__ db) {
    const int i = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);     // over (tap' in [0, taps], m, n)
    const int lane = threadIdx.x & 31;
    const int total = (taps + 1) * m_real * n_real;
    if (i >= total) return;
    const int tap = i / (m_real * n_real), rem = i - tap * m_real * n_real;
    const int o = rem / n_real, c = rem - o * n_real;
    if (tap == taps && (c != 0 || db == nullptr)) return;
    const float* src = partial + ((size_t)tap * kWgMaxM + o) * npad + (tap == taps ? 0 : c);
    const size_t stride = (size_t)kWgMaxTaps * kWgMaxM * npad;
    float acc = 0.f;
    for (int k = lane; k < n_ctas; k += 32) acc += src[(size_t)k * stride];
#pragma unroll
    for (int s = 16; s > 0; s >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, s);
    if (lane == 0) {
        if (tap == taps) db[o] += acc;
        else dw[((size_t)o * n_real + c) * taps + tap] += acc;
    }
}

// the (31,1) layers: CTA (x, group, b) holds taps group * G .. group * G + G - 1 of all 128 A-side channels; dw (m, n, taps) += fixed-order sums
__global__ void wgrad_reduce_groups_kernel(const float* __restrict__ partial, int nx, int n_groups, int nb, int G, int npad, int taps, int m_real,
                                           int n_real, float* __restrict__ dw, float* __restrict__ db) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;              // over (kh in [0, taps], m, n); kh == taps: the bias "tap"
    const int total = (taps + 1) * m_real * n_real;
    if (i >= total) return;
    const int kh = i / (m_real * n_real), rem = i - kh * m_real * n_real;
    const int o = rem / n_real, c = rem - o * n_real;
    if (kh == taps && (c != 0 || db == nullptr)) return;
    const int group = kh == taps ? 0 : kh / G, tl = kh == taps ? G : kh - group * G;
    const size_t cta_stride = (size_t)kWgMaxTaps * 128 * npad;
    const float* src = partial + ((size_t)tl * 128 + o) * npad + (kh == taps ? 0 : c);
    float acc = 0.f;
    for (int b = 0; b < nb; ++b)
        for (int x = 0; x < nx; ++x) acc += src[(((size_t)b * n_groups + group) * nx + x) * cta_stride];
    if (kh == taps) db[o] += acc;
    else dw[((size_t)o * n_real + c) * taps + kh] += acc;
}

// out[c][h] += sum over (b, t) of a C8 planar tensor (B, CG, H, T, 8): two stages, fixed order (the indicator row of Decoder.convin's
// weight gradient and that layer's bias gradient)
__global__ void __launch_bounds__(256) row_channel_sum_c8_kernel(const uint4* __restrict__ x, int CG, int H, int T, float* __restrict__ partial) {
    // grid (H, CG, B)
    const uint4* row = x + (((size_t)blockIdx.z * CG + blockIdx.y) * H + blockIdx.x) * T;
    float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    for (int i = threadIdx.x; i < T; i += 256) {
        const uint4 v = __ldcs(row + i);
        const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&v);
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const float2 f = __bfloat1622float2(h[k]);
            acc[2 * k] += f.x;
            acc[2 * k + 1] += f.y;
        }
    }
    __shared__ float red[8][8];
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        float v = acc[k];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5][k] = v;
    }
    __syncthreads();
    if (threadIdx.x < 8) {
        float v = 0.f;
        for (int w = 0; w < 8; ++w) v += red[w][threadIdx.x];
        partial[(((size_t)blockIdx.z * CG + blockIdx.y) * H + blockIdx.x) * 8 + threadIdx.x] = v;
    }
}
__global__ void row_channel_sum_finish_kernel(const float* __restrict__ partial, int B, int CG, int H, int c_real, float* __restrict__ out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;              // over (c, h)
    if (i >= c_real * H) return;
    const int c = i / H, h = i - c * H;
    float acc = 0.f;
    for (int b = 0; b < B; ++b) acc += partial[(((size_t)b * CG + (c >> 3)) * H + h) * 8 + (c & 7)];
    out[i] += acc;
}

// db[c] += sum over pixels of a C8 planar tensor (B, CG, H, T, 8): per-CTA partials, fixed-order second stage (the transposed layers'
// bias gradient: their weight-gradient GEMM has the layer INPUT on its A side)
__global__ void __launch_bounds__(256) channel_sum_c8_partial_kernel(const uint4* __restrict__ x, int CG, long long hw, float* __restrict__ partial) {
    // grid (chunks, CG, B); thread-strided over the pixels of one (b, cg) plane
    const uint4* plane = x + ((size_t)blockIdx.z * CG + blockIdx.y) * hw;
    float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < hw; i += (long long)gridDim.x * blockDim.x) {
        const uint4 v = __ldcs(plane + i);
        const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&v);
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const float2 f = __bfloat1622float2(h[k]);
            acc[2 * k] += f.x;
            acc[2 * k + 1] += f.y;
        }
    }
    __shared__ float red[8][8];
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        float v = acc[k];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5][k] = v;
    }
    __syncthreads();
    if (threadIdx.x < 8) {
        float v = 0.f;
        for (int w = 0; w < 8; ++w) v += red[w][threadIdx.x];
        partial[(((size_t)blockIdx.z * CG + blockIdx.y) * gridDim.x + blockIdx.x) * 8 + threadIdx.x] = v;
    }
}
__global__ void channel_sum_c8_finish_kernel(const float* __restrict__ partial, int B, int CG, int chunks, int c_real, float* __restrict__ db) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= c_real) return;
    const int cg = c >> 3, k = c & 7;
    float acc = 0.f;
    for (int b = 0; b < B; ++b)
        for (int i = 0; i < chunks; ++i) acc += partial[(((size_t)b * CG + cg) * chunks + i) * 8 + k];
    db[c] += acc;
}

// ---- element-wise pieces of the backward pass on bf16 tensors of ANY common layout -------------------------------------------------
__device__ __forceinline__ float elu_grad_from_output(float a) { return a > 0.f ? 1.f : a + 1.f; }

// dz = gy * ELU'(z) through the activated output a
__global__ void elu_bwd_bf16_kernel(const uint4* __restrict__ gy, const uint4* __restrict__ a, uint4* __restrict__ dz, long long n8) {
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n8; i += stride) {
        const uint4 g = __ldcs(gy + i), av = __ldcs(a + i);
        const __nv_bfloat162* gh = reinterpret_cast<const __nv_bfloat162*>(&g);
        const __nv_bfloat162* ah = reinterpret_cast<const __nv_bfloat162*>(&av);
        uint4 r;
        uint32_t* rw = reinterpret_cast<uint32_t*>(&r);
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const float2 fg = __bfloat1622float2(gh[k]), fa = __bfloat1622float2(ah[k]);
            rw[k] = pack2(fg.x * elu_grad_from_output(fa.x), fg.y * elu_grad_from_output(fa.y));
        }
        dz[i] = r;
    }
}

// residual block: dz2 = gy * ELU'(z2) with the activated 1x1 output recovered as y - x
__global__ void res_out_bwd_bf16_kernel(const uint4* __restrict__ gy, const uint4* __restrict__ y, const uint4* __restrict__ x, uint4* __restrict__ dz,
                                        long long n8) {
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n8; i += stride) {
        const uint4 g = __ldcs(gy + i), yv = __ldcs(y + i), xv = __ldcs(x + i);
        const __nv_bfloat162* gh = reinterpret_cast<const __nv_bfloat162*>(&g);
        const __nv_bfloat162* yh = reinterpret_cast<const __nv_bfloat162*>(&yv);
        const __nv_bfloat162* xh = reinterpret_cast<const __nv_bfloat162*>(&xv);
        uint4 r;
        uint32_t* rw = reinterpret_cast<uint32_t*>(&r);
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const float2 fg = __bfloat1622float2(gh[k]), fy = __bfloat1622float2(yh[k]), fx = __bfloat1622float2(xh[k]);
            rw[k] = pack2(fg.x * elu_grad_from_output(fy.x - fx.x), fg.y * elu_grad_from_output(fy.y - fx.y));
        }
        dz[i] = r;
    }
}

// packed 4-channel (B, H, T, 4) <-> C8 planar with one channel group (B, 1, H, T, 8): the first / last stage's tensors for the kernels
// that only know C8 planar
__global__ void p4_to_c8_kernel(const uint2* __restrict__ p4, uint4* __restrict__ c8, long long n_px) {
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n_px; i += stride) {
        const uint2 v = __ldcs(p4 + i);
        c8[i] = make_uint4(v.x, v.y, 0u, 0u);
    }
}
__global__ void c8_to_p4_kernel(const uint4* __restrict__ c8, uint2* __restrict__ p4, long long n_px) {
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n_px; i += stride) {
        const uint4 v = __ldcs(c8 + i);
        p4[i] = make_uint2(v.x, v.y);
    }
}

static size_t wgrad_smem(int CGi, int CGo, int xring, int zslots) {
    const size_t z_slot = (size_t)CGo * kStripTileT * 16;
    const size_t x_slot = (size_t)CGi * kStripTileT * 16;
    size_t s = 1024 + 4096 + zslots * z_slot + xring * x_slot + 8 * kStripTileT * 16;   // + the padded N groups read past the last B slot
    // the A operand spans 16 channel groups (32 KB) from the start of an A slot, the ones operand NPAD/8 groups: keep both inside
    s = std::max(s, (size_t)1024 + 4096 + (zslots - 1) * z_slot + 16 * (size_t)kStripTileT * 16 + 1024);
    return s;
}

template <int NPAD, int KH, int MW>
static int launch_wgrad(const void* x, const void* dz, const WgradParams& p, dim3 grid, cudaStream_t stream) {
    const int xring = p.xring;
    TT_REQUIRE(xring <= 16 && xring >= KH + 2, "wgrad: ring of %d rows", xring);
    const size_t smem = wgrad_smem(p.CGi, p.CGo, xring, p.z_slots);
    TT_REQUIRE(smem <= 227 * 1024, "wgrad: %zu bytes of shared memory", smem);
    static size_t configured = 0;
    if (smem > configured) {
        TT_CUDA_CHECK(cudaFuncSetAttribute(wgrad_kernel<NPAD, KH, MW>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        configured = smem;
    }
    CUtensorMap mx, mz;
    int rc = make_row_map(&mx, x, p.B, p.CGi, p.Hx, p.T, kStripTileT);
    if (rc) return rc;
    rc = make_row_map(&mz, dz, p.B, p.CGo, p.Hz, p.T, kStripTileT);
    if (rc) return rc;
    wgrad_kernel<NPAD, KH, MW><<<grid, kWgThreads, smem, stream>>>(mx, mz, p);
    TT_CUDA_CHECK(cudaGetLastError());
    tt_count_launches(1);
    return TT_OK;
}

static long long wgrad_strips(int B, int Hz, int T) {
    // about six CTAs per SM in total (several are co-resident: the accumulators of a CTA take 128-512 TMEM columns): evens out
    // the load over the 148 SMs at the price of more partial buffers for the reduction
    const long long tiles = (long long)B * ((T + kStripTileT - 1) / kStripTileT);
    return std::max<long long>(1, std::min<long long>((6 * 148 + tiles - 1) / tiles, std::max(1, Hz / 8)));
}

// ---- row-stationary 3x3: strip geometry (shared by the launch and the scratch bound) ----
struct Wg3Plan {
    int rows, strips, xring, per_cta;
    size_t smem;
};

static Wg3Plan wg3_plan(int B, int CGi, int CGo, int H, int T, int d) {
    Wg3Plan g;
    const size_t z_slot = (size_t)CGo * kStripTileT * 16, x_slot = ((size_t)CGi * (kStripTileT + 2 * d) * 16 + 127) & ~(size_t)127;
    g.xring = 4;
    // everything a strip touches of dZ stays resident: rows + 2 d slots, and the A operand reads 32 KB from its first slot
    // one resident strip per SM leaves the tensor pipe idle while the strip's first rows are in flight: with small rows (C <= 16) take
    // half of the shared memory, so that two CTAs share an SM and one computes while the other loads
    const size_t cap = (size_t)(CGo <= 2 ? 112 : 226) * 1024;
    const size_t budget = cap - 2048 - g.xring * x_slot - 32 * 1024;
    int max_rows = (int)std::min<size_t>(budget / z_slot, (size_t)kWg3MaxRows) - (3 * d - 1);   // the residue-class layout rounds the row count up to a multiple of d
    max_rows = std::max(max_rows, 1);
    const long long tiles = (long long)B * ((T + kStripTileT - 1) / kStripTileT);
    // at least ~4 CTAs per SM in total (one is resident at a time), never more rows than shared memory holds
    long long strips = std::max<long long>((H + max_rows - 1) / max_rows, std::min<long long>((4 * 148 + tiles - 1) / tiles, std::max(1, H / 4)));
    g.rows = (int)((H + strips - 1) / strips);
    g.strips = (H + g.rows - 1) / g.rows;
    const int nk = CGi == 1 ? 32 : (CGi == 2 ? 16 : 32), ncol = nk * (CGi == 1 ? 1 : 3);
    g.per_cta = 3 * CGo * 8 * ncol + CGo * 8;
    const size_t nzpos = (size_t)d * ((g.rows + 2 * d + d - 1) / d);
    g.smem = 2048 + g.xring * x_slot + std::max(nzpos * z_slot, (nzpos - 3) * z_slot + 32 * 1024) + 1024;
    return g;
}

struct WgUdPlan {
    int rows, strips, xring, per_cta;
    size_t smem;
};

static WgUdPlan wgud_plan(int B, int CGf, int CGc, int Hc, int T) {
    WgUdPlan g;
    const size_t c_slot = (size_t)CGc * kStripTileT * 16, f_slot = (size_t)CGf * kStripTileT * 16;
    g.xring = 4;
    const size_t cap = (size_t)(CGc <= 2 ? 112 : 226) * 1024;          // small rows: two strips per SM (see wg3_plan)
    const size_t budget = cap - 2048 - g.xring * f_slot - 32 * 1024;
    int max_rows = (int)std::min<size_t>(budget / c_slot, (size_t)kWg3MaxRows) - 1;     // values of q0 per strip (+ 1 coarse row)
    max_rows = std::max(max_rows, 1);
    const int nq = Hc + 1;
    const long long tiles = (long long)B * ((T + kStripTileT - 1) / kStripTileT);
    long long strips = std::max<long long>((nq + max_rows - 1) / max_rows, std::min<long long>((4 * 148 + tiles - 1) / tiles, std::max(1, nq / 4)));
    g.rows = (int)((nq + strips - 1) / strips);
    g.strips = (nq + g.rows - 1) / g.rows;
    const int nk = CGf <= 2 ? 16 : 32;
    g.per_cta = 2 * CGc * 8 * 2 * nk + CGc * 8;
    const size_t nrows = (size_t)g.rows + 1;
    g.smem = 2048 + g.xring * f_slot + std::max(nrows * c_slot, (nrows - 2) * c_slot + 32 * 1024) + 1024;
    return g;
}

}  // namespace tt

using namespace tt;

extern "C" int64_t tt_wgrad_scratch_floats(int B, int H, int T) {
    // upper bound over the strip splits the weight-gradient entry points choose (H = rows of the A-side tensor)
    const long long tiles = (long long)B * ((T + kStripTileT - 1) / kStripTileT);
    long long need = tiles * (wgrad_strips(B, H, T) + 1) * kWgMaxTaps * kWgMaxM * 32;
    // the row-stationary 3x3 kernel: its strips are bounded by shared memory, its partial blocks are smaller
    for (int cgi = 1; cgi <= 4; cgi *= 2)
        for (int cgo = 1; cgo <= 4; cgo *= 2)
            for (int d = 1; d <= 3; ++d) {
                const Wg3Plan g = wg3_plan(B, cgi, cgo, H, T, d);
                need = std::max(need, tiles * g.strips * (long long)g.per_cta);
            }
    for (int cgc = 1; cgc <= 8; cgc *= 2) {
        const WgUdPlan g = wgud_plan(B, std::max(1, cgc / 2), cgc, H, T);
        need = std::max(need, tiles * g.strips * (long long)g.per_cta);
    }
    return need;
}

// 1x1 layers: the ring kernel, A side dz (channels Cout), B side x (channels Cin)
static int wgrad1x1(const void* x, const void* dz, float* dw, float* db, int B, int Cin, int Cout, int cin_real, int cout_real, int H, int T,
                    float* scratch, cudaStream_t stream) {
    WgradParams p;
    p.partial = scratch;
    p.B = B; p.T = T; p.Hz = H; p.Hx = H; p.CGi = Cin / 8; p.CGo = Cout / 8;
    p.tap_group = 0;
    // ring depths: the loads are 2-16 KB rows with ~1 us latency each, so the prefetch distance - not bandwidth - sets the pace;
    // take up to 8 A-side rows and up to 8 B-side rows ahead, within ~170 KB of shared memory
    {
        const size_t z_slot = (size_t)(Cout / 8) * kStripTileT * 16, x_slot = (size_t)(Cin / 8) * kStripTileT * 16 + 128;
        p.z_slots = (int)std::max<size_t>(3, std::min<size_t>(kWgZSlots, (48 * 1024) / z_slot));
        int pf = 8;
        while (pf > 2 && (1 + pf) * x_slot > 120 * 1024) --pf;
        p.xring = 1 + pf;
    }
    const long long strips = wgrad_strips(B, H, T);
    p.rows_per_strip = (int)((H + strips - 1) / strips);
    dim3 grid((T + kStripTileT - 1) / kStripTileT, (H + p.rows_per_strip - 1) / p.rows_per_strip, B);
    const int n_ctas = (int)(grid.x * grid.y * grid.z);
    const int npad = Cin >= 32 ? 32 : 16;
    const int rc = npad == 32 ? launch_wgrad<32, 1, 2>(x, dz, p, grid, stream) : launch_wgrad<16, 1, 2>(x, dz, p, grid, stream);
    if (rc) return rc;
    const int total = 2 * cout_real * cin_real;
    wgrad_reduce_kernel<<<(total + 7) / 8, 256, 0, stream>>>(scratch, n_ctas, npad, 1, cout_real, cin_real, dw, db);
    tt_count_launches(1);
    TT_CUDA_CHECK(cudaGetLastError());
    return TT_OK;
}

template <int CGO, int CGI>
static int launch_wgrad3(const void* x, const void* dz, float* dw, float* db, int B, int cin_real, int cout_real, int H, int T, int d,
                         float* scratch, cudaStream_t stream) {
    constexpr int KH = 3;
    const Wg3Plan g = wg3_plan(B, CGI, CGO, H, T, d);
    TT_REQUIRE(g.smem <= 227 * 1024 && g.rows + 2 * d <= kWg3MaxRows, "wgrad3: %zu bytes of shared memory, %d rows", g.smem, g.rows);
    static size_t configured = 0;
    if (g.smem > configured) {
        TT_CUDA_CHECK(cudaFuncSetAttribute(wgrad3_kernel<CGO, CGI>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)g.smem));
        configured = g.smem;
    }
    CUtensorMap mx, mz;
    int rc = make_row_map(&mx, x, B, CGI, H, T, kStripTileT + 2 * d);
    if (rc) return rc;
    rc = make_row_map(&mz, dz, B, CGO, H, T, kStripTileT);
    if (rc) return rc;
    Wgrad3Params p;
    p.partial = scratch; p.B = B; p.T = T; p.H = H; p.d = d; p.rows_per_strip = g.rows; p.xring = g.xring; p.per_cta = g.per_cta;
    dim3 grid((T + kStripTileT - 1) / kStripTileT, g.strips, B);
    wgrad3_kernel<CGO, CGI><<<grid, kWgThreads, g.smem, stream>>>(mx, mz, p);
    TT_CUDA_CHECK(cudaGetLastError());
    const int n_ctas = (int)(grid.x * grid.y * grid.z);
    constexpr int NK = CGI == 1 ? 32 : (CGI == 2 ? 16 : 32), NCOL = NK * (CGI == 1 ? 1 : 3);
    const int total = (KH * KH + 1) * cout_real * cin_real;
    wgrad3_reduce_kernel<<<(total + 31) / 32, 32 * kWg3RedSeg, 0, stream>>>(scratch, n_ctas, g.per_cta, CGO, NCOL, NK, CGI == 1, KH, cout_real, cin_real, dw, db);
    tt_count_launches(2);
    TT_CUDA_CHECK(cudaGetLastError());
    return TT_OK;
}

static int wgrad3_dispatch(const void* x, const void* dz, float* dw, float* db, int B, int Cin, int Cout, int cin_real, int cout_real, int H, int T,
                           int d, float* scratch, cudaStream_t stream) {
#define TT_WG3(CO, CI) if (Cout == CO * 8 && Cin == CI * 8) return launch_wgrad3<CO, CI>(x, dz, dw, db, B, cin_real, cout_real, H, T, d, scratch, stream);
    TT_WG3(1, 1) TT_WG3(2, 2) TT_WG3(4, 4) TT_WG3(1, 2) TT_WG3(2, 1) TT_WG3(2, 4) TT_WG3(4, 2) TT_WG3(1, 4) TT_WG3(4, 1)
#undef TT_WG3
    return TT_ERR_UNSUPPORTED;
}

extern "C" int tt_conv_wgrad_same(const void* x, const void* dz, float* dw, float* db, int B, int Cin, int Cout, int cin_real, int cout_real,
                                  int H, int T, int k, int dilation, float* scratch, void* stream_) {
    TT_REQUIRE(x && dz && dw && scratch, "null argument");
    TT_REQUIRE((Cin == 8 || Cin == 16 || Cin == 32) && (Cout == 8 || Cout == 16 || Cout == 32), "wgrad: padded channel counts must be 8, 16 or 32");
    TT_REQUIRE(cin_real >= 1 && cin_real <= Cin && cout_real >= 1 && cout_real <= Cout, "wgrad: bad real channel counts");
    TT_REQUIRE((k == 3 && dilation >= 1 && dilation <= 3) || k == 1, "wgrad: 3x3 (dilation 1..3) or 1x1");
    if (B <= 0 || H <= 0 || T <= 0) return TT_OK;
    cudaStream_t stream = (cudaStream_t)stream_;
    if (k == 3) return wgrad3_dispatch(x, dz, dw, db, B, Cin, Cout, cin_real, cout_real, H, T, dilation, scratch, stream);
    // (1x1 layers through resident strips - plain or with four image rows per MMA - were measured slower than the ring kernel with its
    // co-resident CTAs: 293 vs 205 us at the largest stage; the ring kernel without its "ones" MMA stays)
    return wgrad1x1(x, dz, dw, db, B, Cin, Cout, cin_real, cout_real, H, T, scratch, stream);
}

template <int CGC, int CGF>
static int launch_wgrad_ud(const void* fine, const void* coarse, float* dw, float* db, int B, int cfine_real, int ccoarse_real, int Hfine, int Hcoarse,
                           int T, float* scratch, cudaStream_t stream) {
    const WgUdPlan g = wgud_plan(B, CGF, CGC, Hcoarse, T);
    TT_REQUIRE(g.smem <= 227 * 1024 && g.rows + 1 <= kWg3MaxRows, "wgrad_ud: %zu bytes of shared memory, %d rows", g.smem, g.rows);
    static size_t configured = 0;
    if (g.smem > configured) {
        TT_CUDA_CHECK(cudaFuncSetAttribute(wgrad_ud_kernel<CGC, CGF>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)g.smem));
        configured = g.smem;
    }
    CUtensorMap mf, mc;
    int rc = make_row_map(&mf, fine, B, CGF, Hfine, T, kStripTileT);
    if (rc) return rc;
    rc = make_row_map(&mc, coarse, B, CGC, Hcoarse, T, kStripTileT);
    if (rc) return rc;
    WgradUdParams p;
    p.partial = scratch; p.B = B; p.T = T; p.Hc = Hcoarse; p.rows_per_strip = g.rows; p.xring = g.xring; p.per_cta = g.per_cta;
    dim3 grid((T + kStripTileT - 1) / kStripTileT, g.strips, B);
    wgrad_ud_kernel<CGC, CGF><<<grid, kWgThreads, g.smem, stream>>>(mf, mc, p);
    TT_CUDA_CHECK(cudaGetLastError());
    const int n_ctas = (int)(grid.x * grid.y * grid.z);
    const int total = 5 * ccoarse_real * cfine_real;
    wgrad_ud_reduce_kernel<<<(total + 31) / 32, 32 * kWg3RedSeg, 0, stream>>>(scratch, n_ctas, g.per_cta, CGC, CGF <= 2 ? 16 : 32, ccoarse_real, cfine_real, dw, db);
    tt_count_launches(2);
    TT_CUDA_CHECK(cudaGetLastError());
    return TT_OK;
}

static int wgrad_ud_dispatch(const void* fine, const void* coarse, float* dw, float* db, int B, int Cfine, int Ccoarse, int cfine_real,
                             int ccoarse_real, int Hfine, int Hcoarse, int T, float* scratch, cudaStream_t stream) {
#define TT_WGUD(CC, CF) if (Ccoarse == CC * 8 && Cfine == CF * 8) return launch_wgrad_ud<CC, CF>(fine, coarse, dw, db, B, cfine_real, ccoarse_real, Hfine, Hcoarse, T, scratch, stream);
    TT_WGUD(1, 1) TT_WGUD(2, 1) TT_WGUD(4, 2) TT_WGUD(8, 4)
#undef TT_WGUD
    tt_set_error("wgrad_updown: no kernel for %d coarse / %d fine channels (padded)", Ccoarse, Cfine);
    return TT_ERR_UNSUPPORTED;
}

extern "C" int tt_conv_wgrad_updown(const void* fine, const void* coarse, float* dw, float* db, int B, int Cfine, int Ccoarse, int cfine_real,
                                    int ccoarse_real, int Hfine, int Hcoarse, int T, int transposed, float* scratch, void* stream_) {
    TT_REQUIRE(fine && coarse && dw && scratch, "null argument");
    TT_REQUIRE(Cfine % 8 == 0 && Ccoarse % 8 == 0 && Cfine >= 8 && Ccoarse >= 8 && Cfine <= 32 && Ccoarse <= 64,
               "wgrad_updown: fine side up to 32 channels, coarse side up to 64 (padded)");
    TT_REQUIRE(Hfine >= 2 * Hcoarse + 2, "wgrad_updown: the fine tensor must hold rows 2q .. 2q+3 of every coarse row q");
    if (B <= 0 || T <= 0 || Hcoarse <= 0) return TT_OK;
    cudaStream_t stream = (cudaStream_t)stream_;
    // the coarse tensor (sconv: the output gradient; tconv: the layer input) is the A side, the fine one (rows 2q + kh) the B side
    const int rc = wgrad_ud_dispatch(fine, coarse, dw, transposed ? nullptr : db, B, Cfine, Ccoarse, cfine_real, ccoarse_real, Hfine, Hcoarse, T,
                                     scratch, stream);
    if (rc || !transposed || !db) return rc;
    // ConvTranspose2d bias: sum of the FINE tensor (the output gradient) over all pixels
    const int CG = Cfine / 8, chunks = 64;
    const long long hw = (long long)Hfine * T;
    channel_sum_c8_partial_kernel<<<dim3(chunks, CG, B), 256, 0, stream>>>((const uint4*)fine, CG, hw, scratch);
    channel_sum_c8_finish_kernel<<<1, 64, 0, stream>>>(scratch, B, CG, chunks, cfine_real, db);
    tt_count_launches(2);
    TT_CUDA_CHECK(cudaGetLastError());
    return TT_OK;
}

constexpr int kLatTapGroup = 7;       // vertical taps per CTA of the (H, 1)-kernel layers: (7 + 1 bias) x 64 accumulator columns = all of TMEM

extern "C" int64_t tt_wgrad_lat_scratch_floats(int B, int H, int T) {
    const long long nx = (T + kStripTileT - 1) / kStripTileT, groups = (H + kLatTapGroup - 1) / kLatTapGroup;
    return std::max<long long>(nx * groups * B * kWgMaxTaps * 128 * 64, (long long)B * 8 * H * 8);
}

extern "C" int tt_conv_wgrad_lat(const void* tall, const void* flat, float* dw, float* db, float* tall_row_sums, int B, int Ctall, int Cflat,
                                 int ctall_real, int cflat_real, int H, int T, float* scratch, void* stream_) {
    TT_REQUIRE(tall && flat && dw && scratch, "null argument");
    TT_REQUIRE(Ctall % 8 == 0 && Cflat % 8 == 0 && Ctall >= 8 && Ctall <= 64 && Cflat >= 8 && Cflat <= 128,
               "wgrad_lat: up to 64 tall-side and 128 flat-side (padded) channels (got %d, %d)", Ctall, Cflat);
    TT_REQUIRE(ctall_real >= 1 && ctall_real <= Ctall && cflat_real >= 1 && cflat_real <= Cflat && H >= 1, "wgrad_lat: bad sizes");
    if (B <= 0 || T <= 0) return TT_OK;
    cudaStream_t stream = (cudaStream_t)stream_;
    WgradParams p;
    p.partial = scratch;
    p.B = B; p.T = T; p.Hz = 1; p.Hx = H; p.CGi = Ctall / 8; p.CGo = Cflat / 8;
    p.rows_per_strip = 1; p.z_slots = 1; p.tap_group = kLatTapGroup; p.xring = kLatTapGroup + 2;
    const int groups = (H + kLatTapGroup - 1) / kLatTapGroup;
    dim3 grid((T + kStripTileT - 1) / kStripTileT, groups, B);
    const int rc = launch_wgrad<64, kLatTapGroup, 4>(tall, flat, p, grid, stream);
    if (rc) return rc;
    const int total = (H + 1) * cflat_real * ctall_real;
    wgrad_reduce_groups_kernel<<<(total + 127) / 128, 128, 0, stream>>>(scratch, (int)grid.x, groups, B, kLatTapGroup, 64, H, cflat_real, ctall_real, dw, db);
    tt_count_launches(1);
    if (tall_row_sums) {
        // (ctall_real, H) += sum over (b, t) of the tall tensor (after the reduction above has consumed the scratch: same stream)
        row_channel_sum_c8_kernel<<<dim3(H, Ctall / 8, B), 256, 0, stream>>>((const uint4*)tall, Ctall / 8, H, T, scratch);
        row_channel_sum_finish_kernel<<<(ctall_real * H + 127) / 128, 128, 0, stream>>>(scratch, B, Ctall / 8, H, ctall_real, tall_row_sums);
        tt_count_launches(2);
    }
    TT_CUDA_CHECK(cudaGetLastError());
    return TT_OK;
}

static int ew_grid(long long n) { return (int)std::min<long long>((n + 255) / 256, 148 * 16); }

extern "C" int tt_elu_bwd_bf16(const void* gy, const void* a, void* dz, int64_t n, void* stream) {
    TT_REQUIRE(gy && a && dz && n % 8 == 0, "elu_bwd_bf16: null argument or element count not a multiple of 8");
    if (n <= 0) return TT_OK;
    elu_bwd_bf16_kernel<<<ew_grid(n / 8), 256, 0, (cudaStream_t)stream>>>((const uint4*)gy, (const uint4*)a, (uint4*)dz, n / 8);
    tt_count_launches(1);
    TT_CUDA_CHECK(cudaGetLastError());
    return TT_OK;
}

extern "C" int tt_res_out_bwd_bf16(const void* gy, const void* y, const void* x, void* dz, int64_t n, void* stream) {
    TT_REQUIRE(gy && y && x && dz && n % 8 == 0, "res_out_bwd_bf16: null argument or element count not a multiple of 8");
    if (n <= 0) return TT_OK;
    res_out_bwd_bf16_kernel<<<ew_grid(n / 8), 256, 0, (cudaStream_t)stream>>>((const uint4*)gy, (const uint4*)y, (const uint4*)x, (uint4*)dz, n / 8);
    tt_count_launches(1);
    TT_CUDA_CHECK(cudaGetLastError());
    return TT_OK;
}

extern "C" int tt_p4_to_c8(const void* p4, void* c8, int64_t n_pixels, void* stream) {
    TT_REQUIRE(p4 && c8, "null argument");
    if (n_pixels <= 0) return TT_OK;
    p4_to_c8_kernel<<<ew_grid(n_pixels), 256, 0, (cudaStream_t)stream>>>((const uint2*)p4, (uint4*)c8, n_pixels);
    tt_count_launches(1);
    TT_CUDA_CHECK(cudaGetLastError());
    return TT_OK;
}

extern "C" int tt_c8_to_p4(const void* c8, void* p4, int64_t n_pixels, void* stream) {
    TT_REQUIRE(p4 && c8, "null argument");
    if (n_pixels <= 0) return TT_OK;
    c8_to_p4_kernel<<<ew_grid(n_pixels), 256, 0, (cudaStream_t)stream>>>((const uint4*)c8, (uint2*)p4, n_pixels);
    tt_count_launches(1);
    TT_CUDA_CHECK(cudaGetLastError());
    return TT_OK;
}
