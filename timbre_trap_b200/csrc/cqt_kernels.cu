// NSGT / sliCQ analysis and synthesis for B200 (sm_100a).
//
// Replaces cqt_pytorch.CQT.encode / decode as called from the reference wrapper
// (timbre_trap/framework/cqtwrapper.py:67 and :207) plus the wrapper's own to_real / to_complex
// re-layouts (:74-120) and the global peak normalise (:209-211), which are fused here.
//
// Per block of L samples (F bins, M frames):
//
//   analysis    A1  cols_fwd   length-N1 real FFTs down the columns of the (N1 x N2) view of the block,
//                              two real columns per complex transform, four-step twiddle   -> T (L2)
//               A2  rows_fwd   length-N2 complex FFTs along the rows, Hermitian mirror     -> S (L2)
//               A3  bins_fwd   one warp per bin: gather len_k taps of S, window, input-pruned
//                              M-point inverse FFT in registers (32 x 32, one smem transpose),
//                              coalesced streaming store of the (F, T, 2) interleaved row    -> HBM
//   synthesis   S1  bins_inv   one warp per bin: streaming load of the row, M-point FFT, output-pruned
//                              to the len_k taps, dual window, red.add into the block spectrum -> S (L2)
//               S2  rows_inv   Hermitian gather of S, length-N2 inverse FFTs, four-step twiddle -> T (L2)
//               S3  cols_inv   length-N1 inverse FFTs (two real columns per transform), 1/L, per-CTA
//                              max|y| -> atomicMax on the peak scalar, audio store            -> HBM
//               S4  scale      audio *= 1/peak (only when asked to normalise)
//
// T and S are plan-owned scratch sized for `max_blocks` blocks; launches walk the batch in groups of
// that many blocks so the scratch stays L2-resident while the coefficient tensor streams past it.
//
// Algorithmic HBM bytes per block (the roofline numerator): 4*L + 8*F*M in either direction.

#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <string.h>

#include <vector>

#include "../../include/timbre_trap_b200.h"
#include "fft_device.cuh"

// ---------------------------------------------------------------------------------------------
// error plumbing
// ---------------------------------------------------------------------------------------------
static thread_local char g_err[512] = "";

void tt_set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

extern "C" const char* tt_last_error(void) { return g_err; }
extern "C" int tt_version(void) { return 1; }

#include <atomic>
static std::atomic<long long> g_launches{0};
void tt_count_launches(int n) { g_launches.fetch_add(n, std::memory_order_relaxed); }
extern "C" long long tt_launch_count(int reset) {
    return reset ? g_launches.exchange(0, std::memory_order_relaxed) : g_launches.load(std::memory_order_relaxed);
}

namespace tt {

constexpr int kColsPerCta = 32;   // A1 / S3: real columns per CTA (even: two per complex transform; 32 floats = 128 B runs)
constexpr int kRowsPerCta = 16;   // A2 / S2: rows per CTA (16 complex = 128 B runs in S)
constexpr int kFftThreads = 256;
constexpr int kBinWarps = 4;      // A3 / S1: warps (= bins) per CTA (small CTAs: 5 per SM at 88 registers)

// ---------------------------------------------------------------------------------------------
// A1: forward column transforms
//   x viewed as x[N2 * n1 + n2].  For each column n2: A[k1] = sum_n1 x[n1, n2] w_N1^{k1 n1}, kept for
//   k1 <= N1/2 (x is real), multiplied by w_L^{k1 n2} and stored as T[k1][n2].
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kFftThreads)
cols_fwd_kernel(const float* __restrict__ audio, float2* __restrict__ T, FftSpec spec, int N2, int K1, int L,
                const float2* __restrict__ tw_n1, const float2* __restrict__ tw_L) {
    extern __shared__ float2 smem[];
    const int N1 = spec.n;
    constexpr int G = kColsPerCta;
    float2* buf_a = smem;
    float2* buf_b = smem + (G / 2) * N1;
    float2* tw = buf_b + (G / 2) * N1;
    const int tid = threadIdx.x;
    const int n2_0 = blockIdx.x * G;
    const float* x = audio + (size_t)blockIdx.y * L;

    for (int i = tid; i < N1; i += kFftThreads) tw[i] = tw_n1[i];
    float* buf_f = reinterpret_cast<float*>(buf_a);
#pragma unroll 8
    for (int i = tid; i < N1 * G; i += kFftThreads) {
        const int n1 = i / G, g = i - n1 * G;
        const int n2 = n2_0 + g;
        const float v = n2 < N2 ? __ldg(x + (size_t)N2 * n1 + n2) : 0.f;
        buf_f[((g >> 1) * N1 + n1) * 2 + (g & 1)] = v;
    }
    __syncthreads();
    const float2* Z = run_passes<-1>(spec, buf_a, buf_b, tw, G / 2, tid, kFftThreads);

    float2* Tb = T + (size_t)blockIdx.y * K1 * N2;
#pragma unroll 4
    for (int i = tid; i < K1 * G; i += kFftThreads) {
        const int k1 = i / G, g = i - k1 * G;
        const int n2 = n2_0 + g;
        if (n2 >= N2) continue;
        const float2* z = Z + (g >> 1) * N1;
        const float2 a = z[k1];
        const float2 b = cconj(z[k1 == 0 ? 0 : N1 - k1]);
        // column pair (xa, xb) packed as xa + i xb:  Xa = (Z + Zr)/2,  Xb = (Z - Zr)/(2i)
        float2 r;
        if ((g & 1) == 0) r = cscale(cadd(a, b), 0.5f);
        else r = cscale(cmul_mi(csub(a, b)), 0.5f);
        r = cmul(r, tw_L[k1 * n2]);          // k1 <= N1/2 and n2 < N2, so k1 * n2 < L/2: no reduction mod L needed
        Tb[(size_t)k1 * N2 + n2] = r;
    }
}

// ---------------------------------------------------------------------------------------------
// A2: forward row transforms.  X[k1 + N1 k2] = sum_n2 T[k1][n2] w_N2^{k2 n2}; the other half of the
// spectrum follows from X[L - j] = conj(X[j]).  Only j <= L/2 is stored (S, natural order).
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kFftThreads)
rows_fwd_kernel(const float2* __restrict__ T, float2* __restrict__ S, FftSpec spec, int N1, int K1, int L, int SP,
                const float2* __restrict__ tw_n2) {
    extern __shared__ float2 smem[];
    const int N2 = spec.n;
    constexpr int R = kRowsPerCta;
    float2* buf_a = smem;
    float2* buf_b = smem + R * N2;
    float2* tw = buf_b + R * N2;
    const int tid = threadIdx.x;
    const int k1_0 = blockIdx.x * R;
    const int rows = min(R, K1 - k1_0);
    const float2* Tb = T + ((size_t)blockIdx.y * K1 + k1_0) * N2;

    for (int i = tid; i < N2; i += kFftThreads) tw[i] = tw_n2[i];
#pragma unroll 8
    for (int i = tid; i < rows * N2; i += kFftThreads) buf_a[i] = Tb[i];
    __syncthreads();
    const float2* X = run_passes<-1>(spec, buf_a, buf_b, tw, rows, tid, kFftThreads);

    float2* Sb = S + (size_t)blockIdx.y * SP;
    const int half = L / 2;
    for (int i = tid; i < rows * N2; i += kFftThreads) {
        const int k2 = i / rows, r = i - k2 * rows;
        const int j = k1_0 + r + N1 * k2;
        const float2 v = X[r * N2 + k2];
        if (j <= half) Sb[j] = v;
        // mirror only into slots no row computes directly (jm mod N1 > N1/2): every S[j] has exactly one writer,
        // so the spectrum is bit-reproducible
        const int jm = L - j;
        if (j != 0 && jm <= half && (jm % N1) >= K1) Sb[jm] = cconj(v);
    }
}

// ---------------------------------------------------------------------------------------------
// A3: per-bin window + inverse M-point FFT, M = 1024 = 32 x 32, one warp per (block, bin).
//
//   c[n] = sum_m a[m] e^{+2 pi i m n / M},  a[m] = X[start + (m - first)] * win[m - first] / M  on the
//   len taps m in [first, first+len) and 0 elsewhere.  With pp = 32*floor(first/32), m = pp + 32 m1 + m0
//   (m0 = lane) and n = n0 + 32 n1:
//       B[m0][n0] = sum_{m1 < Z} a[m1][m0] w32^{m1 n0}            (input-pruned: Z rows are non-zero)
//       B[m0][n0] *= w1024^{(m0 + pp) n0}
//       c[n0 + 32 n1] = sum_{m0} B[m0][n0] w32^{m0 n1}             (after a 32x32 transpose through smem)
// ---------------------------------------------------------------------------------------------
struct BinTables {
    const int* start;
    const int* length;
    const int* first;
    const int* offset;
    const float* win;    // window / M   (analysis)
    const float* dual;   // dual window  (synthesis)
};

// Offset (in float2) of the row of bin k in block gb of a (items, F, n_blocks * M) interleaved coefficient tensor.  Uniform items of
// n_blocks_item blocks, or - clip_block0 non-null - clips of clip_block0[c + 1] - clip_block0[c] blocks packed one after the other
// (the many-clip calls, find_clip), each in the layout a one-clip call has.
__device__ __forceinline__ size_t coeff_row(int gb, int k, int F, int M, int n_blocks_item, const int* __restrict__ clip_block0,
                                            int n_clips) {
    int first, n;
    if (clip_block0) {
        const int c = find_clip(clip_block0, n_clips, gb);
        first = __ldg(clip_block0 + c) - __ldg(clip_block0);
        n = __ldg(clip_block0 + c + 1) - __ldg(clip_block0 + c);
    } else {
        first = gb / n_blocks_item * n_blocks_item;
        n = n_blocks_item;
    }
    return (size_t)first * F * M + (size_t)k * n * M + (size_t)(gb - first) * M;
}

template <int Z>
__device__ __forceinline__ void bin_fwd_stage1(const float2* __restrict__ spec_taps, const float* __restrict__ win,
                                               int len, int shift, int lane, float2 (&B)[32]) {
    // a[m1] for m1 < Z;  tap index i = 32 m1 + lane - shift  (shift = first - pp)
    float2 a[Z];
#pragma unroll
    for (int m1 = 0; m1 < Z; ++m1) {
        const int i = 32 * m1 + lane - shift;
        float2 v = make_float2(0.f, 0.f);
        if (i >= 0 && i < len) {
            const float w = __ldg(win + i);
            const float2 x = __ldg(spec_taps + i);
            v = make_float2(x.x * w, x.y * w);
        }
        a[m1] = v;
    }
    constexpr int D = 32 / Z;
    // B[D q + r] = sum_{m1<Z} (a[m1] w32^{m1 r}) e^{2 pi i m1 q / Z}
#pragma unroll
    for (int r = 0; r < D; ++r) {
        float2 t[Z];
#pragma unroll
        for (int m1 = 0; m1 < Z; ++m1) t[m1] = mul_tw32<+1>(a[m1], m1 * r);
        if constexpr (Z > 1) {
            // Z-point DIF with table stride 32/Z: reuse the 32-table by scaling indices
            // (fft_reg_dif<Z> indexes the 32-point table as j*(16/half); for a Z-point transform the
            //  twiddle is exp(2 pi i j/(2 half)) = w32^{j*16/half}, identical expression)
            fft_reg_dif<Z, +1>(t);
        }
#pragma unroll
        for (int q = 0; q < Z; ++q) B[D * q + r] = t[brev<Z>(q)];
    }
}

__global__ void __launch_bounds__(kBinWarps * 32, 6)
bins_fwd_kernel(const float2* __restrict__ S, float* __restrict__ coeffs, BinTables tab, int F, int SP,
                int n_blocks_item, int block0, int n_blocks_launch, const float2* __restrict__ tw_m) {
    constexpr int M = 1024;
    extern __shared__ float2 smem[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    float2* tile = smem + warp * (32 * 33);
    // exp(+2 pi i k / 1024): five reads per transform, straight from the 8 KB global table (L1-resident) - no shared-memory copy, so
    // six 4-warp CTAs fit an SM

    const long long w = (long long)blockIdx.x * kBinWarps + warp;
    if (w >= (long long)n_blocks_launch * F) return;
    const int lb = (int)(w / F);             // block within this launch
    const int k = (int)(w - (long long)lb * F);
    const int gb = block0 + lb;              // global block index = item * n_blocks_item + blk
    const int item = gb / n_blocks_item, blk = gb - item * n_blocks_item;

    const int len = tab.length[k], first = tab.first[k];
    const int pp = first & ~31;
    const int shift = first - pp;
    const int rows = (shift + len + 31) >> 5;
    const float2* taps = S + (size_t)lb * SP + tab.start[k];
    const float* win = tab.win + tab.offset[k];

    float2 B[32];
    if (rows <= 1) bin_fwd_stage1<1>(taps, win, len, shift, lane, B);
    else if (rows <= 2) bin_fwd_stage1<2>(taps, win, len, shift, lane, B);
    else if (rows <= 4) bin_fwd_stage1<4>(taps, win, len, shift, lane, B);
    else if (rows <= 8) bin_fwd_stage1<8>(taps, win, len, shift, lane, B);
    else if (rows <= 16) bin_fwd_stage1<16>(taps, win, len, shift, lane, B);
    else bin_fwd_stage1<32>(taps, win, len, shift, lane, B);

    // twiddle w1024^{(m0 + pp) n0} and transpose.  The factors of one lane are a geometric sequence in n0: re-seeded from the table
    // every 8 steps and advanced by one complex multiply in between (4 table reads instead of 32; error <= 8 roundings)
    const int base = (lane + pp) & (M - 1);
    const float2 w1 = __ldg(tw_m + base);
#pragma unroll
    for (int n0 = 0; n0 < 32; n0 += 8) {
        float2 t = __ldg(tw_m + ((base * n0) & (M - 1)));
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            tile[(n0 + q) * 33 + lane] = (n0 + q == 0) ? B[0] : cmul(B[n0 + q], t);
            if (q < 7) t = cmul(t, w1);
        }
    }
    __syncwarp();
    float2 E[32];
#pragma unroll
    for (int m0 = 0; m0 < 32; ++m0) E[m0] = tile[lane * 33 + m0];
    fft_reg_dif<32, +1>(E);

    float2* out = reinterpret_cast<float2*>(coeffs) +
                  ((size_t)item * F + k) * ((size_t)n_blocks_item * M) + (size_t)blk * M;
#pragma unroll
    for (int n1 = 0; n1 < 32; ++n1) st_stream(out + lane + 32 * n1, E[brev<32>(n1)]);
}

// ---------------------------------------------------------------------------------------------
// S1: per-bin M-point FFT of a coefficient row, output-pruned to the bin's taps, dual window,
// overlap-add into the block spectrum.  Transposed data flow of A3:
//       D[n0][m0] = sum_{n1} c[n0 + 32 n1] w32^{-m0 n1}
//       D[n0][m0] *= w1024^{-(m0 + pp) n0}
//       C[pp + 32 m1 + m0] = sum_{n0} D[n0][m0] w32^{-m1 n0}      for m1 < Z only
// ---------------------------------------------------------------------------------------------
template <int Z>
__device__ __forceinline__ void bin_inv_stage3(float2 (&E)[32], float2* __restrict__ spec_taps,
                                               const float* __restrict__ dual, int len, int shift, int lane) {
    constexpr int D = 32 / Z;
    float2 C[Z];
#pragma unroll
    for (int m1 = 0; m1 < Z; ++m1) C[m1] = make_float2(0.f, 0.f);
    // C[m1] = sum_{r<D} w32^{-m1 r} * DFT_Z( E[D q + r] over q )[m1]
#pragma unroll
    for (int r = 0; r < D; ++r) {
        float2 t[Z];
#pragma unroll
        for (int q = 0; q < Z; ++q) t[q] = E[D * q + r];
        if constexpr (Z > 1) fft_reg_dif<Z, -1>(t);
#pragma unroll
        for (int m1 = 0; m1 < Z; ++m1) C[m1] = cadd2(C[m1], mul_tw32<-1>(t[brev<Z>(m1)], m1 * r));
    }
#pragma unroll
    for (int m1 = 0; m1 < Z; ++m1) {
        const int i = 32 * m1 + lane - shift;
        if (i >= 0 && i < len) {
            const float w = __ldg(dual + i);
            atomicAdd(spec_taps + i, make_float2(C[m1].x * w, C[m1].y * w));      // one 64-bit vector reduction (sm_90+)
        }
    }
}

__global__ void __launch_bounds__(kBinWarps * 32, 6)
bins_inv_kernel(const float* __restrict__ coeffs, float2* __restrict__ S, BinTables tab, int F, int SP,
                int n_blocks_item, int block0, int n_blocks_launch, const float2* __restrict__ tw_m,
                const int* __restrict__ clip_block0, int n_clips) {
    constexpr int M = 1024;
    extern __shared__ float2 smem[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    float2* tile = smem + warp * (32 * 33);

    const long long w = (long long)blockIdx.x * kBinWarps + warp;
    if (w >= (long long)n_blocks_launch * F) return;
    const int lb = (int)(w / F);
    const int k = (int)(w - (long long)lb * F);
    const float2* in = reinterpret_cast<const float2*>(coeffs) + coeff_row(block0 + lb, k, F, M, n_blocks_item, clip_block0, n_clips);
    float2 v[32];
#pragma unroll
    for (int n1 = 0; n1 < 32; ++n1) v[n1] = ld_stream(in + lane + 32 * n1);
    fft_reg_dif<32, -1>(v);      // v[brev(m0)] = D[n0 = lane][m0]

    const int len = tab.length[k], first = tab.first[k];
    const int pp = first & ~31;
    const int shift = first - pp;
    const int rows = (shift + len + 31) >> 5;
    // twiddle w1024^{-(m0 + pp) n0}, n0 = lane: geometric in m0 with ratio w1024^{lane}, re-seeded every 8 steps (see bins_fwd)
    const float2 wl = __ldg(tw_m + lane);
#pragma unroll
    for (int m0 = 0; m0 < 32; m0 += 8) {
        float2 t = __ldg(tw_m + ((((m0 + pp) & (M - 1)) * lane) & (M - 1)));
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            tile[(m0 + q) * 33 + lane] = cmulc(v[brev<32>(m0 + q)], t);
            if (q < 7) t = cmul(t, wl);
        }
    }
    __syncwarp();
    float2 E[32];
#pragma unroll
    for (int n0 = 0; n0 < 32; ++n0) E[n0] = tile[lane * 33 + n0];   // lane = m0

    float2* taps = S + (size_t)lb * SP + tab.start[k];
    const float* dual = tab.dual + tab.offset[k];
    if (rows <= 1) bin_inv_stage3<1>(E, taps, dual, len, shift, lane);
    else if (rows <= 2) bin_inv_stage3<2>(E, taps, dual, len, shift, lane);
    else if (rows <= 4) bin_inv_stage3<4>(E, taps, dual, len, shift, lane);
    else if (rows <= 8) bin_inv_stage3<8>(E, taps, dual, len, shift, lane);
    else if (rows <= 16) bin_inv_stage3<16>(E, taps, dual, len, shift, lane);
    else bin_inv_stage3<32>(E, taps, dual, len, shift, lane);
}

// ---------------------------------------------------------------------------------------------
// Generic-M variants (any power of two M >= 4 other than 1024): one CTA per (block, bin), the M-point
// transform runs as shared-memory Stockham passes.  Correct for every configuration the wrapper can
// be constructed with; the 1024 path above is the tuned one (the reference's base configuration).
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128)
bins_fwd_generic_kernel(const float2* __restrict__ S, float* __restrict__ coeffs, BinTables tab, int F, int SP,
                        int n_blocks_item, int block0, FftSpec spec, const float2* __restrict__ tw_m_fwd) {
    extern __shared__ float2 smem[];
    const int M = spec.n;
    float2* buf_a = smem;
    float2* buf_b = smem + M;
    float2* tw = smem + 2 * M;
    const int tid = threadIdx.x;
    const int k = blockIdx.x, lb = blockIdx.y;
    const int gb = block0 + lb;
    const int item = gb / n_blocks_item, blk = gb - item * n_blocks_item;
    const int len = tab.length[k], first = tab.first[k];
    const float2* taps = S + (size_t)lb * SP + tab.start[k];
    const float* win = tab.win + tab.offset[k];
    for (int i = tid; i < M; i += 128) {
        tw[i] = tw_m_fwd[i];
        const int t = i - first;
        float2 v = make_float2(0.f, 0.f);
        if (t >= 0 && t < len) v = cscale(taps[t], win[t]);
        buf_a[i] = v;
    }
    __syncthreads();
    const float2* c = run_passes<+1>(spec, buf_a, buf_b, tw, 1, tid, 128);
    float2* out = reinterpret_cast<float2*>(coeffs) +
                  ((size_t)item * F + k) * ((size_t)n_blocks_item * M) + (size_t)blk * M;
    for (int i = tid; i < M; i += 128) st_stream(out + i, c[i]);
}

__global__ void __launch_bounds__(128)
bins_inv_generic_kernel(const float* __restrict__ coeffs, float2* __restrict__ S, BinTables tab, int F, int SP,
                        int n_blocks_item, int block0, FftSpec spec, const float2* __restrict__ tw_m_fwd,
                        const int* __restrict__ clip_block0, int n_clips) {
    extern __shared__ float2 smem[];
    const int M = spec.n;
    float2* buf_a = smem;
    float2* buf_b = smem + M;
    float2* tw = smem + 2 * M;
    const int tid = threadIdx.x;
    const int k = blockIdx.x, lb = blockIdx.y;
    const float2* in = reinterpret_cast<const float2*>(coeffs) + coeff_row(block0 + lb, k, F, M, n_blocks_item, clip_block0, n_clips);
    for (int i = tid; i < M; i += 128) {
        tw[i] = tw_m_fwd[i];
        buf_a[i] = ld_stream(in + i);
    }
    __syncthreads();
    const float2* C = run_passes<-1>(spec, buf_a, buf_b, tw, 1, tid, 128);
    const int len = tab.length[k], first = tab.first[k];
    float2* taps = S + (size_t)lb * SP + tab.start[k];
    const float* dual = tab.dual + tab.offset[k];
    for (int t = tid; t < len; t += 128) {
        atomicAdd(taps + t, cscale(C[first + t], dual[t]));
    }
}

// ---------------------------------------------------------------------------------------------
// S2: inverse row transforms.  y = Re ifft_L(Y) with Y one-sided, i.e. ifft of the Hermitian
//   H[0] = Re Y[0], H[L/2] = Re Y[L/2] (L even), H[j] = Y[j]/2, H[L-j] = conj(Y[j])/2.
//   G[k1][n2] = w_L^{-k1 n2} sum_k2 H[k1 + N1 k2] w_N2^{-k2 n2}          for k1 <= N1/2
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kFftThreads)
rows_inv_kernel(const float2* __restrict__ S, float2* __restrict__ T, FftSpec spec, int N1, int K1, int L, int SP,
                const float2* __restrict__ tw_n2, const float2* __restrict__ tw_L) {
    extern __shared__ float2 smem[];
    const int N2 = spec.n;
    constexpr int R = kRowsPerCta;
    float2* buf_a = smem;
    float2* buf_b = smem + R * N2;
    float2* tw = buf_b + R * N2;
    const int tid = threadIdx.x;
    const int k1_0 = blockIdx.x * R;
    const int rows = min(R, K1 - k1_0);
    const float2* Sb = S + (size_t)blockIdx.y * SP;
    const int half = L / 2;
    const bool even = (L & 1) == 0;

    for (int i = tid; i < N2; i += kFftThreads) tw[i] = tw_n2[i];
    for (int i = tid; i < rows * N2; i += kFftThreads) {
        const int k2 = i / rows, r = i - k2 * rows;
        const int j = k1_0 + r + N1 * k2;
        float2 h;
        if (j == 0) h = make_float2(Sb[0].x, 0.f);
        else if (even && j == half) h = make_float2(Sb[half].x, 0.f);
        else if (j <= half) h = cscale(Sb[j], 0.5f);
        else h = cscale(cconj(Sb[L - j]), 0.5f);
        buf_a[r * N2 + k2] = h;
    }
    __syncthreads();
    const float2* Gm = run_passes<+1>(spec, buf_a, buf_b, tw, rows, tid, kFftThreads);

    float2* Tb = T + ((size_t)blockIdx.y * K1 + k1_0) * N2;
    for (int i = tid; i < rows * N2; i += kFftThreads) {
        const int r = i / N2, n2 = i - r * N2;
        Tb[i] = cmulc(Gm[i], tw_L[(k1_0 + r) * n2]);      // (k1 <= N1/2) * (n2 < N2) < L/2
    }
}

// ---------------------------------------------------------------------------------------------
// S3: inverse column transforms + 1/L + peak.   y[N2 n1 + n2] = (1/L) sum_k1 G[k1][n2] w_N1^{-k1 n1},
// G Hermitian in k1; two real columns share one complex transform (Z = Ga + i Gb -> ya = Re, yb = Im).
// One peak for the whole call, or - clip_block0 non-null - one per clip (block block0 + blockIdx.y is in clip find_clip(..)).
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kFftThreads)
cols_inv_kernel(const float2* __restrict__ T, float* __restrict__ audio, FftSpec spec, int N2, int K1, int L,
                const float2* __restrict__ tw_n1, unsigned int* __restrict__ peak_bits, const int* __restrict__ clip_block0,
                int n_clips, int block0) {
    extern __shared__ float2 smem[];
    const int N1 = spec.n;
    constexpr int G = kColsPerCta;
    float2* buf_a = smem;
    float2* buf_b = smem + (G / 2) * N1;
    float2* tw = buf_b + (G / 2) * N1;
    __shared__ float red[kFftThreads / 32];
    const int tid = threadIdx.x;
    const int n2_0 = blockIdx.x * G;
    const float2* Tb = T + (size_t)blockIdx.y * K1 * N2;

    for (int i = tid; i < N1; i += kFftThreads) tw[i] = tw_n1[i];
    for (int i = tid; i < N1 * (G / 2); i += kFftThreads) {
        const int k1 = i / (G / 2), f = i - k1 * (G / 2);
        const int na = n2_0 + 2 * f, nb = na + 1;
        const int ks = k1 < K1 ? k1 : N1 - k1;          // Hermitian source row
        float2 ga = make_float2(0.f, 0.f), gb = make_float2(0.f, 0.f);
        if (na < N2) ga = Tb[(size_t)ks * N2 + na];
        if (nb < N2) gb = Tb[(size_t)ks * N2 + nb];
        if (k1 >= K1) { ga = cconj(ga); gb = cconj(gb); }
        buf_a[f * N1 + k1] = cadd(ga, cmul_i(gb));
    }
    __syncthreads();
    const float2* y = run_passes<+1>(spec, buf_a, buf_b, tw, G / 2, tid, kFftThreads);

    float* out = audio + (size_t)blockIdx.y * L;
    const float inv_l = 1.0f / (float)L;
    float peak = 0.f;
    for (int i = tid; i < N1 * G; i += kFftThreads) {
        const int n1 = i / G, g = i - n1 * G;
        const int n2 = n2_0 + g;
        if (n2 >= N2) continue;
        const float2 z = y[(g >> 1) * N1 + n1];
        const float v = ((g & 1) ? z.y : z.x) * inv_l;
        out[(size_t)N2 * n1 + n2] = v;
        peak = fmaxf(peak, fabsf(v));
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) peak = fmaxf(peak, __shfl_xor_sync(0xffffffffu, peak, o));
    if ((tid & 31) == 0) red[tid >> 5] = peak;
    __syncthreads();
    if (tid == 0) {
        for (int i = 1; i < kFftThreads / 32; ++i) peak = fmaxf(peak, red[i]);
        const int clip = clip_block0 ? find_clip(clip_block0, n_clips, block0 + (int)blockIdx.y) : 0;
        atomicMax(peak_bits + clip, __float_as_uint(peak));   // non-negative floats order like their bit patterns
    }
}

__global__ void scale_by_peak_kernel(float* __restrict__ audio, long long n, const float* __restrict__ peak) {
    const float p = *peak;
    if (!(p > 0.f)) return;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) audio[i] = audio[i] / p;
}

// the same per clip: block blockIdx.y (L samples) is divided by the peak of its clip
__global__ void scale_by_clip_peak_kernel(float* __restrict__ audio, int L, const int* __restrict__ clip_block0, int n_clips,
                                          const float* __restrict__ peaks) {
    const float p = peaks[find_clip(clip_block0, n_clips, blockIdx.y)];
    if (!(p > 0.f)) return;
    float* a = audio + (size_t)blockIdx.y * L;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < L; i += gridDim.x * blockDim.x) a[i] = a[i] / p;
}

// ---------------------------------------------------------------------------------------------
// element-wise readers of the interleaved coefficient layout
// ---------------------------------------------------------------------------------------------
__global__ void magnitude_kernel(const float2* __restrict__ c, long long n, int apply_tanh, float* __restrict__ out) {
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const float2 v = ld_stream(c + i);
        float m = sqrtf(v.x * v.x + v.y * v.y);
        if (apply_tanh) m = tanhf(m);
        out[i] = m;
    }
}

__global__ void item_max_kernel(const float* __restrict__ x, long long per_item, unsigned int* __restrict__ item_max) {
    const float* p = x + (size_t)blockIdx.y * per_item;
    float m = 0.f;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < per_item; i += stride) m = fmaxf(m, p[i]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    if ((threadIdx.x & 31) == 0) atomicMax(item_max + blockIdx.y, __float_as_uint(fmaxf(m, 0.f)));
}

__global__ void decibels_kernel(const float* __restrict__ x, long long per_item, int rescale, float* __restrict__ out,
                                const float* __restrict__ item_max) {
    // AmplitudeToDB(stype='amplitude', top_db=80): 20 log10(clamp(x, 1e-10)), floored at (item max dB - 80)
    const float top = 20.f * log10f(fmaxf(item_max[blockIdx.y], 1e-10f));
    const float* p = x + (size_t)blockIdx.y * per_item;
    float* q = out + (size_t)blockIdx.y * per_item;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < per_item; i += stride) {
        float d = 20.f * log10f(fmaxf(p[i], 1e-10f));
        d = fmaxf(d, top - 80.f);
        if (rescale) d = 1.f + (d - top) / 80.f;
        q[i] = d;
    }
}


// Cross-fade of 50 %-overlapped chunk outputs (TimbreTrap.chunked_inference, modules.py:259-267), as a gather: output
// frame t (after the M/2 trim) receives chunk i1 = (t + M/2) / (M/2) at position p1 = (t + M/2) mod (M/2) and chunk
// i1 - 1 at position p1 + M/2, each scaled by the window.  Products are rounded separately and added in chunk order,
// like the reference's `coefficients[...] += window * output_chunk`.
// blockIdx.z is the item: batch items of n_chunks chunks each, or - clip_chunk0 non-null - clip z of the chunk prefix table
// (find_clip), whose chunks and whose (F, (n - 1) M/2) output rows follow those of the clips before it.
__global__ void crossfade_kernel(const float2* __restrict__ chunks, const float* __restrict__ window, int n_chunks, int F,
                                 int M, float2* __restrict__ coeffs_out, float* __restrict__ act_out, const int* __restrict__ clip_chunk0) {
    const int half = M / 2;
    const int b = blockIdx.z, f = blockIdx.y;
    size_t chunk0 = (size_t)b * n_chunks, out0 = (size_t)b * F * ((size_t)(n_chunks - 1) * half);
    if (clip_chunk0) {
        const int c0 = __ldg(clip_chunk0 + b) - __ldg(clip_chunk0);
        n_chunks = __ldg(clip_chunk0 + b + 1) - __ldg(clip_chunk0 + b);
        chunk0 = (size_t)c0;
        out0 = (size_t)F * half * (size_t)(c0 - b);       // sum over earlier clips of F (n_c - 1) M/2
    }
    const long long n_out = (long long)(n_chunks - 1) * half;
    const float2* base = chunks + (chunk0 * F + f) * M;       // chunk i of the item: + i * F * M
    const size_t chunk_stride = (size_t)F * M;
    const size_t out_row = out0 + (size_t)f * n_out;
    for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < n_out; t += (long long)gridDim.x * blockDim.x) {
        const long long tf = t + half;
        const int i1 = (int)(tf / half);
        const int p1 = (int)(tf - (long long)i1 * half);
        const float2 c0 = ld_stream(base + (size_t)(i1 - 1) * chunk_stride + p1 + half);
        const float2 c1 = ld_stream(base + (size_t)i1 * chunk_stride + p1);
        const float w0 = window[p1 + half], w1 = window[p1];
        float2 r;
        r.x = __fadd_rn(__fmul_rn(w0, c0.x), __fmul_rn(w1, c1.x));
        r.y = __fadd_rn(__fmul_rn(w0, c0.y), __fmul_rn(w1, c1.y));
        if (coeffs_out) coeffs_out[out_row + t] = r;
        if (act_out) act_out[out_row + t] = tanhf(sqrtf(r.x * r.x + r.y * r.y));
    }
}

// The chunk matrix of the many-clip calls (TimbreTrap._chunks of every clip, modules.py:226-234): clip c of n_c samples, zero-padded
// to a whole number of blocks and by half a block on either side, cut into 50 %-overlapped chunks of L samples.  Row r of `out` is
// chunk chunk_lo + r of the clip list; clip_chunk0 is the chunk prefix table (find_clip), clips[c] = (address, samples) of clip c.
__global__ void gather_chunks_kernel(const longlong2* __restrict__ clips, const int* __restrict__ clip_chunk0, int n_clips,
                                     int chunk_lo, int L, float* __restrict__ out) {
    const int g = chunk_lo + (int)blockIdx.y;
    const int c = find_clip(clip_chunk0, n_clips, g);
    const longlong2 clip = clips[c];
    const float* x = reinterpret_cast<const float*>(clip.x);
    const int hop = L / 2;
    const long long s0 = (long long)(g - (__ldg(clip_chunk0 + c) - __ldg(clip_chunk0))) * hop - hop;
    float* o = out + (size_t)blockIdx.y * L;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < L; i += gridDim.x * blockDim.x) {
        const long long s = s0 + i;
        o[i] = (s >= 0 && s < clip.y) ? __ldg(x + s) : 0.f;
    }
}

}  // namespace tt

// =============================================================================================
// host side: plan
// =============================================================================================
using namespace tt;

constexpr int kMaxLanes = 4;

struct tt_cqt_plan {
    int L, F, M, n_taps;
    int N1, N2, K1, SP;
    int max_blocks;
    FftSpec spec_n1, spec_n2, spec_m;
    // device tables
    int *d_start, *d_length, *d_first, *d_offset;
    float *d_win, *d_dual;
    float2 *d_tw_n1, *d_tw_n2, *d_tw_L, *d_tw_m_inv, *d_tw_m_fwd;
    // scratch
    // two scratch sets + two internal streams: consecutive groups of blocks run on alternating lanes, so the FFT front end of
    // group g+1 overlaps the HBM-bound per-bin kernel of group g
    float2 *d_T[kMaxLanes], *d_S[kMaxLanes];
    cudaStream_t lane[kMaxLanes];
    cudaEvent_t ev_start, ev_done[kMaxLanes];
    int n_lanes;                   // lanes in use (consecutive groups of blocks rotate over them)
    int64_t scratch_bytes;
};

static bool factor_2357(int n, FftSpec* spec) {
    memset(spec, 0, sizeof(*spec));
    spec->n = n;
    int r = n;
    // composite radices first (fewer shared-memory passes), then the primes; radix 4 before 2
    const int order[] = {10, 9, 6, 7, 5, 4, 3, 2};
    for (int p : order)
        while (r % p == 0) {
            if (spec->n_passes >= kMaxPasses) return false;
            spec->radix[spec->n_passes++] = p;
            r /= p;
        }
    if (r != 1) return false;
    int s = 1;
    for (int i = 0; i < spec->n_passes; ++i) {
        const unsigned per = (unsigned)(n / spec->radix[i]);
        spec->magic_per[i] = (unsigned)(0x100000000ull / per) + 1u;
        spec->magic_s[i] = (unsigned)(0x100000000ull / (unsigned)s) + 1u;     // unused when s == 1
        s *= spec->radix[i];
    }
    return true;
}

static void make_twiddles(std::vector<float2>& out, int n, int sign) {
    out.resize(n);
    for (int k = 0; k < n; ++k) {
        const double a = sign * 2.0 * M_PI * (double)k / (double)n;
        out[k] = make_float2((float)cos(a), (float)sin(a));
    }
}

template <typename T>
static int upload(T** dst, const T* src, size_t count) {
    TT_CUDA_CHECK(cudaMalloc((void**)dst, count * sizeof(T)));
    TT_CUDA_CHECK(cudaMemcpy(*dst, src, count * sizeof(T), cudaMemcpyHostToDevice));
    return TT_OK;
}

static size_t cols_smem(const tt_cqt_plan* p) { return ((size_t)kColsPerCta * p->N1 + p->N1) * sizeof(float2); }
static size_t rows_smem(const tt_cqt_plan* p) { return ((size_t)2 * kRowsPerCta * p->N2 + p->N2) * sizeof(float2); }
static size_t bins_smem() { return ((size_t)kBinWarps * 32 * 33) * sizeof(float2); }

extern "C" int tt_cqt_plan_create(tt_cqt_plan** out, int block_length, int n_bins, int max_window_length,
                                  const int32_t* start, const int32_t* length, const int32_t* first,
                                  const int32_t* offset, const float* win_packed, const float* dual_packed,
                                  int n_taps, int max_blocks_per_launch) {
    TT_REQUIRE(out && start && length && first && offset && win_packed && dual_packed, "null argument");
    TT_REQUIRE(block_length >= 4 && n_bins >= 1 && max_blocks_per_launch >= 1, "bad sizes");
    const int L = block_length, F = n_bins, M = max_window_length;
    TT_REQUIRE(M >= 4 && (M & (M - 1)) == 0 && M <= 8192, "max_window_length must be a power of two in [4, 8192], got %d", M);
    TT_REQUIRE(offset[F] == n_taps, "offset[F] != n_taps");
    for (int k = 0; k < F; ++k) {
        TT_REQUIRE(length[k] >= 1 && first[k] >= 0 && first[k] + length[k] <= M, "bin %d: taps outside the crop", k);
        TT_REQUIRE(start[k] >= 0 && start[k] + length[k] - 1 <= L / 2,
                   "bin %d: taps outside the one-sided spectrum [0, L/2] (start %d, len %d)", k, start[k], length[k]);
    }

    tt_cqt_plan* p = new tt_cqt_plan();
    memset(p, 0, sizeof(*p));
    p->L = L; p->F = F; p->M = M; p->n_taps = n_taps; p->max_blocks = max_blocks_per_launch;

    // four-step split L = N1 * N2, both {2,3,5,7}-smooth, as square as possible, small enough for smem
    int best = 0;
    for (int n1 = 1; (long long)n1 * n1 <= (long long)L; ++n1) {
        if (L % n1) continue;
        FftSpec a, b;
        if (!factor_2357(n1, &a) || !factor_2357(L / n1, &b)) continue;
        best = n1;
    }
    if (best == 0 || L / best > 4096) {
        delete p;
        tt_set_error("block_length %d is not {2,3,5,7}-smooth (or its factors exceed 4096): unsupported", L);
        return TT_ERR_UNSUPPORTED;
    }
    // prefer the larger factor for the column (real) transforms
    p->N2 = best;
    p->N1 = L / best;
    factor_2357(p->N1, &p->spec_n1);
    factor_2357(p->N2, &p->spec_n2);
    factor_2357(M, &p->spec_m);
    p->K1 = p->N1 / 2 + 1;
    p->SP = (L / 2 + 1 + 1) & ~1;

    std::vector<float2> tw;
    int rc;
    make_twiddles(tw, p->N1, -1); if ((rc = upload(&p->d_tw_n1, tw.data(), tw.size()))) return rc;
    make_twiddles(tw, p->N2, -1); if ((rc = upload(&p->d_tw_n2, tw.data(), tw.size()))) return rc;
    make_twiddles(tw, L, -1);     if ((rc = upload(&p->d_tw_L, tw.data(), tw.size()))) return rc;
    make_twiddles(tw, M, +1);     if ((rc = upload(&p->d_tw_m_inv, tw.data(), tw.size()))) return rc;
    make_twiddles(tw, M, -1);     if ((rc = upload(&p->d_tw_m_fwd, tw.data(), tw.size()))) return rc;
    make_twiddles(tw, 32, +1);
    TT_CUDA_CHECK(cudaMemcpyToSymbol(c_tw32, tw.data(), 32 * sizeof(float2)));

    std::vector<float> win(n_taps);
    for (int i = 0; i < n_taps; ++i) win[i] = win_packed[i] / (float)M;     // the 1/M of the analysis ifft
    if ((rc = upload(&p->d_start, start, F))) return rc;
    if ((rc = upload(&p->d_length, length, F))) return rc;
    if ((rc = upload(&p->d_first, first, F))) return rc;
    if ((rc = upload(&p->d_offset, offset, F + 1))) return rc;
    if ((rc = upload(&p->d_win, win.data(), n_taps))) return rc;
    if ((rc = upload(&p->d_dual, dual_packed, n_taps))) return rc;

    const size_t t_bytes = (size_t)p->max_blocks * p->K1 * p->N2 * sizeof(float2);
    const size_t s_bytes = (size_t)p->max_blocks * p->SP * sizeof(float2);
    p->n_lanes = 2;
    for (int i = 0; i < kMaxLanes; ++i) {
        TT_CUDA_CHECK(cudaMalloc((void**)&p->d_T[i], t_bytes));
        TT_CUDA_CHECK(cudaMalloc((void**)&p->d_S[i], s_bytes));
        TT_CUDA_CHECK(cudaStreamCreateWithFlags(&p->lane[i], cudaStreamNonBlocking));
        TT_CUDA_CHECK(cudaEventCreateWithFlags(&p->ev_done[i], cudaEventDisableTiming));
    }
    TT_CUDA_CHECK(cudaEventCreateWithFlags(&p->ev_start, cudaEventDisableTiming));
    p->scratch_bytes = (int64_t)(kMaxLanes * (t_bytes + s_bytes));

    TT_REQUIRE(cols_smem(p) <= 200 * 1024 && rows_smem(p) <= 200 * 1024, "block_length %d needs too much shared memory", L);
    TT_CUDA_CHECK(cudaFuncSetAttribute(cols_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)cols_smem(p)));
    TT_CUDA_CHECK(cudaFuncSetAttribute(cols_inv_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)cols_smem(p)));
    TT_CUDA_CHECK(cudaFuncSetAttribute(rows_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)rows_smem(p)));
    TT_CUDA_CHECK(cudaFuncSetAttribute(rows_inv_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)rows_smem(p)));
    TT_CUDA_CHECK(cudaFuncSetAttribute(bins_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bins_smem()));
    TT_CUDA_CHECK(cudaFuncSetAttribute(bins_inv_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bins_smem()));
    if (M != 1024) {
        const int gs = 3 * M * (int)sizeof(float2);
        TT_CUDA_CHECK(cudaFuncSetAttribute(bins_fwd_generic_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, gs));
        TT_CUDA_CHECK(cudaFuncSetAttribute(bins_inv_generic_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, gs));
    }
    *out = p;
    return TT_OK;
}

extern "C" int tt_cqt_plan_destroy(tt_cqt_plan* p) {
    if (!p) return TT_OK;
    cudaFree(p->d_start); cudaFree(p->d_length); cudaFree(p->d_first); cudaFree(p->d_offset);
    cudaFree(p->d_win); cudaFree(p->d_dual);
    cudaFree(p->d_tw_n1); cudaFree(p->d_tw_n2); cudaFree(p->d_tw_L); cudaFree(p->d_tw_m_inv); cudaFree(p->d_tw_m_fwd);
    for (int i = 0; i < kMaxLanes; ++i) {
        cudaFree(p->d_T[i]); cudaFree(p->d_S[i]);
        if (p->lane[i]) cudaStreamDestroy(p->lane[i]);
        if (p->ev_done[i]) cudaEventDestroy(p->ev_done[i]);
    }
    if (p->ev_start) cudaEventDestroy(p->ev_start);
    delete p;
    return TT_OK;
}

extern "C" int64_t tt_cqt_plan_scratch_bytes(const tt_cqt_plan* p) { return p ? p->scratch_bytes : 0; }

extern "C" int tt_cqt_plan_set_lanes(tt_cqt_plan* p, int n_lanes) {
    TT_REQUIRE(p && n_lanes >= 1 && n_lanes <= kMaxLanes, "lanes must be in [1, %d]", kMaxLanes);
    p->n_lanes = n_lanes;
    return TT_OK;
}

static BinTables bin_tables(const tt_cqt_plan* p) {
    BinTables t;
    t.start = p->d_start; t.length = p->d_length; t.first = p->d_first; t.offset = p->d_offset;
    t.win = p->d_win; t.dual = p->d_dual;
    return t;
}

extern "C" int tt_cqt_forward(tt_cqt_plan* p, const float* audio, int batch, int n_blocks, float* coeffs, void* stream_) {
    TT_REQUIRE(p && audio && coeffs, "null argument");
    TT_REQUIRE(batch >= 0 && n_blocks >= 0, "negative sizes");
    cudaStream_t user = (cudaStream_t)stream_;
    const long long total = (long long)batch * n_blocks;
    const BinTables tab = bin_tables(p);
    if (total == 0) return TT_OK;
    const int n_groups = (int)((total + p->max_blocks - 1) / p->max_blocks);
    const int n_lanes = std::min(n_groups, p->n_lanes);
    TT_CUDA_CHECK(cudaEventRecord(p->ev_start, user));
    for (int i = 0; i < n_lanes; ++i) TT_CUDA_CHECK(cudaStreamWaitEvent(p->lane[i], p->ev_start, 0));
    int g = 0;
    for (long long b0 = 0; b0 < total; b0 += p->max_blocks, ++g) {
        const int nb = (int)std::min<long long>(p->max_blocks, total - b0);
        cudaStream_t stream = p->lane[g % n_lanes];
        float2 *T = p->d_T[g % n_lanes], *S = p->d_S[g % n_lanes];
        dim3 g1((p->N2 + kColsPerCta - 1) / kColsPerCta, nb);
        cols_fwd_kernel<<<g1, kFftThreads, cols_smem(p), stream>>>(audio + (size_t)b0 * p->L, T, p->spec_n1, p->N2,
                                                                    p->K1, p->L, p->d_tw_n1, p->d_tw_L);
        dim3 g2((p->K1 + kRowsPerCta - 1) / kRowsPerCta, nb);
        rows_fwd_kernel<<<g2, kFftThreads, rows_smem(p), stream>>>(T, S, p->spec_n2, p->N1, p->K1, p->L, p->SP, p->d_tw_n2);
        if (p->M == 1024) {
            const long long warps = (long long)nb * p->F;
            const unsigned g3 = (unsigned)((warps + kBinWarps - 1) / kBinWarps);
            bins_fwd_kernel<<<g3, kBinWarps * 32, bins_smem(), stream>>>(S, coeffs, tab, p->F, p->SP, n_blocks, (int)b0, nb,
                                                                          p->d_tw_m_inv);
        } else {
            dim3 g3(p->F, nb);
            bins_fwd_generic_kernel<<<g3, 128, 3 * p->M * sizeof(float2), stream>>>(S, coeffs, tab, p->F, p->SP, n_blocks,
                                                                                     (int)b0, p->spec_m, p->d_tw_m_fwd);
        }
        tt_count_launches(3);
    }
    TT_CUDA_CHECK(cudaGetLastError());
    for (int i = 0; i < n_lanes; ++i) {
        TT_CUDA_CHECK(cudaEventRecord(p->ev_done[i], p->lane[i]));
        TT_CUDA_CHECK(cudaStreamWaitEvent(user, p->ev_done[i], 0));
    }
    return TT_OK;
}

extern "C" int tt_scale_by_peak(float* audio, int64_t n, const float* peak, void* stream_) {
    TT_REQUIRE(audio && peak, "null argument");
    if (n <= 0) return TT_OK;
    cudaStream_t stream = (cudaStream_t)stream_;
    const int grid = (int)std::min<long long>((n + 255) / 256, 148 * 8);
    scale_by_peak_kernel<<<grid, 256, 0, stream>>>(audio, n, peak);
    tt_count_launches(1);
    TT_CUDA_CHECK(cudaGetLastError());
    return TT_OK;
}

// batch uniform items of n_blocks_item blocks (one peak), or the clips of clip_block0 (one peak each); `total` blocks in all
static int cqt_inverse(tt_cqt_plan* p, const float* coeffs, long long total, int n_blocks_item, const int* clip_block0, int n_clips,
                       float* audio, float* peak, cudaStream_t user) {
    const BinTables tab = bin_tables(p);
    TT_CUDA_CHECK(cudaMemsetAsync(peak, 0, (clip_block0 ? n_clips : 1) * sizeof(float), user));
    if (total == 0) return TT_OK;
    const int n_groups = (int)((total + p->max_blocks - 1) / p->max_blocks);
    const int n_lanes = std::min(n_groups, p->n_lanes);
    TT_CUDA_CHECK(cudaEventRecord(p->ev_start, user));
    for (int i = 0; i < n_lanes; ++i) TT_CUDA_CHECK(cudaStreamWaitEvent(p->lane[i], p->ev_start, 0));
    int g = 0;
    for (long long b0 = 0; b0 < total; b0 += p->max_blocks, ++g) {
        const int nb = (int)std::min<long long>(p->max_blocks, total - b0);
        cudaStream_t stream = p->lane[g % n_lanes];
        float2 *T = p->d_T[g % n_lanes], *S = p->d_S[g % n_lanes];
        TT_CUDA_CHECK(cudaMemsetAsync(S, 0, (size_t)nb * p->SP * sizeof(float2), stream));
        if (p->M == 1024) {
            const long long warps = (long long)nb * p->F;
            const unsigned g1 = (unsigned)((warps + kBinWarps - 1) / kBinWarps);
            bins_inv_kernel<<<g1, kBinWarps * 32, bins_smem(), stream>>>(coeffs, S, tab, p->F, p->SP, n_blocks_item, (int)b0, nb,
                                                                          p->d_tw_m_inv, clip_block0, n_clips);
        } else {
            dim3 g1(p->F, nb);
            bins_inv_generic_kernel<<<g1, 128, 3 * p->M * sizeof(float2), stream>>>(coeffs, S, tab, p->F, p->SP, n_blocks_item,
                                                                                     (int)b0, p->spec_m, p->d_tw_m_fwd, clip_block0,
                                                                                     n_clips);
        }
        dim3 g2((p->K1 + kRowsPerCta - 1) / kRowsPerCta, nb);
        rows_inv_kernel<<<g2, kFftThreads, rows_smem(p), stream>>>(S, T, p->spec_n2, p->N1, p->K1, p->L, p->SP, p->d_tw_n2,
                                                                    p->d_tw_L);
        dim3 g3((p->N2 + kColsPerCta - 1) / kColsPerCta, nb);
        cols_inv_kernel<<<g3, kFftThreads, cols_smem(p), stream>>>(T, audio + (size_t)b0 * p->L, p->spec_n1, p->N2, p->K1, p->L,
                                                                    p->d_tw_n1, (unsigned int*)peak, clip_block0, n_clips, (int)b0);
        tt_count_launches(3);
    }
    TT_CUDA_CHECK(cudaGetLastError());
    for (int i = 0; i < n_lanes; ++i) {
        TT_CUDA_CHECK(cudaEventRecord(p->ev_done[i], p->lane[i]));
        TT_CUDA_CHECK(cudaStreamWaitEvent(user, p->ev_done[i], 0));
    }
    return TT_OK;
}

extern "C" int tt_cqt_inverse(tt_cqt_plan* p, const float* coeffs, int batch, int n_blocks, float* audio, float* peak,
                              int normalise, void* stream_) {
    TT_REQUIRE(p && coeffs && audio && peak, "null argument");
    TT_REQUIRE(batch >= 0 && n_blocks >= 0, "negative sizes");
    const long long total = (long long)batch * n_blocks;
    const int rc = cqt_inverse(p, coeffs, total, n_blocks, nullptr, 0, audio, peak, (cudaStream_t)stream_);
    if (rc != TT_OK || total == 0) return rc;
    if (normalise) return tt_scale_by_peak(audio, total * p->L, peak, stream_);
    return TT_OK;
}

extern "C" int tt_scale_by_clip_peak(float* audio, const int* clip_block0, int n_clips, int n_blocks, int block_length,
                                     const float* peaks, void* stream_) {
    TT_REQUIRE(audio && clip_block0 && peaks, "null argument");
    TT_REQUIRE(n_blocks <= 65535, "at most 65535 blocks per call (got %d)", n_blocks);
    if (n_clips <= 0 || n_blocks <= 0 || block_length <= 0) return TT_OK;
    dim3 grid((unsigned)std::min((block_length + 1023) / 1024, 64), n_blocks);
    scale_by_clip_peak_kernel<<<grid, 256, 0, (cudaStream_t)stream_>>>(audio, block_length, clip_block0, n_clips, peaks);
    tt_count_launches(1);
    TT_CUDA_CHECK(cudaGetLastError());
    return TT_OK;
}

extern "C" int tt_cqt_inverse_clips(tt_cqt_plan* p, const float* coeffs, const int* clip_block0, int n_clips, int n_blocks,
                                    float* audio, float* peaks, int normalise, void* stream_) {
    TT_REQUIRE(p && coeffs && clip_block0 && audio && peaks, "null argument");
    TT_REQUIRE(n_clips >= 0 && n_blocks >= 0, "negative sizes");
    if (n_clips == 0) return TT_OK;
    const int rc = cqt_inverse(p, coeffs, n_blocks, 1, clip_block0, n_clips, audio, peaks, (cudaStream_t)stream_);
    if (rc != TT_OK || n_blocks == 0) return rc;
    if (normalise) return tt_scale_by_clip_peak(audio, clip_block0, n_clips, n_blocks, p->L, peaks, stream_);
    return TT_OK;
}

extern "C" int tt_magnitude(const float* coeffs, int64_t n, int apply_tanh, float* out, void* stream_) {
    TT_REQUIRE(coeffs && out, "null argument");
    if (n <= 0) return TT_OK;
    const int grid = (int)std::min<long long>((n + 255) / 256, 148 * 16);
    magnitude_kernel<<<grid, 256, 0, (cudaStream_t)stream_>>>((const float2*)coeffs, n, apply_tanh, out);
    tt_count_launches(1);
    TT_CUDA_CHECK(cudaGetLastError());
    return TT_OK;
}

extern "C" int tt_to_decibels(const float* magnitude, int batch, int64_t per_item, int rescale, float* out,
                              float* item_max, void* stream_) {
    TT_REQUIRE(magnitude && out && item_max, "null argument");
    if (batch <= 0 || per_item <= 0) return TT_OK;
    cudaStream_t stream = (cudaStream_t)stream_;
    TT_CUDA_CHECK(cudaMemsetAsync(item_max, 0, batch * sizeof(float), stream));
    const int gx = (int)std::min<long long>((per_item + 255) / 256, 1024);
    dim3 grid(gx, batch);
    item_max_kernel<<<grid, 256, 0, stream>>>(magnitude, per_item, (unsigned int*)item_max);
    decibels_kernel<<<grid, 256, 0, stream>>>(magnitude, per_item, rescale, out, item_max);
    tt_count_launches(2);
    TT_CUDA_CHECK(cudaGetLastError());
    return TT_OK;
}

extern "C" int tt_chunk_crossfade(const float* chunks, const float* window, int batch, int n_chunks, int n_bins, int frames_per_chunk,
                                  float* coeffs_out, float* act_out, void* stream_) {
    TT_REQUIRE(chunks && window && (coeffs_out || act_out), "null argument");
    TT_REQUIRE(n_chunks >= 2 && frames_per_chunk % 2 == 0, "need at least two chunks and an even chunk length");
    if (batch <= 0 || n_bins <= 0) return TT_OK;
    const long long n_out = (long long)(n_chunks - 1) * (frames_per_chunk / 2);
    dim3 grid((unsigned)std::min<long long>((n_out + 255) / 256, 64), n_bins, batch);
    crossfade_kernel<<<grid, 256, 0, (cudaStream_t)stream_>>>((const float2*)chunks, window, n_chunks, n_bins, frames_per_chunk,
                                                              (float2*)coeffs_out, act_out, nullptr);
    tt_count_launches(1);
    TT_CUDA_CHECK(cudaGetLastError());
    return TT_OK;
}

extern "C" int tt_chunk_crossfade_clips(const float* chunks, const float* window, const int* clip_chunk0, int n_clips,
                                        int max_chunks, int n_bins, int frames_per_chunk, float* coeffs_out, float* act_out,
                                        void* stream_) {
    TT_REQUIRE(chunks && window && clip_chunk0 && (coeffs_out || act_out), "null argument");
    TT_REQUIRE(max_chunks >= 2 && frames_per_chunk % 2 == 0, "need at least two chunks and an even chunk length");
    TT_REQUIRE(n_clips <= 65535, "at most 65535 clips per call (got %d)", n_clips);
    if (n_clips <= 0 || n_bins <= 0) return TT_OK;
    const long long n_out = (long long)(max_chunks - 1) * (frames_per_chunk / 2);
    dim3 grid((unsigned)std::min<long long>((n_out + 255) / 256, 64), n_bins, n_clips);
    crossfade_kernel<<<grid, 256, 0, (cudaStream_t)stream_>>>((const float2*)chunks, window, 0, n_bins, frames_per_chunk,
                                                              (float2*)coeffs_out, act_out, clip_chunk0);
    tt_count_launches(1);
    TT_CUDA_CHECK(cudaGetLastError());
    return TT_OK;
}

extern "C" int tt_gather_chunks(const int64_t* clips, const int* clip_chunk0, int n_clips, int chunk_lo, int n_rows, int block_length,
                                float* out, void* stream_) {
    TT_REQUIRE(clips && clip_chunk0 && out, "null argument");
    TT_REQUIRE(n_rows <= 65535, "at most 65535 chunks per call (got %d)", n_rows);
    if (n_clips <= 0 || n_rows <= 0 || block_length <= 0) return TT_OK;
    dim3 grid((unsigned)std::min((block_length + 2047) / 2048, 64), n_rows);
    gather_chunks_kernel<<<grid, 256, 0, (cudaStream_t)stream_>>>((const longlong2*)clips, clip_chunk0, n_clips, chunk_lo,
                                                                  block_length, out);
    tt_count_launches(1);
    TT_CUDA_CHECK(cudaGetLastError());
    return TT_OK;
}
