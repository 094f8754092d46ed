// Backward half of the loss step (reference: experiments/train.py:470-496 = autograd through timbre_trap/framework/modules.py
// and objectives.py, clip_grad_norm_, AdamW): the gradients of the losses with respect to their inputs, and clip + AdamW over the
// flat parameter / gradient buckets.  The layers' weight gradients are in wgrad_tc.cu; their data gradients run through the
// forward kernels (framework/train.py).
#include <math.h>

#include <algorithm>

#include "../../include/timbre_trap_b200.h"
#include "tt_common.cuh"

namespace tt {

// objectives.py:11-33 backward: loss = scale * sum (a-b)^2 ;  ga = gout * 2 scale (a-b),  gb = -ga  (either may be null)
__global__ void sq_diff_bwd_kernel(const float* __restrict__ a, const float* __restrict__ b, const float* __restrict__ gout, float scale,
                                   float* __restrict__ ga, float* __restrict__ gb, long long n) {
    const float s = 2.f * scale * gout[0];
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const float d = s * (a[i] - b[i]);
        if (ga) ga[i] = d;
        if (gb) gb[i] = -d;
    }
}

// objectives.py:36-74 backward w.r.t. the estimate (B, F, T) and / or the target (either output may be null); one thread per frame.
// With the positive-class weight S = neg / (pos + eps) (neg = sum_f (1 - t_f), pos = sum_f t_f) on the bins whose target is 1, the
// target also moves S:  dL/dt_k = -dL/de_k + gout / (B T) * dS/dt_k * sum_{f: t_f = 1} (e_f - t_f)^2,  dS/dt_k = -(neg + pos + eps) / (pos + eps)^2
// (no such term where S = 0, which the forward replaces by 1).
__global__ void transcription_bwd_kernel(const float* __restrict__ est, const float* __restrict__ tgt, const float* __restrict__ gout,
                                         int B, int F, int T, int weighted, float* __restrict__ gest, float* __restrict__ gtgt) {
    const long long frames = (long long)B * T;
    const float s = 2.f * gout[0] / (float)frames;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < frames; i += (long long)gridDim.x * blockDim.x) {
        const long long b = i / T, t = i - b * T;
        const float* e = est + (size_t)b * F * T + t;
        const float* gt = tgt + (size_t)b * F * T + t;
        float scale = 1.f, pos = 0.f;
        if (weighted) {
            for (int f = 0; f < F; ++f) pos += gt[(size_t)f * T];
            scale = ((float)F - pos) / (pos + 1.1920928955078125e-07f);
            if (scale == 0.f) scale = 1.f;
        }
        if (gest) {
            float* ge = gest + (size_t)b * F * T + t;
            for (int f = 0; f < F; ++f) {
                const float gv = gt[(size_t)f * T];
                ge[(size_t)f * T] = s * (gv == 1.f ? scale : 1.f) * (e[(size_t)f * T] - gv);
            }
        }
        if (gtgt) {
            float dscale = 0.f;                       // dL/dS * dS/dt_k, the same for every bin of the frame
            if (weighted && (float)F - pos != 0.f) {
                float q = 0.f;
                for (int f = 0; f < F; ++f) {
                    const float gv = gt[(size_t)f * T];
                    if (gv == 1.f) {
                        const float d = e[(size_t)f * T] - gv;
                        q += d * d;
                    }
                }
                const float den = pos + 1.1920928955078125e-07f;
                dscale = -0.5f * s * q * ((float)F + 1.1920928955078125e-07f) / (den * den);
            }
            float* gg = gtgt + (size_t)b * F * T + t;
            for (int f = 0; f < F; ++f) {
                const float gv = gt[(size_t)f * T];
                gg[(size_t)f * T] = dscale - s * (gv == 1.f ? scale : 1.f) * (e[(size_t)f * T] - gv);
            }
        }
    }
}

// activations = tanh(|c|) backward (modules.py:271-289): dc = dact * (1 - act^2) * c / |c|   (0 where |c| = 0)
__global__ void activations_bwd_kernel(const float2* __restrict__ c, const float* __restrict__ dact, float2* __restrict__ dc, long long n) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const float2 v = c[i];
        const float m = sqrtf(v.x * v.x + v.y * v.y);
        const float a = tanhf(m);
        const float k = m > 0.f ? dact[i] * (1.f - a * a) / m : 0.f;
        dc[i] = make_float2(k * v.x, k * v.y);
    }
}

// TimbreTrapFiLM's Decoder.convin (modules.py:801-809, 838-840): y = ConvTranspose2d(W (D, C0, H0, 1), b)(u), u = gamma * z + beta per
// latent channel, gamma = film_layer.gamma(cond), beta = film_layer.beta(cond), cond one-hot with its 1 in column `hot`.  From the
// tensor-core sums G[d,c,h] = sum_{b,t} dz[c,h,t] z[d,t] and rows[c,h] = sum_{b,t} dz[c,h,t] (tt_conv_wgrad_lat):
//   dW[d] = gamma[d] G[d] + beta[d] rows,  db[c] = sum_h rows[c,h],  dgamma[d] = <W[d], G[d]>,  dbeta[d] = <W[d], rows>,
// and the nn.Linear gradients: weight (D, 2) = dgamma (dbeta) in column `hot`, 0 in the other; bias = dgamma (dbeta).
// One CTA per latent channel, fixed-order reductions (bit-reproducible).
__global__ void __launch_bounds__(256) film_convin_grad_kernel(const float* __restrict__ G, const float* __restrict__ rows,
                                                               const float* __restrict__ w, const float* __restrict__ gamma_w,
                                                               const float* __restrict__ gamma_b, const float* __restrict__ beta_w,
                                                               const float* __restrict__ beta_b, int C0, int H0, int hot,
                                                               float* __restrict__ dw, float* __restrict__ db, float* __restrict__ dgamma_w,
                                                               float* __restrict__ dgamma_b, float* __restrict__ dbeta_w,
                                                               float* __restrict__ dbeta_b) {
    const int d = blockIdx.x;
    const int n = C0 * H0;
    const float gamma = gamma_w[2 * d + hot] + gamma_b[d];         // F.linear(one-hot cond): the forward's fold reads the same value
    const float beta = beta_w[2 * d + hot] + beta_b[d];
    const float* Gd = G + (size_t)d * n;
    const float* Wd = w + (size_t)d * n;
    float* dWd = dw + (size_t)d * n;
    float sg = 0.f, sb = 0.f;
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        const float g = Gd[i], r = rows[i], wi = Wd[i];
        dWd[i] = fmaf(gamma, g, beta * r);
        sg = fmaf(wi, g, sg);
        sb = fmaf(wi, r, sb);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        sg += __shfl_xor_sync(0xffffffffu, sg, o);
        sb += __shfl_xor_sync(0xffffffffu, sb, o);
    }
    __shared__ float red[2][8];
    if ((threadIdx.x & 31) == 0) {
        red[0][threadIdx.x >> 5] = sg;
        red[1][threadIdx.x >> 5] = sb;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        float a = 0.f, b = 0.f;
        for (int k = 0; k < (int)(blockDim.x >> 5); ++k) {
            a += red[0][k];
            b += red[1][k];
        }
        dgamma_w[2 * d + hot] = a;
        dgamma_w[2 * d + 1 - hot] = 0.f;
        dgamma_b[d] = a;
        dbeta_w[2 * d + hot] = b;
        dbeta_w[2 * d + 1 - hot] = 0.f;
        dbeta_b[d] = b;
    }
    for (int c = blockIdx.x * blockDim.x + threadIdx.x; c < C0; c += gridDim.x * blockDim.x) {
        float s = 0.f;
        for (int h = 0; h < H0; ++h) s += rows[(size_t)c * H0 + h];
        db[c] = s;
    }
}

// sum of squares of one gradient tensor into a double accumulator (for clip_grad_norm_, train.py:493)
__global__ void sumsq_kernel(const float* __restrict__ g, long long n, double* __restrict__ acc) {
    __shared__ double red[8];
    double s = 0.0;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) s += (double)g[i] * g[i];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int i = 1; i < 8; ++i) s += red[i];
        atomicAdd(acc, s);
    }
}

// AdamW step with the clip factor applied on the fly (torch.optim.AdamW defaults, train.py:334,496):
//   g *= min(1, max_norm / (||g|| + 1e-6));  p *= 1 - lr*wd;  m = b1 m + (1-b1) g;  v = b2 v + (1-b2) g^2;
//   p -= lr * (m / (1 - b1^t)) / (sqrt(v / (1 - b2^t)) + eps)
__global__ void adamw_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m, float* __restrict__ v, long long n,
                             const double* __restrict__ sumsq, float max_norm, float lr, float b1, float b2, float eps, float wd,
                             float bc1, float bc2) {
    const float norm = (float)sqrt(*sumsq);
    const float clip = fminf(1.f, max_norm / (norm + 1e-6f));
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const float gi = g[i] * clip;
        float pi = p[i] * (1.f - lr * wd);
        const float mi = b1 * m[i] + (1.f - b1) * gi;
        const float vi = b2 * v[i] + (1.f - b2) * gi * gi;
        m[i] = mi;
        v[i] = vi;
        pi -= lr * (mi / bc1) / (sqrtf(vi / bc2) + eps);
        p[i] = pi;
    }
}

static inline int grid_for(long long n) { return (int)std::max<long long>(1, std::min<long long>((n + 255) / 256, 148 * 16)); }

}  // namespace tt

using namespace tt;

extern "C" int tt_sum_sq_diff_bwd(const float* a, const float* b, const float* gout, double scale, float* ga, float* gb, int64_t n,
                                  void* stream) {
    TT_REQUIRE(a && b && gout && (ga || gb), "null argument");
    if (n <= 0) return TT_OK;
    sq_diff_bwd_kernel<<<grid_for(n), 256, 0, (cudaStream_t)stream>>>(a, b, gout, (float)scale, ga, gb, n);
    TT_CUDA_CHECK(cudaGetLastError());
    tt_count_launches(1);
    return TT_OK;
}

extern "C" int tt_transcription_loss_bwd(const float* estimate, const float* target, const float* gout, int B, int F, int T,
                                         int weight_positive_class, float* gest, float* gtarget, void* stream) {
    TT_REQUIRE(estimate && target && gout && (gest || gtarget), "null argument");
    const long long frames = (long long)B * T;
    if (frames <= 0) return TT_OK;
    transcription_bwd_kernel<<<grid_for(frames), 256, 0, (cudaStream_t)stream>>>(estimate, target, gout, B, F, T, weight_positive_class, gest,
                                                                                  gtarget);
    TT_CUDA_CHECK(cudaGetLastError());
    tt_count_launches(1);
    return TT_OK;
}

extern "C" int tt_activations_bwd(const float* coeffs, const float* dact, float* dcoeffs, int64_t n, void* stream) {
    TT_REQUIRE(coeffs && dact && dcoeffs, "null argument");
    if (n <= 0) return TT_OK;
    activations_bwd_kernel<<<grid_for(n), 256, 0, (cudaStream_t)stream>>>((const float2*)coeffs, dact, (float2*)dcoeffs, n);
    TT_CUDA_CHECK(cudaGetLastError());
    tt_count_launches(1);
    return TT_OK;
}

extern "C" int tt_film_convin_grad(const float* G, const float* rows, const float* w, const float* gamma_w, const float* gamma_b,
                                   const float* beta_w, const float* beta_b, int D, int C0, int H0, int hot, float* dw, float* db,
                                   float* dgamma_w, float* dgamma_b, float* dbeta_w, float* dbeta_b, void* stream) {
    TT_REQUIRE(G && rows && w && gamma_w && gamma_b && beta_w && beta_b && dw && db && dgamma_w && dgamma_b && dbeta_w && dbeta_b,
               "null argument");
    TT_REQUIRE(D > 0 && C0 > 0 && H0 > 0, "film_convin_grad: bad shape D %d C0 %d H0 %d", D, C0, H0);
    TT_REQUIRE(hot == 0 || hot == 1, "film_convin_grad: hot must be 0 (transcribe) or 1 (reconstruct)");
    film_convin_grad_kernel<<<D, 256, 0, (cudaStream_t)stream>>>(G, rows, w, gamma_w, gamma_b, beta_w, beta_b, C0, H0, hot, dw, db, dgamma_w,
                                                                dgamma_b, dbeta_w, dbeta_b);
    TT_CUDA_CHECK(cudaGetLastError());
    tt_count_launches(1);
    return TT_OK;
}

extern "C" int tt_grad_sumsq(const float* g, int64_t n, double* acc, void* stream) {
    TT_REQUIRE(g && acc, "null argument");
    if (n <= 0) return TT_OK;
    sumsq_kernel<<<grid_for(n), 256, 0, (cudaStream_t)stream>>>(g, n, acc);
    TT_CUDA_CHECK(cudaGetLastError());
    tt_count_launches(1);
    return TT_OK;
}

extern "C" int tt_adamw_step(float* p, const float* g, float* m, float* v, int64_t n, const double* sumsq, float max_norm, float lr,
                             float beta1, float beta2, float eps, float weight_decay, int step, void* stream) {
    TT_REQUIRE(p && g && m && v && sumsq && step >= 1, "bad argument");
    if (n <= 0) return TT_OK;
    const float bc1 = 1.f - powf(beta1, (float)step), bc2 = 1.f - powf(beta2, (float)step);
    adamw_kernel<<<grid_for(n), 256, 0, (cudaStream_t)stream>>>(p, g, m, v, n, sumsq, max_norm, lr, beta1, beta2, eps, weight_decay, bc1, bc2);
    TT_CUDA_CHECK(cudaGetLastError());
    tt_count_launches(1);
    return TT_OK;
}
