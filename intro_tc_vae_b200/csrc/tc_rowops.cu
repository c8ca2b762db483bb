// Row-wise companions of the TC estimator (all HBM-bound, one warp per row, coalesced over D):
//   KL to the unit Gaussian          ops.py:136-163
//   reparameterisation               ops.py:166-185
//   row-wise Gaussian log-density    ops.py:24-29 (+ .sum(dim=1), solvers/tc.py:107,112)
#include "tc_common.cuh"
#include "tc_rowops.h"
#include "tc_instr.h"

namespace tcelbo {

constexpr int kRowWarps = 8;

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

__global__ void kl_fwd_kernel(const float* __restrict__ lv, int64_t ldlv, const float* __restrict__ mu, int64_t ldmu,
                              int b, int d, float* __restrict__ kl_rows) {
    const int row = blockIdx.x * kRowWarps + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (row >= b) return;
    float acc = 0.0f;
    for (int dd = lane; dd < d; dd += 32) {
        const float l = lv[(int64_t)row * ldlv + dd], m = mu[(int64_t)row * ldmu + dd];
        acc += 1.0f + l - expf(l) - m * m;
    }
    acc = warp_sum(acc);
    if (lane == 0) kl_rows[row] = -0.5f * acc;
}

__global__ void kl_bwd_kernel(const float* __restrict__ lv, int64_t ldlv, const float* __restrict__ mu, int64_t ldmu,
                              const float* __restrict__ g_rows, int b, int d,
                              float* __restrict__ glv, int64_t ldglv, float* __restrict__ gmu, int64_t ldgmu) {
    const int64_t n = (int64_t)b * d;
    for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < n; idx += (int64_t)gridDim.x * blockDim.x) {
        const int i = (int)(idx / d), dd = (int)(idx % d);
        const float g = g_rows[i];
        glv[(int64_t)i * ldglv + dd] = g * 0.5f * (expf(lv[(int64_t)i * ldlv + dd]) - 1.0f);
        gmu[(int64_t)i * ldgmu + dd] = g * mu[(int64_t)i * ldmu + dd];
    }
}

__global__ void reparam_fwd_kernel(const float* __restrict__ mu, int64_t ldmu, const float* __restrict__ lv, int64_t ldlv,
                                   const float* __restrict__ eps, int64_t ldeps, int b, int d,
                                   float* __restrict__ z, int64_t ldz) {
    const int64_t n = (int64_t)b * d;
    for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < n; idx += (int64_t)gridDim.x * blockDim.x) {
        const int i = (int)(idx / d), dd = (int)(idx % d);
        z[(int64_t)i * ldz + dd] = reparam_z(mu[(int64_t)i * ldmu + dd], lv[(int64_t)i * ldlv + dd], eps[(int64_t)i * ldeps + dd]);
    }
}

template <bool ACC>     // ACC: add to grad_mu / grad_logvar (they already hold the gradients of the loss terms that read mu, logvar)
__global__ void reparam_bwd_kernel(const float* __restrict__ lv, int64_t ldlv, const float* __restrict__ eps, int64_t ldeps,
                                   const float* __restrict__ gz, int64_t ldgz, int b, int d,
                                   float* __restrict__ gmu, int64_t ldgmu, float* __restrict__ glv, int64_t ldglv) {
    const int64_t n = (int64_t)b * d;
    for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < n; idx += (int64_t)gridDim.x * blockDim.x) {
        const int i = (int)(idx / d), dd = (int)(idx % d);
        const float g = gz[(int64_t)i * ldgz + dd];
        const float std = expf(0.5f * lv[(int64_t)i * ldlv + dd]);
        const float dl = g * eps[(int64_t)i * ldeps + dd] * (0.5f * std);
        if (ACC) { gmu[(int64_t)i * ldgmu + dd] += g; glv[(int64_t)i * ldglv + dd] += dl; }
        else     { gmu[(int64_t)i * ldgmu + dd] = g;  glv[(int64_t)i * ldglv + dd] = dl; }
    }
}

// lp = max(-0.5*((x-mu)^2*exp(-lv) + lv + log2pi), -50) (tc_common.cuh: lp_unfloored); the reference's log 2pi is an fp32
// constant (ops.py:25)
__global__ void rowdensity_fwd_kernel(const float* __restrict__ x, int64_t ldx, const float* __restrict__ mu, int64_t ldmu,
                                      const float* __restrict__ lv, int64_t ldlv, int b, int d, float* __restrict__ out) {
    const int row = blockIdx.x * kRowWarps + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (row >= b) return;
    float acc = 0.0f;
    for (int dd = lane; dd < d; dd += 32) {
        const float xv = x[(int64_t)row * ldx + dd];
        const float m = mu ? mu[(int64_t)row * ldmu + dd] : 0.0f;
        const float l = lv ? lv[(int64_t)row * ldlv + dd] : 0.0f;
        float t, iv;
        acc += lp_clamped(lp_unfloored(xv, m, l, t, iv));
    }
    acc = warp_sum(acc);
    if (lane == 0) out[row] = acc;
}

__global__ void rowdensity_bwd_kernel(const float* __restrict__ x, int64_t ldx, const float* __restrict__ mu, int64_t ldmu,
                                      const float* __restrict__ lv, int64_t ldlv, const float* __restrict__ g_rows, int b, int d,
                                      float* __restrict__ gx, int64_t ldgx, float* __restrict__ gmu, int64_t ldgmu,
                                      float* __restrict__ glv, int64_t ldglv) {
    const int64_t n = (int64_t)b * d;
    for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < n; idx += (int64_t)gridDim.x * blockDim.x) {
        const int i = (int)(idx / d), dd = (int)(idx % d);
        const float xv = x[(int64_t)i * ldx + dd];
        const float m = mu ? mu[(int64_t)i * ldmu + dd] : 0.0f;
        const float l = lv ? lv[(int64_t)i * ldlv + dd] : 0.0f;
        float t, iv;
        const float lp = lp_unfloored(xv, m, l, t, iv);
        const float g = lp_passes_grad(lp) ? g_rows[i] : 0.0f;            // clamp passes gradient where lp >= -50
        if (gx) gx[(int64_t)i * ldgx + dd] = -g * t * iv;
        if (gmu) gmu[(int64_t)i * ldgmu + dd] = g * t * iv;
        if (glv) glv[(int64_t)i * ldglv + dd] = g * 0.5f * (t * t * iv - 1.0f);
    }
}

// ------------------------------------------------------------------------------------------------------
// Per-sample reconstruction loss (ops.py:188-236): sum over the C*H*W pixels of mse / l1 / bce, x detached.
// grid = (chunks, samples); each CTA reduces one chunk of one sample with float4 loads, a second tiny kernel adds
// the chunk partials in a fixed order (deterministic).  kind: 0 = mse, 1 = l1, 2 = bce (log clamped at -100 as in
// torch.nn.functional.binary_cross_entropy).
// ------------------------------------------------------------------------------------------------------
__device__ __forceinline__ float rec_elem(int kind, float x, float r) {
    if (kind == 0) { const float t = r - x; return t * t; }
    if (kind == 1) return fabsf(r - x);
    return -(x * fmaxf(logf(r), -100.0f) + (1.0f - x) * fmaxf(logf(1.0f - r), -100.0f));
}
__device__ __forceinline__ float rec_grad(int kind, float x, float r) {
    if (kind == 0) return 2.0f * (r - x);
    if (kind == 1) return (r > x) ? 1.0f : ((r < x) ? -1.0f : 0.0f);
    const float a = (logf(r) > -100.0f) ? -x / r : 0.0f;
    const float b = (logf(1.0f - r) > -100.0f) ? (1.0f - x) / (1.0f - r) : 0.0f;
    return a + b;
}

__global__ void recloss_partial_kernel(const float* __restrict__ x, const float* __restrict__ r, int64_t n, int kind,
                                       float* __restrict__ partial /*[samples][chunks]*/) {
    __shared__ float sh[8];
    const int chunk = blockIdx.x, nchunk = gridDim.x, i = blockIdx.y;
    const int64_t per = (n + nchunk - 1) / nchunk;
    const int64_t lo = (int64_t)chunk * per, hi = (lo + per < n) ? lo + per : n;
    const float* xs = x + (int64_t)i * n;
    const float* rs = r + (int64_t)i * n;
    float acc = 0.0f;
    for (int64_t k = lo + threadIdx.x; k < hi; k += blockDim.x) acc += rec_elem(kind, xs[k], rs[k]);
    acc = warp_sum(acc);
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        float t = 0.0f;
        for (int w = 0; w < (blockDim.x >> 5); ++w) t += sh[w];
        partial[(int64_t)i * nchunk + chunk] = t;
    }
}

__global__ void recloss_finish_kernel(const float* __restrict__ partial, int b, int nchunk, float* __restrict__ out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= b) return;
    float t = 0.0f;
    for (int c = 0; c < nchunk; ++c) t += partial[(int64_t)i * nchunk + c];
    out[i] = t;
}

__global__ void recloss_bwd_kernel(const float* __restrict__ x, const float* __restrict__ r, const float* __restrict__ g_rows,
                                   int64_t n, int64_t total, int kind, float* __restrict__ gr) {
    for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (int64_t)gridDim.x * blockDim.x)
        gr[idx] = g_rows[idx / n] * rec_grad(kind, x[idx], r[idx]);
}

// Soft-intro exp-ELBO term (solvers/intro.py:102-103): out = mean_i exp(-2*scale*(rec_i + kl_i)); one CTA.
__global__ void expelbo_fwd_kernel(const float* __restrict__ rec, const float* __restrict__ kl, int b, float scale,
                                   float* __restrict__ out, float* __restrict__ e_rows) {
    __shared__ float sh[8];
    float acc = 0.0f;
    for (int i = threadIdx.x; i < b; i += blockDim.x) {
        const float e = expf(-2.0f * scale * (rec[i] + kl[i]));
        e_rows[i] = e;
        acc += e;
    }
    acc = warp_sum(acc);
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        float t = 0.0f;
        for (int w = 0; w < (blockDim.x >> 5); ++w) t += sh[w];
        out[0] = t / (float)b;
    }
}

__global__ void expelbo_bwd_kernel(const float* __restrict__ e_rows, const float* __restrict__ g, int b, float scale,
                                   float* __restrict__ g_rows) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < b) g_rows[i] = g[0] * (-2.0f * scale / (float)b) * e_rows[i];      // same gradient for rec_i and kl_i
}

cudaError_t launch_recloss_fwd(const float* x, const float* r, int b, int64_t n, int kind, float* partial, int nchunk, float* out, cudaStream_t st) {
    { LaunchScope scope(kKernNone, st); recloss_partial_kernel<<<dim3(nchunk, b), 256, 0, st>>>(x, r, n, kind, partial); }
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    { LaunchScope scope(kKernNone, st); recloss_finish_kernel<<<(b + 127) / 128, 128, 0, st>>>(partial, b, nchunk, out); }
    return cudaGetLastError();
}
cudaError_t launch_recloss_bwd(const float* x, const float* r, const float* g_rows, int b, int64_t n, int kind, float* gr, cudaStream_t st) {
    const int64_t total = (int64_t)b * n;
    int64_t g = (total + 255) / 256; if (g > 148 * 16) g = 148 * 16; if (g < 1) g = 1;
    LaunchScope scope(kKernNone, st);
    recloss_bwd_kernel<<<(int)g, 256, 0, st>>>(x, r, g_rows, n, total, kind, gr);
    return cudaGetLastError();
}
cudaError_t launch_expelbo_fwd(const float* rec, const float* kl, int b, float scale, float* out, float* e_rows, cudaStream_t st) {
    LaunchScope scope(kKernNone, st);
    expelbo_fwd_kernel<<<1, 256, 0, st>>>(rec, kl, b, scale, out, e_rows);
    return cudaGetLastError();
}
cudaError_t launch_expelbo_bwd(const float* e_rows, const float* g, int b, float scale, float* g_rows, cudaStream_t st) {
    LaunchScope scope(kKernNone, st);
    expelbo_bwd_kernel<<<(b + 255) / 256, 256, 0, st>>>(e_rows, g, b, scale, g_rows);
    return cudaGetLastError();
}

// MUFU.EX2 saturation probe: 8 independent dependency chains per thread, nothing but ex2 in the loop.
__global__ void __launch_bounds__(256) ex2_peak_kernel(float* __restrict__ out, int iters) {
    float v[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) v[k] = -1.0f - 0.001f * (float)(threadIdx.x + k);
    for (int it = 0; it < iters; ++it) {
#pragma unroll
        for (int k = 0; k < 8; ++k) v[k] = ex2(-v[k]);          // maps (0,1] <-> [0.5,1): stays finite forever
    }
    float acc = 0.0f;
#pragma unroll
    for (int k = 0; k < 8; ++k) acc += v[k];
    if (acc == 12345.678f) out[0] = acc;                          // keep the chains alive without real traffic
}

cudaError_t launch_ex2_peak(float* out, int iters, int ctas, cudaStream_t st) {
    LaunchScope scope(kKernNone, st);
    ex2_peak_kernel<<<ctas, 256, 0, st>>>(out, iters);
    return cudaGetLastError();
}

static inline int grid1d(int64_t n, int block) {
    int64_t g = (n + block - 1) / block;
    if (g > 148 * 16) g = 148 * 16;
    if (g < 1) g = 1;
    return (int)g;
}

cudaError_t launch_kl_fwd(const float* lv, int64_t ldlv, const float* mu, int64_t ldmu, int b, int d, float* kl_rows, cudaStream_t st) {
    LaunchScope scope(kKernNone, st);
    kl_fwd_kernel<<<(b + kRowWarps - 1) / kRowWarps, kRowWarps * 32, 0, st>>>(lv, ldlv, mu, ldmu, b, d, kl_rows);
    return cudaGetLastError();
}
cudaError_t launch_kl_bwd(const float* lv, int64_t ldlv, const float* mu, int64_t ldmu, const float* g_rows, int b, int d,
                          float* glv, int64_t ldglv, float* gmu, int64_t ldgmu, cudaStream_t st) {
    LaunchScope scope(kKernNone, st);
    kl_bwd_kernel<<<grid1d((int64_t)b * d, 256), 256, 0, st>>>(lv, ldlv, mu, ldmu, g_rows, b, d, glv, ldglv, gmu, ldgmu);
    return cudaGetLastError();
}
cudaError_t launch_reparam_fwd(const float* mu, int64_t ldmu, const float* lv, int64_t ldlv, const float* eps, int64_t ldeps,
                               int b, int d, float* z, int64_t ldz, cudaStream_t st) {
    LaunchScope scope(kKernNone, st);
    reparam_fwd_kernel<<<grid1d((int64_t)b * d, 256), 256, 0, st>>>(mu, ldmu, lv, ldlv, eps, ldeps, b, d, z, ldz);
    return cudaGetLastError();
}
cudaError_t launch_reparam_bwd(const float* lv, int64_t ldlv, const float* eps, int64_t ldeps, const float* gz, int64_t ldgz,
                               int b, int d, float* gmu, int64_t ldgmu, float* glv, int64_t ldglv, bool accumulate, cudaStream_t st) {
    LaunchScope scope(kKernNone, st);
    if (accumulate) reparam_bwd_kernel<true><<<grid1d((int64_t)b * d, 256), 256, 0, st>>>(lv, ldlv, eps, ldeps, gz, ldgz, b, d, gmu, ldgmu, glv, ldglv);
    else            reparam_bwd_kernel<false><<<grid1d((int64_t)b * d, 256), 256, 0, st>>>(lv, ldlv, eps, ldeps, gz, ldgz, b, d, gmu, ldgmu, glv, ldglv);
    return cudaGetLastError();
}
cudaError_t launch_rowdensity_fwd(const float* x, int64_t ldx, const float* mu, int64_t ldmu, const float* lv, int64_t ldlv,
                                  int b, int d, float* out, cudaStream_t st) {
    LaunchScope scope(kKernNone, st);
    rowdensity_fwd_kernel<<<(b + kRowWarps - 1) / kRowWarps, kRowWarps * 32, 0, st>>>(x, ldx, mu, ldmu, lv, ldlv, b, d, out);
    return cudaGetLastError();
}
cudaError_t launch_rowdensity_bwd(const float* x, int64_t ldx, const float* mu, int64_t ldmu, const float* lv, int64_t ldlv,
                                  const float* g_rows, int b, int d, float* gx, int64_t ldgx, float* gmu, int64_t ldgmu,
                                  float* glv, int64_t ldglv, cudaStream_t st) {
    LaunchScope scope(kKernNone, st);
    rowdensity_bwd_kernel<<<grid1d((int64_t)b * d, 256), 256, 0, st>>>(x, ldx, mu, ldmu, lv, ldlv, g_rows, b, d,
                                                                        gx, ldgx, gmu, ldgmu, glv, ldglv);
    return cudaGetLastError();
}

}  // namespace tcelbo
