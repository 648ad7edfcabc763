// Training-step building blocks (BASELINE config 5; reference train.py:96-135 runs the same modules in .train() mode and
// lets autograd differentiate them).  fp32 throughout - the reference trains in fp32 - token-major [rows][C] maps.
//
// A training step of the path is a chain of a few op families; each gets one kernel (pair) here and the host side
// (cfpnet_b200/train.py) sequences them in the order of the closed-form backward (DESIGN.md section 8):
//   * tr_gemm            C[M][N] (+)= A . B with arbitrary row / column strides: every pointwise projection forward
//                        (x W^T + b), its input gradient (dy W) and its weight gradient (dy^T x, a reduction over all
//                        rows: split over K across CTAs, fp32 atomics);
//   * tr_colstats        per-channel sums over rows: BatchNorm batch statistics (two passes: mean, then centred sum of
//                        squares - E[x^2] - mean^2 loses the variance of a channel whose mean dominates), bias gradients;
//   * tr_bn_*            train-mode BatchNorm forward (batch statistics, running-stat update with the unbiased variance,
//                        per replica as under nn.DataParallel, train.py:45) and backward (two more channel sums);
//   * tr_ln_*            LayerNorm forward / backward over the channel dim (warp per row);
//   * tr_gelu_*, tr_ew   erf GELU and its derivative, add / ReLU-mask elementwise;
//   * tr_dwconv_wgrad    weight gradient of the k x k depthwise conv (k*k correlations per channel plane).  The input
//                        gradient is the forward depthwise kernel fed with the flipped taps (k_lkpm.cu).
#include "cfp_common.cuh"
#include "cfp_internal.h"

namespace cfp {

// ------------------------------------------------------------------------------------------------ strided GEMM
// 64 x 64 x 16 tiles, 256 threads, 4 x 4 outputs per thread.  The tile loads pick the thread -> element map by which
// index of the operand is contiguous in memory, so both orientations of every operand read coalesced segments.
template <bool A_MC, bool B_NC>
__global__ void __launch_bounds__(256) tr_gemm_kernel(const float* __restrict__ A, int64_t a_rs, int64_t a_cs,
                                                      const float* __restrict__ B, int64_t b_rs, int64_t b_cs,
                                                      float* __restrict__ C, int64_t c_rs, int M, int N, int K, int kchunk,
                                                      const float* __restrict__ bias, int accumulate) {
    __shared__ float As[16][64 + 4], Bs[16][64 + 4];
    const int t = threadIdx.x, tx = t & 15, ty = t >> 4;
    const int m0 = blockIdx.y * 64, n0 = blockIdx.x * 64;
    const int k_begin = blockIdx.z * kchunk, k_end = min(K, k_begin + kchunk);
    float acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
    for (int k0 = k_begin; k0 < k_end; k0 += 16) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            int m, k;
            if (A_MC) { m = t & 63; k = (t >> 6) + 4 * j; } else { k = t & 15; m = (t >> 4) + 16 * j; }
            const int gm = m0 + m, gk = k0 + k;
            As[k][m] = (gm < M && gk < k_end) ? A[(int64_t)gm * a_rs + (int64_t)gk * a_cs] : 0.f;
            int n, kb;
            if (B_NC) { n = t & 63; kb = (t >> 6) + 4 * j; } else { kb = t & 15; n = (t >> 4) + 16 * j; }
            const int gn = n0 + n, gkb = k0 + kb;
            Bs[kb][n] = (gn < N && gkb < k_end) ? B[(int64_t)gkb * b_rs + (int64_t)gn * b_cs] : 0.f;
        }
        __syncthreads();
#pragma unroll
        for (int k = 0; k < 16; ++k) {
            const float4 a = *reinterpret_cast<const float4*>(&As[k][ty * 4]);
            const float4 b = *reinterpret_cast<const float4*>(&Bs[k][tx * 4]);
            const float av[4] = {a.x, a.y, a.z, a.w}, bv[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
        }
        __syncthreads();
    }
    const bool split = gridDim.z > 1;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int gm = m0 + ty * 4 + i;
        if (gm >= M) continue;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int gn = n0 + tx * 4 + j;
            if (gn >= N) continue;
            float v = acc[i][j];
            if (bias && blockIdx.z == 0) v += bias[gn];
            float* dst = C + (int64_t)gm * c_rs + gn;
            if (split) atomicAdd(dst, v);                 // C was zeroed by the launcher (or holds the value to add to)
            else *dst = accumulate ? *dst + v : v;
        }
    }
}

int tr_gemm(const float* A, int64_t a_rs, int64_t a_cs, const float* B, int64_t b_rs, int64_t b_cs, float* C, int64_t c_rs,
            int M, int N, int K, const float* bias, int accumulate, cudaStream_t st) {
    CFP_REQUIRE(M > 0 && N > 0 && K > 0, "tr_gemm: empty problem %dx%dx%d", M, N, K);
    const int tiles = ((M + 63) / 64) * ((N + 63) / 64);
    int ksplit = 1;
    if (tiles < 2 * sm_count() && K >= 1024) {            // few output tiles, long reduction (weight gradients): split K
        ksplit = (4 * sm_count() + tiles - 1) / tiles;
        const int max_split = (K + 255) / 256;
        if (ksplit > max_split) ksplit = max_split;
    }
    int kchunk = ((K + ksplit - 1) / ksplit + 15) / 16 * 16;
    ksplit = (K + kchunk - 1) / kchunk;
    if (ksplit > 1 && !accumulate) {
        cudaError_t e = cudaMemset2DAsync(C, (size_t)c_rs * sizeof(float), 0, (size_t)N * sizeof(float), (size_t)M, st);
        if (e != cudaSuccess) return fail("tr_gemm: cudaMemset2DAsync: %s", cudaGetErrorString(e));
    }
    dim3 grid((N + 63) / 64, (M + 63) / 64, ksplit);
    const bool amc = a_rs == 1 && a_cs != 1, bnc = b_cs == 1;
#define CFP_TR_GEMM(AM, BN) tr_gemm_kernel<AM, BN><<<grid, 256, 0, st>>>(A, a_rs, a_cs, B, b_rs, b_cs, C, c_rs, M, N, K, kchunk, bias, accumulate)
    if (amc && bnc) CFP_TR_GEMM(true, true);
    else if (amc) CFP_TR_GEMM(true, false);
    else if (bnc) CFP_TR_GEMM(false, true);
    else CFP_TR_GEMM(false, false);
#undef CFP_TR_GEMM
    return check_launch("tr_gemm");
}

// ------------------------------------------------------------------------------------------------ channel sums
// s1[c] += sum_r w(r,c) * (x[r][c] - shift[c]),  s2[c] += sum_r w * (x - shift)^2 over this CTA's rows (32 channels x 8 row
// lanes per CTA, rows strided over gridDim.y), fp32 atomics into the (pre-zeroed) outputs.
__global__ void __launch_bounds__(256) tr_colstats_kernel(const float* __restrict__ x, const float* __restrict__ shift,
                                                          float* __restrict__ s1, float* __restrict__ s2, int64_t rows, int C) {
    __shared__ float r1[8][33], r2[8][33];
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    const int c = blockIdx.x * 32 + tx;
    float a1 = 0.f, a2 = 0.f;
    if (c < C) {
        const float sh = shift ? shift[c] : 0.f;
        for (int64_t r = (int64_t)blockIdx.y * 8 + ty; r < rows; r += (int64_t)gridDim.y * 8) {
            const float v = x[r * C + c] - sh;
            a1 += v;
            a2 = fmaf(v, v, a2);
        }
    }
    r1[ty][tx] = a1; r2[ty][tx] = a2;
    __syncthreads();
    if (ty == 0 && c < C) {
#pragma unroll
        for (int i = 1; i < 8; ++i) { a1 += r1[i][tx]; a2 += r2[i][tx]; }
        atomicAdd(s1 + c, a1);
        if (s2) atomicAdd(s2 + c, a2);
    }
}
static int colstats_launch(const float* x, const float* shift, float* s1, float* s2, int64_t rows, int C, cudaStream_t st) {
    const int gx = (C + 31) / 32;
    int64_t gy = (rows + 63) / 64;
    const int64_t cap = (int64_t)(4 * sm_count() + gx - 1) / gx;
    if (gy > cap) gy = cap;
    if (gy < 1) gy = 1;
    tr_colstats_kernel<<<dim3(gx, (unsigned)gy), 256, 0, st>>>(x, shift, s1, s2, rows, C);
    return check_launch("tr_colstats");
}
int tr_colsum(const float* x, float* out, int64_t rows, int C, cudaStream_t st) {
    cudaError_t e = cudaMemsetAsync(out, 0, (size_t)C * sizeof(float), st);
    if (e != cudaSuccess) return fail("tr_colsum: cudaMemsetAsync: %s", cudaGetErrorString(e));
    return colstats_launch(x, nullptr, out, nullptr, rows, C, st);
}

// ------------------------------------------------------------------------------------------------ BatchNorm (train mode)
// phase 0: mean = s1 / n.   phase 1: var = css / n (biased, what normalises the batch), rstd; running statistics with the
// UNBIASED variance (torch.nn.functional.batch_norm), momentum as nn.BatchNorm's (0.1 by default).
__global__ void tr_bn_finalize_kernel(const float* __restrict__ s, float n, float eps, float momentum, float* __restrict__ mean,
                                      float* __restrict__ rstd, float* __restrict__ running_mean, float* __restrict__ running_var,
                                      int C, int phase) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= C) return;
    if (phase == 0) {
        mean[c] = s[c] / n;
    } else {
        const float var = s[c] / n;
        rstd[c] = 1.f / sqrtf(var + eps);         // correctly rounded: a weight in front of a batch-statistics BatchNorm has a
                                                  // gradient of relative size eps / var, an rsqrtf ulp error swamps it
        if (running_mean) running_mean[c] = (1.f - momentum) * running_mean[c] + momentum * mean[c];
        if (running_var) running_var[c] = (1.f - momentum) * running_var[c] + momentum * var * (n > 1.f ? n / (n - 1.f) : 1.f);
    }
}
int tr_bn_stats(const float* x, int64_t rows, int C, float eps, float momentum, float* mean, float* rstd, float* running_mean,
                float* running_var, float* scratch /* [2C] */, cudaStream_t st) {
    CFP_REQUIRE(rows > 0 && C > 0, "tr_bn_stats: empty input");
    cudaError_t e = cudaMemsetAsync(scratch, 0, (size_t)2 * C * sizeof(float), st);
    if (e != cudaSuccess) return fail("tr_bn_stats: cudaMemsetAsync: %s", cudaGetErrorString(e));
    if (int err = colstats_launch(x, nullptr, scratch, nullptr, rows, C, st)) return err;
    tr_bn_finalize_kernel<<<(C + 127) / 128, 128, 0, st>>>(scratch, (float)rows, eps, momentum, mean, rstd, nullptr, nullptr, C, 0);
    if (int err = check_launch("tr_bn_finalize")) return err;
    e = cudaMemsetAsync(scratch, 0, (size_t)2 * C * sizeof(float), st);
    if (e != cudaSuccess) return fail("tr_bn_stats: cudaMemsetAsync: %s", cudaGetErrorString(e));
    if (int err = colstats_launch(x, mean, scratch, scratch + C, rows, C, st)) return err;
    tr_bn_finalize_kernel<<<(C + 127) / 128, 128, 0, st>>>(scratch + C, (float)rows, eps, momentum, mean, rstd, running_mean, running_var, C, 1);
    return check_launch("tr_bn_finalize");
}

// y = (x - mean) * rstd * gamma + beta  [ReLU]
__global__ void __launch_bounds__(256) tr_bn_apply_kernel(const float* __restrict__ x, const float* __restrict__ mean,
                                                          const float* __restrict__ rstd, const float* __restrict__ gamma,
                                                          const float* __restrict__ beta, float* __restrict__ y, int64_t total4, int C,
                                                          int relu) {
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total4; i += (int64_t)gridDim.x * blockDim.x) {
        const int c = (int)((i * 4) % C);
        const float4 v = reinterpret_cast<const float4*>(x)[i];
        const float4 m = *reinterpret_cast<const float4*>(mean + c), r = *reinterpret_cast<const float4*>(rstd + c);
        const float4 g = *reinterpret_cast<const float4*>(gamma + c), b = *reinterpret_cast<const float4*>(beta + c);
        float4 o = make_float4(fmaf((v.x - m.x) * r.x, g.x, b.x), fmaf((v.y - m.y) * r.y, g.y, b.y),
                               fmaf((v.z - m.z) * r.z, g.z, b.z), fmaf((v.w - m.w) * r.w, g.w, b.w));
        if (relu) o = make_float4(fmaxf(o.x, 0.f), fmaxf(o.y, 0.f), fmaxf(o.z, 0.f), fmaxf(o.w, 0.f));
        reinterpret_cast<float4*>(y)[i] = o;
    }
}
static inline unsigned ew_grid(int64_t n) {
    const int64_t want = (n + 255) / 256, cap = (int64_t)sm_count() * 16;
    return (unsigned)(want < cap ? (want > 0 ? want : 1) : cap);
}
int tr_bn_apply(const float* x, const float* mean, const float* rstd, const float* gamma, const float* beta, float* y,
                int64_t rows, int C, int relu, cudaStream_t st) {
    CFP_REQUIRE(C % 4 == 0, "tr_bn_apply: C=%d is not a multiple of 4", C);
    const int64_t total4 = rows * C / 4;
    tr_bn_apply_kernel<<<ew_grid(total4), 256, 0, st>>>(x, mean, rstd, gamma, beta, y, total4, C, relu);
    return check_launch("tr_bn_apply");
}

// backward, pass 1: g = dy * [bn(x) > 0 if relu];  s1[c] = sum g, s2[c] = sum g * xhat   (= dbeta, dgamma)
__global__ void __launch_bounds__(256) tr_bn_bwd_stats_kernel(const float* __restrict__ dy, const float* __restrict__ x,
                                                              const float* __restrict__ mean, const float* __restrict__ rstd,
                                                              const float* __restrict__ gamma, const float* __restrict__ beta,
                                                              float* __restrict__ s1, float* __restrict__ s2, int64_t rows, int C,
                                                              int relu) {
    __shared__ float r1[8][33], r2[8][33];
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    const int c = blockIdx.x * 32 + tx;
    float a1 = 0.f, a2 = 0.f;
    if (c < C) {
        const float m = mean[c], r = rstd[c], g = gamma[c], b = beta[c];
        for (int64_t row = (int64_t)blockIdx.y * 8 + ty; row < rows; row += (int64_t)gridDim.y * 8) {
            const float xh = (x[row * C + c] - m) * r;
            float d = dy[row * C + c];
            if (relu && fmaf(xh, g, b) <= 0.f) d = 0.f;
            a1 += d;
            a2 = fmaf(d, xh, a2);
        }
    }
    r1[ty][tx] = a1; r2[ty][tx] = a2;
    __syncthreads();
    if (ty == 0 && c < C) {
#pragma unroll
        for (int i = 1; i < 8; ++i) { a1 += r1[i][tx]; a2 += r2[i][tx]; }
        atomicAdd(s1 + c, a1);
        atomicAdd(s2 + c, a2);
    }
}
// pass 2: dx = gamma * rstd / n * (n g - s1 - xhat s2)
__global__ void __launch_bounds__(256) tr_bn_bwd_apply_kernel(const float* __restrict__ dy, const float* __restrict__ x,
                                                              const float* __restrict__ mean, const float* __restrict__ rstd,
                                                              const float* __restrict__ gamma, const float* __restrict__ beta,
                                                              const float* __restrict__ s1, const float* __restrict__ s2,
                                                              float* __restrict__ dx, int64_t total, int C, float n, int relu) {
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int c = (int)(i % C);
        const float r = rstd[c], g = gamma[c];
        const float xh = (x[i] - mean[c]) * r;
        float d = dy[i];
        if (relu && fmaf(xh, g, beta[c]) <= 0.f) d = 0.f;
        dx[i] = g * r / n * (n * d - s1[c] - xh * s2[c]);
    }
}
int tr_bn_bwd(const float* dy, const float* x, const float* mean, const float* rstd, const float* gamma, const float* beta,
              float* dx, float* dgamma, float* dbeta, int64_t rows, int C, int relu, cudaStream_t st) {
    cudaError_t e = cudaMemsetAsync(dgamma, 0, (size_t)C * sizeof(float), st);
    if (e == cudaSuccess) e = cudaMemsetAsync(dbeta, 0, (size_t)C * sizeof(float), st);
    if (e != cudaSuccess) return fail("tr_bn_bwd: cudaMemsetAsync: %s", cudaGetErrorString(e));
    const int gx = (C + 31) / 32;
    int64_t gy = (rows + 63) / 64;
    const int64_t cap = (int64_t)(4 * sm_count() + gx - 1) / gx;
    if (gy > cap) gy = cap;
    tr_bn_bwd_stats_kernel<<<dim3(gx, (unsigned)gy), 256, 0, st>>>(dy, x, mean, rstd, gamma, beta, dbeta, dgamma, rows, C, relu);
    if (int err = check_launch("tr_bn_bwd_stats")) return err;
    const int64_t total = rows * C;
    tr_bn_bwd_apply_kernel<<<ew_grid(total), 256, 0, st>>>(dy, x, mean, rstd, gamma, beta, dbeta, dgamma, dx, total, C, (float)rows, relu);
    return check_launch("tr_bn_bwd_apply");
}

// ------------------------------------------------------------------------------------------------ LayerNorm
// Warp per row, C <= 512 (up to 16 channels per lane).
template <int PER>
__global__ void __launch_bounds__(256) tr_ln_fwd_kernel(const float* __restrict__ x, const float* __restrict__ g,
                                                        const float* __restrict__ b, float* __restrict__ y, int64_t rows, int C, float eps) {
    const int lane = threadIdx.x & 31;
    for (int64_t row = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5); row < rows; row += (int64_t)gridDim.x * 8) {
        float v[PER], s = 0.f;
#pragma unroll
        for (int i = 0; i < PER; ++i) { const int c = lane + 32 * i; v[i] = c < C ? x[row * C + c] : 0.f; s += v[i]; }
        const float mean = warp_sum(s) / C;
        float q = 0.f;
#pragma unroll
        for (int i = 0; i < PER; ++i) { const int c = lane + 32 * i; v[i] = c < C ? v[i] - mean : 0.f; q = fmaf(v[i], v[i], q); }
        const float rstd = 1.f / sqrtf(warp_sum(q) / C + eps);
#pragma unroll
        for (int i = 0; i < PER; ++i) { const int c = lane + 32 * i; if (c < C) y[row * C + c] = fmaf(v[i] * rstd, g[c], b[c]); }
    }
}
// dx = rstd * (gy - mean(gy) - xhat * mean(gy * xhat)), gy = dy * g;  dg += dy * xhat, db += dy  (per-warp partial sums
// over the warp's rows, then one atomic per (warp, channel))
template <int PER>
__global__ void __launch_bounds__(256) tr_ln_bwd_kernel(const float* __restrict__ x, const float* __restrict__ g,
                                                        const float* __restrict__ dy, float* __restrict__ dx, float* __restrict__ dg,
                                                        float* __restrict__ db, int64_t rows, int C, float eps) {
    const int lane = threadIdx.x & 31;
    float pg[PER], pb[PER];
#pragma unroll
    for (int i = 0; i < PER; ++i) pg[i] = pb[i] = 0.f;
    for (int64_t row = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5); row < rows; row += (int64_t)gridDim.x * 8) {
        float v[PER], d[PER], s = 0.f;
#pragma unroll
        for (int i = 0; i < PER; ++i) {
            const int c = lane + 32 * i;
            v[i] = c < C ? x[row * C + c] : 0.f;
            d[i] = c < C ? dy[row * C + c] : 0.f;
            s += v[i];
        }
        const float mean = warp_sum(s) / C;
        float q = 0.f;
#pragma unroll
        for (int i = 0; i < PER; ++i) { const int c = lane + 32 * i; v[i] = c < C ? v[i] - mean : 0.f; q = fmaf(v[i], v[i], q); }
        const float rstd = 1.f / sqrtf(warp_sum(q) / C + eps);
        float m1 = 0.f, m2 = 0.f;
#pragma unroll
        for (int i = 0; i < PER; ++i) {
            const int c = lane + 32 * i;
            v[i] *= rstd;                                  // xhat
            pg[i] = fmaf(d[i], v[i], pg[i]);
            pb[i] += d[i];
            d[i] = c < C ? d[i] * g[c] : 0.f;              // gy
            m1 += d[i];
            m2 = fmaf(d[i], v[i], m2);
        }
        m1 = warp_sum(m1) / C;
        m2 = warp_sum(m2) / C;
#pragma unroll
        for (int i = 0; i < PER; ++i) { const int c = lane + 32 * i; if (c < C) dx[row * C + c] = rstd * (d[i] - m1 - v[i] * m2); }
    }
#pragma unroll
    for (int i = 0; i < PER; ++i) {
        const int c = lane + 32 * i;
        if (c < C) { atomicAdd(dg + c, pg[i]); atomicAdd(db + c, pb[i]); }
    }
}
static inline unsigned ln_grid(int64_t rows) {
    const int64_t want = (rows + 7) / 8, cap = (int64_t)sm_count() * 8;
    return (unsigned)(want < cap ? (want > 0 ? want : 1) : cap);
}
int tr_ln_fwd(const float* x, const float* g, const float* b, float* y, int64_t rows, int C, float eps, cudaStream_t st) {
    CFP_REQUIRE(C >= 1 && C <= 512, "tr_ln_fwd: C=%d outside [1, 512]", C);
    if (C <= 32) tr_ln_fwd_kernel<1><<<ln_grid(rows), 256, 0, st>>>(x, g, b, y, rows, C, eps);
    else if (C <= 64) tr_ln_fwd_kernel<2><<<ln_grid(rows), 256, 0, st>>>(x, g, b, y, rows, C, eps);
    else if (C <= 128) tr_ln_fwd_kernel<4><<<ln_grid(rows), 256, 0, st>>>(x, g, b, y, rows, C, eps);
    else tr_ln_fwd_kernel<16><<<ln_grid(rows), 256, 0, st>>>(x, g, b, y, rows, C, eps);
    return check_launch("tr_ln_fwd");
}
int tr_ln_bwd(const float* x, const float* g, const float* dy, float* dx, float* dg, float* db, int64_t rows, int C, float eps,
              cudaStream_t st) {
    CFP_REQUIRE(C >= 1 && C <= 512, "tr_ln_bwd: C=%d outside [1, 512]", C);
    cudaError_t e = cudaMemsetAsync(dg, 0, (size_t)C * sizeof(float), st);
    if (e == cudaSuccess) e = cudaMemsetAsync(db, 0, (size_t)C * sizeof(float), st);
    if (e != cudaSuccess) return fail("tr_ln_bwd: cudaMemsetAsync: %s", cudaGetErrorString(e));
    if (C <= 32) tr_ln_bwd_kernel<1><<<ln_grid(rows), 256, 0, st>>>(x, g, dy, dx, dg, db, rows, C, eps);
    else if (C <= 64) tr_ln_bwd_kernel<2><<<ln_grid(rows), 256, 0, st>>>(x, g, dy, dx, dg, db, rows, C, eps);
    else if (C <= 128) tr_ln_bwd_kernel<4><<<ln_grid(rows), 256, 0, st>>>(x, g, dy, dx, dg, db, rows, C, eps);
    else tr_ln_bwd_kernel<16><<<ln_grid(rows), 256, 0, st>>>(x, g, dy, dx, dg, db, rows, C, eps);
    return check_launch("tr_ln_bwd");
}

// ------------------------------------------------------------------------------------------------ elementwise
// op 0: out = a + b            op 1: out = a * (b > 0)        (ReLU mask)
// op 2: out = gelu_erf(a)      op 3: out = a * gelu_erf'(b)   (convnext.py:33: nn.GELU(), erf form)
// op 4: out = relu(a)          op 5: out = a * elu1'(b) = a * (b > 0 ? 1 : exp(b))
// op 6: out = elu(a) + 1       op 7: out = -a / b             (attention.py:10-11; the normaliser's gradient)
// op 8: out = leaky_relu(a)    op 9: out = a * (b > 0 ? 1 : 0.01)  (nn.LeakyReLU() of decoder.py, slope 0.01)
__global__ void __launch_bounds__(256) tr_ew_kernel(const float* __restrict__ a, const float* __restrict__ b, float* __restrict__ out,
                                                    int64_t n, int op) {
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const float x = a[i];
        float r;
        switch (op) {
            case 0: r = x + b[i]; break;
            case 1: r = b[i] > 0.f ? x : 0.f; break;
            case 2: r = gelu_erf(x); break;
            case 3: {
                const float t = b[i];
                r = x * (0.5f * (1.f + erff(t * 0.70710678118654752440f)) + t * __expf(-0.5f * t * t) * 0.39894228040143267794f);
                break;
            }
            case 4: r = fmaxf(x, 0.f); break;
            case 6: r = x > 0.f ? x + 1.f : expf(x); break;
            case 7: r = -x / b[i]; break;
            case 8: r = x > 0.f ? x : 0.01f * x; break;
            case 9: r = b[i] > 0.f ? x : 0.01f * x; break;
            default: { const float t = b[i]; r = t > 0.f ? x : x * __expf(t); break; }
        }
        out[i] = r;
    }
}
int tr_ew(const float* a, const float* b, float* out, int64_t n, int op, cudaStream_t st) {
    CFP_REQUIRE(op >= 0 && op <= 9, "tr_ew: unknown op %d", op);
    CFP_REQUIRE(b != nullptr || op == 2 || op == 4 || op == 6 || op == 8, "tr_ew: op %d needs a second operand", op);
    if (n == 0) return 0;
    tr_ew_kernel<<<ew_grid(n), 256, 0, st>>>(a, b, out, n, op);
    return check_launch("tr_ew");
}

// ------------------------------------------------------------------------------------------------ depthwise weight gradient
// dw[c][i][j] = sum_{b,y,x} dy[b][y][x][c] * x[b][y+i-p][x+j-p][c]        (DESIGN.md section 8)
// CTA = (16 x 16 pixel tile position, 16 channels), walks over the frames with the 16 x 16 x K x K partial products of its
// 16 channels in registers: thread = (channel, group of taps); a tap row slides along x with the row segment in registers,
// so a pixel costs one shared-memory load per tap row.  One atomic per (CTA, tap, channel) at the end.
template <int K>
__global__ void __launch_bounds__(256) tr_dwconv_wgrad_kernel(const float* __restrict__ x, const float* __restrict__ dy,
                                                              float* __restrict__ dw, int B, int H, int W, int C) {
    constexpr int T = 16, HP = T + K - 1, PAD = (K - 1) / 2, CH = 16, NG = 256 / CH;     // 16 tap groups
    constexpr int ROWS = (K + NG - 1) / NG;                                              // tap rows per thread (2 for K = 31)
    extern __shared__ __align__(16) float sm[];
    float* halo = sm;                     // [HP][HP][CH]
    float* dys = halo + HP * HP * CH;     // [T][T][CH]
    const int c = threadIdx.x & 15, tg = threadIdx.x >> 4;
    const int cgroups = C / CH;
    const int c0 = (blockIdx.z % cgroups) * CH;
    const int y0 = blockIdx.y * T, x0 = blockIdx.x * T;
    float acc[ROWS][K];
#pragma unroll
    for (int r = 0; r < ROWS; ++r)
#pragma unroll
        for (int j = 0; j < K; ++j) acc[r][j] = 0.f;
    for (int b = 0; b < B; ++b) {
        const size_t frame = (size_t)b * H * W;
        __syncthreads();
        for (int i = threadIdx.x; i < HP * HP * (CH / 4); i += 256) {
            const int cell = i / (CH / 4), cc = (i % (CH / 4)) * 4;
            const int y = y0 - PAD + cell / HP, xx = x0 - PAD + cell % HP;
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            if (y >= 0 && y < H && xx >= 0 && xx < W) v = *reinterpret_cast<const float4*>(x + (frame + (size_t)y * W + xx) * C + c0 + cc);
            *reinterpret_cast<float4*>(halo + cell * CH + cc) = v;
        }
        for (int i = threadIdx.x; i < T * T * (CH / 4); i += 256) {
            const int cell = i / (CH / 4), cc = (i % (CH / 4)) * 4;
            const int y = y0 + cell / T, xx = x0 + cell % T;
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            if (y < H && xx < W) v = *reinterpret_cast<const float4*>(dy + (frame + (size_t)y * W + xx) * C + c0 + cc);
            *reinterpret_cast<float4*>(dys + cell * CH + cc) = v;
        }
        __syncthreads();
#pragma unroll
        for (int r = 0; r < ROWS; ++r) {
            const int ti = tg + NG * r;                                      // tap row of this thread
            if (ti >= K) continue;
#pragma unroll 1
            for (int py = 0; py < T; ++py) {
                // x segment [px + j], j < K, kept in registers while px slides over the 16 pixels of the row
                float seg[K + T - 1];
                const float* hrow = halo + ((py + ti) * HP) * CH + c;
#pragma unroll
                for (int i = 0; i < K + T - 1; ++i) seg[i] = hrow[i * CH];
#pragma unroll
                for (int px = 0; px < T; ++px) {
                    const float d = dys[(py * T + px) * CH + c];
#pragma unroll
                    for (int j = 0; j < K; ++j) acc[r][j] = fmaf(d, seg[px + j], acc[r][j]);
                }
            }
        }
    }
#pragma unroll
    for (int r = 0; r < ROWS; ++r) {
        const int ti = tg + NG * r;
        if (ti >= K) continue;
#pragma unroll
        for (int j = 0; j < K; ++j) atomicAdd(dw + ((size_t)(c0 + c) * K + ti) * K + j, acc[r][j]);
    }
}
template <int K>
static int dwconv_wgrad_launch(const float* x, const float* dy, float* dw, int B, int H, int W, int C, cudaStream_t st) {
    constexpr int T = 16, HP = T + K - 1;
    const size_t smem = (size_t)(HP * HP * 16 + T * T * 16) * sizeof(float);
    auto k = tr_dwconv_wgrad_kernel<K>;
    if (int e = set_smem(k, smem)) return e;
    cudaError_t e = cudaMemsetAsync(dw, 0, (size_t)C * K * K * sizeof(float), st);
    if (e != cudaSuccess) return fail("tr_dwconv_wgrad: cudaMemsetAsync: %s", cudaGetErrorString(e));
    dim3 grid((W + T - 1) / T, (H + T - 1) / T, C / 16);
    k<<<grid, 256, smem, st>>>(x, dy, dw, B, H, W, C);
    return check_launch(K == 31 ? "tr_dwconv_wgrad<31>" : K == 15 ? "tr_dwconv_wgrad<15>" : "tr_dwconv_wgrad<7>");
}
int tr_dwconv_wgrad(const float* x, const float* dy, float* dw, int B, int H, int W, int C, int K, cudaStream_t st) {
    CFP_REQUIRE(C % 16 == 0, "tr_dwconv_wgrad: C=%d is not a multiple of 16", C);
    if (K == 7) return dwconv_wgrad_launch<7>(x, dy, dw, B, H, W, C, st);
    if (K == 15) return dwconv_wgrad_launch<15>(x, dy, dw, B, H, W, C, st);
    if (K == 31) return dwconv_wgrad_launch<31>(x, dy, dw, B, H, W, C, st);
    return fail("tr_dwconv_wgrad: unsupported kernel size %d (decoder.py:92-94 uses 7 / 15 / 31)", K);
}

// ------------------------------------------------------------------------------------------------ optimizer step
// The reference's step after loss.backward() (train.py:124-129): clip_grad_norm_(parameters, 0.1) then AdamW.  Gradients
// and parameters live in flat fp32 buffers (cfpnet_b200/train.py: FlatTrainer - the gradient bucket the NCCL all-reduce ran
// on), so the step is two launches: sum of squares of the whole bucket, then one elementwise update that reads the clip
// coefficient from device memory (no host synchronisation anywhere in the step).
// Deterministic (replicas must stay bit-identical: every rank derives its clip coefficient from this number): each CTA
// writes the partial sum of its fixed slice to out[1 + blockIdx.x], the last CTA to finish (ticket in out[1 + kSumsqParts],
// re-armed for the next call) adds the partials in index order.
constexpr int kSumsqParts = 1024;
__global__ void __launch_bounds__(256) tr_sumsq_kernel(const float* __restrict__ x, int64_t n, float scale, float* __restrict__ out) {
    float a = 0.f;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const float v = x[i] * scale;
        a = fmaf(v, v, a);
    }
    __shared__ float part[8];
    __shared__ bool last;
    a = warp_sum(a);
    if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = a;
    __syncthreads();
    if (threadIdx.x == 0) {
        float t = 0.f;
#pragma unroll
        for (int i = 0; i < 8; ++i) t += part[i];
        out[1 + blockIdx.x] = t;
        __threadfence();
        unsigned* ticket = reinterpret_cast<unsigned*>(out + 1 + kSumsqParts);
        last = atomicAdd(ticket, 1u) == gridDim.x - 1;
    }
    __syncthreads();
    if (!last) return;
    __threadfence();
    float t = 0.f;
    for (int i = threadIdx.x; i < (int)gridDim.x; i += 256) t += __ldcg(out + 1 + i);      // fixed assignment, fixed order
    t = warp_sum(t);
    if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = t;
    __syncthreads();
    if (threadIdx.x == 0) {
        float r = 0.f;
#pragma unroll
        for (int i = 0; i < 8; ++i) r += part[i];
        out[0] = r;
        *reinterpret_cast<unsigned*>(out + 1 + kSumsqParts) = 0u;
    }
}
int tr_sumsq(const float* x, int64_t n, float scale, float* out, cudaStream_t st) {
    if (n == 0) {
        cudaError_t e = cudaMemsetAsync(out, 0, sizeof(float), st);
        return e == cudaSuccess ? 0 : fail("tr_sumsq: cudaMemsetAsync: %s", cudaGetErrorString(e));
    }
    unsigned grid = ew_grid(n);
    if (grid > (unsigned)kSumsqParts) grid = kSumsqParts;
    tr_sumsq_kernel<<<grid, 256, 0, st>>>(x, n, scale, out);
    return check_launch("tr_sumsq");
}
// torch.optim.AdamW (decoupled weight decay, bias-corrected moments, eps added to sqrt(v_hat)); grad = g * grad_scale (the
// 1 / world of the gradient average) * min(1, max_norm / (||grad|| + 1e-6)) - torch.nn.utils.clip_grad_norm_'s coefficient.
// seg_lr: per-segment learning rates (the reference's 1x / 10x parameter groups, train.py:75-76): element i belongs to the
// segment s with seg_end[s-1] <= i < seg_end[s].
__global__ void __launch_bounds__(256) tr_adamw_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                                                       float* __restrict__ v, int64_t n, const int64_t* __restrict__ seg_end,
                                                       const float* __restrict__ seg_lr, int nseg, float beta1, float beta2,
                                                       float eps, float wd, float bc1, float bc2, float grad_scale,
                                                       const float* __restrict__ sumsq, float max_norm) {
    float coef = grad_scale;
    if (max_norm > 0.f) {
        const float c = max_norm / (sqrtf(*sumsq) + 1e-6f);
        coef *= c < 1.f ? c : 1.f;
    }
    int s = 0;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        while (s + 1 < nseg && i >= seg_end[s]) ++s;               // i only grows: the segment pointer never moves back
        const float lr = seg_lr[s];
        const float gi = g[i] * coef;
        const float mi = beta1 * m[i] + (1.f - beta1) * gi;
        const float vi = beta2 * v[i] + (1.f - beta2) * gi * gi;
        m[i] = mi;
        v[i] = vi;
        const float denom = sqrtf(vi) / sqrtf(bc2) + eps;
        p[i] = p[i] * (1.f - lr * wd) - (lr / bc1) * (mi / denom);
    }
}
int tr_adamw(float* p, const float* g, float* m, float* v, int64_t n, const int64_t* seg_end, const float* seg_lr, int nseg,
             float beta1, float beta2, float eps, float wd, int step, float grad_scale, const float* sumsq, float max_norm,
             cudaStream_t st) {
    CFP_REQUIRE(step >= 1 && nseg >= 1, "tr_adamw: step %d / %d segments", step, nseg);
    CFP_REQUIRE(max_norm <= 0.f || sumsq != nullptr, "tr_adamw: clipping needs the gradient sum of squares");
    if (n == 0) return 0;
    const float bc1 = 1.f - powf(beta1, (float)step), bc2 = 1.f - powf(beta2, (float)step);
    tr_adamw_kernel<<<ew_grid(n), 256, 0, st>>>(p, g, m, v, n, seg_end, seg_lr, nseg, beta1, beta2, eps, wd, bc1, bc2, grad_scale,
                                                sumsq, max_norm);
    return check_launch("tr_adamw");
}

}  // namespace cfp
