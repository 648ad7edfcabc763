// Decoder shell and adaptive-bins head in train mode: the adjoints no forward kernel already computes (SURVEY.md section 8
// f1 / f2, config 5).  fp32 FFMA with fp32 accumulation, no atomics: every output is summed in one fixed order, so two
// launches give the same bits.  The forward convs and the conv input gradients run on conv_f32 (k_dec_f32.cu).
//
//   conv_wgrad_f32         dW[tap][ci][co] = sum_{b,p} x[b][p + off(tap)][ci] dy[b][p][co] as an implicit GEMM (no im2col):
//                          a CTA owns a 64 (ci) x 64 (co) tile of one tap and a contiguous range of the B*H*W pixels; each
//                          pixel range writes its own partial, a second pass adds the partials in range order.
//   upsample_concat_bwd_f32  adjoint of upsample_concat_f32: every low-resolution pixel gathers the high-resolution pixels
//                          whose source coordinate lies within one pixel of it (weights from the forward's float arithmetic);
//                          the skip slice is transposed back to NCHW.
//   head_expect_bwd_f32    dlogit = p (c - pred) dpred channels-last (c - pred taken relative to the pixel's most probable
//                          bin), and per-tile partials of sum_pixels p dpred (the centres' gradient), added in tile order.
//   head_bins_bwd_f32      one CTA per frame: cotangents of the bin edges / centres back through the cumsum, the min_val
//                          pad, the normalisation and relu + 0.1 to the regressor's pre-ReLU output.
#include "cfp_common.cuh"
#include "cfp_internal.h"

namespace cfp {

static unsigned grid_cap(int64_t total) {
    const int64_t want = (total + 255) / 256, cap = (int64_t)sm_count() * 16;
    return (unsigned)(want < cap ? want : cap);
}

// ------------------------------------------------------------------------------------------------ conv weight gradient
namespace wg {
constexpr int BM = 64, BN = 64, BK = 32, LD = 68;      // ci x co tile, pixels per step, smem row pitch
constexpr int kTargetCtas = 1184;                      // 8 per SM of a 148-SM B200; a constant, so the split (and the
                                                       // summation order) does not depend on the device
constexpr int kMinPixels = 512;                        // least pixels per split

struct Plan {
    int splits;
    int64_t kchunk;
};
inline Plan plan(int64_t K, int cin, int cout, int taps) {
    const int64_t tiles = (int64_t)((cin + BM - 1) / BM) * ((cout + BN - 1) / BN) * taps;
    int64_t s = (kTargetCtas + tiles - 1) / tiles;
    const int64_t smax = (K + kMinPixels - 1) / kMinPixels;
    if (s > smax) s = smax;
    if (s < 1) s = 1;
    int64_t kchunk = ((K + s - 1) / s + BK - 1) / BK * BK;
    return {(int)((K + kchunk - 1) / kchunk), kchunk};
}
}  // namespace wg

size_t conv_wgrad_scratch_floats(int B, int H, int W, int cin, int cout, int taps) {
    if (B <= 0 || H <= 0 || W <= 0 || cin <= 0 || cout <= 0 || (taps != 1 && taps != 9)) return 0;
    const wg::Plan p = wg::plan((int64_t)B * H * W, cin, cout, taps);
    return p.splits > 1 ? (size_t)p.splits * taps * cin * cout : 0;
}

// Thread t: loads pixel rows (t / 16) and (t / 16 + 16) of the step, float4 group t % 16 of the tile's 64 channels, for
// both operands; computes ci rows 4 (t / 16) .. +4 and co columns 4 (t % 16) .. +4 of the tile.
__global__ void __launch_bounds__(256) conv_wgrad_f32_kernel(const float* __restrict__ x, const float* __restrict__ dy,
                                                             float* __restrict__ out, int H, int W, int cin, int cout, int k,
                                                             int64_t K, int64_t kchunk) {
    using namespace wg;
    __shared__ __align__(16) float As[BK][LD], Bs[BK][LD];
    const int taps = k * k, t = threadIdx.x, g = t & 15, r = t >> 4;
    const int tap = blockIdx.y % taps, ci0 = (blockIdx.y / taps) * BM, co0 = blockIdx.x * BN;
    const int oy = tap / k - k / 2, ox = tap % k - k / 2;
    const int64_t p_begin = blockIdx.z * kchunk, p_end = min(K, p_begin + kchunk);
    const int64_t HW = (int64_t)H * W;
    const int ci = ci0 + 4 * g, co = co0 + 4 * g;
    const float4 zero = make_float4(0.f, 0.f, 0.f, 0.f);

    float4 ra[2], rb[2];
    auto load = [&](int64_t p0) {
#pragma unroll
        for (int j = 0; j < 2; ++j) {
            const int64_t p = p0 + r + 16 * j;
            ra[j] = rb[j] = zero;
            if (p < p_end) {
                const int64_t b = p / HW;
                const int rem = (int)(p - b * HW), y = rem / W + oy, xx = rem % W + ox;
                if (ci < cin && y >= 0 && y < H && xx >= 0 && xx < W)
                    ra[j] = *reinterpret_cast<const float4*>(x + ((b * H + y) * W + xx) * cin + ci);
                if (co < cout) rb[j] = *reinterpret_cast<const float4*>(dy + p * cout + co);
            }
        }
    };

    float acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i) acc[i][0] = acc[i][1] = acc[i][2] = acc[i][3] = 0.f;
    const int ty = r, tx = g;
    load(p_begin);
#pragma unroll 1
    for (int64_t p0 = p_begin; p0 < p_end; p0 += BK) {
#pragma unroll
        for (int j = 0; j < 2; ++j) {
            *reinterpret_cast<float4*>(&As[r + 16 * j][4 * g]) = ra[j];
            *reinterpret_cast<float4*>(&Bs[r + 16 * j][4 * g]) = rb[j];
        }
        __syncthreads();
        if (p0 + BK < p_end) load(p0 + BK);              // next step's operands in flight during this step's FFMAs
#pragma unroll
        for (int kk = 0; kk < BK; ++kk) {
            const float4 a = *reinterpret_cast<const float4*>(&As[kk][4 * ty]);
            const float4 b = *reinterpret_cast<const float4*>(&Bs[kk][4 * tx]);
            const float av[4] = {a.x, a.y, a.z, a.w}, bv[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int jj = 0; jj < 4; ++jj) acc[i][jj] = fmaf(av[i], bv[jj], acc[i][jj]);
        }
        __syncthreads();
    }
    const int cc = co0 + 4 * tx;
    if (cc >= cout) return;
    float* dst = out + ((size_t)blockIdx.z * taps + tap) * cin * cout;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int c = ci0 + 4 * ty + i;
        if (c < cin) *reinterpret_cast<float4*>(dst + (size_t)c * cout + cc) = make_float4(acc[i][0], acc[i][1], acc[i][2], acc[i][3]);
    }
}

// out[i] = sum_s part[s][i], s ascending
__global__ void __launch_bounds__(256) sum_partials_kernel(const float* __restrict__ part, float* __restrict__ out, int64_t n,
                                                           int splits) {
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        float s = 0.f;
        for (int j = 0; j < splits; ++j) s += part[(size_t)j * n + i];
        out[i] = s;
    }
}

int conv_wgrad_f32(const float* x, const float* dy, float* dw, float* scratch, int B, int H, int W, int cin, int cout, int taps,
                   cudaStream_t st) {
    CFP_REQUIRE(cin % 4 == 0 && cout % 4 == 0 && cin > 0 && cout > 0, "conv_wgrad_f32: %d -> %d channels (multiples of 4)", cin, cout);
    CFP_REQUIRE(taps == 1 || taps == 9, "conv_wgrad_f32: %d taps (1 x 1 and 3 x 3 convolutions are served)", taps);
    CFP_REQUIRE(B > 0 && H > 0 && W > 0, "conv_wgrad_f32: bad shape");
    const int64_t K = (int64_t)B * H * W;
    const wg::Plan p = wg::plan(K, cin, cout, taps);
    CFP_REQUIRE(p.splits == 1 || scratch, "conv_wgrad_f32: %d pixel ranges need cfp_tr_conv_wgrad_scratch_floats() of scratch", p.splits);
    const int64_t gy = (int64_t)((cin + wg::BM - 1) / wg::BM) * taps;
    CFP_REQUIRE(gy <= 65535 && p.splits <= 65535, "conv_wgrad_f32: grid too large");
    dim3 grid((cout + wg::BN - 1) / wg::BN, (unsigned)gy, p.splits);
    conv_wgrad_f32_kernel<<<grid, 256, 0, st>>>(x, dy, p.splits > 1 ? scratch : dw, H, W, cin, cout, taps == 9 ? 3 : 1, K, p.kchunk);
    if (int e = check_launch("conv_wgrad_f32")) return e;
    if (p.splits == 1) return 0;
    const int64_t n = (int64_t)taps * cin * cout;
    sum_partials_kernel<<<grid_cap(n), 256, 0, st>>>(scratch, dw, n, p.splits);
    return check_launch("conv_wgrad_sum_f32");
}

// ------------------------------------------------------------------------------------------------ upsample + concat adjoint
// Weight of source row j in the value the forward kernel forms at destination row y (upsample_concat_f32_kernel: fy = s y,
// y0 = min(int(fy), n - 1), y1 = y0 + (y0 < n - 1), weights (1 - l, l)).
__device__ __forceinline__ float interp_weight(int y, int j, float s, int n) {
    const float fy = s * y;
    int y0 = (int)fy;
    if (y0 > n - 1) y0 = n - 1;
    const int y1 = y0 + (y0 < n - 1 ? 1 : 0);
    const float l = fy - (float)y0;
    return (y0 == j ? 1.f - l : 0.f) + (y1 == j ? l : 0.f);
}

// Destination rows whose source coordinate s y lies within one pixel of j (one more row each side covers the float
// rounding of s y; interp_weight is exact and gives 0 outside).
__device__ __forceinline__ void gather_range(int j, float s, int N, int& lo, int& hi) {
    if (!(s > 0.f)) { lo = 0; hi = N - 1; return; }
    const float a = fminf((float)(j - 1) / s, (float)N), b = fminf((float)(j + 1) / s, (float)N);
    lo = max(0, (int)floorf(a) - 1);
    hi = min(N - 1, (int)ceilf(b) + 1);
}

__global__ void __launch_bounds__(256) upsample_concat_bwd_f32_kernel(const float* __restrict__ dcat, int pitch, float* __restrict__ d_lo,
                                                                      int h, int w, int c_lo, float* __restrict__ d_skip, int c_skip,
                                                                      int B, int H, int W) {
    const int g_lo = c_lo / 4;
    const int64_t n_lo = (int64_t)B * h * w * g_lo, total = n_lo + (int64_t)B * c_skip * H * W;
    const float sy = H > 1 ? (float)(h - 1) / (float)(H - 1) : 0.f, sx = W > 1 ? (float)(w - 1) / (float)(W - 1) : 0.f;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        if (i < n_lo) {
            const int64_t pix = i / g_lo;
            const int c0 = (int)(i - pix * g_lo) * 4;
            const int xl = (int)(pix % w), yl = (int)((pix / w) % h), b = (int)(pix / ((int64_t)w * h));
            int ya, yb, xa, xb;
            gather_range(yl, sy, H, ya, yb);
            gather_range(xl, sx, W, xa, xb);
            float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
            for (int y = ya; y <= yb; ++y) {
                const float wy = interp_weight(y, yl, sy, h);
                if (wy == 0.f) continue;
                const float* row = dcat + ((size_t)b * H + y) * W * pitch + c0;
                for (int x = xa; x <= xb; ++x) {
                    const float wx = interp_weight(x, xl, sx, w);
                    if (wx == 0.f) continue;
                    const float wt = wy * wx;
                    const float4 v = *reinterpret_cast<const float4*>(row + (size_t)x * pitch);
                    acc.x = fmaf(wt, v.x, acc.x); acc.y = fmaf(wt, v.y, acc.y); acc.z = fmaf(wt, v.z, acc.z); acc.w = fmaf(wt, v.w, acc.w);
                }
            }
            *reinterpret_cast<float4*>(d_lo + (size_t)pix * c_lo + c0) = acc;
        } else {
            const int64_t j = i - n_lo;                   // NCHW index of d_skip
            const int x = (int)(j % W), y = (int)((j / W) % H);
            const int64_t bc = j / ((int64_t)W * H);
            const int c = (int)(bc % c_skip), b = (int)(bc / c_skip);
            d_skip[j] = dcat[(((size_t)b * H + y) * W + x) * pitch + c_lo + c];
        }
    }
}
int upsample_concat_bwd_f32(const float* dcat, int pitch, float* d_lo, int h, int w, int c_lo, float* d_skip, int c_skip, int B, int H, int W,
                            cudaStream_t st) {
    CFP_REQUIRE(c_lo % 4 == 0 && pitch % 4 == 0 && c_lo >= 0 && c_skip >= 0 && c_lo + c_skip <= pitch,
                "upsample_concat_bwd_f32: channels %d + %d of pitch %d", c_lo, c_skip, pitch);
    CFP_REQUIRE(B > 0 && h > 0 && w > 0 && H > 0 && W > 0, "upsample_concat_bwd_f32: bad shape");
    CFP_REQUIRE(c_lo == 0 || d_lo != nullptr, "upsample_concat_bwd_f32: null d_lo");
    CFP_REQUIRE(c_skip == 0 || d_skip != nullptr, "upsample_concat_bwd_f32: null d_skip");
    const int64_t total = (int64_t)B * h * w * (c_lo / 4) + (int64_t)B * c_skip * H * W;
    if (total == 0) return 0;
    upsample_concat_bwd_f32_kernel<<<grid_cap(total), 256, 0, st>>>(dcat, pitch, d_lo, h, w, c_lo, d_skip, c_skip, B, H, W);
    return check_launch("upsample_concat_bwd_f32");
}

// ------------------------------------------------------------------------------------------------ head: softmax-expectation adjoint
// CTA = 32 pixels of one frame x all NB bins.  c_i - pred is formed as (c_i - c_m) - e with m the pixel's most probable bin
// and e = sum_j p_j (c_j - c_m) (= pred - c_m): a peaked softmax (p_m ~ 1, pred ~ c_m) would otherwise lose the small
// difference c_m - pred to the rounding of pred.  Warp w takes bins w, w + 8, ... (lane = pixel) to read prob and to write
// the [32][NB] dlogit tile, which is transposed through shared memory so that rows are written whole; the per-pixel scans
// take 8 threads per pixel.
constexpr int kHeadBwdPix = 32;
template <int NB>
__global__ void __launch_bounds__(256) head_expect_bwd_f32_kernel(const float* __restrict__ prob, const float* __restrict__ pred,
                                                                  const float* __restrict__ centres, const float* __restrict__ dpred,
                                                                  float* __restrict__ dlogit, float* __restrict__ part, int npix) {
    __shared__ float tile[kHeadBwdPix][NB + 1];
    __shared__ float cen[NB], cm_s[kHeadBwdPix], e_s[kHeadBwdPix];
    const int b = blockIdx.y, p0 = blockIdx.x * kHeadBwdPix, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int p = p0 + lane;
    const bool ok = p < npix;
    const float dv = ok ? dpred[(size_t)b * npix + p] : 0.f;
    for (int i = threadIdx.x; i < NB; i += 256) cen[i] = centres[(size_t)b * NB + i];
    for (int i = warp; i < NB; i += 8) tile[lane][i] = ok ? prob[((size_t)b * NB + i) * npix + p] : 0.f;
    __syncthreads();
    {
        const int r = threadIdx.x >> 3, q = threadIdx.x & 7;           // 8 threads per pixel, lanes 8 r' .. 8 r' + 7 of a warp
        float best = -1.f;
        int m = 0;
        for (int i = q; i < NB; i += 8)
            if (tile[r][i] > best) { best = tile[r][i]; m = i; }
#pragma unroll
        for (int o = 1; o < 8; o <<= 1) {
            const float ob = __shfl_xor_sync(0xffffffffu, best, o);
            const int om = __shfl_xor_sync(0xffffffffu, m, o);
            if (ob > best || (ob == best && om < m)) { best = ob; m = om; }
        }
        const float cm = cen[m];
        float e = 0.f;
        for (int i = q; i < NB; i += 8) e = fmaf(tile[r][i], cen[i] - cm, e);
#pragma unroll
        for (int o = 1; o < 8; o <<= 1) e += __shfl_xor_sync(0xffffffffu, e, o);
        if (q == 0) { cm_s[r] = cm; e_s[r] = e; }
    }
    __syncthreads();
    const float cm = cm_s[lane], e = e_s[lane];
    for (int i = warp; i < NB; i += 8) {
        const float pr = tile[lane][i];
        tile[lane][i] = pr * ((cen[i] - cm) - e) * dv;
        const float s = warp_sum(pr * dv);
        if (lane == 0) part[((size_t)b * gridDim.x + blockIdx.x) * NB + i] = s;
    }
    __syncthreads();
    for (int e2 = threadIdx.x; e2 < kHeadBwdPix * NB; e2 += 256) {
        const int r = e2 / NB, i = e2 % NB;
        if (p0 + r < npix) dlogit[((size_t)b * npix + p0 + r) * NB + i] = tile[r][i];
    }
}
// dcentres[b][i] = sum over the frame's tiles (in order) of part[b][tile][i]
__global__ void __launch_bounds__(256) head_centre_sum_kernel(const float* __restrict__ part, float* __restrict__ dcentres, int B, int nb,
                                                              int tiles) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= B * nb) return;
    const int b = i / nb, c = i % nb;
    float s = 0.f;
    for (int t = 0; t < tiles; ++t) s += part[((size_t)b * tiles + t) * nb + c];
    dcentres[i] = s;
}
int head_expect_bwd_f32(const float* prob, const float* pred, const float* centres, const float* dpred, int B, int npix, int nb, float* dlogit,
                        float* dcentres, float* scratch, cudaStream_t st) {
    CFP_REQUIRE(nb == 256 || nb == 128, "head_expect_bwd_f32: %d bins (128 and 256 are served)", nb);
    CFP_REQUIRE(B > 0 && npix > 0 && B <= 65535, "head_expect_bwd_f32: bad shape");
    const int tiles = (npix + kHeadBwdPix - 1) / kHeadBwdPix;
    dim3 grid(tiles, B);
    if (nb == 256) head_expect_bwd_f32_kernel<256><<<grid, 256, 0, st>>>(prob, pred, centres, dpred, dlogit, scratch, npix);
    else head_expect_bwd_f32_kernel<128><<<grid, 256, 0, st>>>(prob, pred, centres, dpred, dlogit, scratch, npix);
    if (int e = check_launch(nb == 256 ? "head_expect_bwd_f32<256>" : "head_expect_bwd_f32<128>")) return e;
    head_centre_sum_kernel<<<(B * nb + 255) / 256, 256, 0, st>>>(scratch, dcentres, B, nb, tiles);
    return check_launch("head_centre_sum_f32");
}

// ------------------------------------------------------------------------------------------------ head: bin geometry adjoint
// edges = cumsum([min_val, R y / sum(y)]), y = relu(z) + 0.1, R = max_val - min_val, centres = (edges[i] + edges[i + 1]) / 2.
// The scans and sums are done by thread 0 in index order (NB + 1 terms); the per-bin work by thread i.
__global__ void __launch_bounds__(256) head_bins_bwd_f32_kernel(const float* __restrict__ z, const float* __restrict__ d_edges,
                                                                const float* __restrict__ d_centres, float* __restrict__ dz, int nb,
                                                                float range) {
    __shared__ float de[257], dwid[256], y[256], sums[2];
    const int b = blockIdx.x, i = threadIdx.x;
    for (int e = i; e <= nb; e += blockDim.x) de[e] = d_edges ? d_edges[(size_t)b * (nb + 1) + e] : 0.f;
    float zi = 0.f;
    if (i < nb) {
        zi = z[(size_t)b * nb + i];
        y[i] = fmaxf(zi, 0.f) + 0.1f;
    }
    __syncthreads();
    if (i == 0) {
        if (d_centres)
            for (int e = 0; e < nb; ++e) {
                const float h = 0.5f * d_centres[(size_t)b * nb + e];
                de[e] += h;
                de[e + 1] += h;
            }
        float acc = 0.f;
        for (int e = nb; e >= 1; --e) {             // adjoint of the cumsum; edge 0 is the constant min_val
            acc += de[e];
            dwid[e - 1] = acc;
        }
        float s = 0.f, t = 0.f;
        for (int e = 0; e < nb; ++e) {
            s += y[e];
            t = fmaf(dwid[e], y[e], t);
        }
        sums[0] = s;
        sums[1] = t;
    }
    __syncthreads();
    if (i < nb) {
        const float s = sums[0];
        const float dy = range * (dwid[i] / s - sums[1] / (s * s));
        dz[(size_t)b * nb + i] = zi > 0.f ? dy : 0.f;
    }
}
int head_bins_bwd_f32(const float* z, const float* d_edges, const float* d_centres, float* dz, int B, int nb, float min_val, float max_val,
                      cudaStream_t st) {
    CFP_REQUIRE(nb > 0 && nb <= 256, "head_bins_bwd_f32: %d bins (at most 256)", nb);
    CFP_REQUIRE(B > 0, "head_bins_bwd_f32: bad shape");
    head_bins_bwd_f32_kernel<<<B, 256, 0, st>>>(z, d_edges, d_centres, dz, nb, max_val - min_val);
    return check_launch("head_bins_bwd_f32");
}

}  // namespace cfp
