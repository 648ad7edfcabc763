// Decoder shell and adaptive-bins head, exact fp32 engine (SURVEY.md section 8 f1 / f2): the fp32 counterparts of the
// tcgen05 kernels of k_dec_tc.cu, on the same channels-last [B][H][W][C] maps.  Every product is an fp32 FFMA with fp32
// accumulation (no TF32 / bf16 operands: one TF32 rounding of the decoder's features already costs 2.5e-3 abs-rel of final
// depth), no atomics: each output is summed in one fixed order, so two runs give the same bits.
//
//   conv_f32          k x k (k = 1, 3) convolution as an implicit GEMM: a CTA owns a TH x TW pixel tile and NT output
//                     channels; the tile + halo of one 32-channel K-chunk sits in shared memory, the taps are shifted
//                     views of it (conv3x3_kernel of k_conv.cu), and the [32 x NT] weight block of every (chunk, tap) is
//                     streamed through a cp.async double buffer together with the next chunk's halo.
//   upsample_concat_f32, posenc_tokens_nhwc_f32, copy_channels_f32: element-wise, float4 per thread.
//   channel_mean_f32  per-frame channel mean, one CTA per frame (fixed-order tree, no atomics); the regressor behind it is
//                     head_regressor of k_dec_tc.cu, which is fp32 already.
//   head_expect_f32   conv_out 1x1 (RowsGemm) + softmax over the bins + expectation: a warp owns a pixel row's n_bins
//                     logits (8 per lane at 256 bins), the row max and sums are warp reductions; accurate expf and true
//                     divisions.
#include "cfp_common.cuh"
#include "cfp_internal.h"

namespace cfp {

// ------------------------------------------------------------------------------------------------ conv
// Thread (tr, tc): tc owns output channels [4 tc, 4 tc + 4) of the CTA's NT, tr owns RM pixels r = tr + i * NTR of the tile.
template <int NT> struct ConvF32 {
    static constexpr int CG = NT / 4;                 // column groups
    static constexpr int NTR = kThreads / CG;         // row lanes
    static constexpr int RM = 8;                      // pixels per thread
    static constexpr int BM = NTR * RM;               // 64 / 128 / 256 pixels for NT = 128 / 64 / 32
    static constexpr int TW = BM >= 128 ? 16 : 8, TH = BM / TW;
    static constexpr int HW2 = TW + 2, CELLS = (TH + 2) * HW2;
    static constexpr int KC = 32, LDA = KC + 4;       // channels per K-chunk; halo row pitch (conflict-free float4 reads)
    static constexpr size_t kSmemFloats = 2 * (size_t)CELLS * LDA + 2 * (size_t)KC * NT;
};

__device__ __forceinline__ void cp_async16_zfill(float* smem, const float* gmem, bool valid) {
    const uint32_t s = static_cast<uint32_t>(__cvta_generic_to_shared(smem));
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;\n" ::"r"(s), "l"(gmem), "r"(valid ? 16 : 0) : "memory");
}

template <int NT>
__global__ void __launch_bounds__(kThreads, 2) conv_f32_kernel(const float* __restrict__ in, int cin, int cout, int taps,
                                                               const float* __restrict__ w, const float* __restrict__ shift,
                                                               float slope, float* __restrict__ out, int out_pitch, int out_coff,
                                                               int H, int W, int nsplit) {
    using P = ConvF32<NT>;
    extern __shared__ __align__(16) float smem[];
    float* halo = smem;                                   // [2][CELLS][LDA]
    float* wbuf = smem + 2 * P::CELLS * P::LDA;           // [2][KC][NT]
    const int tid = threadIdx.x, tc = tid % P::CG, tr = tid / P::CG;
    const int b = blockIdx.z / nsplit, n0 = (blockIdx.z % nsplit) * NT;
    const int y0 = blockIdx.y * P::TH, x0 = blockIdx.x * P::TW;
    const size_t frame = (size_t)b * H * W;
    const int nchunk = (cin + P::KC - 1) / P::KC, nblk = nchunk * taps;

    // one cp.async group per block j = (chunk, tap): the weight block, plus the chunk's halo when tap == 0
    auto issue = [&](int j) {
        const int c = j / taps, tap = j - c * taps, c0 = c * P::KC;
        if (tap == 0) {
            float* dst = halo + (c & 1) * P::CELLS * P::LDA;
            for (int i = tid; i < P::CELLS * (P::KC / 4); i += kThreads) {
                const int cell = i / (P::KC / 4), ch = c0 + (i % (P::KC / 4)) * 4;
                const int y = y0 - 1 + cell / P::HW2, x = x0 - 1 + cell % P::HW2;
                const bool ok = y >= 0 && y < H && x >= 0 && x < W && ch < cin;
                cp_async16_zfill(dst + cell * P::LDA + (ch - c0), ok ? in + (frame + (size_t)y * W + x) * cin + ch : in, ok);
            }
        }
        float* dst = wbuf + (j & 1) * P::KC * NT;
        const float* src = w + ((size_t)tap * cin + c0) * cout + n0;
        for (int i = tid; i < P::KC * P::CG; i += kThreads) {
            const int kk = i / P::CG, g = i % P::CG;
            const bool ok = c0 + kk < cin;                 // rows past cin: zeros (the halo is zero there too)
            cp_async16_zfill(dst + kk * NT + 4 * g, ok ? src + (size_t)kk * cout + 4 * g : w, ok);
        }
        cp_async_commit();
    };

    float acc[P::RM][4];
#pragma unroll
    for (int i = 0; i < P::RM; ++i) acc[i][0] = acc[i][1] = acc[i][2] = acc[i][3] = 0.f;
    int cell0[P::RM];                                     // halo cell of each pixel at tap (0, 0)
#pragma unroll
    for (int i = 0; i < P::RM; ++i) {
        const int r = tr + i * P::NTR;
        cell0[i] = ((r / P::TW) * P::HW2 + r % P::TW) * P::LDA;
    }

    issue(0);
#pragma unroll 1
    for (int j = 0; j < nblk; ++j) {
        if (j + 1 < nblk) {
            issue(j + 1);
            cp_async_wait<1>();
        } else {
            cp_async_wait<0>();
        }
        __syncthreads();
        const int c = j / taps, tap = j - c * taps;
        const int dy = taps == 9 ? tap / 3 : 1, dx = taps == 9 ? tap % 3 : 1;
        const float* A = halo + (c & 1) * P::CELLS * P::LDA + (dy * P::HW2 + dx) * P::LDA;
        const float* Wb = wbuf + (j & 1) * P::KC * NT + 4 * tc;
#pragma unroll
        for (int kk = 0; kk < P::KC; kk += 4) {
            const float4 w0 = *reinterpret_cast<const float4*>(Wb + (kk + 0) * NT);
            const float4 w1 = *reinterpret_cast<const float4*>(Wb + (kk + 1) * NT);
            const float4 w2 = *reinterpret_cast<const float4*>(Wb + (kk + 2) * NT);
            const float4 w3 = *reinterpret_cast<const float4*>(Wb + (kk + 3) * NT);
#pragma unroll
            for (int i = 0; i < P::RM; ++i) {
                const float4 a = *reinterpret_cast<const float4*>(A + cell0[i] + kk);
                float* s = acc[i];
                s[0] = fmaf(a.x, w0.x, s[0]); s[1] = fmaf(a.x, w0.y, s[1]); s[2] = fmaf(a.x, w0.z, s[2]); s[3] = fmaf(a.x, w0.w, s[3]);
                s[0] = fmaf(a.y, w1.x, s[0]); s[1] = fmaf(a.y, w1.y, s[1]); s[2] = fmaf(a.y, w1.z, s[2]); s[3] = fmaf(a.y, w1.w, s[3]);
                s[0] = fmaf(a.z, w2.x, s[0]); s[1] = fmaf(a.z, w2.y, s[1]); s[2] = fmaf(a.z, w2.z, s[2]); s[3] = fmaf(a.z, w2.w, s[3]);
                s[0] = fmaf(a.w, w3.x, s[0]); s[1] = fmaf(a.w, w3.y, s[1]); s[2] = fmaf(a.w, w3.z, s[2]); s[3] = fmaf(a.w, w3.w, s[3]);
            }
        }
        __syncthreads();                                  // the buffers of block j are re-filled by issue(j + 2)
    }

    const float4 sh = *reinterpret_cast<const float4*>(shift + n0 + 4 * tc);
#pragma unroll
    for (int i = 0; i < P::RM; ++i) {
        const int r = tr + i * P::NTR, y = y0 + r / P::TW, x = x0 + r % P::TW;
        if (y < H && x < W) {
            float v[4] = {acc[i][0] + sh.x, acc[i][1] + sh.y, acc[i][2] + sh.z, acc[i][3] + sh.w};
#pragma unroll
            for (int q = 0; q < 4; ++q) v[q] = v[q] > 0.f ? v[q] : v[q] * slope;
            *reinterpret_cast<float4*>(out + (frame + (size_t)y * W + x) * out_pitch + out_coff + n0 + 4 * tc) =
                make_float4(v[0], v[1], v[2], v[3]);
        }
    }
}

template <int NT>
static int conv_f32_launch(const float* in, int cin, int cout, int taps, const float* w, const float* shift, float slope, float* out,
                           int out_pitch, int out_coff, int B, int H, int W, cudaStream_t st) {
    using P = ConvF32<NT>;
    const int nsplit = cout / NT;
    CFP_REQUIRE((int64_t)B * nsplit <= 65535, "conv_f32: %d frames x %d channel slices exceed grid.z", B, nsplit);
    const size_t smem = P::kSmemFloats * sizeof(float);
    auto k = conv_f32_kernel<NT>;
    if (int e = set_smem(k, smem)) return e;
    dim3 grid((W + P::TW - 1) / P::TW, (H + P::TH - 1) / P::TH, B * nsplit);
    k<<<grid, kThreads, smem, st>>>(in, cin, cout, taps, w, shift, slope, out, out_pitch, out_coff, H, W, nsplit);
    return check_launch(NT == 128 ? "conv_f32<128>" : NT == 64 ? "conv_f32<64>" : "conv_f32<32>");
}

int conv_f32(const float* in, int cin, int taps, const float* w, const float* shift, float slope, float* out, int out_pitch, int out_coff,
             int B, int H, int W, int cout, cudaStream_t st) {
    CFP_REQUIRE(cin >= 4 && cin % 4 == 0, "conv_f32: input channels %d must be a positive multiple of 4", cin);
    CFP_REQUIRE(taps == 1 || taps == 9, "conv_f32: %d taps (1 x 1 and 3 x 3 convolutions are served)", taps);
    CFP_REQUIRE(out_pitch % 4 == 0 && out_coff % 4 == 0 && out_coff >= 0 && out_coff + cout <= out_pitch,
                "conv_f32: output slice [%d, %d) of pitch %d", out_coff, out_coff + cout, out_pitch);
    CFP_REQUIRE(B > 0 && H > 0 && W > 0 && H <= 65535 * 8, "conv_f32: bad shape");
    if (cout == 256 || cout == 128) return conv_f32_launch<128>(in, cin, cout, taps, w, shift, slope, out, out_pitch, out_coff, B, H, W, st);
    if (cout == 64) return conv_f32_launch<64>(in, cin, cout, taps, w, shift, slope, out, out_pitch, out_coff, B, H, W, st);
    if (cout == 32) return conv_f32_launch<32>(in, cin, cout, taps, w, shift, slope, out, out_pitch, out_coff, B, H, W, st);
    return fail("conv_f32: %d output channels (32 / 64 / 128 / 256 are served)", cout);
}

static unsigned grid_for(int64_t total) {
    const int64_t want = (total + 255) / 256, cap = (int64_t)sm_count() * 16;
    return (unsigned)(want < cap ? want : cap);
}

// ------------------------------------------------------------------------------------------------ upsample + concat
// upsample_concat_kernel of k_dec_tc.cu on fp32 maps, in 4-channel groups; the interpolation is F.interpolate's
// (align_corners: source = scale * destination, weights (1 - l, l) per axis, rows blended last).
__global__ void __launch_bounds__(256) upsample_concat_f32_kernel(const float* __restrict__ lo, int h, int w, int c_lo, int lo_pitch,
                                                                  const float* __restrict__ skip, int c_skip, float* __restrict__ out,
                                                                  int B, int H, int W, int c_out) {
    const int g_lo = c_lo / 4, g_rest = (c_out - c_lo) / 4;
    const int64_t npix = (int64_t)B * H * W, n_lo = npix * g_lo, total = n_lo + npix * g_rest;
    const float sy = H > 1 ? (float)(h - 1) / (float)(H - 1) : 0.f, sx = W > 1 ? (float)(w - 1) / (float)(W - 1) : 0.f;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        float4 v;
        int64_t pix;
        int c0;
        if (i < n_lo) {
            pix = i / g_lo;
            c0 = (int)(i - pix * g_lo) * 4;
            const int x = (int)(pix % W), y = (int)((pix / W) % H), b = (int)(pix / ((int64_t)W * H));
            const float fy = sy * y, fx = sx * x;
            int y0 = (int)fy, x0 = (int)fx;
            if (y0 > h - 1) y0 = h - 1;
            if (x0 > w - 1) x0 = w - 1;
            const int y1 = y0 + (y0 < h - 1 ? 1 : 0), x1 = x0 + (x0 < w - 1 ? 1 : 0);
            const float ly = fy - (float)y0, lx = fx - (float)x0, hy = 1.f - ly, hx = 1.f - lx;
            const float* base = lo + (size_t)b * h * w * lo_pitch + c0;
            const float4 q00 = *reinterpret_cast<const float4*>(base + ((size_t)y0 * w + x0) * lo_pitch);
            const float4 q01 = *reinterpret_cast<const float4*>(base + ((size_t)y0 * w + x1) * lo_pitch);
            const float4 q10 = *reinterpret_cast<const float4*>(base + ((size_t)y1 * w + x0) * lo_pitch);
            const float4 q11 = *reinterpret_cast<const float4*>(base + ((size_t)y1 * w + x1) * lo_pitch);
            v.x = hy * (hx * q00.x + lx * q01.x) + ly * (hx * q10.x + lx * q11.x);
            v.y = hy * (hx * q00.y + lx * q01.y) + ly * (hx * q10.y + lx * q11.y);
            v.z = hy * (hx * q00.z + lx * q01.z) + ly * (hx * q10.z + lx * q11.z);
            v.w = hy * (hx * q00.w + lx * q01.w) + ly * (hx * q10.w + lx * q11.w);
        } else {
            const int64_t j = i - n_lo;
            pix = j % npix;
            c0 = c_lo + (int)(j / npix) * 4;
            const int x = (int)(pix % W), y = (int)((pix / W) % H), b = (int)(pix / ((int64_t)W * H));
            float t[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const int c = c0 + k - c_lo;
                t[k] = c < c_skip ? skip[(((size_t)b * c_skip + c) * H + y) * W + x] : 0.f;
            }
            v = make_float4(t[0], t[1], t[2], t[3]);
        }
        *reinterpret_cast<float4*>(out + (size_t)pix * c_out + c0) = v;
    }
}
int upsample_concat_f32(const float* lo, int h, int w, int c_lo, int lo_pitch, const float* skip, int c_skip, float* out, int B, int H, int W,
                        int c_out, cudaStream_t st) {
    CFP_REQUIRE(c_lo % 4 == 0 && lo_pitch % 4 == 0 && c_out % 4 == 0 && c_lo >= 0 && c_skip >= 0 && c_lo <= lo_pitch &&
                    c_lo + c_skip <= c_out,
                "upsample_concat_f32: channels %d + %d -> %d (pitch %d)", c_lo, c_skip, c_out, lo_pitch);
    CFP_REQUIRE(B > 0 && h > 0 && w > 0 && H > 0 && W > 0, "upsample_concat_f32: bad shape");
    CFP_REQUIRE(c_lo == 0 || lo != nullptr, "upsample_concat_f32: null map");
    CFP_REQUIRE(c_skip == 0 || skip != nullptr, "upsample_concat_f32: null skip feature");
    upsample_concat_f32_kernel<<<grid_for((int64_t)B * H * W * (c_out / 4)), 256, 0, st>>>(lo, h, w, c_lo, lo_pitch, skip, c_skip, out, B,
                                                                                          H, W, c_out);
    return check_launch("upsample_concat_f32");
}

// ------------------------------------------------------------------------------------------------ channel copy / pos-enc add
__global__ void __launch_bounds__(256) copy_channels_f32_kernel(const float* __restrict__ src, int src_pitch, float* __restrict__ dst,
                                                                int dst_pitch, int coff, int C, int64_t rows) {
    const int groups = C / 4;
    const int64_t total = rows * groups;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = i / groups;
        const int g = (int)(i - r * groups);
        *reinterpret_cast<float4*>(dst + r * dst_pitch + coff + g * 4) = *reinterpret_cast<const float4*>(src + r * src_pitch + g * 4);
    }
}
int copy_channels_f32(const float* src, int src_pitch, float* dst, int dst_pitch, int coff, int C, int64_t rows, cudaStream_t st) {
    CFP_REQUIRE(C % 4 == 0 && src_pitch % 4 == 0 && dst_pitch % 4 == 0 && coff % 4 == 0 && coff >= 0 && coff + C <= dst_pitch && C <= src_pitch,
                "copy_channels_f32: %d channels from pitch %d into [%d, %d) of pitch %d", C, src_pitch, coff, coff + C, dst_pitch);
    if (rows == 0) return 0;
    copy_channels_f32_kernel<<<grid_for(rows * (C / 4)), 256, 0, st>>>(src, src_pitch, dst, dst_pitch, coff, C, rows);
    return check_launch("copy_channels_f32");
}

// kCropDev: (oy, ox) from device memory, as posenc_tokens_nhwc_kernel (k_dec_tc.cu)
template <bool kCropDev>
__global__ void __launch_bounds__(256) posenc_tokens_nhwc_f32_kernel(const float* __restrict__ x, int x_pitch, const float* __restrict__ pos,
                                                                     float* __restrict__ tokens, int B, int C, int H, int W, int pos_w,
                                                                     int oy, int ox, const int* __restrict__ crop) {
    if (kCropDev) { oy = crop[0]; ox = crop[1]; }
    const int groups = C / 4;
    const int64_t total = (int64_t)B * H * W * groups;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t pix = i / groups;
        const int g = (int)(i - pix * groups);
        const int xx = (int)(pix % W), yy = (int)((pix / W) % H);
        const float4 a = *reinterpret_cast<const float4*>(x + pix * x_pitch + g * 4);
        const float4 p = *reinterpret_cast<const float4*>(pos + ((size_t)(oy + yy) * pos_w + ox + xx) * C + g * 4);
        *reinterpret_cast<float4*>(tokens + pix * C + g * 4) = make_float4(a.x + p.x, a.y + p.y, a.z + p.z, a.w + p.w);
    }
}
int posenc_tokens_nhwc_f32(const float* x, int x_pitch, const float* pos, float* tokens, int B, int C, int H, int W, int pos_w, int oy, int ox,
                           cudaStream_t st, const int* crop) {
    CFP_REQUIRE(C % 4 == 0 && x_pitch % 4 == 0 && C <= x_pitch, "posenc_tokens_nhwc_f32: C = %d, pitch %d", C, x_pitch);
    const auto grid = grid_for((int64_t)B * H * W * (C / 4));
    if (crop) {
        posenc_tokens_nhwc_f32_kernel<true><<<grid, 256, 0, st>>>(x, x_pitch, pos, tokens, B, C, H, W, pos_w, 0, 0, crop);
        return check_launch("posenc_tokens_nhwc_f32_crop");
    }
    posenc_tokens_nhwc_f32_kernel<false><<<grid, 256, 0, st>>>(x, x_pitch, pos, tokens, B, C, H, W, pos_w, oy, ox, nullptr);
    return check_launch("posenc_tokens_nhwc_f32");
}

// ------------------------------------------------------------------------------------------------ head: channel mean
// mean[b][c] = mean over the frame's pixels of x[b][pix][c].  One CTA of 1024 threads per frame: thread (pixel lane pl,
// channel group g) sums every lanes-th pixel of its four channels, then thread c adds the lanes' partial sums in lane order.
__global__ void __launch_bounds__(1024) channel_mean_f32_kernel(const float* __restrict__ x, int pitch, int C, int npix,
                                                                float* __restrict__ mean) {
    extern __shared__ float part[];                      // [lanes][C]
    const int b = blockIdx.x, groups = C / 4, lanes = 1024 / groups;
    const int g = threadIdx.x % groups, pl = threadIdx.x / groups;
    const float* base = x + (size_t)b * npix * pitch + g * 4;
    float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll 4
    for (int p = pl; p < npix; p += lanes) {
        const float4 v = *reinterpret_cast<const float4*>(base + (size_t)p * pitch);
        s.x += v.x; s.y += v.y; s.z += v.z; s.w += v.w;
    }
    *reinterpret_cast<float4*>(part + pl * C + g * 4) = s;
    __syncthreads();
    for (int c = threadIdx.x; c < C; c += 1024) {
        float t = 0.f;
        for (int l = 0; l < lanes; ++l) t += part[l * C + c];
        mean[(size_t)b * C + c] = t / (float)npix;
    }
}
int channel_mean_f32(const float* x, int pitch, int C, int B, int npix, float* mean, cudaStream_t st) {
    CFP_REQUIRE(C % 4 == 0 && C > 0 && C <= 4096 && 1024 % (C / 4) == 0 && pitch % 4 == 0 && C <= pitch,
                "channel_mean_f32: C = %d (pitch %d)", C, pitch);
    CFP_REQUIRE(B > 0 && npix > 0, "channel_mean_f32: bad shape");
    const size_t smem = (size_t)(1024 / (C / 4)) * C * sizeof(float);
    channel_mean_f32_kernel<<<B, 1024, smem, st>>>(x, pitch, C, npix, mean);
    return check_launch("channel_mean_f32");
}

// ------------------------------------------------------------------------------------------------ head: logits -> softmax -> expectation
// pred[row] = sum_j softmax_j(x[row] W + b) centre[frame(row)][j]  (deltar.py:18-19,50,59), w_t = conv_out's weight as [128][NB].
// CTA = 64 rows; warp w owns rows [8 w, 8 w + 8), lane owns NB / 32 bins of every row (RowsGemm<64, NB>::col).
template <int NB>
__global__ void __launch_bounds__(kThreads) head_expect_f32_kernel(const float* __restrict__ x, int pitch, int64_t rows, int npix,
                                                                   const float* __restrict__ w_t, const float* __restrict__ bias,
                                                                   const float* __restrict__ centres, float* __restrict__ pred,
                                                                   float* __restrict__ prob) {
    constexpr int E = 128, BM = 64, LD = E + 4;
    using G = RowsGemm<BM, NB>;
    extern __shared__ __align__(16) float smem[];
    float* xs = smem;                                    // [BM][LD]
    float* wbuf = xs + BM * LD;                          // RowsGemm weight stages
    const int64_t row0 = (int64_t)blockIdx.x * BM;
    for (int i = threadIdx.x; i < BM * (E / 4); i += kThreads) {
        const int r = i / (E / 4), c = (i % (E / 4)) * 4;
        const bool ok = row0 + r < rows;
        cp_async16_zfill(xs + r * LD + c, ok ? x + (row0 + r) * pitch + c : x, ok);
    }
    cp_async_commit();
    cp_async_wait<0>();
    __syncthreads();
    float acc[G::TM][G::TN];
    G::zero(acc);
    G::run(acc, SmemRows{xs, LD}, w_t, NB, E, wbuf);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
#pragma unroll
    for (int i = 0; i < G::TM; ++i) {
        const int64_t row = row0 + warp * G::TM + i;
        if (row >= rows) break;                           // warp-uniform
        const int fr = (int)(row / npix);
        const float* cen = centres + (size_t)fr * NB;
        float l[G::TN], mx = -INFINITY;
#pragma unroll
        for (int j = 0; j < G::TN; ++j) {
            l[j] = acc[i][j] + bias[G::col(lane, j)];
            mx = fmaxf(mx, l[j]);
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
        float se = 0.f, sc = 0.f;
#pragma unroll
        for (int j = 0; j < G::TN; ++j) {
            l[j] = expf(l[j] - mx);
            se += l[j];
            sc = fmaf(l[j], cen[G::col(lane, j)], sc);
        }
        se = warp_sum(se);                                // xor butterfly: every lane holds the same bits
        sc = warp_sum(sc);
        if (lane == 0) pred[row] = sc / se;
        if (prob) {
            const int64_t pix = row - (int64_t)fr * npix;
#pragma unroll
            for (int j = 0; j < G::TN; ++j) prob[((size_t)fr * NB + G::col(lane, j)) * npix + pix] = l[j] / se;
        }
    }
}
int head_expect_f32(const float* x, int pitch, int B, int npix, const float* w_t, const float* bias, const float* centres, int nb, float* pred,
                    float* prob, cudaStream_t st) {
    CFP_REQUIRE(pitch % 4 == 0 && pitch >= 128, "head_expect_f32: pitch %d", pitch);
    CFP_REQUIRE(nb == 256 || nb == 128, "head_expect_f32: %d bins (128 and 256 are served; the reference configs use n_bins 256)", nb);
    CFP_REQUIRE(B > 0 && npix > 0, "head_expect_f32: bad shape");
    const int64_t rows = (int64_t)B * npix;
    const int64_t grid = (rows + 63) / 64;
    CFP_REQUIRE(grid < ((int64_t)1 << 31), "head_expect_f32: %lld rows", (long long)rows);
    if (nb == 256) {
        auto k = head_expect_f32_kernel<256>;
        const size_t smem = (size_t)(64 * 132 + RowsGemm<64, 256>::kWbufFloats) * sizeof(float);
        if (int e = set_smem(k, smem)) return e;
        k<<<(unsigned)grid, kThreads, smem, st>>>(x, pitch, rows, npix, w_t, bias, centres, pred, prob);
    } else {
        auto k = head_expect_f32_kernel<128>;
        const size_t smem = (size_t)(64 * 132 + RowsGemm<64, 128>::kWbufFloats) * sizeof(float);
        if (int e = set_smem(k, smem)) return e;
        k<<<(unsigned)grid, kThreads, smem, st>>>(x, pitch, rows, npix, w_t, bias, centres, pred, prob);
    }
    return check_launch(nb == 256 ? "head_expect_f32<256>" : "head_expect_f32<128>");
}

}  // namespace cfp
