// Decoder shell and adaptive-bins head on the 5th-gen tensor cores (SURVEY.md section 8 f1 / f2; bf16 activations,
// channels-last [B][H][W][C] maps = the token-major layout of the fusion path, so nothing is transposed between them).
//
//   f1  UpSampleBN (decoder.py:40-58) and the decoder's 1x1 / 3x3 convs (:70-80, 107-126):
//         upsample_concat   bilinear (align_corners) resize of the previous level's map + channel concat with the
//                           encoder's skip feature, written once, channels-last, input channels zero-padded to 16;
//         conv_gen_tc       k x k (k = 1, 3) convolution with ANY input width (multiple of 16) and 32 / 64 / 128 / 256
//                           output channels as an implicit GEMM: + shift (folded BatchNorm / bias), LeakyReLU.
//   f2  DepthRegression + conv_out (decoder.py:9-37, deltar.py:18-19,50-61):
//         channel_mean      per-frame mean of every channel (mean commutes with the bias-free 1x1 conv of :24-25);
//         head_regressor    conv1x1 -> 3-layer MLP -> relu + 0.1 -> normalise -> bin edges -> bin centres, one CTA per frame;
//         head_expect_tc    conv_out 1x1 (128 -> n_bins) + softmax over the bins + expectation over the frame's bin
//                           centres in ONE kernel: logits live in TMEM, the [B, n_bins, H, W] probability volume (58 MB per
//                           frame in fp32) is only written when the caller asks for it.
//
// conv_gen_tc generalises k_conv_tc.cu's scheme: a CTA owns a TR x TW block of output pixels; the zero-padded raster of
// the block (+ halo) is staged per K-chunk of KC input channels in the canonical K-major UMMA layout, the taps are MMAs
// over shifted views of it.  New here: 2-D tiles (maps wider than one M-tile), a K loop over chunks with TWO raster
// buffers (chunk c + 1 is staged by the row warps while the MMA warp works on chunk c), N up to 256.
#include "cfp_common.cuh"
#include "cfp_internal.h"
#include "umma.cuh"

namespace cfp {

struct DecBars {
    uint64_t full[3], empty[3], a_ready[2], a_free[2], acc_ready;
    uint32_t tmem_slot;
};

template <int COUT> struct DecTC {
    static constexpr int T = COUT >= 128 ? 2 : 4;        // M-tiles (of 128 raster cells) per CTA
    static constexpr int TCOLS = T * COUT;                // 512 / 256 / 256 / 128 TMEM columns
    static constexpr int NSLOT = 2;
    static constexpr int MAX_SLOT = 40 * 1024;            // bytes of one [COUT x KC] weight block
};

template <int COUT>
__global__ void __launch_bounds__(192) conv_gen_tc_kernel(const bf16* __restrict__ in, int cin, int kc, int taps,
                                                          const bf16* __restrict__ wpk, const float* __restrict__ shift, float slope,
                                                          bf16* __restrict__ out, int out_pitch, int out_coff, int H, int W, int TW,
                                                          int TR, int cells, unsigned wp_magic) {
    using P = DecTC<COUT>;
    extern __shared__ __align__(128) uint8_t smem[];
    __shared__ DecBars bars;
    const int WP = TW + 2, KG = kc / 8, nchunk = cin / kc;
    const uint32_t lbo_a = (uint32_t)cells * 16;
    const uint32_t abuf_bytes = (uint32_t)KG * lbo_a;
    const uint32_t slot_bytes = (uint32_t)COUT * kc * 2;
    uint8_t* a_buf = smem;                                  // 2 x [KG][cells][16 B]
    uint8_t* ring = smem + 2 * (size_t)abuf_bytes;          // [NSLOT][slot_bytes]
    const int tid = threadIdx.x, warp = umma::warp_idx_sync(), lane = tid & 31;
    const int b = blockIdx.z, y0 = blockIdx.y * TR, x0 = blockIdx.x * TW;
    const size_t frame = (size_t)b * H * W;

    if (tid == 0) {
        for (int i = 0; i < P::NSLOT; ++i) { umma::mbar_init(&bars.full[i], 1); umma::mbar_init(&bars.empty[i], 1); }
        for (int i = 0; i < 2; ++i) { umma::mbar_init(&bars.a_ready[i], 128); umma::mbar_init(&bars.a_free[i], 1); }
        umma::mbar_init(&bars.acc_ready, 1);
        umma::fence_mbar_init();
    }
    if (warp == 4) umma::tmem_alloc(&bars.tmem_slot, P::TCOLS);
    umma::fence_before_sync();
    __syncthreads();
    umma::fence_after_sync();
    const uint32_t tmem = bars.tmem_slot;

    if (warp < 4) {
        pdl_wait();
        // ---------------- stage the raster, one K-chunk at a time, alternating between the two buffers
        for (int c = 0; c < nchunk; ++c) {
            const int buf = c & 1;
            if (c >= 2) umma::mbar_wait(&bars.a_free[buf], (uint32_t)(((c >> 1) - 1) & 1));   // MMAs of chunk c - 2 done
            uint8_t* dstb = a_buf + (size_t)buf * abuf_bytes;
            const int total = cells * KG;
            for (int i = tid; i < total; i += 128) {
                const int ci = i / KG, kg = i - ci * KG;
                const int idx = ci - 1;                     // one slack cell in front (tap dx = 0 of cell 0)
                const bf16* g = in;
                uint32_t nbytes = 0;
                if (idx >= 0) {
                    const int pr = (int)__umulhi((unsigned)idx, wp_magic), px = idx - pr * WP;
                    const int y = y0 - 1 + pr, x = x0 - 1 + px;
                    if (pr < TR + 2 && y >= 0 && y < H && x >= 0 && x < W) {
                        g = in + (frame + (size_t)y * W + x) * cin + (size_t)c * kc + kg * 8;
                        nbytes = 16;
                    }
                }
                const uint32_t dst = umma::smem_u32(dstb + (size_t)kg * lbo_a + (size_t)ci * 16);
                asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;\n" ::"r"(dst), "l"(g), "r"(nbytes) : "memory");
            }
            asm volatile("cp.async.commit_group;\n" ::: "memory");
            asm volatile("cp.async.wait_group 0;\n" ::: "memory");
            umma::fence_async_smem();
            asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];\n" ::"r"(umma::smem_u32(&bars.a_ready[buf])) : "memory");
        }
        // ---------------- epilogue: thread = accumulator row = output cell of the padded raster
        umma::mbar_wait(&bars.acc_ready, 0);
        umma::fence_after_sync();
#pragma unroll 1
        for (int t = 0; t < P::T; ++t) {
            const int o = t * 128 + warp * 32 + lane;
            const int r = (int)__umulhi((unsigned)o, wp_magic), px = o - r * WP;
            const int y = y0 + r, x = x0 + px - 1;
            const bool live = r < TR && y < H && px >= 1 && px <= TW && x < W;
            bf16* dst = out + (frame + (size_t)y * W + x) * out_pitch + out_coff;
#pragma unroll 1
            for (int c0 = 0; c0 < COUT; c0 += 16) {
                float v[16];
                umma::tmem_ld16(umma::tmem_addr(tmem, warp * 32, t * COUT + c0), v);   // warp-collective
                if (live) {
#pragma unroll
                    for (int j = 0; j < 16; j += 4) {
                        const float4 sh = *reinterpret_cast<const float4*>(shift + c0 + j);
                        v[j] += sh.x; v[j + 1] += sh.y; v[j + 2] += sh.z; v[j + 3] += sh.w;
                    }
#pragma unroll
                    for (int j = 0; j < 16; ++j) v[j] = v[j] > 0.f ? v[j] : v[j] * slope;
#pragma unroll
                    for (int h = 0; h < 2; ++h) {
                        uint4 u;
                        u.x = umma::pack_bf16(v[8 * h + 0], v[8 * h + 1]);
                        u.y = umma::pack_bf16(v[8 * h + 2], v[8 * h + 3]);
                        u.z = umma::pack_bf16(v[8 * h + 4], v[8 * h + 5]);
                        u.w = umma::pack_bf16(v[8 * h + 6], v[8 * h + 7]);
                        *reinterpret_cast<uint4*>(dst + c0 + 8 * h) = u;
                    }
                }
            }
        }
        umma::fence_before_sync();
    } else if (warp == 4) {
        // ---------------- weight producer: one [COUT x KC] block per (chunk, tap), bulk copies L2 -> shared
        const int nblk = nchunk * taps;
        for (int c = 0; c < nblk; ++c) {
            const int slot = c % P::NSLOT, round = c / P::NSLOT;
            if (round > 0) umma::mbar_wait(&bars.empty[slot], (uint32_t)((round - 1) & 1));
            umma::bulk_load(ring + (size_t)slot * slot_bytes, wpk + (size_t)c * COUT * kc, slot_bytes, &bars.full[slot]);
        }
    } else {
        // ---------------- MMA issuer
        const uint32_t idesc = umma::idesc_bf16(128, COUT);
        const uint32_t a0 = umma::smem_u32(a_buf), w0 = umma::smem_u32(ring);
        constexpr uint32_t lbo_b = COUT * 16;
        int blk = 0;
        for (int c = 0; c < nchunk; ++c) {
            const int buf = c & 1;
            umma::mbar_wait(&bars.a_ready[buf], (uint32_t)((c >> 1) & 1));
            umma::fence_after_sync();
            for (int tap = 0; tap < taps; ++tap, ++blk) {
                const int slot = blk % P::NSLOT, round = blk / P::NSLOT;
                umma::mbar_wait(&bars.full[slot], (uint32_t)(round & 1));
                umma::fence_after_sync();
                // view of the raster for this tap: (+1 slack, -1 for dx) cancel; a 1 x 1 conv reads the centre tap
                const uint32_t tap_cell = taps == 9 ? (uint32_t)((tap / 3) * WP + (tap % 3)) : (uint32_t)(WP + 1);
                const uint64_t wd0 = umma::smem_desc(w0 + slot * slot_bytes, lbo_b);
                uint64_t ad0 = umma::smem_desc(a0 + buf * abuf_bytes + tap_cell * 16, lbo_a);
#pragma unroll 1
                for (int t = 0; t < P::T; ++t) {
                    uint64_t ad = ad0, wd = wd0;
#pragma unroll 1
                    for (int ks = 0; ks < kc / 16; ++ks) {
                        umma::mma_bf16(tmem + t * COUT, ad, wd, idesc, (blk | ks) != 0);
                        ad = umma::desc_advance(ad, 2 * lbo_a);
                        wd = umma::desc_advance(wd, 2 * lbo_b);
                    }
                    ad0 = umma::desc_advance(ad0, 128 * 16);
                }
                umma::commit(&bars.empty[slot]);
            }
            umma::commit(c + 1 < nchunk ? &bars.a_free[buf] : &bars.acc_ready);
        }
    }
    pdl_trigger();
    __syncthreads();
    if (warp == 4) {
        umma::fence_after_sync();
        umma::tmem_dealloc(tmem, P::TCOLS);
    }
}

template <int COUT>
static int conv_gen_launch(const void* in, int cin, int kc, int taps, const void* wpk, const float* shift, float slope, void* out,
                           int out_pitch, int out_coff, int B, int H, int W, cudaStream_t st) {
    using P = DecTC<COUT>;
    CFP_REQUIRE((size_t)COUT * kc * 2 <= (size_t)P::MAX_SLOT, "conv_gen: a [%d x %d] weight block exceeds the %d-byte ring slot", COUT, kc,
                P::MAX_SLOT);
    // tile: the map's width cut into equal column slices of at most 34 / 46 pixels (256 / 512 raster cells per CTA:
    // 7-10 output rows per slice, 73-80 % of the staged cells are outputs), then as many rows as fit the T M-tiles
    const int cap = P::T * 128;
    const int tw_max = cap == 256 ? 34 : 46;
    const int ncol = (W + tw_max - 1) / tw_max;
    const int TW = (W + ncol - 1) / ncol;
    const int WP = TW + 2;
    const int TR = cap / WP;
    CFP_REQUIRE(TR >= 1, "conv_gen: tile width %d leaves no room for a row", TW);
    int cells = cap + 2 * WP + 2;
    while (cells % 8 != 1) ++cells;                             // LBO / 16 = 1 (mod 8): conflict-free staging stores
    const size_t smem = 2 * (size_t)(kc / 8) * cells * 16 + (size_t)P::NSLOT * COUT * kc * 2;
    CFP_REQUIRE(smem <= 220 * 1024, "conv_gen: %zu B of shared memory (COUT %d, KC %d)", smem, COUT, kc);
    auto k = conv_gen_tc_kernel<COUT>;
    if (int e = set_smem(k, smem)) return e;
    dim3 grid((W + TW - 1) / TW, (H + TR - 1) / TR, B);
    const unsigned wp_magic = (unsigned)((((uint64_t)1 << 32) + WP - 1) / WP);
    launch_pdl(k, grid, 192, smem, st, (const bf16*)in, cin, kc, taps, (const bf16*)wpk, shift, slope, (bf16*)out, out_pitch, out_coff, H,
               W, TW, TR, cells, wp_magic);
    return check_launch(COUT == 256 ? "conv_gen_tc<256>" : COUT == 128 ? "conv_gen_tc<128>" : COUT == 64 ? "conv_gen_tc<64>" : "conv_gen_tc<32>");
}

int conv_gen_tc(const void* in, int cin, int kc, int taps, const void* wpk, const float* shift, float slope, void* out, int out_pitch,
                int out_coff, int B, int H, int W, int cout, cudaStream_t st) {
    CFP_REQUIRE(cin >= 16 && cin % 16 == 0, "conv_gen: input channels %d must be a multiple of 16 (zero-pad them)", cin);
    CFP_REQUIRE(kc >= 16 && kc % 16 == 0 && cin % kc == 0, "conv_gen: K-chunk %d must be a multiple of 16 dividing %d", kc, cin);
    CFP_REQUIRE(taps == 1 || taps == 9, "conv_gen: %d taps (1 x 1 and 3 x 3 convolutions are served)", taps);
    CFP_REQUIRE(out_pitch % 8 == 0 && out_coff % 8 == 0 && out_coff + cout <= out_pitch, "conv_gen: output slice [%d, %d) of pitch %d",
                out_coff, out_coff + cout, out_pitch);
    CFP_REQUIRE(B > 0 && B <= 65535 && H > 0 && W > 0, "conv_gen: bad shape");
#define CFP_DEC_ARGS in, cin, kc, taps, wpk, shift, slope, out, out_pitch, out_coff, B, H, W, st
    if (cout == 256) return conv_gen_launch<256>(CFP_DEC_ARGS);
    if (cout == 128) return conv_gen_launch<128>(CFP_DEC_ARGS);
    if (cout == 64) return conv_gen_launch<64>(CFP_DEC_ARGS);
    if (cout == 32) return conv_gen_launch<32>(CFP_DEC_ARGS);
#undef CFP_DEC_ARGS
    return fail("conv_gen: %d output channels (32 / 64 / 128 / 256 are served)", cout);
}

// ------------------------------------------------------------------------------------------------ upsample + concat
// out[b][y][x][:] = [ bilinear_align_corners(lo [B][h][w][c_lo] (pitch lo_pitch))(y, x) | skip [B][c_skip][H][W] (fp32, NCHW: the
// image encoder's layout) | zeros up to c_out ]      (decoder.py:51-58; F.interpolate index arithmetic as in k_io.cu)
// Two thread -> element maps in one launch: the resized part walks (pixel, 8-channel group) with the GROUP fastest - a warp reads
// and writes whole contiguous runs of a pixel's channels; the skip part walks it with the PIXEL fastest, so its NCHW fp32
// reads are coalesced along x (its 16-byte channels-last stores are the strided side).
__global__ void __launch_bounds__(256) upsample_concat_kernel(const bf16* __restrict__ lo, int h, int w, int c_lo, int lo_pitch,
                                                              const float* __restrict__ skip, int c_skip, bf16* __restrict__ out, int B,
                                                              int H, int W, int c_out) {
    pdl_wait();
    const int g_lo = c_lo / 8, g_rest = (c_out - c_lo) / 8;
    const int64_t npix = (int64_t)B * H * W, n_lo = npix * g_lo, total = n_lo + npix * g_rest;
    const float sy = H > 1 ? (float)(h - 1) / (float)(H - 1) : 0.f, sx = W > 1 ? (float)(w - 1) / (float)(W - 1) : 0.f;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        float v[8];
        int64_t pix;
        int c0;
        if (i < n_lo) {
            pix = i / g_lo;
            c0 = (int)(i - pix * g_lo) * 8;
            const int x = (int)(pix % W), y = (int)((pix / W) % H), b = (int)(pix / ((int64_t)W * H));
            const float fy = sy * y, fx = sx * x;
            int y0 = (int)fy, x0i = (int)fx;
            if (y0 > h - 1) y0 = h - 1;
            if (x0i > w - 1) x0i = w - 1;
            const int y1 = y0 + (y0 < h - 1 ? 1 : 0), x1 = x0i + (x0i < w - 1 ? 1 : 0);
            const float ly = fy - (float)y0, lx = fx - (float)x0i;
            const bf16* base = lo + (size_t)b * h * w * lo_pitch + c0;
            const uint4 q00 = *reinterpret_cast<const uint4*>(base + ((size_t)y0 * w + x0i) * lo_pitch);
            const uint4 q01 = *reinterpret_cast<const uint4*>(base + ((size_t)y0 * w + x1) * lo_pitch);
            const uint4 q10 = *reinterpret_cast<const uint4*>(base + ((size_t)y1 * w + x0i) * lo_pitch);
            const uint4 q11 = *reinterpret_cast<const uint4*>(base + ((size_t)y1 * w + x1) * lo_pitch);
            const uint32_t* a = &q00.x; const uint32_t* bq = &q01.x; const uint32_t* cq = &q10.x; const uint32_t* d = &q11.x;
            const float w00 = (1.f - ly) * (1.f - lx), w01 = (1.f - ly) * lx, w10 = ly * (1.f - lx), w11 = ly * lx;
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                v[2 * k] = w00 * __uint_as_float(a[k] << 16) + w01 * __uint_as_float(bq[k] << 16) + w10 * __uint_as_float(cq[k] << 16) +
                           w11 * __uint_as_float(d[k] << 16);
                v[2 * k + 1] = w00 * __uint_as_float(a[k] & 0xffff0000u) + w01 * __uint_as_float(bq[k] & 0xffff0000u) +
                               w10 * __uint_as_float(cq[k] & 0xffff0000u) + w11 * __uint_as_float(d[k] & 0xffff0000u);
            }
        } else {
            const int64_t j = i - n_lo;
            pix = j % npix;
            c0 = c_lo + (int)(j / npix) * 8;
            const int x = (int)(pix % W), y = (int)((pix / W) % H), b = (int)(pix / ((int64_t)W * H));
#pragma unroll
            for (int k = 0; k < 8; ++k) {
                const int c = c0 + k - c_lo;
                v[k] = c < c_skip ? skip[(((size_t)b * c_skip + c) * H + y) * W + x] : 0.f;
            }
        }
        uint4 u;
        u.x = umma::pack_bf16(v[0], v[1]); u.y = umma::pack_bf16(v[2], v[3]);
        u.z = umma::pack_bf16(v[4], v[5]); u.w = umma::pack_bf16(v[6], v[7]);
        *reinterpret_cast<uint4*>(out + (size_t)pix * c_out + c0) = u;
    }
}
int upsample_concat(const void* lo, int h, int w, int c_lo, int lo_pitch, const float* skip, int c_skip, void* out, int B, int H, int W,
                    int c_out, cudaStream_t st) {
    CFP_REQUIRE(c_lo % 8 == 0 && lo_pitch % 8 == 0 && c_out % 8 == 0 && c_lo + c_skip <= c_out, "upsample_concat: channels %d + %d -> %d (pitch %d)",
                c_lo, c_skip, c_out, lo_pitch);
    CFP_REQUIRE(B > 0 && h > 0 && w > 0 && H > 0 && W > 0, "upsample_concat: bad shape");
    CFP_REQUIRE(c_lo == 0 || lo != nullptr, "upsample_concat: null map");
    CFP_REQUIRE(c_skip == 0 || skip != nullptr, "upsample_concat: null skip feature");
    const int64_t total = (int64_t)B * H * W * (c_out / 8);
    const int64_t want = (total + 255) / 256, cap = (int64_t)sm_count() * 16;
    launch_pdl(upsample_concat_kernel, dim3((unsigned)(want < cap ? want : cap)), dim3(256), 0, st, (const bf16*)lo, h, w, c_lo, lo_pitch, skip,
               c_skip, (bf16*)out, B, H, W, c_out);
    return check_launch("upsample_concat");
}

// ------------------------------------------------------------------------------------------------ channel copy
// dst[row][coff : coff + C] = src[row][0 : C]  (pitches in elements): places a token-major map next to another one inside a
// wider channels-last buffer (torch.cat([x_d, x_d_fused], dim=1), decoder.py:112,117,122, without a concatenated copy of both).
__global__ void __launch_bounds__(256) copy_channels_kernel(const bf16* __restrict__ src, int src_pitch, bf16* __restrict__ dst, int dst_pitch,
                                                            int coff, int C, int64_t rows) {
    pdl_wait();
    const int groups = C / 8;
    const int64_t total = rows * groups;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = i / groups;
        const int g = (int)(i - r * groups);
        *reinterpret_cast<uint4*>(dst + r * dst_pitch + coff + g * 8) = *reinterpret_cast<const uint4*>(src + r * src_pitch + g * 8);
    }
}
int copy_channels(const void* src, int src_pitch, void* dst, int dst_pitch, int coff, int C, int64_t rows, cudaStream_t st) {
    CFP_REQUIRE(C % 8 == 0 && src_pitch % 8 == 0 && dst_pitch % 8 == 0 && coff % 8 == 0 && coff + C <= dst_pitch && C <= src_pitch,
                "copy_channels: %d channels from pitch %d into [%d, %d) of pitch %d", C, src_pitch, coff, coff + C, dst_pitch);
    if (rows == 0) return 0;
    const int64_t total = rows * (C / 8);
    const int64_t want = (total + 255) / 256, cap = (int64_t)sm_count() * 16;
    launch_pdl(copy_channels_kernel, dim3((unsigned)(want < cap ? want : cap)), dim3(256), 0, st, (const bf16*)src, src_pitch, (bf16*)dst,
               dst_pitch, coff, C, rows);
    return check_launch("copy_channels");
}

// ------------------------------------------------------------------------------------------------ pos-enc add on a channels-last map
// tokens[b][n][:] = x[b][n][0 : C] (pitch x_pitch) + pos[(oy + y) * pos_w + ox + x][:]   (fusion.py:87-97 for a caller that already
// holds the map channels-last: the decoder shell above - no NCHW round trip between the convs and the fusion layers).
// kCropDev: (oy, ox) = crop[0], crop[1], read from device memory when the kernel runs (a CUDA-graph replay takes fresh draws);
// otherwise the by-value offsets, and `crop` is not read.
template <bool kCropDev>
__global__ void __launch_bounds__(256) posenc_tokens_nhwc_kernel(const bf16* __restrict__ x, int x_pitch, const float* __restrict__ pos,
                                                                 bf16* __restrict__ tokens, int B, int C, int H, int W, int pos_w, int oy,
                                                                 int ox, const int* __restrict__ crop) {
    pdl_wait();
    if (kCropDev) { oy = crop[0]; ox = crop[1]; }
    const int groups = C / 8;
    const int64_t total = (int64_t)B * H * W * groups;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t pix = i / groups;
        const int g = (int)(i - pix * groups);
        const int xx = (int)(pix % W), yy = (int)((pix / W) % H);
        const uint4 q = *reinterpret_cast<const uint4*>(x + pix * x_pitch + g * 8);
        const float* pp = pos + ((size_t)(oy + yy) * pos_w + ox + xx) * C + g * 8;
        const float4 p0 = *reinterpret_cast<const float4*>(pp), p1 = *reinterpret_cast<const float4*>(pp + 4);
        const uint32_t* u = &q.x;
        uint4 o;
        o.x = umma::pack_bf16(__uint_as_float(u[0] << 16) + p0.x, __uint_as_float(u[0] & 0xffff0000u) + p0.y);
        o.y = umma::pack_bf16(__uint_as_float(u[1] << 16) + p0.z, __uint_as_float(u[1] & 0xffff0000u) + p0.w);
        o.z = umma::pack_bf16(__uint_as_float(u[2] << 16) + p1.x, __uint_as_float(u[2] & 0xffff0000u) + p1.y);
        o.w = umma::pack_bf16(__uint_as_float(u[3] << 16) + p1.z, __uint_as_float(u[3] & 0xffff0000u) + p1.w);
        *reinterpret_cast<uint4*>(tokens + pix * C + g * 8) = o;
    }
}
int posenc_tokens_nhwc(const void* x, int x_pitch, const float* pos, void* tokens, int B, int C, int H, int W, int pos_w, int oy, int ox,
                       cudaStream_t st, const int* crop) {
    CFP_REQUIRE(C % 8 == 0 && x_pitch % 8 == 0 && C <= x_pitch, "posenc_tokens_nhwc: C = %d, pitch %d", C, x_pitch);
    const int64_t total = (int64_t)B * H * W * (C / 8);
    const int64_t want = (total + 255) / 256, cap = (int64_t)sm_count() * 16;
    const dim3 grid((unsigned)(want < cap ? want : cap));
    if (crop) {
        launch_pdl(posenc_tokens_nhwc_kernel<true>, grid, dim3(256), 0, st, (const bf16*)x, x_pitch, pos, (bf16*)tokens, B, C, H, W,
                   pos_w, 0, 0, crop);
        return check_launch("posenc_tokens_nhwc_crop");
    }
    launch_pdl(posenc_tokens_nhwc_kernel<false>, grid, dim3(256), 0, st, (const bf16*)x, x_pitch, pos, (bf16*)tokens, B, C, H, W, pos_w,
               oy, ox, (const int*)nullptr);
    return check_launch("posenc_tokens_nhwc");
}

// ------------------------------------------------------------------------------------------------ head: channel mean
// mean[b][c] = mean over the frame's pixels of x[b][pix][c]  (regression_head.mean([2, 3]), decoder.py:25, taken BEFORE the
// bias-free 1x1 conv: the two commute).  CTA = (pixel slice, frame); fp32 partial sums, one atomic per (CTA, channel).
__global__ void __launch_bounds__(256) channel_mean_kernel(const bf16* __restrict__ x, int pitch, int C, int npix, float* __restrict__ mean) {
    extern __shared__ float cm_part[];                   // [rows_per_cta_group][C]
    const int b = blockIdx.y, groups = C / 8, lanes = 256 / groups;      // lanes = pixel lanes per channel group
    const int g = threadIdx.x % groups, pl = threadIdx.x / groups;
    float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    if (pl < lanes) {
        const bf16* base = x + (size_t)b * npix * pitch + g * 8;
        for (int p = blockIdx.x * lanes + pl; p < npix; p += gridDim.x * lanes) {
            const uint4 q = *reinterpret_cast<const uint4*>(base + (size_t)p * pitch);
            const uint32_t* u = &q.x;
#pragma unroll
            for (int k = 0; k < 4; ++k) { acc[2 * k] += __uint_as_float(u[k] << 16); acc[2 * k + 1] += __uint_as_float(u[k] & 0xffff0000u); }
        }
#pragma unroll
        for (int k = 0; k < 8; ++k) cm_part[pl * C + g * 8 + k] = acc[k];
    }
    __syncthreads();
    for (int c = threadIdx.x; c < C; c += 256) {
        float s = 0.f;
        for (int l = 0; l < lanes; ++l) s += cm_part[l * C + c];
        atomicAdd(mean + (size_t)b * C + c, s / (float)npix);
    }
}
int channel_mean(const void* x, int pitch, int C, int B, int npix, float* mean, cudaStream_t st) {
    CFP_REQUIRE(C % 8 == 0 && C <= 2048 && 256 % (C / 8) == 0 && pitch % 8 == 0 && C <= pitch, "channel_mean: C = %d (pitch %d)", C, pitch);
    cudaError_t e = cudaMemsetAsync(mean, 0, (size_t)B * C * sizeof(float), st);
    if (e != cudaSuccess) return fail("channel_mean: cudaMemsetAsync: %s", cudaGetErrorString(e));
    const int lanes = 256 / (C / 8);
    int gx = (npix + lanes * 8 - 1) / (lanes * 8);
    const int cap = (4 * sm_count() + B - 1) / B;
    if (gx > cap) gx = cap;
    if (gx < 1) gx = 1;
    channel_mean_kernel<<<dim3(gx, B), 256, (size_t)lanes * C * sizeof(float), st>>>((const bf16*)x, pitch, C, npix, mean);
    return check_launch("channel_mean");
}

// ------------------------------------------------------------------------------------------------ head: bin regressor
// One CTA of 32 warps per frame (tiny, latency-bound: every warp keeps a weight row's loads in flight) (decoder.py:24-36 with norm = 'linear', deltar.py:52-57): v = Wc mean, h1 = lrelu(W0 v + b0),
// h2 = lrelu(W2 h1 + b2), y = relu(W4 h2 + b4) + 0.1, y /= sum(y), widths = (max - min) y, edges = cumsum([min, widths]),
// centres = (edges[:-1] + edges[1:]) / 2.  Weights row-major [out][in] fp32 as nn.Linear / the squeezed conv keep them.
__global__ void __launch_bounds__(1024) head_regressor_kernel(const float* __restrict__ mean, const float* __restrict__ wc,
                                                             const float* __restrict__ w0, const float* __restrict__ b0,
                                                             const float* __restrict__ w2, const float* __restrict__ b2,
                                                             const float* __restrict__ w4, const float* __restrict__ b4, int E, int Hd,
                                                             int nb, float min_val, float max_val, float* __restrict__ edges,
                                                             float* __restrict__ centres) {
    extern __shared__ float rs[];                        // [E] mean | [E] v | [Hd] h1 | [Hd] h2 | [nb] y | [nb + 1] edges
    float* m = rs; float* v = m + E; float* h1 = v + E; float* h2 = h1 + Hd; float* y = h2 + Hd; float* ed = y + nb;
    const int b = blockIdx.x;
    for (int i = threadIdx.x; i < E; i += blockDim.x) m[i] = mean[(size_t)b * E + i];
    __syncthreads();
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nwarp = blockDim.x >> 5;
    auto dense = [&](const float* W, const float* bias, const float* xin, float* out, int n_out, int n_in, int act) {
        for (int o = wid; o < n_out; o += nwarp) {           // a warp per output: the weight row is read in coalesced segments
            const float* wr = W + (size_t)o * n_in;
            float s = 0.f;
            for (int k = lane; k < n_in; k += 32) s = fmaf(wr[k], xin[k], s);
            s = warp_sum(s);
            if (lane == 0) {
                if (bias) s += bias[o];
                if (act == 1) s = s > 0.f ? s : 0.01f * s;          // nn.LeakyReLU() default slope
                if (act == 2) s = fmaxf(s, 0.f) + 0.1f;
                out[o] = s;
            }
        }
        __syncthreads();
    };
    dense(wc, nullptr, m, v, E, E, 0);
    dense(w0, b0, v, h1, Hd, E, 1);
    dense(w2, b2, h1, h2, Hd, Hd, 1);
    dense(w4, b4, h2, y, nb, Hd, 2);
    if (threadIdx.x == 0) {
        float s = 0.f;
        for (int i = 0; i < nb; ++i) s += y[i];
        float e = min_val;
        ed[0] = e;
        for (int i = 0; i < nb; ++i) { e += (max_val - min_val) * (y[i] / s); ed[i + 1] = e; }
    }
    __syncthreads();
    for (int i = threadIdx.x; i <= nb; i += blockDim.x) edges[(size_t)b * (nb + 1) + i] = ed[i];
    for (int i = threadIdx.x; i < nb; i += blockDim.x) centres[(size_t)b * nb + i] = 0.5f * (ed[i] + ed[i + 1]);
}
int head_regressor(const float* mean, const float* wc, const float* w0, const float* b0, const float* w2, const float* b2, const float* w4,
                   const float* b4, int B, int E, int Hd, int nb, float min_val, float max_val, float* edges, float* centres,
                   cudaStream_t st) {
    CFP_REQUIRE(B > 0 && E > 0 && Hd > 0 && nb > 0, "head_regressor: bad shape");
    const size_t smem = (size_t)(2 * E + 2 * Hd + 2 * nb + 1) * sizeof(float);
    CFP_REQUIRE(smem <= 48 * 1024, "head_regressor: %zu B of shared memory", smem);
    head_regressor_kernel<<<B, 1024, smem, st>>>(mean, wc, w0, b0, w2, b2, w4, b4, E, Hd, nb, min_val, max_val, edges, centres);
    return check_launch("head_regressor");
}

// ------------------------------------------------------------------------------------------------ head: logits -> softmax -> expectation
// pred[row] = sum_j softmax_j(W_out x[row] + b_out) * centre[frame(row)][j]      (deltar.py:18-19,50,59)
// CTA: the [NB x 128] weight block stays in shared memory; per 128-row tile the rows are staged with cp.async, ONE MMA group
// (M = 128, N = NB, K = 128) leaves the logits in TMEM, and row thread r walks its NB logits twice (max, then exp / sums).
// The probability volume [B][NB][H][W] (fp32, NCHW as the reference returns it in eval mode) is written only if asked for.
template <int NB>
__global__ void __launch_bounds__(192) head_expect_tc_kernel(const bf16* __restrict__ x, int pitch, int64_t rows, int npix,
                                                             const bf16* __restrict__ w_tc, const float* __restrict__ bias,
                                                             const float* __restrict__ centres, float* __restrict__ pred,
                                                             float* __restrict__ prob, int ntiles) {
    constexpr int E = 128, KG = E / 8;
    constexpr uint32_t LBO = 129 * 16;
    extern __shared__ __align__(128) uint8_t smem[];
    __shared__ DecBars bars;
    uint8_t* a0 = smem;                                  // [KG][129][16 B]
    uint8_t* wsm = a0 + KG * LBO;                        // [E / 8][NB][16 B]
    const int tid = threadIdx.x, warp = umma::warp_idx_sync();
    if (tid == 0) {
        umma::mbar_init(&bars.full[0], 1);
        umma::mbar_init(&bars.a_ready[0], 128);
        umma::mbar_init(&bars.acc_ready, 1);
        umma::fence_mbar_init();
    }
    if (warp == 4) umma::tmem_alloc(&bars.tmem_slot, NB);
    umma::fence_before_sync();
    __syncthreads();
    umma::fence_after_sync();
    const uint32_t tmem = bars.tmem_slot;
    if (warp < 4) {
        pdl_wait();
        uint32_t ph = 0;
        for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
            const int64_t row = (int64_t)tile * 128 + tid;
            {
                const bf16* src = x + (row < rows ? row : 0) * pitch;
                const uint32_t nbytes = row < rows ? 16u : 0u;
#pragma unroll
                for (int kg = 0; kg < KG; ++kg) {
                    const uint32_t dst = umma::smem_u32(a0 + (size_t)kg * LBO + tid * 16);
                    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;\n" ::"r"(dst), "l"(src + kg * 8), "r"(nbytes) : "memory");
                }
                asm volatile("cp.async.commit_group;\n" ::: "memory");
                asm volatile("cp.async.wait_group 0;\n" ::: "memory");
            }
            umma::fence_async_smem();
            asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];\n" ::"r"(umma::smem_u32(&bars.a_ready[0])) : "memory");
            umma::mbar_wait(&bars.acc_ready, ph); ph ^= 1;
            umma::fence_after_sync();
            const int fr = (int)((row < rows ? row : 0) / npix);
            const float* cen = centres + (size_t)fr * NB;
            // one walk over the logits (pipelined TMEM loads), online softmax: running maximum, sums rescaled per 16-bin piece
            float mx = -3.0e38f, se = 0.f, sc = 0.f;
            umma::tmem_for_each16<NB>(umma::tmem_addr(tmem, warp * 32, 0), [&](int c0, const float (&t)[16]) {
                float l[16], cm = -3.0e38f;
#pragma unroll
                for (int j = 0; j < 16; ++j) { l[j] = t[j] + __ldg(bias + c0 + j); cm = fmaxf(cm, l[j]); }
                if (cm > mx) {
                    const float r = __expf(mx - cm);
                    se *= r; sc *= r; mx = cm;
                }
#pragma unroll
                for (int j = 0; j < 16; ++j) {
                    const float e = __expf(l[j] - mx);
                    se += e;
                    sc = fmaf(e, __ldg(cen + c0 + j), sc);
                }
            });
            if (row < rows) pred[row] = sc / se;
            if (prob) {
                const float inv = 1.f / se;
                const int64_t pix = row - (int64_t)fr * npix;
#pragma unroll 1
                for (int c0 = 0; c0 < NB; c0 += 16) {
                    float v[16];
                    umma::tmem_ld16(umma::tmem_addr(tmem, warp * 32, c0), v);
                    if (row < rows) {
#pragma unroll
                        for (int j = 0; j < 16; ++j)
                            prob[((size_t)fr * NB + c0 + j) * npix + pix] = __expf(v[j] + __ldg(bias + c0 + j) - mx) * inv;
                    }
                }
            }
            umma::fence_before_sync();
            asm volatile("bar.sync 1, 128;\n" ::: "memory");          // every row has read its logits / a0 before the next tile
        }
    } else if (warp == 4) {
        umma::bulk_load(wsm, w_tc, NB * E * 2, &bars.full[0]);
    } else {
        const uint32_t idesc = umma::idesc_bf16(128, NB);
        const uint32_t a0s = umma::smem_u32(a0), ws = umma::smem_u32(wsm);
        constexpr uint32_t LBO_B = NB * 16;
        umma::mbar_wait(&bars.full[0], 0);
        umma::fence_after_sync();
        uint32_t ph = 0;
        for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
            umma::mbar_wait(&bars.a_ready[0], ph); ph ^= 1;
            umma::fence_after_sync();
#pragma unroll
            for (int ks = 0; ks < E / 16; ++ks)
                umma::mma_bf16(tmem, umma::smem_desc(a0s + 2 * ks * LBO, LBO), umma::smem_desc(ws + ks * 2 * LBO_B, LBO_B), idesc, ks > 0);
            umma::commit(&bars.acc_ready);
        }
    }
    pdl_trigger();
    __syncthreads();
    if (warp == 4) {
        umma::fence_after_sync();
        umma::tmem_dealloc(tmem, NB);
    }
}
int head_expect_tc(const void* x, int pitch, int B, int npix, const void* w_tc, const float* bias, const float* centres, int nb, float* pred,
                   float* prob, cudaStream_t st) {
    CFP_REQUIRE(pitch % 8 == 0 && pitch >= 128, "head_expect: pitch %d", pitch);
    CFP_REQUIRE(nb == 256 || nb == 128, "head_expect: %d bins (128 and 256 are served; the reference configs use n_bins 256)", nb);
    const int64_t rows = (int64_t)B * npix;
    CFP_REQUIRE(rows > 0 && rows < ((int64_t)1 << 31), "head_expect: %lld rows", (long long)rows);
    const int ntiles = (int)((rows + 127) / 128);
    const size_t smem = (size_t)16 * 129 * 16 + (size_t)nb * 128 * 2;
    const int per_sm = nb == 256 ? 2 : 2;
    const int grid = ntiles < sm_count() * per_sm ? ntiles : sm_count() * per_sm;
    if (nb == 256) {
        auto k = head_expect_tc_kernel<256>;
        if (int e = set_smem(k, smem)) return e;
        launch_pdl(k, dim3(grid), dim3(192), smem, st, (const bf16*)x, pitch, rows, npix, (const bf16*)w_tc, bias, centres, pred, prob, ntiles);
    } else {
        auto k = head_expect_tc_kernel<128>;
        if (int e = set_smem(k, smem)) return e;
        launch_pdl(k, dim3(grid), dim3(192), smem, st, (const bf16*)x, pitch, rows, npix, (const bf16*)w_tc, bias, centres, pred, prob, ntiles);
    }
    return check_launch(nb == 256 ? "head_expect_tc<256>" : "head_expect_tc<128>");
}

}  // namespace cfp
