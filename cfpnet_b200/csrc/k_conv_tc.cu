// DAPM 3x3 convolutions on the 5th-gen tensor cores (bf16 path).
//
//   out = conv3x3(cat[in0, in1]) (+BN folded) (+ residual)          transformer.py:239-247
//
// Implicit GEMM without im2col.  A CTA owns R consecutive image rows of one frame.  It stages
// the zero-padded raster of those rows (+1 halo row above and below, +1 halo column left and
// right: WP = W + 2 cells per row) ONCE in shared memory in the canonical K-major no-swizzle
// UMMA layout [channel-group][cell][16 B].  Output positions are indexed by the same padded
// raster, so the A operand of tap (dy,dx) for the M-tile of output cells [128 t, 128 t + 128)
// is the same buffer viewed from cell 128 t + dy*WP + dx - 1: nine tcgen05.mma groups over nine
// start addresses.  The two junk columns per raster row cost 2/WP of the MMA work and are
// dropped in the epilogue.
//
// Per CTA:  warps 0-3  stage the raster (per source), then run the epilogue: thread = TMEM lane
//                      = output cell; adds shift (+ residual) and writes bf16 tokens;
//           warp 4     lane 0 streams the per-(source, tap) weight blocks [C x C] (pre-packed in
//                      the canonical layout by the host) through a ring with the bulk-copy (TMA)
//                      engine, mbarrier complete_tx;
//           warp 5     lane 0 issues tcgen05.mma (M=128, N=C, K=16) into T accumulators of C
//                      TMEM columns each and releases ring slots with tcgen05.commit.
// The concatenated input of conv1 is processed as two K-halves (sources) through the same
// raster buffer; the message-map source is zero inside the zone rectangle by construction
// (transformer.py:233-234) and those cells are never read.
#include "cfp_common.cuh"
#include "cfp_internal.h"
#include "umma.cuh"
#include <stdio.h>

namespace cfp {

#ifdef CFP_DEBUG_TIMING
// phase timestamps (globaltimer ns) of CTA (0,0): [0] start, [1] source-0 raster landed, [2] source-1 (or last) raster
// landed, [3] accumulators ready, [4] epilogue done; row thread 0 writes them.  Debug builds only.
__device__ unsigned long long g_conv_dbg[8];
__device__ __forceinline__ unsigned long long dbg_now() { unsigned long long t; asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t)); return t; }
#define CFP_DBG_MARK(i) do { if (blockIdx.x == 1 && blockIdx.y == 1 && threadIdx.x == 0) g_conv_dbg[i] = dbg_now(); } while (0)
#else
#define CFP_DBG_MARK(i) do { } while (0)
#endif

template <int C, int TCOLS> struct ConvTC {
    static constexpr int T = TCOLS / C;               // M-tiles per CTA: T*C = TCOLS TMEM columns (256 or 128)
    // weight ring depth (measured: 2 slots and 9 / 4 slots change nothing or cost occupancy; measured again at C = 32 with the
    // per-stage timeline in hand - 72 MMAs of a source take 4.5 us against 1.5 us of tensor time - nine 2 KB slots, a whole
    // source's taps, still four CTAs per SM: conv3x3_tc<2C->C,32> 0.199 -> 0.207 ms.  The issuer is not waiting for weights.)
    static constexpr int NSLOT = C >= 128 ? 2 : 3;
    static constexpr int SLOT_BYTES = C * C * 2;      // one [C x C] bf16 block
    static constexpr int KG = C / 8;                  // 16-byte channel groups per source
};

struct ConvTCBars {
    uint64_t full[3], empty[3], a_ready, a_free, acc_ready;
    uint32_t tmem_slot;
};

template <int C, int TCOLS>
__global__ void __launch_bounds__(192) conv3x3_tc_kernel(const bf16* __restrict__ in0, const bf16* __restrict__ in1,
                                                         const bf16* __restrict__ wpk,
                                                         const float* __restrict__ shift,
                                                         const bf16* __restrict__ residual, bf16* __restrict__ out,
                                                         int H, int W, int R, int cells, unsigned wp_magic, int zy0,
                                                         int zy1, int zx0, int zx1) {
    using P = ConvTC<C, TCOLS>;
    extern __shared__ __align__(128) uint8_t smem[];
    __shared__ ConvTCBars bars;
    const int WP = W + 2;
    const uint32_t lbo_a = (uint32_t)cells * 16;
    uint8_t* a_buf = smem;                                  // [KG][cells][16 B]
    uint8_t* ring = a_buf + (size_t)P::KG * lbo_a;          // [NSLOT][SLOT_BYTES]
    const int tid = threadIdx.x, warp = umma::warp_idx_sync(), lane = tid & 31;
    const int b = blockIdx.y, y0 = blockIdx.x * R;
    const int nsrc = in1 ? 2 : 1;
    const size_t frame = (size_t)b * H * W;

    if (tid == 0) {
        for (int i = 0; i < P::NSLOT; ++i) { umma::mbar_init(&bars.full[i], 1); umma::mbar_init(&bars.empty[i], 1); }
        umma::mbar_init(&bars.a_ready, 128);
        umma::mbar_init(&bars.a_free, 1);
        umma::mbar_init(&bars.acc_ready, 1);
        umma::fence_mbar_init();
    }
    if (warp == 4) umma::tmem_alloc(&bars.tmem_slot, TCOLS);
    umma::fence_before_sync();
    __syncthreads();
    umma::fence_after_sync();
    const uint32_t tmem = bars.tmem_slot;

    CFP_DBG_MARK(0);
    if (warp < 4) {
        pdl_wait();                       // the maps come from the previous kernels of the stream (weights do not)
        // ---------------- stage the raster, one source at a time
        for (int s = 0; s < nsrc; ++s) {
            if (s > 0) umma::mbar_wait(&bars.a_free, 0);    // all MMAs reading source 0 have completed
            const bf16* src = s == 0 ? in0 : in1;
            // cp.async (LDGSTS) with zero-fill: every 16-byte chunk of the raster is one fire-and-forget copy, so
            // all of a thread's ~40 copies are in flight at once (register staging made this phase latency-bound)
            const int total = cells * P::KG;
            for (int i = tid; i < total; i += 128) {
                const int ci = i / P::KG, kg = i % P::KG;
                const int idx = ci - 1;                     // one slack cell in front (tap dx=0 of cell 0)
                const bf16* g = src;                        // any valid address when the chunk is zero-filled
                uint32_t nbytes = 0;
                if (idx >= 0) {
                    const int pr = (int)__umulhi((unsigned)idx, wp_magic), px = idx - pr * WP;
                    const int y = y0 - 1 + pr, x = px - 1;
                    if (pr < R + 2 && y >= 0 && y < H && x >= 0 && x < W &&
                        !(s == 1 && y >= zy0 && y < zy1 && x >= zx0 && x < zx1)) {
                        g = src + (frame + (size_t)y * W + x) * C + kg * 8;
                        nbytes = 16;
                    }
                }
                const uint32_t dst = umma::smem_u32(a_buf + (size_t)kg * lbo_a + (size_t)ci * 16);
                asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;\n" ::"r"(dst), "l"(g), "r"(nbytes) : "memory");
            }
            asm volatile("cp.async.commit_group;\n" ::: "memory");
            asm volatile("cp.async.wait_group 0;\n" ::: "memory");
            CFP_DBG_MARK(1 + s);
            umma::fence_async_smem();
            asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];\n" ::"r"(umma::smem_u32(&bars.a_ready)) : "memory");
        }
        // ---------------- epilogue: thread = accumulator row = output cell of the padded raster.  The residual row of tile
        // t + 1 is fetched while tile t is processed (and tile 0's while the MMAs still run): its load latency used to be
        // paid eight times per CTA.
        auto cell_of = [&](int t, bool& live) -> size_t {
            const int o = t * 128 + warp * 32 + lane;
            const int r = (int)__umulhi((unsigned)o, wp_magic), px = o - r * WP;   // o / WP (exact: o*WP < 2^32)
            const int y = y0 + r, x = px - 1;
            live = r < R && y < H && x >= 0 && x < W;
            return (frame + (size_t)y * W + x) * C;
        };
        constexpr int NCH = C / 8;
        uint4 res_next[NCH];
        auto fetch_res = [&](int t) {
            bool live;
            const size_t off = cell_of(t, live);
#pragma unroll
            for (int k = 0; k < NCH; ++k)
                res_next[k] = (residual && live) ? *reinterpret_cast<const uint4*>(residual + off + k * 8) : make_uint4(0u, 0u, 0u, 0u);
        };
        fetch_res(0);
        umma::mbar_wait(&bars.acc_ready, 0);
        CFP_DBG_MARK(3);
        umma::fence_after_sync();
#pragma unroll 1
        for (int t = 0; t < P::T; ++t) {
            bool live;
            const size_t off = cell_of(t, live);
            uint4 res[NCH];
#pragma unroll
            for (int k = 0; k < NCH; ++k) res[k] = res_next[k];
            if (t + 1 < P::T) fetch_res(t + 1);
#pragma unroll
            for (int c0 = 0; c0 < C; c0 += 16) {
                float v[16];
                umma::tmem_ld16(umma::tmem_addr(tmem, warp * 32, t * C + c0), v);   // warp-collective
                if (live) {
#pragma unroll
                    for (int j = 0; j < 16; j += 4) {
                        const float4 sh = *reinterpret_cast<const float4*>(shift + c0 + j);
                        v[j] += sh.x; v[j + 1] += sh.y; v[j + 2] += sh.z; v[j + 3] += sh.w;
                    }
#pragma unroll
                    for (int h = 0; h < 2; ++h) {
                        const uint4 rr = res[(c0 >> 3) + h];
                        const uint32_t w4[4] = {rr.x, rr.y, rr.z, rr.w};
                        uint4 u;
                        uint32_t* up = &u.x;
#pragma unroll
                        for (int k = 0; k < 4; ++k)
                            up[k] = umma::pack_bf16(v[8 * h + 2 * k] + __uint_as_float(w4[k] << 16),
                                                    v[8 * h + 2 * k + 1] + __uint_as_float(w4[k] & 0xffff0000u));
                        *reinterpret_cast<uint4*>(out + off + c0 + 8 * h) = u;
                    }
                }
            }
        }
        CFP_DBG_MARK(4);
        umma::fence_before_sync();
    } else if (warp == 4) {
        // ---------------- weight producer (bulk async copies, L2 -> shared)
        const int nchunk = nsrc * 9;
        for (int c = 0; c < nchunk; ++c) {
            const int slot = c % P::NSLOT, round = c / P::NSLOT;
            if (round > 0) umma::mbar_wait(&bars.empty[slot], (round - 1) & 1);
            umma::bulk_load(ring + (size_t)slot * P::SLOT_BYTES, wpk + (size_t)c * C * C, P::SLOT_BYTES, &bars.full[slot]);
        }
    } else {
        // ---------------- MMA issuer (whole warp runs the loop; one elected lane issues)
        {
            const uint32_t idesc = umma::idesc_bf16(128, C);
            const uint32_t a0 = umma::smem_u32(a_buf), w0 = umma::smem_u32(ring);
            constexpr uint32_t lbo_b = C * 16;
            int c = 0;
            for (int s = 0; s < nsrc; ++s) {
                umma::mbar_wait(&bars.a_ready, s & 1);
                umma::fence_after_sync();
                for (int tap = 0; tap < 9; ++tap, ++c) {
                    const int slot = c % P::NSLOT, round = c / P::NSLOT;
                    umma::mbar_wait(&bars.full[slot], round & 1);
                    umma::fence_after_sync();
                    const uint32_t tap_cell = (tap / 3) * WP + (tap % 3);      // (+1 slack, -1 for dx) cancel
                    const uint64_t wd0 = umma::smem_desc(w0 + slot * P::SLOT_BYTES, lbo_b);
                    uint64_t ad0 = umma::smem_desc(a0 + tap_cell * 16, lbo_a);
#pragma unroll 1
                    for (int t = 0; t < P::T; ++t) {
                        uint64_t ad = ad0, wd = wd0;
#pragma unroll
                        for (int ks = 0; ks < C / 16; ++ks) {
                            umma::mma_bf16(tmem + t * C, ad, wd, idesc, (c | ks) != 0);
                            ad = umma::desc_advance(ad, 2 * lbo_a);
                            wd = umma::desc_advance(wd, 2 * lbo_b);
                        }
                        ad0 = umma::desc_advance(ad0, 128 * 16);
                    }
                    umma::commit(&bars.empty[slot]);
                }
                umma::commit(s + 1 < nsrc ? &bars.a_free : &bars.acc_ready);
            }
        }
    }
    pdl_trigger();                         // this CTA's work is done: the next kernel of the stream may start its prologue
    __syncthreads();
    if (warp == 4) {
        umma::fence_after_sync();
        umma::tmem_dealloc(tmem, TCOLS);
    }
}

template <int C, int TCOLS>
static int conv_tc_launch(const void* in0, const void* in1, const void* wpk, const float* shift, const void* residual,
                          void* out, int B, int H, int W, int zy0, int zy1, int zx0, int zx1, cudaStream_t st) {
    using P = ConvTC<C, TCOLS>;
    const int WP = W + 2;
    const int R = (P::T * 128) / WP;
    CFP_REQUIRE(R >= 1, "conv3x3 (tensor-core path): map width %d exceeds %d", W, P::T * 128 - 2);
    int cells = P::T * 128 + 2 * WP + 2;
    while (cells % 8 != 1) ++cells;              // LBO/16 = 1 (mod 8): conflict-free staging stores
    const size_t smem = (size_t)P::KG * cells * 16 + (size_t)P::NSLOT * P::SLOT_BYTES;
    CFP_REQUIRE(smem <= 220 * 1024, "conv3x3 (tensor-core path): %zu B shared memory", smem);
    auto k = conv3x3_tc_kernel<C, TCOLS>;
    if (int e = set_smem(k, smem)) return e;
    dim3 grid((H + R - 1) / R, B);
    const unsigned wp_magic = (unsigned)((((uint64_t)1 << 32) + WP - 1) / WP);   // umulhi(i, magic) == i / WP for i*WP < 2^32
    launch_pdl(k, grid, 192, smem, st, (const bf16*)in0, (const bf16*)in1, (const bf16*)wpk, shift, (const bf16*)residual,
               (bf16*)out, H, W, R, cells, wp_magic, zy0, zy1, zx0, zx1);
#ifdef CFP_DEBUG_TIMING
    {
        cudaStreamSynchronize(st);
        unsigned long long h[8] = {0};
        cudaMemcpyFromSymbol(h, g_conv_dbg, sizeof(h));
        fprintf(stderr, "conv3x3_tc<C=%d,%s> CTA(1,1) ns: stage0 %llu  stage1 %llu  mma-done %llu  epilogue %llu  (grid %d x %d)\n", C,
                in1 ? "2C->C" : "C->C", h[1] - h[0], h[2] - h[0], h[3] - h[0], h[4] - h[0], grid.x, grid.y);
    }
#endif
    return check_launch(in1 ? (C == 32 ? "conv3x3_tc<2C->C,32>" : C == 64 ? "conv3x3_tc<2C->C,64>" : "conv3x3_tc<2C->C,128>")
                            : (C == 32 ? "conv3x3_tc<C->C,32>" : C == 64 ? "conv3x3_tc<C->C,64>" : "conv3x3_tc<C->C,128>"));
}

int conv3x3_tc(const void* in0, const void* in1, const void* wpk, const float* shift, const void* residual, void* out,
               int B, int H, int W, int C, int zy0, int zy1, int zx0, int zx1, cudaStream_t st) {
    CFP_REQUIRE(B <= 65535, "B too large for grid.y");
    // CTA size: 128 accumulator columns (T = 128/C M-tiles) at C <= 64, 256 at C = 128: with half the raster per CTA, twice
    // the CTAs share an SM, and co-resident CTAs are what overlaps the serial stage -> MMA -> epilogue phases of a CTA.
    // Measured (B200, 64 frames): 128 columns win for C = 32 / 64 (0.84x / 0.93x the time), 256 for C = 128.
    // Raster staging by tensor-map TMA was measured and removed: equal at C = 64 / 128, 6 % slower at C = 32, and the
    // cp.async form is 1.3 % faster on the concurrent step.
#define CFP_CONV_ARGS in0, in1, wpk, shift, residual, out, B, H, W, zy0, zy1, zx0, zx1, st
    if (C == 32) return conv_tc_launch<32, 128>(CFP_CONV_ARGS);
    if (C == 64) return conv_tc_launch<64, 128>(CFP_CONV_ARGS);
    if (C == 128) return conv_tc_launch<128, 256>(CFP_CONV_ARGS);
#undef CFP_CONV_ARGS
    return fail("unsupported C=%d", C);
}

}  // namespace cfp
