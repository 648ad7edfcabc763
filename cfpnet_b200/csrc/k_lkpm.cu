// a7. LKPM — large-kernel depthwise propagation, Block14.forward (src/models/convnext.py:42-58):
//   y = ReLU(BN(dwconv_kxk(x) + b))            dwconv_bn_relu_kernel   (FMA-pipe bound for k=31)
//   out = x + W2 GELU(W1 LN(y) + b1) + b2      lkpm_mlp_kernel         (row chain, C -> 4C -> C)
// Eval-mode BN (and the conv bias) are folded by the host wrapper into the taps / `dw_shift`.
#include "cfp_common.cuh"
#include "cfp_internal.h"

namespace cfp {

// ------------------------------------------------------------------ depthwise k x k
// CTA = 16x16 output pixels x 16 channels.  Half-warp lanes are the 16 channels (shared
// memory is [pixel][16 ch], so a half-warp reads 64 contiguous bytes); the two half-warps
// take even / odd output columns so that they always sit on pixels of opposite parity, i.e.
// on opposite halves of the 32 banks.  A thread owns 2 rows x 8 (stride-2) columns and slides
// over the input rows with the row segment held in registers: 2*8*K FMAs per (2K + 2*8+K-2)
// shared loads.
// The tile is TY x TX = (2 x warps) x (2 Q) output pixels: 16 x 16 in general (Q = 8, eight warps); on a small map
// (the 1/16-scale level: 26 x 34, 30 x 40) ONE CTA takes the whole frame (Q = 17 or 20, a warp per two rows) - 16 x 16
// tiles covered 32 x 48 cells of a 26 x 34 map and staged a 22 x 22 halo per 256 outputs (43 % of the FMAs and 1.9x
// of the loads wasted); the frame-sized tile wastes nothing and stages 1.45x.
constexpr int kDwTile = 16, kDwCh = 16;

template <int K, typename T, int Q, int MAXT>
__global__ void __launch_bounds__(MAXT) dwconv_bn_relu_kernel(const T* __restrict__ in, T* __restrict__ out,
                                                              int H, int W, int C,
                                                              const float* __restrict__ dw_t,
                                                              const float* __restrict__ dw_shift, int relu) {
    constexpr int TX = 2 * Q, HPX = TX + K - 1, PADK = (K - 1) / 2, NIN = 2 * (Q - 1) + K;
    const int nthreads = blockDim.x, TY = 2 * (nthreads >> 5), HPY = TY + K - 1;
    extern __shared__ __align__(16) float smem[];
    float* halo = smem;                         // [HPY][HPX][16]
    float* wsm = halo + HPY * HPX * kDwCh;      // [K*K][16]
    const int cgroups = C / kDwCh;
    const int b = blockIdx.z / cgroups, c0 = (blockIdx.z % cgroups) * kDwCh;
    const int y0 = blockIdx.y * TY, x0 = blockIdx.x * TX;
    const size_t frame = (size_t)b * H * W;

    for (int i = threadIdx.x; i < K * K * (kDwCh / 4); i += nthreads) {          // taps: weights, before the wait
        const int tap = i / (kDwCh / 4), c = (i % (kDwCh / 4)) * 4;
        *reinterpret_cast<float4*>(wsm + tap * kDwCh + c) = *reinterpret_cast<const float4*>(dw_t + (size_t)tap * C + c0 + c);
    }
    pdl_wait();
    for (int i = threadIdx.x; i < HPY * HPX * (kDwCh / 4); i += nthreads) {
        const int cell = i / (kDwCh / 4), c = (i % (kDwCh / 4)) * 4;
        const int y = y0 - PADK + cell / HPX, x = x0 - PADK + cell % HPX;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (y >= 0 && y < H && x >= 0 && x < W) v = IO<T>::ld4(in + (frame + (size_t)y * W + x) * C + c0 + c);
        *reinterpret_cast<float4*>(halo + cell * kDwCh + c) = v;
    }
    __syncthreads();

    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int c = lane & 15, xh = lane >> 4, oy = warp * 2;
    float acc[2][Q];
#pragma unroll
    for (int q = 0; q < Q; ++q) acc[0][q] = acc[1][q] = 0.f;

#pragma unroll 1
    for (int iy = 0; iy < K + 1; ++iy) {
        float v[NIN];
        const float* hrow = halo + ((oy + iy) * HPX + xh) * kDwCh + c;
#pragma unroll
        for (int i = 0; i < NIN; ++i) v[i] = hrow[i * kDwCh];
        if (iy < K) {
            const float* wr = wsm + (iy * K) * kDwCh + c;
#pragma unroll
            for (int dx = 0; dx < K; ++dx) {
                const float wv = wr[dx * kDwCh];
#pragma unroll
                for (int q = 0; q < Q; ++q) acc[0][q] = fmaf(wv, v[2 * q + dx], acc[0][q]);
            }
        }
        if (iy >= 1) {
            const float* wr = wsm + ((iy - 1) * K) * kDwCh + c;
#pragma unroll
            for (int dx = 0; dx < K; ++dx) {
                const float wv = wr[dx * kDwCh];
#pragma unroll
                for (int q = 0; q < Q; ++q) acc[1][q] = fmaf(wv, v[2 * q + dx], acc[1][q]);
            }
        }
    }
    pdl_trigger();
    const float sh = dw_shift[c0 + c];
#pragma unroll
    for (int r = 0; r < 2; ++r) {
        const int y = y0 + oy + r;
        if (y >= H) continue;
#pragma unroll
        for (int q = 0; q < Q; ++q) {
            const int x = x0 + 2 * q + xh;
            if (x < W) IO<T>::st(out + (frame + (size_t)y * W + x) * C + c0 + c, relu ? fmaxf(acc[r][q] + sh, 0.f) : acc[r][q] + sh);
        }
    }
}

template <int K, typename T, int Q, int MAXT>
static int dw_launch_tile(const void* in, void* out, int B, int H, int W, int C, const float* dw_t, const float* dw_shift,
                          int relu, int warps, cudaStream_t st) {
    const int TY = 2 * warps, TX = 2 * Q;
    const size_t smem = (size_t)((TY + K - 1) * (TX + K - 1) * kDwCh + K * K * kDwCh) * sizeof(float);
    auto k = dwconv_bn_relu_kernel<K, T, Q, MAXT>;
    if (int e = set_smem(k, smem)) return e;
    dim3 grid((W + TX - 1) / TX, (H + TY - 1) / TY, B * (C / kDwCh));
    launch_pdl(k, grid, warps * 32, smem, st, (const T*)in, (T*)out, H, W, C, dw_t, dw_shift, relu);
    return check_launch(K == 31 ? "dwconv<31>" : K == 15 ? "dwconv<15>" : "dwconv<7>");
}

template <int K, typename T>
static int dw_launch(const void* in, void* out, int B, int H, int W, int C, const float* dw_t, const float* dw_shift,
                     int relu, cudaStream_t st) {
    if constexpr (K == 7) {                     // whole-frame tiles for small maps (measured 0.121 -> 0.116 ms against 16 x 16)
        if (H <= 32 && W <= 40 && H * W > 16 * 16) {
            const int warps = (H + 1) / 2;
            if (W <= 34) return dw_launch_tile<K, T, 17, 512>(in, out, B, H, W, C, dw_t, dw_shift, relu, warps, st);
            return dw_launch_tile<K, T, 20, 512>(in, out, B, H, W, C, dw_t, dw_shift, relu, warps, st);
        }
    }
    return dw_launch_tile<K, T, kDwTile / 2, kThreads>(in, out, B, H, W, C, dw_t, dw_shift, relu, kThreads / 32, st);
}

// relu = 0: the plain depthwise conv + per-channel shift (train mode: shift = the conv bias, BatchNorm follows as its
// own kernels; with the taps flipped in both axes and shift = 0 it is the conv's input gradient)
int dwconv_bn_relu(const void* in, void* out, int B, int H, int W, int C, int ksize, const float* dw_t,
                   const float* dw_shift, int dtype, cudaStream_t st, int relu) {
    CFP_REQUIRE(C % kDwCh == 0, "dwconv: C=%d not a multiple of %d", C, kDwCh);
    CFP_REQUIRE((size_t)B * (C / kDwCh) <= 65535, "dwconv: B*C/16=%zu exceeds grid.z", (size_t)B * (C / kDwCh));
#define CFP_DW(KS)                                                                                       \
    if (ksize == KS)                                                                                     \
        return dtype == CFP_F32 ? dw_launch<KS, float>(in, out, B, H, W, C, dw_t, dw_shift, relu, st)    \
                                : dw_launch<KS, bf16>(in, out, B, H, W, C, dw_t, dw_shift, relu, st);
    CFP_DW(7) CFP_DW(15) CFP_DW(31)
#undef CFP_DW
    return fail("unsupported large_kernel=%d: libcfp serves 7, 15, 31 (decoder.py:92-94)", ksize);
}

// ------------------------------------------------------------------ LN -> C->4C -> GELU -> 4C->C -> +x
template <int C, typename T>
__global__ void __launch_bounds__(kThreads) lkpm_mlp_kernel(T* __restrict__ feat0, const T* __restrict__ y, int64_t rows,
                                                            cfp_lkpm_w w) {
    constexpr int BM = C >= 128 ? 32 : 64, LDY = C + 4, LDH = 4 * C + 4;
    extern __shared__ __align__(16) float smem[];
    float* ys = smem;                   // [BM][LDY]
    float* hs = ys + BM * LDY;          // [BM][LDH]
    float* wbuf = hs + BM * LDH;
    const int64_t row0 = (int64_t)blockIdx.x * BM;
    for (int i = threadIdx.x; i < BM * (C / 4); i += kThreads) {
        int r = i / (C / 4), c = (i % (C / 4)) * 4;
        float4 v = row0 + r < rows ? IO<T>::ld4(y + (row0 + r) * C + c) : make_float4(0.f, 0.f, 0.f, 0.f);
        *reinterpret_cast<float4*>(ys + r * LDY + c) = v;
    }
    __syncthreads();
    layernorm_rows<BM, C>(ys, LDY, w.ln_g, w.ln_b, kLkpmLnEps);
    __syncthreads();
    gemm_to_smem<BM, 4 * C>(SmemRows{ys, LDY}, w.pw1_t, C, wbuf, hs, LDH,
                            [&](int c, float v) { return gelu_erf(v + w.pw1_b[c]); });
    __syncthreads();
    gemm_to_smem<BM, C>(SmemRows{hs, LDH}, w.pw2_t, 4 * C, wbuf, ys, LDY, [&](int c, float v) { return v + w.pw2_b[c]; });
    __syncthreads();
    for (int i = threadIdx.x; i < BM * (C / 4); i += kThreads) {
        int r = i / (C / 4), c = (i % (C / 4)) * 4;
        if (row0 + r < rows) {
            T* p = feat0 + (row0 + r) * C + c;
            float4 x = IO<T>::ld4(p), m = *reinterpret_cast<const float4*>(ys + r * LDY + c);
            IO<T>::st4(p, make_float4(x.x + m.x, x.y + m.y, x.z + m.z, x.w + m.w));
        }
    }
}

template <int C, typename T>
static int mlp_impl(void* feat0, const void* y, int64_t rows, const cfp_lkpm_w& w, cudaStream_t st) {
    constexpr int BM = C >= 128 ? 32 : 64, NT = 4 * C > 256 ? 256 : 4 * C;
    const size_t smem = (size_t)(BM * (C + 4) + BM * (4 * C + 4) + 2 * 32 * NT) * sizeof(float);
    auto k = lkpm_mlp_kernel<C, T>;
    if (int e = set_smem(k, smem)) return e;
    k<<<(unsigned)((rows + BM - 1) / BM), kThreads, smem, st>>>((T*)feat0, (const T*)y, rows, w);
    return check_launch("lkpm_mlp_kernel");
}

int lkpm_mlp(void* feat0, const void* y, int64_t rows, int C, const cfp_lkpm_w& w, int dtype, cudaStream_t st) {
    if (dtype == CFP_F32) {
        if (C == 32) return mlp_impl<32, float>(feat0, y, rows, w, st);
        if (C == 64) return mlp_impl<64, float>(feat0, y, rows, w, st);
        if (C == 128) return mlp_impl<128, float>(feat0, y, rows, w, st);
    } else if (dtype == CFP_BF16) {
        if (C == 32) return mlp_impl<32, bf16>(feat0, y, rows, w, st);
        if (C == 64) return mlp_impl<64, bf16>(feat0, y, rows, w, st);
        if (C == 128) return mlp_impl<128, bf16>(feat0, y, rows, w, st);
    }
    return fail("unsupported (C=%d, dtype=%d): libcfp serves C in {32,64,128}, fp32/bf16", C, dtype);
}

}  // namespace cfp
