// Fused LoFTR query chain on the 5th-gen tensor cores (bf16 path):
//
//   x --Wq--> q --elu+1--> Q --(Q KV)/(Q.Ksum+eps)--> msg --Wm--> LN1 --[x|msg] W1--> relu --W2--> LN2 --(+x)--> out
//
// (transformer.py:54-71, attention.py:31-49).  One CTA keeps a 128-token tile on chip through the
// whole chain: the five GEMMs run as tcgen05.mma (M=128, N=C, K=16) with fp32 accumulators in
// TMEM; between GEMMs the 128 "row" threads (thread r <-> token r <-> TMEM lane r) read their
// accumulator row with tcgen05.ld, apply the row-wise math in registers and write the next A
// operand straight into shared memory in the canonical K-major UMMA layout (umma.cuh).  The tile is
// read from HBM once and written once.
//
// Weights: every GEMM of the chain is cut into [C x C] bf16 blocks (8 per tile: Wq, Wm, four
// quadrants of W1, two K-halves of W2), pre-packed by the host in consumption order; a producer
// lane streams them through a shared-memory ring with the bulk-copy (TMA) engine while MMAs and
// row math of earlier stages run.
//
//   warps 0-3 : row threads (stage x, epilogues)      warp 4 : weight producer      warp 5 : MMA issuer
//
// The same kernel serves hist2image, LSA, GSA (full chain) and the DAPM attention (q -> msg only)
// through the row providers of providers.cuh.
#include "cfp_common.cuh"
#include "cfp_internal.h"
#include "providers.cuh"
#include "umma.cuh"
#include <cuda_fp16.h>
#include <stdlib.h>
#include <stdio.h>

namespace cfp {

#ifdef CFP_DEBUG_TIMING
// phase timestamps (globaltimer ns) of the second tile of CTA 5 of a query-chain launch.  Debug builds only.
__device__ unsigned long long g_chain_dbg[16];
__device__ __forceinline__ unsigned long long chain_now() { unsigned long long t; asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t)); return t; }
#define CFP_CHAIN_MARK(i, it) do { if (blockIdx.x == 5 && threadIdx.x == 0 && (it) == 1) g_chain_dbg[i] = chain_now(); } while (0)
#else
#define CFP_CHAIN_MARK(i, it) do { } while (0)
#endif

template <int C> struct ChainTC {
    static constexpr int KG = C / 8;                       // 16-byte k-groups per C columns
    static constexpr uint32_t LBO = 129 * 16;              // 128 rows + one pad chunk: conflict-free staging
    static constexpr int SLOT = 2 * C * C;                 // bytes of one [C x C] bf16 weight block
    static constexpr int NSLOT = C >= 128 ? 2 : 4;
    static constexpr int ABUF = 2 * KG * (int)LBO;         // a tile of up to 2C columns
    static constexpr int TMEM_COLS = 2 * C < 32 ? 32 : 2 * C;
    static constexpr size_t SMEM = 2 * (size_t)ABUF + (size_t)NSLOT * SLOT;
};

struct ChainBars {
    uint64_t full[4], empty[4], a_ready, acc_ready, kv_full;
    uint32_t tmem_slot;
};

__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];\n" ::"r"(umma::smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void rows_sync() { asm volatile("bar.sync 1, 128;\n" ::: "memory"); }

__device__ __forceinline__ void unpack8(uint4 u, float (&v)[8]) {
    v[0] = __uint_as_float(u.x << 16); v[1] = __uint_as_float(u.x & 0xffff0000u);
    v[2] = __uint_as_float(u.y << 16); v[3] = __uint_as_float(u.y & 0xffff0000u);
    v[4] = __uint_as_float(u.z << 16); v[5] = __uint_as_float(u.z & 0xffff0000u);
    v[6] = __uint_as_float(u.w << 16); v[7] = __uint_as_float(u.w & 0xffff0000u);
}

// Row r's accumulator columns [col0, col0 + N) -> registers.
template <int N>
__device__ __forceinline__ void load_cols(uint32_t tmem, int wq, int col0, float (&v)[N]) {
    umma::tmem_for_each16<N>(umma::tmem_addr(tmem, wq * 32, col0), [&](int c0, const float (&t)[16]) {
#pragma unroll
        for (int j = 0; j < 16; ++j) v[c0 + j] = t[j];
    });
}
template <int C>
__device__ __forceinline__ void layernorm_reg(float (&v)[C], const float* __restrict__ g, const float* __restrict__ b) {
    using namespace umma;
    f32x2 p[C / 2];                                      // the row as C/2 register pairs: every step is one packed op per pair
    f32x2 s2 = pack2(0.f, 0.f);
#pragma unroll
    for (int i = 0; i < C / 2; ++i) { p[i] = pack2(v[2 * i], v[2 * i + 1]); s2 = add2(s2, p[i]); }
    float s_lo, s_hi;
    unpack2(s2, s_lo, s_hi);
    const float mean = (s_lo + s_hi) * (1.f / C);
    const f32x2 nm = pack2(-mean, -mean);
    f32x2 q2 = pack2(0.f, 0.f);
#pragma unroll
    for (int i = 0; i < C / 2; ++i) { p[i] = add2(p[i], nm); q2 = fma2(p[i], p[i], q2); }
    float q_lo, q_hi;
    unpack2(q2, q_lo, q_hi);
    const float rstd = rsqrtf((q_lo + q_hi) * (1.f / C) + kLnEps);
    const f32x2 r2 = pack2(rstd, rstd);
#pragma unroll
    for (int i = 0; i < C / 2; i += 2) {                 // gamma / beta as 16-byte loads (warp-uniform addresses)
        const float4 g4 = *reinterpret_cast<const float4*>(g + 2 * i), b4 = *reinterpret_cast<const float4*>(b + 2 * i);
        const f32x2 o0 = fma2(mul2(p[i], r2), pack2(g4.x, g4.y), pack2(b4.x, b4.y));
        const f32x2 o1 = fma2(mul2(p[i + 1], r2), pack2(g4.z, g4.w), pack2(b4.z, b4.w));
        unpack2(o0, v[2 * i], v[2 * i + 1]);
        unpack2(o1, v[2 * i + 2], v[2 * i + 3]);
    }
}
// Statistics of a row whose C columns are split over two threads (CH = C / 2 each): every thread brings the mean of its
// half and the sum of squares centred on THAT mean; one exchange through shared memory (xch[half][row]) and Chan's
// pairwise combination give the row's mean and 1 / std.  `sync` is a barrier over all threads that share rows.
// Returns {shift, rstd}: (v - mean) = (v - mean_half) + shift.
template <int C, class Sync>
__device__ __forceinline__ float2 ln_combine_halves(float mean_h, float m2_h, float2* xch, int row, int half, float eps, Sync&& sync) {
    constexpr int CH = C / 2;
    xch[half * 128 + row] = make_float2(mean_h, m2_h);
    sync();
    const float2 o = xch[(half ^ 1) * 128 + row];
    const float mean = 0.5f * (mean_h + o.x), d = mean_h - o.x;
    const float var = (m2_h + o.y + d * d * (0.5f * CH)) * (1.f / C);
    return make_float2(mean_h - mean, rsqrtf(var + eps));
}
// LayerNorm of the CH = C / 2 columns this thread holds of a split row (g, b already offset to those columns)
template <int C, class Sync>
__device__ __forceinline__ void layernorm_half(float (&v)[C / 2], const float* __restrict__ g, const float* __restrict__ b,
                                               float2* xch, int row, int half, Sync&& sync) {
    using namespace umma;
    constexpr int CH = C / 2;
    f32x2 p[CH / 2];
    f32x2 s2 = pack2(0.f, 0.f);
#pragma unroll
    for (int i = 0; i < CH / 2; ++i) { p[i] = pack2(v[2 * i], v[2 * i + 1]); s2 = add2(s2, p[i]); }
    float s_lo, s_hi;
    unpack2(s2, s_lo, s_hi);
    const float mean_h = (s_lo + s_hi) * (1.f / CH);
    const f32x2 nm = pack2(-mean_h, -mean_h);
    f32x2 q2 = pack2(0.f, 0.f);
#pragma unroll
    for (int i = 0; i < CH / 2; ++i) { p[i] = add2(p[i], nm); q2 = fma2(p[i], p[i], q2); }
    float q_lo, q_hi;
    unpack2(q2, q_lo, q_hi);
    const float2 st = ln_combine_halves<C>(mean_h, q_lo + q_hi, xch, row, half, kLnEps, sync);
    const f32x2 sh2 = pack2(st.x, st.x), r2 = pack2(st.y, st.y);
#pragma unroll
    for (int i = 0; i < CH / 2; i += 2) {
        const float4 g4 = *reinterpret_cast<const float4*>(g + 2 * i), b4 = *reinterpret_cast<const float4*>(b + 2 * i);
        const f32x2 o0 = fma2(mul2(add2(p[i], sh2), r2), pack2(g4.x, g4.y), pack2(b4.x, b4.y));
        const f32x2 o1 = fma2(mul2(add2(p[i + 1], sh2), r2), pack2(g4.z, g4.w), pack2(b4.z, b4.w));
        unpack2(o0, v[2 * i], v[2 * i + 1]);
        unpack2(o1, v[2 * i + 2], v[2 * i + 3]);
    }
}

// ---------------------------------------------------------------------------------------
// Row-thread stages of the chain, shared by the two kernel organisations below.  A token row is owned by NT threads
// (NT = 1: thread `tid` <-> token row0 + tid <-> TMEM lane tid; NT = 2: two threads of different warps with the same
// TMEM lane quarter share a row, `half` selects which CH = C / NT columns - i.e. which heads, which 16-byte chunks -
// are this thread's).  At C >= 64 a thread per row meant 4-8 warps per SM walking 64-256 accumulator columns each in
// one long dependent instruction stream (issue-slot utilisation 0.11-0.26); two threads per row halve every epilogue
// and double the warps the schedulers can pick from.  Only the two LayerNorms need the other half: one exchange of
// (mean, centred sum of squares) through shared memory each.
template <class Q> struct IsZonePatch { static constexpr bool value = false; };
template <class T, bool F> struct IsZonePatch<ZonePatchRows<T, F>> { static constexpr bool value = true; };

template <int C, int NH, bool kAttnOnly, class Q, int NT = 1>
struct ChainStages {
    using P = ChainTC<C>;
    static constexpr int DH = C / NH, KG = P::KG, G = DH < 16 ? 16 : DH;
    static constexpr int CH = C / NT, KGT = KG / NT;
    static_assert(NT == 1 || NT == 2, "one or two threads per row");
    static_assert(CH % G == 0 && CH % 16 == 0, "a thread owns whole heads and whole 16-column pieces");
    struct Row { typename Q::R ref; int g; };
    // stage x: locate the row once, copy this thread's chunks of its C channels into a0[:, 0:C)
    static __device__ __forceinline__ Row stage_x(const Q& q, int64_t row0, int tid, uint8_t* a0, int half = 0) {
        const int64_t row = row0 + tid;
        const bool live = row < q.rows;
        Row r;
        r.ref = q.locate(live ? row : 0);
        r.g = live ? q.group(r.ref) : -1;
        uint4 v[KGT];
#pragma unroll
        for (int kg = 0; kg < KGT; ++kg) v[kg] = live ? load8_bf16(q, r.ref, (half * KGT + kg) * 8) : make_uint4(0u, 0u, 0u, 0u);
#pragma unroll
        for (int kg = 0; kg < KGT; ++kg) *reinterpret_cast<uint4*>(a0 + (size_t)(half * KGT + kg) * P::LBO + tid * 16) = v[kg];
        return r;
    }
    // epilogue 1: Q = elu(q)+1, msg = (Q KV) / (Q.Ksum + eps) -> a0[:, C:2C)  (or the message map)
    // kv / ksum hold the state of groups g_base, g_base + 1, ... (global arrays: g_base = 0; the shared-memory copy of the
    // tile's groups: g_base = first group of the tile)
    static __device__ __forceinline__ void epi_attention(const Q& q, const Row& r, uint32_t tmem, int warp, int tid, uint8_t* a0,
                                                         const float* __restrict__ kv, const float* __restrict__ ksum, int g_base = 0,
                                                         int half = 0) {
        const int g = r.g;
#pragma unroll 1
        for (int c0 = half * CH; c0 < half * CH + CH; c0 += G) {
            float qv[G], out[G];
#pragma unroll
            for (int j = 0; j < G; j += 16) {
                float t[16];
                umma::tmem_ld16(umma::tmem_addr(tmem, warp * 32, c0 + j), t);
#pragma unroll
                for (int i = 0; i < 16; ++i) qv[j + i] = elu1(t[i]);
            }
#pragma unroll
            for (int hh = 0; hh < G / DH; ++hh) {
                const int h0 = c0 + hh * DH;             // first channel of this head
                float num[DH], den = kAttnEps;
#pragma unroll
                for (int v = 0; v < DH; ++v) num[v] = 0.f;
                if (g >= 0) {
                    const float* kvh = kv + (size_t)(g - g_base) * (C * DH) + (size_t)h0 * DH;
                    const float* ksh = ksum + (size_t)(g - g_base) * C + h0;
                    umma::f32x2 n2[DH / 2];                  // num as register pairs: one FFMA2 per two outputs
#pragma unroll
                    for (int v = 0; v < DH / 2; ++v) n2[v] = umma::pack2(0.f, 0.f);
#pragma unroll
                    for (int d = 0; d < DH; ++d) {
                        const float qd = qv[hh * DH + d];
                        den = fmaf(qd, ksh[d], den);
                        const umma::f32x2 q2 = umma::pack2(qd, qd);
#pragma unroll
                        for (int v = 0; v < DH; v += 4) {
                            const float4 k4 = *reinterpret_cast<const float4*>(kvh + d * DH + v);
                            n2[v / 2] = umma::fma2(q2, umma::pack2(k4.x, k4.y), n2[v / 2]);
                            n2[v / 2 + 1] = umma::fma2(q2, umma::pack2(k4.z, k4.w), n2[v / 2 + 1]);
                        }
                    }
#pragma unroll
                    for (int v = 0; v < DH / 2; ++v) umma::unpack2(n2[v], num[2 * v], num[2 * v + 1]);
                }
                const float inv = __fdividef(1.f, den);     // MUFU.RCP: the bf16 path does not need the IEEE divide
#pragma unroll
                for (int v = 0; v < DH; ++v) out[hh * DH + v] = num[v] * inv;
            }
#pragma unroll
            for (int j = 0; j < G; j += 8) {
                float o8[8];
#pragma unroll
                for (int i = 0; i < 8; ++i) o8[i] = out[j + i];
                if (kAttnOnly) {
                    if (g >= 0) store8(q, r.ref, c0 + j, o8);
                } else {
                    umma::store_chunk(a0, P::LBO, tid, KG + (c0 + j) / 8, o8);
                }
            }
        }
    }
    // epilogue 1, group-stationary form (hist2image at C = 128: dh = 32, 9-row zone groups).  The row-stationary form above
    // has every row walk its group's whole [C x dh] state - 1024 sixteen-byte loads per row, 4-5 distinct addresses per warp
    // instruction because 9 consecutive rows share a group: 37 us of a 65 us tile pair, bound by LSU wavefronts.  Here
    //   phase A (thread = row half, as before): Q = elu(q)+1 -> a0[:, C:2C) as bf16 (where msg will go), 1 / (Q.Ksum + eps)
    //           per head -> inv[row][head];
    //   phase B (warp = task (group segment of the tile, head), lane = value column c2): the lane loads ITS column of the
    //           head's state once (dh coalesced loads) and applies it to the segment's rows, whose Q chunks are warp-wide
    //           broadcast reads of shared memory; msg overwrites Q in place (the task owns those rows x columns).
    // Each state element is loaded once per group and head instead of once per row; Q passes through bf16.
    static constexpr bool kGroupStationary = C >= 128 && DH == 32 && NT == 2 && !kAttnOnly && IsZonePatch<Q>::value;
    template <class Sync>
    static __device__ __forceinline__ void epi_attention_gs(const Q& q, const Row& r, uint32_t tmem, int wq, int tid, uint8_t* a0,
                                                            const float* __restrict__ kv, const float* __restrict__ ksum, int half,
                                                            float* inv, int64_t row0, int wg, int nwarps, Sync&& sync) {
        const int g = r.g;
        // ---- phase A
#pragma unroll 1
        for (int c0 = half * CH; c0 < half * CH + CH; c0 += DH) {
            float qv[DH];
#pragma unroll
            for (int j = 0; j < DH; j += 16) {
                float t[16];
                umma::tmem_ld16(umma::tmem_addr(tmem, wq * 32, c0 + j), t);
#pragma unroll
                for (int i = 0; i < 16; ++i) qv[j + i] = g >= 0 ? elu1(t[i]) : 0.f;
            }
            float den = kAttnEps;
            if (g >= 0) {
                const float* ksh = ksum + (size_t)g * C + c0;
#pragma unroll
                for (int d = 0; d < DH; d += 4) {
                    const float4 k4 = *reinterpret_cast<const float4*>(ksh + d);
                    den = fmaf(qv[d], k4.x, den); den = fmaf(qv[d + 1], k4.y, den);
                    den = fmaf(qv[d + 2], k4.z, den); den = fmaf(qv[d + 3], k4.w, den);
                }
            }
            inv[tid * NH + c0 / DH] = g >= 0 ? __fdividef(1.f, den) : 0.f;
#pragma unroll
            for (int j = 0; j < DH; j += 8) {
                float o8[8];
#pragma unroll
                for (int i = 0; i < 8; ++i) o8[i] = qv[j + i];
                umma::store_chunk(a0, P::LBO, tid, KG + (c0 + j) / 8, o8);
            }
        }
        sync();                                            // Q and inv of the whole tile are in shared memory
        // ---- phase B
        const int lane = threadIdx.x & 31;
        const int rpg = (int)q.rows_per_group();
        const int64_t left = q.rows - row0;
        const int live = left < 128 ? (int)left : 128;
        if (live > 0) {
            const int g0 = q.group_of_row(row0), g1 = q.group_of_row(row0 + live - 1);
            const int ntask = (g1 - g0 + 1) * NH;
#pragma unroll 1
            for (int t = wg; t < ntask; t += nwarps) {
                const int seg = t / NH, h = t - seg * NH, gg = g0 + seg;
                int ra = (int)((int64_t)gg * rpg - row0), rb = ra + rpg;
                ra = ra < 0 ? 0 : ra;
                rb = rb > live ? live : rb;
                float kvc[DH];                               // this lane's column of the head's dh x dh state
                const float* kp = kv + (size_t)gg * (C * DH) + (size_t)(h * DH) * DH + lane;
#pragma unroll
                for (int d = 0; d < DH; ++d) kvc[d] = kp[d * DH];
                uint8_t* qrow = a0 + (size_t)(KG + h * (DH / 8)) * P::LBO;
                uint8_t* mdst = a0 + (size_t)(KG + (h * DH + lane) / 8) * P::LBO + (lane & 7) * 2;
#pragma unroll 1
                for (int rr = ra; rr < rb; ++rr) {
                    float acc = 0.f;
#pragma unroll
                    for (int j = 0; j < DH / 8; ++j) {
                        float q8[8];
                        unpack8(*reinterpret_cast<const uint4*>(qrow + (size_t)j * P::LBO + rr * 16), q8);
#pragma unroll
                        for (int i = 0; i < 8; ++i) acc = fmaf(q8[i], kvc[j * 8 + i], acc);
                    }
                    acc *= inv[rr * NH + h];
                    __syncwarp();                            // every lane has read row rr's Q chunks of this head
                    *reinterpret_cast<__nv_bfloat16*>(mdst + rr * 16) = __float2bfloat16_rn(acc);
                }
            }
        }
        sync();                                            // msg complete for the tile (the caller hands over to the merge MMA)
    }
    // epilogue 2: LN1(merge) -> a0[:, C:2C)
    template <class Sync>
    static __device__ __forceinline__ void epi_ln1(const cfp_loftr_w& w, uint32_t tmem, int warp, int tid, uint8_t* a0, int half,
                                                   float2* xch, Sync&& sync) {
        float v[CH];
        load_cols<CH>(tmem, warp, half * CH, v);
        if constexpr (NT == 1) layernorm_reg<C>(v, w.ln1_g, w.ln1_b);
        else layernorm_half<C>(v, w.ln1_g + half * CH, w.ln1_b + half * CH, xch, tid, half, sync);
#pragma unroll
        for (int j = 0; j < CH; j += 8) {
            float o8[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) o8[i] = v[j + i];
            umma::store_chunk(a0, P::LBO, tid, KG + (half * CH + j) / 8, o8);
        }
    }
    // epilogue 3: relu(W1 [x|msg]) -> a1 (2C columns)
    static __device__ __forceinline__ void epi_relu(uint32_t tmem, int warp, int tid, uint8_t* a1, int half = 0) {
        constexpr int N = 2 * C / NT;
        umma::tmem_for_each16<N>(umma::tmem_addr(tmem, warp * 32, half * N), [&](int c0, const float (&t)[16]) {
#pragma unroll
            for (int j = 0; j < 16; j += 8) {
                float o8[8];
#pragma unroll
                for (int i = 0; i < 8; ++i) o8[i] = fmaxf(t[j + i], 0.f);
                umma::store_chunk(a1, P::LBO, tid, (half * N + c0 + j) / 8, o8);
            }
        });
    }
    // epilogue 4: x + LN2(W2 hidden) -> scatter through the provider.  x comes from a0[:, 0:C) (kReloadX = false) or is
    // read again through the provider when the MLP hidden has overwritten a0 in place (two-group kernel).
    template <bool kReloadX, class Sync>
    static __device__ __forceinline__ void epi_out(const Q& q, const Row& r, const cfp_loftr_w& w, uint32_t tmem, int warp, int tid,
                                                   const uint8_t* a0, int half, float2* xch, Sync&& sync) {
        const int cb = half * CH;                          // this thread's first column
        if constexpr (kReloadX) {
            // C = 128, two-tile kernel: the residual row is fetched through the provider FIRST (all 16-byte loads in
            // flight at once - issued one by one between the stores they used to serialise on each other, 12-38 us per
            // tile), and LayerNorm walks the accumulator three times in 16-column pieces instead of holding all the
            // values in registers next to them (mean, then centred sum of squares, then normalise + residual + store).
            uint4 xr[KGT];
#pragma unroll
            for (int k = 0; k < KGT; ++k) xr[k] = r.g >= 0 ? load8_bf16(q, r.ref, cb + k * 8) : make_uint4(0u, 0u, 0u, 0u);
            float s = 0.f;
#pragma unroll 1
            for (int c0 = 0; c0 < CH; c0 += 16) {
                float t[16];
                umma::tmem_ld16(umma::tmem_addr(tmem, warp * 32, cb + c0), t);
#pragma unroll
                for (int i = 0; i < 16; ++i) s += t[i];
            }
            float mean = s * (1.f / CH);
            float qs = 0.f;
#pragma unroll 1
            for (int c0 = 0; c0 < CH; c0 += 16) {
                float t[16];
                umma::tmem_ld16(umma::tmem_addr(tmem, warp * 32, cb + c0), t);
#pragma unroll
                for (int i = 0; i < 16; ++i) { const float d = t[i] - mean; qs = fmaf(d, d, qs); }
            }
            float rstd;
            if constexpr (NT == 1) {
                rstd = rsqrtf(qs * (1.f / C) + kLnEps);
            } else {
                const float2 st = ln_combine_halves<C>(mean, qs, xch, tid, half, kLnEps, sync);
                mean -= st.x;
                rstd = st.y;
            }
#pragma unroll
            for (int c0 = 0; c0 < CH; c0 += 16) {
                float t[16];
                umma::tmem_ld16(umma::tmem_addr(tmem, warp * 32, cb + c0), t);
                if (r.g >= 0) {
#pragma unroll
                    for (int h = 0; h < 2; ++h) {
                        const int jl = c0 + 8 * h, j = cb + jl;
                        const float4 g0 = *reinterpret_cast<const float4*>(w.ln2_g + j), g1 = *reinterpret_cast<const float4*>(w.ln2_g + j + 4);
                        const float4 b0 = *reinterpret_cast<const float4*>(w.ln2_b + j), b1 = *reinterpret_cast<const float4*>(w.ln2_b + j + 4);
                        const float gg[8] = {g0.x, g0.y, g0.z, g0.w, g1.x, g1.y, g1.z, g1.w};
                        const float bb[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
                        float x8[8], o8[8];
                        unpack8(xr[jl / 8], x8);
#pragma unroll
                        for (int i = 0; i < 8; ++i) o8[i] = x8[i] + fmaf((t[8 * h + i] - mean) * rstd, gg[i], bb[i]);
                        if constexpr (HasPutSum<Q>::value) {
                            if (q.sums_in_place()) { q.put8_sum(r.ref, j, o8, x8); continue; }
                        }
                        store8(q, r.ref, j, o8);
                    }
                }
            }
            return;
        }
        float v[CH];
        load_cols<CH>(tmem, warp, cb, v);
        if constexpr (NT == 1) layernorm_reg<C>(v, w.ln2_g, w.ln2_b);
        else layernorm_half<C>(v, w.ln2_g + cb, w.ln2_b + cb, xch, tid, half, sync);
        if (r.g >= 0) {
#pragma unroll
            for (int jl = 0; jl < CH; jl += 8) {
                const int j = cb + jl;
                float x8[8], o8[8];
                unpack8(*reinterpret_cast<const uint4*>(a0 + (size_t)(j / 8) * P::LBO + tid * 16), x8);
#pragma unroll
                for (int i = 0; i < 8; ++i) o8[i] = x8[i] + v[jl + i];
                if constexpr (HasPutSum<Q>::value && sizeof(typename Q::R) > 0) {
                    if (q.sums_in_place()) { q.put8_sum(r.ref, j, o8, x8); continue; }
                }
                store8(q, r.ref, j, o8);
            }
        }
    }
};

// D[:, dcol:dcol+C] (+)= A[:, kg0*8 : kg0*8+C] * Wblock^T   (called by a converged warp)
template <int C>
__device__ __forceinline__ void issue_block(uint32_t tmem_d, uint32_t a_addr, uint32_t w_addr, uint32_t idesc, bool acc_first) {
    using P = ChainTC<C>;
    uint64_t ad = umma::smem_desc(a_addr, P::LBO);
    uint64_t wd = umma::smem_desc(w_addr, C * 16);
#pragma unroll
    for (int ks = 0; ks < C / 16; ++ks) {
        umma::mma_bf16(tmem_d, ad, wd, idesc, acc_first || ks > 0);
        ad = umma::desc_advance(ad, 2 * P::LBO);
        wd = umma::desc_advance(wd, 2 * C * 16);
    }
}

template <int C> struct ChainOcc { static constexpr int CTAS = C >= 128 ? 1 : (C == 64 ? 2 : 4); };

// ---------------------------------------------------------------------------------------
// Organisation A (C = 128): three warp roles, TWO 128-token tiles per CTA.  At C = 128 the eight [C x C] weight
// blocks of the chain are 256 KB per tile pass - more than shared memory holds and the dominant cost of a tile when
// they are streamed for 128 rows only.  So a CTA runs two row groups (warps 0-3 and 4-7, thread <-> token <-> TMEM
// lane, one tile each) in lockstep: every weight block brought in by the producer (warp 8) is used by the MMA issuer
// (warp 9) for both tiles back to back (two accumulators of 2C TMEM columns), and the eight row warps run the
// epilogues of the two tiles side by side (two warps per scheduler instead of one).  Each group owns ONE operand
// buffer: the MLP hidden overwrites [x | msg] in place once its MMAs have completed, and the residual x is read again
// through the provider (L2-hot) in the last epilogue.
template <int C, int NH, bool kAttnOnly, class Q, int NT>
__global__ void __launch_bounds__((8 * NT + 2) * 32, 1) loftr_query_tc_kernel(Q q, cfp_loftr_w w, const float* __restrict__ kv,
                                                             const float* __restrict__ ksum, int ntiles, int kv_slots) {
    using P = ChainTC<C>;
    using S = ChainStages<C, NH, kAttnOnly, Q, NT>;
    constexpr int KG = P::KG;
    constexpr int NCHUNK = kAttnOnly ? 1 : 8;
    constexpr int RW = 4 * NT, NRW = 2 * RW;                 // row warps per tile group / per CTA; then producer, MMA issuer
    extern __shared__ __align__(128) uint8_t smem[];
    __shared__ ChainBars bars;
    __shared__ float2 ln_xch[2][NT][128];                    // LayerNorm statistics of split rows, per tile group
    __shared__ float inv_den[2][S::kGroupStationary ? 128 * NH : 1];   // 1 / (Q.Ksum + eps) per (row, head), per tile group
    // the attention-only chain (DAPM) stages x only: half an operand buffer per tile, and the shared memory it does not
    // ask for stays L1 - where its per-frame attention state (16 KB a group at C = 128) is read from
    constexpr size_t ABUF = kAttnOnly ? (size_t)KG * P::LBO : (size_t)P::ABUF;
    uint8_t* ring = smem + 2 * ABUF;
    // kv_slots > 0 (groups of a frame - GSA, DAPM - where a tile pair touches two of them and their state fits beside
    // the operand buffers): the pair's group states are brought into shared memory by two bulk copies while x is staged and
    // q is projected, and the attention epilogue reads them with LDS (as the C <= 64 chains do)
    float* kvs = reinterpret_cast<float*>(ring + (size_t)P::NSLOT * P::SLOT);
    float* kss = kvs + (size_t)kv_slots * (C * S::DH);
    const int tid = threadIdx.x, warp = umma::warp_idx_sync();
    // Tiles of round `it`: group g of CTA c takes tile  it * 2 G + 2 c + g - a CTA owns two neighbouring tiles.  A group
    // without a tile (the last one when ntiles is odd) only keeps the hand-over protocol going (arrivals, barrier), and its
    // MMAs are not issued.
    const int round_tiles = 2 * (int)gridDim.x;
    const int first0 = (int)blockIdx.x * 2;

    if (tid == 0) {
        for (int i = 0; i < P::NSLOT; ++i) { umma::mbar_init(&bars.full[i], 1); umma::mbar_init(&bars.empty[i], 1); }
        umma::mbar_init(&bars.a_ready, NRW * 32);
        umma::mbar_init(&bars.acc_ready, 1);
        umma::mbar_init(&bars.kv_full, 1);
        umma::fence_mbar_init();
    }
    if (warp == NRW) umma::tmem_alloc(&bars.tmem_slot, 512);
    umma::fence_before_sync();
    __syncthreads();
    umma::fence_after_sync();

    if (warp < NRW) {
        pdl_wait();                       // rows and attention state come from the previous kernels of the stream
        const int grp = warp / RW, half = (warp % RW) >> 2, wq = warp & 3, tid_g = tid & 127;
        uint8_t* a0 = smem + (size_t)grp * ABUF;             // [x | msg, then LN1(merge(msg))], then the MLP hidden
        const uint32_t tmem = bars.tmem_slot + grp * 256;
        float2* xch = &ln_xch[grp][0][0];
        auto group_sync = [&]() { asm volatile("bar.sync %0, %1;\n" ::"r"(2 + grp), "n"(RW * 32) : "memory"); };
        uint32_t ph = 0, kvph = 0;
        auto hand_over = [&]() {          // operands staged / accumulator consumed -> MMA warp; then wait for its result
            umma::fence_async_smem();
            umma::fence_before_sync();
            mbar_arrive(&bars.a_ready);
            umma::mbar_wait(&bars.acc_ready, ph); ph ^= 1;
            umma::fence_after_sync();
        };
        for (int first = first0; first < ntiles; first += round_tiles) {
            const int tile = first + grp;
            int g_first = 0;
            if (kv_slots > 0) {
                const int64_t r_first = (int64_t)first * 128;
                const int64_t r_last = r_first + 255 < q.rows ? r_first + 255 : q.rows - 1;
                g_first = q.group_of_row(r_first);
                if (tid == 0) {                              // every row thread is past the previous pair's epilogue (bar.sync 1)
                    const uint32_t ng = (uint32_t)(q.group_of_row(r_last) - g_first + 1);
                    umma::mbar_expect_tx(&bars.kv_full, ng * (uint32_t)((C * S::DH + C) * sizeof(float)));
                    umma::bulk_g2s(kvs, kv + (size_t)g_first * (C * S::DH), ng * (uint32_t)(C * S::DH * sizeof(float)), &bars.kv_full);
                    umma::bulk_g2s(kss, ksum + (size_t)g_first * C, ng * (uint32_t)(C * sizeof(float)), &bars.kv_full);
                }
            }
            if (tile >= ntiles) {                            // (group 1 only) no tile this round: keep the protocol going
#pragma unroll 1
                for (int i = 0; i < (kAttnOnly ? 1 : 4); ++i) hand_over();
                umma::fence_before_sync();
                asm volatile("bar.sync 1, %0;\n" ::"n"(NRW * 32) : "memory");
                continue;
            }
            const int64_t row0 = (int64_t)tile * 128;
            [[maybe_unused]] const int dbg_it = 1 - (first - first0) / round_tiles;      // marks on the FIRST pair of CTA 5
            CFP_CHAIN_MARK(0, dbg_it);
            const typename S::Row r = S::stage_x(q, row0, tid_g, a0, half);
            CFP_CHAIN_MARK(1, dbg_it);
            hand_over();
            CFP_CHAIN_MARK(2, dbg_it);
            if constexpr (S::kGroupStationary) {
                S::epi_attention_gs(q, r, tmem, wq, tid_g, a0, kv, ksum, half, &inv_den[grp][0], row0, warp % RW, RW, group_sync);
            } else if (kv_slots > 0) {
                umma::mbar_wait(&bars.kv_full, kvph); kvph ^= 1;
                S::epi_attention(q, r, tmem, wq, tid_g, a0, kvs, kss, g_first, half);
            } else {
                S::epi_attention(q, r, tmem, wq, tid_g, a0, kv, ksum, 0, half);
            }
            CFP_CHAIN_MARK(3, dbg_it);
            if (!kAttnOnly) {
                hand_over();
                CFP_CHAIN_MARK(4, dbg_it);
                S::epi_ln1(w, tmem, wq, tid_g, a0, half, xch, group_sync);
                CFP_CHAIN_MARK(5, dbg_it);
                hand_over();
                CFP_CHAIN_MARK(6, dbg_it);
                S::epi_relu(tmem, wq, tid_g, a0, half);       // in place: the W1 MMAs have consumed [x | LN1]
                CFP_CHAIN_MARK(7, dbg_it);
                hand_over();
                CFP_CHAIN_MARK(8, dbg_it);
                S::template epi_out<true>(q, r, w, tmem, wq, tid_g, a0, half, xch, group_sync);
                CFP_CHAIN_MARK(9, dbg_it);
            }
            umma::fence_before_sync();
            asm volatile("bar.sync 1, %0;\n" ::"n"(NRW * 32) : "memory");  // every row is done with a0 / the accumulators before the next pair
        }
    } else if (warp == NRW) {
        const bf16* wsrc = reinterpret_cast<const bf16*>(w.tc);
        int cc = 0;
        for (int first = first0; first < ntiles; first += round_tiles)
            for (int c = 0; c < NCHUNK; ++c, ++cc) {
                const int slot = cc % P::NSLOT, round = cc / P::NSLOT;
                if (round > 0) umma::mbar_wait(&bars.empty[slot], (round - 1) & 1);
                umma::bulk_load(ring + (size_t)slot * P::SLOT, wsrc + (size_t)c * C * C, P::SLOT, &bars.full[slot]);
            }
    } else {
        const uint32_t idesc = umma::idesc_bf16(128, C);
        const uint32_t a0s = umma::smem_u32(smem), rs = umma::smem_u32(ring);
        const uint32_t tmem = bars.tmem_slot;
        uint32_t ph = 0;
        int cc = 0;
        // one weight block, both tiles: D_g[:, dcol:dcol+C] (+)= A_g[:, kg0*8 : kg0*8+C] * W^T
        int nlive = 2;
        auto block = [&](int kg0, int dcol, bool acc_first) {
            const int slot = cc % P::NSLOT, round = cc / P::NSLOT;
            umma::mbar_wait(&bars.full[slot], round & 1);
            umma::fence_after_sync();
#pragma unroll
            for (int g2 = 0; g2 < 2; ++g2)
                if (g2 < nlive)
                    issue_block<C>(tmem + g2 * 256 + dcol, a0s + g2 * (uint32_t)ABUF + kg0 * P::LBO, rs + slot * P::SLOT, idesc, acc_first);
            umma::commit(&bars.empty[slot]);
            ++cc;
        };
        auto wait_a = [&]() { umma::mbar_wait(&bars.a_ready, ph); ph ^= 1; umma::fence_after_sync(); };
        for (int first = first0; first < ntiles; first += round_tiles) {
            nlive = first + 1 < ntiles ? 2 : 1;
            wait_a();
            block(0, 0, false);                            // q
            umma::commit(&bars.acc_ready);
            if (kAttnOnly) continue;
            wait_a();
            block(KG, 0, false);                           // merge: msg sits in a0[:, C:2C)
            umma::commit(&bars.acc_ready);
            wait_a();
            block(0, 0, false);                            // W1 quadrants: (n0,k0) (n0,k1) (n1,k0) (n1,k1)
            block(KG, 0, true);
            block(0, C, false);
            block(KG, C, true);
            umma::commit(&bars.acc_ready);
            wait_a();
            block(0, 0, false);                            // W2 K-halves (hidden sits in a0[:, 0:2C))
            block(KG, 0, true);
            umma::commit(&bars.acc_ready);
        }
    }
    pdl_trigger();                         // this CTA's work is done: the next kernel of the stream may start its prologue
    __syncthreads();
    if (warp == NRW) {
        umma::fence_after_sync();
        umma::tmem_dealloc(bars.tmem_slot, 512);
    }
}

// ---------------------------------------------------------------------------------------
// Organisation B (C <= 64): one role.  The 128 row threads ARE the CTA; after a block barrier warp 0
// issues the stage's MMAs itself and schedules the weight-block prefetches at the points where the
// ring slots are known to be free (right after an accumulator wait), so there are no service warps
// (their registers bought nothing), no empty-barriers and one mbarrier hand-off per stage instead
// of two.  More CTAs fit per SM, which is what these latency-bound chains need.
// (measured: an in-place hidden buffer + register caps for 8 / 3 CTAs per SM made these kernels 5-25 % SLOWER - they
// are not occupancy-bound)
template <int C> struct MonoOcc { static constexpr int CTAS = C == 32 ? 5 : 2; };
struct MonoBars {
    uint64_t full[4], acc_ready, kv_full;
    uint32_t tmem_slot;
};

template <int C, int NH, bool kAttnOnly, class Q, int NT>
__global__ void __launch_bounds__(128 * NT, MonoOcc<C>::CTAS) loftr_query_mono_kernel(Q q, cfp_loftr_w w, const float* __restrict__ kv,
                                                                const float* __restrict__ ksum, int ntiles, int kv_slots) {
    using P = ChainTC<C>;
    using S = ChainStages<C, NH, kAttnOnly, Q, NT>;
    constexpr int KG = P::KG, NB = kAttnOnly ? 1 : 8;      // weight blocks per tile
    extern __shared__ __align__(128) uint8_t smem[];
    __shared__ MonoBars bars;
    __shared__ float2 ln_xch[NT][128];                      // LayerNorm statistics of split rows
    uint8_t* a0 = smem;
    uint8_t* a1 = a0 + P::ABUF;
    uint8_t* ring = a1 + (kAttnOnly ? 0 : P::ABUF);        // 4 slots
    // attention state of the groups a tile touches (kv_slots of them; 0 = read it from global memory): brought in by two
    // bulk copies while the q projection runs - the per-row loads of the attention epilogue then hit shared memory
    // instead of stalling every FMA chain on an L2 round trip
    float* kvs = reinterpret_cast<float*>(ring + 4 * (size_t)P::SLOT);
    float* kss = kvs + (size_t)kv_slots * (C * S::DH);
    const int warp = umma::warp_idx_sync();
    const int tid = threadIdx.x & 127, half = warp >> 2, wq = warp & 3;   // row of the tile (= TMEM lane), which of its NT threads
    float2* xch = &ln_xch[0][0];
    auto cta_sync = [&]() { __syncthreads(); };

    if (threadIdx.x == 0) {
        for (int i = 0; i < 4; ++i) umma::mbar_init(&bars.full[i], 1);
        umma::mbar_init(&bars.acc_ready, 1);
        umma::mbar_init(&bars.kv_full, 1);
        umma::fence_mbar_init();
    }
    if (warp == 0) umma::tmem_alloc(&bars.tmem_slot, P::TMEM_COLS);
    umma::fence_before_sync();
    __syncthreads();
    umma::fence_after_sync();
    const uint32_t tmem = bars.tmem_slot;
    const uint32_t idesc = umma::idesc_bf16(128, C);
    const uint32_t a0s = umma::smem_u32(a0), a1s = umma::smem_u32(a1), rs = umma::smem_u32(ring);
    const bf16* wsrc = reinterpret_cast<const bf16*>(w.tc);
    const int my_tiles = blockIdx.x < ntiles ? (ntiles - 1 - blockIdx.x) / gridDim.x + 1 : 0;
    const long total_blocks = (long)my_tiles * NB;

    // weight block `seq` (running over this CTA's tiles) lives in slot seq % 4, parity (seq / 4) & 1
    auto prefetch = [&](long seq) {                          // warp 0 only, converged
        if (seq < total_blocks) {
            const int slot = (int)(seq & 3);
            umma::bulk_load(ring + (size_t)slot * P::SLOT, wsrc + (size_t)(seq % NB) * C * C, P::SLOT, &bars.full[slot]);
        }
    };
    auto block = [&](long seq, uint32_t a_addr, int dcol, bool acc_first) {   // warp 0 only
        const int slot = (int)(seq & 3);
        umma::mbar_wait(&bars.full[slot], (uint32_t)((seq >> 2) & 1));
        umma::fence_after_sync();
        issue_block<C>(tmem + dcol, a_addr, rs + slot * P::SLOT, idesc, acc_first);
    };
    uint32_t ph = 0;
    // operands staged by all rows -> barrier -> warp 0 issues `mmas` -> everyone waits for the accumulator
    auto stage = [&](auto mmas) {
        umma::fence_async_smem();
        umma::fence_before_sync();
        __syncthreads();
        if (warp == 0) {
            umma::fence_after_sync();
            mmas();
            umma::commit(&bars.acc_ready);
        }
        umma::mbar_wait(&bars.acc_ready, ph); ph ^= 1;
        umma::fence_after_sync();
    };

    if (warp == 0)
        for (long s0 = 0; s0 < 4; ++s0) prefetch(s0);       // weights: not produced by the previous kernel
    pdl_wait();
    long base = 0;                                          // sequence number of this tile's first block
    uint32_t kvph = 0;
    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x, base += NB) {
        const int64_t row0 = (int64_t)tile * 128;
        [[maybe_unused]] const int dbg_it = (tile - (int)blockIdx.x) / (int)gridDim.x;
        CFP_CHAIN_MARK(0, dbg_it);
        const typename S::Row r = S::stage_x(q, row0, tid, a0, half);
        CFP_CHAIN_MARK(1, dbg_it);
        const int g_first = kv_slots > 0 ? q.group_of_row(row0) : 0;
        stage([&] {                                                                        // q
            if (kv_slots > 0) {            // every row is past the previous tile's attention epilogue (stage barrier)
                const int64_t last = row0 + 127 < q.rows ? row0 + 127 : q.rows - 1;
                const uint32_t ng = (uint32_t)(q.group_of_row(last) - g_first + 1);
                if (umma::elect_one()) {
                    umma::mbar_expect_tx(&bars.kv_full, ng * (uint32_t)((C * S::DH + C) * sizeof(float)));
                    umma::bulk_g2s(kvs, kv + (size_t)g_first * (C * S::DH), ng * (uint32_t)(C * S::DH * sizeof(float)), &bars.kv_full);
                    umma::bulk_g2s(kss, ksum + (size_t)g_first * C, ng * (uint32_t)(C * sizeof(float)), &bars.kv_full);
                }
            }
            block(base + 0, a0s, 0, false);
        });
        // two instantiations of the epilogue, one per address space of the state: selected through one pointer variable
        // its loads were generic (LD.E) - also when they hit the shared-memory copy - instead of LDS / LDG
        auto attention = [&]() {
            if (kv_slots > 0) {
                umma::mbar_wait(&bars.kv_full, kvph); kvph ^= 1;
                S::epi_attention(q, r, tmem, wq, tid, a0, kvs, kss, g_first, half);
            } else {
                S::epi_attention(q, r, tmem, wq, tid, a0, kv, ksum, 0, half);
            }
        };
        if (kAttnOnly) {
            if (warp == 0) prefetch(base + 4);               // slot of block `base` is free again
            attention();
            continue;                                        // next stage() barrier orders a0 / TMEM reuse
        }
        CFP_CHAIN_MARK(2, dbg_it);
        attention();
        CFP_CHAIN_MARK(3, dbg_it);
        stage([&] { block(base + 1, a0s + KG * P::LBO, 0, false); });                     // merge
        CFP_CHAIN_MARK(4, dbg_it);
        if (warp == 0) { prefetch(base + 4); prefetch(base + 5); }                        // blocks 0,1 consumed
        S::epi_ln1(w, tmem, wq, tid, a0, half, xch, cta_sync);
        CFP_CHAIN_MARK(5, dbg_it);
        stage([&] {                                                                        // W1 quadrants
            block(base + 2, a0s, 0, false);
            block(base + 3, a0s + KG * P::LBO, 0, true);
            block(base + 4, a0s, C, false);
            block(base + 5, a0s + KG * P::LBO, C, true);
        });
        if (warp == 0) { prefetch(base + 6); prefetch(base + 7); prefetch(base + 8); prefetch(base + 9); }
        CFP_CHAIN_MARK(6, dbg_it);
        S::epi_relu(tmem, wq, tid, a1, half);
        CFP_CHAIN_MARK(7, dbg_it);
        stage([&] {                                                                        // W2 K-halves
            block(base + 6, a1s, 0, false);
            block(base + 7, a1s + KG * P::LBO, 0, true);
        });
        if (warp == 0) { prefetch(base + 10); prefetch(base + 11); }
        CFP_CHAIN_MARK(8, dbg_it);
        S::template epi_out<false>(q, r, w, tmem, wq, tid, a0, half, xch, cta_sync);
        CFP_CHAIN_MARK(9, dbg_it);
        // the next tile's stage_x overwrites a0[:, 0:C), which epi_out of other rows may still read
        __syncthreads();
    }
    pdl_trigger();                         // this CTA's work is done: the next kernel of the stream may start its prologue
    umma::fence_before_sync();
    __syncthreads();
    if (warp == 0) {
        umma::fence_after_sync();
        umma::tmem_dealloc(tmem, P::TMEM_COLS);
    }
}

template <int C, int NH, bool kAttnOnly, class Q>
static int run_query_tc(const char* name, const Q& q, const cfp_loftr_w& w, const float* kv, const float* ksum,
                        cudaStream_t st) {
    using P = ChainTC<C>;
    constexpr int NT = C >= 64 ? 2 : 1;      // threads per token row (see ChainStages): two win by 10-17 % at C >= 64
    CFP_REQUIRE(w.tc != nullptr, "%s: bf16 path needs the packed tensor-core weights (cfp_loftr_w.tc)", name);
    const int64_t ntiles = (q.rows + 127) / 128;
    CFP_REQUIRE(q.rows < ((int64_t)1 << 31), "%s: %lld rows exceed the 32-bit row index", name, (long long)q.rows);
    if constexpr (C <= 64) {
        constexpr size_t smem0 = (kAttnOnly ? 1 : 2) * (size_t)P::ABUF + 4 * (size_t)P::SLOT;
        const int per_sm = MonoOcc<C>::CTAS;
        // shared-memory copy of the attention state of one tile's groups, if it fits beside the occupancy target
        constexpr int DH = C / NH;
        const uint32_t rpg = q.rows_per_group();
        int kv_slots = (int)((128 + rpg - 2) / rpg + 1);
        const size_t kv_bytes = (size_t)kv_slots * (C * DH + C) * sizeof(float);
        if ((smem0 + kv_bytes + 1024) * per_sm > 227 * 1024) kv_slots = 0;
        const size_t smem = smem0 + (kv_slots > 0 ? kv_bytes : 0);
        const int grid = (int)(ntiles < sm_count() * per_sm ? ntiles : sm_count() * per_sm);
        auto k = loftr_query_mono_kernel<C, NH, kAttnOnly, Q, NT>;
        if (int e = set_smem(k, smem)) return e;
        launch_pdl(k, grid, 128 * NT, smem, st, q, w, kv, ksum, (int)ntiles, kv_slots);
#ifdef CFP_DEBUG_TIMING
        {
            cudaStreamSynchronize(st);
            unsigned long long h[16] = {0};
            cudaMemcpyFromSymbol(h, g_chain_dbg, sizeof(h));
            fprintf(stderr, "%s (C=%d, %d CTAs, %lld tiles) 2nd tile of CTA 5, ns since tile start: stage_x %llu | q-acc %llu | attn %llu | merge-acc %llu | ln1 %llu | W1-acc %llu | relu %llu | W2-acc %llu | out %llu\n",
                    name, C, grid, (long long)ntiles, h[1] - h[0], h[2] - h[0], h[3] - h[0], h[4] - h[0], h[5] - h[0], h[6] - h[0], h[7] - h[0], h[8] - h[0], h[9] - h[0]);
        }
#endif
    } else {
        // two neighbouring tiles per CTA, also in a thin last round: spreading that round one tile per CTA over all SMs was
        // measured slower with the three levels concurrent (3.85 -> 3.91 ms per step)
        const int64_t npairs = (ntiles + 1) / 2;
        const int grid = (int)(npairs < sm_count() ? npairs : sm_count());
        auto k = loftr_query_tc_kernel<C, NH, kAttnOnly, Q, NT>;
        constexpr size_t smem0 = kAttnOnly ? 2 * (size_t)P::KG * P::LBO + (size_t)P::NSLOT * P::SLOT : P::SMEM;
        // shared-memory copy of the group states a tile pair (256 consecutive rows) touches, where it fits (groups of a frame)
        constexpr int DH = C / NH;
        const uint32_t rpg = q.rows_per_group();
        int kv_slots = (int)((256 + rpg - 2) / rpg + 1);
        const size_t kv_bytes = (size_t)kv_slots * (C * DH + C) * sizeof(float);
        if (smem0 + kv_bytes + 1024 > 227 * 1024) kv_slots = 0;
        const size_t smem = smem0 + (kv_slots > 0 ? kv_bytes : 0);
        if (int e = set_smem(k, smem)) return e;
        launch_pdl(k, grid, (8 * NT + 2) * 32, smem, st, q, w, kv, ksum, (int)ntiles, kv_slots);
#ifdef CFP_DEBUG_TIMING
        {
            cudaStreamSynchronize(st);
            unsigned long long h[16] = {0};
            cudaMemcpyFromSymbol(h, g_chain_dbg, sizeof(h));
            fprintf(stderr, "%s (C=%d, %d CTAs, %lld tiles, two per CTA) 1st pair of CTA 5, ns since start: stage_x %llu | q-acc %llu | attn %llu | merge-acc %llu | ln1 %llu | W1-acc %llu | relu %llu | W2-acc %llu | out %llu\n",
                    name, C, grid, (long long)ntiles, h[1] - h[0], h[2] - h[0], h[3] - h[0], h[4] - h[0], h[5] - h[0], h[6] - h[0], h[7] - h[0], h[8] - h[0], h[9] - h[0]);
        }
#endif
    }
    return check_launch(name);
}

// =====================================================================================
// LKPM pointwise half on tensor cores (convnext.py:49-58):
//   out = x + W2 GELU(W1 LN(y) + b1) + b2,   W1: C -> 4C, W2: 4C -> C
// The 4C hidden dimension is walked in 128-wide slices j (1, 2 or 4 of them): h_j = [LNhat(y) | 1] W1_j^T
// (TMEM cols [0,128)), GELU in registers -> fp16 A tile, out += [GELU(h_j) | 1] W2_j^T; the out accumulator stays
// in TMEM across slices (for C = 32 there is a single slice and out reuses the h columns).  MMA2_j and
// MMA1_{j+1} are issued back to back, so the tensor pipe works on slice j+1 while the row threads
// apply GELU to slice j.  Weight blocks in consumption order: W1_0, W2_0, W1_1, ...
// GELU: tanh form evaluated as packed fp16x2 (tanh.approx.f16x2): |dev| <= 5e-4 from the erf form,
// i.e. below 1/8 bf16 ulp of the result for |y| >= 0.06; the epilogue is ALU-bound at small C and this
// is ~3x fewer instructions than erff.
template <int C> struct MlpTC {
    static constexpr int NS = 128;                       // hidden slice width
    static constexpr int NSL = 4 * C / NS;               // slices: 1, 2, 4
    // Both GEMMs carry their bias inside the contraction: the A operands have one extra 16-column K step whose first
    // column is 1 (written once per CTA), the weight blocks one extra K step whose first column is the bias.  The
    // LayerNorm affine is folded into W1 / b1 by the host.  So the epilogues are pure: normalise | GELU | + residual.
    static constexpr int K1 = C + 16;                    // GEMM1: [128 x K1] x W1_j^T (N = 128), bf16
    static constexpr int K2 = NS + 16;                   // GEMM2: [128 x K2] x W2_j^T (N = C), fp16
    static constexpr int BLK1 = NS * K1 * 2, BLK2 = C * K2 * 2;
    static constexpr int BLK = BLK1 > BLK2 ? BLK1 : BLK2;   // ring slot / packed block stride (bytes)
    static constexpr int NBLK = 2 * NSL;                 // blocks per tile
    static constexpr int NSLOT = 2;                      // (4 slots at C = 64 cost the second CTA per SM: 140 KB of shared memory)
    static constexpr int OUT_COL = NSL == 1 ? 0 : NS;    // out accumulator columns
    static constexpr int TMEM_COLS = NSL == 1 ? 128 : 256;
    static constexpr int G0 = K1 / 8, G1 = K2 / 8;       // 16-byte k-groups of the two A buffers
    static constexpr size_t SMEM = (size_t)(G0 + G1) * ChainTC<C>::LBO + (size_t)NSLOT * BLK;
};

// GELU (tanh form) of two fp32 values as packed fp16: the second GEMM consumes fp16 (more mantissa than bf16, and no
// conversion back through fp32).
__device__ __forceinline__ uint32_t gelu_tanh_h2(float x0, float x1) {
    const __half2 h = __floats2half2_rn(x0, x1);
    const __half2 k0 = __float2half2_rn(0.7978845608f), k1 = __float2half2_rn(0.0356774081f);
    const __half2 inner = __hmul2(h, __hfma2(__hmul2(h, h), k1, k0));
    uint32_t ti = *reinterpret_cast<const uint32_t*>(&inner), to;
    asm("tanh.approx.f16x2 %0, %1;\n" : "=r"(to) : "r"(ti));
    const __half2 t = *reinterpret_cast<const __half2*>(&to);
    const __half2 hh = __hmul2(h, __float2half2_rn(0.5f));
    const __half2 r = __hfma2(hh, t, hh);
    return *reinterpret_cast<const uint32_t*>(&r);
}

template <int C>
__global__ void __launch_bounds__(192) lkpm_mlp_tc_kernel(bf16* __restrict__ feat0, const bf16* __restrict__ y,
                                                          int64_t rows, int planar_n, int planar_w, int planar_pitch, cfp_lkpm_w w, int ntiles,
                                                          FastDiv dPn, FastDiv dPw) {
    using P = ChainTC<C>;
    using M = MlpTC<C>;
    constexpr int KG = P::KG;
    extern __shared__ __align__(128) uint8_t smem[];
    __shared__ ChainBars bars;
    uint8_t* a0 = smem;                          // [LNhat(y) | 1 0..0]   [G0][129][16 B]  bf16
    uint8_t* a1 = a0 + M::G0 * P::LBO;           // [GELU(h_j) | 1 0..0]  [G1][129][16 B]  fp16
    uint8_t* ring = a1 + M::G1 * P::LBO;
    const int tid = threadIdx.x, warp = umma::warp_idx_sync();

    if (tid == 0) {
        for (int i = 0; i < M::NSLOT; ++i) { umma::mbar_init(&bars.full[i], 1); umma::mbar_init(&bars.empty[i], 1); }
        umma::mbar_init(&bars.a_ready, 128);
        umma::mbar_init(&bars.acc_ready, 1);
        umma::fence_mbar_init();
    }
    if (warp == 4) umma::tmem_alloc(&bars.tmem_slot, M::TMEM_COLS);
    if (warp < 4) {                              // the constant bias columns of the two A operands (row `tid`)
        *reinterpret_cast<uint4*>(a0 + (size_t)KG * P::LBO + tid * 16) = make_uint4(0x3F80u, 0u, 0u, 0u);        // bf16 1.0
        *reinterpret_cast<uint4*>(a0 + (size_t)(KG + 1) * P::LBO + tid * 16) = make_uint4(0u, 0u, 0u, 0u);
        *reinterpret_cast<uint4*>(a1 + (size_t)(M::NS / 8) * P::LBO + tid * 16) = make_uint4(0x3C00u, 0u, 0u, 0u);  // fp16 1.0
        *reinterpret_cast<uint4*>(a1 + (size_t)(M::NS / 8 + 1) * P::LBO + tid * 16) = make_uint4(0u, 0u, 0u, 0u);
    }
    umma::fence_async_smem();
    umma::fence_before_sync();
    __syncthreads();
    umma::fence_after_sync();
    const uint32_t tmem = bars.tmem_slot;

    if (warp < 4) {
        pdl_wait();
        uint32_t ph = 0;
        for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
            const int64_t row = (int64_t)tile * 128 + tid;
            // residual x of the row, fetched now so that the last epilogue does not stall on it (registers permitting)
            constexpr bool kPrefetchX = C <= 64;
            uint4 xres[kPrefetchX ? C / 8 : 1];
            if constexpr (kPrefetchX) {
#pragma unroll
                for (int j = 0; j < C / 8; ++j)
                    xres[j] = row < rows ? *reinterpret_cast<const uint4*>(feat0 + row * C + j * 8) : make_uint4(0u, 0u, 0u, 0u);
            }
            {   // channels-last LayerNorm (eps 1e-6) of row `tid` -> a0
                float v[C];
                if (planar_n > 0) {
                    // planar dwconv output [frame][C][H][pitch]: lanes are consecutive tokens, so each of the C two-byte
                    // loads of a warp is (mostly) one contiguous 64-byte segment
                    uint32_t fr, n, yy, xx;                       // rows < 2^31; multiply-high divisions
                    dPn.divmod((uint32_t)row, fr, n);
                    dPw.divmod(n, yy, xx);
                    const size_t cstride = (size_t)(planar_n / planar_w) * planar_pitch;
                    const uint16_t* p = reinterpret_cast<const uint16_t*>(y) + (size_t)fr * C * cstride + (size_t)yy * planar_pitch + xx;
#pragma unroll
                    for (int c = 0; c < C; ++c)
                        v[c] = row < rows ? __uint_as_float((uint32_t)__ldg(p + (size_t)c * cstride) << 16) : 0.f;
                } else {
#pragma unroll
                    for (int j = 0; j < C; j += 8) {
                        float t[8];
                        uint4 u = make_uint4(0u, 0u, 0u, 0u);
                        if (row < rows) u = *reinterpret_cast<const uint4*>(y + row * C + j);
                        unpack8(u, t);
#pragma unroll
                        for (int i = 0; i < 8; ++i) v[j + i] = t[i];
                    }
                }
                using namespace umma;                            // packed fp32x2: one instruction per channel pair
                f32x2 p2[C / 2];
                f32x2 s2 = pack2(0.f, 0.f);
#pragma unroll
                for (int i = 0; i < C / 2; ++i) { p2[i] = pack2(v[2 * i], v[2 * i + 1]); s2 = add2(s2, p2[i]); }
                float s_lo, s_hi;
                unpack2(s2, s_lo, s_hi);
                const float mean = (s_lo + s_hi) * (1.f / C);
                const f32x2 nm = pack2(-mean, -mean);
                f32x2 q2 = pack2(0.f, 0.f);
#pragma unroll
                for (int i = 0; i < C / 2; ++i) { p2[i] = add2(p2[i], nm); q2 = fma2(p2[i], p2[i], q2); }
                float q_lo, q_hi;
                unpack2(q2, q_lo, q_hi);
                const float rstd = rsqrtf((q_lo + q_hi) * (1.f / C) + kLkpmLnEps);
                const f32x2 r2 = pack2(rstd, rstd);
#pragma unroll
                for (int j = 0; j < C; j += 8) {                 // gamma / beta live in W1 / b1 (host fold)
                    float o8[8];
#pragma unroll
                    for (int k = 0; k < 4; ++k) unpack2(mul2(p2[j / 2 + k], r2), o8[2 * k], o8[2 * k + 1]);
                    umma::store_chunk(a0, P::LBO, tid, j / 8, o8);
                }
            }
            umma::fence_async_smem();
            mbar_arrive(&bars.a_ready);
#pragma unroll 1
            for (int js = 0; js < M::NSL; ++js) {                // hidden slice js: GELU(h + b1) -> a1
                umma::mbar_wait(&bars.acc_ready, ph); ph ^= 1;
                umma::fence_after_sync();
                umma::tmem_for_each16<M::NS>(umma::tmem_addr(tmem, warp * 32, 0), [&](int c0, const float (&t)[16]) {
#pragma unroll
                    for (int j = 0; j < 16; j += 8) {
                        uint4 u;
                        u.x = gelu_tanh_h2(t[j + 0], t[j + 1]);
                        u.y = gelu_tanh_h2(t[j + 2], t[j + 3]);
                        u.z = gelu_tanh_h2(t[j + 4], t[j + 5]);
                        u.w = gelu_tanh_h2(t[j + 6], t[j + 7]);
                        *reinterpret_cast<uint4*>(a1 + (size_t)((c0 + j) / 8) * P::LBO + tid * 16) = u;
                    }
                });
                umma::fence_async_smem();
                umma::fence_before_sync();
                mbar_arrive(&bars.a_ready);
            }
            umma::mbar_wait(&bars.acc_ready, ph); ph ^= 1;       // out accumulator complete
            umma::fence_after_sync();
#pragma unroll
            for (int c0 = 0; c0 < C; c0 += 16) {
                float t[16];
                umma::tmem_ld16(umma::tmem_addr(tmem, warp * 32, M::OUT_COL + c0), t);
                if (row < rows) {
#pragma unroll
                    for (int j = 0; j < 16; j += 8) {
                        bf16* p = feat0 + row * C + c0 + j;
                        float x8[8];
                        if constexpr (kPrefetchX) unpack8(xres[(c0 + j) / 8], x8);
                        else unpack8(*reinterpret_cast<const uint4*>(p), x8);
                        uint4 u;
                        u.x = umma::pack_bf16(x8[0] + t[j + 0], x8[1] + t[j + 1]);
                        u.y = umma::pack_bf16(x8[2] + t[j + 2], x8[3] + t[j + 3]);
                        u.z = umma::pack_bf16(x8[4] + t[j + 4], x8[5] + t[j + 5]);
                        u.w = umma::pack_bf16(x8[6] + t[j + 6], x8[7] + t[j + 7]);
                        *reinterpret_cast<uint4*>(p) = u;
                    }
                }
            }
            umma::fence_before_sync();
            rows_sync();
        }
    } else if (warp == 4) {
        const bf16* wsrc = reinterpret_cast<const bf16*>(w.tc);
        int cc = 0;
        for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x)
            for (int c = 0; c < M::NBLK; ++c, ++cc) {
                const int slot = cc % M::NSLOT, round = cc / M::NSLOT;
                if (round > 0) umma::mbar_wait(&bars.empty[slot], (round - 1) & 1);
                umma::bulk_load(ring + (size_t)slot * M::BLK, wsrc + (size_t)c * (M::BLK / 2), M::BLK, &bars.full[slot]);
            }
    } else {
        // GEMM1: bf16 x bf16; GEMM2: fp16 x fp16 (a_format = b_format = 0 in the instruction descriptor)
        const uint32_t idesc1 = umma::idesc_bf16(128, M::NS);
        const uint32_t idesc2 = umma::idesc_bf16(128, C) & ~((7u << 7) | (7u << 10));
        const uint32_t a0s = umma::smem_u32(a0), a1s = umma::smem_u32(a1), rs = umma::smem_u32(ring);
        uint32_t ph = 0;
        int cc = 0;
        // h (+)= A0[128 x K1] * W1_j^T (N = 128)   |   out (+)= A1[128 x K2] * W2_j^T (N = C)
        auto block = [&](bool first_gemm, bool acc_first) {
            const int slot = cc % M::NSLOT, round = cc / M::NSLOT;
            umma::mbar_wait(&bars.full[slot], round & 1);
            umma::fence_after_sync();
            const uint32_t lbo_b = (first_gemm ? M::NS : C) * 16;
            uint64_t ad = umma::smem_desc(first_gemm ? a0s : a1s, P::LBO);
            uint64_t wd = umma::smem_desc(rs + slot * M::BLK, lbo_b);
            const int nk = (first_gemm ? M::K1 : M::K2) / 16;
            for (int ks = 0; ks < nk; ++ks) {
                umma::mma_bf16(tmem + (first_gemm ? 0 : M::OUT_COL), ad, wd, first_gemm ? idesc1 : idesc2, acc_first || ks > 0);
                ad = umma::desc_advance(ad, 2 * P::LBO);
                wd = umma::desc_advance(wd, 2 * lbo_b);
            }
            umma::commit(&bars.empty[slot]);
            ++cc;
        };
        auto wait_a = [&]() { umma::mbar_wait(&bars.a_ready, ph); ph ^= 1; umma::fence_after_sync(); };
        for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
            wait_a();
            block(true, false);                                // h_0
            umma::commit(&bars.acc_ready);
            for (int js = 0; js < M::NSL; ++js) {
                wait_a();                                      // GELU(h_js) staged in a1, h columns free
                block(false, js > 0);                          // out += GELU(h_js) W2_js^T
                if (js + 1 < M::NSL) block(true, false);       // h_{js+1}
                umma::commit(&bars.acc_ready);
            }
        }
    }
    pdl_trigger();                         // this CTA's work is done: the next kernel of the stream may start its prologue
    __syncthreads();
    if (warp == 4) {
        umma::fence_after_sync();
        umma::tmem_dealloc(tmem, M::TMEM_COLS);
    }
}

template <int C>
static int run_lkpm_mlp_tc(void* feat0, const void* y, int64_t rows, int planar_n, int planar_w, int planar_pitch, const cfp_lkpm_w& w,
                           cudaStream_t st) {
    CFP_REQUIRE(rows < ((int64_t)1 << 31), "lkpm_mlp: %lld rows exceed the 32-bit row index", (long long)rows);
    using M = MlpTC<C>;
    CFP_REQUIRE(w.tc != nullptr, "lkpm_mlp: bf16 path needs the packed tensor-core weights (cfp_lkpm_w.tc)");
    auto k = lkpm_mlp_tc_kernel<C>;
    if (int e = set_smem(k, M::SMEM)) return e;
    const int64_t ntiles = (rows + 127) / 128;
    const int per_sm = C >= 128 ? 1 : (C == 64 ? 2 : 3);
    const int grid = (int)(ntiles < sm_count() * per_sm ? ntiles : sm_count() * per_sm);
    launch_pdl(k, grid, 192, M::SMEM, st, (bf16*)feat0, (const bf16*)y, rows, planar_n, planar_w, planar_pitch, w, (int)ntiles,
               FastDiv((uint32_t)(planar_n > 0 ? planar_n : 1)), FastDiv((uint32_t)(planar_w > 0 ? planar_w : 1)));
    return check_launch(C == 32 ? "lkpm_mlp_tc<32>" : C == 64 ? "lkpm_mlp_tc<64>" : "lkpm_mlp_tc<128>");
}

int lkpm_mlp_tc(void* feat0, const void* y, int64_t rows, int planar_n, int planar_w, int planar_pitch, int C, const cfp_lkpm_w& w,
                cudaStream_t st) {
    if (C == 32) return run_lkpm_mlp_tc<32>(feat0, y, rows, planar_n, planar_w, planar_pitch, w, st);
    if (C == 64) return run_lkpm_mlp_tc<64>(feat0, y, rows, planar_n, planar_w, planar_pitch, w, st);
    if (C == 128) return run_lkpm_mlp_tc<128>(feat0, y, rows, planar_n, planar_w, planar_pitch, w, st);
    return fail("unsupported C=%d", C);
}

// =====================================================================================
// Attention state on tensor cores (attention.py:31-44):
//   K = elu(x Wk^T)+1, V = x Wv^T,  KV[g][h] = sum_{s in g} K_s^T V_s  (dh x dh),  Ksum[g] = sum_s K_s
// Both contractions are tcgen05.mma:
//   (1) the projection, [128 rows] x [C] x [2C], exactly like a chain stage;
//   (2) the reduction over rows.  The row threads write K and V (bf16) back in the chain's
//       [channel-group][row][16 B] layout; read as an *MN-major* operand (channel = M/N index,
//       row = K index, SBO = group stride, LBO = 128 B) the very same buffer is K^T and V^T, so
//       D[c1][c2] = sum_r K[r][c1] V[r][c2] is one M=128, N=C+16 MMA per 16 rows.  The extra 16
//       columns carry a ones-column, which makes Ksum fall out of the same MMA.  Only the
//       block-diagonal (same-head) part of D is used: thread c1 (TMEM lane c1) reads its head's
//       dh columns and adds them to the fp32 state in global memory.
// Rows are enumerated per group with the group size padded to a multiple of 16, so every
// 16-row MMA step belongs to one group; consecutive steps of a group form a "run" that
// accumulates in TMEM before it is flushed (plain stores when groups never straddle a tile).
template <int C> struct KvTC {
    static constexpr int KG = C / 8;
    static constexpr int A1G = 2 * KG + 2 < 16 ? 16 : 2 * KG + 2;   // K | V | ones | zeros (>= 16 groups: M = 128)
    static constexpr int NRED = C + 16;
    // the reduction accumulator (C + 16 columns) reuses the projection's 2C columns: the reduce MMAs are issued only after
    // every row thread has read its K | V row (a_ready), so the kernel needs max(2C, C + 16) columns - 64 / 128 / 256 -
    // and TMEM stops being what limits the co-resident CTAs at C = 32 / 64
    static constexpr int RED_COL = 0;
    static constexpr int TMEM_COLS = 2 * C <= 64 ? 64 : (2 * C <= 128 ? 128 : 256);
    static constexpr size_t SMEM = (size_t)(KG + A1G) * ChainTC<C>::LBO + 4 * (size_t)C * C;
};

// kZone16 (groups of exactly one 16-row MMA step: the hist2image zones): the per-group reduction is done by the row
// threads themselves with FMAs straight from the bf16 K | V tile - 16 rows x dh products per (channel, group) - instead
// of one MMA + accumulator read-back + flush round trip per group (eight serial round trips per tile).
// NT = threads per row (KvNT<C>): at C = 128 a CTA per SM with four row warps left every scheduler with one warp of long
// serial epilogues; two threads share a row (x chunks, then K columns | V columns, then half of the zones each).
template <int C> struct KvNT { static constexpr int NT = C >= 64 ? 2 : 1; };
template <class S> struct IsZoneTok { static constexpr bool value = false; };
template <> struct IsZoneTok<ZoneTokSrc<bf16>> { static constexpr bool value = true; };
// kZone16 at C = 128 (kZoneMma): the per-zone reduction goes back to the tensor pipe, but without the serial
// accumulate / read / flush of ONE accumulator: the projection's 2C TMEM columns are free once K | V sit in shared
// memory, so two zones are reduced at a time (one M = 128, N = C, K = 16 MMA each, MN-major views of the K | V tile,
// accumulators at columns 0 and C), thread (c1, half) stores its head's dh columns of zone 2 b + half, four batches per
// tile.  The FMA form cost ~4.5 k instructions per thread and tile there (16 rows x dh products per channel and zone,
// half of them bf16 unpacking); Ksum stays a 16-term row-thread sum.
template <int C, int NH, bool kComplete, class Src, bool kZone16 = false>
__global__ void __launch_bounds__((4 * KvNT<C>::NT + 2) * 32) kv_state_tc_kernel(Src src, int S, int S_pad, FastDiv dSp, int groups, const bf16* __restrict__ wkv_tc,
                                                          float* __restrict__ kv, float* __restrict__ ksum, int ntiles) {
    using P = ChainTC<C>;
    using K = KvTC<C>;
    constexpr int DH = C / NH, KG = P::KG, NT = KvNT<C>::NT, ROWT = 128 * NT;
    extern __shared__ __align__(128) uint8_t smem[];
    __shared__ ChainBars bars;
    uint8_t* a0 = smem;                            // x tile                [KG][129][16 B]
    uint8_t* a1 = a0 + KG * P::LBO;                // K | V | ones | zeros  [A1G][129][16 B]
    uint8_t* wsm = a1 + K::A1G * P::LBO;           // Wk, Wv blocks
    const int tid_all = threadIdx.x, warp = umma::warp_idx_sync(), lane = tid_all & 31;
    const int tid = tid_all & 127, half = warp >> 2, wq = warp & 3;       // row, which of the row's NT threads, TMEM lane quarter
    auto rows_barrier = [&]() { asm volatile("bar.sync 1, %0;\n" ::"n"(ROWT) : "memory"); };
    constexpr bool kZoneMma = kZone16 && C >= 128 && DH == 32 && NT == 2;
    constexpr bool kZonePos = kZone16 && IsZoneTok<Src>::value;      // zone tokens: the positional row of a thread never changes

    if (tid_all == 0) {
        umma::mbar_init(&bars.full[0], 1);
        umma::mbar_init(&bars.a_ready, ROWT);
        umma::mbar_init(&bars.acc_ready, 1);
        umma::fence_mbar_init();
    }
    if (warp == 4 * NT) umma::tmem_alloc(&bars.tmem_slot, K::TMEM_COLS);
    if (warp < 4 * NT)                              // zero the groups no one writes later
        for (int i = tid_all; i < (K::A1G - 2 * KG) * 129; i += ROWT)
            *reinterpret_cast<uint4*>(a1 + (size_t)(2 * KG) * P::LBO + (size_t)i * 16) = make_uint4(0u, 0u, 0u, 0u);
    umma::fence_async_smem();
    umma::fence_before_sync();
    __syncthreads();
    umma::fence_after_sync();
    const uint32_t tmem = bars.tmem_slot;
    const uint32_t total = (uint32_t)groups * (uint32_t)S_pad;      // < 2^31 (checked by the launcher): 32-bit index math and
                                                                      // multiply-high division (a 64-bit divide per run used to cost ~25 % here)

    if (warp < 4 * NT) {
        constexpr int KGT = KG / NT;                           // this thread's share of the row's 16-byte chunks
        // S_pad = 16 divides the tile: row `tid` is sample tid % 16 of its zone in EVERY tile, so its slice of the
        // positional table (weights, not produced by the previous kernel) is read once, before the grid dependency
        [[maybe_unused]] float pos[kZonePos ? KGT * 8 : 1];
        if constexpr (kZonePos) {
            const int s = (tid & 15) < S ? (tid & 15) : 0;
#pragma unroll
            for (int k = 0; k < KGT * 2; ++k) {
                const float4 p4 = *reinterpret_cast<const float4*>(src.pos2 + (size_t)s * C + half * (KGT * 8) + k * 4);
                pos[4 * k] = p4.x; pos[4 * k + 1] = p4.y; pos[4 * k + 2] = p4.z; pos[4 * k + 3] = p4.w;
            }
        }
        pdl_wait();
        uint32_t ph = 0;
        for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
            const uint32_t row0 = (uint32_t)tile * 128u;
            const uint32_t myp = row0 + tid;
            const int myg = (int)dSp.div(myp), mys = (int)(myp - (uint32_t)myg * (uint32_t)S_pad);
            const bool real = myp < total && mys < S;
            [[maybe_unused]] const int dbg_it = (tile - (int)blockIdx.x) / (int)gridDim.x;
            CFP_CHAIN_MARK(0, dbg_it);
            {
                const typename Src::R ref = src.locate(real ? (int64_t)myg * S + mys : 0);
                uint4 v[KGT];
                if constexpr (kZonePos) {
                    uint4 raw[KGT];
#pragma unroll
                    for (int k = 0; k < KGT; ++k)
                        raw[k] = real ? *reinterpret_cast<const uint4*>(src.tok + ref.off + (half * KGT + k) * 8) : make_uint4(0u, 0u, 0u, 0u);
#pragma unroll
                    for (int k = 0; k < KGT; ++k) {
                        float x8[8];
                        unpack8(raw[k], x8);
#pragma unroll
                        for (int i = 0; i < 8; ++i) x8[i] += pos[k * 8 + i];
                        v[k] = real ? pack8_bf16(x8) : make_uint4(0u, 0u, 0u, 0u);
                    }
                } else {
#pragma unroll
                    for (int k = 0; k < KGT; ++k) v[k] = real ? load8_bf16(src, ref, (half * KGT + k) * 8) : make_uint4(0u, 0u, 0u, 0u);
                }
#pragma unroll
                for (int k = 0; k < KGT; ++k) *reinterpret_cast<uint4*>(a0 + (size_t)(half * KGT + k) * P::LBO + tid * 16) = v[k];
            }
            umma::fence_async_smem();
            CFP_CHAIN_MARK(1, dbg_it);
            mbar_arrive(&bars.a_ready);

            // ---- K = elu(k)+1 and V of row `tid` -> a1 (zeros for padding rows)
            umma::mbar_wait(&bars.acc_ready, ph); ph ^= 1;
            CFP_CHAIN_MARK(2, dbg_it);
            umma::fence_after_sync();
            // padding rows are zeroed with a multiplicative mask (their x row was staged as zeros, so the accumulator is
            // finite): written as `!real ? 0 : ...` ptxas wrapped every elu in a divergent branch (114 BSSY / BSYNC pairs at
            // C = 128, 5.5 us per tile for ~900 instructions per thread)
            const float live = real ? 1.f : 0.f;
            if constexpr (C >= 64) {                           // NT = 2: thread `half` 0 owns the K columns, 1 the V columns
                static_assert(2 * C / NT == C, "a thread owns exactly K or V");
                const int cb = half * C;
                if (half == 0) {
                    umma::tmem_for_each16<C>(umma::tmem_addr(tmem, wq * 32, 0), [&](int cc, const float (&t)[16]) {
#pragma unroll
                        for (int j = 0; j < 16; j += 8) {
                            float o8[8];
#pragma unroll
                            for (int i = 0; i < 8; ++i) o8[i] = elu1(t[j + i]) * live;
                            umma::store_chunk(a1, P::LBO, tid, (cc + j) / 8, o8);
                        }
                    });
                } else {
                    umma::tmem_for_each16<C>(umma::tmem_addr(tmem, wq * 32, cb), [&](int cc, const float (&t)[16]) {
#pragma unroll
                        for (int j = 0; j < 16; j += 8) {
                            float o8[8];
#pragma unroll
                            for (int i = 0; i < 8; ++i) o8[i] = t[j + i] * live;
                            umma::store_chunk(a1, P::LBO, tid, (cb + cc + j) / 8, o8);
                        }
                    });
                }
            } else {                                           // four pieces only: the rolled loop measured 15 % faster at C = 32
#pragma unroll 1
                for (int c0 = 0; c0 < 2 * C; c0 += 16) {
                    float t[16];
                    umma::tmem_ld16(umma::tmem_addr(tmem, wq * 32, c0), t);
                    const bool isk = c0 < C;                   // warp-uniform
#pragma unroll
                    for (int j = 0; j < 16; j += 8) {
                        float o8[8];
#pragma unroll
                        for (int i = 0; i < 8; ++i) o8[i] = (isk ? elu1(t[j + i]) : t[j + i]) * live;
                        umma::store_chunk(a1, P::LBO, tid, (c0 + j) / 8, o8);
                    }
                }
            }
            if constexpr (kZoneMma) {
                umma::fence_async_smem();
                umma::fence_before_sync();
                CFP_CHAIN_MARK(3, dbg_it);
                mbar_arrive(&bars.a_ready);                    // K | V staged, projection accumulator consumed: batch 0 may issue
                rows_barrier();                                // ... and visible to the other row threads (Ksum below)
                const int c1 = tid;                            // channel = TMEM lane; its head's columns start at wq * 32
                {
                    const uint8_t* kp = a1 + (size_t)(c1 / 8) * P::LBO + (c1 % 8) * 2;
#pragma unroll
                    for (int zz = 0; zz < 4; ++zz) {
                        const int z = half * 4 + zz;
                        float ks = 0.f;
#pragma unroll
                        for (int rr = 0; rr < 16; ++rr)
                            ks += __uint_as_float((uint32_t)*reinterpret_cast<const uint16_t*>(kp + (z * 16 + rr) * 16) << 16);
                        const int64_t g = (int64_t)tile * 8 + z;
                        if (g < groups) ksum[(size_t)g * C + c1] = ks;
                    }
                }
                CFP_CHAIN_MARK(4, dbg_it);
#pragma unroll 1
                for (int b = 0; b < 4; ++b) {
                    umma::mbar_wait(&bars.acc_ready, ph); ph ^= 1;
                    umma::fence_after_sync();
                    const int64_t g = (int64_t)tile * 8 + 2 * b + half;
                    float t0[16], t1[16];
                    umma::tmem_ld16(umma::tmem_addr(tmem, wq * 32, half * C + wq * 32), t0);
                    umma::tmem_ld16(umma::tmem_addr(tmem, wq * 32, half * C + wq * 32 + 16), t1);
                    if (g < groups) {
                        float* dst = kv + (size_t)g * (C * DH) + (size_t)c1 * DH;
#pragma unroll
                        for (int v = 0; v < 16; v += 4) *reinterpret_cast<float4*>(dst + v) = make_float4(t0[v], t0[v + 1], t0[v + 2], t0[v + 3]);
#pragma unroll
                        for (int v = 0; v < 16; v += 4) *reinterpret_cast<float4*>(dst + 16 + v) = make_float4(t1[v], t1[v + 1], t1[v + 2], t1[v + 3]);
                    }
                    umma::fence_before_sync();
                    if (b < 3) mbar_arrive(&bars.a_ready);     // both accumulators read: the next two zones may overwrite them
                }
                CFP_CHAIN_MARK(5, dbg_it);
                continue;                                      // the next tile's a_ready arrival orders a0 / a1 / TMEM reuse
            } else if constexpr (kZone16) {
                umma::fence_before_sync();
                rows_barrier();                                // K | V of all 128 rows staged; accumulator consumed
                constexpr int ZPT = 8 / (ROWT / C);            // zones per thread: thread = (channel c1, zone subset)
                const int c1 = tid_all % C, h0 = (c1 / DH) * DH;
                const uint8_t* kp = a1 + (size_t)(c1 / 8) * P::LBO + (c1 % 8) * 2;
                const uint8_t* vp = a1 + (size_t)(KG + h0 / 8) * P::LBO;
                for (int z = (tid_all / C) * ZPT; z < (tid_all / C) * ZPT + ZPT; ++z) {
                    float acc[DH], ks = 0.f;
#pragma unroll
                    for (int v = 0; v < DH; ++v) acc[v] = 0.f;
#pragma unroll 4
                    for (int rr = 0; rr < 16; ++rr) {
                        const int rw = z * 16 + rr;
                        const float kval = __uint_as_float((uint32_t)*reinterpret_cast<const uint16_t*>(kp + rw * 16) << 16);
                        ks += kval;
#pragma unroll
                        for (int v8 = 0; v8 < DH / 8; ++v8) {
                            float vv[8];
                            unpack8(*reinterpret_cast<const uint4*>(vp + (size_t)v8 * P::LBO + rw * 16), vv);
#pragma unroll
                            for (int i2 = 0; i2 < 8; ++i2) acc[v8 * 8 + i2] = fmaf(kval, vv[i2], acc[v8 * 8 + i2]);
                        }
                    }
                    const int64_t g = (int64_t)tile * 8 + z;
                    if (g < groups) {
                        float* dst = kv + (size_t)g * (C * DH) + (size_t)c1 * DH;
#pragma unroll
                        for (int v = 0; v < DH; v += 4) *reinterpret_cast<float4*>(dst + v) = make_float4(acc[v], acc[v + 1], acc[v + 2], acc[v + 3]);
                        ksum[(size_t)g * C + c1] = ks;
                    }
                }
                rows_barrier();                                // a1 is rewritten by the next tile's epilogue
                continue;
            }
            if (half == 0) {
                const float one8[8] = {real ? 1.f : 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
                umma::store_chunk(a1, P::LBO, tid, 2 * KG, one8);
            }
            umma::fence_async_smem();
            umma::fence_before_sync();
            CFP_CHAIN_MARK(3, dbg_it);
            mbar_arrive(&bars.a_ready);

            // ---- flush the runs: lane c1 adds D[c1][head(c1) block] and D[c1][ones] to the state
            int ks = 0;
            while (ks < 8 && row0 + 16 * ks < total) {
                const int g = (int)dSp.div(row0 + 16 * ks);
                int ke = ks + 1;
                while (ke < 8 && row0 + 16 * ke < total && (int)dSp.div(row0 + 16 * ke) == g) ++ke;
                umma::mbar_wait(&bars.acc_ready, ph); ph ^= 1;
                CFP_CHAIN_MARK(4, dbg_it);
                umma::fence_after_sync();
                if (half == 0 && wq * 32 < C) {
                    const int m = wq * 32 + lane;
                    float t0[16], t1[16], o[16];
                    umma::tmem_ld16(umma::tmem_addr(tmem, wq * 32, K::RED_COL + wq * 32), t0);
                    umma::tmem_ld16(umma::tmem_addr(tmem, wq * 32, K::RED_COL + wq * 32 + 16), t1);
                    umma::tmem_ld16(umma::tmem_addr(tmem, wq * 32, K::RED_COL + C), o);
                    float* dst = kv + (size_t)g * (C * DH) + (size_t)m * DH;
#pragma unroll
                    for (int sb = 0; sb < 32 / DH; ++sb)
                        if (lane / DH == sb) {
#pragma unroll
                            for (int j = 0; j < DH; ++j) {
                                const int col = sb * DH + j;                  // compile-time after unrolling
                                const float val = col < 16 ? t0[col & 15] : t1[col & 15];
                                if (kComplete) dst[j] = val;
                                else atomicAdd(dst + j, val);
                            }
                        }
                    if (kComplete) ksum[(size_t)g * C + m] = o[0];
                    else atomicAdd(ksum + (size_t)g * C + m, o[0]);
                }
                ks = ke;
                const bool last = !(ks < 8 && row0 + 16 * ks < total);
                if (!last) {
                    umma::fence_before_sync();
                    mbar_arrive(&bars.a_ready);
                }
            }
            CFP_CHAIN_MARK(5, dbg_it);
            umma::fence_before_sync();
        }
    } else if (warp == 4 * NT) {
        umma::bulk_load(wsm, wkv_tc, 4 * C * C, &bars.full[0]);
    } else {
        {
            const uint32_t idesc = umma::idesc_bf16(128, C);
            const uint32_t idesc_red = umma::idesc_bf16(128, K::NRED) | (1u << 15) | (1u << 16);   // A, B MN-major
            const uint32_t a0s = umma::smem_u32(a0), a1s = umma::smem_u32(a1), ws = umma::smem_u32(wsm);
            constexpr uint32_t LBO_B = C * 16;
            uint32_t ph = 0;
            auto wait_a = [&]() { umma::mbar_wait(&bars.a_ready, ph); ph ^= 1; umma::fence_after_sync(); };
            umma::mbar_wait(&bars.full[0], 0);
            umma::fence_after_sync();
            for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
                const uint32_t row0 = (uint32_t)tile * 128u;
                wait_a();
#pragma unroll
                for (int half = 0; half < 2; ++half)          // k -> cols [0,C), v -> cols [C,2C)
#pragma unroll
                    for (int ks = 0; ks < C / 16; ++ks)
                        umma::mma_bf16(tmem + half * C, umma::smem_desc(a0s + 2 * ks * P::LBO, P::LBO),
                                       umma::smem_desc(ws + half * 2 * C * C + ks * 2 * LBO_B, LBO_B), idesc, ks > 0);
                umma::commit(&bars.acc_ready);
                if constexpr (kZoneMma) {                     // two zones per batch: K^T V of 16 rows into columns 0 / C
                    const uint32_t idesc_z = umma::idesc_bf16(128, C) | (1u << 15) | (1u << 16);
#pragma unroll 1
                    for (int b = 0; b < 4; ++b) {
                        wait_a();                             // K | V staged (b = 0) / previous batch read
#pragma unroll
                        for (int zz = 0; zz < 2; ++zz)
                            umma::mma_bf16(tmem + zz * C, umma::smem_desc(a1s + (2 * b + zz) * 256, 128, P::LBO),
                                           umma::smem_desc(a1s + KG * P::LBO + (2 * b + zz) * 256, 128, P::LBO), idesc_z, false);
                        umma::commit(&bars.acc_ready);
                    }
                    continue;
                }
                if constexpr (kZone16) continue;              // the row threads reduce the groups themselves
                wait_a();                                     // K | V | ones staged
                int ks = 0;
                bool first = true;
                while (ks < 8 && row0 + 16 * ks < total) {
                    const int g = (int)dSp.div(row0 + 16 * ks);
                    int ke = ks + 1;
                    while (ke < 8 && row0 + 16 * ke < total && (int)dSp.div(row0 + 16 * ke) == g) ++ke;
                    if (!first) wait_a();                     // previous run's accumulator has been read
                    first = false;
                    for (int k = ks; k < ke; ++k)             // MN-major views: SBO = group stride, LBO = 8 rows
                        umma::mma_bf16(tmem + K::RED_COL, umma::smem_desc(a1s + k * 256, 128, P::LBO),
                                       umma::smem_desc(a1s + KG * P::LBO + k * 256, 128, P::LBO), idesc_red, k > ks);
                    umma::commit(&bars.acc_ready);
                    ks = ke;
                }
            }
        }
    }
    pdl_trigger();                         // this CTA's work is done: the next kernel of the stream may start its prologue
    __syncthreads();
    if (warp == 4 * NT) {
        umma::fence_after_sync();
        umma::tmem_dealloc(tmem, K::TMEM_COLS);
    }
}

template <int C, int NH, class Src>
static int run_kv_state_tc(const char* name, const Src& src, int S, int groups, const void* wkv_tc, float* kv, float* ksum,
                           cudaStream_t st) {
    using K = KvTC<C>;
    constexpr int DH = C / NH;
    CFP_REQUIRE(wkv_tc != nullptr, "%s: bf16 path needs the packed tensor-core weights (cfp_loftr_w.kv_tc)", name);
    const int S_pad = (S + 15) / 16 * 16;
    const bool complete = 128 % S_pad == 0;          // groups never straddle a tile: plain stores, no memset
    if (!complete) {
        cudaError_t e = cudaMemsetAsync(kv, 0, (size_t)groups * (C * DH + C) * sizeof(float), st);
        if (e != cudaSuccess) return fail("cudaMemsetAsync(kv state): %s", cudaGetErrorString(e));
    }
    const int64_t ntiles = ((int64_t)groups * S_pad + 127) / 128;
    CFP_REQUIRE((int64_t)groups * S_pad < ((int64_t)1 << 31), "%s: %lld padded rows exceed the 32-bit row index", name, (long long)groups * S_pad);
    const int per_sm = C >= 128 ? 1 : (C == 64 ? 3 : 5);          // shared memory: 169 / 70 / 45 KB per CTA
    const int grid = (int)(ntiles < sm_count() * per_sm ? ntiles : sm_count() * per_sm);
    if (S_pad == 16 && NH == 4) {                     // hist2image zones (dh = C/4 is a multiple of 8)
        auto k = kv_state_tc_kernel<C, NH, true, Src, (NH == 4)>;
        if (int e = set_smem(k, K::SMEM)) return e;
        launch_pdl(k, grid, (4 * KvNT<C>::NT + 2) * 32, K::SMEM, st, src, S, S_pad, FastDiv((uint32_t)S_pad), groups, (const bf16*)wkv_tc, kv, ksum, (int)ntiles);
    } else if (complete) {
        auto k = kv_state_tc_kernel<C, NH, true, Src>;
        if (int e = set_smem(k, K::SMEM)) return e;
        launch_pdl(k, grid, (4 * KvNT<C>::NT + 2) * 32, K::SMEM, st, src, S, S_pad, FastDiv((uint32_t)S_pad), groups, (const bf16*)wkv_tc, kv, ksum, (int)ntiles);
    } else {
        auto k = kv_state_tc_kernel<C, NH, false, Src>;
        if (int e = set_smem(k, K::SMEM)) return e;
        launch_pdl(k, grid, (4 * KvNT<C>::NT + 2) * 32, K::SMEM, st, src, S, S_pad, FastDiv((uint32_t)S_pad), groups, (const bf16*)wkv_tc, kv, ksum, (int)ntiles);
    }
#ifdef CFP_DEBUG_TIMING
    {
        cudaStreamSynchronize(st);
        unsigned long long h[16] = {0};
        cudaMemcpyFromSymbol(h, g_chain_dbg, sizeof(h));
        fprintf(stderr, "%s (C=%d, %d CTAs, %lld tiles, S_pad %d) 2nd tile of CTA 5, ns since tile start: stage_x %llu | proj-acc %llu | K|V epilogue %llu | last run-acc %llu | flushed %llu\n",
                name, C, grid, (long long)ntiles, S_pad, h[1] - h[0], h[2] - h[0], h[3] - h[0], h[4] - h[0], h[5] - h[0]);
    }
#endif
    return check_launch(name);
}

#define CFP_KV_DISPATCH(NH, NAME)                                                                     \
    if (C == 32) return run_kv_state_tc<32, NH>(NAME ",32>", src, S, groups, wkv_tc, kv, ksum, st);   \
    if (C == 64) return run_kv_state_tc<64, NH>(NAME ",64>", src, S, groups, wkv_tc, kv, ksum, st);   \
    if (C == 128) return run_kv_state_tc<128, NH>(NAME ",128>", src, S, groups, wkv_tc, kv, ksum, st); \
    return fail("unsupported C=%d", C);

int kv_tc_h2i(int C, const ZoneTokSrc<bf16>& src, int S, int groups, const void* wkv_tc, float* kv, float* ksum,
              cudaStream_t st) { CFP_KV_DISPATCH(4, "kv_state_tc<hist2image") }
int kv_tc_lsa(int C, const WindowRows<bf16>& src, int S, int groups, const void* wkv_tc, float* kv, float* ksum,
              cudaStream_t st) { CFP_KV_DISPATCH(8, "kv_state_tc<lsa") }
int kv_tc_gsa(int C, const SrTokSrc& src, int S, int groups, const void* wkv_tc, float* kv, float* ksum,
              cudaStream_t st) { CFP_KV_DISPATCH(8, "kv_state_tc<gsa") }
int kv_tc_dapm(int C, const InsideSrc<bf16>& src, int S, int groups, const void* wkv_tc, float* kv, float* ksum,
               cudaStream_t st) { CFP_KV_DISPATCH(4, "kv_state_tc<dapm") }

// =====================================================================================
// GSA sub-sampling conv on tensor cores (transformer.py:144-147): a stride-ws, ws x ws conv is a
// GEMM with K = ws*ws*C whose A rows are gathered per tap.  Only B*Ns (a few thousand) rows exist,
// so the K dimension (taps) is split across CTAs (grid = row tiles x tap splits) and partial sums
// are added atomically into an fp32 accumulator; sr_bias_ln_kernel then applies bias + LayerNorm.
// Per tap the 128 row threads copy the [128 x C] A slice into a ring stage with zero-fill cp.async (every 16-byte chunk
// is one fire-and-forget copy; each thread's chunk addresses are tap-independent up to a common offset and are located
// once) while the bulk-copy engine brings the [C x C] weight block; SrTC::NST taps are in flight, the MMA lane consumes
// a stage and frees it by commit.  (With a 2-stage register-staged gather every tap paid a full global-load round trip.)
template <int C> struct SrTC { static constexpr int NST = C >= 128 ? 3 : (C == 64 ? 4 : 6); };
struct SrBars {
    uint64_t a_full[6], w_full[6], empty[6], acc_ready;
    uint32_t tmem_slot;
};

template <int C>
__global__ void __launch_bounds__(192) sr_conv_tc_kernel(const bf16* __restrict__ feat, float* __restrict__ acc_out,
                                                         int64_t rows, int H, int W, int ws, int nsx, int Ns,
                                                         const bf16* __restrict__ sr_tc, int taps_per_cta, FastDiv dNs, FastDiv dNsx,
                                                         FastDiv dWs) {
    using P = ChainTC<C>;
    constexpr int KG = P::KG, TCOLS = C < 32 ? 32 : C, NST = SrTC<C>::NST;
    extern __shared__ __align__(128) uint8_t smem[];
    __shared__ SrBars bars;
    uint8_t* a_st = smem;                                // [NST][KG][129][16 B]
    uint8_t* w_st = a_st + (size_t)NST * KG * P::LBO;    // [NST][C x C]
    const int tid = threadIdx.x, warp = umma::warp_idx_sync();
    const int ntap = ws * ws;
    const int t0 = blockIdx.y * taps_per_cta, t1 = min(t0 + taps_per_cta, ntap);
    const int64_t row0 = (int64_t)blockIdx.x * 128;

    if (tid == 0) {
        for (int i = 0; i < NST; ++i) {
            umma::mbar_init(&bars.a_full[i], 128);
            umma::mbar_init(&bars.w_full[i], 1);
            umma::mbar_init(&bars.empty[i], 1);
        }
        umma::mbar_init(&bars.acc_ready, 1);
        umma::fence_mbar_init();
    }
    if (warp == 4) umma::tmem_alloc(&bars.tmem_slot, TCOLS);
    umma::fence_before_sync();
    __syncthreads();
    umma::fence_after_sync();
    const uint32_t tmem = bars.tmem_slot;

    if (warp < 4) {
        pdl_wait();
        // chunk k of this thread: (row r_k, channel group kg_k) with r_k * KG + kg_k = tid + 128 k; source element offset of
        // the row's window origin (tap (0,0)) or -1 for rows past the end (zero-filled)
        int64_t base[KG];
        uint32_t dst[KG];
#pragma unroll
        for (int k = 0; k < KG; ++k) {
            const int i = tid + 128 * k, r = i / KG, kg = i % KG;
            const int64_t row = row0 + r;
            base[k] = -1;
            if (row < rows) {
                uint32_t b, sidx, sy, sx;                       // multiply-high divisions (48 integer divisions per thread at C = 128)
                dNs.divmod((uint32_t)row, b, sidx);
                dNsx.divmod(sidx, sy, sx);
                const int y = (int)sy * ws, x = (int)sx * ws;
                base[k] = (((int64_t)b * H + y) * W + x) * C + kg * 8;
            }
            dst[k] = (uint32_t)(kg * P::LBO + r * 16);
        }
        const uint32_t a_base = umma::smem_u32(a_st);
        auto issue = [&](int t) {                        // copies of tap t into stage (t - t0) % NST
            const int n = t - t0, st = n % NST;
            if (n >= NST) umma::mbar_wait(&bars.empty[st], ((n / NST) - 1) & 1);
            uint32_t ty, tx;
            dWs.divmod((uint32_t)t, ty, tx);
            const int64_t toff = ((int64_t)ty * W + tx) * C;
#pragma unroll
            for (int k = 0; k < KG; ++k) {
                const bf16* g = base[k] >= 0 ? feat + base[k] + toff : feat;
                const uint32_t nbytes = base[k] >= 0 ? 16u : 0u;
                asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;\n" ::"r"(a_base + st * (uint32_t)(KG * P::LBO) + dst[k]), "l"(g), "r"(nbytes) : "memory");
            }
        };
        for (int t = t0; t < t0 + NST - 1; ++t) {        // prologue: NST - 1 taps in flight
            if (t < t1) issue(t);
            asm volatile("cp.async.commit_group;\n" ::: "memory");
        }
        for (int t = t0; t < t1; ++t) {
            if (t + NST - 1 < t1) issue(t + NST - 1);
            asm volatile("cp.async.commit_group;\n" ::: "memory");
            asm volatile("cp.async.wait_group %0;\n" ::"n"(NST - 1) : "memory");    // tap t has landed
            umma::fence_async_smem();
            mbar_arrive(&bars.a_full[(t - t0) % NST]);
        }
        umma::mbar_wait(&bars.acc_ready, 0);
        umma::fence_after_sync();
        const int64_t row = row0 + tid;
#pragma unroll 1
        for (int c0 = 0; c0 < C; c0 += 16) {
            float v[16];
            umma::tmem_ld16(umma::tmem_addr(tmem, warp * 32, c0), v);
            if (row < rows) {
#pragma unroll
                for (int j = 0; j < 16; ++j) atomicAdd(acc_out + row * C + c0 + j, v[j]);
            }
        }
        umma::fence_before_sync();
    } else if (warp == 4) {
        for (int t = t0; t < t1; ++t) {
            const int n = t - t0, st = n % NST;
            if (n >= NST) umma::mbar_wait(&bars.empty[st], ((n / NST) - 1) & 1);
            umma::bulk_load(w_st + (size_t)st * P::SLOT, sr_tc + (size_t)t * C * C, P::SLOT, &bars.w_full[st]);
        }
    } else {
        {
            const uint32_t idesc = umma::idesc_bf16(128, C);
            constexpr uint32_t LBO_B = C * 16;
            for (int t = t0; t < t1; ++t) {
                const int n = t - t0, st = n % NST;
                umma::mbar_wait(&bars.a_full[st], (n / NST) & 1);
                umma::mbar_wait(&bars.w_full[st], (n / NST) & 1);
                umma::fence_after_sync();
                const uint32_t ab = umma::smem_u32(a_st) + st * KG * P::LBO, wb = umma::smem_u32(w_st) + st * P::SLOT;
#pragma unroll
                for (int ks = 0; ks < C / 16; ++ks)
                    umma::mma_bf16(tmem, umma::smem_desc(ab + 2 * ks * P::LBO, P::LBO),
                                   umma::smem_desc(wb + ks * 2 * LBO_B, LBO_B), idesc, n > 0 || ks > 0);
                umma::commit(&bars.empty[st]);
            }
            umma::commit(&bars.acc_ready);
        }
    }
    pdl_trigger();                         // this CTA's work is done: the next kernel of the stream may start its prologue
    __syncthreads();
    if (warp == 4) {
        umma::fence_after_sync();
        umma::tmem_dealloc(tmem, TCOLS);
    }
}

// sr_tok[row] = LayerNorm(acc[row] + bias), in place on the fp32 accumulator (warp per row).
template <int C>
__global__ void sr_bias_ln_kernel(float* __restrict__ sr_tok, int64_t rows, const float* __restrict__ bias,
                                  const float* __restrict__ gamma, const float* __restrict__ beta) {
    const int lane = threadIdx.x & 31;
    const int64_t row = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    pdl_trigger();                         // tiny kernel: let the next one come in right away
    pdl_wait();
    if (row >= rows) return;
    constexpr int PER = C / 32;
    float v[PER], s = 0.f;
#pragma unroll
    for (int i = 0; i < PER; ++i) { v[i] = sr_tok[row * C + lane + 32 * i] + bias[lane + 32 * i]; s += v[i]; }
    const float mean = warp_sum(s) * (1.f / C);
    float q = 0.f;
#pragma unroll
    for (int i = 0; i < PER; ++i) { v[i] -= mean; q += v[i] * v[i]; }
    const float rstd = rsqrtf(warp_sum(q) * (1.f / C) + kLnEps);
#pragma unroll
    for (int i = 0; i < PER; ++i) sr_tok[row * C + lane + 32 * i] = v[i] * rstd * gamma[lane + 32 * i] + beta[lane + 32 * i];
}

template <int C>
static int run_sr_conv_tc(const void* feat0, float* sr_tok, int B, int H, int W, int ws, const void* sr_tc,
                          const float* sr_b, const float* g, const float* b, cudaStream_t st) {
    using P = ChainTC<C>;
    CFP_REQUIRE(sr_tc != nullptr, "sr conv: bf16 path needs the packed tensor-core weights (cfp_twins_w.sr_tc)");
    const int nsx = W / ws, Ns = (H / ws) * nsx;
    const int64_t rows = (int64_t)B * Ns;
    if (rows == 0) return 0;
    cudaError_t e = cudaMemsetAsync(sr_tok, 0, (size_t)rows * C * sizeof(float), st);
    if (e != cudaSuccess) return fail("cudaMemsetAsync(sr accumulator): %s", cudaGetErrorString(e));
    const int tiles = (int)((rows + 127) / 128), ntap = ws * ws;
    // split the taps so that the grid is ONE wave of co-resident CTAs (shared memory: 3 / 2 / 1 CTAs per SM at C = 32 / 64 /
    // 128): a second, partial wave of tap slices costs a whole slice latency
    constexpr int per_sm = C >= 128 ? 1 : (C == 64 ? 2 : 3);
    int splits = (sm_count() * per_sm) / tiles;
    if (splits < 1) splits = 1;
    if (splits > ntap) splits = ntap;
    const int taps_per_cta = (ntap + splits - 1) / splits;
    splits = (ntap + taps_per_cta - 1) / taps_per_cta;
    constexpr size_t smem = SrTC<C>::NST * ((size_t)P::KG * P::LBO + (size_t)P::SLOT);
    CFP_REQUIRE(rows < ((int64_t)1 << 31), "sr conv: %lld rows exceed the 32-bit row index", (long long)rows);
    auto k = sr_conv_tc_kernel<C>;
    if (int err = set_smem(k, smem)) return err;
    launch_pdl(k, dim3(tiles, splits), 192, smem, st, (const bf16*)feat0, sr_tok, rows, H, W, ws, nsx, Ns, (const bf16*)sr_tc,
               taps_per_cta, FastDiv((uint32_t)Ns), FastDiv((uint32_t)nsx), FastDiv((uint32_t)ws));
    if (int err = check_launch(C == 32 ? "sr_conv_tc<32>" : C == 64 ? "sr_conv_tc<64>" : "sr_conv_tc<128>")) return err;
    launch_pdl(sr_bias_ln_kernel<C>, (unsigned)((rows + 7) / 8), 256, 0, st, sr_tok, rows, sr_b, g, b);
    return check_launch("sr_bias_ln");
}

int sr_conv_ln_tc(const void* feat0, float* sr_tok, int B, int H, int W, int C, int ws, const void* sr_tc,
                  const float* sr_b, const float* g, const float* b, cudaStream_t st) {
    if (C == 32) return run_sr_conv_tc<32>(feat0, sr_tok, B, H, W, ws, sr_tc, sr_b, g, b, st);
    if (C == 64) return run_sr_conv_tc<64>(feat0, sr_tok, B, H, W, ws, sr_tc, sr_b, g, b, st);
    if (C == 128) return run_sr_conv_tc<128>(feat0, sr_tok, B, H, W, ws, sr_tc, sr_b, g, b, st);
    return fail("unsupported C=%d", C);
}

// ---- entry points used by k_loftr.cu's layer implementations (bf16 only)
#define CFP_TC_DISPATCH(NH, ATTN, NAME)                                                  \
    if (C == 32) return run_query_tc<32, NH, ATTN>(NAME ",32>", q, w, kv, ksum, st);     \
    if (C == 64) return run_query_tc<64, NH, ATTN>(NAME ",64>", q, w, kv, ksum, st);     \
    if (C == 128) return run_query_tc<128, NH, ATTN>(NAME ",128>", q, w, kv, ksum, st);  \
    return fail("unsupported C=%d", C);

template <class Q>
static int query_tc_h2i_impl(int C, const Q& q, const cfp_loftr_w& w, const float* kv, const float* ksum, cudaStream_t st) {
    CFP_TC_DISPATCH(4, false, "loftr_query_tc<hist2image")
}
int query_tc_h2i(int C, const ZonePatchRows<bf16>& q, const cfp_loftr_w& w, const float* kv, const float* ksum,
                 cudaStream_t st) {
    if (q.fast_eligible()) return query_tc_h2i_impl(C, ZonePatchRows<bf16, true>(q), w, kv, ksum, st);
    return query_tc_h2i_impl(C, q, w, kv, ksum, st);
}
int query_tc_lsa(int C, const WindowRows<bf16>& q, const cfp_loftr_w& w, const float* kv, const float* ksum,
                 cudaStream_t st) {
    CFP_TC_DISPATCH(8, false, "loftr_query_tc<lsa")
}
int query_tc_gsa(int C, const FrameRows<bf16>& q, const cfp_loftr_w& w, const float* kv, const float* ksum,
                 cudaStream_t st) {
    CFP_TC_DISPATCH(8, false, "loftr_query_tc<gsa")
}
int query_tc_gsa_nchw(int C, const FrameRowsToNCHW<bf16>& q, const cfp_loftr_w& w, const float* kv, const float* ksum,
                      cudaStream_t st) {
    CFP_TC_DISPATCH(8, false, "loftr_query_tc<gsa")
}
int query_tc_dapm(int C, const OutsideRows<bf16>& q, const cfp_loftr_w& w, const float* kv, const float* ksum,
                  cudaStream_t st) {
    CFP_TC_DISPATCH(4, true, "attn_query_tc<dapm")
}

}  // namespace cfp
