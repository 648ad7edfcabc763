// LKPM large-kernel depthwise convolution on the tensor cores (bf16 path).
//
//   y[b][r][x][c] = ReLU( sum_{dy,dx} w[c][dy][dx] * in[b][r+dy-p][x+dx-p][c] + shift[c] ),  p = (k-1)/2
//                                                                   (convnext.py:45-47, BN folded)
//
// As a direct stencil the 31x31 case is bound by the fp32 FMA pipe (961 FMA per output, SURVEY §7).
// Here each channel plane is a GEMM instead: for one channel and one tile of 32 output columns
//
//   D[r][n] = sum_dy sum_kk  A_dy[r][kk] * T_dy[n][kk],     A_dy[r][kk] = plane[r + dy][x0 + kk]
//                                                            T_dy[n][kk] = w[dy][kk - n]  (0 outside the band)
//
// The banded Toeplitz matrix T_dy carries the horizontal taps; the vertical tap is a row shift.  A row-shifted
// A view (start address + 16 B * dy in the canonical K-major layout, umma.cuh) would work, but with N = 32 every
// MMA is bound by the shared-memory read of its 4 KB A tile (twice that when the shift is not a multiple of
// 8 rows).  So the vertical taps are split as dy = NB a + b (NB = kDwNB = 4): the NB b's of one a use the SAME A view
// (rows m + NB a) and their Toeplitz blocks sit side by side along N:
//
//   E[m][(b, n)] = sum_a sum_kk plane[m + NB a][x0 + kk] * T_{NB a+b}[n][kk]      one M=128 x N=128 x K=16 MMA per (a, kk/16)
//   out[r][n]    = sum_b E[r + b][(b, n)]                                         row shift b applied by the epilogue
//
// One A read feeds NB x 32 accumulator columns, so the MMA runs at the tensor pipe's rate instead of the operand
// fetch rate.  NB is a balance: the epilogue has to read NB x 32 accumulator columns per output row through
// tcgen05.ld (64 B/clk/SM) - at NB = 8 that alone took as long as the MMAs - and needs NB - 1 shuffles per column.
// The epilogue thread of accumulator row m gets E[m + b] from lane m + b with warp shuffles; the rows that live in
// the next TMEM lane quarter travel through a small shared-memory exchange.  Eight epilogue warps (two per lane
// quarter, 16 output columns each) keep two warps on every scheduler.
// About half of every T_dy is structural zeros; the tensor pipe is still >10x faster than the FMA pipe on this op.
//
// Data flow: dw_plane_pack_kernel rewrites the token-major map into zero-padded channel planes stored
// directly in the UMMA layout ([b][c][x-group][padded row][8 columns]), so that the A operand of a
// (frame, channel, column tile) is ONE contiguous block brought in by a single bulk (TMA) copy.
// dwconv_tc_kernel: CTA = (column tile, channel); the channel's K Toeplitz blocks (host-packed) stay
// resident in shared memory while the CTA walks over the frames with a 3-stage A ring and two TMEM
// accumulators (MMA of frame i+1 overlaps the epilogue of frame i).  The epilogue writes planar
// rows ([B][C][H][W]); the pointwise MLP (lkpm_mlp_tc_kernel) reads that map in place - lanes are consecutive
// tokens, so a channel's 32 values are one coalesced 64-byte segment - and no transpose back is needed.
#include "cfp_common.cuh"
#include "cfp_internal.h"
#include "umma.cuh"

namespace cfp {

constexpr int kDwNB = 4;       // vertical taps stacked along the MMA's N dimension (dy = kDwNB * a + b)
constexpr int kDwN = kDwNB * 32;
constexpr int kDwAcc = kDwN <= 128 ? 128 : 256;   // TMEM columns reserved per accumulator (two accumulators)
constexpr int kDwMS = 120;     // output rows per 128-row M block: the epilogue reads accumulator rows m .. m + kDwNB - 1

struct DwGeom {
    int H, W, C, K, PAD;
    int F;         // frames stacked vertically in one plane (PAD zero rows between them): fills the M block
                   // when the map is short (H=52 at 1/8 scale -> 2 frames per MMA)
    int RS;        // row stride between stacked frames = H + PAD
    int NB;        // plane stacks = ceil(B / F)
    int nM;        // M blocks (kDwMS output rows each) per stack
    int HP;        // padded plane rows
    int KS;        // 16-column K-steps per tap group = ceil((32 + K - 1) / 16)
    int NA;        // groups of kDwNB vertical taps = ceil(K / kDwNB)
    int nX;        // 32-column output tiles
    int WG;        // 8-column groups per plane = 4*nX + 2*KS - 4
    int WO;        // row pitch of the planar output = W rounded up to 8 (every row and every 8-column chunk 16-byte aligned)
};
static DwGeom dw_geom(int B, int H, int W, int C, int K) {
    DwGeom g;
    g.H = H; g.W = W; g.C = C; g.K = K; g.PAD = (K - 1) / 2;
    g.RS = H + g.PAD;
    g.F = (kDwMS + g.PAD) / g.RS;                      // F*H + (F-1)*PAD <= kDwMS
    if (g.F < 1) g.F = 1;
    if (g.F > B) g.F = B;
    g.NB = (B + g.F - 1) / g.F;
    const int rows = g.F * H + (g.F - 1) * g.PAD;      // output rows of one stack
    g.nM = (rows + kDwMS - 1) / kDwMS;
    g.KS = (32 + K - 1 + 15) / 16;
    g.NA = (K + kDwNB - 1) / kDwNB;
    // rows an A view can touch: last block start + 128 accumulator rows + 8 rows per further tap group;
    // and every row that feeds a stored output (PAD + F x (H + PAD)) must exist for the pack kernel
    g.HP = (g.nM - 1) * kDwMS + 128 + kDwNB * (g.NA - 1);
    if (g.HP < g.F * g.RS + g.PAD) g.HP = g.F * g.RS + g.PAD;
    g.nX = (W + 31) / 32;
    g.WG = 4 * g.nX + 2 * g.KS - 4;
    g.WO = (W + 7) & ~7;
    return g;
}
size_t dwconv_tc_plane_bytes(int B, int H, int W, int C, int K) {
    DwGeom g = dw_geom(B, H, W, C, K);
    const size_t in_bytes = (size_t)g.NB * C * g.WG * g.HP * 16;
    const size_t out_bytes = (size_t)B * C * H * g.WO * 2;
    return ((in_bytes + 255) & ~(size_t)255) + ((out_bytes + 255) & ~(size_t)255);
}

__host__ __device__ inline int dw_slab_row_words(int W, int C) {
    const int n = W * (C / 2 + 1);
    return n + ((1 - n) % 32 + 32) % 32;
}

// ---------------------------------------------------------------- token-major -> padded planes
// CTA = (plane stack, RPC consecutive PLANE rows): coalesced read of the image rows among them ([W][C] slabs),
// transpose through shared memory, then each thread emits 16-byte chunks (8 columns of one channel, one
// plane row); 8 consecutive rows of one (channel, x-group) are 128 contiguous bytes of the plane.  The kernel
// writes EVERY chunk of the planes - image cells and zeros everywhere else (PAD rows above / between / below the
// stacked frames, PAD columns left and right, the slack rows and column groups the 128-row / 64-column operand
// views reach into) - so the planes need no memset and stale workspace bytes never enter an MMA.
template <int RPC>
__global__ void __launch_bounds__(256) dw_plane_pack_kernel(const bf16* __restrict__ in, bf16* __restrict__ planes, DwGeom g, int B) {
    extern __shared__ __align__(16) uint32_t slab[];          // [8 rows][RS]: per row [W][C/2 + 1] channel pairs + padding
    const int stack = blockIdx.y, pr0 = blockIdx.x * RPC;
    const int C = g.C, W = g.W, C2 = C / 2, LD = C2 + 1;
    // phase 2 reads with a warp = 8 plane rows x 4 consecutive x-groups: word address r * RS + xg * 8 * LD + const.  LD = 1
    // (mod 4) puts the x-groups 8 banks apart; RS = 1 (mod 32) puts the rows on the banks in between - conflict-free (with
    // RS = W * LD the eight rows fell on four banks, the x-groups on the same four: 8-way conflicts on every load)
    const int RS = dw_slab_row_words(W, C);
    pdl_wait();
    // every plane row an A view can touch (HP >= PAD + F x (H + PAD)): the rows below the last frame's halo are only
    // multiplied by all-zero Toeplitz blocks (taps dy >= K of the last group of eight), but a stale NaN would survive that
    const int rows = min(RPC, g.HP - pr0);
    // plane row pr -> (stacked frame f, image row y) -> source row index, or -1 for a zero row
    auto src_row = [&](int r) {
        const int qr = pr0 + r - g.PAD;                        // row relative to the first frame's first row
        int f = 0, y = qr;                                     // F is 1 - 3: subtract instead of an integer division
        for (; f < g.F && y >= g.RS; ++f) y -= g.RS;
        const int frame = stack * g.F + f;
        return (r < rows && qr >= 0 && f < g.F && y < g.H && frame < B) ? frame * g.H + y : -1;
    };
    // phase 1: the image rows among the RPC, 16-byte loads (8 channels), rows one after the other
    {
        const int V = C2 / 4, nvec = W * V;                   // uint4 per pixel (C % 8 == 0), per row
        const bool vp2 = (V & (V - 1)) == 0;                  // a power of two for every served C: shift / mask, not ~50
        const int vsh = 31 - __clz(V);                        // instructions of integer division per 16-byte load
        for (int r = 0; r < RPC; ++r) {
            const int sr = src_row(r);
            if (sr < 0) continue;                             // block-uniform
            const uint4* src = reinterpret_cast<const uint4*>(in) + (size_t)sr * nvec;
            for (int i = threadIdx.x; i < nvec; i += 256) {
                const uint4 v = src[i];
                const int px = vp2 ? i >> vsh : i / V, q4 = vp2 ? i & (V - 1) : i % V;
                uint32_t* d = slab + r * RS + px * LD + q4 * 4;
                d[0] = v.x; d[1] = v.y; d[2] = v.z; d[3] = v.w;
            }
        }
    }
    __syncthreads();
    pdl_trigger();
    // phase 2: thread = (plane row r, slot); a slot walks over the (channel pair, x-group) chunks.  8 consecutive threads
    // (r = 0..7) write 128 contiguous bytes of a plane.  Chunks without image cells are plain zero stores.
    const int r = threadIdx.x & (RPC - 1);
    if (r >= rows) return;
    const bool img_row = src_row(r) >= 0;
    const int npair = C2 * g.WG;
    int pair = threadIdx.x / RPC, c2 = pair / g.WG, xg = pair - c2 * g.WG;
    const size_t plane_stride = (size_t)g.WG * g.HP * 8;       // elements per channel plane
    for (; pair < npair; pair += 256 / RPC) {
        const int xb = xg * 8 - g.PAD;                         // image column of the chunk's first element
        uint4 lo = make_uint4(0u, 0u, 0u, 0u), hi = lo;
        if (img_row && xb + 7 >= 0 && xb < W) {
            uint32_t v[8];
            const uint32_t* sp = slab + r * RS + xb * LD + c2;
#pragma unroll
            for (int j = 0; j < 8; ++j) v[j] = (xb + j >= 0 && xb + j < W) ? sp[j * LD] : 0u;
            lo.x = __byte_perm(v[0], v[1], 0x5410); hi.x = __byte_perm(v[0], v[1], 0x7632);
            lo.y = __byte_perm(v[2], v[3], 0x5410); hi.y = __byte_perm(v[2], v[3], 0x7632);
            lo.z = __byte_perm(v[4], v[5], 0x5410); hi.z = __byte_perm(v[4], v[5], 0x7632);
            lo.w = __byte_perm(v[6], v[7], 0x5410); hi.w = __byte_perm(v[6], v[7], 0x7632);
        }
        const size_t off = ((((size_t)stack * C + 2 * c2) * g.WG + xg) * g.HP + (pr0 + r)) * 8;
        *reinterpret_cast<uint4*>(planes + off) = lo;
        *reinterpret_cast<uint4*>(planes + off + plane_stride) = hi;
        xg += 256 / RPC;
        while (xg >= g.WG) { xg -= g.WG; ++c2; }
    }
}

// ---------------------------------------------------------------- the Toeplitz GEMM
struct DwBars {
    uint64_t t_full, t_empty, a_full[3], a_empty[3], acc_full[2], acc_empty[2];
    uint32_t tmem_slot;
};

// Work items are (channel, column tile, frame stack, row block), channel-major; every CTA takes an equal
// contiguous share, so the grid is one balanced wave and the Toeplitz blocks are reloaded only when
// a CTA's share crosses a channel boundary.
struct DwItem { int c, xt, b, mt; };                      // b = plane stack index
__device__ __forceinline__ DwItem dw_item(int i, const DwGeom& g) {
    DwItem it;
    it.mt = i % g.nM; i /= g.nM;
    it.b = i % g.NB; i /= g.NB;
    it.xt = i % g.nX;
    it.c = i / g.nX;
    return it;
}
// A CTA's items are consecutive: decoded once (four integer divisions, ~25 instructions each - per item and thread that was
// a third of the epilogue's instruction count), then stepped
__device__ __forceinline__ void dw_next(DwItem& it, const DwGeom& g) {
    if (++it.mt < g.nM) return;
    it.mt = 0;
    if (++it.b < g.NB) return;
    it.b = 0;
    if (++it.xt < g.nX) return;
    it.xt = 0;
    ++it.c;
}

constexpr int kXchLd = 36;                                 // floats per exchanged row (16-byte aligned, bank-staggered)
constexpr int kXchRows = kDwNB * (kDwNB - 1) / 2;           // rows a quarter publishes per item: sum_{b=1..NB-1} b
constexpr size_t kXchBytes = 2 * 3 * kXchRows * kXchLd * sizeof(float);
constexpr int kDwParts = 2;                                // epilogue warps per TMEM lane quarter
constexpr int kDwCols = 32 / kDwParts;                     // output columns per epilogue thread
constexpr int kDwEpiWarps = 4 * kDwParts;
constexpr int kDwThreads = (kDwEpiWarps + 2) * 32;         // + bulk-copy producer warp + MMA issuer warp
constexpr size_t kBndBytes = 2 * kDwEpiWarps * (kDwNB - 1) * kDwCols * sizeof(float);   // per (item parity, warp): boundary rows

template <int NC> __device__ __forceinline__ void tmem_ld(uint32_t taddr, float (&v)[NC]);
template <> __device__ __forceinline__ void tmem_ld<16>(uint32_t taddr, float (&v)[16]) { umma::tmem_ld16(taddr, v); }
template <> __device__ __forceinline__ void tmem_ld<8>(uint32_t taddr, float (&v)[8]) {
    uint32_t r[8];
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];\n"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                 : "r"(taddr)
                 : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;\n" ::: "memory");
#pragma unroll
    for (int i = 0; i < 8; ++i) v[i] = __uint_as_float(r[i]);
}

__global__ void __launch_bounds__(kDwThreads) dwconv_tc_kernel(const bf16* __restrict__ planes, const bf16* __restrict__ toep,
                                                        const float* __restrict__ shift, bf16* __restrict__ planar_out,
                                                        int B, DwGeom g, int items_per_cta, int total_items) {
    extern __shared__ __align__(128) uint8_t smem[];
    __shared__ DwBars bars;
    const int tid = threadIdx.x, warp = umma::warp_idx_sync(), lane = tid & 31;
    constexpr uint32_t t_blk = 2 * kDwN * 16;                  // bytes of one (a, ks) block  [2 k-groups][kDwN = (b, n)][8]
    const uint32_t t_bytes = g.NA * g.KS * t_blk;
    const uint32_t lbo_a = g.HP * 16;
    const uint32_t a_bytes = 2 * g.KS * lbo_a;
    uint8_t* t_sm = smem;
    uint8_t* a_sm = smem + t_bytes;                            // [3][a_stride]
    const uint32_t a_stride = (a_bytes + 127) & ~127u;
    float* xch = reinterpret_cast<float*>(a_sm + 3 * (size_t)a_stride);   // [2][3 quarters][28 rows][kXchLd]
    float* bnd = xch + kXchBytes / sizeof(float);                         // [2][epilogue warps][7 rows][kDwCols]
    const int i0 = blockIdx.x * items_per_cta, i1 = min(i0 + items_per_cta, total_items);

    if (tid == 0) {
        umma::mbar_init(&bars.t_full, 1);
        umma::mbar_init(&bars.t_empty, 1);
        for (int i = 0; i < 3; ++i) { umma::mbar_init(&bars.a_full[i], 1); umma::mbar_init(&bars.a_empty[i], 1); }
        for (int i = 0; i < 2; ++i) { umma::mbar_init(&bars.acc_full[i], 1); umma::mbar_init(&bars.acc_empty[i], kDwEpiWarps * 32); }
        umma::fence_mbar_init();
    }
    if (warp == kDwEpiWarps) umma::tmem_alloc(&bars.tmem_slot, 2 * kDwAcc);
    umma::fence_before_sync();
    __syncthreads();
    umma::fence_after_sync();
    const uint32_t tmem = bars.tmem_slot;

    if (warp < kDwEpiWarps) {
        pdl_wait();                       // the planar output may still be read by the previous kernels of the stream
        // ---------------- epilogue: kDwParts warps per TMEM lane quarter.  Thread = (accumulator row m, kDwCols of the
        // 32 output columns):  out[m][n] = sum_b E_b[m + b][n]
        constexpr int NC = kDwCols;
        const int q = warp & 3, part = warp >> 2, row = q * 32 + lane;
        DwItem it = dw_item(i0, g);
        for (int i = i0; i < i1; ++i, dw_next(it, g)) {
            const int n = i - i0, ab = n & 1;
            const float sh = shift[it.c];
            float* xw = xch + (size_t)ab * (3 * kXchRows * kXchLd) + part * NC;
            float* bw = bnd + ((size_t)ab * kDwEpiWarps + warp) * ((kDwNB - 1) * NC);
            umma::mbar_wait(&bars.acc_full[ab], (n >> 1) & 1);
            umma::fence_after_sync();
            float acc[NC];
#pragma unroll
            for (int b = 0; b < kDwNB; ++b) {
                float e[NC];
                tmem_ld<NC>(umma::tmem_addr(tmem, q * 32, ab * kDwAcc + b * 32 + part * NC), e);
                if (b == 0) {
#pragma unroll
                    for (int j = 0; j < NC; ++j) acc[j] = e[j];
                } else {
                    if (q > 0 && lane < b) {                   // rows the quarter below needs: E_b[32 q + lane]
                        float* dst = xw + ((size_t)(q - 1) * kXchRows + b * (b - 1) / 2 + lane) * kXchLd;
#pragma unroll
                        for (int j = 0; j < NC; j += 4) *reinterpret_cast<float4*>(dst + j) = make_float4(e[j], e[j + 1], e[j + 2], e[j + 3]);
                    }
                    float sv[NC];
#pragma unroll
                    for (int j = 0; j < NC; ++j) sv[j] = __shfl_down_sync(0xffffffffu, e[j], b);
                    if (lane + b < 32) {
#pragma unroll
                        for (int j = 0; j < NC; ++j) acc[j] += sv[j];
                    }
                }
            }
            umma::fence_before_sync();
            asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];\n" ::"r"(umma::smem_u32(&bars.acc_empty[ab])) : "memory");
            asm volatile("bar.sync 1, %0;\n" ::"n"(kDwEpiWarps * 32) : "memory");   // boundary rows of this item are published
            if (q < 3) {
                // rows 25..31 of the quarter take E_b[m + b] for m + b >= 32 from the exchange: lane -> (target row 25 + t,
                // four of the NC columns) sums its b's, then hands the partial row over through `bw`
                constexpr int QPR = NC / 4;                    // float4 per row
                const int t = lane / QPR, cq = (lane % QPR) * 4;
                if (t < kDwNB - 1) {
                    float4 sacc = make_float4(0.f, 0.f, 0.f, 0.f);
                    for (int b = kDwNB - 1 - t; b < kDwNB; ++b) {
                        const float4 v = *reinterpret_cast<const float4*>(xw + ((size_t)q * kXchRows + b * (b - 1) / 2 + (t + b - (kDwNB - 1))) * kXchLd + cq);
                        sacc.x += v.x; sacc.y += v.y; sacc.z += v.z; sacc.w += v.w;
                    }
                    *reinterpret_cast<float4*>(bw + t * NC + cq) = sacc;
                }
                __syncwarp();
                if (lane >= 33 - kDwNB) {
#pragma unroll
                    for (int j = 0; j < NC; j += 4) {
                        const float4 v = *reinterpret_cast<const float4*>(bw + (lane - (33 - kDwNB)) * NC + j);
                        acc[j] += v.x; acc[j + 1] += v.y; acc[j + 2] += v.z; acc[j + 3] += v.w;
                    }
                }
                __syncwarp();                                  // `bw` is rewritten two items later (ab parity) - cheap insurance
            }
            const int m = it.mt * kDwMS + row, x0 = it.xt * 32 + part * NC;
            int f = 0, y = m;                                  // stacked frame and its row (F is 1 - 3: no division)
            for (; f < g.F && y >= g.RS; ++f) y -= g.RS;
            const int frame = it.b * g.F + f;
            if (row < kDwMS && f < g.F && y < g.H && frame < B) {
                bf16* dst = planar_out + (((size_t)frame * g.C + it.c) * g.H + y) * g.WO + x0;
#pragma unroll
                for (int j = 0; j < NC; j += 8) {
                    if (x0 + j < g.WO) {                       // WO % 8 == 0: a chunk is inside the (padded) row or not at all
                        uint4 u;
                        u.x = umma::pack_bf16(fmaxf(acc[j + 0] + sh, 0.f), fmaxf(acc[j + 1] + sh, 0.f));
                        u.y = umma::pack_bf16(fmaxf(acc[j + 2] + sh, 0.f), fmaxf(acc[j + 3] + sh, 0.f));
                        u.z = umma::pack_bf16(fmaxf(acc[j + 4] + sh, 0.f), fmaxf(acc[j + 5] + sh, 0.f));
                        u.w = umma::pack_bf16(fmaxf(acc[j + 6] + sh, 0.f), fmaxf(acc[j + 7] + sh, 0.f));
                        *reinterpret_cast<uint4*>(dst + j) = u;
                    }
                }
            }
        }
    } else if (warp == kDwEpiWarps) {
        // ---------------- producer: Toeplitz blocks per channel, one bulk copy per work item
        {
            int cur_c = -1, nt = 0;
            DwItem it = dw_item(i0, g);
            for (int i = i0; i < i1; ++i, dw_next(it, g)) {
                const int n = i - i0, s = n % 3;
                if (it.c != cur_c) {
                    if (nt > 0) umma::mbar_wait(&bars.t_empty, (nt - 1) & 1);   // MMAs on the old blocks are done
                    if (umma::elect_one()) {
                        umma::mbar_expect_tx(&bars.t_full, t_bytes);
                        const uint8_t* src = reinterpret_cast<const uint8_t*>(toep) + (size_t)it.c * t_bytes;
                        for (uint32_t off = 0; off < t_bytes; off += 4 * t_blk)
                            umma::bulk_g2s(t_sm + off, src + off, min(4 * t_blk, t_bytes - off), &bars.t_full);
                    }
                    __syncwarp();
                    cur_c = it.c;
                    ++nt;
                }
                if (i == i0) pdl_wait();  // the first Toeplitz blocks (weights) are on their way; the planes are the previous kernel's
                if (n >= 3) umma::mbar_wait(&bars.a_empty[s], ((n / 3) - 1) & 1);
                const bf16* src = planes + ((((size_t)it.b * g.C + it.c) * g.WG + 4 * it.xt) * g.HP) * 8;
                umma::bulk_load(a_sm + (size_t)s * a_stride, src, a_bytes, &bars.a_full[s]);
            }
        }
    } else {
        // ---------------- MMA issuer (warp-uniform control flow; one elected lane issues)
        {
            const uint32_t idesc = umma::idesc_bf16(128, kDwN);
            const uint64_t tdesc0 = umma::smem_desc(umma::smem_u32(t_sm), kDwN * 16);
            const uint32_t as0 = umma::smem_u32(a_sm);
            int cur_c = -1, nt = 0;
            DwItem it = dw_item(i0, g);
            for (int i = i0; i < i1; ++i, dw_next(it, g)) {
                const int n = i - i0, s = n % 3, ab = n & 1;
                if (it.c != cur_c) {
                    if (nt > 0) umma::commit(&bars.t_empty);
                    umma::mbar_wait(&bars.t_full, nt & 1);
                    cur_c = it.c;
                    ++nt;
                }
                umma::mbar_wait(&bars.a_full[s], (n / 3) & 1);
                if (n >= 2) umma::mbar_wait(&bars.acc_empty[ab], ((n >> 1) - 1) & 1);
                umma::fence_after_sync();
                // vertical taps dy = 8 a + b: the eight b's of one a share ONE (8-row aligned) A view and sit side by
                // side along N (256 = 8 x 32 columns); their row shift b is applied by the epilogue
                uint64_t ad = umma::smem_desc(as0 + s * a_stride + (uint32_t)(it.mt * kDwMS) * 16, lbo_a);
                uint64_t td = tdesc0;
                const uint32_t dcol = tmem + ab * kDwAcc;
                for (int a = 0; a < g.NA; ++a) {
                    uint64_t adj = ad;
                    for (int j = 0; j < g.KS; ++j) {
                        umma::mma_bf16(dcol, adj, td, idesc, (a | j) != 0);
                        adj = umma::desc_advance(adj, 2 * lbo_a);
                        td = umma::desc_advance(td, t_blk);
                    }
                    ad = umma::desc_advance(ad, kDwNB * 16);   // next group of vertical taps: kDwNB rows down (any 16-byte
                                                               // aligned start is a legal operand view; measured: no penalty)
                }
                umma::commit(&bars.a_empty[s]);
                umma::commit(&bars.acc_full[ab]);
            }
        }
    }
    pdl_trigger();                         // this CTA's work is done: the next kernel of the stream may start its prologue
    __syncthreads();
    if (warp == kDwEpiWarps) {
        umma::fence_after_sync();
        umma::tmem_dealloc(tmem, 2 * kDwAcc);
    }
}

int dwconv_tc(const void* in, const void** planar_out_p, int* planar_pitch, int B, int H, int W, int C, int K, const void* toep, const float* shift,
              char* plane_ws, cudaStream_t st) {
    CFP_REQUIRE(toep != nullptr, "dwconv: bf16 path needs the packed Toeplitz blocks (cfp_lkpm_w.dw_toep)");
    CFP_REQUIRE(B <= 65535 && C <= 65535, "grid limits");
    DwGeom g = dw_geom(B, H, W, C, K);
    const size_t in_bytes = ((size_t)g.NB * C * g.WG * g.HP * 16 + 255) & ~(size_t)255;
    bf16* planes = reinterpret_cast<bf16*>(plane_ws);
    bf16* planar_out = reinterpret_cast<bf16*>(plane_ws + in_bytes);
    *planar_out_p = planar_out;          // [B][C][H][WO]; lkpm_mlp_tc reads it in place (no transpose back)
    *planar_pitch = g.WO;
    // refuse a map too tall for the GEMM's shared memory before anything is launched: a refused call leaves the
    // workspace and the stream untouched
    const uint32_t t_bytes = g.NA * g.KS * 2 * kDwN * 16, a_bytes = 2 * g.KS * g.HP * 16;
    const size_t gemm_smem = t_bytes + 3 * (size_t)((a_bytes + 127) & ~127u) + kXchBytes + kBndBytes;
    CFP_REQUIRE(gemm_smem <= 225 * 1024, "dwconv (tensor-core path): %zu B shared memory (H=%d too tall)", gemm_smem, H);
    {
        // plane rows per CTA: 4 (64 contiguous bytes per chunk column, 35 KB slab at L1: six CTAs per SM overlap their load
        // and store phases) - measured 0.149 ms per step against 0.189 ms with 8 rows
        constexpr int rpc = 4;
        const size_t smem = (size_t)rpc * dw_slab_row_words(W, C) * 4;
        CFP_REQUIRE(smem <= 200 * 1024, "dw_plane_pack: %zu B shared memory", smem);
        auto kp = dw_plane_pack_kernel<rpc>;
        if (int err = set_smem(kp, smem)) return err;
        launch_pdl(kp, dim3((g.HP + rpc - 1) / rpc, g.NB), 256, smem, st, (const bf16*)in, planes, g, B);
        if (int err = check_launch("dw_plane_pack")) return err;
    }
    {
        if (int err = set_smem(dwconv_tc_kernel, gemm_smem)) return err;
        const int total = C * g.nX * g.NB * g.nM;
        const int grid = total < sm_count() ? total : sm_count();
        const int per = (total + grid - 1) / grid;
        launch_pdl(dwconv_tc_kernel, (total + per - 1) / per, kDwThreads, gemm_smem, st, planes, (const bf16*)toep, shift, planar_out, B, g, per, total);
        if (int err = check_launch(K == 31 ? "dwconv_tc<31>" : K == 15 ? "dwconv_tc<15>" : "dwconv_tc<7>")) return err;
    }
    return 0;
}

}  // namespace cfp
