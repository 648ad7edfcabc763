// tcgen05 / TMEM / mbarrier / bulk-copy primitives for sm_100a (inline PTX, no CUTLASS).
//
// Operand layout used throughout libcfp's tensor-core kernels: the *canonical K-major,
// no-swizzle* UMMA layout with row-contiguous core matrices.  For an operand tile of R rows
// (M rows of A or N rows of B) and K bf16 columns, element (r, k) lives at byte
//
//        (k / 8) * LBO  +  r * 16  +  (k % 8) * 2          with LBO >= R * 16
//
// i.e. one 16-byte chunk (8 bf16 along K) per (row, k-group), chunks of consecutive rows
// adjacent, k-groups LBO bytes apart.  In descriptor terms: core matrix = 8 rows x 16 B
// (128 contiguous bytes), SBO (8-row group stride) = 128 B, LBO (k-group stride) = LBO.
// Two properties make this the layout of choice here:
//   * a row-shifted view of the same buffer is just "start address + shift*16": the nine taps
//     of a 3x3 convolution become nine MMAs over one staged raster (no im2col);
//   * thread r of an epilogue warp owns accumulator row r (TMEM lane r) and writes its 16-byte
//     chunks at consecutive addresses across the warp: conflict-free stores that are directly
//     the A operand of the next GEMM of a fused chain.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace cfp {
namespace umma {

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

// ---------------------------------------------------------------- descriptors
// Shared-memory matrix descriptor (cute::UMMA::SmemDescriptor bit layout): start address
// [0,14) >>4, LBO [16,30) >>4, SBO [32,46) >>4, version [46,48) = 1, layout type [61,64) = 0.
__device__ __forceinline__ uint64_t smem_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes = 128) {
    return (uint64_t)((saddr >> 4) & 0x3FFFu) | ((uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16) |
           ((uint64_t)((sbo_bytes >> 4) & 0x3FFFu) << 32) | ((uint64_t)1 << 46);
}
// Advance a descriptor's start address by `bytes` (multiple of 16; no carry out of the 14-bit field
// as long as the operand stays inside the CTA's shared-memory window).  One 64-bit add in the MMA
// issue loop instead of rebuilding the descriptor: the single issuing thread is the pacing resource.
__device__ __forceinline__ uint64_t desc_advance(uint64_t desc, uint32_t bytes) { return desc + (uint64_t)(bytes >> 4); }
// Instruction descriptor, kind::f16, A/B = bf16 K-major, D = fp32 (cute::UMMA::InstrDescriptor).
__host__ __device__ constexpr uint32_t idesc_bf16(int M, int N) {
    return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

// ---------------------------------------------------------------- warp-uniform roles
// Warp index as a value the compiler can prove warp-uniform (role branches then stay uniform and
// descriptor arithmetic lives in uniform registers).
__device__ __forceinline__ int warp_idx_sync() { return __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0); }
// elect.sync: exactly one lane of the (converged) warp gets true.  Issuing tcgen05.mma / commit /
// bulk copies under this predicate (instead of `lane == 0`) lets ptxas emit a single predicated
// UTCHMMA with uniform-register operands rather than a per-lane waterfall loop around every MMA.
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile(
        "{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}\n"
        : "=r"(pred));
    return pred != 0;
}

// ---------------------------------------------------------------- MMA issue / commit
// D[tmem] (+)= A[smem] * B[smem]^T, M x N x 16.  Called by ALL lanes of the (converged) MMA warp with
// warp-uniform arguments; one elected lane issues the instruction.
__device__ __forceinline__ void mma_bf16(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                         bool accumulate) {
    if (elect_one()) {
        asm volatile(
            "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
            "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}\n" ::"r"(d_tmem),
            "l"(adesc), "l"(bdesc), "r"(idesc), "r"((uint32_t)accumulate)
            : "memory");
    }
}
// Arrive on an mbarrier when all MMAs issued so far by this warp's elected lane have completed.
// (elect.sync picks the same lane every time for a full mask, so commit tracks the MMAs above.)
__device__ __forceinline__ void commit(uint64_t* mbar) {
    if (elect_one()) {
        asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n" ::"r"(smem_u32(mbar))
                     : "memory");
    }
}
__device__ __forceinline__ void fence_before_sync() { asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory"); }
__device__ __forceinline__ void fence_after_sync() { asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory"); }
// Make generic-proxy shared-memory writes visible to the async proxy (tcgen05.mma operand reads).
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory"); }

// ---------------------------------------------------------------- TMEM
// One full warp allocates `cols` (power of two >= 32) columns; the base address lands in *slot.
__device__ __forceinline__ void tmem_alloc(uint32_t* slot, uint32_t cols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;\n" ::"r"(smem_u32(slot)), "r"(cols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;\n" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t base, uint32_t cols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;\n" ::"r"(base), "r"(cols) : "memory");
}
// Warp-collective: lane t of warp w (w % 4 selects TMEM lanes 32*(w%4)..+31) receives columns
// [col, col+16) of accumulator row 32*(w%4)+t.
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, float (&v)[16]) {
    uint32_t r[16];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];\n"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr)
        : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;\n" ::: "memory");
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(r[i]);
}
// Asynchronous form: the load is only issued; the registers are valid after tmem_wait_ld16() on the SAME array (the wait
// names them as read-write operands, so the compiler cannot move a use above it).
__device__ __forceinline__ void tmem_ld16_async(uint32_t taddr, uint32_t (&r)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];\n"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_wait_ld16(uint32_t (&r)[16]) {
    asm volatile("tcgen05.wait::ld.sync.aligned;\n"
                 : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]), "+r"(r[8]),
                   "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15])
                 :
                 : "memory");
}
// Walk NCOLS accumulator columns of this thread's TMEM lane in 16-column pieces, f(c0, v[16]) on each, with the load of
// piece i+1 in flight while piece i is processed (a tcgen05.ld + wait per piece exposes ~100 cycles of TMEM latency
// every 16 columns - every epilogue used to pay that).
template <int NCOLS, class F>
__device__ __forceinline__ void tmem_for_each16(uint32_t taddr, F&& f) {
    static_assert(NCOLS % 16 == 0, "16-column pieces");
    uint32_t buf[2][16];
    tmem_ld16_async(taddr, buf[0]);
    tmem_wait_ld16(buf[0]);
#pragma unroll
    for (int i = 0; i < NCOLS / 16; ++i) {
        if (i + 1 < NCOLS / 16) tmem_ld16_async(taddr + (uint32_t)((i + 1) * 16), buf[(i + 1) & 1]);
        float v[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) v[j] = __uint_as_float(buf[i & 1][j]);
        f(i * 16, v);
        if (i + 1 < NCOLS / 16) tmem_wait_ld16(buf[(i + 1) & 1]);
    }
}
__device__ __forceinline__ uint32_t tmem_addr(uint32_t base, int lane, int col) {
    return base + ((uint32_t)lane << 16) + (uint32_t)col;
}

// ---------------------------------------------------------------- mbarrier
__device__ __forceinline__ void mbar_init(uint64_t* mbar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"(smem_u32(mbar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint64_t* mbar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(smem_u32(mbar)), "r"(bytes) : "memory");
}
// try_wait is potentially blocking: the hardware may suspend the thread until the phase completes or a time limit
// passes.  A suspend-time hint was measured slower (step 4.05 -> 4.09 ms): the wake-up costs more than the polling.
__device__ __forceinline__ bool mbar_try_wait(uint64_t* mbar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}\n"
        : "=r"(ok)
        : "r"(smem_u32(mbar)), "r"(parity)
        : "memory");
    return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t* mbar, uint32_t parity) {
    while (!mbar_try_wait(mbar, parity)) {
    }
}

// ---------------------------------------------------------------- bulk async copy (TMA engine, 1-D)
// global -> shared, completion signalled on `mbar` via complete_tx; bytes % 16 == 0, 16-B aligned.
__device__ __forceinline__ void bulk_g2s(void* smem_dst, const void* gmem_src, uint32_t bytes, uint64_t* mbar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n" ::"r"(
                     smem_u32(smem_dst)),
                 "l"(gmem_src), "r"(bytes), "r"(smem_u32(mbar))
                 : "memory");
}

// expect_tx + bulk copy by one elected lane; called by all lanes of the (converged) producer warp.
__device__ __forceinline__ void bulk_load(void* smem_dst, const void* gmem_src, uint32_t bytes, uint64_t* mbar) {
    if (elect_one()) {
        mbar_expect_tx(mbar, bytes);
        bulk_g2s(smem_dst, gmem_src, bytes, mbar);
    }
}

// ---------------------------------------------------------------- packed fp32x2 arithmetic (sm_100: FFMA2 / FADD2 / FMUL2)
// Two IEEE fp32 operations per instruction on a 64-bit register pair; the row-wise epilogues (LayerNorm, attention
// apply) are instruction-issue bound at small C, and every lane computes exactly what fmaf / + / * would.
typedef unsigned long long f32x2;
__device__ __forceinline__ f32x2 pack2(float lo, float hi) { f32x2 r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi)); return r; }
__device__ __forceinline__ void unpack2(f32x2 v, float& lo, float& hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v)); }
__device__ __forceinline__ f32x2 fma2(f32x2 a, f32x2 b, f32x2 c) { f32x2 d; asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c)); return d; }
__device__ __forceinline__ f32x2 add2(f32x2 a, f32x2 b) { f32x2 d; asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b)); return d; }
__device__ __forceinline__ f32x2 mul2(f32x2 a, f32x2 b) { f32x2 d; asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b)); return d; }

// ---------------------------------------------------------------- packing helpers
__device__ __forceinline__ uint32_t pack_bf16(float lo, float hi) {
    __nv_bfloat162 t = __floats2bfloat162_rn(lo, hi);
    return *reinterpret_cast<uint32_t*>(&t);
}
// 8 consecutive-K values of one row -> the 16-byte chunk of the canonical layout.
__device__ __forceinline__ void store_chunk(void* tile, uint32_t lbo_bytes, int row, int kgroup, const float (&v)[8]) {
    uint4 u;
    u.x = pack_bf16(v[0], v[1]);
    u.y = pack_bf16(v[2], v[3]);
    u.z = pack_bf16(v[4], v[5]);
    u.w = pack_bf16(v[6], v[7]);
    *reinterpret_cast<uint4*>(reinterpret_cast<char*>(tile) + (size_t)kgroup * lbo_bytes + (size_t)row * 16) = u;
}

}  // namespace umma
}  // namespace cfp
