// Thin PTX wrappers for the Blackwell (sm_100a) tensor-core path: mbarriers, TMA tile loads,
// tcgen05.mma (kind::i8, kind::mxf4) with operands from shared memory or tensor memory, TMEM allocation and
// tcgen05.ld/st.  Shared by the Hamming scan (scan_mma.cu), the signature filter (sig_filter.cu) and the
// exact-similarity path (exact.cu).  Nothing here comes from the reference (it has no tensor-core code).
#pragma once

#include <cuda.h>
#include <cuda_runtime.h>
#include <cstdint>

struct em2_context;

namespace em2 {
namespace tc05 {

__device__ __forceinline__ uint32_t smemAddr(const void* p) { return uint32_t(__cvta_generic_to_shared(p)); }

// ---- mbarriers ---------------------------------------------------------------------------------
__device__ __forceinline__ void mbarInit(uint64_t* bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smemAddr(bar)), "r"(count));
}
__device__ __forceinline__ void mbarInitFence()
{
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbarExpectTx(uint64_t* bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smemAddr(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbarArrive(uint64_t* bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smemAddr(bar)) : "memory");
}
__device__ __forceinline__ void mbarWait(uint64_t* bar, uint32_t parity)
{
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "WAIT_LOOP:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE;\n\t"
        "bra WAIT_LOOP;\n\t"
        "DONE:\n\t"
        "}\n" ::"r"(smemAddr(bar)),
        "r"(parity)
        : "memory");
}

// ---- TMA ---------------------------------------------------------------------------------------
// 2-D tile load; coordinates are (innermost = byte offset along K, row).
__device__ __forceinline__ void tmaLoad2d(void* smemDst, const CUtensorMap* map, uint64_t* bar, int32_t c0, int32_t c1)
{
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(smemAddr(smemDst)), "l"(map), "r"(smemAddr(bar)), "r"(c0), "r"(c1)
        : "memory");
}
__device__ __forceinline__ void prefetchMap(const CUtensorMap* map)
{
    asm volatile("prefetch.tensormap [%0];" ::"l"(map) : "memory");
}

// One lane of the (converged) warp: the issue loops of the MMA warps run on all 32 lanes with uniform control flow and
// only the tcgen05 instructions sit behind this predicate -- inside an `if (lane == 0)` region the compiler cannot keep
// the descriptors in uniform registers and wraps every tcgen05.mma in an ELECT / R2UR.BROADCAST / BRA.U.ANY loop
// (~20 SASS instructions per MMA from one thread: as long as the MMA itself at K = 32).
__device__ __forceinline__ bool electOne()
{
    uint32_t pred;
    asm volatile(
        "{\n\t"
        ".reg .pred P;\n\t"
        "elect.sync _|P, 0xffffffff;\n\t"
        "selp.u32 %0, 1, 0, P;\n\t"
        "}\n"
        : "=r"(pred));
    return pred != 0;
}

// ---- tcgen05 -----------------------------------------------------------------------------------
__device__ __forceinline__ void fenceBefore() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void fenceAfter() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void commit(uint64_t* bar)
{
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smemAddr(bar))
                 : "memory");
}
// D[tmem] (+)= A[tmem] * B[smem]
__device__ __forceinline__ void mmaI8Ts(uint32_t tmemD, uint32_t tmemA, uint64_t descB, uint32_t idesc, uint32_t accumulate)
{
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::i8 [%0], [%1], %2, %3, p;\n\t"
        "}\n" ::"r"(tmemD),
        "r"(tmemA), "l"(descB), "r"(idesc), "r"(accumulate)
        : "memory");
}
// D[tmem] (+)= A[smem] * B[smem]
__device__ __forceinline__ void mmaI8Ss(uint32_t tmemD, uint64_t descA, uint64_t descB, uint32_t idesc, uint32_t accumulate)
{
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n\t"
        "}\n" ::"r"(tmemD),
        "l"(descA), "l"(descB), "r"(idesc), "r"(accumulate)
        : "memory");
}
// Whole-warp TMEM allocation of `cols` (power of two >= 32) columns; the base address lands in *slot.
__device__ __forceinline__ void tmemAlloc(uint32_t* slot, uint32_t cols)
{
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smemAddr(slot)), "r"(cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmemDealloc(uint32_t base, uint32_t cols)
{
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(base), "r"(cols) : "memory");
}
__device__ __forceinline__ void tmemStore32(uint32_t taddr, const uint32_t (&v)[32])
{
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
        "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
        "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};"
        ::"r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]),
          "r"(v[9]), "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15]), "r"(v[16]),
          "r"(v[17]), "r"(v[18]), "r"(v[19]), "r"(v[20]), "r"(v[21]), "r"(v[22]), "r"(v[23]), "r"(v[24]),
          "r"(v[25]), "r"(v[26]), "r"(v[27]), "r"(v[28]), "r"(v[29]), "r"(v[30]), "r"(v[31])
        : "memory");
}
__device__ __forceinline__ void tmemStoreWait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
// 32 consecutive accumulator columns of this thread's TMEM lane.
__device__ __forceinline__ void tmemLoad32(uint32_t taddr, uint32_t (&v)[32])
{
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
          "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
          "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
          "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
        : "r"(taddr));
}
__device__ __forceinline__ void tmemLoadWait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// ---- CTA pairs (cta_group::2): two CTAs of a cluster, on the two SMs of one TPC, run ONE M=256 MMA -----------
// Each CTA holds its 128 rows of A and D in its own TMEM and HALF of the B tile (N/2 rows) in its own shared
// memory; the leader (cluster rank 0) issues the instruction.  In a 2-CTA cluster the rank sits in bit 24 of a
// shared-memory address, so clearing it names the same location in the leader CTA.
constexpr uint32_t kPeerBitMask = 0xFEFFFFFFu;
__device__ __forceinline__ uint32_t clusterRank()
{
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void clusterSync()
{
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ uint32_t leaderAddr(const void* p) { return smemAddr(p) & kPeerBitMask; }
// arrive on the LEADER CTA's copy of a barrier (from either CTA of the pair)
__device__ __forceinline__ void mbarArriveLeader(uint64_t* bar)
{
    asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(leaderAddr(bar)) : "memory");
}
// TMA tile load into THIS CTA's shared memory whose completion bytes are credited to the leader's barrier
__device__ __forceinline__ void tmaLoad2dPair(void* smemDst, const CUtensorMap* map, uint64_t* bar, int32_t c0, int32_t c1)
{
    const uint64_t evictNormal = 0x1000000000000000ull;
    asm volatile(
        "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint"
        " [%0], [%1, {%3, %4}], [%2], %5;"
        ::"r"(smemAddr(smemDst)), "l"(map), "r"(leaderAddr(bar)), "r"(c0), "r"(c1), "l"(evictNormal)
        : "memory");
}
// completion of all prior MMAs of the pair -> one arrival on the same barrier offset in BOTH CTAs
__device__ __forceinline__ void commitPair(uint64_t* bar)
{
    const uint16_t mask = 3;
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                 ::"r"(smemAddr(bar)), "h"(mask)
                 : "memory");
}
__device__ __forceinline__ void mmaI8TsPair(uint32_t tmemD, uint32_t tmemA, uint64_t descB, uint32_t idesc, uint32_t accumulate)
{
    const uint32_t z = 0;
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::i8 [%0], [%1], %2, %3, {%5, %5, %5, %5, %5, %5, %5, %5}, p;\n\t"
        "}\n" ::"r"(tmemD),
        "r"(tmemA), "l"(descB), "r"(idesc), "r"(accumulate), "r"(z)
        : "memory");
}
__device__ __forceinline__ void mmaI8SsPair(uint32_t tmemD, uint64_t descA, uint64_t descB, uint32_t idesc, uint32_t accumulate)
{
    const uint32_t z = 0;
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::i8 [%0], %1, %2, %3, {%5, %5, %5, %5, %5, %5, %5, %5}, p;\n\t"
        "}\n" ::"r"(tmemD),
        "l"(descA), "l"(descB), "r"(idesc), "r"(accumulate), "r"(z)
        : "memory");
}
// kind::mxf4 (e2m1 operands packed two per byte, K = 64 per instruction, f32 accumulator), both operands in shared
// memory; sfA / sfB: tensor-memory addresses of the UE8M0 scale factors (one per 32 elements along K)
__device__ __forceinline__ void mmaMxf4Ss(uint32_t tmemD, uint64_t descA, uint64_t descB, uint32_t idesc, uint32_t sfA, uint32_t sfB,
                                          uint32_t accumulate)
{
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %6, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::mxf4.block_scale.scale_vec::2X [%0], %1, %2, %3, [%4], [%5], p;\n\t"
        "}\n" ::"r"(tmemD),
        "l"(descA), "l"(descB), "r"(idesc), "r"(sfA), "r"(sfB), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void mmaMxf4SsPair(uint32_t tmemD, uint64_t descA, uint64_t descB, uint32_t idesc, uint32_t sfA, uint32_t sfB,
                                              uint32_t accumulate)
{
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %6, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::mxf4.block_scale.scale_vec::2X [%0], %1, %2, %3, [%4], [%5], p;\n\t"
        "}\n" ::"r"(tmemD),
        "l"(descA), "l"(descB), "r"(idesc), "r"(sfA), "r"(sfB), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void tmemAllocPair(uint32_t* slot, uint32_t cols)
{
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smemAddr(slot)), "r"(cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmemDeallocPair(uint32_t base, uint32_t cols)
{
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(base), "r"(cols) : "memory");
}

// Shared-memory matrix descriptor: K-major operand tile whose rows are 128 bytes (one swizzle atom) apart and
// whose 8-row groups are 1024 bytes apart, 128-byte swizzle (the layout a TMA box of {128 bytes, rows} with
// CU_TENSOR_MAP_SWIZZLE_128B produces).  Encoding per the PTX ISA matrix-descriptor table, version 1 (sm_100).
__device__ __forceinline__ uint64_t makeSmemDesc(uint32_t saddr)
{
    uint64_t d = 0;
    d |= uint64_t((saddr & 0x3FFFF) >> 4);          // start address, bits [0,14)
    d |= uint64_t(1) << 16;                          // leading byte offset (ignored for swizzled K-major; 1)
    d |= uint64_t(1024 >> 4) << 32;                  // stride byte offset = 1024 B between 8-row groups
    d |= uint64_t(1) << 46;                          // descriptor version
    d |= uint64_t(2) << 61;                          // layout type: SWIZZLE_128B
    return d;
}

// Instruction descriptor of kind::i8: D = s32, A/B 8-bit K-major, signedness per operand.
__host__ __device__ constexpr uint32_t instrDescI8(bool aSigned, bool bSigned, uint32_t m, uint32_t n)
{
    return (2u << 4)                          // c_format = S32
           | (uint32_t(aSigned ? 1 : 0) << 7) // a_format: 0 = unsigned 8-bit, 1 = signed 8-bit
           | (uint32_t(bSigned ? 1 : 0) << 10)
           | ((n >> 3) << 17)                 // n_dim
           | ((m >> 4) << 24);                // m_dim
}

// Instruction descriptor of kind::mxf4 (block-scaled): D = f32, A/B e2m1 K-major, UE8M0 scale factors, dense K = 64.
__host__ __device__ constexpr uint32_t instrDescMxf4(uint32_t m, uint32_t n)
{
    return (1u << 7)                          // a_format: e2m1
           | (1u << 10)                       // b_format: e2m1
           | ((n >> 3) << 17)                 // n_dim
           | (1u << 23)                       // scale_format: UE8M0
           | ((m >> 4) << 24);                // m_dim
}

}  // namespace tc05

// Host: 2-D uint8 tensor map over a row-major [rows][pitchBytes] matrix whose logical width is `widthBytes`
// (out-of-bounds bytes/rows read as zero), box = {128 bytes, boxRows}, 128-byte swizzle.
int makeTensorMapU8(::em2_context* ctx, CUtensorMap* map, const void* base, uint64_t rows, uint64_t widthBytes,
                    uint64_t pitchBytes, uint32_t boxRows);

}  // namespace em2
