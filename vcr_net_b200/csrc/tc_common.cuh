// sm_100a building blocks shared by the tensor-core kernels: mbarrier, TMA (cp.async.bulk.tensor),
// TMEM allocation, tcgen05.mma / commit / ld wrappers and the UMMA descriptors.
// Field layouts follow the PTX ISA "tcgen05 matrix / instruction descriptor" tables (the same bit
// positions CUTLASS's cute/arch/mma_sm100_desc.hpp encodes).
#pragma once
#include <cuda.h>
#include <cuda_fp16.h>
#include <cuda_bf16.h>
#include "common.cuh"

namespace tc {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// ---------------------------------------------------------------- operand format ---------------------
__device__ __forceinline__ uint32_t pack_h2(float a, float b, int bf16) {
    if (bf16) {
        __nv_bfloat162 v = __floats2bfloat162_rn(a, b);
        return *reinterpret_cast<uint32_t*>(&v);
    }
    __half2 v = __floats2half2_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&v);
}
__device__ __forceinline__ float lo_part(float x, int bf16) {
    // residual of the 16-bit rounding, scaled by 2^11 (fp16) / 2^8 (bf16) so it stays normal
    if (bf16) return (x - __bfloat162float(__float2bfloat16_rn(x))) * 256.f;
    return (x - __half2float(__float2half_rn(x))) * 2048.f;
}

// ---------------------------------------------------------------- exp2 -------------------------------
// (Round 2 tried moving a share of the attention kernels' exponentials to the FMA pipe -- Cody-Waite split + degree-6
// polynomial, 7.9e-8 relative error -- on the theory that MUFU.EX2 paced the softmax: no gain at any share, in either
// kernel (profiles/r02_colsum_diag.txt, r02_flash_organisations_v2.txt), so every exponential stays on the XU pipe.)
__device__ __forceinline__ float ex2_mufu(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

// ---------------------------------------------------------------- mbarrier --------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    const uint32_t addr = smem_u32(bar);
    uint32_t done;
    do {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done)
            : "r"(addr), "r"(parity)
            : "memory");
    } while (!done);
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "elect.sync _|p, 0xffffffff;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(pred));
    return pred != 0;
}

// ---------------------------------------------------------------- TMA -------------------------------
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* m) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
__device__ __forceinline__ void tma_load_3d(void* smem_dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1, int c2) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
        ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
        : "memory");
}

// ---------------------------------------------------------------- TMEM ------------------------------
__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem, uint32_t cols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(cols));
}
__device__ __forceinline__ void tmem_relinquish() { asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::); }
__device__ __forceinline__ void tmem_dealloc(uint32_t addr, uint32_t cols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(addr), "r"(cols));
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// 32 lanes x 32 consecutive 32-bit columns: thread t of the warp gets row (lane base + t), cols c..c+31
__device__ __forceinline__ void tmem_ld_32x32(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
          "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
          "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr));
}

// 32 lanes x 16 consecutive 32-bit columns
__device__ __forceinline__ void tmem_ld_32x16(uint32_t taddr, uint32_t (&r)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr));
}

// ---------------------------------------------------------------- UMMA ------------------------------
// shared-memory matrix descriptor, K-major operand, 128-byte swizzle: rows of 128 B, 8-row swizzle
// atoms of 1024 B (SBO), tile base 1024-B aligned.
__device__ __forceinline__ uint64_t umma_desc_k_sw128(uint32_t smem_addr) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr & 0x3FFFF) >> 4);        // start address      bits [0,14)
    d |= (uint64_t)1 << 16;                              // leading byte offset (unused for swizzled K-major)
    d |= (uint64_t)(1024 >> 4) << 32;                    // stride byte offset  bits [32,46)
    d |= (uint64_t)1 << 46;                              // descriptor version (Blackwell)
    d |= (uint64_t)2 << 61;                              // layout type: SWIZZLE_128B
    return d;
}
// instruction descriptor for kind::f16 (fmt 0 = fp16, 1 = bf16) or kind::tf32 (fmt 2), fp32 accumulate,
// both operands K-major, dense
__host__ __device__ constexpr uint32_t umma_idesc(int M, int N, int fmt) {
    return (1u << 4) | ((uint32_t)fmt << 7) | ((uint32_t)fmt << 10) | ((uint32_t)(N >> 3) << 17) |
           ((uint32_t)(M >> 4) << 24);
}
__device__ __forceinline__ void umma_f16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}
// D = A*B + D * 2^-11 (tcgen05.mma's optional scale-input-d immediate): folds the 2^-11 of the 3-term split's correction
// accumulator into the tensor core when ALL correction products of a tile are issued before its main products, so main
// and correction terms share ONE TMEM accumulator (half the tcgen05.ld traffic and TMEM columns of a D0 | D1 pair).
__device__ __forceinline__ void umma_f16_scale_d11(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, 1, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p, 11;\n\t}"
        ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc)
        : "memory");
}
// arrives on the mbarrier once every previously issued tcgen05.mma of this thread has completed
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// A operand in tensor memory (lane = row, 16-bit elements packed two per 32-bit column: k = 2c in the low half), B from a
// shared-memory descriptor
__device__ __forceinline__ void umma_f16_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
        ::"r"(tmem_d), "r"(tmem_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void umma_f16_ts_scale_d11(uint32_t tmem_d, uint32_t tmem_a, uint64_t desc_b, uint32_t idesc) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, 1, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p, 11;\n\t}"
        ::"r"(tmem_d), "r"(tmem_a), "l"(desc_b), "r"(idesc)
        : "memory");
}
__device__ __forceinline__ void tmem_st_32x16(uint32_t taddr, const uint32_t (&r)[16]) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
        "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};"
        ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]),
          "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
        : "memory");
}

__device__ __forceinline__ void tmem_st_32x32(uint32_t taddr, const uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
        "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
        "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};"
        ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]),
          "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]),
          "r"(r[16]), "r"(r[17]), "r"(r[18]), "r"(r[19]), "r"(r[20]), "r"(r[21]), "r"(r[22]), "r"(r[23]),
          "r"(r[24]), "r"(r[25]), "r"(r[26]), "r"(r[27]), "r"(r[28]), "r"(r[29]), "r"(r[30]), "r"(r[31])
        : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// ---------------------------------------------------------------- CTA pairs (cta_group::2) ----------
// Two CTAs of a cluster (same TPC) execute ONE tcgen05.mma with M = 256: each CTA holds its 128 rows of A and of the
// accumulator (own TMEM) and HALF of the B tile; only the leader (cluster rank 0) issues the MMA and owns the "full"
// barriers, which both CTAs' TMA loads signal (barrier address with the peer bit cleared, as CUTLASS's
// SM100_TMA_2SM_LOAD does); completion is multicast to the same barrier offset in both CTAs.
constexpr uint32_t kPeerBitMask = 0xFEFFFFFFu;
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ int cluster_nctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_nctarank;" : "=r"(r));
    return (int)r;
}
// address of the same shared-memory object in CTA `rank` of the cluster
__device__ __forceinline__ uint32_t cluster_addr(const void* p, int rank) {
    uint32_t a;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(a) : "r"(smem_u32(p)), "r"(rank));
    return a;
}
__device__ __forceinline__ void tma_load_3d_2sm(void* smem_dst, const CUtensorMap* m, uint64_t* leader_bar, int c0, int c1, int c2) {
    asm volatile(
        "cp.async.bulk.tensor.3d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
        ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(leader_bar) & kPeerBitMask), "r"(c0), "r"(c1), "r"(c2)
        : "memory");
}
// the same load written to the same smem offset of every CTA in cta_mask; each destination pair's leader barrier gets the bytes
__device__ __forceinline__ void tma_load_3d_2sm_mc(void* smem_dst, const CUtensorMap* m, uint64_t* leader_bar, int c0, int c1, int c2,
                                                   uint16_t cta_mask) {
    asm volatile(
        "cp.async.bulk.tensor.3d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster [%0], [%1, {%4, %5, %6}], [%2], %3;"
        ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(leader_bar) & kPeerBitMask), "h"(cta_mask),
          "r"(c0), "r"(c1), "r"(c2)
        : "memory");
}
__device__ __forceinline__ void tmem_alloc_2sm(uint32_t* dst_smem, uint32_t cols) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(cols));
}
__device__ __forceinline__ void tmem_relinquish_2sm() { asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::); }
__device__ __forceinline__ void tmem_dealloc_2sm(uint32_t addr, uint32_t cols) {
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(addr), "r"(cols));
}
__device__ __forceinline__ void umma_f16_2sm(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}
// arrives on the barrier at this offset in BOTH CTAs of the pair once the previously issued MMAs have completed
__device__ __forceinline__ void umma_commit_2sm(uint64_t* bar, uint16_t cta_mask = 3) {
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                 ::"r"(smem_u32(bar)), "h"(cta_mask) : "memory");
}
// arrive on the barrier at the same offset in CTA `rank` of the cluster
__device__ __forceinline__ void mbar_arrive_cluster(uint64_t* bar, uint32_t rank) {
    uint32_t remote;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(remote) : "r"(smem_u32(bar)), "r"(rank));
    asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(remote) : "memory");
}

}  // namespace tc

// ---------------------------------------------------------------- host: tensor maps ------------------
// cuTensorMapEncodeTiled is fetched through the runtime's driver entry point so the library does not
// link libcuda (it must load on CPU-only hosts for the symbol checks).
typedef CUresult (*vcr_tmap_encode_fn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                       const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                       CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
vcr_tmap_encode_fn vcr_get_tmap_encoder();

// 3-D map over an operand buffer of 16-bit elements laid out [planes][rows][ld] (row-major, K contiguous):
// box = 64 elements (128 B) x box_rows x 1, 128-B swizzle, zero fill out of bounds.
int vcr_make_operand_tmap(CUtensorMap* out, const void* base, int cols, long long rows, int ld_elems,
                          long long plane_stride_elems, int planes, int box_rows);
