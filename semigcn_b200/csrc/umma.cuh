// tcgen05 / TMEM / mbarrier / bulk-copy / TMA PTX wrappers of the fp16-split tensor-core GEMM (gemm_f16.cu; sm_100a only).
#pragma once
#include "common.cuh"
#include <cuda.h>

namespace sgb {

// ------------------------------------------------------------------------------------------
// PTX helpers
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "WAIT_LOOP:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE;\n\t"
        "bra WAIT_LOOP;\n\t"
        "DONE:\n\t"
        "}" ::"r"(smem_u32(bar)), "r"(parity)
        : "memory");
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ void bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst_smem)),
                 "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

__device__ __forceinline__ void tmem_alloc(uint32_t* slot_smem, uint32_t cols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(slot_smem)), "r"(cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t addr, uint32_t cols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(addr), "r"(cols) : "memory");
}

__device__ __forceinline__ void umma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// 32 lanes x 32 columns of 32-bit: thread (lane) receives 32 consecutive columns of its row
__device__ __forceinline__ void tmem_ld_32x32(uint32_t taddr, float* v) {
    uint32_t r[32];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
          "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]),
          "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]),
          "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr)
        : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}

// shared-memory matrix descriptor, no swizzle (cute::UMMA::SmemDescriptor: start>>4 [0,14), LBO>>4 [16,30),
// SBO>>4 [32,46), version=1 [46,48), layout_type=0 [61,64))
__device__ __forceinline__ uint64_t make_desc(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes, uint32_t layout_type = 0) {
    uint64_t d = (uint64_t)(layout_type & 7) << 61;
    d |= (uint64_t)((smem_addr >> 4) & 0x3FFF);
    d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
    d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
    d |= (uint64_t)1 << 46;
    return d;
}

// instruction descriptor (cute::UMMA::InstrDescriptor) of kind::f16 with fp16 operands and fp32 accumulate: c_format F32 = 1 @4,
// a/b_format F16 = 0 @7/@10, a_major @15, b_major @16 (0 = K-major, 1 = MN-major), n>>3 @17, m>>4 @24
__host__ __device__ constexpr uint32_t make_idesc_f16(int m, int n, int a_mn_major, int b_mn_major) {
    return (1u << 4) | ((uint32_t)a_mn_major << 15) | ((uint32_t)b_mn_major << 16) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}

__device__ __forceinline__ void umma_f16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
        "}" ::"r"(d_tmem),
        "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
}

// ---- CTA pairs (cta_group::2): two CTAs of one cluster (the two SMs of a TPC) execute ONE MMA of M = 256 -------------------
// Each CTA holds its 128 rows of the A operand and HALF of the B operand (N / 2 rows) in its own shared memory; the tensor
// cores exchange the B halves, so per CTA the operand traffic of an M = 256, N = 256 MMA is that of a 128 x 128 one.  The even
// CTA (cluster rank 0) issues the MMAs and owns the barriers the pair synchronises on.
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// arrive on the barrier at the same shared-memory offset in CTA `rank` of the cluster (rank may be the caller's own).
// Default semantics (release at CTA scope): a cluster-scope release compiles to MEMBAR.ALL.GPU per arrive (measured: 29 % of all
// stall samples of the pair kernel).  What the arrive publishes here is shared memory of the ARRIVING CTA that only this SM's
// tensor core reads (made visible to the async proxy by fence.proxy.async before the arrive) or TMEM reads that have retired.
__device__ __forceinline__ void mbar_arrive_cluster(uint64_t* bar, uint32_t rank) {
    asm volatile(
        "{\n\t"
        ".reg .b32 ra;\n\t"
        "mapa.shared::cluster.u32 ra, %0, %1;\n\t"
        "mbarrier.arrive.shared::cluster.b64 _, [ra];\n\t"
        "}" ::"r"(smem_u32(bar)), "r"(rank)
        : "memory");
}
__device__ __forceinline__ void mbar_wait_cluster(uint64_t* bar, uint32_t parity) {      // acquire at cluster scope
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "WAIT_LOOP_C:\n\t"
        "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE_C;\n\t"
        "bra WAIT_LOOP_C;\n\t"
        "DONE_C:\n\t"
        "}" ::"r"(smem_u32(bar)), "r"(parity)
        : "memory");
}
__device__ __forceinline__ void tmem_alloc_pair(uint32_t* slot_smem, uint32_t cols) {    // one warp in EACH CTA of the pair
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(slot_smem)), "r"(cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_pair(uint32_t addr, uint32_t cols) {
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(addr), "r"(cols) : "memory");
}
__device__ __forceinline__ void umma_f16_pair(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t"
        "}" ::"r"(d_tmem),
        "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// completion of all MMAs issued so far by this thread -> one arrive on the barrier at this offset in BOTH CTAs of the pair
__device__ __forceinline__ void umma_commit_pair(uint64_t* bar) {
    const uint16_t mask = 3;
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(smem_u32(bar)), "h"(mask)
                 : "memory");
}

// ---- TMA (cp.async.bulk.tensor): 2-D tiled loads of row-major fp32 matrices --------------------------------
// box = {box_cols, box_rows} elements starting at (col, row); out-of-range elements are written as zeros and the
// mbarrier always receives the full box byte count.
__device__ __forceinline__ void tma_load_2d(void* dst_smem, const CUtensorMap* tmap, int col, int row, uint64_t* bar) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(
                     smem_u32(dst_smem)),
                 "l"(reinterpret_cast<uint64_t>(tmap)), "r"(col), "r"(row), "r"(smem_u32(bar))
                 : "memory");
}
// L2 eviction priorities: the weight-gradient kernels stream G and A once (evict_first) while re-reading and re-writing a running
// partial tile per CTA once per segment (evict_last) -- without the hints the stream pushes the partials out to DRAM
// (measured: 0.47 GB of extra traffic on a 2.05 GB launch).
__device__ __forceinline__ uint64_t l2_policy_evict_first() {
    uint64_t p;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
    return p;
}
__device__ __forceinline__ uint64_t l2_policy_evict_last() {
    uint64_t p;
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));
    return p;
}
__device__ __forceinline__ void tma_load_2d_hint(void* dst_smem, const CUtensorMap* tmap, int col, int row, uint64_t* bar, uint64_t policy) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1, {%2, %3}], [%4], %5;" ::"r"(
                     smem_u32(dst_smem)),
                 "l"(reinterpret_cast<uint64_t>(tmap)), "r"(col), "r"(row), "r"(smem_u32(bar)), "l"(policy)
                 : "memory");
}
__device__ __forceinline__ float4 ldcg_hint(const float4* p, uint64_t policy) {
    float4 v;
    asm volatile("ld.global.cg.L2::cache_hint.v4.f32 {%0, %1, %2, %3}, [%4], %5;" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p), "l"(policy) : "memory");
    return v;
}
__device__ __forceinline__ void stcg_hint(float4* p, float4 v, uint64_t policy) {
    asm volatile("st.global.cg.L2::cache_hint.v4.f32 [%0], {%1, %2, %3, %4}, %5;" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w), "l"(policy) : "memory");
}
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* tmap) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(tmap)) : "memory");
}

// host: tensor map of a row-major [rows, cols] fp32 matrix with leading dimension ld (elements); swizzle128 = the
// 128-byte swizzle (16-byte chunk index XOR row % 8; box_cols * 4 must be 128), else a dense box image.
int make_tmap_2d(CUtensorMap* out, const float* base, int64_t rows, int64_t cols, int64_t ld, int box_cols, int box_rows, bool swizzle128);

}  // namespace sgb
