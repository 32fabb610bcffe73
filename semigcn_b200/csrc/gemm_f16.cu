// tcgen05 tiles for the dense feature transform with a 2 x FP16 operand split (engine 3).
//
// Each fp32 operand is scaled by a per-tensor power of two s (exact) so that max |x s| lies in
// [2^14, 2^15), then split   x s = hi + lo,  hi = rn_f16(x s),  lo = rn_f16(x s - hi)   (22 significant
// bits), and the product is evaluated as   A*B ~= (A_lo*B_hi + A_hi*B_lo + A_hi*B_hi) / (s_A s_B)
// with fp32 accumulation in TMEM.  kind::f16 runs at twice the tf32 rate and every operand byte
// (shared memory, L2 -> SM weight traffic) is half of a tf32 one: at these rates both kernels are bound
// by the HBM stream of the activation operand, which is what the feature transform algorithmically has to read.
// Accuracy contract: max |C - C_exact| <= ~4e-7 * sum_k |A||B| (norm-relative, like fp32 SIMT);
// elements more than ~2^-23 below their tensor's maximum lose relative (not absolute) precision,
// since fp16 has 5 exponent bits -- see DESIGN.md "engine 3".
//
// k_gemm_f16    C[M,N] (+)= A[M,K] * Wp^T + bias      (forward transform and dX)
//   persistent, one CTA per SM; 8 producer warps (global -> scale/split -> K-major no-swizzle smem,
//   conflict-free 16-byte stores), 1 lane bulk-copies the pre-split weight image (cp.async.bulk +
//   mbarrier complete_tx), 1 lane issues tcgen05.mma.kind::f16 128 x N x 16, 4 epilogue warps
//   (tcgen05.ld -> unscale -> bias / accumulate -> global); double-buffered TMEM accumulators.
// k_gemm_tn_f16 D[N,K] = G[M,N]^T A[M,K]                 (weight gradient, reduction over vertices)
//   both operands K-major with "K" = vertex: a producer thread loads 8 vertices x 4 columns
//   (8 float4), which is exactly four 16-byte core-matrix rows after conversion -- the transposition
//   happens in registers.  Split over vertices across CTAs, 512-vertex TMEM segments drained with
//   round-to-nearest adds, fixed-order reduction of the per-CTA partial tiles (deterministic).
#include "common.cuh"
#include "umma.cuh"
#include <cuda_fp16.h>
#include <stdlib.h>

namespace sgb {

// ------------------------------------------------------------------------------------------
// per-tensor power-of-two scale from max |x|
// ------------------------------------------------------------------------------------------
// s = 2^(14 - floor(log2 amax)) -> amax * s in [2^14, 2^15); amax == 0 / non-finite -> 1 (every max |x| handed to the
// engine is taken over the finite entries, so an inf or NaN operand entry does not reach here)
__host__ __device__ __forceinline__ void f16_scale_from_amax(float amax, float& s, float& inv) {
    uint32_t bits;
#ifdef __CUDA_ARCH__
    bits = __float_as_uint(amax);
#else
    union { float f; uint32_t u; } cv; cv.f = amax; bits = cv.u;
#endif
    const int e = (int)((bits >> 23) & 0xff);
    int se = 127 + 14 - (e - 127);
    if (e == 0 || e == 255) se = 127;
    if (se < 2) se = 2;
    if (se > 252) se = 252;
#ifdef __CUDA_ARCH__
    s = __uint_as_float((uint32_t)se << 23);
    inv = __uint_as_float((uint32_t)(254 - se) << 23);
#else
    cv.u = (uint32_t)se << 23; s = cv.f;
    cv.u = (uint32_t)(254 - se) << 23; inv = cv.f;
#endif
}

// max |x| over the finite entries of an [m, c] matrix (finite_abs) -> atomicMax on the float bits (non-negative floats order
// like uints).  The slot must be zero before the launch.
__global__ void __launch_bounds__(256) k_amax(const float* __restrict__ x, int64_t ldx, int64_t m, int c, uint32_t* __restrict__ slot) {
    const int cv = c >> 2;
    const int64_t total = m * cv;
    float mx = 0.f;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = i / cv;
        const int ch = (int)(i % cv) * 4;
        const float4 v = ldg4(x + r * ldx + ch);
        mx = fmaxf(mx, fmaxf(fmaxf(finite_abs(v.x), finite_abs(v.y)), fmaxf(finite_abs(v.z), finite_abs(v.w))));
    }
    uint32_t b = __float_as_uint(mx);
    b = __reduce_max_sync(0xffffffffu, b);
    __shared__ uint32_t sm[8];
    if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = b;
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < 8; ++w) b = max(b, sm[w]);
        if (b) atomicMax(slot, b);
    }
}

int amax_launch(const float* x, int64_t ldx, int64_t m, int c, uint32_t* slot, cudaStream_t stream) {
    SGB_CUDA(cudaMemsetAsync(slot, 0, sizeof(uint32_t), stream));
    const int64_t total = m * (c / 4);
    const int grid = (int)min64(ceil_div(total > 0 ? total : 1, 256 * 8), (int64_t)num_sms() * 8);
    k_amax<<<grid, 256, 0, stream>>>(x, ldx, m, c, slot);
    SGB_CHECK_LAUNCH("k_amax");
    return SGB_OK;
}

__device__ __forceinline__ void split_f16x2(float x0, float x1, uint32_t& hi, uint32_t& lo) {
    const __half2 h = __floats2half2_rn(x0, x1);
    const float2 f = __half22float2(h);
    const __half2 l = __floats2half2_rn(x0 - f.x, x1 - f.y);
    hi = *reinterpret_cast<const uint32_t*>(&h);
    lo = *reinterpret_cast<const uint32_t*>(&l);
}

// ------------------------------------------------------------------------------------------
// forward / dX kernel geometry
// ------------------------------------------------------------------------------------------
constexpr int kHBM = 128;                       // rows per tile == UMMA M
constexpr int kHBK = 32;                        // K elements per pipeline stage (2 MMA k-slices of 16)
constexpr int kHCols = kHBK / 8;                // 16-byte core-matrix columns per stage
constexpr int kHALbo = 128;                     // bytes between K-adjacent core matrices of A (dense; a quarter-warp of converters fills one whole core matrix)
constexpr int kHASbo = kHCols * kHALbo;         // bytes between M-adjacent core matrices of A
constexpr int kHATile = (kHBM / 8) * kHASbo;    // per hi (or lo)
constexpr int kHBLbo = 128;
constexpr int kHBSbo = kHCols * kHBLbo;
constexpr int kHConvWarps = 4;                  // warps 0..3: converters, raw fp32 (TMA) -> scaled hi/lo fp16 operand tiles
constexpr int kHEpiWarps = 8;                   // warps 4..11: epilogue; TMEM lane quarter = warp % 4, two warps per quarter (even / odd 32-column chunks)
constexpr int kHWarpB = kHConvWarps + kHEpiWarps;      // B copy
constexpr int kHWarpMma = kHWarpB + 1;                 // MMA issuer, TMEM owner
constexpr int kHWarpLoad = kHWarpB + 2;                // A TMA loader
constexpr int kHThreads = (kHWarpLoad + 1) * 32;       // 480
constexpr int kHRawBytes = kHBM * kHBK * 4;     // one raw A stage: 128 rows x 32 fp32, 128-byte rows, TMA 128B swizzle
constexpr int kHMaxRawStages = 6;               // raw fp32 A stages in flight (runtime: HArgs::raw_stages)
constexpr int kHBarBytes = 512;                 // forward kernel: barrier block between the operand ring and the epilogue staging
constexpr int kHMaxStages = 6;
constexpr int kHEpiLd = 36;                     // weight-gradient kernel: floats per row of a drain warp's 32 x 32 staging tile (+4: conflict-free)
constexpr int kHEpiBytes = kHEpiWarps * 32 * 32 * 4;  // forward kernel: dense 32 x 32 tiles, 16-byte chunks XOR-swizzled by the row (conflict-free both ways)
constexpr int kTEpiBytes = 4 * 32 * kHEpiLd * 4;      // the weight-gradient kernel has four drain warps
static const int kHSmemBudget = 227 * 1024;

__host__ __device__ constexpr int h_b_tile_bytes(int bn) { return (bn / 8) * kHBSbo; }
__host__ __device__ constexpr int h_stage_bytes(int bn) { return (2 * kHATile + 2 * h_b_tile_bytes(bn) + 1023) / 1024 * 1024; }
// CTA pairs (cta_group::2): each CTA stages its own 128 rows of A and HALF of the weight tile (bn / 2 rows of B, hi and lo)
__host__ __device__ constexpr int h_stage_bytes_pair(int bn) { return (2 * kHATile + h_b_tile_bytes(bn) + 1023) / 1024 * 1024; }

struct HArgs {
    CUtensorMap a_map;                // A as a [m, k] fp32 tensor, box {32, 128}, 128-byte swizzle
    const float* a; int64_t lda;
    const uint8_t* wp;                // prepped weights: [n_tiles][k_chunks][hi|lo][tile image]
    const float* wscale;              // [0] = s_W, [1] = 1 / s_W   (written by k_prep_weights_f16)
    const float* a_amax;              // device scalar: max |A|
    float* c; int64_t ldc;
    int64_t m; int n; int k;
    int bn; int n_tiles; int k_chunks; int stages; int raw_stages;
    const float* bias; int accumulate;
    float* stat_partials;             // optional BatchNorm partials of C: [4 * gridDim.x / n_tiles][3][n] (count, mean, M2), one row per epilogue warp
    uint32_t tmem_cols; int acc_stride;
};

// weights -> scale, hi/lo fp16 split, zero padded, in the exact per-stage shared-memory image.
// Small grid; every CTA first reduces max |W| (finite entries) itself (W is at most 1 MB and L2-resident), so one launch
// does amax + prep and the scale never round-trips through the host.
__global__ void __launch_bounds__(256) k_prep_weights_f16(const float* __restrict__ w, int64_t ldw, int transb, int n, int k, int bn,
                                                          int n_tiles, int k_chunks, __half* __restrict__ wp, float* __restrict__ wscale) {
    __shared__ float sm[8];
    const int rows = transb ? n : k, cols = transb ? k : n;
    float mx = 0.f;
    if (ldw == cols && (reinterpret_cast<uintptr_t>(w) & 15) == 0 && ((rows * cols) & 3) == 0) {       // dense, aligned: flat 128-bit scan
        for (int i = threadIdx.x; i < (rows * cols) >> 2; i += blockDim.x) {
            const float4 v = ldg4(w + 4 * i);
            mx = fmaxf(mx, fmaxf(fmaxf(finite_abs(v.x), finite_abs(v.y)), fmaxf(finite_abs(v.z), finite_abs(v.w))));
        }
    } else {
        for (int r = 0; r < rows; ++r)
            for (int i = threadIdx.x; i < cols; i += blockDim.x) mx = fmaxf(mx, finite_abs(w[(int64_t)r * ldw + i]));
    }
    mx = __uint_as_float(__reduce_max_sync(0xffffffffu, __float_as_uint(mx)));
    if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = mx;
    __syncthreads();
    mx = sm[0];
    for (int i = 1; i < 8; ++i) mx = fmaxf(mx, sm[i]);
    float s, inv;
    f16_scale_from_amax(mx, s, inv);
    if (blockIdx.x == 0 && threadIdx.x == 0) { wscale[0] = s; wscale[1] = inv; }
    const int tile_halves = h_b_tile_bytes(bn) / 2;
    const int64_t total = (int64_t)n_tiles * k_chunks * tile_halves;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int h = (int)(i % tile_halves);
        const int64_t blk = i / tile_halves;
        const int q = (int)(blk % k_chunks), t = (int)(blk / k_chunks);
        const int core_n = h / (kHBSbo / 2);
        const int rem = h % (kHBSbo / 2);
        const int core_k = rem / 64, in_core = rem % 64;
        const int nl = core_n * 8 + in_core / 8, kl = core_k * 8 + in_core % 8;
        const int gn = t * bn + nl, gk = q * kHBK + kl;
        float v = 0.f;
        if (gn < n && gk < k) v = transb ? w[(int64_t)gn * ldw + gk] : w[(int64_t)gk * ldw + gn];
        v *= s;
        const __half hi = __float2half_rn(v);
        const __half lo = __float2half_rn(v - __half2float(hi));
        __half* base = wp + (blk * 2) * tile_halves;
        base[h] = hi;
        base[tile_halves + h] = lo;
    }
}

// One 32-column chunk of an epilogue warp's 32-row block: TMEM -> registers -> unscale -> transpose through the warp's
// staging tile -> (+C) + bias -> coalesced 128-byte row-segment stores, and (optionally) the chunk's column moments.
// FULL: all 32 rows of the block and all 32 columns of the chunk are inside C (no per-row / per-column predicates).
template <bool FULL>
__device__ __forceinline__ void h_epi_chunk(const HArgs& g, uint32_t taddr, float* __restrict__ stg, float* __restrict__ cp /* row grp, column cc of the chunk */,
                                            const float* __restrict__ bias_p, int lane, int grp, int cc, int nvalid, bool col_ok, float sc1, float sc2,
                                            bool stats, float inv_nb, float (&blk_mean)[4], float (&blk_m2)[4]) {
    float4 b = make_float4(0.f, 0.f, 0.f, 0.f);
    if (bias_p && (FULL || col_ok)) b = ldg4(bias_p);      // issued first: its latency hides behind the TMEM load
    float v[32];
    tmem_ld_32x32(taddr, v);                 // warp-collective: lane = row, registers = 32 consecutive columns
    if (sc2 == 1.f) {                        // 1 / (s_A s_W) is one exact power-of-two factor in all but extreme-range cases
#pragma unroll
        for (int e = 0; e < 32; e += 4)      // row `lane`, 16-byte chunk e / 4 stored at chunk position (e / 4) ^ (lane % 8)
            *reinterpret_cast<float4*>(stg + lane * 32 + (((e >> 2) ^ (lane & 7)) << 2)) = make_float4(v[e] * sc1, v[e + 1] * sc1, v[e + 2] * sc1, v[e + 3] * sc1);
    } else {
#pragma unroll
        for (int e = 0; e < 32; e += 4)
            *reinterpret_cast<float4*>(stg + lane * 32 + (((e >> 2) ^ (lane & 7)) << 2)) =
                make_float4((v[e] * sc1) * sc2, (v[e + 1] * sc1) * sc2, (v[e + 2] * sc1) * sc2, (v[e + 3] * sc1) * sc2);
    }
    __syncwarp();
    // read back transposed: lane -> rows grp, grp + 4, ..., 16 bytes at column cc: a store instruction then writes four whole
    // 128-byte row segments (a lane-per-row store touches 32 different lines per instruction and saturates the L1 data pipe)
    const int64_t ld4 = 4 * g.ldc;
    float4 o[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const bool on = FULL || (col_ok && i * 4 + grp < nvalid);
        o[i] = on ? *reinterpret_cast<const float4*>(stg + (i * 4 + grp) * 32 + ((((lane & 7) ^ ((i * 4 + grp) & 7))) << 2)) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
    if (g.accumulate) {                      // all eight loads in flight before the first add
        float4 old[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const bool on = FULL || (col_ok && i * 4 + grp < nvalid);
            old[i] = on ? *reinterpret_cast<const float4*>(cp + i * ld4) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
#pragma unroll
        for (int i = 0; i < 8; ++i) { o[i].x += old[i].x; o[i].y += old[i].y; o[i].z += old[i].z; o[i].w += old[i].w; }
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const bool on = FULL || (col_ok && i * 4 + grp < nvalid);
        if (on) {
            o[i].x += b.x; o[i].y += b.y; o[i].z += b.z; o[i].w += b.w;
            *reinterpret_cast<float4*>(cp + i * ld4) = o[i];
        }
    }
    if (stats) {
        // block mean, then centred second moment (two passes over registers: no cancellation), each reduced over the four
        // row groups with two butterfly steps (lanes l, l^8, l^16, l^24 hold the same columns); rows / columns outside C are zeros
        float sm[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int i = 0; i < 8; ++i) { sm[0] += o[i].x; sm[1] += o[i].y; sm[2] += o[i].z; sm[3] += o[i].w; }
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            sm[q] += __shfl_xor_sync(0xffffffffu, sm[q], 8);
            sm[q] += __shfl_xor_sync(0xffffffffu, sm[q], 16);
            sm[q] *= inv_nb;
        }
        float d2[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            if (FULL || i * 4 + grp < nvalid) {
                const float dx = o[i].x - sm[0], dy = o[i].y - sm[1], dz = o[i].z - sm[2], dw = o[i].w - sm[3];
                d2[0] = fmaf(dx, dx, d2[0]); d2[1] = fmaf(dy, dy, d2[1]); d2[2] = fmaf(dz, dz, d2[2]); d2[3] = fmaf(dw, dw, d2[3]);
            }
        }
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            d2[q] += __shfl_xor_sync(0xffffffffu, d2[q], 8);
            d2[q] += __shfl_xor_sync(0xffffffffu, d2[q], 16);
            blk_mean[q] = sm[q];
            blk_m2[q] = d2[q];
        }
    }
    __syncwarp();                            // the staging tile is free for the next chunk
}

// PAIR: the kernel runs as clusters of two CTAs (launch attribute) on UMMA M = 256: CTA r of a pair owns the m-tile 2 u + r of its
// unit's tile pair u and the B rows [r ncols / 2, + ncols / 2) of the n-tile; the tensor cores exchange the B halves, so a stage
// costs each SM 16 KB less weight copy and 24 KB less operand reads (the kernel is bound by the shared-memory data pipe).  The
// leader (cluster rank 0) issues the MMAs and owns full[] / tempty[]; commits arrive on empty[] / tfull[] of both CTAs.
template <bool PAIR>
__global__ void __launch_bounds__(kHThreads, 1) k_gemm_f16(const __grid_constant__ HArgs g) {
    extern __shared__ __align__(1024) uint8_t smem[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t rank = PAIR ? cluster_ctarank() : 0u;
    const int stage_bytes = PAIR ? h_stage_bytes_pair(g.bn) : h_stage_bytes(g.bn);
    const int b_tile_bytes = h_b_tile_bytes(g.bn);                       // one full hi (or lo) weight tile of the global image
    const int b_smem_bytes = PAIR ? b_tile_bytes / 2 : b_tile_bytes;     // what this CTA stages of it
    const uint32_t stages = (uint32_t)g.stages;
    // smem: [raw ring: raw_stages x 16 KB][operand ring: stages x stage_bytes][barriers 512 B][epilogue staging: 8 x 4 KB]
    uint8_t* const raw_base = smem;
    const uint32_t raw_stages = (uint32_t)g.raw_stages;
    uint8_t* const op_base = smem + raw_stages * kHRawBytes;
    uint64_t* full = reinterpret_cast<uint64_t*>(op_base + (size_t)g.stages * stage_bytes);
    uint64_t* empty = full + kHMaxStages;
    uint64_t* tfull = empty + kHMaxStages;
    uint64_t* tempty = tfull + 2;
    uint64_t* rfull = tempty + 2;               // raw stage landed (TMA complete_tx)
    uint64_t* rempty = rfull + kHMaxRawStages;  // raw stage consumed by all converter threads
    uint64_t* bfull = rempty + kHMaxRawStages;  // PAIR: this CTA's half of the weight tile landed (bulk copy complete_tx)
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bfull + kHMaxStages);

    if (threadIdx.x == 0) {
        for (int s = 0; s < g.stages; ++s) {
            // single CTA: one converter group (64 threads) + the B copy's expect_tx arrive;  PAIR: one elected lane per warp of the
            // stage's converter group, in both CTAs (each arrives once its CTA's A tile is converted AND its B half has landed)
            mbar_init(&full[s], PAIR ? 2 * (kHConvWarps / 2) : kHConvWarps * 32 / 2 + 1);
            mbar_init(&empty[s], 1);
            mbar_init(&bfull[s], 1);
        }
        for (int b = 0; b < 2; ++b) {
            mbar_init(&tfull[b], 1);
            mbar_init(&tempty[b], PAIR ? 2 * kHEpiWarps : kHEpiWarps);
        }
        for (uint32_t s = 0; s < raw_stages; ++s) {
            mbar_init(&rfull[s], 1);
            mbar_init(&rempty[s], kHConvWarps * 32 / 2);
        }
        fence_barrier_init();
    }
    if (PAIR) {
        __syncthreads();
        cluster_sync_all();                     // both CTAs' barriers exist before anyone arrives remotely
        if (warp == kHWarpMma) tmem_alloc_pair(tmem_slot, g.tmem_cols);
    } else {
        if (warp == kHWarpMma) tmem_alloc(tmem_slot, g.tmem_cols);
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    // A unit (a CTA, or a CTA pair) works on the tiles unit, + units, ... of the (m-tile or m-tile pair) x n-tile grid; the number
    // of units is a multiple of n_tiles, so the n-tile of a unit never changes.  m0_of(tile): first row of THIS CTA's m-tile.
    // All ring positions / phases below are carried incrementally (no per-iteration division by a runtime stage count).
    const uint32_t unit = PAIR ? blockIdx.x >> 1 : blockIdx.x, units = PAIR ? gridDim.x >> 1 : gridDim.x;
    const int64_t m_tiles = (g.m + kHBM - 1) / kHBM;
    const int64_t total_tiles = (PAIR ? (m_tiles + 1) / 2 : m_tiles) * g.n_tiles;
    const uint32_t my_tiles = total_tiles > unit ? (uint32_t)((total_tiles - 1 - unit) / units + 1) : 0u;
    const uint32_t k_chunks = (uint32_t)g.k_chunks;
    const int nt = (int)(unit % (uint32_t)g.n_tiles);
#define SGB_H_M0_OF(tile) ((PAIR ? ((tile) / g.n_tiles) * 2 + (int64_t)rank : (tile) / g.n_tiles) * kHBM)

    if (warp < kHConvWarps) {
        // ================= A converters: raw fp32 stage (TMA) -> regs (scale, hi/lo fp16) -> operand stage =================
        // Two groups of two warps, group g takes the stages g, g + 2, g + 4, ...: a group's chain for one stage (wait for the TMA
        // -> shared-memory loads -> convert -> fence -> wait for the operand slot -> stores -> fence -> arrive) is long and strictly
        // serial; with ONE group it was the period of the whole pipeline (measured: every shape ran ~0.4 us per stage above its
        // HBM time).  Two groups overlap stage i + 1's loads / conversion with stage i's stores / fences.
        float sa, inva;
        f16_scale_from_amax(__ldg(g.a_amax), sa, inva);
        constexpr int GROUPS = 2, GTHREADS = kHConvWarps * 32 / GROUPS;        // 64 threads per group
        const int grp = warp / (kHConvWarps / GROUPS);                          // 0: warps 0-1, 1: warps 2-3
        const int gt = threadIdx.x - grp * GTHREADS;                            // 0..63 inside the group
        // stage = 128 rows x kHCols core columns (8 K elements = 32 bytes of the raw row).  A quarter-warp (the unit a 16-byte
        // shared-memory access is processed in) takes the 8 rows of ONE core matrix at one core column: its reads hit 8
        // distinct swizzled chunks of the raw rows, its writes fill one dense 128-byte core matrix -- conflict-free both ways
        // without padding the operand tile.  Thread: core column cq, rows r0 + 16 i (8 row slots, converted four at a time).
        const int cq = (gt >> 3) & (kHCols - 1), r0 = (gt & 7) + 8 * (gt >> 5);      // r0 in 0..15
        static_assert(kHCols == 4, "converter thread mapping assumes 4 core columns per stage");
        constexpr int RPT = kHBM * kHCols / GTHREADS;                           // row slots per thread (8)
        constexpr int RSTEP = GTHREADS / kHCols;                                // 16
        constexpr int HALF = RPT / 2;
        const uint32_t total_it = my_tiles * k_chunks;
        uint32_t s = (uint32_t)grp % stages, ph = ((uint32_t)grp / stages) & 1u;
        uint32_t rs = (uint32_t)grp % raw_stages, rph = ((uint32_t)grp / raw_stages) & 1u;
        for (uint32_t it = (uint32_t)grp; it < total_it; it += GROUPS) {
            // The previous user of this raw slot (stage it - raw_stages) is the OTHER group when the ring length is odd, and
            // TMA completions are not ordered: without this wait a group that runs ahead could test rfull[rs] while the slot's
            // previous phase has not even completed -- the parity test would alias (phase p - 1 incomplete looks like phase p
            // complete) and the group would convert stale data and release the slot twice.  rempty[rs] completes only after the
            // previous user has seen its data, and its next phase cannot complete without this group: no aliasing here.
            mbar_wait(&rempty[rs], rph ^ 1);
            mbar_wait(&rfull[rs], rph);
            const uint8_t* raw = raw_base + (size_t)rs * kHRawBytes;
            uint4 h[RPT], l[RPT];
#pragma unroll
            for (int hf = 0; hf < 2; ++hf) {
                float4 v[HALF][2];
#pragma unroll
                for (int i = 0; i < HALF; ++i) {
                    const int r = r0 + RSTEP * (hf * HALF + i);
                    // 128-byte swizzle: 16-byte chunk j of row r sits at chunk position j ^ (r % 8)
                    v[i][0] = *reinterpret_cast<const float4*>(raw + r * 128 + (((2 * cq) ^ (r & 7)) << 4));
                    v[i][1] = *reinterpret_cast<const float4*>(raw + r * 128 + (((2 * cq + 1) ^ (r & 7)) << 4));
                }
#pragma unroll
                for (int i = 0; i < HALF; ++i) {
                    const int k = hf * HALF + i;
                    split_f16x2(v[i][0].x * sa, v[i][0].y * sa, h[k].x, l[k].x);
                    split_f16x2(v[i][0].z * sa, v[i][0].w * sa, h[k].y, l[k].y);
                    split_f16x2(v[i][1].x * sa, v[i][1].y * sa, h[k].z, l[k].z);
                    split_f16x2(v[i][1].z * sa, v[i][1].w * sa, h[k].w, l[k].w);
                }
            }
            // converted first: the shared-memory reads must have returned before the raw slot is handed back to the TMA
            // engine (an arrive issued right behind the loads can overtake them in the memory pipeline)
            fence_proxy_async();
            mbar_arrive(&rempty[rs]);
            mbar_wait(&empty[s], ph ^ 1);
            uint8_t* a_hi = op_base + (size_t)s * stage_bytes;
            uint8_t* a_lo = a_hi + kHATile;
#pragma unroll
            for (int i = 0; i < RPT; ++i) {
                const int r = r0 + RSTEP * i;
                const uint32_t off = (uint32_t)(r >> 3) * kHASbo + (uint32_t)cq * kHALbo + (uint32_t)(r & 7) * 16;
                *reinterpret_cast<uint4*>(a_hi + off) = h[i];
                *reinterpret_cast<uint4*>(a_lo + off) = l[i];
            }
            fence_proxy_async();          // generic-proxy smem writes -> visible to the tensor core (async proxy)
            if (PAIR) {
                __syncwarp();
                if (lane == 0) {
                    mbar_wait(&bfull[s], ph);                 // this CTA's B half is in place as well (bfull[s] cannot run ahead: its next copy needs empty[s])
                    mbar_arrive_cluster(&full[s], 0);
                }
            } else {
                mbar_arrive(&full[s]);
            }
            s += GROUPS;
            if (s >= stages) { s -= stages; ph ^= 1; }
            rs += GROUPS;
            if (rs >= raw_stages) { rs -= raw_stages; rph ^= 1; }
        }
    } else if (warp == kHWarpLoad) {
        // ================= A loader: one lane streams the raw A tiles (TMA 2-D, 128B swizzle, zero fill past m / k) =================
        if (lane == 0) {
            tma_prefetch_desc(&g.a_map);
            uint32_t rs = 0, rph = 0;
            int64_t tile = unit;
            for (uint32_t t = 0; t < my_tiles; ++t, tile += units) {
                const int m0 = (int)SGB_H_M0_OF(tile);
                for (uint32_t q = 0; q < k_chunks; ++q) {
                    mbar_wait(&rempty[rs], rph ^ 1);
                    mbar_arrive_expect_tx(&rfull[rs], kHRawBytes);
                    tma_load_2d(raw_base + (size_t)rs * kHRawBytes, &g.a_map, (int)(q * kHBK), m0, &rfull[rs]);
                    if (++rs == raw_stages) { rs = 0; rph ^= 1; }
                }
            }
        }
    } else if (warp == kHWarpB) {
        // ================= B copy: one bulk copy of the pre-tiled hi|lo weight image per stage =================
        if (lane == 0) {
            const uint8_t* src0 = g.wp + (size_t)nt * g.k_chunks * 2 * b_tile_bytes;
            // PAIR: rows [rank ncols / 2, + ncols / 2) of the hi and of the lo tile (whole 8-row core-matrix rows, contiguous in the image)
            const int ncols = min(g.bn, g.n - nt * g.bn);
            const uint32_t half_bytes = (uint32_t)(ncols / 16) * kHBSbo;
            const uint8_t* src_half = src0 + (size_t)rank * half_bytes;
            uint32_t s = 0, ph = 0;
            for (uint32_t t = 0; t < my_tiles; ++t) {
                for (uint32_t q = 0; q < k_chunks; ++q) {
                    mbar_wait(&empty[s], ph ^ 1);
                    uint8_t* b_dst = op_base + (size_t)s * stage_bytes + 2 * kHATile;
                    if (PAIR) {
                        mbar_arrive_expect_tx(&bfull[s], 2 * half_bytes);
                        bulk_g2s(b_dst, src_half + (size_t)q * 2 * b_tile_bytes, half_bytes, &bfull[s]);
                        bulk_g2s(b_dst + b_smem_bytes, src_half + (size_t)q * 2 * b_tile_bytes + b_tile_bytes, half_bytes, &bfull[s]);
                    } else {
                        mbar_arrive_expect_tx(&full[s], 2 * b_tile_bytes);
                        bulk_g2s(b_dst, src0 + (size_t)q * 2 * b_tile_bytes, 2 * b_tile_bytes, &full[s]);
                    }
                    if (++s == stages) { s = 0; ph ^= 1; }
                }
            }
        }
    } else if (warp == kHWarpMma) {
        // ================= MMA issuer =================
        if (lane == 0 && rank == 0) {
            const int ncols = min(g.bn, g.n - nt * g.bn);                     // multiple of 16
            const uint32_t idesc = make_idesc_f16(PAIR ? 2 * kHBM : kHBM, ncols, 0, 0);
            uint32_t s = 0, ph = 0;
            for (uint32_t tcount = 0; tcount < my_tiles; ++tcount) {
                const uint32_t acc = tcount & 1;
                if (PAIR) mbar_wait_cluster(&tempty[acc], ((tcount >> 1) & 1) ^ 1);      // drained in BOTH CTAs
                else mbar_wait(&tempty[acc], ((tcount >> 1) & 1) ^ 1);
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + acc * (uint32_t)g.acc_stride;
                for (uint32_t q = 0; q < k_chunks; ++q) {
                    if (PAIR) mbar_wait_cluster(&full[s], ph);                           // converted / landed in BOTH CTAs
                    else mbar_wait(&full[s], ph);
                    tc_fence_after();
                    const uint32_t a_hi = smem_u32(op_base + (size_t)s * stage_bytes);
                    const uint32_t a_lo = a_hi + kHATile;
                    const uint32_t b_hi = a_hi + 2 * kHATile;
                    const uint32_t b_lo = b_hi + b_smem_bytes;
#pragma unroll
                    for (int j = 0; j < kHBK / 16; ++j) {
                        const uint64_t dah = make_desc(a_hi + j * 2 * kHALbo, kHALbo, kHASbo);
                        const uint64_t dal = make_desc(a_lo + j * 2 * kHALbo, kHALbo, kHASbo);
                        const uint64_t dbh = make_desc(b_hi + j * 2 * kHBLbo, kHBLbo, kHBSbo);
                        const uint64_t dbl = make_desc(b_lo + j * 2 * kHBLbo, kHBLbo, kHBSbo);
                        // small terms first, the dominant hi*hi product last
                        if (PAIR) {
                            umma_f16_pair(d_tmem, dal, dbh, idesc, (q | (uint32_t)j) ? 1u : 0u);
                            umma_f16_pair(d_tmem, dah, dbl, idesc, 1u);
                            umma_f16_pair(d_tmem, dah, dbh, idesc, 1u);
                        } else {
                            umma_f16(d_tmem, dal, dbh, idesc, (q | (uint32_t)j) ? 1u : 0u);
                            umma_f16(d_tmem, dah, dbl, idesc, 1u);
                            umma_f16(d_tmem, dah, dbh, idesc, 1u);
                        }
                    }
                    if (PAIR) umma_commit_pair(&empty[s]);       // frees the smem slot (in both CTAs) when the MMAs above have read it
                    else umma_commit(&empty[s]);
                    if (++s == stages) { s = 0; ph ^= 1; }
                }
                if (PAIR) umma_commit_pair(&tfull[acc]);         // accumulator complete
                else umma_commit(&tfull[acc]);
            }
        }
    } else {
        // ================= epilogue (8 warps): TMEM -> registers -> unscale (+bias, +C) -> global (+ BatchNorm moments) =================
        // The epilogue of a 128 x 256 tile is a long dependent chain per warp (TMEM load -> staging -> read back -> store);
        // with four warps it took ~20 k cycles per tile and bounded every K <= 256 shape (ncu, profiles/r2_*): two warps per
        // TMEM lane quarter, each taking every other 32-column chunk, halve it.
        float sa, inva;
        f16_scale_from_amax(__ldg(g.a_amax), sa, inva);
        const float invw = __ldg(g.wscale + 1);
        float sc1 = inva * invw, sc2 = 1.f;
        if (!(fabsf(sc1) >= 1.1754944e-38f && fabsf(sc1) <= 3.4028235e38f)) { sc1 = inva; sc2 = invw; }   // product out of range: two exact factors
        const int ew = warp - kHConvWarps;           // 0..7
        const int quarter = warp & 3;                // TMEM lanes 32*quarter .. +31 are accessible to this warp
        const int half = ew >> 2;                    // chunks half, half + 2, half + 4, half + 6 of the n-tile
        float* stg = reinterpret_cast<float*>(op_base + (size_t)g.stages * stage_bytes + kHBarBytes) + ew * 32 * 32;
        const int grp = lane >> 3;                   // row group of the transposed read-back: rows grp, grp + 4, ...
        const int cc = (lane & 7) * 4;               // this lane's float4 inside a 32-column chunk
        const bool stats = g.stat_partials != nullptr;
        const int n0 = nt * g.bn;
        const int ncols = min(g.bn, g.n - n0);
        // Running column moments (count, mean, M2) of every row this warp has stored, Chan-merged one 32-row block at a
        // time while the block is still in registers (no second pass over C).  A CTA only ever sees one n-tile, so the
        // count is the same for all of its columns.  Of the warp's four chunks, chunk t is owned by the lanes of row group t.
        float st_mean[4] = {0.f, 0.f, 0.f, 0.f}, st_m2[4] = {0.f, 0.f, 0.f, 0.f}, st_n = 0.f;
        int64_t tile = unit;
        for (uint32_t tcount = 0; tcount < my_tiles; ++tcount, tile += units) {
            const int64_t m0 = SGB_H_M0_OF(tile);
            const uint32_t acc = tcount & 1;
            mbar_wait(&tfull[acc], (tcount >> 1) & 1);
            tc_fence_after();
            const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + acc * (uint32_t)g.acc_stride;
            const int64_t rows_left = g.m - (m0 + quarter * 32);
            const int nvalid = rows_left >= 32 ? 32 : (rows_left > 0 ? (int)rows_left : 0);   // rows of this warp's block inside C
            const float nb = (float)nvalid;
            const float inv_nb = nvalid ? 1.f / nb : 0.f;
            const float wgt = nvalid ? nb / (st_n + nb) : 0.f;                                // Chan weight of the new block
            float* crow = g.c + (m0 + quarter * 32 + grp) * g.ldc + n0 + cc;
#pragma unroll
            for (int t = 0; t < 4; ++t) {            // unrolled: the moment registers are indexed statically
                const int c0 = (2 * t + half) * 32;
                if (c0 < ncols) {
                    float bm[4], bq[4];
                    const bool col_ok = c0 + cc < ncols;             // ncols is a multiple of 16 => whole float4 valid
                    const float* bias_p = g.bias ? g.bias + n0 + c0 + cc : nullptr;
                    if (nvalid == 32 && c0 + 32 <= ncols)
                        h_epi_chunk<true>(g, taddr + c0, stg, crow + c0, bias_p, lane, grp, cc, nvalid, col_ok, sc1, sc2, stats, inv_nb, bm, bq);
                    else
                        h_epi_chunk<false>(g, taddr + c0, stg, crow + c0, bias_p, lane, grp, cc, nvalid, col_ok, sc1, sc2, stats && nvalid > 0, inv_nb, bm, bq);
                    if (stats && nvalid > 0 && grp == t) {
#pragma unroll
                        for (int q = 0; q < 4; ++q) {
                            const float delta = bm[q] - st_mean[q];
                            st_mean[q] = fmaf(delta, wgt, st_mean[q]);
                            st_m2[q] += bq[q] + delta * delta * st_n * wgt;
                        }
                    }
                }
            }
            st_n += nb;
            tc_fence_before();
            __syncwarp();
            if (lane == 0) {
                if (PAIR) mbar_arrive_cluster(&tempty[acc], 0);
                else mbar_arrive(&tempty[acc]);
            }
        }
        if (stats) {
            const int64_t group = PAIR ? (int64_t)(unit / (uint32_t)g.n_tiles) * 2 + rank : (int64_t)(blockIdx.x / g.n_tiles);
            float* row = g.stat_partials + (group * 4 + quarter) * 3 * g.n;
            const int c0 = (2 * grp + half) * 32;        // the chunk whose moments this lane holds
            if (c0 + cc < ncols) {
                st4(row + 0 * (int64_t)g.n + n0 + c0 + cc, make_float4(st_n, st_n, st_n, st_n));
                st4(row + 1 * (int64_t)g.n + n0 + c0 + cc, make_float4(st_mean[0], st_mean[1], st_mean[2], st_mean[3]));
                st4(row + 2 * (int64_t)g.n + n0 + c0 + cc, make_float4(st_m2[0], st_m2[1], st_m2[2], st_m2[3]));
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (PAIR) cluster_sync_all();                // neither CTA may free its TMEM (or exit) while the pair's MMAs can still touch it
    if (warp == kHWarpMma) {
        tc_fence_after();
        if (PAIR) tmem_dealloc_pair(tmem_base, g.tmem_cols);
        else tmem_dealloc(tmem_base, g.tmem_cols);
    }
#undef SGB_H_M0_OF
}

// fixed-order split reduction -- gemm_simt.cu
int reduce_splits_launch(const float* partial, int splits, int n, int k, float* d, int64_t ldd, int accumulate, cudaStream_t stream);

// ------------------------------------------------------------------------------------------
// weight gradient:  D[n,k] = sum_m G[m,n] * A[m,k];   UMMA M = 128 rows of n, N = k-tile, K = 16 vertices
// ------------------------------------------------------------------------------------------
constexpr int kTBM = 128;                        // rows of D (n) per CTA
constexpr int kTBV = 32;                         // vertices per pipeline stage
constexpr int kTCols = kTBV / 8;                 // 16-byte core-matrix columns (8 vertices each) per stage
constexpr int kTLbo = 128;                       // vertex-adjacent core matrices
constexpr int kTSbo = kTCols * kTLbo + 16;       // row-adjacent core matrices (+16: spreads the transposing stores over the banks)
constexpr int kTGTile = (kTBM / 8) * kTSbo;      // per hi (or lo)
constexpr int kTProducerWarps = 12;              // 384 threads: one (8 vertices x 4 columns) item each per stage
constexpr int kTDrainWarps = 4;
constexpr int kTThreads = (kTProducerWarps + 1 + kTDrainWarps + 1) * 32;   // converters, MMA, drain, TMA loader
constexpr int kTRawStages = 2;                   // single-CTA kernel: fewest raw (TMA) stages (the wide shapes, where shared memory is short)
constexpr int kTMaxRawStages = 8;                // single-CTA kernel: most raw stages in flight, chosen per shape (TArgs::raw_stages)
constexpr int kTBarBytes = 512;                  // single-CTA kernel: barrier block between the operand ring and the drain staging
constexpr int kTSegChunks = 16;                  // 512 vertices per TMEM accumulation segment (tensor-core accumulation truncates)

__host__ __device__ constexpr int t_a_tile_bytes(int bk) { return (bk / 8) * kTSbo; }
__host__ __device__ constexpr int t_stage_bytes(int bk) { return 2 * kTGTile + 2 * t_a_tile_bytes(bk); }

struct TArgs {
    CUtensorMap g_map, a_map;         // G [m, n] box {gbox, 32}; A [m, k] box {abox, 32}; dense (no swizzle) box images
    int gbox, abox;                   // box widths in columns (multiples of 4)
    const float* g; int64_t ldg;
    const float* a; int64_t lda;
    const float* g_amax; const float* a_amax;   // device scalars
    float* partial;                   // [splits][n][k]
    int64_t m; int n; int k;
    int bk;                           // UMMA N: columns of D per CTA (multiple of 16, <= 256)
    int k_tiles; int stages; int raw_stages;
    int conv_groups;                  // 1: all 384 converter threads take every stage; 2: two groups of 192 alternate stages (narrow shapes)
    int64_t m_per_split;              // multiple of kTBV
    uint32_t tmem_cols; int acc_stride;
};

__global__ void __launch_bounds__(kTThreads, 1) k_gemm_tn_f16(const __grid_constant__ TArgs t) {
    extern __shared__ __align__(1024) uint8_t smem[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int stage_bytes = t_stage_bytes(t.bk);
    const int a_tile_bytes = t_a_tile_bytes(t.bk);
    // smem: [raw ring: raw_stages x (G box | A box), fp32][operand ring: stages x stage_bytes][barriers 512 B][drain staging]
    const int raw_g_bytes = kTBV * t.gbox * 4, raw_a_bytes = kTBV * t.abox * 4;
    const int raw_bytes = (raw_g_bytes + raw_a_bytes + 127) / 128 * 128;
    uint8_t* const raw_base = smem;
    const uint32_t raw_stages = (uint32_t)t.raw_stages;
    uint8_t* const op_base = smem + (size_t)raw_stages * raw_bytes;
    uint64_t* full = reinterpret_cast<uint64_t*>(op_base + (size_t)t.stages * stage_bytes);
    uint64_t* empty = full + kHMaxStages;
    uint64_t* tfull = empty + kHMaxStages;      // [2]
    uint64_t* tempty = tfull + 2;               // [2]
    uint64_t* rfull = tempty + 2;               // [raw_stages]
    uint64_t* rempty = rfull + kTMaxRawStages;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(rempty + kTMaxRawStages);

    if (threadIdx.x == 0) {
        for (int s = 0; s < t.stages; ++s) {
            mbar_init(&full[s], kTProducerWarps * 32 / t.conv_groups);
            mbar_init(&empty[s], 1);
        }
        for (int b = 0; b < 2; ++b) {
            mbar_init(&tfull[b], 1);
            mbar_init(&tempty[b], kTDrainWarps);
        }
        for (uint32_t s = 0; s < raw_stages; ++s) {
            mbar_init(&rfull[s], 1);
            mbar_init(&rempty[s], kTProducerWarps * 32 / t.conv_groups);
        }
        fence_barrier_init();
    }
    if (warp == kTProducerWarps) tmem_alloc(tmem_slot, t.tmem_cols);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    const int n0 = (blockIdx.x / t.k_tiles) * kTBM;
    const int k0 = (blockIdx.x % t.k_tiles) * t.bk;
    const int64_t ms = (int64_t)blockIdx.y * t.m_per_split;
    const int64_t me = min64(t.m, ms + t.m_per_split);
    const int chunks = me > ms ? (int)((me - ms + kTBV - 1) / kTBV) : 0;
    const int segments = (chunks + kTSegChunks - 1) / kTSegChunks;
    float sg, invg, sa, inva;
    f16_scale_from_amax(__ldg(t.g_amax), sg, invg);
    f16_scale_from_amax(__ldg(t.a_amax), sa, inva);

    if (warp < kTProducerWarps) {
        // converter item: 8 consecutive vertices (core column mg) x 4 consecutive columns (float4 index c4) of G
        // (threads 0..127) or of A (threads 128..383), read from the raw fp32 stage; the 8 x 4 register block is four
        // 16-byte K-major rows after conversion (the transposition happens in registers)
        // Narrow shapes (gbox + abox <= 192 columns): the stage is too small to keep 384 threads busy and the kernel sits on the
        // length of ONE converter chain per stage (wait -> load -> convert -> fence -> wait -> store -> fence -> arrive, ~0.8 us
        // whatever the shape); two groups of 192 threads alternate stages, so two chains are in flight.
        const int tid = threadIdx.x;
        const int groups = t.conv_groups, gthreads = kTProducerWarps * 32 / groups;
        const int grp = tid / gthreads, lt = tid - grp * gthreads;
        bool is_g, active = true;
        int mg, c4;
        if (groups == 1) {
            is_g = tid < 128;
            const int idx = is_g ? tid : tid - 128;
            const int per_mg = is_g ? 32 : 64;
            mg = idx / per_mg; c4 = idx % per_mg;
        } else {
            const int qg = t.gbox >> 2, qa = t.abox >> 2;            // float4 items per 8-vertex core column
            is_g = lt < 4 * qg;
            const int la = is_g ? lt : lt - 4 * qg;
            const int q = is_g ? qg : qa;
            active = la < 4 * q;
            mg = active ? la / q : 0; c4 = active ? la % q : 0;
        }
        const int box = is_g ? t.gbox : t.abox;
        const bool col_ok = active && c4 * 4 < box;                       // inside the TMA box (zero-filled past n / k)
        const bool in_tile = active && c4 * 4 < (is_g ? kTBM : t.bk);     // inside the operand tile the tensor core reads
        const float sc = is_g ? sg : sa;
        const uint32_t raw_off = (is_g ? 0u : (uint32_t)raw_g_bytes) + (uint32_t)(mg * 8) * (uint32_t)box * 4u + (uint32_t)c4 * 16u;
        const uint32_t tile_off = is_g ? 0u : (uint32_t)(2 * kTGTile);
        const uint32_t lo_off = is_g ? (uint32_t)kTGTile : (uint32_t)a_tile_bytes;
        // rows 4*c4 .. 4*c4+3 of the operand tile, core column mg
        const uint32_t base_off = tile_off + (uint32_t)((c4 * 4) >> 3) * kTSbo + (uint32_t)mg * kTLbo + (uint32_t)((c4 * 4) & 7) * 16;
        // ring positions / phases carried incrementally (no division by a runtime stage count in the loop)
        const uint32_t ug = (uint32_t)groups, ustages = (uint32_t)t.stages;
        uint32_t s = (uint32_t)grp % ustages, ph = ((uint32_t)grp / ustages) & 1u, rs = (uint32_t)grp % raw_stages, rph = ((uint32_t)grp / raw_stages) & 1u;
        for (int it = grp; it < chunks; it += groups) {
            // two groups: the slot's previous user may be the OTHER group and TMA completions are unordered -- wait for that use's
            // release before testing rfull (parity aliasing, see k_gemm_f16)
            if (groups == 2) mbar_wait(&rempty[rs], rph ^ 1);
            mbar_wait(&rfull[rs], rph);
            const uint8_t* raw = raw_base + (size_t)rs * raw_bytes + raw_off;
            uint4 h[4], l[4];
            if (col_ok) {
                float4 v[8];
#pragma unroll
                for (int r = 0; r < 8; ++r) v[r] = *reinterpret_cast<const float4*>(raw + (size_t)r * box * 4);
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const float x0 = (&v[0].x)[q], x1 = (&v[1].x)[q], x2 = (&v[2].x)[q], x3 = (&v[3].x)[q];
                    const float x4 = (&v[4].x)[q], x5 = (&v[5].x)[q], x6 = (&v[6].x)[q], x7 = (&v[7].x)[q];
                    split_f16x2(x0 * sc, x1 * sc, h[q].x, l[q].x);
                    split_f16x2(x2 * sc, x3 * sc, h[q].y, l[q].y);
                    split_f16x2(x4 * sc, x5 * sc, h[q].z, l[q].z);
                    split_f16x2(x6 * sc, x7 * sc, h[q].w, l[q].w);
                }
            } else {
#pragma unroll
                for (int q = 0; q < 4; ++q) { h[q] = make_uint4(0u, 0u, 0u, 0u); l[q] = make_uint4(0u, 0u, 0u, 0u); }
            }
            // the conversion above consumed the loaded values: only now may the raw slot go back to the TMA engine
            fence_proxy_async();
            mbar_arrive(&rempty[rs]);
            mbar_wait(&empty[s], ph ^ 1);
            if (in_tile) {
                uint8_t* st = op_base + (size_t)s * stage_bytes + base_off;
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    *reinterpret_cast<uint4*>(st + q * 16) = h[q];
                    *reinterpret_cast<uint4*>(st + lo_off + q * 16) = l[q];
                }
            }
            fence_proxy_async();
            mbar_arrive(&full[s]);
            s += ug;
            if (s >= ustages) { s -= ustages; ph ^= 1; }
            rs += ug;
            if (rs >= raw_stages) { rs -= raw_stages; rph ^= 1; }
        }
    } else if (warp == kTProducerWarps + 1 + kTDrainWarps) {
        // ================= loader: one lane streams the raw G and A boxes of each 32-vertex stage (TMA 2-D, zero fill) =================
        if (lane == 0) {
            tma_prefetch_desc(&t.g_map);
            tma_prefetch_desc(&t.a_map);
            const uint64_t stream_policy = l2_policy_evict_first();      // G and A are read once: do not push the partial tiles out of L2
            uint32_t rs = 0, rph = 0;
            for (int it = 0; it < chunks; ++it) {
                mbar_wait(&rempty[rs], rph ^ 1);
                mbar_arrive_expect_tx(&rfull[rs], (uint32_t)(raw_g_bytes + raw_a_bytes));
                uint8_t* dst = raw_base + (size_t)rs * raw_bytes;
                const int row = (int)(ms + (int64_t)it * kTBV);
                tma_load_2d_hint(dst, &t.g_map, n0, row, &rfull[rs], stream_policy);
                tma_load_2d_hint(dst + raw_g_bytes, &t.a_map, k0, row, &rfull[rs], stream_policy);
                if (++rs == raw_stages) { rs = 0; rph ^= 1; }
            }
        }
    } else if (warp == kTProducerWarps) {
        if (lane == 0) {
            const uint32_t idesc = make_idesc_f16(kTBM, t.bk, 0, 0);        // both operands K-major (K = vertex)
            uint32_t s = 0, ph = 0;
            for (int it = 0; it < chunks; ++it) {
                const int seg = it / kTSegChunks, in_seg = it % kTSegChunks;
                const int acc = seg & 1;
                if (in_seg == 0) {
                    mbar_wait(&tempty[acc], ((seg >> 1) & 1) ^ 1);          // drained (passes at once for the first two segments)
                    tc_fence_after();
                }
                const uint32_t d_tmem = tmem_base + (uint32_t)(acc * t.acc_stride);
                mbar_wait(&full[s], ph);
                tc_fence_after();
                const uint32_t g_hi = smem_u32(op_base + (size_t)s * stage_bytes);
                const uint32_t g_lo = g_hi + kTGTile;
                const uint32_t a_hi = g_lo + kTGTile;
                const uint32_t a_lo = a_hi + a_tile_bytes;
#pragma unroll
                for (int j = 0; j < kTBV / 16; ++j) {
                    const uint64_t dgh = make_desc(g_hi + j * 2 * kTLbo, kTLbo, kTSbo);
                    const uint64_t dgl = make_desc(g_lo + j * 2 * kTLbo, kTLbo, kTSbo);
                    const uint64_t dah = make_desc(a_hi + j * 2 * kTLbo, kTLbo, kTSbo);
                    const uint64_t dal = make_desc(a_lo + j * 2 * kTLbo, kTLbo, kTSbo);
                    umma_f16(d_tmem, dgl, dah, idesc, (in_seg | j) ? 1u : 0u);
                    umma_f16(d_tmem, dgh, dal, idesc, 1u);
                    umma_f16(d_tmem, dgh, dah, idesc, 1u);
                }
                umma_commit(&empty[s]);
                if (in_seg == kTSegChunks - 1 || it == chunks - 1) umma_commit(&tfull[acc]);
                if (++s == (uint32_t)t.stages) { s = 0; ph ^= 1; }
            }
        }
    } else {
        // drain warps: TMEM lane quarter = warp % 4; running total lives in the CTA's partial tile (L2-resident),
        // always updated by the same thread in the same order -> deterministic
        const int quarter = warp & 3;
        float* out = t.partial + (int64_t)blockIdx.y * t.n * t.k;
        const int gn = n0 + quarter * 32 + lane;
        const int kcols = min(t.bk, t.k - k0);
        const bool vec_ok = (t.k % 4 == 0) && (k0 % 4 == 0) && ((reinterpret_cast<uintptr_t>(out) & 15) == 0);
        const uint64_t keep_policy = l2_policy_evict_last();             // the running partial tile stays in L2 between segments
        if (segments == 0) {
            if (gn < t.n)
                for (int c = 0; c < kcols; ++c) out[(int64_t)gn * t.k + k0 + c] = 0.f;
        }
        float* stg = reinterpret_cast<float*>(op_base + (size_t)t.stages * stage_bytes + kTBarBytes) + quarter * 32 * kHEpiLd;
        for (int seg = 0; seg < segments; ++seg) {
            const int acc = seg & 1;
            mbar_wait(&tfull[acc], (seg >> 1) & 1);
            tc_fence_after();
            const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(acc * t.acc_stride);
            for (int c0 = 0; c0 < kcols; c0 += 32) {
                float v[32];
                tmem_ld_32x32(taddr + (uint32_t)c0, v);          // lane = row of D, registers = 32 consecutive columns
#pragma unroll
                for (int e = 0; e < 32; ++e) v[e] = (v[e] * invg) * inva;
                if (vec_ok) {
                    // transpose through the warp's staging tile: the read-modify-write of the partial tile then moves whole
                    // 128-byte row segments (a lane-per-row access touches 32 lines per instruction)
#pragma unroll
                    for (int e = 0; e < 32; e += 4) *reinterpret_cast<float4*>(stg + lane * kHEpiLd + e) = make_float4(v[e], v[e + 1], v[e + 2], v[e + 3]);
                    __syncwarp();
                    const int cc = (lane & 7) * 4;
                    if (c0 + cc < kcols) {                       // kcols is a multiple of 4 here
                        float* const op0 = out + (int64_t)(n0 + quarter * 32 + (lane >> 3)) * t.k + k0 + c0 + cc;
                        const int nrows = t.n - (n0 + quarter * 32 + (lane >> 3));       // rows j = i*4 + (lane>>3) valid while 4*i < nrows
                        float4 old[8];
                        if (seg != 0) {                          // all eight loads in flight before the first add
#pragma unroll
                            for (int i = 0; i < 8; ++i)
                                old[i] = (4 * i < nrows) ? ldcg_hint(reinterpret_cast<const float4*>(op0 + (int64_t)(4 * i) * t.k), keep_policy) : make_float4(0.f, 0.f, 0.f, 0.f);
                        }
#pragma unroll
                        for (int i = 0; i < 8; ++i) {
                            if (4 * i < nrows) {
                                float4 o = *reinterpret_cast<const float4*>(stg + (i * 4 + (lane >> 3)) * kHEpiLd + cc);
                                if (seg != 0) { o.x += old[i].x; o.y += old[i].y; o.z += old[i].z; o.w += old[i].w; }
                                stcg_hint(reinterpret_cast<float4*>(op0 + (int64_t)(4 * i) * t.k), o, keep_policy);
                            }
                        }
                    }
                    __syncwarp();
                } else if (gn < t.n) {
                    float* op = out + (int64_t)gn * t.k + k0 + c0;
#pragma unroll
                    for (int e = 0; e < 32; ++e)
                        if (c0 + e < kcols) op[e] = seg == 0 ? v[e] : op[e] + v[e];
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(&tempty[acc]);
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == kTProducerWarps) {
        tc_fence_after();
        tmem_dealloc(tmem_base, t.tmem_cols);
    }
}

// ------------------------------------------------------------------------------------------
// weight gradient on CTA PAIRS (cta_group::2):  D[256 n-rows, bk k-cols] per pair, UMMA M = 256 (128 rows per CTA), N = bk.
//   k_gemm_tn_f16 is bound by the shared-memory data pipe (ncu: 79 %; 216 KB of shared-memory traffic per 32-vertex stage against
//   48 KB of HBM traffic).  In a pair, CTA r converts its own G box (32 vertices x its 128 n-rows) and only HALF of the A box (the
//   k-columns [k0 + r bk/2, + bk/2)): the tensor cores exchange the B-operand halves, so the per-CTA traffic of a stage drops to
//   144 KB (raw boxes in + out 64, operand tiles in 32, tensor-core reads 48) and every A element is converted once per pair.
//   Protocol: every CTA has its own raw ring (TMA, local barriers).  Operand ring: the converter warps of BOTH CTAs arrive (one
//   elected lane per warp, after the warp's stores and proxy fences) on the LEADER's (cluster rank 0) full[s]; the leader's MMA lane
//   issues tcgen05.mma.cta_group::2 and commits with a multicast arrive on empty[s] / tfull[acc] of both CTAs; each CTA's drain
//   warps read their own TMEM lanes and arrive on the leader's tempty[acc].
// ------------------------------------------------------------------------------------------
constexpr int kPConvWarps = 8;                   // warps 0..3: G box, warps 4..7: this CTA's half of the A box
constexpr int kPWarpMma = kPConvWarps;           // MMA issuer (leader only) and TMEM owner (both CTAs)
constexpr int kPWarpDrain0 = kPConvWarps + 1;    // warps 9..12 (TMEM lane quarter = warp % 4)
constexpr int kPWarpLoad = kPWarpDrain0 + kTDrainWarps;
constexpr int kPThreads = (kPWarpLoad + 1) * 32; // 448
constexpr int kPMaxRawStages = 4;

struct TPArgs {
    CUtensorMap g_map, a_map;         // G [m, n] box {128, 32}; A [m, k] box {ah, 32}; dense (no swizzle) box images
    int ah;                           // k-columns per CTA = bk / 2 (multiple of 8, <= 128)
    const float* g_amax; const float* a_amax;
    float* partial;                   // [splits][n][k]
    int64_t m; int n; int k;
    int bk;                           // UMMA N (multiple of 16, <= 256)
    int k_tiles; int stages; int raw_stages;
    int64_t m_per_split;
    uint32_t tmem_cols; int acc_stride;
};

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kPThreads, 1) k_gemm_tn_f16_pair(const __grid_constant__ TPArgs t) {
    extern __shared__ __align__(1024) uint8_t smem[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t rank = cluster_ctarank();                 // 0 = leader
    const int a_tile_bytes = t_a_tile_bytes(t.ah);
    const int stage_bytes = 2 * kTGTile + 2 * a_tile_bytes;
    constexpr int raw_g_bytes = kTBV * kTBM * 4;
    const int raw_a_bytes = kTBV * t.ah * 4;
    const int raw_bytes = (raw_g_bytes + raw_a_bytes + 127) / 128 * 128;
    uint8_t* const raw_base = smem;
    uint8_t* const op_base = smem + (size_t)t.raw_stages * raw_bytes;
    uint64_t* full = reinterpret_cast<uint64_t*>(op_base + (size_t)t.stages * stage_bytes);
    uint64_t* empty = full + kHMaxStages;
    uint64_t* tfull = empty + kHMaxStages;      // [2]
    uint64_t* tempty = tfull + 2;               // [2]
    uint64_t* rfull = tempty + 2;               // [raw_stages]
    uint64_t* rempty = rfull + kPMaxRawStages;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(rempty + kPMaxRawStages);

    if (threadIdx.x == 0) {
        for (int s = 0; s < t.stages; ++s) {
            mbar_init(&full[s], 2 * kPConvWarps);            // one elected lane per converter warp, both CTAs (leader's copy is the live one)
            mbar_init(&empty[s], 1);                         // multicast commit
        }
        for (int b = 0; b < 2; ++b) {
            mbar_init(&tfull[b], 1);                         // multicast commit
            mbar_init(&tempty[b], 2 * kTDrainWarps);         // drain warps of both CTAs (leader's copy is the live one)
        }
        for (int s = 0; s < t.raw_stages; ++s) {
            mbar_init(&rfull[s], 1);
            mbar_init(&rempty[s], kPConvWarps * 32);
        }
        fence_barrier_init();
    }
    __syncthreads();
    cluster_sync_all();                                      // both CTAs' barriers exist before anyone arrives remotely
    if (warp == kPWarpMma) tmem_alloc_pair(tmem_slot, t.tmem_cols);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    const int pair = blockIdx.x >> 1;
    const int n0 = (pair / t.k_tiles) * 2 * kTBM + (int)rank * kTBM;      // this CTA's 128 n-rows
    const int k0 = (pair % t.k_tiles) * t.bk;                              // the pair's k-tile
    const int ka = k0 + (int)rank * t.ah;                                  // the k-columns this CTA converts
    const int64_t ms = (int64_t)blockIdx.y * t.m_per_split;
    const int64_t me = min64(t.m, ms + t.m_per_split);
    const int chunks = me > ms ? (int)((me - ms + kTBV - 1) / kTBV) : 0;
    const int segments = (chunks + kTSegChunks - 1) / kTSegChunks;
    float sg, invg, sa, inva;
    f16_scale_from_amax(__ldg(t.g_amax), sg, invg);
    f16_scale_from_amax(__ldg(t.a_amax), sa, inva);

    if (warp < kPConvWarps) {
        // converter item: 8 consecutive vertices (core column mg) x 4 consecutive columns (float4 index c4); threads 0..127 take the
        // G box, 128..255 the A half box; the 8 x 4 register block is four 16-byte K-major rows (the transposition happens in registers)
        const int tid = threadIdx.x;
        const bool is_g = tid < 128;
        const int idx = tid & 127;
        const int mg = idx >> 5, c4 = idx & 31;
        const int box = is_g ? kTBM : t.ah;
        const bool in_tile = c4 * 4 < box;
        const float sc = is_g ? sg : sa;
        const uint32_t raw_off = (is_g ? 0u : (uint32_t)raw_g_bytes) + (uint32_t)(mg * 8) * (uint32_t)box * 4u + (uint32_t)c4 * 16u;
        const uint32_t tile_off = is_g ? 0u : (uint32_t)(2 * kTGTile);
        const uint32_t lo_off = is_g ? (uint32_t)kTGTile : (uint32_t)a_tile_bytes;
        const uint32_t base_off = tile_off + (uint32_t)((c4 * 4) >> 3) * kTSbo + (uint32_t)mg * kTLbo + (uint32_t)((c4 * 4) & 7) * 16;
        uint32_t s = 0, ph = 0, rs = 0, rph = 0;
        for (int it = 0; it < chunks; ++it) {
            mbar_wait(&rfull[rs], rph);
            const uint8_t* raw = raw_base + (size_t)rs * raw_bytes + raw_off;
            uint4 h[4], l[4];
            if (in_tile) {
                float4 v[8];
#pragma unroll
                for (int r = 0; r < 8; ++r) v[r] = *reinterpret_cast<const float4*>(raw + (size_t)r * box * 4);
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const float x0 = (&v[0].x)[q], x1 = (&v[1].x)[q], x2 = (&v[2].x)[q], x3 = (&v[3].x)[q];
                    const float x4 = (&v[4].x)[q], x5 = (&v[5].x)[q], x6 = (&v[6].x)[q], x7 = (&v[7].x)[q];
                    split_f16x2(x0 * sc, x1 * sc, h[q].x, l[q].x);
                    split_f16x2(x2 * sc, x3 * sc, h[q].y, l[q].y);
                    split_f16x2(x4 * sc, x5 * sc, h[q].z, l[q].z);
                    split_f16x2(x6 * sc, x7 * sc, h[q].w, l[q].w);
                }
            }
            fence_proxy_async();                 // the conversion consumed the loaded values: the raw slot may go back to the TMA engine
            mbar_arrive(&rempty[rs]);
            mbar_wait(&empty[s], ph ^ 1);        // multicast commit of the leader's MMAs that read this slot (in BOTH CTAs)
            if (in_tile) {
                uint8_t* st = op_base + (size_t)s * stage_bytes + base_off;
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    *reinterpret_cast<uint4*>(st + q * 16) = h[q];
                    *reinterpret_cast<uint4*>(st + lo_off + q * 16) = l[q];
                }
            }
            fence_proxy_async();                 // generic-proxy stores -> visible to the tensor cores
            __syncwarp();
            if (lane == 0) mbar_arrive_cluster(&full[s], 0);     // this warp's part of the stage is in place (leader's barrier)
            if (++s == (uint32_t)t.stages) { s = 0; ph ^= 1; }
            if (++rs == (uint32_t)t.raw_stages) { rs = 0; rph ^= 1; }
        }
    } else if (warp == kPWarpLoad) {
        if (lane == 0) {
            tma_prefetch_desc(&t.g_map);
            tma_prefetch_desc(&t.a_map);
            const uint64_t stream_policy = l2_policy_evict_first();      // G and A are read once: do not push the partial tiles out of L2
            uint32_t rs = 0, rph = 0;
            for (int it = 0; it < chunks; ++it) {
                mbar_wait(&rempty[rs], rph ^ 1);
                mbar_arrive_expect_tx(&rfull[rs], (uint32_t)(raw_g_bytes + raw_a_bytes));
                uint8_t* dst = raw_base + (size_t)rs * raw_bytes;
                const int row = (int)(ms + (int64_t)it * kTBV);
                tma_load_2d_hint(dst, &t.g_map, n0, row, &rfull[rs], stream_policy);
                tma_load_2d_hint(dst + raw_g_bytes, &t.a_map, ka, row, &rfull[rs], stream_policy);
                if (++rs == (uint32_t)t.raw_stages) { rs = 0; rph ^= 1; }
            }
        }
    } else if (warp == kPWarpMma) {
        if (lane == 0 && rank == 0) {
            const uint32_t idesc = make_idesc_f16(2 * kTBM, t.bk, 0, 0);      // M = 256 over the pair; both operands K-major (K = vertex)
            uint32_t s = 0, ph = 0;
            for (int it = 0; it < chunks; ++it) {
                const int seg = it / kTSegChunks, in_seg = it % kTSegChunks;
                const int acc = seg & 1;
                if (in_seg == 0) {
                    mbar_wait_cluster(&tempty[acc], ((seg >> 1) & 1) ^ 1);    // drained in BOTH CTAs
                    tc_fence_after();
                }
                const uint32_t d_tmem = tmem_base + (uint32_t)(acc * t.acc_stride);
                mbar_wait_cluster(&full[s], ph);                              // converted in BOTH CTAs
                tc_fence_after();
                const uint32_t g_hi = smem_u32(op_base + (size_t)s * stage_bytes);
                const uint32_t g_lo = g_hi + kTGTile;
                const uint32_t a_hi = g_lo + kTGTile;
                const uint32_t a_lo = a_hi + a_tile_bytes;
#pragma unroll
                for (int j = 0; j < kTBV / 16; ++j) {
                    const uint64_t dgh = make_desc(g_hi + j * 2 * kTLbo, kTLbo, kTSbo);
                    const uint64_t dgl = make_desc(g_lo + j * 2 * kTLbo, kTLbo, kTSbo);
                    const uint64_t dah = make_desc(a_hi + j * 2 * kTLbo, kTLbo, kTSbo);
                    const uint64_t dal = make_desc(a_lo + j * 2 * kTLbo, kTLbo, kTSbo);
                    umma_f16_pair(d_tmem, dgl, dah, idesc, (in_seg | j) ? 1u : 0u);
                    umma_f16_pair(d_tmem, dgh, dal, idesc, 1u);
                    umma_f16_pair(d_tmem, dgh, dah, idesc, 1u);
                }
                umma_commit_pair(&empty[s]);
                if (in_seg == kTSegChunks - 1 || it == chunks - 1) umma_commit_pair(&tfull[acc]);
                if (++s == (uint32_t)t.stages) { s = 0; ph ^= 1; }
            }
        }
    } else {
        // drain warps: TMEM lane quarter = warp % 4 (this CTA's 128 rows of D, all bk columns); running total in the partial tile
        const int quarter = warp & 3;
        float* out = t.partial + (int64_t)blockIdx.y * t.n * t.k;
        const int kcols = min(t.bk, t.k - k0);
        float* stg = reinterpret_cast<float*>(op_base + (size_t)t.stages * stage_bytes + 256) + quarter * 32 * kHEpiLd;
        const int cc = (lane & 7) * 4;
        const uint64_t keep_policy = l2_policy_evict_last();             // the running partial tile stays in L2 between segments
        float* const orow = out + (int64_t)(n0 + quarter * 32 + (lane >> 3)) * t.k + k0 + cc;
        if (segments == 0) {
            for (int c0 = 0; c0 < kcols; c0 += 32)
                if (c0 + cc < kcols)
#pragma unroll
                    for (int i = 0; i < 8; ++i) __stcg(reinterpret_cast<float4*>(orow + (int64_t)(4 * i) * t.k + c0), make_float4(0.f, 0.f, 0.f, 0.f));
        }
        for (int seg = 0; seg < segments; ++seg) {
            const int acc = seg & 1;
            mbar_wait(&tfull[acc], (seg >> 1) & 1);
            tc_fence_after();
            const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(acc * t.acc_stride);
            for (int c0 = 0; c0 < kcols; c0 += 32) {
                float v[32];
                tmem_ld_32x32(taddr + (uint32_t)c0, v);          // lane = row of D, registers = 32 consecutive columns
#pragma unroll
                for (int e = 0; e < 32; e += 4)
                    *reinterpret_cast<float4*>(stg + lane * kHEpiLd + e) =
                        make_float4((v[e] * invg) * inva, (v[e + 1] * invg) * inva, (v[e + 2] * invg) * inva, (v[e + 3] * invg) * inva);
                __syncwarp();
                if (c0 + cc < kcols) {                           // kcols is a multiple of 32 here (k % 32 == 0)
                    float4 old[8];
                    if (seg != 0) {                              // all eight loads in flight before the first add
#pragma unroll
                        for (int i = 0; i < 8; ++i) old[i] = ldcg_hint(reinterpret_cast<const float4*>(orow + (int64_t)(4 * i) * t.k + c0), keep_policy);
                    }
#pragma unroll
                    for (int i = 0; i < 8; ++i) {
                        float4 o = *reinterpret_cast<const float4*>(stg + (i * 4 + (lane >> 3)) * kHEpiLd + cc);
                        if (seg != 0) { o.x += old[i].x; o.y += old[i].y; o.z += old[i].z; o.w += old[i].w; }
                        stcg_hint(reinterpret_cast<float4*>(orow + (int64_t)(4 * i) * t.k + c0), o, keep_policy);
                    }
                }
                __syncwarp();
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive_cluster(&tempty[acc], 0);
        }
    }
    tc_fence_before();
    __syncthreads();
    cluster_sync_all();                          // neither CTA may free its TMEM (or exit) while the pair's MMAs can still touch it
    if (warp == kPWarpMma) {
        tc_fence_after();
        tmem_dealloc_pair(tmem_base, t.tmem_cols);
    }
}

// ------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------
struct HPlan {
    int bn, n_tiles, k_chunks, stages, raw_stages, acc_stride;
    size_t smem_bytes, img_bytes;
    uint32_t tmem_cols;
    bool pair;
};

// what the forward kernels take: n a multiple of 16, 16-byte aligned rows of A and C (TMA loads, float4 stores)
bool gemm_f16_supported(int64_t m, int n, int k, int64_t lda, int64_t ldc, const void* a, const void* c, const void* bias) {
    auto al16 = [](const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; };
    return n >= 16 && n % 16 == 0 && k >= 8 && k % 4 == 0 && lda % 4 == 0 && ldc % 4 == 0 && al16(a) && al16(c) &&
           (!bias || al16(bias)) && m >= 1;
}

// CTA pairs: every n-tile must split into two halves of whole core-matrix rows (ncols % 16 == 0), and there must be enough
// m-tiles to keep 74 pairs busy.  SGB_F16_PAIR=0 / 1 forces the single-CTA / pair kernel (from m > 128 rows), so that
// tests and tools/bench_small_shapes.py can run both on small operands.
static bool h_pair_wanted(int64_t m, int n) {
    if (m <= kHBM) return false;                 // a single m-tile: nothing to pair
    if (const char* e = getenv("SGB_F16_PAIR")) return atoi(e) != 0 && n % 16 == 0 && n >= 32;
    return n % 32 == 0 && m >= 32768;
}

static HPlan h_plan(int n, int k, bool pair = false) {
    HPlan p;
    p.pair = pair;
    p.bn = n <= 256 ? n : 256;
    p.n_tiles = (n + p.bn - 1) / p.bn;
    p.k_chunks = (k + kHBK - 1) / kHBK;
    int sb = pair ? h_stage_bytes_pair(p.bn) : h_stage_bytes(p.bn);
    p.raw_stages = 3;
    int st = (kHSmemBudget - kHBarBytes - kHEpiBytes - p.raw_stages * kHRawBytes - 1024) / sb;
    p.stages = st > kHMaxStages ? kHMaxStages : st;
    p.smem_bytes = (size_t)p.raw_stages * kHRawBytes + (size_t)p.stages * sb + kHBarBytes + kHEpiBytes;
    p.img_bytes = (size_t)p.n_tiles * p.k_chunks * 2 * h_b_tile_bytes(p.bn);
    p.acc_stride = (p.bn + 31) / 32 * 32;
    uint32_t cols = 32;
    while (cols < (uint32_t)(2 * p.acc_stride)) cols <<= 1;
    p.tmem_cols = cols;
    return p;
}

// workspace: [0,256) header (w scale, 1/scale, internal amax slot), then the weight image
size_t gemm_f16_workspace(int n, int k) { return h_plan(n, k).img_bytes + 512; }

int gemm_f16_launch(const GemmArgs& g, const float* a_amax, void* ws, size_t ws_bytes, cudaStream_t stream) {
    HPlan p = h_plan(g.n, g.k, h_pair_wanted(g.m, g.n));
    if (!ws || ws_bytes < p.img_bytes + 512) {
        set_error("sgb_gemm: fp16-split engine needs %zu bytes of workspace, got %zu", p.img_bytes + 512, ws_bytes);
        return SGB_ENOSPC;
    }
    if (p.stages < 2) {
        set_error("sgb_gemm: tile does not fit shared memory");
        return SGB_ENOTSUP;
    }
    uint8_t* base = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(ws) + 255) & ~(uintptr_t)255);
    float* hdr = reinterpret_cast<float*>(base);
    uint8_t* img = base + 256;
    if (!a_amax) {
        int rc = amax_launch(g.a, g.lda, g.m, g.k, reinterpret_cast<uint32_t*>(hdr + 2), stream);
        if (rc != SGB_OK) return rc;
        a_amax = hdr + 2;
    }
    k_prep_weights_f16<<<num_sms(), 256, 0, stream>>>(g.b, g.ldb, g.transb, g.n, g.k, p.bn, p.n_tiles, p.k_chunks, reinterpret_cast<__half*>(img), hdr);
    SGB_CHECK_LAUNCH("k_prep_weights_f16");
    {
        static std::atomic<uint64_t> optin{0}, optin_pair{0};
        int rc = p.pair ? smem_optin(reinterpret_cast<const void*>(k_gemm_f16<true>), kHSmemBudget, &optin_pair)
                        : smem_optin(reinterpret_cast<const void*>(k_gemm_f16<false>), kHSmemBudget, &optin);
        if (rc != SGB_OK) return rc;
    }
    HArgs t{};
    {
        int rc = make_tmap_2d(&t.a_map, g.a, g.m, g.k, g.lda, kHBK, kHBM, true);
        if (rc != SGB_OK) return rc;
    }
    t.a = g.a; t.lda = g.lda; t.wp = img; t.wscale = hdr; t.a_amax = a_amax; t.c = g.c; t.ldc = g.ldc; t.m = g.m; t.n = g.n; t.k = g.k;
    t.bn = p.bn; t.n_tiles = p.n_tiles; t.k_chunks = p.k_chunks; t.stages = p.stages; t.raw_stages = p.raw_stages;
    t.bias = g.bias; t.accumulate = g.accumulate; t.stat_partials = g.stat_partials; t.tmem_cols = p.tmem_cols; t.acc_stride = p.acc_stride;
    // grid = (m-tile groups) x n_tiles, a multiple of n_tiles: CTA b always works on n-tile b % n_tiles (its BatchNorm
    // moments then cover one fixed column range) and on the m-tiles b / n_tiles, + groups, ...
    const int64_t m_tiles = ceil_div(g.m, kHBM);
    int groups = num_sms() / p.n_tiles;
    if (groups < 1) groups = 1;
    if (groups > m_tiles) groups = (int)m_tiles;
    if (p.pair) groups = groups / 2 * 2;         // pairs: CTAs 2 u, 2 u + 1 form unit u; the CTA's moment-row group is 2 (u / n_tiles) + rank
    if (p.pair && groups < 2) {
        set_error("sgb_gemm: too few rows for CTA pairs");
        return SGB_ENOTSUP;
    }
    const int grid = groups * p.n_tiles;
    if (g.stat_partials) {
        SGB_CHECK_ARG((reinterpret_cast<uintptr_t>(g.stat_partials) & 15) == 0, "sgb_gemm: stat_partials must be 16-byte aligned");
        const int rows = gemm_stat_rows(g.m), written = 4 * groups;       // one row per epilogue warp; the rest of the caller's rows are empty
        if (rows > written)
            SGB_CUDA(cudaMemsetAsync(g.stat_partials + (size_t)written * 3 * g.n, 0, (size_t)(rows - written) * 3 * g.n * sizeof(float), stream));
    }
    if (p.pair) {
        cudaLaunchConfig_t cfg{};
        cfg.gridDim = dim3((unsigned)grid);
        cfg.blockDim = dim3(kHThreads);
        cfg.dynamicSmemBytes = p.smem_bytes;
        cfg.stream = stream;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeClusterDimension;
        attr[0].val.clusterDim.x = 2; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
        cfg.attrs = attr;
        cfg.numAttrs = 1;
        SGB_CUDA(cudaLaunchKernelEx(&cfg, k_gemm_f16<true>, t));
    } else {
        k_gemm_f16<false><<<grid, kHThreads, p.smem_bytes, stream>>>(t);
    }
    SGB_CHECK_LAUNCH("k_gemm_f16");
    return SGB_OK;
}

// ---- weight gradient ----
struct TPlan {
    int bk, k_tiles, n_tiles, stages, raw_stages, conv_groups, splits, acc_stride, gbox, abox;
    int64_t m_per_split;
    size_t smem_bytes, ws_bytes;
    uint32_t tmem_cols;
};

static TPlan t_plan(int64_t m, int n, int k) {
    TPlan p;
    int kpad = (k + 15) / 16 * 16;
    p.bk = kpad <= 256 ? kpad : 256;
    p.k_tiles = (k + p.bk - 1) / p.bk;
    p.n_tiles = (n + kTBM - 1) / kTBM;
    int sb = t_stage_bytes(p.bk);
    p.gbox = n < kTBM ? n : kTBM;
    p.abox = k < p.bk ? k : p.bk;
    int raw = (kTBV * (p.gbox + p.abox) * 4 + 127) / 128 * 128;
    int st = (kHSmemBudget - kTBarBytes - kTEpiBytes - kTRawStages * raw) / sb;
    p.stages = st > 4 ? 4 : st;
    // The raw ring is what hides the HBM latency: bytes in flight per SM = raw_stages x box bytes.  The narrow layers have 2.5 - 12 KB
    // boxes (32 vertices x (n + k) floats), so two stages left them latency-bound (~0.17 ms whatever the shape): as deep as fits, <= 8.
    int rs = (kHSmemBudget - kTBarBytes - kTEpiBytes - p.stages * sb) / raw;
    p.raw_stages = rs > kTMaxRawStages ? kTMaxRawStages : (rs < kTRawStages ? kTRawStages : rs);
    p.conv_groups = (p.gbox + p.abox <= kTProducerWarps * 32 / 2 && p.stages >= 2 && p.raw_stages >= 2) ? 2 : 1;
    p.smem_bytes = (size_t)p.raw_stages * raw + (size_t)p.stages * sb + kTBarBytes + kTEpiBytes;
    int tiles = p.k_tiles * p.n_tiles;
    int64_t want = num_sms() / tiles;
    if (want < 1) want = 1;
    int64_t maxs = ceil_div(m > 0 ? m : 1, 1024);
    p.splits = (int)(want < maxs ? want : maxs);
    p.m_per_split = ceil_div(ceil_div(m, p.splits), kTBV) * kTBV;
    p.ws_bytes = (size_t)p.splits * n * k * sizeof(float) + 512;
    p.acc_stride = (p.bk + 31) / 32 * 32;
    uint32_t cols = 32;
    while (cols < (uint32_t)(2 * p.acc_stride)) cols <<= 1;
    p.tmem_cols = cols;
    return p;
}

size_t gemm_tn_f16_workspace(int64_t m, int n, int k) { return t_plan(m, n, k).ws_bytes; }

// what both weight-gradient kernels take: 16-byte aligned rows of G and A (TMA loads)
bool gemm_tn_f16_supported(int64_t m, int n, int k, int64_t ldg, int64_t lda, const void* g, const void* a) {
    auto al16 = [](const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; };
    return n % 4 == 0 && k % 4 == 0 && ldg % 4 == 0 && lda % 4 == 0 && al16(g) && al16(a) && m >= 1;
}

int gemm_tn_f16_launch(const float* g, int64_t ldg, const float* a, int64_t lda, const float* g_amax, const float* a_amax, float* d,
                       int64_t ldd, int64_t m, int n, int k, int accumulate, void* ws, size_t ws_bytes, cudaStream_t stream) {
    TPlan p = t_plan(m, n, k);
    if (!ws || ws_bytes < p.ws_bytes) {
        set_error("sgb_gemm_tn: fp16-split engine needs %zu bytes of workspace, got %zu", p.ws_bytes, ws_bytes);
        return SGB_ENOSPC;
    }
    if (p.stages < 2) {
        set_error("sgb_gemm_tn: tile does not fit shared memory");
        return SGB_ENOTSUP;
    }
    uint8_t* base = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(ws) + 255) & ~(uintptr_t)255);
    float* hdr = reinterpret_cast<float*>(base);
    float* partial = reinterpret_cast<float*>(base + 256);
    if (!g_amax) {
        int rc = amax_launch(g, ldg, m, n, reinterpret_cast<uint32_t*>(hdr + 0), stream);
        if (rc != SGB_OK) return rc;
        g_amax = hdr + 0;
    }
    if (!a_amax) {
        int rc = amax_launch(a, lda, m, k, reinterpret_cast<uint32_t*>(hdr + 1), stream);
        if (rc != SGB_OK) return rc;
        a_amax = hdr + 1;
    }
    {
        static std::atomic<uint64_t> optin{0};
        int rc = smem_optin(reinterpret_cast<const void*>(k_gemm_tn_f16), kHSmemBudget, &optin);
        if (rc != SGB_OK) return rc;
    }
    TArgs t{};
    {
        int rc = make_tmap_2d(&t.g_map, g, m, n, ldg, p.gbox, kTBV, false);
        if (rc == SGB_OK) rc = make_tmap_2d(&t.a_map, a, m, k, lda, p.abox, kTBV, false);
        if (rc != SGB_OK) return rc;
        t.gbox = p.gbox; t.abox = p.abox;
    }
    t.g = g; t.ldg = ldg; t.a = a; t.lda = lda; t.g_amax = g_amax; t.a_amax = a_amax; t.partial = partial; t.m = m; t.n = n; t.k = k;
    t.bk = p.bk; t.k_tiles = p.k_tiles; t.stages = p.stages; t.raw_stages = p.raw_stages; t.conv_groups = p.conv_groups; t.m_per_split = p.m_per_split; t.tmem_cols = p.tmem_cols; t.acc_stride = p.acc_stride;
    dim3 grid((unsigned)(p.n_tiles * p.k_tiles), (unsigned)p.splits);
    k_gemm_tn_f16<<<grid, kTThreads, p.smem_bytes, stream>>>(t);
    SGB_CHECK_LAUNCH("k_gemm_tn_f16");
    return reduce_splits_launch(partial, p.splits, n, k, d, ldd, accumulate, stream);
}

// ---- weight gradient on CTA pairs ----
bool gemm_tn_pair_ok(int64_t m, int n, int k) { return n % 256 == 0 && k % 32 == 0 && (k <= 256 || k % 256 == 0) && m >= 4096; }

struct PPlan {
    int bk, ah, k_tiles, pairs, stages, raw_stages, splits, acc_stride;
    int64_t m_per_split;
    size_t smem_bytes, ws_bytes;
    uint32_t tmem_cols;
};

static PPlan p_plan(int64_t m, int n, int k) {
    PPlan p;
    p.bk = k <= 256 ? k : 256;
    p.ah = p.bk / 2;
    p.k_tiles = k / p.bk;
    p.pairs = (n / 256) * p.k_tiles;
    const int sb = 2 * kTGTile + 2 * t_a_tile_bytes(p.ah);
    const int raw = (kTBV * (kTBM + p.ah) * 4 + 127) / 128 * 128;
    p.raw_stages = 3;
    int st = (kHSmemBudget - 256 - kTEpiBytes - p.raw_stages * raw) / sb;
    p.stages = st > kHMaxStages ? kHMaxStages : st;
    p.smem_bytes = (size_t)p.raw_stages * raw + (size_t)p.stages * sb + 256 + kTEpiBytes;
    int64_t want = num_sms() / (2 * p.pairs);
    if (want < 1) want = 1;
    const int64_t maxs = ceil_div(m > 0 ? m : 1, 1024);
    p.splits = (int)(want < maxs ? want : maxs);
    p.m_per_split = ceil_div(ceil_div(m, p.splits), kTBV) * kTBV;
    p.ws_bytes = (size_t)p.splits * n * k * sizeof(float) + 512;
    p.acc_stride = (p.bk + 31) / 32 * 32;
    uint32_t cols = 32;
    while (cols < (uint32_t)(2 * p.acc_stride)) cols <<= 1;
    p.tmem_cols = cols;
    return p;
}

size_t gemm_tn_pair_workspace(int64_t m, int n, int k) { return gemm_tn_pair_ok(m, n, k) ? p_plan(m, n, k).ws_bytes : 0; }

int gemm_tn_pair_launch(const float* g, int64_t ldg, const float* a, int64_t lda, const float* g_amax, const float* a_amax, float* d,
                        int64_t ldd, int64_t m, int n, int k, int accumulate, void* ws, size_t ws_bytes, cudaStream_t stream) {
    PPlan p = p_plan(m, n, k);
    if (!ws || ws_bytes < p.ws_bytes) {
        set_error("sgb_gemm_tn: pair engine needs %zu bytes of workspace, got %zu", p.ws_bytes, ws_bytes);
        return SGB_ENOSPC;
    }
    if (p.stages < 2) {
        set_error("sgb_gemm_tn: pair tile does not fit shared memory");
        return SGB_ENOTSUP;
    }
    uint8_t* base = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(ws) + 255) & ~(uintptr_t)255);
    float* hdr = reinterpret_cast<float*>(base);
    float* partial = reinterpret_cast<float*>(base + 256);
    if (!g_amax) {
        int rc = amax_launch(g, ldg, m, n, reinterpret_cast<uint32_t*>(hdr + 0), stream);
        if (rc != SGB_OK) return rc;
        g_amax = hdr + 0;
    }
    if (!a_amax) {
        int rc = amax_launch(a, lda, m, k, reinterpret_cast<uint32_t*>(hdr + 1), stream);
        if (rc != SGB_OK) return rc;
        a_amax = hdr + 1;
    }
    {
        static std::atomic<uint64_t> optin{0};
        int rc = smem_optin(reinterpret_cast<const void*>(k_gemm_tn_f16_pair), kHSmemBudget, &optin);
        if (rc != SGB_OK) return rc;
    }
    TPArgs t{};
    {
        int rc = make_tmap_2d(&t.g_map, g, m, n, ldg, kTBM, kTBV, false);
        if (rc == SGB_OK) rc = make_tmap_2d(&t.a_map, a, m, k, lda, p.ah, kTBV, false);
        if (rc != SGB_OK) return rc;
    }
    t.ah = p.ah; t.g_amax = g_amax; t.a_amax = a_amax; t.partial = partial; t.m = m; t.n = n; t.k = k;
    t.bk = p.bk; t.k_tiles = p.k_tiles; t.stages = p.stages; t.raw_stages = p.raw_stages; t.m_per_split = p.m_per_split; t.tmem_cols = p.tmem_cols; t.acc_stride = p.acc_stride;
    dim3 grid((unsigned)(2 * p.pairs), (unsigned)p.splits);
    k_gemm_tn_f16_pair<<<grid, kPThreads, p.smem_bytes, stream>>>(t);
    SGB_CHECK_LAUNCH("k_gemm_tn_f16_pair");
    return reduce_splits_launch(partial, p.splits, n, k, d, ldd, accumulate, stream);
}

}  // namespace sgb

extern "C" int sgb_amax(const float* x, int64_t ldx, int64_t m, int c, float* amax_out, void* stream) {
    SGB_CHECK_ARG(x && amax_out && m >= 0 && c > 0 && ldx >= c, "sgb_amax: bad argument");
    SGB_CHECK_ARG(c % 4 == 0 && ldx % 4 == 0 && (reinterpret_cast<uintptr_t>(x) & 15) == 0, "sgb_amax: needs c %% 4 == 0 and 16-byte aligned rows");
    return sgb::amax_launch(x, ldx, m, c, reinterpret_cast<uint32_t*>(amax_out), (cudaStream_t)stream);
}
