// Row-parallel SpMM over the mesh vertex graph:  Y = alpha * (S f(X)) + beta * ADDEND + bias.
//
// Replaces PyG's MessagePassing.propagate (x.index_select(0,row) -> norm.view(-1,1)*x_j ->
// scatter_add at col), SURVEY.md §3.2 / A.1 step 3 / A.2 step 3, forward and -- on the
// transpose CSR -- backward.  No [nnz, C] message tensor, no atomics.  The normalised edge weights are
// computed once per edge_index by the graph builder (graph_build.cu, bit-identical to gcn_norm /
// ChebConv.__norm__) and read as a packed (column, weight) stream in CSR order; the slice of a run of
// vertices is staged into a warp-private shared-memory buffer with cp.async.
//
// Mapping: one sub-warp of LPV lanes per vertex, each lane owns VEC contiguous channels per
// iteration (128-bit loads when C % 4 == 0), ITERS iterations cover up to LPV*VEC*ITERS
// channels per pass; persistent grid, every warp owns runs of consecutive vertices and the co-resident
// warps sweep one window of X together (their neighbourhoods overlap -> L1/L2 hits; DRAM sees X
// once).  Up to NB (6 or 8) x ITERS independent 128-bit gathers in flight per lane.
//
// Arithmetic order is the reference's: per row, messages in CSR (= edge) order, each
// msg = fl(w * x_j) with w = fl(dis_j * dis_i), acc = fl(acc + msg); then the self-loop
// term(s): GCN  acc += fl(fl(dis_i*dis_i) * x_i);  CHEB  acc = fl(fl(acc + x_i) - x_i).
// => bit-identical to the CPU oracle on the same inputs.
//
// HBM roofline: algorithmic bytes = 2*N*C*4 + (nnz + 2N + 1)*4 (SURVEY.md §8(d)).
#include "common.cuh"
#include <stdlib.h>
#include <type_traits>

namespace sgb {

#ifndef SGB_SPMM_MINB2
#define SGB_SPMM_MINB2 4          // resident CTAs per SM for the two-float4-per-lane configurations
#endif
#ifndef SGB_SPMM_NB2
#define SGB_SPMM_NB2 6
#endif
#ifndef SGB_SPMM_ITERS
#define SGB_SPMM_ITERS 2
#endif

constexpr int kSpmmThreads = 128;                       // 4 autonomous warps per CTA
constexpr int kSpmmWarps = kSpmmThreads / 32;

template <int VEC>
struct Vec;
template <>
struct Vec<4> {
    float v[4];
    __device__ __forceinline__ void load(const float* p) {
        float4 t = ldg4(p);
        v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
    }
    __device__ __forceinline__ void store(float* p) const { st4(p, make_float4(v[0], v[1], v[2], v[3])); }
};
template <>
struct Vec<1> {
    float v[1];
    __device__ __forceinline__ void load(const float* p) { v[0] = __ldg(p); }
    __device__ __forceinline__ void store(float* p) const { *p = v[0]; }
};

struct SpmmArgs {
    const int32_t* rowptr;
    const int2* edges;                // [nnz] (col, float bits of the edge weight), CSR order
    const float* dis;
    int mode;
    const float* x;
    int64_t ldx;
    int64_t n;
    int c;
    const float* in_mean;
    const float* in_scale;
    const float* in_shift;
    float slope;
    float alpha;
    const float* addend;
    int64_t ld_addend;
    float beta;
    const float* bias;
    float* y;
    int64_t ldy;
    float* stat_partials;
    const float* xg;                  // ghost rows (vertex-partitioned mode): neighbour ids >= split read xg[(id - split)]
    int64_t ldxg;
    int32_t split;                    // INT32_MAX when there are no ghost rows
    float* amax;                      // optional: max |y| (atomicMax on the float bits; caller zeroes it)
    int64_t row0;                     // first row of the range this launch computes (rows row0 .. row0 + n - 1 of the operator)
};

// A warp owns "runs" of VPW consecutive vertices; run r of the grid goes to warp (r mod total warps), so the
// co-resident warps sweep one window of X together (neighbour rows are served by L1/L2, DRAM sees X once) and the
// warps of a CTA cover 4 adjacent runs (L1 reuse along a mesh row).
#ifndef SGB_SPMM_VPW32
#define SGB_SPMM_VPW32 8
#endif
#ifndef SGB_SPMM_VPW16
#define SGB_SPMM_VPW16 16
#endif
#ifndef SGB_SPMM_VPW8
#define SGB_SPMM_VPW8 32
#endif
// vertices per run.  Full-warp rows (C >= 256) touch 1 KB+ per vertex: a shorter run keeps the window the grid sweeps
// (and with it the reuse distance of a neighbour row in L2) at the size the narrower widths have.
__host__ __device__ constexpr int spmm_vpw(int lpv) { return lpv == 32 ? SGB_SPMM_VPW32 : lpv == 16 ? SGB_SPMM_VPW16 : lpv == 8 ? SGB_SPMM_VPW8 : 32; }
__host__ __device__ constexpr int spmm_ecap(int lpv) { return spmm_vpw(lpv) * 8; }      // staged edges per run (mean degree 6)
__host__ __device__ constexpr int kSpmmNB(int vec, int iters) { return vec * iters >= 8 ? SGB_SPMM_NB2 : 8; }
constexpr int kSpmmSlack = 8;                           // >= NB: a round may read up to NB - 1 slots past the staged slice
__host__ __device__ constexpr int spmm_smem_ints(int lpv, int vec, int iters, bool stats, int nw) {
    const int stage = nw * 2 * ((spmm_vpw(lpv) + 2) + 2 * (spmm_ecap(lpv) + kSpmmSlack));
    const int stat = stats ? 2 * nw * 32 * vec * iters + nw * 32 : 0;
    return stage > stat ? stage : stat;
}

__device__ __forceinline__ void cp_async4(void* smem_dst, const void* gmem_src) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"((uint32_t)__cvta_generic_to_shared(smem_dst)), "l"(gmem_src) : "memory");
}
__device__ __forceinline__ void cp_async8(void* smem_dst, const void* gmem_src) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"((uint32_t)__cvta_generic_to_shared(smem_dst)), "l"(gmem_src) : "memory");
}
__device__ __forceinline__ void cp_async_commit_wait_all() {
    asm volatile("cp.async.commit_group;\n\tcp.async.wait_group 0;" ::: "memory");
}

// Warp-autonomous pipeline (no CTA barrier in the main loop): while run i is gathered, the (col, weight) slice
// of run i+1 and the row pointers of run i+2 are in flight (cp.async into the warp's private double buffer).
// Per vertex there is ONE round of dependent global loads for degree <= NB: the NB neighbour rows and the self
// row are issued together, branch-free -- slots past the row's degree re-read its last neighbour with weight 0
// (acc + 0*x is exact), so the gather code is straight-line and the loads of a whole round are in flight at once.
// FULL: c is a multiple of the pass width (every lane active, no channel predicates).
template <int LPV, int VEC, int ITERS, bool FULL, bool HALO, bool PRO, bool STATS>
__global__ void __launch_bounds__(kSpmmThreads, (VEC * ITERS >= 8) ? (STATS ? SGB_SPMM_MINB2 - 1 : SGB_SPMM_MINB2) : 6) k_spmm(const SpmmArgs a) {
    constexpr int NB = kSpmmNB(VEC, ITERS);                 // neighbour rows in flight per round (register budget)
    constexpr int CH = LPV * VEC * ITERS;                   // channels per pass
    constexpr int SUB = 32 / LPV;                           // sub-warps (vertices in lock-step) per warp
    constexpr int VPW = spmm_vpw(LPV);
    constexpr int ECAP = spmm_ecap(LPV);
    constexpr int NW = kSpmmWarps, THREADS = kSpmmThreads;
    constexpr int STAT_FLOATS = STATS ? 2 * THREADS * VEC * ITERS + THREADS : 0;
    constexpr int EBUF = ECAP + kSpmmSlack;                 // int2 slots per edge buffer
    constexpr int STAGE_INTS = NW * 2 * ((VPW + 2) + 2 * EBUF);
    constexpr int SMEM_INTS = spmm_smem_ints(LPV, VEC, ITERS, STATS, NW);
    static_assert(SMEM_INTS >= STAGE_INTS && SMEM_INTS >= STAT_FLOATS, "shared-memory sizing");
    __shared__ __align__(16) int smem_raw[SMEM_INTS];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int l = lane & (LPV - 1);
    const int sub = lane / LPV;
    // warp-private staging: [2][ECAP] int2 edges, then [2][VPW + 2] row pointers
    int2* const w_edge = reinterpret_cast<int2*>(smem_raw) + (size_t)warp * 2 * EBUF;
    int* const w_rp = smem_raw + NW * 4 * EBUF + warp * 2 * (VPW + 2);
    const uint32_t ldx_b = (uint32_t)a.ldx * 4u, ldxg_b = (uint32_t)a.ldxg * 4u;     // row strides in bytes (host checks they fit)
    auto row_of = [](const float* base, uint32_t row, uint32_t stride_b) {           // one IMAD.WIDE.U32
        return reinterpret_cast<const float*>(reinterpret_cast<const char*>(base) + (uint64_t)row * stride_b);
    };

    // Run schedule: position ri of this warp is run  gw + ri * tw, i.e. run r of the grid goes to warp r mod (#warps in the
    // grid).  (A per-SM contiguous-span schedule with channel slices was measured slower: DESIGN.md §5.2.)
    const int64_t nruns = (a.n + VPW - 1) / VPW;
    const int64_t gw = (int64_t)blockIdx.x * NW + warp;
    const int64_t tw = (int64_t)gridDim.x * NW;
    const int64_t rcount = nruns > gw ? (nruns - 1 - gw) / tw + 1 : 0;

    auto stage_rowptr = [&](int64_t ri, int buf) {         // async; ri (schedule position) may be past the end
        if (ri < rcount) {
            const int64_t v0 = a.row0 + (gw + ri * tw) * VPW;
            const int nv = (int)min64(VPW, a.row0 + a.n - v0);
            for (int i = lane; i <= nv; i += 32) cp_async4(&w_rp[buf * (VPW + 2) + i], a.rowptr + v0 + i);
        }
    };
    auto stage_edges = [&](int64_t ri, int buf) {          // needs the row pointers of that run to be visible
        if (ri < rcount) {
            const int64_t v0 = a.row0 + (gw + ri * tw) * VPW;
            const int nv = (int)min64(VPW, a.row0 + a.n - v0);
            const int e0 = w_rp[buf * (VPW + 2)], ne = w_rp[buf * (VPW + 2) + nv] - e0;
            if (ne <= ECAP)
                for (int i = lane; i < ne; i += 32) cp_async8(&w_edge[buf * EBUF + i], a.edges + e0 + i);
        }
    };

    for (int c0 = 0; c0 < a.c; c0 += CH) {
        // every staged slot must always hold a valid vertex id: rounds read (and discard, weight 0) slots past a row's
        // end.  (Per pass: the statistics merge of the previous pass reused this memory.)
        for (int i = lane; i < 2 * EBUF; i += 32) w_edge[i] = make_int2(0, 0);
        int ch[ITERS];
        bool act[ITERS];
        Vec<VEC> mu[ITERS], sc[ITERS], sh[ITERS];
#pragma unroll
        for (int t = 0; t < ITERS; ++t) {
            ch[t] = c0 + (t * LPV + l) * VEC;
            act[t] = FULL || ch[t] < a.c;
#pragma unroll
            for (int q = 0; q < VEC; ++q) { mu[t].v[q] = 0.f; sc[t].v[q] = 1.f; sh[t].v[q] = 0.f; }
            if (PRO && a.in_scale && act[t]) { mu[t].load(a.in_mean + ch[t]); sc[t].load(a.in_scale + ch[t]); sh[t].load(a.in_shift + ch[t]); }
        }
        // inactive lanes (c not a multiple of the pass width) gather channel 0 of their slot instead: harmless, never stored
        const float* xl = a.x + (act[0] ? ch[0] : 0);
        const float* xgl = HALO ? a.xg + (act[0] ? ch[0] : 0) : nullptr;
        // statistics: pivot-shifted sums per thread (pivot = first value seen), see common.cuh
        float s1[ITERS][VEC], s2[ITERS][VEC], pv[ITERS][VEC];
        float nseen = 0.f;
        float amx = 0.f;
#pragma unroll
        for (int t = 0; t < ITERS; ++t)
#pragma unroll
            for (int q = 0; q < VEC; ++q) { s1[t][q] = 0.f; s2[t][q] = 0.f; pv[t][q] = 0.f; }

        // ---- pipeline prologue: rowptr(0) -> edges(0) + rowptr(1)
        __syncwarp();
        stage_rowptr(0, 0);
        cp_async_commit_wait_all();
        __syncwarp();
        stage_edges(0, 0);
        stage_rowptr(1, 1);

        for (int64_t ri = 0; ri < rcount; ++ri) {
            const int buf = (int)(ri & 1);
            cp_async_commit_wait_all();
            __syncwarp();                                     // this run's edges + next run's row pointers have landed
            stage_edges(ri + 1, buf ^ 1);
            const int64_t v0 = a.row0 + (gw + ri * tw) * VPW;
            const int nv = (int)min64(VPW, a.row0 + a.n - v0);
            const int* srp = w_rp + buf * (VPW + 2);
            const int e0 = srp[0];
            const bool staged = (srp[nv] - e0) <= ECAP;
            const int2* sedge = w_edge + buf * EBUF;

            // one instantiation per edge source (the warp's shared-memory slice, or global memory for runs whose
            // rows are too long to stage)
            auto gather = [&](auto staged_tag) {
                constexpr bool STAGED = decltype(staged_tag)::value;
                // The self-row registers live across the vertex loop (zeroed once, reloaded per vertex): re-zeroing them per
                // vertex made the next vertex's address arithmetic wait on the previous vertex's loads (13-18 % slower, §5.2).
                // (Keeping the rows of v-1 / v cached in registers to save 2 of the 7 gathers was measured slower as well.)
                Vec<VEC> xself[ITERS];
#pragma unroll
                for (int t = 0; t < ITERS; ++t)
#pragma unroll
                    for (int q = 0; q < VEC; ++q) xself[t].v[q] = 0.f;
#pragma unroll 1
                for (int vi = sub; vi < nv; vi += SUB) {
                    const int kb = srp[vi] - e0, ke = srp[vi + 1] - e0;
                    const int64_t v = v0 + vi;
                    Vec<VEC> acc[ITERS];
                    float di = 0.f;
#pragma unroll
                    for (int t = 0; t < ITERS; ++t)
#pragma unroll
                        for (int q = 0; q < VEC; ++q) acc[t].v[q] = 0.f;
                    if (a.mode != SGB_MODE_ADJ) {                 // the self row rides along with the first round of gathers
                        if (a.mode == SGB_MODE_GCN) di = __ldg(a.dis + v);
                        const float* xs = row_of(xl, (uint32_t)v, ldx_b);
#pragma unroll
                        for (int t = 0; t < ITERS; ++t)
                            if (t == 0 || act[t]) xself[t].load(xs + t * LPV * VEC);
                    }
#pragma unroll 1
                    for (int r = kb; r < ke; r += NB) {
                        Vec<VEC> xv[NB][ITERS];
                        float w[NB];
                        const int left = ke - r;
#pragma unroll
                        for (int b = 0; b < NB; ++b) {
                            // slots past the row's end: a valid (stale or next-row) vertex id with weight 0
                            const int2 ed = STAGED ? sedge[r + b] : __ldg(a.edges + e0 + min(r + b, ke - 1));
                            w[b] = (b < left) ? __int_as_float(ed.y) : 0.f;
                            // owned rows live in x, halo (ghost) rows of the partitioned mode in xg
                            const float* xr = (!HALO || ed.x < a.split) ? row_of(xl, (uint32_t)ed.x, ldx_b) : row_of(xgl, (uint32_t)(ed.x - a.split), ldxg_b);
#pragma unroll
                            for (int t = 0; t < ITERS; ++t) {
                                if (t == 0 || act[t]) xv[b][t].load(xr + t * LPV * VEC);
                                else {
#pragma unroll
                                    for (int q = 0; q < VEC; ++q) xv[b][t].v[q] = 0.f;
                                }
                            }
                        }
#pragma unroll
                        for (int b = 0; b < NB; ++b) {
                            // msg = fl(w * x_j), acc = fl(acc + msg): PyG's message / aggregate op order (A.1 step 3)
#pragma unroll
                            for (int t = 0; t < ITERS; ++t)
#pragma unroll
                                for (int q = 0; q < VEC; ++q) {
                                    float xx = xv[b][t].v[q];
                                    if (PRO) xx = bn_lrelu(xx, mu[t].v[q], sc[t].v[q], sh[t].v[q], a.slope);
                                    acc[t].v[q] = __fadd_rn(acc[t].v[q], __fmul_rn(w[b], xx));
                                }
                        }
                    }
                    const float wii = __fmul_rn(di, di);
#pragma unroll
                    for (int t = 0; t < ITERS; ++t) {
                        if (!act[t]) continue;
                        Vec<VEC> out = acc[t];
                        if (a.mode != SGB_MODE_ADJ) {
#pragma unroll
                            for (int q = 0; q < VEC; ++q) {
                                float xx = xself[t].v[q];
                                if (PRO) xx = bn_lrelu(xx, mu[t].v[q], sc[t].v[q], sh[t].v[q], a.slope);
                                if (a.mode == SGB_MODE_GCN) {
                                    out.v[q] = __fadd_rn(out.v[q], __fmul_rn(wii, xx));
                                } else {   // CHEB: the (+1, -1) loop pair of ChebConv.__norm__, not cancelled
                                    out.v[q] = __fadd_rn(__fadd_rn(out.v[q], xx), -xx);
                                }
                            }
                        }
                        if (a.addend) {
                            Vec<VEC> ad;
                            ad.load(a.addend + v * a.ld_addend + ch[t]);
#pragma unroll
                            for (int q = 0; q < VEC; ++q)
                                out.v[q] = __fadd_rn(__fmul_rn(a.alpha, out.v[q]), __fmul_rn(a.beta, ad.v[q]));
                        } else if (a.alpha != 1.f) {
#pragma unroll
                            for (int q = 0; q < VEC; ++q) out.v[q] = __fmul_rn(a.alpha, out.v[q]);
                        }
                        if (a.bias) {                             // L1-resident; not worth 4*ITERS registers across the gather loop
                            Vec<VEC> bs;
                            bs.load(a.bias + ch[t]);
#pragma unroll
                            for (int q = 0; q < VEC; ++q) out.v[q] = __fadd_rn(out.v[q], bs.v[q]);
                        }
                        out.store(a.y + v * a.ldy + ch[t]);
                        if (a.amax) {
#pragma unroll
                            for (int q = 0; q < VEC; ++q) amx = fmaxf(amx, finite_abs(out.v[q]));
                        }
                        if (STATS) {
#pragma unroll
                            for (int q = 0; q < VEC; ++q) {
                                if (nseen == 0.f) pv[t][q] = out.v[q];
                                const float dv = out.v[q] - pv[t][q];
                                s1[t][q] += dv;
                                s2[t][q] = fmaf(dv, dv, s2[t][q]);
                            }
                        }
                    }
                    nseen += 1.f;
                }
            };
            if (staged) gather(std::true_type{});
            else gather(std::false_type{});
            __syncwarp();                                     // every lane is done reading this run's row pointers
            stage_rowptr(ri + 2, buf);
        }
        cp_async_commit_wait_all();
        if (a.amax) {
            __syncthreads();                                  // all warps are done with their staging buffers
            publish_amax(amx, reinterpret_cast<uint32_t*>(smem_raw), a.amax);
            __syncthreads();
        }
        if (STATS) {   // fixed-order block merge (Chan) -> partials[blockIdx.x][3][c] = (count, mean, M2)
            constexpr int GROUPS = THREADS / LPV;
            float* red0 = reinterpret_cast<float*>(smem_raw);
            float* red1 = red0 + THREADS * VEC * ITERS;
            float* redn = red1 + THREADS * VEC * ITERS;
            const int grp = threadIdx.x / LPV;
            __syncthreads();                                  // all warps are done with their staging buffers
#pragma unroll
            for (int t = 0; t < ITERS; ++t)
#pragma unroll
                for (int q = 0; q < VEC; ++q) {
                    const int cl = (t * LPV + l) * VEC + q;     // channel within the pass
                    const Moments mo = from_shifted(nseen, pv[t][q], s1[t][q], s2[t][q]);
                    red0[grp * CH + cl] = mo.mean;
                    red1[grp * CH + cl] = mo.m2;
                }
            if (l == 0) redn[grp] = nseen;
            __syncthreads();
            for (int cl = threadIdx.x; cl < CH; cl += THREADS) {
                if (c0 + cl < a.c) {
                    Moments acc{0.f, 0.f, 0.f};
                    for (int g = 0; g < GROUPS; ++g) acc = merge(acc, Moments{redn[g], red0[g * CH + cl], red1[g * CH + cl]});
                    a.stat_partials[((int64_t)blockIdx.x * 3 + 0) * a.c + c0 + cl] = acc.n;
                    a.stat_partials[((int64_t)blockIdx.x * 3 + 1) * a.c + c0 + cl] = acc.mean;
                    a.stat_partials[((int64_t)blockIdx.x * 3 + 2) * a.c + c0 + cl] = acc.m2;
                }
            }
            __syncthreads();
        }
    }
}

struct SpmmCfg {
    int lpv, vec, iters;
};

static SpmmCfg pick_cfg(int c, bool aligned) {
    SpmmCfg k;
    if (c % 4 == 0 && aligned) {
        // 128-bit lanes, two per lane wherever the row is wide enough: halves the per-vertex index / address
        // instruction overhead (the kernel is issue-bound, not DRAM-bound, at one float4 per lane)
        k.vec = 4;
        const int lanes = c / 4;
        if (lanes == 1) { k.lpv = 1; k.iters = 1; }
        else {
            int p = 1;
            while (p * 2 < lanes && p < 32) p <<= 1;
            k.lpv = p;
            k.iters = 2;
            if (SGB_SPMM_ITERS == 1) {     // experiment: one float4 per lane (more warps per SM, more index instructions per byte)
                p = 1;
                while (p < lanes && p < 32) p <<= 1;
                k.lpv = p;
                k.iters = 1;
            }
        }
    } else {
        k.vec = 1;
        k.lpv = c <= 4 ? 4 : 32;
        k.iters = 1;
    }
    return k;
}

static int spmm_per_sm(const SpmmCfg& k, bool stats) { return (k.vec * k.iters >= 8) ? (stats ? SGB_SPMM_MINB2 - 1 : SGB_SPMM_MINB2) : 6; }

static int spmm_grid(int64_t n, const SpmmCfg& k, bool stats) {
    int64_t need = ceil_div(ceil_div(n > 0 ? n : 1, spmm_vpw(k.lpv)), kSpmmWarps);
    int64_t cap = (int64_t)num_sms() * spmm_per_sm(k, stats);
    return (int)(need < cap ? need : cap);
}

}  // namespace sgb

extern "C" int sgb_spmm_stat_rows(int64_t n, int c) {
    if (n < 0 || c <= 0) return 0;
    // alignment of x/y is not known here: the row count must not depend on it, so both
    // candidate configurations are sized and the larger grid is reported.
    int g1 = sgb::spmm_grid(n, sgb::pick_cfg(c, true), true);
    int g2 = sgb::spmm_grid(n, sgb::pick_cfg(c, false), true);
    return g1 > g2 ? g1 : g2;
}

extern "C" int sgb_spmm(const int32_t* rowptr, const sgb_edge_t* edges, const float* dis, int mode,
                        const float* x, int64_t ldx, int64_t n, int c,
                        const float* in_mean, const float* in_scale, const float* in_shift, float slope,
                        float alpha, const float* addend, int64_t ld_addend, float beta,
                        const float* bias, float* y, int64_t ldy, float* stat_partials, float* amax_out, void* stream_) {
    return sgb_spmm_halo(rowptr, edges, dis, mode, x, ldx, n, c, nullptr, 0, n, in_mean, in_scale, in_shift, slope, alpha, addend, ld_addend,
                         beta, bias, y, ldy, stat_partials, amax_out, stream_);
}

extern "C" int sgb_spmm_halo(const int32_t* rowptr, const sgb_edge_t* edges, const float* dis, int mode,
                             const float* x, int64_t ldx, int64_t n, int c, const float* x_ghost, int64_t ld_ghost, int64_t n_split,
                             const float* in_mean, const float* in_scale, const float* in_shift, float slope,
                             float alpha, const float* addend, int64_t ld_addend, float beta,
                             const float* bias, float* y, int64_t ldy, float* stat_partials, float* amax_out, void* stream_) {
    return sgb_spmm_range(rowptr, edges, dis, mode, x, ldx, 0, n, c, x_ghost, ld_ghost, n_split, in_mean, in_scale, in_shift, slope, alpha, addend,
                          ld_addend, beta, bias, y, ldy, stat_partials, amax_out, stream_);
}

extern "C" int sgb_spmm_range(const int32_t* rowptr, const sgb_edge_t* edges, const float* dis, int mode,
                              const float* x, int64_t ldx, int64_t row_begin, int64_t n, int c, const float* x_ghost, int64_t ld_ghost, int64_t n_split,
                              const float* in_mean, const float* in_scale, const float* in_shift, float slope,
                              float alpha, const float* addend, int64_t ld_addend, float beta,
                              const float* bias, float* y, int64_t ldy, float* stat_partials, float* amax_out, void* stream_) {
    using namespace sgb;
    cudaStream_t stream = (cudaStream_t)stream_;
    SGB_CHECK_ARG(n >= 0 && c > 0, "sgb_spmm: bad shape n=%lld c=%d", (long long)n, c);
    SGB_CHECK_ARG(mode == SGB_MODE_GCN || mode == SGB_MODE_CHEB || mode == SGB_MODE_ADJ, "sgb_spmm: bad mode %d", mode);
    SGB_CHECK_ARG(rowptr && dis && x && y, "sgb_spmm: null pointer");
    SGB_CHECK_ARG((reinterpret_cast<uintptr_t>(edges) & 7) == 0, "sgb_spmm: edges must be 8-byte aligned");
    SGB_CHECK_ARG(ldx >= c && ldy >= c && (!addend || ld_addend >= c), "sgb_spmm: leading dimension < c");
    SGB_CHECK_ARG((in_scale == nullptr) == (in_shift == nullptr) && (in_scale == nullptr) == (in_mean == nullptr),
                  "sgb_spmm: in_mean / in_scale / in_shift must come together");
    SGB_CHECK_ARG(x != y, "sgb_spmm: in-place aggregation is not supported");
    SGB_CHECK_ARG(row_begin >= 0 && ldx < (int64_t)1 << 30 && ld_ghost < (int64_t)1 << 30 && row_begin + n < (int64_t)0x7fffffff,
                  "sgb_spmm: row stride / vertex count out of range");
    SGB_CHECK_ARG(!x_ghost || (ld_ghost >= c && n_split >= 0 && n_split < (int64_t)0x7fffffff), "sgb_spmm_halo: bad ghost block");
    if (n == 0) return SGB_OK;
    auto al16 = [](const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; };
    bool aligned = al16(x) && al16(y) && ldx % 4 == 0 && ldy % 4 == 0 && (!x_ghost || (al16(x_ghost) && ld_ghost % 4 == 0)) && (!addend || (al16(addend) && ld_addend % 4 == 0)) &&
                   (!bias || al16(bias)) && (!in_scale || (al16(in_scale) && al16(in_shift) && al16(in_mean)));
    SpmmCfg k = pick_cfg(c, aligned);
    int grid = spmm_grid(n, k, stat_partials != nullptr);
    if (stat_partials) {
        // rows the caller sized for; unused rows must read as zero
        int rows = sgb_spmm_stat_rows(n, c);
        if (rows > grid)
            SGB_CUDA(cudaMemsetAsync(stat_partials + (size_t)grid * 3 * c, 0, (size_t)(rows - grid) * 3 * c * sizeof(float), stream));
    }
    const bool pro = in_scale != nullptr, st = stat_partials != nullptr, halo = x_ghost != nullptr;
    if (!pro) slope = 1.f;            // the general instantiation applies lrelu((x - 0) * 1 + 0, slope): identity
    SpmmArgs a{rowptr, reinterpret_cast<const int2*>(edges), dis, mode, x, ldx, n, c, in_mean, in_scale, in_shift, slope, alpha, addend, ld_addend, beta, bias, y, ldy, stat_partials,
               x_ghost, ld_ghost, x_ghost ? (int32_t)n_split : (int32_t)0x7fffffff, amax_out, row_begin};
    // the BatchNorm prologue and ragged widths are rare operands: they share one (slower, fully general) instantiation
#define SGB_SPMM_CASE(L, V, I)                                                                                  \
    if (k.lpv == L && k.vec == V && k.iters == I) {                                                             \
        if (pro || c % (L * V * I) != 0) {                                                                      \
            if (st) k_spmm<L, V, I, false, true, true, true><<<grid, kSpmmThreads, 0, stream>>>(a);             \
            else k_spmm<L, V, I, false, true, true, false><<<grid, kSpmmThreads, 0, stream>>>(a);               \
        } else if (halo) { /* vertex-partitioned mode: the fast path plus the ghost-block select */              \
            if (st) k_spmm<L, V, I, true, true, false, true><<<grid, kSpmmThreads, 0, stream>>>(a);             \
            else k_spmm<L, V, I, true, true, false, false><<<grid, kSpmmThreads, 0, stream>>>(a);               \
        } else if (st) k_spmm<L, V, I, true, false, false, true><<<grid, kSpmmThreads, 0, stream>>>(a);         \
        else k_spmm<L, V, I, true, false, false, false><<<grid, kSpmmThreads, 0, stream>>>(a);                  \
        SGB_CHECK_LAUNCH("k_spmm");                                                                             \
        return SGB_OK;                                                                                          \
    }
    SGB_SPMM_CASE(1, 4, 1)
    SGB_SPMM_CASE(1, 4, 2)
#if SGB_SPMM_ITERS == 1
    SGB_SPMM_CASE(2, 4, 1)
    SGB_SPMM_CASE(4, 4, 1)
    SGB_SPMM_CASE(8, 4, 1)
    SGB_SPMM_CASE(16, 4, 1)
    SGB_SPMM_CASE(32, 4, 1)
#endif
    SGB_SPMM_CASE(2, 4, 2)
    SGB_SPMM_CASE(4, 4, 2)
    SGB_SPMM_CASE(8, 4, 2)
    SGB_SPMM_CASE(16, 4, 2)
    SGB_SPMM_CASE(32, 4, 2)
    SGB_SPMM_CASE(4, 1, 1)
    SGB_SPMM_CASE(32, 1, 1)
#undef SGB_SPMM_CASE
    set_error("sgb_spmm: no kernel configuration for c=%d", c);
    return SGB_ENOTSUP;
}

// ---------------- row gather (halo pack): out[k, :] = x[idx[k], :] ----------------
namespace sgb {
template <int VEC>
__global__ void __launch_bounds__(256) k_gather_rows(const float* __restrict__ x, int64_t ldx, const int32_t* __restrict__ idx, int64_t count,
                                                     int c, float* __restrict__ out, int64_t ldo) {
    const int per_row = (c + VEC - 1) / VEC;
    const int64_t total = count * per_row;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t k = i / per_row;
        const int ch = (int)(i % per_row) * VEC;
        const int64_t r = idx[k];
        if (VEC == 4) st4(out + k * ldo + ch, ldg4(x + r * ldx + ch));
        else out[k * ldo + ch] = __ldg(x + r * ldx + ch);
    }
}
}  // namespace sgb

extern "C" int sgb_gather_rows(const float* x, int64_t ldx, const int32_t* idx, int64_t count, int c, float* out, int64_t ldo, void* stream_) {
    using namespace sgb;
    cudaStream_t stream = (cudaStream_t)stream_;
    SGB_CHECK_ARG(count >= 0 && c > 0 && ldx >= c && ldo >= c, "sgb_gather_rows: bad shape");
    if (count == 0) return SGB_OK;
    SGB_CHECK_ARG(x && idx && out, "sgb_gather_rows: null pointer");
    auto al16 = [](const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; };
    const bool vec = c % 4 == 0 && ldx % 4 == 0 && ldo % 4 == 0 && al16(x) && al16(out);
    const int64_t total = count * (vec ? c / 4 : c);
    const int grid = (int)min64(ceil_div(total, 256), (int64_t)num_sms() * 16);
    if (vec) k_gather_rows<4><<<grid, 256, 0, stream>>>(x, ldx, idx, count, c, out, ldo);
    else k_gather_rows<1><<<grid, 256, 0, stream>>>(x, ldx, idx, count, c, out, ldo);
    SGB_CHECK_LAUNCH("k_gather_rows");
    return SGB_OK;
}
