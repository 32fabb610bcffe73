// fp32 CUDA-core tiles for the dense feature transform and its gradients (engine 1).
//
// Replaces F.linear inside GCNConv.lin / ChebConv.lins[k] / nn.Linear (util/networks.py:25,35,
// 42,52,58-61) at widths where the contraction is too thin for the tensor pipe (K or N < 64,
// SURVEY.md §8(d)) and serves as the always-available exact-fp32 path; the tcgen05 fp16-split
// tiles live in gemm_f16.cu.  Fused: bias and per-tile BatchNorm statistics in the epilogue
// (no extra pass over C).
#include "common.cuh"

namespace sgb {

constexpr int kGemmBM = 128;   // rows per CTA tile == rows per stat partial (all engines)
constexpr int kGemmBK = 16;
constexpr int kGemmThreads = 256;


// C tile BM x BN, thread micro-tile TM x TN with TM = 8, TN = BN / 16.
template <int BN>
__global__ void __launch_bounds__(kGemmThreads) k_gemm_simt(const GemmArgs g) {
    constexpr int BM = kGemmBM, BK = kGemmBK, TM = 8, TN = BN / 16;
    __shared__ __align__(16) float smem_ab[BK * (BM + 4) + BK * (BN + 4)];
    float (*As)[BM + 4] = reinterpret_cast<float (*)[BM + 4]>(smem_ab);
    float (*Bs)[BN + 4] = reinterpret_cast<float (*)[BN + 4]>(smem_ab + BK * (BM + 4));
    const int tid = threadIdx.x;
    const int tx = tid % 16, ty = tid / 16;
    const int n0 = blockIdx.y * BN;
    const bool a_vec = (g.lda % 4 == 0) && ((reinterpret_cast<uintptr_t>(g.a) & 15) == 0);
    const bool b_vec = (g.ldb % 4 == 0) && ((reinterpret_cast<uintptr_t>(g.b) & 15) == 0);

    // persistent over the 128-row tiles blockIdx.x, + gridDim.x, ...: the BatchNorm moments of all of a CTA's tiles are
    // Chan-merged in registers, so the partials buffer holds gridDim.x <= gemm_stat_rows(m) rows however large m is
    Moments run[TN];
#pragma unroll
    for (int j = 0; j < TN; ++j) run[j] = Moments{0.f, 0.f, 0.f};
    const int64_t m_tiles = (g.m + BM - 1) / BM;
    for (int64_t mt = blockIdx.x; mt < m_tiles; mt += gridDim.x) {
    const int64_t m0 = mt * BM;
    float acc[TM][TN];
#pragma unroll
    for (int i = 0; i < TM; ++i)
#pragma unroll
        for (int j = 0; j < TN; ++j) acc[i][j] = 0.f;

    for (int k0 = 0; k0 < g.k; k0 += BK) {
        // ---- A tile: BM x BK, k contiguous in memory; stored transposed As[k][m]
#pragma unroll
        for (int i = 0; i < (BM * BK / 4) / kGemmThreads; ++i) {
            const int s = tid + i * kGemmThreads;
            const int r = s / (BK / 4), kq = (s % (BK / 4)) * 4;
            const int64_t gm = m0 + r;
            float v[4] = {0.f, 0.f, 0.f, 0.f};
            if (gm < g.m) {
                const float* p = g.a + gm * g.lda + k0 + kq;
                if (a_vec && k0 + kq + 3 < g.k) {
                    float4 t = ldg4(p);
                    v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
                } else {
#pragma unroll
                    for (int q = 0; q < 4; ++q)
                        if (k0 + kq + q < g.k) v[q] = __ldg(p + q);
                }
            }
#pragma unroll
            for (int q = 0; q < 4; ++q) As[kq + q][r] = v[q];
        }
        // ---- B tile -> Bs[k][n]
        if (g.transb) {   // B is [n, k], k contiguous
            for (int s = tid; s < BN * BK / 4; s += kGemmThreads) {
                const int r = s / (BK / 4), kq = (s % (BK / 4)) * 4;
                const int gn = n0 + r;
                float v[4] = {0.f, 0.f, 0.f, 0.f};
                if (gn < g.n) {
                    const float* p = g.b + (int64_t)gn * g.ldb + k0 + kq;
                    if (b_vec && k0 + kq + 3 < g.k) {
                        float4 t = ldg4(p);
                        v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
                    } else {
#pragma unroll
                        for (int q = 0; q < 4; ++q)
                            if (k0 + kq + q < g.k) v[q] = __ldg(p + q);
                    }
                }
#pragma unroll
                for (int q = 0; q < 4; ++q) Bs[kq + q][r] = v[q];
            }
        } else {          // B is [k, n], n contiguous
            for (int s = tid; s < BK * BN / 4; s += kGemmThreads) {
                const int kr = s / (BN / 4), nq = (s % (BN / 4)) * 4;
                const int gk = k0 + kr;
                float v[4] = {0.f, 0.f, 0.f, 0.f};
                if (gk < g.k) {
                    const float* p = g.b + (int64_t)gk * g.ldb + n0 + nq;
                    if (b_vec && n0 + nq + 3 < g.n) {
                        float4 t = ldg4(p);
                        v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
                    } else {
#pragma unroll
                        for (int q = 0; q < 4; ++q)
                            if (n0 + nq + q < g.n) v[q] = __ldg(p + q);
                    }
                }
#pragma unroll
                for (int q = 0; q < 4; ++q) Bs[kr][nq + q] = v[q];
            }
        }
        __syncthreads();
#pragma unroll
        for (int kk = 0; kk < BK; ++kk) {
            float av[TM], bv[TN];
#pragma unroll
            for (int i = 0; i < TM; i += 4) {
                float4 t = *reinterpret_cast<const float4*>(&As[kk][ty * TM + i]);
                av[i] = t.x; av[i + 1] = t.y; av[i + 2] = t.z; av[i + 3] = t.w;
            }
#pragma unroll
            for (int j = 0; j < TN; ++j) bv[j] = Bs[kk][tx + 16 * j];   // column n0 + tx + 16 j: conflict-free
#pragma unroll
            for (int i = 0; i < TM; ++i)
#pragma unroll
                for (int j = 0; j < TN; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
        }
        __syncthreads();
    }

    // ---- epilogue: (+C) + bias, store, per-tile column moments (count, mean, M2)
    Moments mo[TN];
#pragma unroll
    for (int j = 0; j < TN; ++j) {
        mo[j] = Moments{0.f, 0.f, 0.f};
        const int gn = n0 + tx + 16 * j;
        if (gn >= g.n) continue;
        const float bj = g.bias ? __ldg(g.bias + gn) : 0.f;
        float vals[TM];
        float cnt = 0.f, sum = 0.f;
#pragma unroll
        for (int i = 0; i < TM; ++i) {
            const int64_t gm = m0 + ty * TM + i;
            vals[i] = 0.f;
            if (gm >= g.m) continue;
            float* cp = g.c + gm * g.ldc + gn;
            float v = acc[i][j];
            if (g.accumulate) v += *cp;
            v += bj;
            *cp = v;
            vals[i] = v;
            cnt += 1.f;
            sum += v;
        }
        if (cnt > 0.f) {          // two-pass over the thread's own 8 rows
            const float mean = sum / cnt;
            float m2 = 0.f;
#pragma unroll
            for (int i = 0; i < TM; ++i)
                if (m0 + ty * TM + i < g.m) { const float d = vals[i] - mean; m2 = fmaf(d, d, m2); }
            mo[j] = Moments{cnt, mean, m2};
        }
    }
#pragma unroll
    for (int j = 0; j < TN; ++j) run[j] = merge(run[j], mo[j]);
    }   // m-tile loop
    if (g.stat_partials) {
        __syncthreads();
        __shared__ float red[3 * 16 * BN];   // 3 planes of [16 ty][BN]
        float* r0 = red;
        float* r1 = r0 + 16 * BN;
        float* r2 = r1 + 16 * BN;
#pragma unroll
        for (int j = 0; j < TN; ++j) {
            r0[ty * BN + tx + 16 * j] = run[j].n;
            r1[ty * BN + tx + 16 * j] = run[j].mean;
            r2[ty * BN + tx + 16 * j] = run[j].m2;
        }
        __syncthreads();
        for (int cl = tid; cl < BN; cl += kGemmThreads) {
            if (n0 + cl < g.n) {
                Moments a{0.f, 0.f, 0.f};
#pragma unroll
                for (int r = 0; r < 16; ++r) a = merge(a, Moments{r0[r * BN + cl], r1[r * BN + cl], r2[r * BN + cl]});
                g.stat_partials[((int64_t)blockIdx.x * 3 + 0) * g.n + n0 + cl] = a.n;
                g.stat_partials[((int64_t)blockIdx.x * 3 + 1) * g.n + n0 + cl] = a.mean;
                g.stat_partials[((int64_t)blockIdx.x * 3 + 2) * g.n + n0 + cl] = a.m2;
            }
        }
    }
}

int gemm_simt_launch(const GemmArgs& g, cudaStream_t stream) {
    int bn = g.n <= 16 ? 16 : g.n <= 32 ? 32 : g.n <= 64 ? 64 : 128;
    const int rows = gemm_stat_rows(g.m);
    const int gx = (int)min64(ceil_div(g.m, kGemmBM), rows);
    dim3 grid((unsigned)gx, (unsigned)ceil_div(g.n, bn));
    if (g.stat_partials && rows > gx)
        SGB_CUDA(cudaMemsetAsync(g.stat_partials + (size_t)gx * 3 * g.n, 0, (size_t)(rows - gx) * 3 * g.n * sizeof(float), stream));
    switch (bn) {
        case 16: k_gemm_simt<16><<<grid, kGemmThreads, 0, stream>>>(g); break;
        case 32: k_gemm_simt<32><<<grid, kGemmThreads, 0, stream>>>(g); break;
        case 64: k_gemm_simt<64><<<grid, kGemmThreads, 0, stream>>>(g); break;
        default: k_gemm_simt<128><<<grid, kGemmThreads, 0, stream>>>(g); break;
    }
    SGB_CHECK_LAUNCH("k_gemm_simt");
    return SGB_OK;
}

// ---------------------------------------------------------------------------------------
// Weight gradient D[n,k] (+)= G[m,n]^T A[m,k]: reduction over the (huge) vertex dimension.
// Each CTA owns a 64x64 tile of D and one m-slice; slices are summed afterwards in a fixed
// order (deterministic, no atomics).
// ---------------------------------------------------------------------------------------
constexpr int kTnTile = 64;
constexpr int kTnStep = 16;

__global__ void __launch_bounds__(256) k_gemm_tn_partial(const float* __restrict__ gmat, int64_t ldg, const float* __restrict__ amat,
                                                         int64_t lda, int64_t m, int n, int k, int64_t m_per_split,
                                                         float* __restrict__ partial) {
    __shared__ __align__(16) float Gs[kTnStep][kTnTile + 4];
    __shared__ __align__(16) float As[kTnStep][kTnTile + 4];
    const int tiles_k = (k + kTnTile - 1) / kTnTile;
    const int n0 = (blockIdx.x / tiles_k) * kTnTile;
    const int k0 = (blockIdx.x % tiles_k) * kTnTile;
    const int64_t ms = (int64_t)blockIdx.y * m_per_split;
    const int64_t me = min(m, ms + m_per_split);
    const int tid = threadIdx.x, tx = tid % 16, ty = tid / 16;
    const bool g_vec = (ldg % 4 == 0) && ((reinterpret_cast<uintptr_t>(gmat) & 15) == 0);
    const bool a_vec = (lda % 4 == 0) && ((reinterpret_cast<uintptr_t>(amat) & 15) == 0);
    float acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
    const int lr = tid / 16, lc = (tid % 16) * 4;     // one float4 of each tile per thread
    for (int64_t mm = ms; mm < me; mm += kTnStep) {
        float gv[4] = {0.f, 0.f, 0.f, 0.f}, av[4] = {0.f, 0.f, 0.f, 0.f};
        const int64_t gm = mm + lr;
        if (gm < me) {
            const float* gp = gmat + gm * ldg + n0 + lc;
            if (g_vec && n0 + lc + 3 < n) {
                float4 t = ldg4(gp);
                gv[0] = t.x; gv[1] = t.y; gv[2] = t.z; gv[3] = t.w;
            } else {
#pragma unroll
                for (int q = 0; q < 4; ++q)
                    if (n0 + lc + q < n) gv[q] = __ldg(gp + q);
            }
            const float* ap = amat + gm * lda + k0 + lc;
            if (a_vec && k0 + lc + 3 < k) {
                float4 t = ldg4(ap);
                av[0] = t.x; av[1] = t.y; av[2] = t.z; av[3] = t.w;
            } else {
#pragma unroll
                for (int q = 0; q < 4; ++q)
                    if (k0 + lc + q < k) av[q] = __ldg(ap + q);
            }
        }
        *reinterpret_cast<float4*>(&Gs[lr][lc]) = make_float4(gv[0], gv[1], gv[2], gv[3]);
        *reinterpret_cast<float4*>(&As[lr][lc]) = make_float4(av[0], av[1], av[2], av[3]);
        __syncthreads();
#pragma unroll
        for (int s = 0; s < kTnStep; ++s) {
            float4 gq = *reinterpret_cast<const float4*>(&Gs[s][ty * 4]);
            float4 aq = *reinterpret_cast<const float4*>(&As[s][tx * 4]);
            const float gg[4] = {gq.x, gq.y, gq.z, gq.w};
            const float aa[4] = {aq.x, aq.y, aq.z, aq.w};
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(gg[i], aa[j], acc[i][j]);
        }
        __syncthreads();
    }
    float* out = partial + (int64_t)blockIdx.y * n * k;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int gn = n0 + ty * 4 + i;
        if (gn >= n) continue;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int gk = k0 + tx * 4 + j;
            if (gk < k) out[(int64_t)gn * k + gk] = acc[i][j];
        }
    }
}

__global__ void k_reduce_splits(const float* __restrict__ partial, int splits, int n, int k, float* __restrict__ d, int64_t ldd,
                                int accumulate) {
    const int64_t total = (int64_t)n * k;
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        float s = 0.f;
        for (int sidx = 0; sidx < splits; ++sidx) s += partial[(int64_t)sidx * total + i];
        float* dp = d + (i / k) * ldd + (i % k);
        *dp = accumulate ? *dp + s : s;
    }
}

// D (+)= the sum of `splits` partial [n, k] tiles, added in split order (deterministic); also ends the tcgen05 weight
// gradients of gemm_f16.cu
int reduce_splits_launch(const float* partial, int splits, int n, int k, float* d, int64_t ldd, int accumulate, cudaStream_t stream) {
    const int64_t total = (int64_t)n * k;
    const int rgrid = (int)min64(ceil_div(total, 256), (int64_t)num_sms() * 8);
    k_reduce_splits<<<rgrid, 256, 0, stream>>>(partial, splits, n, k, d, ldd, accumulate);
    SGB_CHECK_LAUNCH("k_reduce_splits");
    return SGB_OK;
}

// ---------------------------------------------------------------------------------------
// Thin weight gradient  D[n,k] = sum_m G[m,n] A[m,k]  with n <= 32, k <= 64 (the 4-16-32 / 32-16-3 ends of the SGCN
// stack): a pure HBM stream of two narrow matrices.  A CTA walks a contiguous row range in 32-row stages
// (cp.async, 3-deep); a warp takes 4 rows of a stage, every lane owns KPL columns of k and all NT rows of n
// (G values are shared-memory broadcasts), so the whole D tile lives in registers.  Fixed-order merge of the 8
// warps, one partial tile per CTA, then k_reduce_splits (deterministic).
// ---------------------------------------------------------------------------------------
constexpr int kThinRows = 32;
constexpr int kThinStages = 3;
constexpr int kThinThreads = 256;

__device__ __forceinline__ void cp_async_4(void* smem_dst, const void* gmem_src) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"((uint32_t)__cvta_generic_to_shared(smem_dst)), "l"(gmem_src) : "memory");
}
__device__ __forceinline__ void cp_async_16(void* smem_dst, const void* gmem_src) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((uint32_t)__cvta_generic_to_shared(smem_dst)), "l"(gmem_src) : "memory");
}

template <int NT, int KPL>
__global__ void __launch_bounds__(kThinThreads) k_gemm_tn_thin(const float* __restrict__ gmat, int64_t ldg, const float* __restrict__ amat,
                                                               int64_t lda, int64_t m, int n, int k, int64_t rows_per_cta,
                                                               float* __restrict__ partial) {
    constexpr int KW = 32 * KPL;
    __shared__ __align__(16) float Gs[kThinStages][kThinRows][NT];
    __shared__ __align__(16) float As[kThinStages][kThinRows][KW];
    __shared__ float red[NT][KW];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int64_t ms = (int64_t)blockIdx.x * rows_per_cta;
    const int64_t me = min64(m, ms + rows_per_cta);
    const int nstages = me > ms ? (int)((me - ms + kThinRows - 1) / kThinRows) : 0;
    const bool g_vec = (n % 4 == 0) && (ldg % 4 == 0) && ((reinterpret_cast<uintptr_t>(gmat) & 15) == 0);
    const bool a_vec = (k % 4 == 0) && (lda % 4 == 0) && ((reinterpret_cast<uintptr_t>(amat) & 15) == 0);
    // padding columns (>= n, >= k) are never written again: zero everything once
    for (int i = tid; i < kThinStages * kThinRows * NT; i += kThinThreads) (&Gs[0][0][0])[i] = 0.f;
    for (int i = tid; i < kThinStages * kThinRows * KW; i += kThinThreads) (&As[0][0][0])[i] = 0.f;
    __syncthreads();

    auto stage_load = [&](int st, int buf) {
        if (st < nstages) {
            const int64_t r0 = ms + (int64_t)st * kThinRows;
            const int rows = (int)min64(kThinRows, me - r0);
            if (g_vec) {
                const int per = n >> 2;
                for (int i = tid; i < kThinRows * per; i += kThinThreads) {
                    const int r = i / per, c = (i % per) * 4;
                    if (r < rows) cp_async_16(&Gs[buf][r][c], gmat + (r0 + r) * ldg + c);
                    else *reinterpret_cast<float4*>(&Gs[buf][r][c]) = make_float4(0.f, 0.f, 0.f, 0.f);
                }
            } else {
                for (int i = tid; i < kThinRows * n; i += kThinThreads) {
                    const int r = i / n, c = i % n;
                    if (r < rows) cp_async_4(&Gs[buf][r][c], gmat + (r0 + r) * ldg + c);
                    else Gs[buf][r][c] = 0.f;
                }
            }
            if (a_vec) {
                const int per = k >> 2;
                for (int i = tid; i < kThinRows * per; i += kThinThreads) {
                    const int r = i / per, c = (i % per) * 4;
                    if (r < rows) cp_async_16(&As[buf][r][c], amat + (r0 + r) * lda + c);
                    else *reinterpret_cast<float4*>(&As[buf][r][c]) = make_float4(0.f, 0.f, 0.f, 0.f);
                }
            } else {
                for (int i = tid; i < kThinRows * k; i += kThinThreads) {
                    const int r = i / k, c = i % k;
                    if (r < rows) cp_async_4(&As[buf][r][c], amat + (r0 + r) * lda + c);
                    else As[buf][r][c] = 0.f;
                }
            }
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
    };

    float acc[NT][KPL];
#pragma unroll
    for (int i = 0; i < NT; ++i)
#pragma unroll
        for (int j = 0; j < KPL; ++j) acc[i][j] = 0.f;

    stage_load(0, 0);
    stage_load(1, 1);
    for (int st = 0; st < nstages; ++st) {
        const int buf = st % kThinStages;
        stage_load(st + 2, (st + 2) % kThinStages);                 // buffer (st + 2) % 3 was consumed at iteration st - 1
        asm volatile("cp.async.wait_group 2;" ::: "memory");         // stage st has landed (two younger groups may be in flight)
        __syncthreads();
#pragma unroll
        for (int rr = 0; rr < kThinRows / 8; ++rr) {
            const int r = warp * (kThinRows / 8) + rr;
            float av[KPL];
#pragma unroll
            for (int j = 0; j < KPL; ++j) av[j] = As[buf][r][lane + 32 * j];
#pragma unroll
            for (int i = 0; i < NT; i += 4) {
                const float4 gq = *reinterpret_cast<const float4*>(&Gs[buf][r][i]);   // broadcast
                const float gg[4] = {gq.x, gq.y, gq.z, gq.w};
#pragma unroll
                for (int q = 0; q < 4; ++q)
#pragma unroll
                    for (int j = 0; j < KPL; ++j) acc[i + q][j] = fmaf(gg[q], av[j], acc[i + q][j]);
            }
        }
        __syncthreads();                                             // everyone is done with buf before it is refilled
    }
    asm volatile("cp.async.wait_group 0;" ::: "memory");
    // fixed-order merge of the warps
    for (int w = 0; w < kThinThreads / 32; ++w) {
        if (warp == w) {
#pragma unroll
            for (int i = 0; i < NT; ++i)
#pragma unroll
                for (int j = 0; j < KPL; ++j) red[i][lane + 32 * j] = (w == 0 ? 0.f : red[i][lane + 32 * j]) + acc[i][j];
        }
        __syncthreads();
    }
    float* out = partial + (int64_t)blockIdx.x * n * k;
    for (int i = tid; i < n * k; i += kThinThreads) out[i] = red[i / k][i % k];
}

static bool tn_thin_ok(int n, int k) { return n <= 32 && k <= 64; }
static int tn_thin_grid(int64_t m) {
    int64_t g = ceil_div(m > 0 ? m : 1, 8 * kThinRows);
    int64_t cap = (int64_t)num_sms() * 2;
    return (int)(g < cap ? g : cap);
}

static int tn_splits(int64_t m, int n, int k) {
    int64_t tiles = ceil_div(n, kTnTile) * ceil_div(k, kTnTile);
    int64_t want = ceil_div((int64_t)num_sms() * 4, tiles);
    int64_t maxs = ceil_div(m > 0 ? m : 1, 512);
    int64_t s = want < maxs ? want : maxs;
    return (int)(s < 1 ? 1 : s);
}

int gemm_tn_simt_launch(const float* g, int64_t ldg, const float* a, int64_t lda, float* d, int64_t ldd, int64_t m, int n, int k,
                        int accumulate, void* ws, size_t ws_bytes, cudaStream_t stream) {
    if (tn_thin_ok(n, k) && m > 0) {
        const int grid = tn_thin_grid(m);
        const size_t need = (size_t)grid * n * k * sizeof(float);
        if (ws_bytes < need || !ws) {
            set_error("sgb_gemm_tn: workspace %zu < required %zu", ws_bytes, need);
            return SGB_ENOSPC;
        }
        const int64_t rpc = ceil_div(ceil_div(m, grid), kThinRows) * kThinRows;
        const int nt = n <= 4 ? 4 : (n <= 16 ? 16 : 32), kpl = k <= 32 ? 1 : 2;
#define SGB_THIN_CASE(NTV, KPLV)                                                                                            \
        if (nt == NTV && kpl == KPLV) k_gemm_tn_thin<NTV, KPLV><<<grid, kThinThreads, 0, stream>>>(g, ldg, a, lda, m, n, k, rpc, (float*)ws);
        SGB_THIN_CASE(4, 1) SGB_THIN_CASE(4, 2) SGB_THIN_CASE(16, 1) SGB_THIN_CASE(16, 2) SGB_THIN_CASE(32, 1) SGB_THIN_CASE(32, 2)
#undef SGB_THIN_CASE
        SGB_CHECK_LAUNCH("k_gemm_tn_thin");
        return reduce_splits_launch((const float*)ws, grid, n, k, d, ldd, accumulate, stream);
    }
    int splits = tn_splits(m, n, k);
    size_t need = (size_t)splits * n * k * sizeof(float);
    if (ws_bytes < need || !ws) {
        set_error("sgb_gemm_tn: workspace %zu < required %zu", ws_bytes, need);
        return SGB_ENOSPC;
    }
    int64_t mps = ceil_div(ceil_div(m, splits), kTnStep) * kTnStep;
    dim3 grid((unsigned)(ceil_div(n, kTnTile) * ceil_div(k, kTnTile)), (unsigned)splits);
    k_gemm_tn_partial<<<grid, 256, 0, stream>>>(g, ldg, a, lda, m, n, k, mps, (float*)ws);
    SGB_CHECK_LAUNCH("k_gemm_tn_partial");
    return reduce_splits_launch((const float*)ws, splits, n, k, d, ldd, accumulate, stream);
}

size_t gemm_tn_simt_workspace(int64_t m, int n, int k) {
    size_t a = (size_t)tn_splits(m, n, k) * n * k * sizeof(float);
    size_t b = tn_thin_ok(n, k) ? (size_t)tn_thin_grid(m) * n * k * sizeof(float) : 0;
    return a > b ? a : b;
}

}  // namespace sgb
