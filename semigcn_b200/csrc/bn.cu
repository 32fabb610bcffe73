// BatchNorm1d (batch statistics over all vertices) + LeakyReLU, forward and backward, and the
// generic deterministic column reductions they share (also used for bias gradients).
//
// Replaces nn.BatchNorm1d(h) + nn.LeakyReLU() between the convs (util/networks.py:26-27,
// 43-44; util/meshnet.py:41-42) -- in the reference 2 reductions + 1 elementwise pass forward
// and the mirror image backward, each a separate ATen kernel.  Here the forward statistics
// normally arrive as per-CTA partials from the producing SpMM / GEMM epilogue; this file
// holds the fp64 finalisation, the stand-alone column-statistics kernel for foreign inputs,
// and the elementwise apply / backward kernels.  All HBM-bound streaming kernels, float4.
#include "common.cuh"

namespace sgb {

constexpr int kColThreads = 256;

enum ColOp { COL_STATS = 0, COL_BN_BWD = 1, COL_SUM = 2 };

struct ColArgs {
    const float* y; int64_t ldy;        // STATS: matrix; BN_BWD: Y (pre-BN conv output); SUM: matrix
    const float* dz; int64_t lddz;      // BN_BWD: upstream gradient
    int64_t m; int c;
    const float* scale; const float* shift; const float* mean; const float* invstd;
    float slope;
    float* partials;                    // STATS: [gridDim.x][3][c] (count, mean, M2); others: [gridDim.x][2][c] sums
    float* amax;                        // SUM only, optional: receives max |y| (atomicMax on the float bits; zeroed by the launcher)
};

// One thread owns VEC channels of one row-lane; rows are grid-strided; fixed-order smem
// reduction over the row-lanes of the CTA at the end.
template <int OP, int VEC>
__global__ void __launch_bounds__(kColThreads) k_col_reduce(const ColArgs a, int tpr /* threads per row, pow2 <= 256 */) {
    __shared__ float red[2][kColThreads * VEC];
    __shared__ float redn[kColThreads];
    float amx = 0.f;
    const int cl = threadIdx.x % tpr;
    const int rl = threadIdx.x / tpr;
    const int rows_per_pass = kColThreads / tpr;
    for (int c0 = 0; c0 < a.c; c0 += tpr * VEC) {
        const int ch = c0 + cl * VEC;
        const bool act = ch < a.c;
        double s1[VEC], s2[VEC];   // fp64 running sums: hundreds of rows per thread
        float sc[VEC], sh[VEC], mu[VEC], is[VEC];
#pragma unroll
        for (int q = 0; q < VEC; ++q) {
            s1[q] = 0.0; s2[q] = 0.0;
            sc[q] = 1.f; sh[q] = 0.f; mu[q] = 0.f; is[q] = 1.f;
            if (OP == COL_BN_BWD && act) {
                sc[q] = __ldg(a.scale + ch + q); sh[q] = __ldg(a.shift + ch + q);
                mu[q] = __ldg(a.mean + ch + q);  is[q] = __ldg(a.invstd + ch + q);
            }
        }
        if (act) {
            for (int64_t r = (int64_t)blockIdx.x * rows_per_pass + rl; r < a.m; r += (int64_t)gridDim.x * rows_per_pass) {
                float yv[VEC], dv[VEC];
                if (VEC == 4) {
                    float4 t = ldg4(a.y + r * a.ldy + ch);
                    yv[0] = t.x; yv[1] = t.y; yv[2] = t.z; yv[3] = t.w;
                    if (OP == COL_BN_BWD) {
                        float4 u = ldg4(a.dz + r * a.lddz + ch);
                        dv[0] = u.x; dv[1] = u.y; dv[2] = u.z; dv[3] = u.w;
                    }
                } else {
                    yv[0] = __ldg(a.y + r * a.ldy + ch);
                    if (OP == COL_BN_BWD) dv[0] = __ldg(a.dz + r * a.lddz + ch);
                }
#pragma unroll
                for (int q = 0; q < VEC; ++q) {
                    if (OP == COL_STATS) {
                        s1[q] += (double)yv[q];
                        s2[q] += (double)yv[q] * (double)yv[q];
                    } else if (OP == COL_SUM) {
                        s1[q] += (double)yv[q];
                        amx = fmaxf(amx, finite_abs(yv[q]));
                    } else {
                        const float ctr = yv[q] - mu[q];
                        const float pre = fmaf(ctr, sc[q], sh[q]);
                        const float da = pre > 0.f ? dv[q] : dv[q] * a.slope;
                        const float xh = ctr * is[q];
                        s1[q] += (double)da;
                        s2[q] += (double)da * (double)xh;
                    }
                }
            }
        }
        if (OP == COL_STATS) {
            // rows this thread visited: r = blockIdx.x*rpp + rl + i*gridDim.x*rpp < m
            const int64_t first = (int64_t)blockIdx.x * rows_per_pass + rl;
            const int64_t stride = (int64_t)gridDim.x * rows_per_pass;
            const double nrows = first < a.m ? (double)((a.m - 1 - first) / stride + 1) : 0.0;
#pragma unroll
            for (int q = 0; q < VEC; ++q) {
                const double mean = nrows > 0.0 ? s1[q] / nrows : 0.0;
                double m2 = nrows > 0.0 ? s2[q] - s1[q] * mean : 0.0;
                if (m2 < 0.0) m2 = 0.0;
                red[0][(rl * tpr + cl) * VEC + q] = (float)mean;
                red[1][(rl * tpr + cl) * VEC + q] = (float)m2;
            }
            if (cl == 0) redn[rl] = (float)nrows;
        } else {
#pragma unroll
            for (int q = 0; q < VEC; ++q) {
                red[0][(rl * tpr + cl) * VEC + q] = (float)s1[q];
                red[1][(rl * tpr + cl) * VEC + q] = (float)s2[q];
            }
        }
        __syncthreads();
        for (int i = threadIdx.x; i < tpr * VEC; i += kColThreads) {
            if (c0 + i < a.c) {
                if (OP == COL_STATS) {
                    Moments acc{0.f, 0.f, 0.f};
                    for (int r = 0; r < rows_per_pass; ++r)
                        acc = merge(acc, Moments{redn[r], red[0][r * tpr * VEC + i], red[1][r * tpr * VEC + i]});
                    a.partials[((int64_t)blockIdx.x * 3 + 0) * a.c + c0 + i] = acc.n;
                    a.partials[((int64_t)blockIdx.x * 3 + 1) * a.c + c0 + i] = acc.mean;
                    a.partials[((int64_t)blockIdx.x * 3 + 2) * a.c + c0 + i] = acc.m2;
                } else {
                    float t1 = 0.f, t2 = 0.f;
                    for (int r = 0; r < rows_per_pass; ++r) {
                        t1 += red[0][r * tpr * VEC + i];
                        t2 += red[1][r * tpr * VEC + i];
                    }
                    a.partials[((int64_t)blockIdx.x * 2 + 0) * a.c + c0 + i] = t1;
                    a.partials[((int64_t)blockIdx.x * 2 + 1) * a.c + c0 + i] = t2;
                }
            }
        }
        __syncthreads();
    }
    if (OP == COL_SUM && a.amax) publish_amax(amx, reinterpret_cast<uint32_t*>(redn), a.amax);
}

static int col_tpr(int c, int vec) {
    int lanes = (c + vec - 1) / vec;
    int p = 1;
    while (p < lanes && p < kColThreads) p <<= 1;
    return p;
}

static int col_rows_cfg(int64_t m, int c, int vec) {
    int tpr = col_tpr(c, vec);
    int rpp = kColThreads / tpr;
    int64_t need = ceil_div(m > 0 ? m : 1, (int64_t)rpp * 4);   // >= 4 rows per row-lane
    int64_t cap = (int64_t)num_sms() * 4;
    int64_t g = need < cap ? need : cap;
    return (int)(g < 1 ? 1 : g);
}

static int col_rows(int64_t m, int c) {
    int g4 = col_rows_cfg(m, c, 4), g1 = col_rows_cfg(m, c, 1);
    return g4 > g1 ? g4 : g1;
}

template <int OP>
static int col_launch(const ColArgs& a, bool vec_ok, cudaStream_t stream) {
    int vec = (a.c % 4 == 0 && vec_ok) ? 4 : 1;
    int grid = col_rows_cfg(a.m, a.c, vec);
    int rows = col_rows(a.m, a.c);
    const int planes = OP == COL_STATS ? 3 : 2;
    if (rows > grid)
        if (cudaMemsetAsync(a.partials + (size_t)grid * planes * a.c, 0, (size_t)(rows - grid) * planes * a.c * sizeof(float), stream) != cudaSuccess) {
            set_error("col_reduce: memset failed");
            return SGB_ECUDA;
        }
    int tpr = col_tpr(a.c, vec);
    if (vec == 4) k_col_reduce<OP, 4><<<grid, kColThreads, 0, stream>>>(a, tpr);
    else k_col_reduce<OP, 1><<<grid, kColThreads, 0, stream>>>(a, tpr);
    SGB_CHECK_LAUNCH("k_col_reduce");
    return SGB_OK;
}

static bool al16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

// ---- fp64 finalisation of [rows][2][c] partials: 32 channels x 32 row-lanes per CTA ----
struct FinArgs {
    const float* partials; int rows; int c; int64_t count;
    const float* gamma; const float* beta; float eps; float momentum;
    float* running_mean; float* running_var;
    float* mean; float* invstd; float* scale; float* shift;   // BN forward outputs
    float* sums; float* dgamma; float* dbeta; int accumulate; // BN backward / colsum outputs
    int kind;                                                  // 0 = BN fwd, 1 = BN bwd sums, 2 = column sum, 3 = merge moment rows -> sums[3][c]
};

__global__ void __launch_bounds__(1024) k_finalize(const FinArgs f) {
    __shared__ double r1[32][33], r2[32][33], r3[32][33];
    const int ch = blockIdx.x * 32 + threadIdx.x;
    double s1 = 0.0, s2 = 0.0, s3 = 0.0;
    if (ch < f.c) {
        if (f.kind == 0 || f.kind == 3) {
            // (count, mean, M2) rows.  Per row lane: division-free sums around a pivot (the mean of the lane's first
            // non-empty row), S0 = sum n, S1 = sum n (mean - p), S2 = sum M2 + n (mean - p)^2, in fp64 -- then one Chan
            // merge per lane below.  (A Chan merge per row costs two fp64 divisions per row and serialises them.)
            double p = 0.0;
            bool have = false;
            for (int r = threadIdx.y; r < f.rows; r += 32) {
                const double nb = (double)__ldg(f.partials + ((int64_t)r * 3 + 0) * f.c + ch);
                if (nb == 0.0) continue;
                const double mb = (double)__ldg(f.partials + ((int64_t)r * 3 + 1) * f.c + ch);
                const double qb = (double)__ldg(f.partials + ((int64_t)r * 3 + 2) * f.c + ch);
                if (!have) { p = mb; have = true; }
                const double d = mb - p;
                s1 += nb;
                s2 = fma(nb, d, s2);
                s3 += fma(nb * d, d, qb);
            }
            if (have) {           // -> (n, mean, M2) of this lane's rows
                const double dm = s2 / s1;
                s3 -= s2 * dm;
                if (s3 < 0.0) s3 = 0.0;
                s2 = p + dm;
            }
        } else {
            for (int r = threadIdx.y; r < f.rows; r += 32) {
                s1 += (double)__ldg(f.partials + ((int64_t)r * 2 + 0) * f.c + ch);
                s2 += (double)__ldg(f.partials + ((int64_t)r * 2 + 1) * f.c + ch);
            }
        }
    }
    r1[threadIdx.y][threadIdx.x] = s1;
    r2[threadIdx.y][threadIdx.x] = s2;
    r3[threadIdx.y][threadIdx.x] = s3;
    __syncthreads();
    if (threadIdx.y == 0 && ch < f.c) {
        if (f.kind == 0 || f.kind == 3) {
            double n = 0.0, mean = 0.0, m2 = 0.0;
            for (int r = 0; r < 32; ++r) {
                const double nb = r1[r][threadIdx.x];
                if (nb == 0.0) continue;
                const double nt = n + nb, d = r2[r][threadIdx.x] - mean;
                m2 += r3[r][threadIdx.x] + d * d * n * nb / nt;
                mean += d * nb / nt;
                n = nt;
            }
            if (f.kind == 3) {       // merged row only (SyncBN: one row per rank goes into the all-gather)
                f.sums[ch] = (float)n;
                f.sums[f.c + ch] = (float)mean;
                f.sums[2 * f.c + ch] = (float)m2;
                return;
            }
            double var = n > 0.0 ? m2 / n : 0.0;
            if (var < 0.0) var = 0.0;
            const double invstd = 1.0 / sqrt(var + (double)f.eps);
            const double g = f.gamma ? (double)f.gamma[ch] : 1.0;
            const double b = f.beta ? (double)f.beta[ch] : 0.0;
            f.mean[ch] = (float)mean;
            f.invstd[ch] = (float)invstd;
            f.scale[ch] = (float)(g * invstd);
            f.shift[ch] = (float)b;            // centred form: z = (y - mean) * scale + beta
            if (f.running_mean) {
                const double unb = n > 1.0 ? m2 / (n - 1.0) : var;
                f.running_mean[ch] = (float)((1.0 - f.momentum) * (double)f.running_mean[ch] + f.momentum * mean);
                f.running_var[ch] = (float)((1.0 - f.momentum) * (double)f.running_var[ch] + f.momentum * unb);
            }
        } else {
            double t1 = 0.0, t2 = 0.0;
            for (int r = 0; r < 32; ++r) { t1 += r1[r][threadIdx.x]; t2 += r2[r][threadIdx.x]; }
            if (f.kind == 1) {
                f.sums[ch] = (float)t1;
                f.sums[f.c + ch] = (float)t2;
                if (f.dbeta) f.dbeta[ch] = f.accumulate ? f.dbeta[ch] + (float)t1 : (float)t1;
                if (f.dgamma) f.dgamma[ch] = f.accumulate ? f.dgamma[ch] + (float)t2 : (float)t2;
            } else {
                f.sums[ch] = f.accumulate ? f.sums[ch] + (float)t1 : (float)t1;
            }
        }
    }
}

// ---- elementwise ------------------------------------------------------------------------
// A thread keeps its VEC channels for the whole kernel (per-channel parameters live in registers, loaded once)
// and walks rows with a grid stride: `tpr` threads cover one row chunk, 256 / tpr rows per CTA pass.
constexpr int kEwThreads = 256;

static int ew_tpr(int c, int vec) {
    int lanes = (c + vec - 1) / vec;
    int p = 1;
    while (p < lanes && p < kEwThreads) p <<= 1;
    return p;
}

template <int VEC>
__global__ void __launch_bounds__(kEwThreads) k_bn_act_apply(const float* __restrict__ y, int64_t ldy, int64_t m, int c, const float* __restrict__ mean,
                                                             const float* __restrict__ scale, const float* __restrict__ shift, float slope,
                                                             float* __restrict__ z, int64_t ldz, float* __restrict__ amax, int tpr) {
    __shared__ uint32_t s_amax[32];
    float amx = 0.f;
    const int cl = threadIdx.x % tpr, rl = threadIdx.x / tpr, rpp = kEwThreads / tpr;
    for (int c0 = 0; c0 < c; c0 += tpr * VEC) {
        const int ch = c0 + cl * VEC;
        if (ch >= c) continue;
        float mu[VEC], sc[VEC], sh[VEC];
#pragma unroll
        for (int q = 0; q < VEC; ++q) { mu[q] = __ldg(mean + ch + q); sc[q] = __ldg(scale + ch + q); sh[q] = __ldg(shift + ch + q); }
        for (int64_t r = (int64_t)blockIdx.x * rpp + rl; r < m; r += (int64_t)gridDim.x * rpp) {
            if (VEC == 4) {
                const float4 v = ldg4(y + r * ldy + ch);
                float4 o;
                o.x = bn_lrelu(v.x, mu[0], sc[0], sh[0], slope); o.y = bn_lrelu(v.y, mu[1], sc[1], sh[1], slope);
                o.z = bn_lrelu(v.z, mu[2], sc[2], sh[2], slope); o.w = bn_lrelu(v.w, mu[3], sc[3], sh[3], slope);
                st4(z + r * ldz + ch, o);
                amx = fmaxf(amx, fmaxf(fmaxf(finite_abs(o.x), finite_abs(o.y)), fmaxf(finite_abs(o.z), finite_abs(o.w))));
            } else {
                const float o = bn_lrelu(__ldg(y + r * ldy + ch), mu[0], sc[0], sh[0], slope);
                z[r * ldz + ch] = o;
                amx = fmaxf(amx, finite_abs(o));
            }
        }
    }
    if (amax) publish_amax(amx, s_amax, amax);
}

struct BwdArgs {
    const float* dz; int64_t lddz; const float* y; int64_t ldy; int64_t m; int c;
    const float* scale; const float* shift; const float* mean; const float* invstd; const float* sums;
    float slope; int training; float* dy; int64_t lddy; float* amax;
};

template <int VEC>
__global__ void __launch_bounds__(kEwThreads) k_bn_act_bwd_apply(const BwdArgs a, int tpr) {
    __shared__ uint32_t s_amax[32];
    float amx = 0.f;
    const float inv_m = 1.0f / (float)a.m;
    const int cl = threadIdx.x % tpr, rl = threadIdx.x / tpr, rpp = kEwThreads / tpr;
    for (int c0 = 0; c0 < a.c; c0 += tpr * VEC) {
        const int ch = c0 + cl * VEC;
        if (ch >= a.c) continue;
        float mu[VEC], sc[VEC], sh[VEC], is[VEC], sb[VEC], sg[VEC];
#pragma unroll
        for (int q = 0; q < VEC; ++q) {
            mu[q] = __ldg(a.mean + ch + q); sc[q] = __ldg(a.scale + ch + q); sh[q] = __ldg(a.shift + ch + q);
            is[q] = 0.f; sb[q] = 0.f; sg[q] = 0.f;
            if (a.training) {
                is[q] = __ldg(a.invstd + ch + q);
                sb[q] = __ldg(a.sums + ch + q) * inv_m;
                sg[q] = __ldg(a.sums + a.c + ch + q) * inv_m;
            }
        }
        for (int64_t r = (int64_t)blockIdx.x * rpp + rl; r < a.m; r += (int64_t)gridDim.x * rpp) {
            float yv[VEC], dv[VEC], out[VEC];
            if (VEC == 4) {
                float4 t = ldg4(a.y + r * a.ldy + ch), u = ldg4(a.dz + r * a.lddz + ch);
                yv[0] = t.x; yv[1] = t.y; yv[2] = t.z; yv[3] = t.w;
                dv[0] = u.x; dv[1] = u.y; dv[2] = u.z; dv[3] = u.w;
            } else {
                yv[0] = __ldg(a.y + r * a.ldy + ch);
                dv[0] = __ldg(a.dz + r * a.lddz + ch);
            }
#pragma unroll
            for (int q = 0; q < VEC; ++q) {
                const float ctr = yv[q] - mu[q];
                const float pre = fmaf(ctr, sc[q], sh[q]);
                const float da = pre > 0.f ? dv[q] : dv[q] * a.slope;
                if (a.training) {
                    const float xh = ctr * is[q];
                    out[q] = sc[q] * (da - sb[q] - xh * sg[q]);
                } else {
                    out[q] = sc[q] * da;
                }
                amx = fmaxf(amx, finite_abs(out[q]));
            }
            if (VEC == 4) st4(a.dy + r * a.lddy + ch, make_float4(out[0], out[1], out[2], out[3]));
            else a.dy[r * a.lddy + ch] = out[0];
        }
    }
    if (a.amax) publish_amax(amx, s_amax, a.amax);
}

static int ew_grid(int64_t m, int tpr) {
    const int rpp = kEwThreads / tpr;
    int64_t g = ceil_div(m > 0 ? m : 1, (int64_t)rpp * 4);   // >= 4 rows per row-lane
    int64_t cap = (int64_t)num_sms() * 8;
    g = g < cap ? g : cap;
    return (int)(g < 1 ? 1 : g);
}

}  // namespace sgb

using namespace sgb;

extern "C" int sgb_col_stat_rows(int64_t m, int c) {
    if (m < 0 || c <= 0) return 0;
    return col_rows(m, c);
}

extern "C" int sgb_col_stats(const float* y, int64_t ldy, int64_t m, int c, float* partials, void* stream) {
    SGB_CHECK_ARG(y && partials && m >= 0 && c > 0 && ldy >= c, "sgb_col_stats: bad argument");
    ColArgs a{};
    a.y = y; a.ldy = ldy; a.m = m; a.c = c; a.partials = partials;
    return col_launch<COL_STATS>(a, al16(y) && ldy % 4 == 0, (cudaStream_t)stream);
}

extern "C" int sgb_bn_finalize(const float* partials, int rows, int c, int64_t count, const float* gamma, const float* beta,
                               float eps, float momentum, float* running_mean, float* running_var, float* mean, float* invstd,
                               float* scale, float* shift, void* stream) {
    SGB_CHECK_ARG(partials && rows > 0 && c > 0 && count > 0 && mean && invstd && scale && shift, "sgb_bn_finalize: bad argument");
    SGB_CHECK_ARG((running_mean == nullptr) == (running_var == nullptr), "sgb_bn_finalize: running stats must come together");
    FinArgs f{};
    f.partials = partials; f.rows = rows; f.c = c; f.count = count; f.gamma = gamma; f.beta = beta; f.eps = eps;
    f.momentum = momentum; f.running_mean = running_mean; f.running_var = running_var;
    f.mean = mean; f.invstd = invstd; f.scale = scale; f.shift = shift; f.kind = 0;
    k_finalize<<<(c + 31) / 32, dim3(32, 32), 0, (cudaStream_t)stream>>>(f);
    SGB_CHECK_LAUNCH("k_finalize");
    return SGB_OK;
}

extern "C" int sgb_moments_merge(const float* partials, int rows, int c, float* merged, void* stream) {
    SGB_CHECK_ARG(partials && rows > 0 && c > 0 && merged, "sgb_moments_merge: bad argument");
    FinArgs f{};
    f.partials = partials; f.rows = rows; f.c = c; f.sums = merged; f.kind = 3;
    k_finalize<<<(c + 31) / 32, dim3(32, 32), 0, (cudaStream_t)stream>>>(f);
    SGB_CHECK_LAUNCH("k_finalize");
    return SGB_OK;
}

extern "C" int sgb_bn_act_apply(const float* y, int64_t ldy, int64_t m, int c, const float* mean, const float* scale,
                                const float* shift, float slope, float* z, int64_t ldz, float* amax_out, void* stream) {
    SGB_CHECK_ARG(y && z && mean && scale && shift && m >= 0 && c > 0 && ldy >= c && ldz >= c, "sgb_bn_act_apply: bad argument");
    if (m == 0) return SGB_OK;
    bool vec = c % 4 == 0 && al16(y) && al16(z) && al16(mean) && al16(scale) && al16(shift) && ldy % 4 == 0 && ldz % 4 == 0;
    const int tpr = ew_tpr(c, vec ? 4 : 1);
    if (vec) k_bn_act_apply<4><<<ew_grid(m, tpr), kEwThreads, 0, (cudaStream_t)stream>>>(y, ldy, m, c, mean, scale, shift, slope, z, ldz, amax_out, tpr);
    else k_bn_act_apply<1><<<ew_grid(m, tpr), kEwThreads, 0, (cudaStream_t)stream>>>(y, ldy, m, c, mean, scale, shift, slope, z, ldz, amax_out, tpr);
    SGB_CHECK_LAUNCH("k_bn_act_apply");
    return SGB_OK;
}

extern "C" int sgb_bn_act_bwd_reduce(const float* dz, int64_t lddz, const float* y, int64_t ldy, int64_t m, int c, const float* scale,
                                     const float* shift, const float* mean, const float* invstd, float slope, float* partials,
                                     void* stream) {
    SGB_CHECK_ARG(dz && y && scale && shift && mean && invstd && partials && m >= 0 && c > 0 && ldy >= c && lddz >= c,
                  "sgb_bn_act_bwd_reduce: bad argument");
    ColArgs a{};
    a.y = y; a.ldy = ldy; a.dz = dz; a.lddz = lddz; a.m = m; a.c = c;
    a.scale = scale; a.shift = shift; a.mean = mean; a.invstd = invstd; a.slope = slope; a.partials = partials;
    return col_launch<COL_BN_BWD>(a, al16(y) && al16(dz) && ldy % 4 == 0 && lddz % 4 == 0, (cudaStream_t)stream);
}

extern "C" int sgb_bn_bwd_finalize(const float* partials, int rows, int c, float* sums, float* dgamma, float* dbeta, int accumulate,
                                   void* stream) {
    SGB_CHECK_ARG(partials && rows > 0 && c > 0 && sums, "sgb_bn_bwd_finalize: bad argument");
    FinArgs f{};
    f.partials = partials; f.rows = rows; f.c = c; f.sums = sums; f.dgamma = dgamma; f.dbeta = dbeta; f.accumulate = accumulate;
    f.kind = 1;
    k_finalize<<<(c + 31) / 32, dim3(32, 32), 0, (cudaStream_t)stream>>>(f);
    SGB_CHECK_LAUNCH("k_finalize");
    return SGB_OK;
}

extern "C" int sgb_bn_act_bwd_apply(const float* dz, int64_t lddz, const float* y, int64_t ldy, int64_t m, int c, const float* scale,
                                    const float* shift, const float* mean, const float* invstd, const float* sums, float slope,
                                    int training, float* dy, int64_t lddy, float* amax_out, void* stream) {
    SGB_CHECK_ARG(dz && y && dy && scale && shift && m >= 0 && c > 0 && ldy >= c && lddz >= c && lddy >= c,
                  "sgb_bn_act_bwd_apply: bad argument");
    SGB_CHECK_ARG(mean && (!training || (invstd && sums)), "sgb_bn_act_bwd_apply: mean required; training mode also needs invstd/sums");
    if (m == 0) return SGB_OK;
    BwdArgs a{dz, lddz, y, ldy, m, c, scale, shift, mean, invstd, sums, slope, training, dy, lddy, amax_out};
    bool vec = c % 4 == 0 && al16(y) && al16(dz) && al16(dy) && ldy % 4 == 0 && lddz % 4 == 0 && lddy % 4 == 0;
    const int tpr = ew_tpr(c, vec ? 4 : 1);
    if (vec) k_bn_act_bwd_apply<4><<<ew_grid(m, tpr), kEwThreads, 0, (cudaStream_t)stream>>>(a, tpr);
    else k_bn_act_bwd_apply<1><<<ew_grid(m, tpr), kEwThreads, 0, (cudaStream_t)stream>>>(a, tpr);
    SGB_CHECK_LAUNCH("k_bn_act_bwd_apply");
    return SGB_OK;
}

extern "C" size_t sgb_colsum_workspace_bytes(int64_t m, int n) {
    if (m < 0 || n <= 0) return 0;
    return (size_t)col_rows(m, n) * 2 * n * sizeof(float);
}

extern "C" int sgb_colsum(const float* g, int64_t ldg, int64_t m, int n, float* out, int accumulate, float* amax_out, void* workspace,
                          size_t workspace_bytes, void* stream) {
    SGB_CHECK_ARG(g && out && m >= 0 && n > 0 && ldg >= n, "sgb_colsum: bad argument");
    size_t need = sgb_colsum_workspace_bytes(m, n);
    if (!workspace || workspace_bytes < need) {
        set_error("sgb_colsum: workspace %zu < required %zu", workspace_bytes, need);
        return SGB_ENOSPC;
    }
    ColArgs a{};
    a.y = g; a.ldy = ldg; a.m = m; a.c = n; a.partials = (float*)workspace; a.amax = amax_out;
    if (amax_out) SGB_CUDA(cudaMemsetAsync(amax_out, 0, sizeof(float), (cudaStream_t)stream));
    int rc = col_launch<COL_SUM>(a, al16(g) && ldg % 4 == 0, (cudaStream_t)stream);
    if (rc != SGB_OK) return rc;
    FinArgs f{};
    f.partials = (const float*)workspace; f.rows = col_rows(m, n); f.c = n; f.sums = out; f.accumulate = accumulate; f.kind = 2;
    k_finalize<<<(n + 31) / 32, dim3(32, 32), 0, (cudaStream_t)stream>>>(f);
    SGB_CHECK_LAUNCH("k_finalize");
    return SGB_OK;
}
