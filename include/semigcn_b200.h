/*
 * semigcn_b200 -- C-ABI of the B200 (sm_100a) graph-convolution hot path of SeMIGCN.
 *
 * Drop-in boundary (SURVEY.md §8(b)): the reference reaches this arithmetic through three
 * torch_geometric symbols -- `from torch_geometric.nn import GCNConv, ChebConv, Sequential`
 * (reference util/networks.py:4, util/meshnet.py:6).  The Python host layer
 * (semigcn_b200/nn.py) re-exposes those classes; every FLOP and byte they move goes through
 * the entry points below, loaded with ctypes (INTEGRATION.md).
 *
 * Conventions
 *   - plain pointers + sizes; every pointer is a DEVICE pointer unless the name ends in
 *     `_host`; the caller owns every buffer, including workspaces (the library allocates
 *     nothing);
 *   - all work is enqueued on `stream` (a cudaStream_t passed as void*); no internal
 *     synchronisation -> CUDA-graph capturable;
 *   - return 0 on success, a negative SGB_E* code otherwise; never throws, never exits;
 *     `sgb_last_error()` returns a thread-local message for the last failing call;
 *   - all matrices are dense row-major fp32 with an explicit leading dimension (elements);
 *   - deterministic: no floating-point atomics anywhere (integer atomics only in the
 *     one-off graph builder, whose output is order-independent).
 */
#ifndef SEMIGCN_B200_H
#define SEMIGCN_B200_H

#include <stddef.h>
#include <stdint.h>

#if defined(__GNUC__)
#define SGB_API __attribute__((visibility("default")))
#else
#define SGB_API
#endif

#ifdef __cplusplus
extern "C" {
#endif

#define SGB_VERSION 100

#define SGB_OK 0
#define SGB_EINVAL (-1)   /* bad argument (null pointer, negative size, bad enum, alignment) */
#define SGB_ECUDA (-2)    /* a CUDA runtime call / kernel launch failed                       */
#define SGB_ENOSPC (-3)   /* caller-provided workspace too small                              */
#define SGB_ENOTSUP (-4)  /* shape not supported by this entry point                          */

/* normalisation modes (which PyG operator the sparse matrix stands for) */
#define SGB_MODE_GCN 0  /* D~^-1/2 (A+I) D~^-1/2, degree over targets (+1 self loop); replaces
                           torch_geometric gcn_norm as called by GCNConv (util/networks.py:25) */
#define SGB_MODE_CHEB 1 /* -D^-1/2 A D^-1/2 with the explicit (+x_i, -x_i) loop pair of
                           ChebConv.__norm__ (util/networks.py:42), degree over sources        */
#define SGB_MODE_ADJ 2  /* plain adjacency sum (weights 1, no loops): mesh_laplacian_loss
                           (util/loss.py:60-76), mask dilation (util/datamaker.py:124-127)    */

/* one CSR entry as the aggregation kernel consumes it: neighbour id + its normalised weight
 * (GCN: dis[src]*dis[dst]; CHEB: -dis[src]*dis[dst]; ADJ: 1), 8 bytes, streamed once per SpMM */
typedef struct sgb_edge {
    int32_t col;
    float w;
} sgb_edge_t;

SGB_API int sgb_version(void);
SGB_API const char* sgb_last_error(void);
/* number of SMs of the current device (used by callers to size stat-partial buffers) */
SGB_API int sgb_num_sms(void);

/* ------------------------------------------------------------------------------------ *
 * 1. Graph builder: edge_index[2, nnz] (int64, row 0 = sources, row 1 = targets)
 *    -> CSR grouped by target (transpose = 0; forward aggregation) or by source
 *    (transpose = 1; backward aggregation), STABLE in edge order inside each row, self
 *    loops removed (GCN re-adds exactly one per vertex implicitly), plus dis[i] =
 *    1/sqrt(deg_i) computed as IEEE div(1, sqrt(deg)) -- bit-exact against torch-CPU
 *    `deg.pow_(-0.5)` (SURVEY.md A.5); deg = 0 -> 0.
 *    Replaces: gcn_norm / get_laplacian / add_remaining_self_loops executed inside every
 *    GCNConv / ChebConv forward (SURVEY.md §8(a3)); input contract util/mesh.py:229-230.
 *    edges[slot] = (colidx[slot], weight) with weight = fl(dis[src] * dis[dst]) (negated for
 *    CHEB, 1 for ADJ) -- the per-edge `norm` of gcn_norm / ChebConv.__norm__, bit-exact; this
 *    packed stream is what sgb_spmm reads (one 8-byte load per neighbour).
 *    perm[e] = slot of edge e in colidx, or -1 for a dropped self loop.
 *    err_flag (device int32[1], zero-initialised by the call): 1 if an index was outside
 *    [0, n).
 * ------------------------------------------------------------------------------------ */
/* out[0..1] (device uint64[2], zeroed by the call) = 128-bit content fingerprint of an int64 array, one streaming pass.
 * The host layer keys its CSR cache on it when the caller passes a fresh device copy of the same edge_index every
 * forward (the reference does: `data.edge_index.to(self.device)`, util/networks.py:65), so the copy costs one hash pass
 * instead of a CSR rebuild. */
SGB_API int sgb_fingerprint(const int64_t* values, int64_t count, uint64_t* out /* [2] */, void* stream);
SGB_API size_t sgb_graph_build_workspace_bytes(int64_t nnz, int64_t n);
SGB_API int sgb_graph_build(const int64_t* edge_index, int64_t nnz, int64_t n, int mode, int transpose,
                    int32_t* rowptr /* [n+1] */, int32_t* colidx /* [nnz] */, sgb_edge_t* edges /* [nnz] or NULL */,
                    float* dis /* [n] */, int32_t* perm /* [nnz] or NULL */, int32_t* err_flag /* [1] */,
                    void* workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------ *
 * 2. SpMM: Y = alpha * (S f(X)) + beta * ADDEND + bias, row-parallel gather, one
 *    sub-warp per vertex, 128-bit loads, atomic-free; S is defined by (rowptr, edges,
 *    dis, mode); accumulation order per row = CSR order then the self-loop term(s), with
 *    separately rounded multiply and add -- the op order of PyG's message/aggregate
 *    (SURVEY.md A.1 step 3, A.6), so the result is bit-identical to the CPU path.
 *    f (optional, in_scale != NULL): per-channel BatchNorm + LeakyReLU applied to every
 *    gathered element in CENTRED form, f(x) = lrelu((x - in_mean[c]) * in_scale[c] +
 *    in_shift[c], slope) with in_scale = gamma*invstd, in_shift = beta: the fused
 *    BatchNorm1d + LeakyReLU of the previous block (util/networks.py:26-27).  (The uncentred
 *    x*scale + shift' form cancels catastrophically on near-constant channels.)
 *    stat_partials (optional): per-CTA column moments of Y as (count, mean, M2) triples,
 *    laid out [sgb_spmm_stat_rows(n, c)][3][c]; feeds sgb_bn_finalize (Chan merge).
 *    Replaces MessagePassing.propagate (index_select -> mul -> scatter_add), fwd and,
 *    called with the transpose CSR, bwd.
 *    amax_out (optional, device float zeroed by the caller) receives max |Y| over the finite entries
 *    (atomicMax on the float bits): the scale of the fp16-split GEMM engine that consumes Y (sgb_gemm a_amax), for free.
 *    SGB_MODE_ADJ takes any CSR whose packed stream carries its own weights -- also a RECTANGULAR one
 *    (n = rows of Y; column ids index rows of X, which may have any row count > max column id; dis is
 *    not read): this is how MeshPool / MeshUnpool (reference util/meshnet.py:9-27, torch.sparse.mm of
 *    the pool / unpool "hash" matrices) run, forward on the by-row CSR, backward on the by-column one.
 * ------------------------------------------------------------------------------------ */
SGB_API int sgb_spmm_stat_rows(int64_t n, int c);
SGB_API int sgb_spmm(const int32_t* rowptr, const sgb_edge_t* edges, const float* dis, int mode,
             const float* x, int64_t ldx, int64_t n, int c,
             const float* in_mean, const float* in_scale, const float* in_shift, float slope,
             float alpha, const float* addend, int64_t ld_addend, float beta,
             const float* bias, float* y, int64_t ldy, float* stat_partials, float* amax_out, void* stream);

/* Vertex-partitioned variant (one mesh over several GPUs, SURVEY.md §8(e)): rows [0, n) are the
 * vertices this rank owns; neighbour ids >= n_split address the halo block x_ghost (rows received
 * from the owning ranks, sgb_gather_rows + all-to-all).  x_ghost = NULL is sgb_spmm.          */
SGB_API int sgb_spmm_halo(const int32_t* rowptr, const sgb_edge_t* edges, const float* dis, int mode,
                  const float* x, int64_t ldx, int64_t n, int c, const float* x_ghost, int64_t ld_ghost, int64_t n_split,
                  const float* in_mean, const float* in_scale, const float* in_shift, float slope,
                  float alpha, const float* addend, int64_t ld_addend, float beta,
                  const float* bias, float* y, int64_t ldy, float* stat_partials, float* amax_out, void* stream);
/* Rows [row_begin, row_begin + n) of the same operator (all pointers are the whole-matrix ones; y / addend / x are addressed
 * by absolute row).  With the owned vertices numbered interior-first, the rows without ghost columns run as one launch
 * (x_ghost = NULL) WHILE the halo all-to-all of the boundary rows is in flight, the boundary rows as a second launch after
 * it: the exchange hides behind the interior aggregation.  stat_partials: sgb_spmm_stat_rows(n, c) rows PER LAUNCH. */
SGB_API int sgb_spmm_range(const int32_t* rowptr, const sgb_edge_t* edges, const float* dis, int mode,
                   const float* x, int64_t ldx, int64_t row_begin, int64_t n, int c, const float* x_ghost, int64_t ld_ghost, int64_t n_split,
                   const float* in_mean, const float* in_scale, const float* in_shift, float slope,
                   float alpha, const float* addend, int64_t ld_addend, float beta,
                   const float* bias, float* y, int64_t ldy, float* stat_partials, float* amax_out, void* stream);
/* out[k, :] = x[idx[k], :] (halo pack; also MeshUnpool-style row gathers), c floats per row */
SGB_API int sgb_gather_rows(const float* x, int64_t ldx, const int32_t* idx, int64_t count, int c, float* out, int64_t ldo, void* stream);

/* ------------------------------------------------------------------------------------ *
 * 3. Dense feature transform (the per-layer `lin` of GCNConv / `lins[k]` of ChebConv,
 *    nn.Linear of util/networks.py:35,52,58-61) and its two gradients.
 *    sgb_gemm:       C[m,n] (+)= f(A)[m,k] * op(B) + bias,  op(B) = B^T for transb=1
 *                    (B is [n,k], i.e. a torch Linear weight) or B for transb=0 (B is [k,n]).
 *                    f = optional per-k-channel centred BatchNorm + LeakyReLU on A (as in sgb_spmm).
 *                    stat_partials: [sgb_gemm_stat_rows(m)][3][n] column (count, mean, M2) of C.
 *    sgb_gemm_tn:    D[n,k] (+)= G[m,n]^T * A[m,k]   (weight gradient; split over m with a
 *                    fixed-order two-stage reduction -> deterministic).
 *    sgb_colsum:     out[n] (+)= sum_m G[m,n]        (bias gradient).
 *    stat_partials rows: every engine writes per-CTA (not per-tile) moments, at most
 *    sgb_gemm_stat_rows(m) = 4 * min(ceil(m/128), #SMs) rows, and zero-fills the rows it does not use
 *    (count 0 rows drop out of the merge) -- the finalisation cost no longer grows with m.
 *    `engine`: 0 = auto, 1 = fp32 CUDA-core tiles, 2 = tcgen05 3xTF32 tensor-core tiles
 *    (error-compensated: hi*hi + lo*hi + hi*lo, fp32 accumulate in TMEM).  The tensor-core
 *    engine stages the split / pre-tiled weights in `workspace` (sgb_gemm_workspace_bytes).
 *    3 = tcgen05 2xFP16-split tiles: operands scaled by a per-tensor power of two and split into
 *    fp16 hi + lo (22 significant bits), the same three products at the fp16 rate; bound by the HBM
 *    stream of the activation operand.  `a_amax` / `g_amax` (optional device scalars, max |A| /
 *    max |G| over the FINITE entries, e.g. from the amax_out of the kernel that produced the
 *    operand) save the engine its own reduction pass over that operand; NULL = computed internally.
 *    Every amax_out of this library and the internal reduction skip inf and NaN, so an operand with
 *    a non-finite entry keeps its scale: inf stays inf, NaN stays NaN, and the other rows of the
 *    result stay finite.  A supplied maximum smaller than the true one overflows the fp16 split;
 *    a larger one costs precision.  Accuracy is norm-relative
 *    (elements > 2^23 below the tensor maximum lose relative precision).  engine 0 picks 3 for
 *    real contractions (n >= 32, k >= 16), 1 for thin ones.  On large operands (m >= 32 768) engine 3
 *    runs as clusters of two CTAs (tcgen05 cta_group::2, UMMA M = 256: each CTA stages its own 128
 *    rows of the activation operand and half of the other operand; sgb_gemm when n % 32 == 0,
 *    sgb_gemm_tn as `engine` 4 when n % 256 == 0, k % 32 == 0 and k <= 256 or k % 256 == 0 -- engine
 *    4 may also be requested explicitly from m >= 4096, SGB_ENOTSUP otherwise).  The results of the
 *    pair and single-CTA variants agree to fp32 rounding of the accumulation order, both are
 *    deterministic run to run.
 * ------------------------------------------------------------------------------------ */
SGB_API int sgb_gemm_stat_rows(int64_t m);
SGB_API size_t sgb_gemm_workspace_bytes(int64_t m, int n, int k, int engine);
SGB_API int sgb_gemm(int transb, const float* a, int64_t lda, const float* b, int64_t ldb,
             float* c, int64_t ldc, int64_t m, int n, int k,
             const float* a_mean, const float* a_scale, const float* a_shift, float slope,
             const float* bias, int accumulate, float* stat_partials, const float* a_amax,
             void* workspace, size_t workspace_bytes, int engine, void* stream);
SGB_API size_t sgb_gemm_tn_workspace_bytes(int64_t m, int n, int k);
SGB_API int sgb_gemm_tn(const float* g, int64_t ldg, const float* a, int64_t lda, float* d, int64_t ldd,
                int64_t m, int n, int k, int accumulate, const float* g_amax, const float* a_amax,
                void* workspace, size_t workspace_bytes, int engine, void* stream);
SGB_API size_t sgb_colsum_workspace_bytes(int64_t m, int n);
SGB_API int sgb_colsum(const float* g, int64_t ldg, int64_t m, int n, float* out, int accumulate,
               float* amax_out /* optional: max |G| from the same pass (feeds g_amax / a_amax of the GEMMs that read G next) */,
               void* workspace, size_t workspace_bytes, void* stream);
/* amax_out[0] = max |X| over an [m, c] matrix (one streaming pass; c % 4 == 0, 16-byte aligned rows): the per-tensor
 * scale of the fp16-split engine for an operand that none of our kernels produced (e.g. the upstream gradient of a bare
 * GCNConv), computed ONCE and shared by every GEMM that reads the operand. */
SGB_API int sgb_amax(const float* x, int64_t ldx, int64_t m, int c, float* amax_out, void* stream);

/* ------------------------------------------------------------------------------------ *
 * 4. BatchNorm1d (batch statistics over all vertices) + LeakyReLU, forward and backward.
 *    Replaces nn.BatchNorm1d + nn.LeakyReLU between convs (util/networks.py:26-27,43-44).
 *    sgb_col_stats      : partials[rows][3][c] of (count, mean, M2) for a matrix that was
 *                         not produced by one of our kernels.
 *    sgb_bn_finalize    : fp64 Chan merge of the partials -> mean, invstd (biased var, eps),
 *                         scale = gamma*invstd, shift = beta; updates running stats
 *                         (momentum, unbiased var) when running_mean != NULL.
 *    sgb_bn_act_apply   : Z = lrelu((Y - mean)*scale + shift, slope).
 *    sgb_bn_act_bwd_reduce / _apply : dY from dZ (two-pass: per-channel sums, then apply).
 * ------------------------------------------------------------------------------------ */
SGB_API int sgb_col_stat_rows(int64_t m, int c);
SGB_API int sgb_col_stats(const float* y, int64_t ldy, int64_t m, int c, float* partials, void* stream);
SGB_API int sgb_bn_finalize(const float* partials, int rows, int c, int64_t count,
                    const float* gamma, const float* beta, float eps, float momentum,
                    float* running_mean, float* running_var,
                    float* mean, float* invstd, float* scale, float* shift, void* stream);
/* merged[3][c] = Chan merge (fp64) of partials[rows][3][c]: ONE (count, mean, M2) row.  Vertex-partitioned SyncBN
 * all-gathers this row per rank (a rank-invariant 12*c bytes) instead of the raw per-CTA rows. */
SGB_API int sgb_moments_merge(const float* partials, int rows, int c, float* merged /* [3][c] */, void* stream);
SGB_API int sgb_bn_act_apply(const float* y, int64_t ldy, int64_t m, int c, const float* mean, const float* scale,
                     const float* shift, float slope, float* z, int64_t ldz, float* amax_out /* optional: max |Z| */, void* stream);
/* partials[rows][2][c]: (sum dA, sum dA*xhat) with dA = dZ * lrelu'((Y-mean)*scale+shift) */
SGB_API int sgb_bn_act_bwd_reduce(const float* dz, int64_t lddz, const float* y, int64_t ldy, int64_t m, int c,
                          const float* scale, const float* shift, const float* mean, const float* invstd,
                          float slope, float* partials, void* stream);
/* sums[2][c] = fp64-reduced partials (as float); dY = scale * (dA - sum0/m - xhat*sum1/m);
 * also emits dgamma = sums[1], dbeta = sums[0] (accumulating when accumulate != 0).      */
SGB_API int sgb_bn_bwd_finalize(const float* partials, int rows, int c, float* sums, float* dgamma,
                        float* dbeta, int accumulate, void* stream);
SGB_API int sgb_bn_act_bwd_apply(const float* dz, int64_t lddz, const float* y, int64_t ldy, int64_t m, int c,
                         const float* scale, const float* shift, const float* mean, const float* invstd,
                         const float* sums, float slope, int training, float* dy, int64_t lddy,
                         float* amax_out /* optional: max |dY| */, void* stream);

/* ------------------------------------------------------------------------------------ *
 * 5. Step-path mesh losses as fused gather/reduce kernels (fp64 accumulation, deterministic).
 *    Replaces Models.compute_fn (util/models.py:121-126), Loss.mask_pos_rec_loss "rmse"
 *    (util/loss.py:14-34), Loss.mask_norm_rec_loss "l1mae" (util/loss.py:78-107) as called
 *    per step by sgcn.py:130-132 / mgcn.py:137-143, and Loss.mesh_laplacian_loss "rmse"
 *    (util/loss.py:60-76).
 *    sgb_incidence_build: faces[nf,3] (int64) -> vertex -> face-corner CSR (entries 3*f + corner,
 *                         ascending inside a row); the backward pass gathers over it (no atomics).
 *    sgb_step_loss_fwd  : out[0] = loss_p = sqrt(sum_{vmask} |target_pos - pos|^2 / |vmask| + 1e-6)
 *                         out[1] = loss_n = sum_{fmask} |n_f(pos) - target_fn_f|_1 / |fmask|
 *                         out[2], out[3] = |vmask|, |fmask|.  target_* are fp64 (target_f64 = 1, the
 *                         sgcn.py case) or fp32; NULL target_pos / faces skip that term; NULL masks =
 *                         all; fn_out (optional, [nf,3]) receives the unit face normals (compute_fn).
 *                         partials: double[sgb_loss_partial_rows()][4].
 *    sgb_step_loss_bwd  : dpos[n,3] = grads[0] * dloss_p/dpos + grads[1] * dloss_n/dpos.
 *    sgb_lap_loss_fwd   : diff[n,3] = pos - (Adj pos)/deg over an SGB_MODE_ADJ (or any) CSR;
 *                         out[0] = sqrt(mean_v |diff_v|^2 + 1e-12).   _bwd: dpos from diff.
 * ------------------------------------------------------------------------------------ */
SGB_API int sgb_loss_partial_rows(void);
SGB_API size_t sgb_incidence_build_workspace_bytes(int64_t nf, int64_t n);
SGB_API int sgb_incidence_build(const int64_t* faces, int64_t nf, int64_t n, int32_t* rowptr /* [n+1] */, int32_t* inc /* [3 nf] */,
                        int32_t* err_flag, void* workspace, size_t workspace_bytes, void* stream);
SGB_API int sgb_step_loss_fwd(const float* pos, int64_t ldp, int64_t n, const void* target_pos, int target_f64, const uint8_t* vmask,
                      const int64_t* faces, int64_t nf, const void* target_fn, const uint8_t* fmask, float* fn_out,
                      double* partials, double* out /* [4] */, void* stream);
SGB_API int sgb_step_loss_bwd(const float* pos, int64_t ldp, int64_t n, const void* target_pos, int target_f64, const uint8_t* vmask,
                      const int64_t* faces, int64_t nf, const void* target_fn, const uint8_t* fmask,
                      const int32_t* inc_rowptr, const int32_t* inc, const double* out, const double* grads /* [2] */,
                      float* dpos, int64_t lddpos, void* stream);
SGB_API int sgb_lap_loss_fwd(const float* pos, int64_t ldp, int64_t n, const int32_t* rowptr, const sgb_edge_t* edges, float* diff /* [n,3] */,
                     double* partials, double* out /* [1] */, void* stream);
SGB_API int sgb_lap_loss_bwd(const float* diff, int64_t n, const int32_t* rowptr, const int32_t* rowptr_t, const sgb_edge_t* edges_t,
                     const double* out, const double* grad /* [1] */, float* dpos, int64_t lddpos, void* stream);

/* ------------------------------------------------------------------------------------ *
 * 6. Bilateral-normal-filter regulariser (the `-CAD` term of the step, sgcn.py:133-136):
 *    replaces Loss.fn_bnf_detach_loss(pos, fn, mesh, ltype, loop) (util/loss.py:197-253).
 *    pos [n,3] (treated as detached), fn [nf,3] = compute_fn(pos) (the differentiable input),
 *    f2f [nf,3] int32 = the faces across the three sides, -1 where a side is on a boundary
 *    (Mesh.f2f, util/mesh.py:215-227).  `loop` detached filter iterations with weights
 *    exp(-|dc|^2 / 2 sigma_c^2) exp(-|dn|^2 / 2 sigma_s^2) area (sigma_s = 0.3, sigma_c = mean
 *    centroid distance), then the distance of fn to the filtered normals.
 *    ltype: 0 "mae", 1 "l1mae" (the default), 2 "rmse", 3 "l1rmse".
 *    work: float[sgb_bnf_work_floats(nf)], partials: double[sgb_bnf_partial_rows()];
 *    new_fn [nf,3] receives the filtered normals; out[0] = loss, out[1] = internal (for _bwd).
 *    _bwd: dfn [nf,3] = grad[0] * dloss/dfn (the filtered normals are detached, so this is the
 *    whole gradient).  fp32 arithmetic like the reference, fp64 sums, deterministic.
 * ------------------------------------------------------------------------------------ */
SGB_API size_t sgb_bnf_work_floats(int64_t nf);
SGB_API int sgb_bnf_partial_rows(void);
SGB_API int sgb_bnf_loss_fwd(const float* pos, int64_t ldp, int64_t n, const int64_t* faces, const int32_t* f2f, int64_t nf,
                     const float* fn, int loop, int ltype, float* work, double* partials, float* new_fn, double* out /* [2] */,
                     void* stream);
SGB_API int sgb_bnf_loss_bwd(const float* fn, const float* new_fn, int64_t nf, int ltype, const double* out, const double* grad /* [1] */,
                     float* dfn, void* stream);

/* ------------------------------------------------------------------------------------ *
 * 7. Input preparation of the network forward (util/networks.py:67-79, util/meshnet.py:282-293):
 *    x[n,4] = (dm * ((z1 - zc) / z_sc), dm) with zc = (min + max) / 2 and z_sc = max_d (max - min) of
 *    z1 over the vertices -- the reference's ~10 ATen launches as a bounding-box reduction + one
 *    elementwise pass, bit-identical arithmetic.  dm [n] (NULL = all ones, the reference's default
 *    mask); scratch: float[16] (receives zc[3], z_sc at scratch[8..11] for inspection).
 * ------------------------------------------------------------------------------------ */
SGB_API int sgb_input_prep(const float* z1, int64_t ldz, int64_t n, const float* dm, float* x, float* scratch /* [16] */, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* SEMIGCN_B200_H */
