// C-ABI entry points of the dense feature transform; dispatch between the fp32 CUDA-core
// tiles (gemm_simt.cu) and the tcgen05 fp16-split tiles (gemm_f16.cu).
#include "common.cuh"

namespace sgb {
int gemm_simt_launch(const GemmArgs& g, cudaStream_t stream);
int gemm_tn_simt_launch(const float* g, int64_t ldg, const float* a, int64_t lda, float* d, int64_t ldd, int64_t m, int n, int k,
                        int accumulate, void* ws, size_t ws_bytes, cudaStream_t stream);
size_t gemm_tn_simt_workspace(int64_t m, int n, int k);
bool gemm_f16_supported(int64_t m, int n, int k, int64_t lda, int64_t ldc, const void* a, const void* c, const void* bias);
bool gemm_tn_f16_supported(int64_t m, int n, int k, int64_t ldg, int64_t lda, const void* g, const void* a);
size_t gemm_f16_workspace(int n, int k);
int gemm_f16_launch(const GemmArgs& g, const float* a_amax, void* ws, size_t ws_bytes, cudaStream_t stream);
size_t gemm_tn_f16_workspace(int64_t m, int n, int k);
int gemm_tn_f16_launch(const float* g, int64_t ldg, const float* a, int64_t lda, const float* g_amax, const float* a_amax, float* d,
                       int64_t ldd, int64_t m, int n, int k, int accumulate, void* ws, size_t ws_bytes, cudaStream_t stream);
bool gemm_tn_pair_ok(int64_t m, int n, int k);
size_t gemm_tn_pair_workspace(int64_t m, int n, int k);
int gemm_tn_pair_launch(const float* g, int64_t ldg, const float* a, int64_t lda, const float* g_amax, const float* a_amax, float* d,
                        int64_t ldd, int64_t m, int n, int k, int accumulate, void* ws, size_t ws_bytes, cudaStream_t stream);
// (998 562 rows, two alternating converter groups for the narrow stages: 32x64 0.130 ms against 0.241 on the CUDA-core split-K kernel,
// 32x16 0.122 / 0.159, 16x32 and below equal -- tools/bench_small_shapes.py)
static bool tn_tc_worthwhile(int64_t m, int n, int k) { return n >= 32 && k >= 16 && m >= 4096; }

// auto policy: the tensor pipe only where the transform is a real dense contraction (SURVEY.md §8(d))
// (measured on 998 562 rows: n32_k64 0.195 ms on the CUDA-core tiles, 0.085 ms on the fp16-split CTA pairs; n32_k16 0.087 / 0.071;
// n16_k32 equal -- tools/bench_small_shapes.py)
static bool tc_worthwhile(int64_t m, int n, int k) { return n >= 32 && k >= 16 && m >= 2048; }
}  // namespace sgb

using namespace sgb;

namespace sgb {
int gemm_stat_rows(int64_t m) {
    if (m <= 0) return 0;
    const int64_t tiles = ceil_div(m, 128);
    return 4 * (int)(tiles < num_sms() ? tiles : num_sms());
}
}  // namespace sgb

extern "C" int sgb_gemm_stat_rows(int64_t m) { return gemm_stat_rows(m); }

extern "C" size_t sgb_gemm_workspace_bytes(int64_t m, int n, int k, int engine) {
    if (m < 0 || n <= 0 || k <= 0 || n % 16 != 0 || k % 4 != 0) return 0;
    if (engine == 3 || (engine == 0 && tc_worthwhile(m, n, k))) return gemm_f16_workspace(n, k);
    return 0;
}

extern "C" int sgb_gemm(int transb, const float* a, int64_t lda, const float* b, int64_t ldb, float* c, int64_t ldc, int64_t m,
                        int n, int k, const float* bias, int accumulate, float* stat_partials, const float* a_amax, void* workspace,
                        size_t workspace_bytes, int engine, void* stream) {
    SGB_CHECK_ARG(a && b && c && m >= 0 && n > 0 && k > 0, "sgb_gemm: bad argument m=%lld n=%d k=%d", (long long)m, n, k);
    SGB_CHECK_ARG(lda >= k && ldc >= n && ldb >= (transb ? k : n), "sgb_gemm: leading dimension too small");
    SGB_CHECK_ARG(engine == 0 || engine == 1 || engine == 3, "sgb_gemm: bad engine %d", engine);
    if (m == 0) return SGB_OK;
    GemmArgs g{transb, a, lda, b, ldb, c, ldc, m, n, k, bias, accumulate, stat_partials};
    const bool tc_ok = gemm_f16_supported(m, n, k, lda, ldc, a, c, bias);
    if (engine == 3) {
        if (!tc_ok) {
            set_error("sgb_gemm: fp16-split engine needs n %% 16 == 0, k %% 4 == 0 and 16-byte aligned operands (n=%d k=%d)", n, k);
            return SGB_ENOTSUP;
        }
        return gemm_f16_launch(g, a_amax, workspace, workspace_bytes, (cudaStream_t)stream);
    }
    // auto: the fp16-split tiles (HBM-bound) for real contractions
    if (engine == 0 && tc_ok && tc_worthwhile(m, n, k) && workspace && workspace_bytes >= gemm_f16_workspace(n, k))
        return gemm_f16_launch(g, a_amax, workspace, workspace_bytes, (cudaStream_t)stream);
    return gemm_simt_launch(g, (cudaStream_t)stream);
}

extern "C" size_t sgb_gemm_tn_workspace_bytes(int64_t m, int n, int k) {
    if (m < 0 || n <= 0 || k <= 0) return 0;
    size_t a = gemm_tn_simt_workspace(m, n, k);
    size_t c = (n % 4 == 0 && k % 4 == 0) ? gemm_tn_f16_workspace(m, n, k) : 0;
    size_t e = gemm_tn_pair_workspace(m, n, k);
    a = a > c ? a : c;
    return a > e ? a : e;
}

extern "C" int sgb_gemm_tn(const float* g, int64_t ldg, const float* a, int64_t lda, float* d, int64_t ldd, int64_t m, int n, int k,
                           int accumulate, const float* g_amax, const float* a_amax, void* workspace, size_t workspace_bytes, int engine,
                           void* stream) {
    SGB_CHECK_ARG(g && a && d && m >= 0 && n > 0 && k > 0, "sgb_gemm_tn: bad argument");
    SGB_CHECK_ARG(ldg >= n && lda >= k && ldd >= k, "sgb_gemm_tn: leading dimension too small");
    SGB_CHECK_ARG(engine == 0 || engine == 1 || engine == 3 || engine == 4, "sgb_gemm_tn: bad engine %d", engine);
    const bool tc_ok = gemm_tn_f16_supported(m, n, k, ldg, lda, g, a);
    // auto: 256-row multiples of D go to CTA pairs (measured on 998 562 vertices, amax supplied: n256_k256 0.517 -> 0.425 ms,
    // n512_k256 0.994 -> 0.839 ms, n256_k64 0.390 -> 0.310 ms against the single-CTA engine)
    if (engine == 0 && tc_ok && gemm_tn_pair_ok(m, n, k) && m >= 32768) engine = 4;
    if (engine == 4) {       // tcgen05 fp16-split tiles on CTA pairs (cta_group::2)
        if (!tc_ok || !gemm_tn_pair_ok(m, n, k)) {
            set_error("sgb_gemm_tn: the pair engine needs n %% 256 == 0, k %% 32 == 0 (k <= 256 or k %% 256 == 0), m >= 4096 and 16-byte aligned operands");
            return SGB_ENOTSUP;
        }
        return gemm_tn_pair_launch(g, ldg, a, lda, g_amax, a_amax, d, ldd, m, n, k, accumulate, workspace, workspace_bytes, (cudaStream_t)stream);
    }
    if (engine == 3 || (engine == 0 && tc_ok && tn_tc_worthwhile(m, n, k))) {
        if (!tc_ok) {
            set_error("sgb_gemm_tn: fp16-split engine needs n %% 4 == 0, k %% 4 == 0 and 16-byte aligned operands");
            return SGB_ENOTSUP;
        }
        return gemm_tn_f16_launch(g, ldg, a, lda, g_amax, a_amax, d, ldd, m, n, k, accumulate, workspace, workspace_bytes, (cudaStream_t)stream);
    }
    return gemm_tn_simt_launch(g, ldg, a, lda, d, ldd, m, n, k, accumulate, workspace, workspace_bytes, (cudaStream_t)stream);
}
