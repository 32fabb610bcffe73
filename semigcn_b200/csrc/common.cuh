// Shared helpers for the semigcn_b200 C-ABI library (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdarg.h>
#include <atomic>
#include "../../include/semigcn_b200.h"

namespace sgb {

void set_error(const char* fmt, ...);   // thread-local message (api.cu)
int num_sms();                           // cached per process (api.cu)
int smem_optin(const void* func, int bytes, std::atomic<uint64_t>* done_mask);   // dynamic shared memory opt-in, once per device (api.cu)

#define SGB_CHECK_ARG(cond, ...)                 \
    do {                                         \
        if (!(cond)) {                           \
            sgb::set_error(__VA_ARGS__);         \
            return SGB_EINVAL;                   \
        }                                        \
    } while (0)

#define SGB_CHECK_LAUNCH(name)                                                        \
    do {                                                                              \
        cudaError_t e__ = cudaGetLastError();                                         \
        if (e__ != cudaSuccess) {                                                     \
            sgb::set_error("%s: launch failed: %s", name, cudaGetErrorString(e__));   \
            return SGB_ECUDA;                                                         \
        }                                                                             \
    } while (0)

#define SGB_CUDA(call)                                                                \
    do {                                                                              \
        cudaError_t e__ = (call);                                                     \
        if (e__ != cudaSuccess) {                                                     \
            sgb::set_error("%s failed: %s", #call, cudaGetErrorString(e__));          \
            return SGB_ECUDA;                                                         \
        }                                                                             \
    } while (0)

static inline int64_t ceil_div(int64_t a, int64_t b) { return (a + b - 1) / b; }
__host__ __device__ static inline int64_t min64(int64_t a, int64_t b) { return a < b ? a : b; }
static inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

__device__ __forceinline__ float lrelu(float v, float slope) { return v > 0.f ? v : v * slope; }

// fused BatchNorm + LeakyReLU on load: centred form (x - mean) * scale + beta.  The uncentred
// x*scale + (beta - mean*scale) cancels catastrophically when |mean| >> std (near-constant channels).
__device__ __forceinline__ float bn_lrelu(float x, float mean, float scale, float beta, float slope) {
    return lrelu(fmaf(x - mean, scale, beta), slope);
}

// BatchNorm statistic partials are (count, mean, M2 = sum (x-mean)^2) triples, merged with Chan's
// parallel formula -- sum / sum-of-squares partials lose the variance of near-constant channels.
struct Moments {
    float n, mean, m2;
};
__device__ __forceinline__ Moments merge(Moments a, Moments b) {
    if (b.n == 0.f) return a;
    if (a.n == 0.f) return b;
    Moments r;
    r.n = a.n + b.n;
    const float d = b.mean - a.mean;
    const float w = b.n / r.n;
    r.mean = fmaf(d, w, a.mean);
    r.m2 = a.m2 + b.m2 + d * d * a.n * w;
    return r;
}
// from pivot-shifted sums: s1 = sum (x - p), s2 = sum (x - p)^2 over n values
__device__ __forceinline__ Moments from_shifted(float n, float p, float s1, float s2) {
    Moments r;
    r.n = n;
    if (n == 0.f) { r.mean = 0.f; r.m2 = 0.f; return r; }
    const float dm = s1 / n;
    r.mean = p + dm;
    r.m2 = fmaxf(s2 - s1 * dm, 0.f);
    return r;
}

// streaming 128-bit load/store helpers (read-only path; Y/Z outputs are written once)
__device__ __forceinline__ float4 ldg4(const float* p) { return __ldg(reinterpret_cast<const float4*>(p)); }
__device__ __forceinline__ void st4(float* p, float4 v) { *reinterpret_cast<float4*>(p) = v; }

// |x| as it enters a published max |x|: inf and NaN count as 0.  The fp16-split engine scales an operand by a power of two
// taken from that maximum; an inf there would leave the scale at 1 and overflow every finite entry above 65504 in the fp16
// split, so rows without any inf would turn inf / NaN.  With the finite maximum an inf entry stays inf and a NaN stays NaN.
__device__ __forceinline__ float finite_abs(float x) {
    const float a = fabsf(x);
    return a <= 3.402823466e+38f ? a : 0.f;
}

// max |x| of a produced tensor, published for the fp16-split GEMM engine that consumes it (sgb_gemm a_amax):
// per-thread running maximum -> warp -> CTA -> one atomicMax on the float bits (non-negative floats order like
// unsigned ints; max is order-independent, so the result is deterministic).  `scratch`: >= 32 uint32 of shared memory.
// Callers accumulate `mx` with finite_abs.
__device__ __forceinline__ void publish_amax(float mx, uint32_t* scratch, float* slot) {
    uint32_t b = __reduce_max_sync(0xffffffffu, __float_as_uint(mx));
    const int warp = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
    if ((threadIdx.x & 31) == 0) scratch[warp] = b;
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < nw; ++w) b = max(b, scratch[w]);
        if (b) atomicMax(reinterpret_cast<uint32_t*>(slot), b);
    }
}

// rows of the BatchNorm-partials buffer of sgb_gemm (every engine writes at most this many (count, mean, M2) rows and
// zero-fills the rest): 4 * min(ceil(m / 128), #SMs) -- gemm.cu
int gemm_stat_rows(int64_t m);

// arguments of the dense transform C (+)= A op(B) + bias (see sgb_gemm)
struct GemmArgs {
    int transb;
    const float* a; int64_t lda;
    const float* b; int64_t ldb;
    float* c; int64_t ldc;
    int64_t m; int n; int k;
    const float* bias; int accumulate; float* stat_partials;
};

}  // namespace sgb
