// Exact point-to-surface distance: nearest triangle of a target mesh for every query point, over a uniform grid.
//
// The grid (built once per target mesh by semigcn_b200/distance.py::SurfaceIndex) lists every face in every cell that its
// bounding box, widened by a small relative epsilon, overlaps.  A face's closest point to any query lies inside that box,
// so it lies in a cell that lists the face: a search that has visited every cell whose box is not farther than the best
// distance found has seen the nearest face.  One thread per query visits Chebyshev rings r = 0, 1, ... around the query's
// cell (clamped into the grid), skips cells whose box is farther than the current best, and stops once the best distance
// is below the distance to the nearest inner face of the visited block (the block's sides on the grid boundary have no
// cells beyond them).  The ring loop is bounded by the largest grid dimension, so it terminates for any input.
//
// Point-to-triangle runs in fp64 on the fp32 coordinates: Ericson's Voronoi-region test (Real-Time Collision Detection,
// 5.1.5) translated to the first corner, with the closest point q formed explicitly and the distance taken as |p - q|
// (the expanded quadratic form loses sqrt(eps) near the surface).  A zero-area face falls back to the nearest of its three
// edge segments.  Candidates compare lexicographically on (squared distance, face id), so the answer is the smallest face
// id among exact ties, independent of the visit order and therefore of the grid.  No floating-point atomics, no
// synchronisation: the call is stream-ordered and CUDA-graph capturable.
#include "common.cuh"
#include <math.h>

namespace sgb {

struct D3 {
    double x, y, z;
};
__host__ __device__ __forceinline__ D3 sub(D3 a, D3 b) { return {a.x - b.x, a.y - b.y, a.z - b.z}; }
__host__ __device__ __forceinline__ D3 scale(D3 a, double s) { return {a.x * s, a.y * s, a.z * s}; }
__host__ __device__ __forceinline__ D3 add(D3 a, D3 b) { return {a.x + b.x, a.y + b.y, a.z + b.z}; }
__host__ __device__ __forceinline__ double dot(D3 a, D3 b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
__host__ __device__ __forceinline__ double norm2(D3 a) { return dot(a, a); }

// squared distance from ap (the query relative to the segment start) to the segment [0, ab]
__host__ __device__ __forceinline__ double seg_dist2(D3 ap, D3 ab) {
    const double l2 = norm2(ab);
    double t = l2 > 0.0 ? dot(ap, ab) / l2 : 0.0;
    t = fmin(fmax(t, 0.0), 1.0);
    return norm2(sub(ap, scale(ab, t)));
}

__host__ __device__ __forceinline__ D3 cross(D3 a, D3 b) { return {a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x}; }

// squared distance from p to the closed triangle (a, b, c); exactly 0 when p is one of the corners.  Ericson's region
// tests, except that the three barycentric numerators are taken in the form n . (u x v) (Lagrange's identity) instead of
// d1 d4 - d3 d2 etc.: the difference form cancels catastrophically on slivers, whose |n|^2 is far below |ab|^2 |ac|^2.
__host__ __device__ __forceinline__ double tri_dist2(D3 p, D3 a, D3 b, D3 c) {
    const D3 ab = sub(b, a), ac = sub(c, a), ap = sub(p, a);
    const D3 n = cross(ab, ac);
    const double nn = norm2(n);
    if (nn == 0.0)   // zero area (collinear or coincident corners): the nearest of the three edge segments
        return fmin(fmin(seg_dist2(ap, ab), seg_dist2(ap, ac)), seg_dist2(sub(p, b), sub(c, b)));
    const double d1 = dot(ab, ap), d2 = dot(ac, ap);
    if (d1 <= 0.0 && d2 <= 0.0) return norm2(ap);                                   // corner a
    const D3 bp = sub(ap, ab);
    const double d3 = dot(ab, bp), d4 = dot(ac, bp);
    if (d3 >= 0.0 && d4 <= d3) return norm2(bp);                                    // corner b
    const double vc = dot(n, cross(ap, bp));                                        // = d1 d4 - d3 d2
    if (vc <= 0.0 && d1 >= 0.0 && d3 <= 0.0) return norm2(sub(ap, scale(ab, d1 / (d1 - d3))));   // edge ab
    const D3 cp = sub(ap, ac);
    const double d5 = dot(ab, cp), d6 = dot(ac, cp);
    if (d6 >= 0.0 && d5 <= d6) return norm2(cp);                                    // corner c
    const double vb = dot(n, cross(cp, ap));                                        // = d5 d2 - d1 d6
    if (vb <= 0.0 && d2 >= 0.0 && d6 <= 0.0) return norm2(sub(ap, scale(ac, d2 / (d2 - d6))));   // edge ac
    const double va = dot(n, cross(bp, cp));                                        // = d3 d6 - d5 d4
    if (va <= 0.0 && d4 - d3 >= 0.0 && d5 - d6 >= 0.0) {                           // edge bc
        const double w = (d4 - d3) / ((d4 - d3) + (d5 - d6));
        return norm2(sub(bp, scale(sub(ac, ab), w)));
    }
    return norm2(sub(ap, add(scale(ab, vb / nn), scale(ac, vc / nn))));             // interior (va + vb + vc = |n|^2)
}

__host__ __device__ __forceinline__ int imax(int a, int b) { return a > b ? a : b; }
__host__ __device__ __forceinline__ int imin(int a, int b) { return a < b ? a : b; }

// Boxes and the stopping bound are compared with a relative margin of 1e-9 in the conservative direction, so fp64
// rounding of the cell borders can neither skip a cell that holds the answer nor stop before it.
constexpr double kPruneSlack = 1.0 + 1e-9;

// The search for query i.  __host__ __device__ so that a host build can step through it.
__host__ __device__ __forceinline__ void search_one(int64_t i, const float* __restrict__ points, int64_t ldp, const float* __restrict__ tris,
                                                   const int32_t* __restrict__ cell_start, const int32_t* __restrict__ cell_faces,
                                                   float ox, float oy, float oz, float hf, int gx, int gy, int gz,
                                                   float* __restrict__ dist, int32_t* __restrict__ face) {
    const float px = points[i * ldp], py = points[i * ldp + 1], pz = points[i * ldp + 2];
    // NaN guard: with a NaN coordinate every comparison below is false; such a query never enters the search
    if (!(isfinite(px) && isfinite(py) && isfinite(pz))) {
        dist[i] = NAN;
        face[i] = -1;
        return;
    }
    const D3 p = {px, py, pz};
    const double h = hf, o[3] = {ox, oy, oz};
    const int g[3] = {gx, gy, gz};
    const double pc[3] = {p.x, p.y, p.z};
    int home[3];
#pragma unroll
    for (int d = 0; d < 3; ++d) home[d] = (int)fmin(fmax(floor((pc[d] - o[d]) / h), 0.0), (double)(g[d] - 1));

    double best = INFINITY;   // squared distance
    int32_t best_f = -1;
#ifdef SGB_SURFACE_COUNT_CANDIDATES
    int32_t tested = 0;
#endif
    const int rmax = imax(gx, imax(gy, gz));
    for (int r = 0; r < rmax; ++r) {
        const int lx = imax(home[0] - r, 0), hx = imin(home[0] + r, gx - 1);
        const int ly = imax(home[1] - r, 0), hy = imin(home[1] + r, gy - 1);
        for (int cx = lx; cx <= hx; ++cx) {
            const bool x_shell = cx == home[0] - r || cx == home[0] + r;
            for (int cy = ly; cy <= hy; ++cy) {
                const bool xy_shell = x_shell || cy == home[1] - r || cy == home[1] + r;
                // inside the shell in x and y only the two z layers at distance r belong to ring r
                const int zstep = xy_shell ? 1 : imax(2 * r, 1);
                for (int cz = home[2] - r; cz <= home[2] + r; cz += zstep) {
                    if (cz < 0 || cz >= gz) continue;
                    const int cc[3] = {cx, cy, cz};
                    double box = 0.0;
#pragma unroll
                    for (int d = 0; d < 3; ++d) {
                        const double b0 = o[d] + cc[d] * h, b1 = b0 + h;
                        const double e = fmax(fmax(b0 - pc[d], pc[d] - b1), 0.0);
                        box += e * e;
                    }
                    if (box > best * kPruneSlack) continue;
                    const int64_t cell = ((int64_t)cz * gy + cy) * gx + cx;
                    const int32_t s = cell_start[cell], t = cell_start[cell + 1];
                    for (int32_t k = s; k < t; ++k) {
                        const int32_t f = cell_faces[k];
                        const float4* tf = reinterpret_cast<const float4*>(tris + (int64_t)f * 12);
                        const float4 t0 = tf[0], t1 = tf[1], t2 = tf[2];
                        const double d2 = tri_dist2(p, {t0.x, t0.y, t0.z}, {t0.w, t1.x, t1.y}, {t1.z, t1.w, t2.x});
#ifdef SGB_SURFACE_COUNT_CANDIDATES
                        ++tested;
#endif
                        if (d2 < best || (d2 == best && f < best_f)) { best = d2; best_f = f; }
                    }
                }
            }
        }
        // every cell not yet visited lies beyond one of the block's sides that are not on the grid boundary
        double bound = INFINITY;
#pragma unroll
        for (int d = 0; d < 3; ++d) {
            if (home[d] - r > 0) bound = fmin(bound, pc[d] - (o[d] + (home[d] - r) * h));
            if (home[d] + r < g[d] - 1) bound = fmin(bound, (o[d] + (home[d] + r + 1) * h) - pc[d]);
        }
        if (bound == INFINITY) break;                                   // the block is the whole grid
        if (bound > 0.0 && best * kPruneSlack < bound * bound) break;   // nothing beyond the block can be closer
    }
    dist[i] = (float)sqrt(best);
#ifdef SGB_SURFACE_COUNT_CANDIDATES
    face[i] = tested;   // counting build (tools/bench_mesh_distance.py): candidates tested instead of the face id
#else
    face[i] = best_f;
#endif
}

__global__ void k_point_surface_distance(
    const float* __restrict__ points, int64_t ldp, int64_t n, const float* __restrict__ tris,
    const int32_t* __restrict__ cell_start, const int32_t* __restrict__ cell_faces,
    float ox, float oy, float oz, float h, int gx, int gy, int gz, float* __restrict__ dist, int32_t* __restrict__ face) {
    const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    if (i < n) search_one(i, points, ldp, tris, cell_start, cell_faces, ox, oy, oz, h, gx, gy, gz, dist, face);
}

}  // namespace sgb

using namespace sgb;

extern "C" int sgb_point_surface_distance(const float* points, int64_t ldp, int64_t n, const float* tris, int64_t nf,
                                          const int32_t* cell_start, const int32_t* cell_faces, float ox, float oy, float oz,
                                          float h, int gx, int gy, int gz, float* dist, int32_t* face, void* stream_) {
    cudaStream_t stream = (cudaStream_t)stream_;
    SGB_CHECK_ARG(n >= 0 && ldp >= 3 && nf > 0 && nf <= INT32_MAX, "sgb_point_surface_distance: bad sizes (n %lld, ldp %lld, nf %lld)",
                  (long long)n, (long long)ldp, (long long)nf);
    SGB_CHECK_ARG(gx >= 1 && gy >= 1 && gz >= 1 && (int64_t)gx * gy * gz <= INT32_MAX, "sgb_point_surface_distance: bad grid %d x %d x %d",
                  gx, gy, gz);
    SGB_CHECK_ARG(isfinite(ox) && isfinite(oy) && isfinite(oz) && isfinite(h) && h > 0.f, "sgb_point_surface_distance: bad grid origin / cell size");
    if (n == 0) return SGB_OK;
    SGB_CHECK_ARG(points && tris && cell_start && cell_faces && dist && face, "sgb_point_surface_distance: null pointer");
    SGB_CHECK_ARG((reinterpret_cast<uintptr_t>(tris) & 15) == 0, "sgb_point_surface_distance: tris must be 16-byte aligned");
    k_point_surface_distance<<<(unsigned)ceil_div(n, 128), 128, 0, stream>>>(points, ldp, n, tris, cell_start, cell_faces, ox, oy, oz, h,
                                                                             gx, gy, gz, dist, face);
    SGB_CHECK_LAUNCH("k_point_surface_distance");
    return SGB_OK;
}
