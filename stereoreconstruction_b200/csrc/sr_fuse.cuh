// sr_fuse.cuh — one de-duplicated, coloured point cloud from the depth maps of all views (sr_fuse_points; the
// model is stated in include/sr_b200.h).  The views' clouds are those of sr_points.cuh; a source pixel p of view v
// with point X is confirmed by each other view u whose pixel q under X has a point X_u within max_dist of X.
//
//   fuse_support_kernel  one thread per pixel of every view: support(p), and the fused point and colour (the
//                        mean over X and the confirming X_u) into per-pixel scratch
//   fuse_emit_kernel     one block per (view, row): which kept pixels are emitted (no confirming lower view
//                        whose pixel q is itself kept), and the row's count
//   points_scan_kernel   (sr_points.cuh) over the V * h row counts
//   fuse_write_kernel    one block per (view, row): the row's emitted points from its offset on, ballot-compacted
//
// The emit pass projects into the lower views again rather than storing a matched pixel per view pair, so the
// scratch stays at 32 bytes per pixel of each view.  Every pixel is computed by one thread from maps no pass
// writes, so there are no atomics and every call gives the same bits.
#pragma once
#include "sr_points.cuh"

namespace sr {

constexpr int FUSE_THREADS = 128;
constexpr uint32_t FUSE_EMITTED = 1u << 24;  // in FuseArgs::rgbe, above the fused colour

struct FuseArgs {
    const sr_camera *cams;        // [V]
    double *const *depth;         // [V] -> [h][w]
    const uchar4 *const *rgba;    // [V] -> [h][w]
    int V, w, h;
    double scale, min_depth, max_dist;
    int min_views;
    // per-pixel scratch, index (v * h + y) * w + x
    double *fxyz;                 // [3][V * h * w] fused position (planes x, y, z)
    int32_t *support;             // [V * h * w] support, -1: the pixel has no point
    uint32_t *rgbe;               // [V * h * w] fused r | g << 8 | b << 16, | FUSE_EMITTED; 0 without a point
    long long *offsets;           // [V * h + 1] row counts, then their exclusive prefix sums
    double *xyz;                  // [points][3]
    uint8_t *rgb;                 // [points][3]
    int32_t *source;              // [points][2] (view, y * w + x), or null
};

// Whether view u confirms the point X: X projects (cam_project, times scale) into the image of u, the pixel q
// there has a point X_u (taken at q's centre), and |X - X_u| < max_dist.  q is the pixel index y * w + x.
__device__ __forceinline__ bool fuse_match(const FuseArgs &a, int u, d3 X, size_t &q, d3 &Xu) {
    const sr_camera &B = a.cams[u];
    double x2, y2;
    if (!cam_project(B, X, x2, y2)) return false;
    x2 *= a.scale;
    y2 *= a.scale;
    if (!(x2 >= 0 && y2 >= 0 && x2 < a.w && y2 < a.h)) return false;
    const int qx = (int)x2, qy = (int)y2;
    if (!point_of_pixel(B, a.depth[u], a.w, qx, qy, a.scale, a.min_depth, Xu)) return false;
    q = (size_t)qy * a.w + qx;
    const d3 df = X - Xu;
    const double dist = sqrt(dot(df, df));
    return isfinite(dist) && dist < a.max_dist;
}

__global__ void __launch_bounds__(FUSE_THREADS) fuse_support_kernel(const FuseArgs a) {
    const size_t n = (size_t)a.w * a.h;
    const size_t i = (size_t)blockIdx.x * FUSE_THREADS + threadIdx.x;
    if (i >= (size_t)a.V * n) return;
    const int v = (int)(i / n);
    const size_t pix = i - (size_t)v * n;
    const int x = (int)(pix % a.w), y = (int)(pix / a.w);
    d3 X;
    if (!point_of_pixel(a.cams[v], a.depth[v], a.w, x, y, a.scale, a.min_depth, X)) {
        a.support[i] = -1;
        a.rgbe[i] = 0;
        return;
    }
    const uchar4 c = a.rgba[v][pix];
    d3 sum = X;  // X first, then the confirming views in ascending order
    unsigned r = c.x, g = c.y, b = c.z;
    int support = 0;
    for (int u = 0; u < a.V; ++u) {
        if (u == v) continue;
        size_t q;
        d3 Xu;
        if (!fuse_match(a, u, X, q, Xu)) continue;
        sum = sum + Xu;
        const uchar4 cu = a.rgba[u][q];
        r += cu.x;
        g += cu.y;
        b += cu.z;
        ++support;
    }
    const double m = 1.0 + support;
    a.fxyz[i] = sum.x / m;
    a.fxyz[n * a.V + i] = sum.y / m;
    a.fxyz[2 * n * a.V + i] = sum.z / m;
    const unsigned k = 1u + (unsigned)support;
    a.rgbe[i] = (r + k / 2) / k | (g + k / 2) / k << 8 | (b + k / 2) / k << 16;
    a.support[i] = support;
}

__global__ void __launch_bounds__(POINTS_THREADS) fuse_emit_kernel(const FuseArgs a) {
    const int row = blockIdx.x;  // v * h + y
    const int v = row / a.h, y = row - v * a.h;
    const size_t n = (size_t)a.w * a.h;
    int count = 0;
    for (int x0 = 0; x0 < a.w; x0 += POINTS_THREADS) {
        const int x = x0 + threadIdx.x;
        bool emit = false;
        if (x < a.w) {
            const size_t i = (size_t)row * a.w + x;
            d3 X;
            // a kept pixel has a point (support -1 < min_views), which the support pass computed the same way
            if (a.support[i] >= a.min_views && point_of_pixel(a.cams[v], a.depth[v], a.w, x, y, a.scale, a.min_depth, X)) {
                emit = true;
                for (int u = 0; u < v && emit; ++u) {
                    size_t q;
                    d3 Xu;
                    if (fuse_match(a, u, X, q, Xu) && a.support[(size_t)u * n + q] >= a.min_views) emit = false;
                }
                if (emit) a.rgbe[i] |= FUSE_EMITTED;
            }
        }
        count += __syncthreads_count(emit);
    }
    if (threadIdx.x == 0) a.offsets[row] = count;
}

__global__ void __launch_bounds__(POINTS_THREADS) fuse_write_kernel(const FuseArgs a) {
    __shared__ int warp_count[POINTS_THREADS / 32];
    const int row = blockIdx.x;
    const int v = row / a.h, y = row - v * a.h;
    const size_t N = (size_t)a.V * a.w * a.h;
    long long base = a.offsets[row];
    for (int x0 = 0; x0 < a.w; x0 += POINTS_THREADS) {
        const int x = x0 + threadIdx.x;
        const size_t i = (size_t)row * a.w + x;
        const uint32_t e = x < a.w ? a.rgbe[i] : 0u;
        const bool keep = (e & FUSE_EMITTED) != 0;
        int chunk;
        const int before = chunk_rank(keep, warp_count, chunk);
        if (keep) {
            const long long o = base + before;
            a.xyz[3 * o] = a.fxyz[i];
            a.xyz[3 * o + 1] = a.fxyz[N + i];
            a.xyz[3 * o + 2] = a.fxyz[2 * N + i];
            a.rgb[3 * o] = (uint8_t)e;
            a.rgb[3 * o + 1] = (uint8_t)(e >> 8);
            a.rgb[3 * o + 2] = (uint8_t)(e >> 16);
            if (a.source) {
                a.source[2 * o] = v;
                a.source[2 * o + 1] = y * a.w + x;
            }
        }
        base += chunk;
        __syncthreads();  // warp_count is rewritten by the next chunk
    }
}

}  // namespace sr
