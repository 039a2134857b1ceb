// sr_points.cuh — the coloured point cloud of one view's depth map (sr_get_points): the input of
// MultiViewStereo's outputPLYFile (multiviewstereo.cpp:291-315), one point per kept pixel as
// pointFromDepth makes it (:740-750), in row-major pixel order.
//
//   points_count_kernel  one block per image row: the number of the row's kept pixels
//   points_scan_kernel   one block: exclusive prefix sums of the row counts, and the total
//   points_write_kernel  one block per image row: the row's points from its offset on, ordered
//                        within the row by warp ballots
//
// Both row passes evaluate the same test per pixel (filter, Camera::unproject, plane intersection).
// It is deterministic, so the write pass keeps exactly the pixels the count pass counted; this
// costs a second unproject but keeps no per-pixel ray table resident.
#pragma once
#include "sr_kernels.cuh"

namespace sr {

constexpr int POINTS_THREADS = 256;
constexpr int POINTS_SCAN_THREADS = 1024;  // any number of rows: fusion (sr_fuse.cuh) scans the rows of all V views

struct PointsArgs {
    sr_camera cam;
    const double *depth;  // [h][w]
    const uchar4 *rgba;   // [h][w]
    int w, h;
    double scale, min_depth;
    long long *offsets;   // [h + 1]: row counts, then their exclusive prefix sums; [h] = number of points
    double *xyz;          // [points][3]
    uint8_t *rgb;         // [points][3]
    int32_t *pixel;       // [points] y * w + x, or null
};

// The point of pixel (x, y) of a view with camera `cam` and depth map `depth` (row pitch w), if it has one: the
// filter and plane of MultiViewStereo::pointCloud.
__device__ __forceinline__ bool point_of_pixel(const sr_camera &cam, const double *depth, int w, int x, int y, double scale,
                                               double min_depth, d3 &p) {
    const double d = depth[(size_t)y * w + x];
    if (!isfinite(d) || d + 1e-5 < min_depth) return false;
    d3 src, dir;
    cam_unproject(cam, (x + 0.5) / scale, (y + 0.5) / scale, src, dir);
    return point_from_depth(src, dir, ld3(cam.prin_dir), ld3(cam.C), d, p);
}
__device__ __forceinline__ bool point_of_pixel(const PointsArgs &a, int x, int y, d3 &p) {
    return point_of_pixel(a.cam, a.depth, a.w, x, y, a.scale, a.min_depth, p);
}

__global__ void __launch_bounds__(POINTS_THREADS) points_count_kernel(const PointsArgs a) {
    const int y = blockIdx.x;
    int count = 0;
    for (int x0 = 0; x0 < a.w; x0 += POINTS_THREADS) {
        const int x = x0 + threadIdx.x;
        d3 p;
        count += __syncthreads_count(x < a.w && point_of_pixel(a, x, y, p));
    }
    if (threadIdx.x == 0) a.offsets[y] = count;
}

__device__ __forceinline__ long long warp_inclusive_sum(long long v, int lane) {
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const long long t = __shfl_up_sync(0xffffffffu, v, o);
        if (lane >= o) v += t;
    }
    return v;
}

// In place: offsets[r] = sum of the counts of rows < r, offsets[h] = sum of all (h: any number of rows).  Each
// thread owns a run of consecutive rows.
__global__ void __launch_bounds__(POINTS_SCAN_THREADS) points_scan_kernel(long long *offsets, int h) {
    __shared__ long long warp_base[POINTS_SCAN_THREADS / 32];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int per = (h + POINTS_SCAN_THREADS - 1) / POINTS_SCAN_THREADS;
    const int r0 = min(h, (int)threadIdx.x * per), r1 = min(h, r0 + per);
    long long own = 0;
    for (int r = r0; r < r1; ++r) own += offsets[r];
    const long long inc = warp_inclusive_sum(own, lane);
    if (lane == 31) warp_base[wid] = inc;
    __syncthreads();
    if (wid == 0) {
        const long long tot = warp_base[lane];
        warp_base[lane] = warp_inclusive_sum(tot, lane) - tot;
    }
    __syncthreads();
    long long run = warp_base[wid] + inc - own;
    for (int r = r0; r < r1; ++r) {
        const long long c = offsets[r];
        offsets[r] = run;
        run += c;
    }
    if (threadIdx.x == POINTS_SCAN_THREADS - 1) offsets[h] = run;
}

// Compaction of one POINTS_THREADS-wide chunk of a row: the number of keeping threads of the block before this
// one, in thread order; `chunk` receives the block's total.  The caller synchronises before reusing warp_count.
__device__ __forceinline__ int chunk_rank(bool keep, int *warp_count, int &chunk) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const unsigned ballot = __ballot_sync(0xffffffffu, keep);
    if (lane == 0) warp_count[wid] = __popc(ballot);
    __syncthreads();
    int before = __popc(ballot & ((1u << lane) - 1u));
    chunk = 0;
#pragma unroll
    for (int k = 0; k < POINTS_THREADS / 32; ++k) {
        const int c = warp_count[k];
        if (k < wid) before += c;
        chunk += c;
    }
    return before;
}

__global__ void __launch_bounds__(POINTS_THREADS) points_write_kernel(const PointsArgs a) {
    __shared__ int warp_count[POINTS_THREADS / 32];
    const int y = blockIdx.x;
    long long base = a.offsets[y];
    for (int x0 = 0; x0 < a.w; x0 += POINTS_THREADS) {
        const int x = x0 + threadIdx.x;
        d3 p;
        const bool keep = x < a.w && point_of_pixel(a, x, y, p);
        int chunk;
        const int before = chunk_rank(keep, warp_count, chunk);
        if (keep) {
            const long long o = base + before;
            const size_t i = (size_t)y * a.w + x;
            a.xyz[3 * o] = p.x;
            a.xyz[3 * o + 1] = p.y;
            a.xyz[3 * o + 2] = p.z;
            const uchar4 c = a.rgba[i];
            a.rgb[3 * o] = c.x;
            a.rgb[3 * o + 1] = c.y;
            a.rgb[3 * o + 2] = c.z;
            if (a.pixel) a.pixel[o] = (int32_t)i;
        }
        base += chunk;
        __syncthreads();  // warp_count is rewritten by the next chunk
    }
}

}  // namespace sr
