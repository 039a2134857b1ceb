// sr_kernels.cuh — hand-written sm_100a kernels of the dense-matching hot path.
//
//   prep_view_kernel      RGBA8 + mask  -> FP64 gray planes (validity folded in as NaN) and the
//                         four colour-edge planes the geodesic sweeps walk on
//   rays_kernel           Camera::unproject on every pixel centre        (camera.cpp:423-459)
//   build_kernel          stage (1): per (pixel, depth label, neighbour view) refractive
//                         reprojection -> packed integer tap volume      (twoviewstereo.cpp:308-316,
//                                                                         multiviewstereo.cpp:768-775)
//   weights_*_kernel      AdaptiveWeight / GeodesicWeight::init_weights  (adaptiveweight.cpp:47-79,
//                                                                         geodesicweight.cpp:59-131)
//   match_kernel<R,G,C>   stages (2)+(3): weighted window cost with the support weights, WTA fused
//                         in the epilogue; streams the tap volume once   (twoviewstereo.cpp:909-977,
//                                                                         multiviewstereo.cpp:113-189,589-602)
//   cross_check_kernel    crossCheck                                      (twoviewstereo.cpp:596-672,
//                                                                         multiviewstereo.cpp:666-729)
//
// Data layout in HBM (all row-major, x fastest):
//   gray planes  double [h][w]            per view, 3 variants (see prep_view_kernel)
//   edge planes  double [4][h][w]         per view: |rgb(p) - rgb(p + e)|, e = E, S, SE, SW
//   rays         double [6][h][w]         SoA: source xyz, direction xyz
//   tap volume   int32  [nbr][D][rows][w] (ty<<16 | tx&0xffff), TAP_NONE where the label cannot
//                                         be evaluated; x fastest: one warp reads/writes 128
//                                         contiguous bytes per label
//   weights      double [WN][rows*w]      support weights of the current row band, tap-major so
//                                         that neighbouring pixels' weights are contiguous
//   cost volume  float  [nbr][D][rows][w] optional (keep_cost_volume)
//   outputs      int32 index [h][w], double depth [h][w], double best [h][w]
#pragma once
#include "sr_geometry.cuh"

namespace sr {

constexpr int SR_MAX_NBRS = 8;
// Row pitch of the FP32 gray planes: the smallest of 1024/2048/4096/16384 that holds a row.
inline int screen_pitch(int w) { return w <= 1024 ? 1024 : w <= 2048 ? 2048 : w <= 4096 ? 4096 : 16384; }
constexpr int32_t TAP_NONE = INT32_MIN;
constexpr int TAP_CLAMP = 20000;  // |coordinate| beyond this is outside any image for any window

__device__ __forceinline__ double gray_of(uchar4 p) {
    // RGBA::toGray(), util/vectorimage.hpp:60-62 (no FMA contraction: same roundings as the
    // reference's plain expression)
    return __dadd_rn(__dadd_rn(__dmul_rn(0.11, (double)p.x), __dmul_rn(0.59, (double)p.y)),
                     __dmul_rn(0.3, (double)p.z));
}
__device__ __forceinline__ double qnan() { return __longlong_as_double(0x7ff8000000000000LL); }
__device__ __forceinline__ double dinf() { return __longlong_as_double(0x7ff0000000000000LL); }

__device__ __forceinline__ double color_dist(uchar4 a, uchar4 b) {
    // sqrt(dr^2 + dg^2 + db^2) on exact small integers (adaptiveweight.cpp:66-69, geodesicweight.cpp:92-94)
    const double dr = (double)((int)b.x - (int)a.x), dg = (double)((int)b.y - (int)a.y), db = (double)((int)b.z - (int)a.z);
    return sqrt(__dadd_rn(__dadd_rn(__dmul_rn(dr, dr), __dmul_rn(dg, dg)), __dmul_rn(db, db)));
}

// gray_pix: valid wherever in bounds              (VectorImage::pixel, vectorimage.cpp:115-119)
// gray_two: NaN unless mask WHITE and x+1<w,y+1<h (mask test twoviewstereo.cpp:920-924 +
//                                                  VectorImage::sample validity, vectorimage.cpp:132)
// gray_msk: NaN unless mask WHITE                 (cost_sad right taps, twoviewstereo.cpp:877,885)
// edges[e][p]: colour distance between pixel p and p + (1,0), (0,1), (1,1), (-1,1); +INF when the
//              other end is outside the image (an edge the geodesic sweeps may not use).
__global__ void prep_view_kernel(const uchar4 *__restrict__ rgba, const uint8_t *__restrict__ mask, int w, int h,
                                 double *__restrict__ gray_pix, double *__restrict__ gray_two,
                                 double *__restrict__ gray_msk, double *__restrict__ edges,
                                 float *__restrict__ gray_pix_f, int pitch_f) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= w * h) return;
    const int x = i % w, y = i / w;
    const uchar4 c = rgba[i];
    const double g = gray_of(c);
    const bool white = mask[i] == 255;
    gray_pix[i] = g;
    // FP32 copy read by the screening pass of match_mvs_screen_kernel; its row pitch is a power of
    // two (screen_pitch) so that the 25 window loads are one base register + immediate offsets
    gray_pix_f[(size_t)y * pitch_f + x] = (float)g;
    gray_msk[i] = white ? g : qnan();
    gray_two[i] = (white && x + 1 < w && y + 1 < h) ? g : qnan();
    const size_t n = (size_t)w * h;
    edges[i] = (x + 1 < w) ? color_dist(c, rgba[i + 1]) : dinf();
    edges[n + i] = (y + 1 < h) ? color_dist(c, rgba[i + w]) : dinf();
    edges[2 * n + i] = (x + 1 < w && y + 1 < h) ? color_dist(c, rgba[i + w + 1]) : dinf();
    edges[3 * n + i] = (x >= 1 && y + 1 < h) ? color_dist(c, rgba[i + w - 1]) : dinf();
}

// Rows [y0, y0 + ny) of the [6][h][w] ray table (a rank that owns a row band computes only its rows).
__global__ void rays_kernel(sr_camera cam, int w, int h, int y0, int ny, double scale, double *__restrict__ rays) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= w * ny) return;
    const int x = k % w, y = y0 + k / w;
    const size_t i = (size_t)y * w + x;
    d3 s, d;
    cam_unproject(cam, (x + 0.5) / scale, (y + 0.5) / scale, s, d);
    const size_t n = (size_t)w * h;
    rays[i] = s.x;
    rays[n + i] = s.y;
    rays[2 * n + i] = s.z;
    rays[3 * n + i] = d.x;
    rays[4 * n + i] = d.y;
    rays[5 * n + i] = d.z;
}

__global__ void project_points_kernel(sr_camera cam, int n, const double *__restrict__ xyz, double *__restrict__ out_xy,
                                      int32_t *__restrict__ out_ok) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    double u = qnan(), v = qnan();
    const bool ok = cam_project(cam, d3{xyz[3 * i], xyz[3 * i + 1], xyz[3 * i + 2]}, u, v);
    out_xy[2 * i] = ok ? u : qnan();
    out_xy[2 * i + 1] = ok ? v : qnan();
    out_ok[i] = ok;
}

// ---------------------------------------------------------------------------------------------
// Stage (1): tap-volume build.
struct BuildArgs {
    sr_camera nbr;               // target view
    double prin[3], C[3];        // reference view principal direction and centre
    const double *rays;          // [6][h][w] of the reference view
    const double *depth_table;   // [D] depthFromLabel(d)
    const uint8_t *ref_mask;     // [h][w]
    const uint8_t *nbr_mask;     // [h][w]
    int32_t *taps;               // [D][rows][w] for this neighbour
    int w, h, row0, rows, D, d_chunk;
    double scale;
    int mvs;                     // 1: tap = trunc(p*scale), neighbour mask must be WHITE
                                 // 0: tap = trunc(p*scale - 0.5)
};

__global__ void __launch_bounds__(128) build_kernel(const BuildArgs a) {
    const int pid = blockIdx.x * blockDim.x + threadIdx.x;
    if (pid >= a.rows * a.w) return;
    const int x = pid % a.w, y = a.row0 + pid / a.w;
    const size_t pix = (size_t)y * a.w + x;
    if (a.ref_mask[pix] != 255) return;  // match_kernel never reads taps of masked-out pixels
    const size_t n = (size_t)a.w * a.h;
    const d3 src = {a.rays[pix], a.rays[n + pix], a.rays[2 * n + pix]};
    const d3 dir = {a.rays[3 * n + pix], a.rays[4 * n + pix], a.rays[5 * n + pix]};
    // pointFromDepth (multiviewstereo.cpp:740-750): Plane3d(normal, C + normal*depth) then
    // intersect(); everything independent of the label is hoisted.
    const d3 prin = ld3(a.prin);
    const d3 nrm = normalized(prin);
    const double nd = dot(nrm, dir);
    const bool ray_ok = !(fabs(nd) < 1e-10);
    const double inv_nd = 1.0 / nd;
    const double nC = dot(nrm, ld3(a.C)), npn = dot(nrm, prin), nn = dot(nrm, nrm), ns = dot(nrm, src);
    const bool exact = !a.nbr.is_refractive;  // uniform: op-for-op IEEE path (see cam_project_exact)
    const RayInView rv = {fmul3(a.nbr.R, src) + ld3(a.nbr.t), fmul3(a.nbr.R, dir)};
    const ProjConsts pc = proj_consts(a.nbr);
    const double scale = a.scale, shift = a.mvs ? 0.0 : -0.5;
    const int d0 = blockIdx.y * a.d_chunk;
    const int d1 = min(d0 + a.d_chunk, a.D);
    const size_t plane = (size_t)a.rows * a.w;
    float w0 = -1.0f, w1 = -1.0f;
#pragma unroll 1
    for (int d = d0; d < d1; ++d) {
        int32_t tap = TAP_NONE;
        const double depth = a.depth_table[d];
        bool ok = false;
        double u, v;
        if (exact) {
            // Plane3d(normal, C + normal*depth); intersect(ray, plane, p)  — reference op order
            const d3 x0 = ld3(a.C) + depth * prin;
            const double dist = dot(nrm, x0);
            if (ray_ok) {
                const double t = dot(nrm, dist * nrm - src) / nd;
                if (!(t < 1e-10)) {
                    cam_project_exact(a.nbr, src + t * dir, u, v);
                    ok = true;
                }
            }
        } else {
            const double dist = fma(depth, npn, nC);
            const double t = fma(dist, nn, -ns) * inv_nd;
            if (ray_ok && !(t < 1e-10)) ok = cam_project_local(a.nbr, pc, faxpy(t, rv.Ld, rv.Ls), w0, w1, u, v);
        }
        if (ok) {
            int tx, ty;
            if (exact) {
                tx = to_int_x86(u * scale + shift);
                ty = to_int_x86(v * scale + shift);
            } else {
                tx = to_int_x86(fma(u, scale, shift));
                ty = to_int_x86(fma(v, scale, shift));
            }
            bool keep = true;
            if (a.mvs) {  // multiviewstereo.cpp:787: only WHITE neighbour-mask pixels are candidates
                keep = tx >= 0 && ty >= 0 && tx < a.w && ty < a.h && a.nbr_mask[(size_t)ty * a.w + tx] == 255;
            }
            if (keep) {
                tx = max(-TAP_CLAMP, min(TAP_CLAMP, tx));
                ty = max(-TAP_CLAMP, min(TAP_CLAMP, ty));
                tap = (int32_t)(((uint32_t)(ty & 0xffff) << 16) | (uint32_t)(tx & 0xffff));
            }
        }
        a.taps[(size_t)d * plane + pid] = tap;
    }
}

// ---------------------------------------------------------------------------------------------
// Support weights -> W[k][pid], k = (row+R)*(2R+1) + (col+R), pid = pixel index inside the band.
struct WeightArgs {
    const uchar4 *rgba;
    const uint8_t *mask;
    const double *edges;   // [4][h][w]
    double *W;             // [WN][npix]
    int w, h, row0, rows, radius;
    // list mode (sr_compute_weights): explicit window centres instead of a row band; no mask test
    const int32_t *list_x, *list_y;
    int list_n;
};
__device__ __forceinline__ bool weight_centre(const WeightArgs &a, int pid, size_t &npix, int &cx, int &cy) {
    if (a.list_x) {
        npix = (size_t)a.list_n;
        if (pid >= a.list_n) return false;
        cx = a.list_x[pid];
        cy = a.list_y[pid];
        return true;
    }
    npix = (size_t)a.rows * a.w;
    if (pid >= (int)npix) return false;
    cx = pid % a.w;
    cy = a.row0 + pid / a.w;
    return a.mask[(size_t)cy * a.w + cx] == 255;
}

// AdaptiveWeight::weight (stereo/adaptiveweight.cpp:62-79) for every tap of every band pixel.
__global__ void __launch_bounds__(128) weights_adaptive_kernel(const WeightArgs a) {
    extern __shared__ double dw[];  // distance_weights[i] = exp(-i / radius), adaptiveweight.cpp:36-38
    const int R = a.radius, WS = 2 * R + 1;
    if ((int)threadIdx.x <= R) dw[threadIdx.x] = exp(-(double)threadIdx.x / (1.0 * R));
    __syncthreads();
    const int pid = blockIdx.x * blockDim.x + threadIdx.x;
    size_t npix;
    int cx, cy;
    if (!weight_centre(a, pid, npix, cx, cy)) return;
    const bool centre_ok = cx >= 0 && cy >= 0 && cx < a.w && cy < a.h;
    const uchar4 c = centre_ok ? a.rgba[(size_t)cy * a.w + cx] : make_uchar4(0, 0, 0, 0);
    for (int row = -R; row <= R; ++row) {
        const int y = cy + row;
        for (int col = -R; col <= R; ++col) {
            const int x = cx + col;
            double wt = 0.0;
            if (centre_ok && x >= 0 && y >= 0 && x < a.w && y < a.h) {  // invalid centre: NaN weight -> 0
                const double diff = color_dist(c, a.rgba[(size_t)y * a.w + x]);
                wt = (dw[abs(row)] * dw[abs(col)]) * exp(-diff / 10.0);
            }
            a.W[(size_t)((row + R) * WS + (col + R)) * npix + pid] = wt;
        }
    }
}

// GeodesicWeight::init_weights (stereo/geodesicweight.cpp:59-131): 3 x (forward + backward)
// in-place raster sweeps over the window.  One thread per reference pixel; the (2R+1)^2 grid is
// the thread's own column of W (coalesced across the warp), the update order is the
// reference's, and the colour distances come from the precomputed edge planes, so the result is
// the reference's up to the final exp().  Cells whose pixel is outside the image are never
// updated and every edge into them is +INF, which reproduces the reference's validity tests.
// SMEM: the grid lives in shared memory ([cell][thread], conflict-free) during the sweeps and is
// written to W once at the end — used when (2R+1)^2 * 128 doubles fit (R <= 2); otherwise the grid
// is the thread's column of W itself.
// fmin(a, b) for operands that are never NaN (distances: finite or +INF, never negative zero) as
// compare + select: min.f64 expands to 7 instructions on sm_100a (NaN canonicalisation), and the
// compiler turns `b < a ? b : a` back into min.f64, hence PTX.
__device__ __forceinline__ double min_sel(double a, double b) {
    double r;
    asm("{\n\t.reg .pred p;\n\tsetp.lt.f64 p, %2, %1;\n\tselp.f64 %0, %2, %1, p;\n\t}" : "=d"(r) : "d"(a), "d"(b));
    return r;
}

// RT > 0: the radius as a compile-time constant (the sweeps are unrolled: every cell index, shared-memory
// offset and window-edge test folds away); RT = 0: a.radius.  Same updates in the same order either way.
#ifndef SR_GEO_MINBLOCKS  // resident blocks per SM the register allocation must allow (6: 80 registers, no spills;
#define SR_GEO_MINBLOCKS 6  // unbounded the unrolled sweeps take 96, bounded to 8 blocks they spill)
#endif
#define SR_GEO_BOUNDS __launch_bounds__(128, SR_GEO_MINBLOCKS)
template <bool SMEM, int RT>
__global__ void SR_GEO_BOUNDS weights_geodesic_kernel(const WeightArgs a) {
    extern __shared__ double grid_s[];
    const int R = RT > 0 ? RT : a.radius, WS = 2 * R + 1;
    const int pid = blockIdx.x * blockDim.x + threadIdx.x;
    size_t npix;
    int cx, cy;
    if (!weight_centre(a, pid, npix, cx, cy)) return;
    double *const out = a.W + pid;
    const size_t out_stride = npix;
    double *c = SMEM ? (grid_s + threadIdx.x) : out;
    if (SMEM) npix = 128;  // stride of the grid the sweeps walk on
    for (int k = 0; k < WS * WS; ++k) c[(size_t)k * npix] = 1000000.0;
    c[(size_t)(R * WS + R) * npix] = 0.0;
    const size_t n = (size_t)a.w * a.h;
    const double *eE = a.edges, *eS = a.edges + n, *eSE = a.edges + 2 * n, *eSW = a.edges + 3 * n;
    const int w = a.w, h = a.h;
    // forward pass: neighbours (-1,-1), (0,-1), (1,-1), (-1,0)
    auto forward = [&](int y, int x) {
        const int py = cy + y, px = cx + x;
        if (py < 0 || py >= h || px < 0 || px >= w) return;
        const size_t p = (size_t)py * w + px;
        const int k = (y + R) * WS + (x + R);
        double wt = c[(size_t)k * npix];
        if (y > -R && py >= 1) {  // row above (inside the image): edges stored at the upper pixel
            if (x > -R && px >= 1) wt = min_sel(wt, c[(size_t)(k - WS - 1) * npix] + eSE[p - w - 1]);
            wt = min_sel(wt, c[(size_t)(k - WS) * npix] + eS[p - w]);
            if (x < R && px + 1 < w) wt = min_sel(wt, c[(size_t)(k - WS + 1) * npix] + eSW[p - w + 1]);
        }
        if (x > -R && px >= 1) wt = min_sel(wt, c[(size_t)(k - 1) * npix] + eE[p - 1]);
        c[(size_t)k * npix] = wt;
    };
    // backward pass: neighbours (-1,1), (0,1), (1,1), (1,0)
    auto backward = [&](int y, int x) {
        const int py = cy + y, px = cx + x;
        if (py < 0 || py >= h || px < 0 || px >= w) return;
        const size_t p = (size_t)py * w + px;
        const int k = (y + R) * WS + (x + R);
        double wt = c[(size_t)k * npix];
        if (y < R) {  // row below: edges stored at this pixel
            if (x > -R) wt = min_sel(wt, c[(size_t)(k + WS - 1) * npix] + eSW[p]);
            wt = min_sel(wt, c[(size_t)(k + WS) * npix] + eS[p]);
            if (x < R) wt = min_sel(wt, c[(size_t)(k + WS + 1) * npix] + eSE[p]);
        }
        if (x < R) wt = min_sel(wt, c[(size_t)(k + 1) * npix] + eE[p]);
        c[(size_t)k * npix] = wt;
    };
#pragma unroll 1
    for (int iter = 0; iter < 3; ++iter) {
        if (RT > 0) {
#pragma unroll
            for (int y = -RT; y <= RT; ++y)
#pragma unroll
                for (int x = -RT; x <= RT; ++x) forward(y, x);
#pragma unroll
            for (int y = RT; y >= -RT; --y)
#pragma unroll
                for (int x = RT; x >= -RT; --x) backward(y, x);
        } else {
#pragma unroll 1
            for (int y = -R; y <= R; ++y)
#pragma unroll 1
                for (int x = -R; x <= R; ++x) forward(y, x);
#pragma unroll 1
            for (int y = R; y >= -R; --y)
#pragma unroll 1
                for (int x = R; x >= -R; --x) backward(y, x);
        }
    }
    for (int k = 0; k < WS * WS; ++k) out[(size_t)k * out_stride] = exp(-c[(size_t)k * npix] / 50.0);
}

// ---------------------------------------------------------------------------------------------
// Stages (2)+(3): windowed cost + WTA.
struct MatchArgs {
    const uint8_t *maskL;           // reference view mask
    const double *grayL;            // reference taps  (gray_pix for C1, gray_two for C2/C3)
    const double *grayR[SR_MAX_NBRS];  // neighbour taps (gray_pix C1, gray_two C2, gray_msk C3)
    const float *grayRf[SR_MAX_NBRS];  // FP32 copies of gray_pix (screening pass, MVS selection only)
    int pitch_f;                       // row pitch of the FP32 planes, in floats (screen_pitch(w))
    const double *W;                // [WN][rows*w] support weights of this band
    const int32_t *taps;            // [nbr][D][rows][w]
    const double *depth_table;      // [D]
    int32_t *out_index;             // [h][w]
    double *out_depth;              // [h][w]
    double *out_best;               // [h][w]
    float *out_volume;              // [nbr][D][rows][w] or null
    double *out_peaks;              // [9][2][h*w] or null: the K = 9 largest (ncc, depth) pairs per pixel,
                                    // ascending (CostFunction::peakPairs, multiviewstereo.cpp:479-482,600-602)
    int w, h, row0, rows, D, num_nbrs;
    int win_w, win_h;               // w - 2*radius, h - 2*radius: tap positions whose whole window is inside
    int tap_planes;                 // planes per neighbour in `taps` when it is larger than D (curve mode), else 0
    int select_kind;
    int depth_up;                   // depth_table is increasing in the label (max_depth > min_depth)
    // curve mode (sr_curve.cuh): the "labels" are the candidates of the rasterised epipolar curve and
    // a candidate's depth is the closest approach of the two viewing rays
    int curve;
    const double *raysL;               // [6][h][w] rays of the reference view
    const double *raysR[SR_MAX_NBRS];  // [6][h][w] rays of the neighbour views
    double camR[9], camT[3];           // reference camera: fromGlobalToLocal (camera.cpp:346-348)
    unsigned long long *stats;      // optional [8]: pixels, screened, forced, verified, all_slow (debug)
    int use_screen;                 // MVS selection: FP32 screen + FP64 verify (sr_match_screen.cuh)
    double second_best_factor, ncc_threshold;
};

template <int G>
__device__ __forceinline__ double group_sum(double v, unsigned gmask) {
#pragma unroll
    for (int o = G / 2; o > 0; o >>= 1) v += __shfl_xor_sync(gmask, v, o);
    return v;
}
template <int G>
__device__ __forceinline__ int group_sum_i(int v, unsigned gmask) {
#pragma unroll
    for (int o = G / 2; o > 0; o >>= 1) v += __shfl_xor_sync(gmask, v, o);
    return v;
}

// The exact tap filter of the reference (a tap counts only if both pixels are valid and the
// weight exceeds 1e-10), used for the few windows that touch an image border or an invalid
// (masked) pixel.  Runtime loops, weights re-read from W: small code, no register arrays.
template <int R, int G, int COST>
// wloc: this pixel's support weights by tap index in shared memory (match_kernel with G > 1 lanes per pixel
// stages them there: in the [tap][pixel] layout of W the G lanes of a pixel read G different planes, 32 sectors
// per request, for every border label again), or null: read W.
__device__ __noinline__ double slow_cost(const MatchArgs &a, const double *__restrict__ gR, int x, int y, int tx, int ty,
                                         int pid, int sub, unsigned gmask, const double *wloc = nullptr) {
    constexpr int WS = 2 * R + 1, WN = WS * WS;
    constexpr bool NCC = (COST != SR_COST_SAD_TWOVIEW);
    const int w = a.w, h = a.h;
    const size_t npix = (size_t)a.rows * w;
    // A window that lies entirely outside the neighbour image has no valid tap: the filter below would find
    // cnt = 0, tw = 0.  (Rectified pairs: every label whose disparity exceeds the pixel's column by more than
    // the radius — a tenth of cfg3's evaluations, each of which walked all (2R+1)^2 taps to learn that.)
    if (tx + R < 0 || ty + R < 0 || tx - R >= w || ty - R >= h) return (COST == SR_COST_NCC_MVS) ? 0.0 : 1000.0;
    double mL = 0.0, mR = 0.0, tw = 0.0;
    int cnt = 0;
    auto first = [&](double gl, double gr, double wt) {
        if (gl == gl && gr == gr && wt > 1e-10) {
            if (NCC) {
                mL += wt * gl;
                mR += wt * gr;
            } else {
                mL += wt * fmin(120.0, fabs(gl - gr));
            }
            tw += wt;
            ++cnt;
        }
    };
    // One lane per window (G = 1, the thread-per-pixel screen's verifications): the taps with both pixels
    // inside their images are a sub-rectangle of the window, walked in the reference's row-major order with
    // running pointers instead of eight bound tests and three 64-bit index products per tap.
    const int row_lo = max(-R, max(-ty, -y)), row_hi = min(R, min(h - 1 - ty, h - 1 - y));
    const int col_lo = max(-R, max(-tx, -x)), col_hi = min(R, min(w - 1 - tx, w - 1 - x));
    auto walk = [&](auto &&body) {
#pragma unroll 1
        for (int row = row_lo; row <= row_hi; ++row) {
            const double *__restrict__ pl = a.grayL + ((size_t)(y + row) * w + (x + col_lo));
            const double *__restrict__ pr = gR + ((size_t)(ty + row) * w + (tx + col_lo));
            const double *__restrict__ pw = a.W + ((size_t)((row + R) * WS + (col_lo + R)) * npix + pid);
#pragma unroll 1
            for (int col = col_lo; col <= col_hi; ++col, ++pl, ++pr, pw += npix) body(*pl, *pr, *pw);
        }
    };
    // G lanes per window (taps dealt round-robin): four of the lane's taps per step, their loads issued
    // together (a tap outside either image reads as NaN, which the filter skips) and consumed in tap order —
    // the loop used to wait for each tap's three loads in turn, at 8 warps per SM (cfg3: 70 % of the kernel).
    constexpr int UNR = 4;
    auto strided = [&](auto &&body) {
        // (`a` arrives by reference: its pointers are read once here, not for every tap)
        const double *__restrict__ const gLp = a.grayL;
        const double *__restrict__ const Wp = a.W;
#pragma unroll 1
        for (int k0 = sub; k0 < WN; k0 += UNR * G) {
            double gl[UNR], gr[UNR], wt[UNR];
            bool in[UNR];
#pragma unroll
            for (int u = 0; u < UNR; ++u) {  // unconditional loads from clamped addresses: nothing to branch around
                const int k = min(k0 + u * G, WN - 1);
                const int row = k / WS - R, col = k % WS - R;
                const int xr = tx + col, yr = ty + row, xl = x + col, yl = y + row;
                in[u] = k0 + u * G < WN && !(xr < 0 || yr < 0 || xr >= w || yr >= h || xl < 0 || yl < 0 || xl >= w || yl >= h);
                const size_t il = in[u] ? (size_t)yl * w + xl : 0, ir = in[u] ? (size_t)yr * w + xr : 0;
                gl[u] = gLp[il];
                gr[u] = gR[ir];
                wt[u] = wloc ? wloc[k] : Wp[(size_t)k * npix + pid];
            }
#pragma unroll
            for (int u = 0; u < UNR; ++u) body(in[u] ? gl[u] : __longlong_as_double(0x7ff8000000000000ll), gr[u], wt[u]);
        }
    };
    if (G == 1) walk(first);
    else strided(first);
    mL = group_sum<G>(mL, gmask);
    mR = group_sum<G>(mR, gmask);
    tw = group_sum<G>(tw, gmask);
    cnt = group_sum_i<G>(cnt, gmask);
    if (!NCC) return (cnt <= 4 || tw <= 1e-10) ? 1000.0 : mL / tw;
    if (tw < 1e-10) return (COST == SR_COST_NCC_MVS) ? 0.0 : 1000.0;
    mL /= tw;
    mR /= tw;
    double q1 = 0.0, q2 = 0.0, q3 = 0.0;
    auto second = [&](double gl, double gr, double wt) {
        if (gl == gl && gr == gr && wt > 1e-10) {
            const double pl = wt * gl - mL, pr = wt * gr - mR;
            q1 += pl * pr;
            q2 += pl * pl;
            q3 += pr * pr;
        }
    };
    if (G == 1) walk(second);
    else strided(second);
    q1 = group_sum<G>(q1, gmask);
    q2 = group_sum<G>(q2, gmask);
    q3 = group_sum<G>(q3, gmask);
    if (COST == SR_COST_NCC_MVS) return (q2 * q3 < 1e-10) ? 0.0 : q1 / sqrt(q2 * q3);
    const double v = 255.0 * (1.0 - fabs(q1) / sqrt(q2 * q3));
    return (v < 120.0) ? v : 120.0;
}

__device__ double curve_depth(const double *__restrict__ raysA, const double *__restrict__ raysB, size_t n, size_t pixA,
                              size_t pixB, const double *R, const double *t);  // sr_curve.cuh

#ifndef SR_MATCH_MINBLOCKS
#define SR_MATCH_MINBLOCKS 3
#endif
#ifndef SR_MATCH_SMEM_C1
#define SR_MATCH_SMEM_C1 1
#endif
constexpr int TAP_CHUNK = 16;  // labels per cp.async stage of the tap stream

// The tap volume is read exactly once: fetch it with an L2 evict-first policy so that it does
// not push the (re-used) neighbour gray planes out of the 126 MB L2.
__device__ __forceinline__ uint64_t l2_evict_first_policy() {
    uint64_t pol;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
__device__ __forceinline__ void cp_async4(void *smem_dst, const void *gmem_src, uint64_t pol) {
    asm volatile("cp.async.ca.shared.global.L2::cache_hint [%0], [%1], 4, %2;" ::"r"((unsigned)__cvta_generic_to_shared(smem_dst)),
                 "l"(gmem_src), "l"(pol));
}
// (shared-window address already converted: callers that issue many copies convert the base once)
__device__ __forceinline__ void cp_async4_saddr(unsigned smem_addr, const void *gmem_src, uint64_t pol) {
    asm volatile("cp.async.ca.shared.global.L2::cache_hint [%0], [%1], 4, %2;" ::"r"(smem_addr), "l"(gmem_src), "l"(pol));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
    asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory");
}

// R: window radius; G: lanes cooperating on one reference pixel (taps are dealt round-robin to
// the G lanes and live in registers); COST: SR_COST_*.
//
// Inner-loop shape (what the FP64 pipe sees): per (label, neighbour) one streaming pass over the
// lane's taps — gr = neighbour gray; p = w*gr; S1 += p; S2 += p*p; S3 += (w*dl)*gr — i.e. 4
// FP64 instructions and one 8-byte L1 load per tap, then a ~25-instruction tail.
// The tap volume streams HBM -> shared memory through a two-stage cp.async ring (TAP_CHUNK
// labels per stage, each thread fetching its own pixel's taps: a warp moves 128 contiguous
// bytes per label), so the HBM latency of the volume is never on a warp's critical path.
template <int R, int G, int COST>
__global__ void __launch_bounds__(128, (R <= 2) ? SR_MATCH_MINBLOCKS : 2) match_kernel(const __grid_constant__ MatchArgs a) {
    constexpr int WS = 2 * R + 1;
    constexpr int WN = WS * WS;
    constexpr int TPL = (WN + G - 1) / G;
    constexpr bool NCC = (COST != SR_COST_SAD_TWOVIEW);
    constexpr int PIX_PER_BLOCK = 128 / G;
    __shared__ int32_t tap_ring[2][TAP_CHUNK][128];
    // thread-per-pixel variant: the second per-tap constant (w*dl / gl) lives in shared memory,
    // [tap][thread] so a warp's LDS.64 is conflict-free; this halves the register arrays and lets
    // 4 blocks (16 warps) share an SM, which is what hides the FP64 issue latency.
    constexpr bool SMEM_C1 = (G == 1) && (SR_MATCH_SMEM_C1 != 0);
    __shared__ double c1s[SMEM_C1 ? TPL : 1][128];
    // G > 1: the pixel's raw support weights by tap index, for slow_cost (dynamic: PIX_PER_BLOCK * WN doubles);
    // every lane reads back only what it wrote (tap k belongs to lane k % G in both places)
    extern __shared__ double wstage[];
    double *const wloc = (G > 1) ? wstage + (size_t)(threadIdx.x / G) * WN : nullptr;

    const int lane = threadIdx.x & 31;
    const int sub = threadIdx.x % G;
    const unsigned gmask = (G == 32) ? 0xffffffffu : (((1u << G) - 1u) << (lane & ~(G - 1)));
    const int pid = blockIdx.x * PIX_PER_BLOCK + threadIdx.x / G;
    if (pid >= a.rows * a.w) return;  // whole group leaves together
    const int x = pid % a.w, y = a.row0 + pid / a.w;
    const size_t pix = (size_t)y * a.w + x;
    const int w = a.w, h = a.h;
    const size_t npix = (size_t)a.rows * w;

    if (a.maskL[pix] != 255) {  // twoviewstereo.cpp:269-271 (NaN) / multiviewstereo.cpp:559,565 (INF)
        if (sub == 0) {
            a.out_index[pix] = SR_INDEX_MASKED;
            a.out_depth[pix] = (a.select_kind == SR_SELECT_MVS) ? dinf() : qnan();
            a.out_best[pix] = qnan();
        }
        return;
    }

    // ---- reference-window invariants (hoisted out of the label sweep) -----------------------
    // wt[i]: support weight of this lane's i-th tap (0 for taps the reference skips on the
    //        reference side: invalid pixel or weight <= 1e-10);
    // c1[i]: NCC: wt*(wt*gl - meanL);  SAD: gl.
    double wt[TPL], c1[TPL];
    double totW = 0.0, SL = 0.0;
    int nact = 0;
#pragma unroll
    for (int i = 0; i < TPL; ++i) {
        const int k = sub + G * i;
        const int row = k / WS - R, col = k % WS - R;
        const int xl = x + col, yl = y + row;
        double gl = qnan(), wv = 0.0;
        if (k < WN && xl >= 0 && yl >= 0 && xl < w && yl < h) {
            gl = a.grayL[(size_t)yl * w + xl];
            wv = a.W[(size_t)k * npix + pid];
        }
        if (G > 1 && k < WN) wloc[k] = wv;
        const bool active = (gl == gl) && (wv > 1e-10);
        wt[i] = active ? wv : 0.0;
        c1[i] = active ? gl : 0.0;
        if (active) {
            totW += wv;
            SL += wv * gl;
            ++nact;
        }
    }
    totW = group_sum<G>(totW, gmask);
    SL = group_sum<G>(SL, gmask);
    nact = group_sum_i<G>(nact, gmask);
    const double meanL = SL / totW;
    const double inv_totW = 1.0 / totW;
    double s2 = 0.0, SD = 0.0;
    if (NCC) {
#pragma unroll
        for (int i = 0; i < TPL; ++i) {
            const double dl = (wt[i] > 0.0) ? wt[i] * c1[i] - meanL : 0.0;
            s2 += dl * dl;
            SD += dl;
            c1[i] = wt[i] * dl;
        }
        s2 = group_sum<G>(s2, gmask);
        SD = group_sum<G>(SD, gmask);
    }
    if (SMEM_C1) {
#pragma unroll
        for (int i = 0; i < TPL; ++i) c1s[i][threadIdx.x] = c1[i];  // only this thread reads its column
    }
    const bool degenerate = (COST == SR_COST_SAD_TWOVIEW) ? (nact <= 4 || totW <= 1e-10) : (totW < 1e-10);
    const double dnact = (double)nact;
    // Error bar of the one-pass NCC (fast_one) against the reference's two passes, in FP64 (u = 2^-53).
    //   S1 = sum p, S2 = sum p^2, S3 = sum (w dl) g with p = w g over the lane's taps in two chains, then
    //   S + T and the lane butterfly: at most M roundings per term.  With A = S2 + 2 |meanR S1| + nact meanR^2
    //   (S1 = meanR totW, so A = S2 + (2 totW + nact) meanR^2) and kappa = A / s3:
    //     |dS1| <= M u S1 (terms >= 0),  |dS2| <= M u S2,  |dS3| <= M u sum |dl p| <= M u sqrt(s2 S2)
    //     meanR = S1 / totW: (M + 2) u relative;  s3 = S2 - 2 meanR S1 + nact meanR^2 (two roundings),
    //     whose derivative in meanR is 2 (nact meanR - S1):      |ds3| <= (3M + 7) u A
    //     SD = sum dl (one chain of <= 2M), |SD| <= sqrt(nact s2):  |d(meanR SD)| <= (3M + 3) u |meanR| sqrt(nact s2)
    //     s1 = S3 - meanR SD:                                       |ds1| <= u sqrt(s2) [(M + 1) sqrt(S2) + (3M + 3) |meanR| sqrt(nact)]
    //   rho = s1 / sqrt(s2 s3) with |rho| <= 1 (Cauchy-Schwarz), S2 <= A and nact meanR^2 <= A:
    //     |drho| <= |ds1| / sqrt(s2 s3) + |ds3| / (2 s3) + |ds2| / (2 s2) + rsqrt and the last products
    //            <= u [(4M + 4) sqrt(kappa) + (1.5M + 3.5) kappa + M + 4]
    //            <= u [(3.5M + 5.5) kappa + 3M + 6]                     (sqrt(kappa) <= (1 + kappa) / 2)
    //   and, as A = s3 + 4 totW meanR^2 = s3 + 4 meanR S1, the bar exceeds RHO_TOL iff
    //     meanR S1 * 4 u (3.5M + 5.5) / (RHO_TOL - u (6.5M + 11.5)) > s3             (two instructions a label)
    //   A label whose bar exceeds RHO_TOL (5e-11 on the 255-scaled two-view cost, half the reference's 1e-10
    //   selection margin; the MVS NCC is then within 2e-13) returns NaN: slow_cost, the reference's two-pass
    //   filter, decides.  The bar is a worst case, and the one-pass error is a few u kappa at most in practice
    //   (measured on the CPU: <= 40 u kappa, r = 1..16), so RHO_TOL is set well above the observed errors to
    //   keep the fallback rare: kappa stays near 1 under adaptive weights (the reference's w g - meanR keeps s3
    //   large), under geodesic weights it is mostly below the ~20-30 the bar allows (flagged: < 1 % of the labels
    //   of a textured rectified pair, 6 % at r = 2 on an arc scene), and flat or smooth neighbour windows under
    //   geodesic weights (kappa in the hundreds to millions, where s3 is a true variance) are flagged whole.
    constexpr int M = (TPL + 1) / 2 + 1 + ((G >= 2) + (G >= 4) + (G >= 8) + (G >= 16) + (G >= 32));
    constexpr double U = 1.1102230246251565e-16, RHO_TOL = 5e-11 / 255.0;
    constexpr double ERR_K = U * (3.5 * M + 5.5), ERR_ROOM = RHO_TOL - U * (6.5 * M + 11.5);
    static_assert(ERR_ROOM > 0.0, "RHO_TOL below the rounding floor of the window");
    constexpr double ERR_C = 4.0 * ERR_K / ERR_ROOM;  // flag iff ERR_C meanR S1 > s3

    // one label, fast path: whole neighbour window in bounds; one streaming pass over the taps.
    // Returns NaN iff a neighbour tap was invalid (NaN), the NCC's error bar exceeds RHO_TOL or
    // the two-view q is out of range — then the exact tap filter (slow_cost) decides.  A legitimately evaluated cost is never NaN
    // (two-view: NaN -> 120 as std::min does; MVS: q < 1e-10 -> 0).
    auto fast_one = [&](const double *__restrict__ base) -> double {
        double S1 = 0.0, S2 = 0.0, S3 = 0.0, T1 = 0.0, T2 = 0.0, T3 = 0.0;
        if (G == 1) {
            // thread-per-pixel: row pointers + compile-time column offsets
#pragma unroll
            for (int row = 0; row < WS; ++row) {
                const double *__restrict__ rp = base + (row - R) * w;
#pragma unroll
                for (int col = 0; col < WS; ++col) {
                    const int i = row * WS + col;
                    const double gr = rp[col - R];
                    const double ci = SMEM_C1 ? c1s[i][threadIdx.x] : c1[i];
                    if (NCC) {
                        const double p = wt[i] * gr;
                        if (i & 1) {
                            T1 += p;
                            T2 = fma(p, p, T2);
                            T3 = fma(ci, gr, T3);
                        } else {
                            S1 += p;
                            S2 = fma(p, p, S2);
                            S3 = fma(ci, gr, S3);
                        }
                    } else {
                        const double ad = fabs(ci - gr);  // (ad > 120 ? 120 : ad) keeps a NaN tap visible
                        if (i & 1) T1 = fma(wt[i], (ad > 120.0) ? 120.0 : ad, T1);
                        else S1 = fma(wt[i], (ad > 120.0) ? 120.0 : ad, S1);
                    }
                }
            }
        } else {
#pragma unroll
            for (int i = 0; i < TPL; ++i) {
                const int k = sub + G * i;
                if (k < WN) {
                    const double gr = base[(k / WS - R) * w + (k % WS - R)];
                    if (NCC) {
                        const double p = wt[i] * gr;
                        if (i & 1) {
                            T1 += p;
                            T2 = fma(p, p, T2);
                            T3 = fma(c1[i], gr, T3);
                        } else {
                            S1 += p;
                            S2 = fma(p, p, S2);
                            S3 = fma(c1[i], gr, S3);
                        }
                    } else {
                        const double ad = fabs(c1[i] - gr);
                        if (i & 1) T1 = fma(wt[i], (ad > 120.0) ? 120.0 : ad, T1);
                        else S1 = fma(wt[i], (ad > 120.0) ? 120.0 : ad, S1);
                    }
                }
            }
        }
        S1 = group_sum<G>(S1 + T1, gmask);
        if (!NCC) {
            if (S1 != S1) return qnan();
            return degenerate ? 1000.0 : S1 * inv_totW;
        }
        S2 = group_sum<G>(S2 + T2, gmask);
        S3 = group_sum<G>(S3 + T3, gmask);
        // gray_pix (COST NCC_MVS) holds no NaN inside the image: no invalid-tap test needed there
        if (COST != SR_COST_NCC_MVS && (S1 != S1 || S3 != S3)) return qnan();
        if (degenerate) return (COST == SR_COST_NCC_MVS) ? 0.0 : 1000.0;
        const double meanR = S1 * inv_totW;
        const double s1 = fma(-meanR, SD, S3);
        const double s3 = fma(dnact * meanR, meanR, fma(-2.0 * meanR, S1, S2));
        const double q = s2 * s3;
        if (COST == SR_COST_NCC_MVS) {
            if (fma(ERR_C * meanR, S1, -s3) > 0.0) return qnan();  // error bar > RHO_TOL
            return (q < 1e-10) ? 0.0 : s1 * fast_rsqrt(q);
        }
        // two-view: 255*(1 - |s1|/sqrt(q)); an error bar > RHO_TOL, or q <= 0, denormal or huge (the IEEE
        // inf/NaN -> 120 cases): slow_cost
        if (fma(ERR_C * meanR, S1, -s3) > 0.0 || !(q > 1e-280 && q < 1e280)) return qnan();
        const double v = 255.0 * (1.0 - fabs(s1) * fast_rsqrt(q));
        return (v < 120.0) ? v : 120.0;
    };

    // ---- label sweep -------------------------------------------------------------------------
    double minCost = dinf(), secondBest = dinf();  // two-view selection
    double bestC = 0.0;                            // MVS selection
    double bestZ = -1.0;                           // MVS curve mode: depth of the winning candidate
    int bestIdx = SR_INDEX_NONE;
    int32_t bestTap = TAP_NONE;                    // curve mode: the winning candidate's pixel
    const bool mvs = a.select_kind == SR_SELECT_MVS;
    const int D = a.D;
    const bool depth_up = a.depth_up != 0;
    const int nchunks = (D + TAP_CHUNK - 1) / TAP_CHUNK;
    const int total_chunks = nchunks * a.num_nbrs;
    const int tid = threadIdx.x;
    const uint64_t pol = l2_evict_first_policy();
    // stage `c` of the tap stream = labels [ (c % nchunks)*TAP_CHUNK, +TAP_CHUNK ) of neighbour c / nchunks
    auto issue_chunk = [&](int c) {
        if (c < total_chunks) {
            const int j = c / nchunks, d0 = (c % nchunks) * TAP_CHUNK;
            const int32_t *src = a.taps + ((size_t)j * (a.tap_planes ? a.tap_planes : D) + d0) * npix + pid;
            const int nl = min(TAP_CHUNK, D - d0);
            for (int l = 0; l < nl; ++l) cp_async4(&tap_ring[c & 1][l][tid], src + (size_t)l * npix, pol);
        }
        cp_async_commit();
    };
    issue_chunk(0);

#pragma unroll 1
    for (int c = 0; c < total_chunks; ++c) {
        issue_chunk(c + 1);
        cp_async_wait<1>();  // stage c has landed (this thread's own copies; no cross-thread sharing)
        const int j = c / nchunks, d0 = (c % nchunks) * TAP_CHUNK;
        const int nl = min(TAP_CHUNK, D - d0);
        const double *__restrict__ gR = a.grayR[j];
        float *vol = a.out_volume ? a.out_volume + ((size_t)j * D + d0) * npix + pid : nullptr;
#pragma unroll 1
        for (int l = 0; l < nl; ++l) {
            const int32_t tap = tap_ring[c & 1][l][tid];
            double cost = qnan();
            if (tap != TAP_NONE) {
                const int tx = (int)(short)(tap & 0xffff), ty = (int)(short)((uint32_t)tap >> 16);
                if (tx >= R && ty >= R && tx < w - R && ty < h - R) cost = fast_one(gR + ((size_t)ty * w + tx));
                // windows touching a border / an invalid pixel: the reference's exact tap filter
                if (cost != cost) cost = slow_cost<R, G, COST>(a, gR, x, y, tx, ty, pid, sub, gmask, wloc);
                // ---- stage (3): winner-take-all, fused ----
                const int d = d0 + l;
                // curve mode (multiviewstereo.cpp:583-588): a candidate's depth is the camera-space z of
                // the closest approach of the two viewing rays, computed only for the few candidates
                // above the threshold
                double zc = 0.0;
                if (mvs && a.curve && cost > a.ncc_threshold)
                    zc = curve_depth(a.raysL, a.raysR[j], (size_t)w * h, pix, (size_t)ty * w + tx, a.camR, a.camT);
                if (mvs && a.out_peaks && sub == 0 && cost > a.ncc_threshold) {
                    // peaks.push_back(pair(ncc, depth)); sort; keep the last K (multiviewstereo.cpp:589-602):
                    // kept incrementally as an ascending list, smallest entry first
                    const size_t n = (size_t)w * h;
                    double *pk = a.out_peaks + pix;  // entry k: pk[(2k)*n] = ncc, pk[(2k+1)*n] = depth
                    const double dep = a.curve ? zc : a.depth_table[d0 + l];
                    const double c0 = pk[0], z0 = pk[n];
                    if (cost > c0 || (cost == c0 && dep > z0)) {
                        int k = 0;  // drop entry 0, shift smaller entries down, insert in order
                        for (; k + 1 < 9; ++k) {
                            const double ck = pk[(size_t)(2 * k + 2) * n], zk = pk[(size_t)(2 * k + 3) * n];
                            if (cost > ck || (cost == ck && dep > zk)) {
                                pk[(size_t)(2 * k) * n] = ck;
                                pk[(size_t)(2 * k + 1) * n] = zk;
                            } else {
                                break;
                            }
                        }
                        pk[(size_t)(2 * k) * n] = cost;
                        pk[(size_t)(2 * k + 1) * n] = dep;
                    }
                }
                if (mvs) {  // multiviewstereo.cpp:589-602,654-660: max over (ncc, depth) pairs
                    // depthFromLabel is strictly monotone in the label, so "depth > bestD" is decided
                    // on the indices (deeper == d > bestIdx iff depth_up); the table is read once at
                    // the end instead of once per label on the critical path.
                    if (cost > a.ncc_threshold) {
                        const bool deeper = a.curve ? (zc > bestZ) : (depth_up ? (d > bestIdx) : (d < bestIdx));
                        if (bestIdx == SR_INDEX_NONE || cost > bestC || (cost == bestC && deeper)) {
                            bestC = cost;
                            bestIdx = d;
                            bestZ = zc;
                        }
                    }
                } else {  // twoviewstereo.cpp:320-325
                    if (cost + 1e-10 < minCost) {
                        secondBest = minCost;
                        minCost = cost;
                        bestIdx = d;
                        bestTap = tap;
                    }
                }
            }
            if (vol && sub == 0) vol[(size_t)l * npix] = (float)cost;
        }
    }
    cp_async_wait<0>();

    if (sub == 0) {
        if (mvs) {
            a.out_index[pix] = bestIdx;
            a.out_depth[pix] = (bestIdx >= 0) ? (a.curve ? bestZ : a.depth_table[bestIdx]) : -1.0;
            a.out_best[pix] = bestC;
        } else {
            double depth = (bestIdx >= 0) ? a.depth_table[a.curve ? 0 : bestIdx] : qnan();
            if (a.curve && bestIdx >= 0) {  // twoviewstereo.cpp:286-299: z of the rays' closest approach
                const int tx = (int)(short)(bestTap & 0xffff), ty = (int)(short)((uint32_t)bestTap >> 16);
                depth = curve_depth(a.raysL, a.raysR[0], (size_t)w * h, pix, (size_t)ty * w + tx, a.camR, a.camT);
            }
            if (a.second_best_factor > 0.0 && minCost > a.second_best_factor * secondBest) {  // :304-305
                depth = dinf();
                bestIdx = SR_INDEX_REJECTED;
            }
            a.out_index[pix] = bestIdx;
            a.out_depth[pix] = depth;
            a.out_best[pix] = minCost;
        }
    }
}

// ---------------------------------------------------------------------------------------------
// crossCheck.  One launch per checked view; the launch order on the stream reproduces the
// reference's in-place, view-by-view semantics.
struct CrossArgs {
    const sr_camera *cams;       // device array of all views' cameras
    double *const *depth_ptrs;   // device array of all views' depth maps
    int32_t *indexA;
    int viewA, num_views;
    int w, h;
    double scale, thresh;
    int two_view;                // 1: failing -> +INF (must pass against the other view);
                                 // 0: any other view may confirm, failing -> NaN
};

__device__ __forceinline__ bool point_from_depth(d3 src, d3 dir, d3 normal, d3 C, double depth, d3 &p) {
    const d3 nrm = normalized(normal);
    const d3 x0 = C + depth * normal;
    return ray_plane(src, dir, nrm, dot(nrm, x0), p);
}

__global__ void __launch_bounds__(128) cross_check_kernel(const CrossArgs a) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.w * a.h) return;
    double *depthA = a.depth_ptrs[a.viewA];
    const double depth = depthA[i];
    if (!isfinite(depth)) return;
    const int x = i % a.w, y = i / a.w;
    const sr_camera &A = a.cams[a.viewA];
    d3 src, dir, p1;
    cam_unproject(A, (x + 0.5) / a.scale, (y + 0.5) / a.scale, src, dir);
    if (!point_from_depth(src, dir, ld3(A.prin_dir), ld3(A.C), depth, p1)) return;
    bool found = false, fail = false;
    for (int b = 0; b < a.num_views && !found; ++b) {
        if (b == a.viewA) continue;
        const sr_camera &B = a.cams[b];
        double x2, y2;
        fail = true;
        if (cam_project(B, p1, x2, y2)) {
            x2 *= a.scale;
            y2 *= a.scale;
            if (x2 >= 0 && y2 >= 0 && x2 < a.w && y2 < a.h) {
                const double od = a.depth_ptrs[b][(size_t)((int)y2) * a.w + (int)x2];
                if (isfinite(od)) {
                    d3 s2, d2, p2;
                    cam_unproject(B, (x2 + 0.5) / a.scale, (y2 + 0.5) / a.scale, s2, d2);
                    if (point_from_depth(s2, d2, ld3(B.prin_dir), ld3(B.C), od, p2)) {
                        const d3 df = p1 - p2;
                        const double nrm = sqrt(dot(df, df));
                        if (a.two_view) {
                            fail = (!isfinite(nrm) || nrm > a.thresh);
                        } else if (isfinite(nrm) && nrm < a.thresh) {
                            found = true;
                        }
                    }
                }
            }
        }
    }
    if (a.two_view) {
        if (fail) {
            depthA[i] = dinf();
            a.indexA[i] = SR_INDEX_REJECTED;
        }
    } else if (!found) {
        depthA[i] = qnan();
        a.indexA[i] = SR_INDEX_NONE;
    }
}

// RefractiveCalibrationFunction::diff (stereo/refractioncalibration.cpp:175-201): the residual the
// interface calibration minimises, one thread per correspondence.  (The Levenberg-Marquardt outer
// loop, util/lm.cpp, stays on the host: a handful of parameters.)
// blockIdx.y selects one of gridDim.y camera sets (the base model of the Levenberg-Marquardt step
// and its finite-difference perturbations are evaluated in one launch).
__global__ void calibration_residual_kernel(const sr_camera *__restrict__ cams, int num_cams, int n,
                                            const int32_t *__restrict__ pairs, const double *__restrict__ pix,
                                            double *__restrict__ out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    cams += (size_t)blockIdx.y * num_cams;
    out += (size_t)blockIdx.y * n;
    const sr_camera &v1 = cams[pairs[2 * i]], &v2 = cams[pairs[2 * i + 1]];
    d3 s1, d1, s2, d2;
    cam_unproject(v1, pix[4 * i], pix[4 * i + 1], s1, d1);
    cam_unproject(v2, pix[4 * i + 2], pix[4 * i + 3], s2, d2);
    const d3 w0 = s1 - s2;  // Ray3d::closestPoints, util/ray.cpp:53-74
    const double aa = dot(d1, d1), bb = dot(d1, d2), cc = dot(d2, d2), dd = dot(d1, w0), ee = dot(d2, w0);
    const double den = 1.0 / (aa * cc - bb * bb);
    const double tl = (bb * ee - cc * dd) * den, tr = (aa * ee - bb * dd) * den;
    d3 p1 = s1, p2 = s2;
    if (tl > 0) p1 = p1 + tl * d1;
    if (tr > 0) p2 = p2 + tr * d2;
    const d3 df = p1 - p2;
    const double dist = sqrt(dot(df, df));
    const d3 mid = 0.5 * (p1 + p2);
    const double z1 = (mul3(v1.R, mid) + ld3(v1.t)).z, z2 = (mul3(v2.R, mid) + ld3(v2.t)).z;
    out[i] = (0.5 * v1.K[0] * dist) / z1 + (0.5 * v2.K[0] * dist) / z2;
}

// colorFromDepth of MultiViewStereo (multiviewstereo.cpp:257-278) + the WHITE fill for masked
// pixels (:381-395) -> RGBA8.
__global__ void depth_image_mvs_kernel(const double *__restrict__ depth, const uint8_t *__restrict__ mask, int n,
                                       double min_depth, double max_depth, uchar4 *__restrict__ out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    unsigned char g = 255;
    const double d = depth[i];
    if (mask[i] == 255 && isfinite(d) && !(d + 1e-5 < min_depth)) {
        const double t = fmin(1.0, fmax(0.0, (d - min_depth) / (max_depth - min_depth)));
        g = (unsigned char)(int)(255 * t);
    }
    out[i] = make_uchar4(g, g, g, 255);
}

}  // namespace sr
