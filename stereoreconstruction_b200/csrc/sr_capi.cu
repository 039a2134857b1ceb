// sr_capi.cu — the C ABI of include/sr_b200.h: context, device memory, launches.
// Host code is C++; everything numeric runs in the kernels of sr_kernels.cuh / sr_curve.cuh.
// There is no CPU fallback: every entry point that computes launches CUDA kernels.
#include <atomic>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <dlfcn.h>
#include <string>
#include <vector>
#include <algorithm>

#include "sr_kernels.cuh"
#include "sr_match_dispatch.cuh"
#include "sr_build_refr.cuh"
#include "sr_curve.cuh"
#include "sr_points.cuh"
#include "sr_fuse.cuh"
#include "sr_mrf.cuh"

using namespace sr;

namespace {

std::string g_create_error;

constexpr int REFR_CHUNK = 256;  // labels per thread of build_refr_kernel
static_assert(REFR_CHUNK % BUILD_STRIDE == 0, "build_refr_sweep takes label ranges that start on an anchor");

struct ViewDev {
    uchar4 *rgba = nullptr;
    uint8_t *mask = nullptr;
    double *gray_pix = nullptr, *gray_two = nullptr, *gray_msk = nullptr, *edges = nullptr;
    float *gray_pix_f = nullptr;
    bool have_image = false; // sr_set_views received pixels for this view
    bool all_white = false;  // no mask was passed for this view: every pixel is WHITE
    double *rays = nullptr;  // [6][h][w] Camera::unproject of every pixel centre (curve mode), lazily
    double rays_scale = 0.0; // image_scale the table was computed for (0: stale)
    int32_t *index = nullptr;
    double *depth = nullptr, *best = nullptr;
};

// Scratch of the view searches, one set per stream that runs them; grow-only, capacities in bytes.
struct Scratch {
    double *rays = nullptr;     // [6][h][w] rays of the reference view
    int32_t *taps = nullptr;    // tap volume of one row band
    double *weights = nullptr;  // [WN][band pixels]
    size_t rays_cap = 0, taps_cap = 0, weights_cap = 0;
};

// ---- NCCL through dlopen (the library loads without NCCL; sr_comm_* fail loudly) ------------
typedef struct ncclComm *ncclComm_t;
struct Uid128 {
    char b[128];
};
struct NcclApi {
    void *handle = nullptr;
    int (*GetUniqueId)(void *) = nullptr;
    int (*CommInitRank)(ncclComm_t *, int, Uid128 /* ncclUniqueId by value */, int) = nullptr;
    int (*CommDestroy)(ncclComm_t) = nullptr;
    int (*Broadcast)(const void *, void *, size_t, int, int, ncclComm_t, cudaStream_t) = nullptr;
    int (*GroupStart)() = nullptr;
    int (*GroupEnd)() = nullptr;
    const char *(*GetErrorString)(int) = nullptr;
};
NcclApi g_nccl;
const int NCCL_CHAR = 0;

bool load_nccl(std::string &err) {
    static bool loaded = false;  // set only once every symbol has resolved
    if (loaded) return true;
    const char *names[] = {"libnccl.so.2", "libnccl.so"};
    void *handle = nullptr;
    for (const char *n : names) {
        handle = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
        if (handle) break;
    }
    if (!handle) {
        err = std::string("cannot dlopen libnccl.so.2: ") + dlerror();
        return false;
    }
    NcclApi api;
    api.handle = handle;
#define LD(field, sym)                                                    \
    *(void **)(&api.field) = dlsym(handle, sym);                          \
    if (!api.field) {                                                     \
        err = std::string("NCCL symbol missing: ") + sym;                 \
        dlclose(handle);                                                  \
        return false;                                                     \
    }
    LD(GetUniqueId, "ncclGetUniqueId");
    LD(CommInitRank, "ncclCommInitRank");
    LD(CommDestroy, "ncclCommDestroy");
    LD(Broadcast, "ncclBroadcast");
    LD(GroupStart, "ncclGroupStart");
    LD(GroupEnd, "ncclGroupEnd");
    LD(GetErrorString, "ncclGetErrorString");
#undef LD
    g_nccl = api;
    loaded = true;
    return true;
}

}  // namespace

struct sr_ctx {
    int device = 0;
    cudaStream_t own_stream = nullptr, stream = nullptr;
    std::string err;
    std::atomic<bool> cancel{false};
    int V = 0, w = 0, h = 0;
    std::vector<sr_camera> cams;
    sr_camera *d_cams = nullptr;
    std::vector<ViewDev> views;
    double **d_depth_ptrs = nullptr;  // device array of per-view depth map pointers
    uchar4 **d_rgba_ptrs = nullptr;   // device array of per-view image pointers
    sr_params params{};
    bool have_params = false;
    std::vector<double> depth_table;
    double *d_depth_table = nullptr;
    size_t depth_table_cap = 0;  // bytes
    Scratch s;                   // of the views run on `stream`
    float *d_volume = nullptr;
    size_t vol_cap = 0, vol_elems = 0;
    double *d_peaks = nullptr;  // [9][2][h*w] of the last view run with keep_cost_volume & 2
    size_t peaks_cap = 0;       // bytes
    int peaks_view = -1;
    void *d_scratch = nullptr;
    size_t scratch_cap = 0;
    void *d_out = nullptr;  // variable-length results (point clouds), apart from the scratch that counts them
    size_t out_cap = 0;
    int64_t launches = 0;
    size_t tap_budget = (size_t)8 << 30;
    unsigned long long *d_stats = nullptr;  // SR_MATCH_STATS=1: counters of the screened match kernel
    bool use_refr_build = true;  // SR_BUILD_REFR=0: refractive views through the generic build_kernel (A/B aid)
    bool use_screen = true;  // SR_MATCH_SCREEN=0: MVS selection through the all-FP64 match_kernel (A/B aid)
    // "Lanes" (stream + private scratch; two by default) that consecutive sr_run_view calls alternate between: the
    // ramp-down of one view's kernels (the last, partially filled wave of 0.5 ms blocks) overlaps the
    // next view's launches.  Everything else runs on `stream`, after join_lanes().  SR_LANES=1 turns it off.
    struct Lane {
        cudaStream_t stream = nullptr;
        cudaEvent_t done = nullptr;
        bool pending = false;
        Scratch s;
    };
    static constexpr int MAX_LANES = 4;
    Lane lanes[MAX_LANES];
    int num_lanes = 2, next_lane = 0;
    cudaEvent_t ev_fork = nullptr;
    std::vector<int> view_lane;  // lane that last ran each reference view (-1: none pending)
    // Downloads of a view that is still on a lane wait for THAT view only (its own event) and run on a copy
    // stream: sr_get_depth(v) overlaps the views enqueued after v instead of joining all of them.
    std::vector<cudaEvent_t> view_done;
    cudaStream_t copy_stream = nullptr;
    ncclComm_t comm = nullptr;
    int rank = 0, nranks = 1;
    // per-stage CUDA-event timing (sr_set_profiling): [begin, after build, after match] per band
    bool profiling = false;
    std::vector<cudaEvent_t> prof_events;
};

namespace {

int fail(sr_ctx *c, int code, const std::string &msg) {
    if (c) c->err = msg;
    else g_create_error = msg;
    return code;
}
#define CK(call)                                                                                       \
    do {                                                                                               \
        cudaError_t e_ = (call);                                                                       \
        if (e_ != cudaSuccess)                                                                         \
            return fail(ctx, SR_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_));         \
    } while (0)
// SR_DEBUG_SYNC=1: synchronise after every launch, so that a faulting kernel is reported at its own line
static const bool g_debug_sync = getenv("SR_DEBUG_SYNC") && atoi(getenv("SR_DEBUG_SYNC")) != 0;
#define CKL()                                                                                          \
    do {                                                                                               \
        ++ctx->launches;                                                                               \
        cudaError_t e_ = cudaGetLastError();                                                           \
        if (e_ == cudaSuccess && g_debug_sync) e_ = cudaStreamSynchronize(ctx->stream);                \
        if (e_ != cudaSuccess)                                                                         \
            return fail(ctx, SR_ERR_CUDA, std::string("kernel launch (" __FILE__ ":") +                \
                                              std::to_string(__LINE__) + "): " + cudaGetErrorString(e_)); \
    } while (0)
// a call that returns an SR_* code
#define CKR(call)                 \
    do {                          \
        int rc_ = (call);         \
        if (rc_) return rc_;      \
    } while (0)

template <typename T>
void dfree(T *&p) {
    if (p) cudaFree(p);
    p = nullptr;
}

void free_scratch(Scratch &s) {
    dfree(s.rays);
    dfree(s.taps);
    dfree(s.weights);
    s = Scratch();
}

void free_views(sr_ctx *c) {
    for (ViewDev &v : c->views) {
        dfree(v.rgba);
        dfree(v.mask);
        dfree(v.gray_pix);
        dfree(v.gray_pix_f);
        dfree(v.rays);
        dfree(v.gray_two);
        dfree(v.gray_msk);
        dfree(v.edges);
        dfree(v.index);
        dfree(v.depth);
        dfree(v.best);
    }
    c->views.clear();
    for (cudaEvent_t e : c->view_done)
        if (e) cudaEventDestroy(e);
    c->view_done.clear();
    c->view_lane.clear();
    c->peaks_view = -1;  // peak lists belong to the image size they were computed at
    dfree(c->d_cams);
    dfree(c->d_depth_ptrs);
    dfree(c->d_rgba_ptrs);
    free_scratch(c->s);  // sized for the old images
}

// Grow-only device buffer: kept while it holds `bytes`; otherwise `st` (the stream that uses it) is drained and
// the buffer reallocated, its capacity recorded only once the allocation has succeeded.
template <typename T>
int grow(sr_ctx *ctx, cudaStream_t st, T *&p, size_t &cap, size_t bytes) {
    if (bytes <= cap) return SR_OK;
    CK(cudaStreamSynchronize(st));
    dfree(p);
    cap = 0;
    CK(cudaMalloc(&p, bytes));
    cap = bytes;
    return SR_OK;
}

int ensure_scratch(sr_ctx *ctx, size_t bytes) { return grow(ctx, ctx->stream, ctx->d_scratch, ctx->scratch_cap, bytes); }

// Byte offsets of the pieces carved out of one buffer start on 256-byte boundaries.
constexpr size_t align256(size_t bytes) { return (bytes + 255) / 256 * 256; }

// Camera::unproject of the pixel centres of rows [row0, row0 + rows) into the [6][h][w] table `out`.
int launch_rays(sr_ctx *ctx, const sr_camera &cam, int row0, int rows, double scale, double *out, cudaStream_t st) {
    rays_kernel<<<(unsigned)(((size_t)rows * ctx->w + 127) / 128), 128, 0, st>>>(cam, ctx->w, ctx->h, row0, rows, scale, out);
    CKL();
    return SR_OK;
}

// The maps of a view read "not computed": NaN depth (twoviewstereo.cpp:118-119) and best cost, index NONE.
int reset_maps(sr_ctx *ctx, ViewDev &v) {
    const size_t n = (size_t)ctx->w * ctx->h;
    CK(cudaMemsetAsync(v.depth, 0xff, n * 8, ctx->stream));
    CK(cudaMemsetAsync(v.best, 0xff, n * 8, ctx->stream));
    CK(cudaMemsetAsync(v.index, 0xff, n * 4, ctx->stream));
    return SR_OK;
}

// Support weights (kind: SR_WEIGHT_*) of view v into W: of the pixels of rows [row0, row0 + rows), or, when
// list_x is given, of the list_n window centres (list_x, list_y).
int launch_weights(sr_ctx *ctx, const ViewDev &v, int kind, int radius, double *W, int row0, int rows, cudaStream_t st,
                   const int32_t *list_x = nullptr, const int32_t *list_y = nullptr, int list_n = 0) {
    WeightArgs wa;
    memset(&wa, 0, sizeof(wa));
    wa.rgba = v.rgba;
    wa.mask = v.mask;
    wa.edges = v.edges;
    wa.W = W;
    wa.w = ctx->w;
    wa.h = ctx->h;
    wa.row0 = row0;
    wa.rows = rows;
    wa.radius = radius;
    wa.list_x = list_x;
    wa.list_y = list_y;
    wa.list_n = list_n;
    const size_t npix = list_x ? (size_t)list_n : (size_t)rows * ctx->w;
    const unsigned gx = (unsigned)((npix + 127) / 128);
    const size_t smem = (size_t)(2 * radius + 1) * (2 * radius + 1) * 128 * sizeof(double);
    // From r = 3 up the shared-memory grid ((2r+1)^2 * 128 doubles, 49 KB at r = 3) exceeds 48 KB: the grid
    // is the thread's column of W.
    if (kind == SR_WEIGHT_ADAPTIVE)
        weights_adaptive_kernel<<<gx, 128, (radius + 1) * sizeof(double), st>>>(wa);
    else if (radius == 2)  // MultiViewStereo's window (multiviewstereo.cpp:91): sweeps unrolled
        weights_geodesic_kernel<true, 2><<<gx, 128, smem, st>>>(wa);
    else if (radius == 1)
        weights_geodesic_kernel<true, 1><<<gx, 128, smem, st>>>(wa);
    else
        weights_geodesic_kernel<false, 0><<<gx, 128, 0, st>>>(wa);
    CKL();
    return SR_OK;
}

double depth_from_label(const sr_params &p, int label) {
    double t = label / (p.num_levels - 1.0);
    if (p.depth_kind == SR_DEPTH_INV5) t /= (5 - 4 * t);  // stereo/twoviewstereo.cpp:981-985
    return p.min_depth * (1 - t) + p.max_depth * t;        // stereo/multiviewstereo.cpp:733-736
}

// K (rows 0/1 normalised for a distorted view) and the map from normalised/pixel coordinates to the
// coordinate that is truncated: scale and the tap rule's shift (label mode: MVS 0, two-view -0.5; curve mode 0)
// folded in.
void refr_pixel_map(const sr_camera &nb, double shift, double sc, double *Kn, double &fxs, double &cxs, double &fys, double &cys) {
    memcpy(Kn, nb.K, 9 * sizeof(double));
    if (nb.is_distorted) {
        const double fx = nb.K[0], fy = nb.K[4], cx = nb.K[2], cy = nb.K[5];
        for (int c = 0; c < 3; ++c) {
            Kn[c] = (nb.K[c] - cx * nb.K[6 + c]) / fx;
            Kn[3 + c] = (nb.K[3 + c] - cy * nb.K[6 + c]) / fy;
        }
        fxs = fx * sc;
        cxs = cx * sc + shift;
        fys = fy * sc;
        cys = cy * sc + shift;
    } else {
        fxs = fys = sc;
        cxs = cys = shift;
    }
}

// Make the context stream wait for the lanes' pending views (no host synchronisation).
int join_lanes(sr_ctx *ctx) {
    for (sr_ctx::Lane &L : ctx->lanes)
        if (L.pending) {
            CK(cudaStreamWaitEvent(ctx->stream, L.done, 0));
            L.pending = false;
        }
    std::fill(ctx->view_lane.begin(), ctx->view_lane.end(), -1);
    return SR_OK;
}

// The preamble of every entry point that touches the device: select the context's device, then (join) order the
// views still running on the lanes before the context stream.
int enter(sr_ctx *ctx, bool join = true) {
    CK(cudaSetDevice(ctx->device));
    return join ? join_lanes(ctx) : SR_OK;
}

int check_view(sr_ctx *ctx, int v) {
    if (!ctx) return SR_ERR_INVALID;
    if (ctx->V == 0) return fail(ctx, SR_ERR_STATE, "sr_set_views has not been called");
    if (v < 0 || v >= ctx->V) return fail(ctx, SR_ERR_INVALID, "view index out of range");
    return SR_OK;
}

int check_params(sr_ctx *ctx) {
    return ctx->have_params ? SR_OK : fail(ctx, SR_ERR_STATE, "sr_set_params has not been called");
}

// Arguments of sr_run_view / sr_run_view_curve; [r0, r1) is the row range to compute.
int check_run(sr_ctx *ctx, int ref, const int32_t *nbrs, int nn, int &r0, int &r1) {
    CKR(check_view(ctx, ref));
    CKR(check_params(ctx));
    if (!nbrs || nn <= 0 || nn > SR_MAX_NBRS) return fail(ctx, SR_ERR_INVALID, "1..8 neighbour views required");
    for (int j = 0; j < nn; ++j)
        if (nbrs[j] < 0 || nbrs[j] >= ctx->V || nbrs[j] == ref) return fail(ctx, SR_ERR_INVALID, "bad neighbour index");
    if (!ctx->views[ref].have_image) return fail(ctx, SR_ERR_STATE, "the reference view was given no image in sr_set_views");
    for (int j = 0; j < nn; ++j)
        if (!ctx->views[nbrs[j]].have_image) return fail(ctx, SR_ERR_STATE, "a neighbour view was given no image in sr_set_views");
    const sr_params &P = ctx->params;
    if (P.select_kind == SR_SELECT_TWOVIEW && nn != 1)
        return fail(ctx, SR_ERR_INVALID, "two-view selection takes exactly one neighbour");
    r0 = std::max(P.row_begin, 0);
    r1 = (P.row_end > 0 && P.row_end < ctx->h) ? P.row_end : ctx->h;
    if (r0 >= r1) return fail(ctx, SR_ERR_INVALID, "empty row range");
    return SR_OK;
}

// Stage timing of one band (sr_set_profiling): ev = [begin, after build, after match], handed to prof_events
// (read by sr_get_stage_ms) once the band's match kernel is enqueued.
int prof_begin(sr_ctx *ctx, cudaStream_t st, cudaEvent_t (&ev)[3]) {
    if (!ctx->profiling) return SR_OK;
    for (int k = 0; k < 3; ++k) CK(cudaEventCreate(&ev[k]));
    CK(cudaEventRecord(ev[0], st));
    return SR_OK;
}
int prof_mark(sr_ctx *ctx, cudaStream_t st, cudaEvent_t (&ev)[3], int k) {
    if (!ctx->profiling) return SR_OK;
    CK(cudaEventRecord(ev[k], st));
    if (k == 2) ctx->prof_events.insert(ctx->prof_events.end(), ev, ev + 3);
    return SR_OK;
}

// The MatchArgs of rows [row0, row0 + rows) of view ref that both searches fill alike; each adds what its mode
// differs in.
MatchArgs match_args(const sr_ctx *ctx, int ref, const int32_t *nbrs, int nn, const Scratch &S, int row0, int rows) {
    const sr_params &P = ctx->params;
    const ViewDev &A = ctx->views[ref];
    MatchArgs ma;
    memset(&ma, 0, sizeof(ma));
    ma.W = S.weights;
    ma.maskL = A.mask;
    ma.grayL = (P.cost_kind == SR_COST_NCC_MVS) ? A.gray_pix : A.gray_two;
    for (int j = 0; j < nn; ++j) {
        const ViewDev &B = ctx->views[nbrs[j]];
        ma.grayR[j] = (P.cost_kind == SR_COST_NCC_MVS) ? B.gray_pix
                      : (P.cost_kind == SR_COST_NCC_TWOVIEW) ? B.gray_two : B.gray_msk;
        ma.grayRf[j] = B.gray_pix_f;
    }
    ma.pitch_f = screen_pitch(ctx->w);
    ma.taps = S.taps;
    ma.depth_table = ctx->d_depth_table;
    ma.out_index = A.index;
    ma.out_depth = A.depth;
    ma.out_best = A.best;
    ma.out_peaks = (P.keep_cost_volume & 2) ? ctx->d_peaks : nullptr;
    ma.w = ctx->w;
    ma.win_w = std::max(0, ctx->w - 2 * P.radius);  // (compared as unsigned: an image smaller than the window has no interior)
    ma.win_h = std::max(0, ctx->h - 2 * P.radius);
    ma.h = ctx->h;
    ma.row0 = row0;
    ma.rows = rows;
    ma.D = P.num_levels;
    ma.num_nbrs = nn;
    ma.select_kind = P.select_kind;
    ma.depth_up = (P.max_depth >= P.min_depth) ? 1 : 0;
    ma.use_screen = ctx->use_screen ? 1 : 0;
    ma.stats = ctx->d_stats;
    ma.second_best_factor = P.second_best_factor;
    ma.ncc_threshold = P.ncc_threshold;
    return ma;
}

int run_match(sr_ctx *ctx, const MatchArgs &ma, cudaStream_t st) {
    cudaError_t e = launch_match(ctx->params.radius, ctx->params.cost_kind, ma, st);
    ++ctx->launches;
    if (e != cudaSuccess) return fail(ctx, SR_ERR_CUDA, std::string("match kernel: ") + cudaGetErrorString(e));
    return SR_OK;
}

// The fields the candidate builds of the reference view `ref` against neighbour `nbr` (BuildArgs, BuildRefrArgs,
// CurveArgs) share, for rows [row0, row0 + rows) and the reference's ray table `rays`.
template <typename A>
void pair_fields(A &a, const sr_ctx *ctx, int ref, int nbr, const double *rays, int row0, int rows, bool mvs) {
    a.nbr = ctx->cams[nbr];
    memcpy(a.prin, ctx->cams[ref].prin_dir, sizeof(a.prin));
    memcpy(a.C, ctx->cams[ref].C, sizeof(a.C));
    a.rays = rays;
    a.depth_table = ctx->d_depth_table;
    a.ref_mask = ctx->views[ref].mask;
    a.w = ctx->w;
    a.h = ctx->h;
    a.row0 = row0;
    a.rows = rows;
    a.D = ctx->params.num_levels;
    a.mvs = mvs;
}

int d2h(sr_ctx *ctx, void *dst, const void *src, size_t bytes, int view = -1) {
    // a view still on a lane: nothing on the context stream has touched its maps since (that would have joined
    // the lanes), so its own event is all this copy has to wait for
    const bool on_lane = view >= 0 && view < (int)ctx->view_lane.size() && ctx->view_lane[view] >= 0 &&
                         view < (int)ctx->view_done.size() && ctx->view_done[view] && ctx->copy_stream;
    CKR(enter(ctx, !on_lane));
    if (on_lane) CK(cudaStreamWaitEvent(ctx->copy_stream, ctx->view_done[view], 0));
    cudaStream_t st = on_lane ? ctx->copy_stream : ctx->stream;
    CK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    return SR_OK;
}

// Downloads the device's [k][n] planes at src into the [n][k] layout the API documents.
int d2h_transposed(sr_ctx *ctx, double *out, const double *src, size_t n, size_t k) {
    if (!out) return fail(ctx, SR_ERR_INVALID, "the output array is null");
    std::vector<double> planar(n * k);
    CKR(d2h(ctx, planar.data(), src, n * k * sizeof(double)));
    for (size_t i = 0; i < n; ++i)
        for (size_t j = 0; j < k; ++j) out[i * k + j] = planar[j * n + i];
    return SR_OK;
}

// Uploads the host's [n][k] layout at in as the device's [k][n] planes at dst.
int h2d_transposed(sr_ctx *ctx, double *dst, const double *in, size_t n, size_t k) {
    std::vector<double> planar(n * k);
    for (size_t i = 0; i < n; ++i)
        for (size_t j = 0; j < k; ++j) planar[j * n + i] = in[i * k + j];
    CK(cudaMemcpyAsync(dst, planar.data(), n * k * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return SR_OK;
}

// The second half of count-then-fill (sr_get_points, sr_fuse_points), once the counting kernels have left the
// number of points at d_total.  *out_count receives it; a call with capacity 0, or without points, ends there.
// Otherwise write(xyz, extra, rgb) fills the output buffer [xyz 3n doubles][extra n * extra_ints][rgb 3n]
// (extra is null when out_extra is) and the arrays are downloaded.
template <typename Write>
int fill_points(sr_ctx *ctx, const long long *d_total, int64_t capacity, int64_t *out_count, const char *too_small,
                double *out_xyz, uint8_t *out_rgb, int32_t *out_extra, int extra_ints, Write write) {
    long long total = 0;
    CKR(d2h(ctx, &total, d_total, sizeof(total)));
    *out_count = total;
    if (capacity == 0 || total == 0) return SR_OK;
    if (capacity < total) return fail(ctx, SR_ERR_INVALID, too_small);
    const size_t n = (size_t)total;
    CKR(grow(ctx, ctx->stream, ctx->d_out, ctx->out_cap, n * (3 * sizeof(double) + extra_ints * sizeof(int32_t) + 3)));
    double *xyz = (double *)ctx->d_out;
    int32_t *extra = (int32_t *)(xyz + 3 * n);
    uint8_t *rgb = (uint8_t *)(extra + extra_ints * n);
    CKR(write(xyz, out_extra ? extra : nullptr, rgb));
    CKR(d2h(ctx, out_xyz, xyz, n * 3 * sizeof(double)));
    CKR(d2h(ctx, out_rgb, rgb, n * 3));
    if (out_extra) CKR(d2h(ctx, out_extra, extra, n * extra_ints * sizeof(int32_t)));
    return SR_OK;
}

}  // namespace

extern "C" {

int sr_ctx_create(int device, sr_ctx **out) {
    if (!out) return fail(nullptr, SR_ERR_INVALID, "out is null");
    *out = nullptr;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0)
        return fail(nullptr, SR_ERR_CUDA,
                    std::string("no CUDA device (this library has no CPU fallback): ") + cudaGetErrorString(e));
    if (device < 0 || device >= n) return fail(nullptr, SR_ERR_INVALID, "device index out of range");
    e = cudaSetDevice(device);
    if (e != cudaSuccess) return fail(nullptr, SR_ERR_CUDA, cudaGetErrorString(e));
    sr_ctx *c = new sr_ctx;
    c->device = device;
    e = cudaStreamCreateWithFlags(&c->own_stream, cudaStreamNonBlocking);
    if (e != cudaSuccess) {
        delete c;
        return fail(nullptr, SR_ERR_CUDA, cudaGetErrorString(e));
    }
    c->stream = c->own_stream;
    {   // scratch budget of one row band: a quarter of the device memory, at most 32 GiB (a B200 has
        // 180 GB: cfg5's 51 GB tap volume runs in 2 bands), at least 1 GiB
        size_t free_b = 0, total_b = 0;
        if (cudaMemGetInfo(&free_b, &total_b) == cudaSuccess && total_b > 0)
            c->tap_budget = std::max<size_t>((size_t)1 << 30, std::min<size_t>((size_t)32 << 30, total_b / 4));
    }
    if (const char *mb = getenv("SR_TAP_BUDGET_MB")) c->tap_budget = (size_t)atoll(mb) << 20;
    if (const char *sc = getenv("SR_MATCH_SCREEN")) c->use_screen = atoi(sc) != 0;
    if (const char *sb = getenv("SR_BUILD_REFR")) c->use_refr_build = atoi(sb) != 0;
    if (const char *sn = getenv("SR_LANES")) c->num_lanes = std::min((int)sr_ctx::MAX_LANES, std::max(1, atoi(sn)));
    if (c->num_lanes > 1) {
        bool ok = cudaEventCreateWithFlags(&c->ev_fork, cudaEventDisableTiming) == cudaSuccess;
        for (int i = 0; i < c->num_lanes && ok; ++i)
            ok = cudaStreamCreateWithFlags(&c->lanes[i].stream, cudaStreamNonBlocking) == cudaSuccess &&
                 cudaEventCreateWithFlags(&c->lanes[i].done, cudaEventDisableTiming) == cudaSuccess;
        ok = ok && cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking) == cudaSuccess;
        if (!ok) c->num_lanes = 1;
    }
    if (const char *ss = getenv("SR_MATCH_STATS")) {
        if (atoi(ss) != 0 && cudaMalloc(&c->d_stats, 16 * sizeof(unsigned long long)) == cudaSuccess)
            cudaMemset(c->d_stats, 0, 16 * sizeof(unsigned long long));
    }
    *out = c;
    return SR_OK;
}

void sr_ctx_destroy(sr_ctx *c) {
    if (!c) return;
    cudaSetDevice(c->device);
    for (sr_ctx::Lane &L : c->lanes)
        if (L.stream) cudaStreamSynchronize(L.stream);
    cudaStreamSynchronize(c->stream);
    if (c->comm && g_nccl.CommDestroy) g_nccl.CommDestroy(c->comm);
    free_views(c);
    dfree(c->d_depth_table);
    dfree(c->d_volume);
    dfree(c->d_peaks);
    dfree(c->d_stats);
    for (sr_ctx::Lane &L : c->lanes) {
        if (L.stream) cudaStreamSynchronize(L.stream);
        free_scratch(L.s);
        if (L.done) cudaEventDestroy(L.done);
        if (L.stream) cudaStreamDestroy(L.stream);
    }
    if (c->ev_fork) cudaEventDestroy(c->ev_fork);
    if (c->copy_stream) cudaStreamDestroy(c->copy_stream);
    dfree(c->d_scratch);
    dfree(c->d_out);
    cudaStreamDestroy(c->own_stream);
    delete c;
}

const char *sr_last_error(const sr_ctx *c) { return c ? c->err.c_str() : g_create_error.c_str(); }
void sr_request_cancel(sr_ctx *c) {
    if (c) c->cancel.store(true);
}
void sr_clear_cancel(sr_ctx *c) {
    if (c) c->cancel.store(false);
}
int sr_set_stream(sr_ctx *c, void *s) {
    if (!c) return SR_ERR_INVALID;
    CKR(enter(c));  // views still running on the lanes are ordered before whatever follows on the old stream
    c->stream = s ? (cudaStream_t)s : c->own_stream;
    return SR_OK;
}
int64_t sr_launch_count(const sr_ctx *c) { return c ? c->launches : 0; }

void sr_params_default(sr_params *p, int multi_view) {
    memset(p, 0, sizeof(*p));
    p->min_depth = 10.0;  // gui/forms/stereowidget.ui defaults
    p->max_depth = 100.0;
    p->num_levels = 100;
    p->image_scale = 1.0;
    p->weight_kind = SR_WEIGHT_GEODESIC;  // typedef GeodesicWeight WeightFunc
    p->second_best_factor = 0.95;
    p->ncc_threshold = 0.95;
    if (multi_view) {
        p->radius = 2;
        p->cost_kind = SR_COST_NCC_MVS;
        p->depth_kind = SR_DEPTH_LINEAR;
        p->select_kind = SR_SELECT_MVS;
    } else {
        p->radius = 5;
        p->cost_kind = SR_COST_NCC_TWOVIEW;
        p->depth_kind = SR_DEPTH_INV5;
        p->select_kind = SR_SELECT_TWOVIEW;
    }
}

int sr_set_views(sr_ctx *ctx, int V, const sr_camera *cams, const uint8_t *const *rgba8, const uint8_t *const *mask8,
                 int w, int h) {
    if (!ctx) return SR_ERR_INVALID;
    if (V <= 0 || !cams || !rgba8 || w <= 0 || h <= 0 || w > 16384 || h > 16384)
        return fail(ctx, SR_ERR_INVALID, "sr_set_views: bad arguments (1 <= w,h <= 16384)");
    CKR(enter(ctx));
    const size_t n = (size_t)w * h;
    if (V != ctx->V || w != ctx->w || h != ctx->h) {
        CK(cudaStreamSynchronize(ctx->stream));
        free_views(ctx);
        ctx->V = ctx->w = ctx->h = 0;  // nothing is usable until every allocation below has succeeded
        ctx->views.resize(V);
        int rc_alloc = [&]() -> int {
            for (ViewDev &v : ctx->views) {
                CK(cudaMalloc(&v.rgba, n * 4));
                CK(cudaMalloc(&v.mask, n));
                CK(cudaMalloc(&v.gray_pix, n * 8));
                CK(cudaMalloc(&v.gray_pix_f, (size_t)screen_pitch(w) * h * 4));
                CK(cudaMalloc(&v.gray_two, n * 8));
                CK(cudaMalloc(&v.gray_msk, n * 8));
                CK(cudaMalloc(&v.edges, n * 8 * 4));
                CK(cudaMalloc(&v.index, n * 4));
                CK(cudaMalloc(&v.depth, n * 8));
                CK(cudaMalloc(&v.best, n * 8));
            }
            CK(cudaMalloc(&ctx->d_cams, sizeof(sr_camera) * V));
            CK(cudaMalloc(&ctx->d_depth_ptrs, sizeof(double *) * V));
            CK(cudaMalloc(&ctx->d_rgba_ptrs, sizeof(uchar4 *) * V));
            CKR(grow(ctx, ctx->stream, ctx->s.rays, ctx->s.rays_cap, n * 6 * 8));
            std::vector<double *> ptrs(V);
            std::vector<uchar4 *> rgba_ptrs(V);
            for (int i = 0; i < V; ++i) {
                ptrs[i] = ctx->views[i].depth;
                rgba_ptrs[i] = ctx->views[i].rgba;
            }
            CK(cudaMemcpyAsync(ctx->d_depth_ptrs, ptrs.data(), sizeof(double *) * V, cudaMemcpyHostToDevice, ctx->stream));
            CK(cudaMemcpyAsync(ctx->d_rgba_ptrs, rgba_ptrs.data(), sizeof(uchar4 *) * V, cudaMemcpyHostToDevice, ctx->stream));
            CK(cudaStreamSynchronize(ctx->stream));
            return SR_OK;
        }();
        if (rc_alloc != SR_OK) {
            free_views(ctx);  // (the error message of the failing call is kept)
            return rc_alloc;
        }
        ctx->V = V;
        ctx->w = w;
        ctx->h = h;
        // A view this context is only told the camera of (another rank computes it) still has defined
        // results: "not computed" (NaN depth, index NONE) under an all-WHITE mask, until a gather fills them.
        for (ViewDev &v : ctx->views) {
            CK(cudaMemsetAsync(v.mask, 255, n, ctx->stream));
            CKR(reset_maps(ctx, v));
        }
    }
    ctx->cams.assign(cams, cams + V);
    CK(cudaMemcpyAsync(ctx->d_cams, ctx->cams.data(), sizeof(sr_camera) * V, cudaMemcpyHostToDevice, ctx->stream));
    for (int i = 0; i < V; ++i) {
        ViewDev &v = ctx->views[i];
        v.rays_scale = 0.0;  // cameras may have changed
        v.have_image = rgba8[i] != nullptr;
        if (!v.have_image) continue;  // a view this context only knows the camera of (another rank computes it)
        CK(cudaMemcpyAsync(v.rgba, rgba8[i], n * 4, cudaMemcpyHostToDevice, ctx->stream));
        v.all_white = !(mask8 && mask8[i]);
        if (!v.all_white) CK(cudaMemcpyAsync(v.mask, mask8[i], n, cudaMemcpyHostToDevice, ctx->stream));
        else CK(cudaMemsetAsync(v.mask, 255, n, ctx->stream));
        prep_view_kernel<<<(unsigned)((n + 255) / 256), 256, 0, ctx->stream>>>(v.rgba, v.mask, w, h, v.gray_pix,
                                                                             v.gray_two, v.gray_msk, v.edges, v.gray_pix_f, screen_pitch(w));
        CKL();
        CKR(reset_maps(ctx, v));  // results start as "not computed"
    }
    return SR_OK;
}

int sr_set_params(sr_ctx *ctx, const sr_params *p) {
    if (!ctx || !p) return SR_ERR_INVALID;
    if (p->num_levels < 2 || p->num_levels > 65536) return fail(ctx, SR_ERR_INVALID, "num_levels must be in [2,65536]");
    if (!(p->image_scale > 0)) return fail(ctx, SR_ERR_INVALID, "image_scale must be > 0");
    if (!match_supported(p->radius))
        return fail(ctx, SR_ERR_INVALID, "unsupported window radius (supported: " SR_RADII_TEXT ")");
    if (p->weight_kind < 0 || p->weight_kind > 1 || p->cost_kind < 0 || p->cost_kind > 2 || p->depth_kind < 0 ||
        p->depth_kind > 1 || p->select_kind < 0 || p->select_kind > 1)
        return fail(ctx, SR_ERR_INVALID, "bad enum in sr_params");
    ctx->params = *p;
    ctx->have_params = true;
    ctx->depth_table.resize(p->num_levels);
    for (int d = 0; d < p->num_levels; ++d) ctx->depth_table[d] = depth_from_label(*p, d);
    CKR(enter(ctx));
    CKR(grow(ctx, ctx->stream, ctx->d_depth_table, ctx->depth_table_cap, sizeof(double) * p->num_levels));
    CK(cudaMemcpyAsync(ctx->d_depth_table, ctx->depth_table.data(), sizeof(double) * p->num_levels,
                       cudaMemcpyHostToDevice, ctx->stream));
    return SR_OK;
}

// The K = 9 peak pairs per pixel of the view about to run (keep_cost_volume & 2), initialised to
// (0, -1) as multiviewstereo.cpp:562 does; label and curve mode share it.
static int init_peaks(sr_ctx *ctx, int ref) {
    const sr_params &P = ctx->params;
    ctx->peaks_view = -1;
    if (!(P.keep_cost_volume & 2)) return SR_OK;
    if (P.select_kind != SR_SELECT_MVS) return fail(ctx, SR_ERR_INVALID, "peak lists belong to the multi-view selection");
    const size_t n = (size_t)ctx->w * ctx->h;
    CKR(grow(ctx, ctx->stream, ctx->d_peaks, ctx->peaks_cap, n * 18 * 8));  // (a context may be given larger images later)
    std::vector<double> init(n * 18);
    for (int k = 0; k < 9; ++k) {
        std::fill(init.begin() + (size_t)(2 * k) * n, init.begin() + (size_t)(2 * k + 1) * n, 0.0);
        std::fill(init.begin() + (size_t)(2 * k + 1) * n, init.begin() + (size_t)(2 * k + 2) * n, -1.0);
    }
    CK(cudaMemcpyAsync(ctx->d_peaks, init.data(), n * 18 * 8, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    ctx->peaks_view = ref;
    return SR_OK;
}

int sr_run_view(sr_ctx *ctx, int ref, const int32_t *nbrs, int nn) {
    int r0, r1;
    CKR(check_run(ctx, ref, nbrs, nn, r0, r1));
    const sr_params &P = ctx->params;
    const int w = ctx->w, h = ctx->h, D = P.num_levels;
    const size_t n = (size_t)w * h;
    ViewDev &A = ctx->views[ref];

    // Where this view runs: one of the two lanes (its own stream and scratch), or the context stream when
    // something context-wide is written (kept volume, peak lists, statistics, per-stage timing).
    const bool on_lane = ctx->num_lanes > 1 && !ctx->profiling && !P.keep_cost_volume && !ctx->d_stats;
    CKR(enter(ctx, !on_lane));
    sr_ctx::Lane *L = on_lane ? &ctx->lanes[ctx->next_lane] : nullptr;
    cudaStream_t st = on_lane ? L->stream : ctx->stream;
    Scratch &S = on_lane ? L->s : ctx->s;
    if (on_lane) {
        const int li = ctx->next_lane;
        ctx->next_lane = (ctx->next_lane + 1) % ctx->num_lanes;
        CK(cudaEventRecord(ctx->ev_fork, ctx->stream));  // inputs uploaded on the context stream are visible
        CK(cudaStreamWaitEvent(st, ctx->ev_fork, 0));
        // the same view still in flight on the other lane (it writes the same output maps): order them
        if ((int)ctx->view_lane.size() != ctx->V) ctx->view_lane.assign(ctx->V, -1);
        const int prev = ctx->view_lane[ref];
        if (prev >= 0 && prev != li && ctx->lanes[prev].pending) CK(cudaStreamWaitEvent(st, ctx->lanes[prev].done, 0));
        ctx->view_lane[ref] = li;
    }
    CKR(grow(ctx, st, S.rays, S.rays_cap, n * 6 * 8));  // (the context's set has it from sr_set_views)

    CKR(launch_rays(ctx, ctx->cams[ref], r0, r1 - r0, P.image_scale, S.rays, st));

    // Row bands bound the scratch (tap volume nn*D*rows*w*4 bytes + support weights
    // WN*rows*w*8 bytes); a kept cost volume needs one band.
    const size_t wn = (size_t)(2 * P.radius + 1) * (2 * P.radius + 1);
    const size_t per_row = (size_t)nn * D * w * 4;
    const size_t per_row_w = wn * w * 8;
    int band = (int)std::min<size_t>((size_t)(r1 - r0), std::max<size_t>(1, ctx->tap_budget / (per_row + per_row_w)));
    if (P.keep_cost_volume & 1) band = r1 - r0;
    const size_t need = per_row * band;
    CKR(grow(ctx, st, S.weights, S.weights_cap, per_row_w * band));
    CKR(grow(ctx, st, S.taps, S.taps_cap, need));
    CKR(init_peaks(ctx, ref));
    ctx->vol_elems = 0;
    if (P.keep_cost_volume & 1) {
        CKR(grow(ctx, st, ctx->d_volume, ctx->vol_cap, need));
        ctx->vol_elems = need / 4;
        CK(cudaMemsetAsync(ctx->d_volume, 0xff, need, st));  // NaN: labels / pixels never evaluated
    }

    for (int b0 = r0; b0 < r1; b0 += band) {
        if (ctx->cancel.load()) return fail(ctx, SR_ERR_CANCELLED, "cancelled");
        cudaEvent_t ev[3] = {};
        CKR(prof_begin(ctx, st, ev));
        const int rows = std::min(band, r1 - b0);
        const size_t plane = (size_t)rows * w;
        const unsigned gx = (unsigned)((plane + 127) / 128);
        const int d_chunk = 32;
        for (int j = 0; j < nn; ++j) {
            const sr_camera &nb = ctx->cams[nbrs[j]];
            const bool mvs = (P.select_kind == SR_SELECT_MVS);
            if (nb.is_refractive && ctx->use_refr_build) {
                // refractive target view: hoisted-affine reprojection + Newton on the quartic in x/r
                BuildRefrArgs ra;
                pair_fields(ra, ctx, ref, nbrs[j], S.rays, b0, rows, mvs);
                refr_pixel_map(nb, mvs ? 0.0 : -0.5, P.image_scale, ra.Kn, ra.fxs, ra.cxs, ra.fys, ra.cys);
                ra.nbr_mask = ctx->views[nbrs[j]].all_white ? nullptr : ctx->views[nbrs[j]].mask;
                ra.taps = S.taps + (size_t)j * D * plane;
                ra.d_chunk = REFR_CHUNK;
                ra.check = ctx->d_stats ? ctx->d_stats + 8 : nullptr;
                const dim3 grid(gx, (D + ra.d_chunk - 1) / ra.d_chunk);
                if (!mvs) build_refr_kernel<false, false><<<grid, 128, 0, st>>>(ra);
                else if (ra.nbr_mask) build_refr_kernel<true, true><<<grid, 128, 0, st>>>(ra);
                else build_refr_kernel<true, false><<<grid, 128, 0, st>>>(ra);
                CKL();
                continue;
            }
            BuildArgs ba;
            pair_fields(ba, ctx, ref, nbrs[j], S.rays, b0, rows, mvs);
            ba.nbr_mask = ctx->views[nbrs[j]].mask;
            ba.taps = S.taps + (size_t)j * D * plane;
            ba.d_chunk = d_chunk;
            ba.scale = P.image_scale;
            build_kernel<<<dim3(gx, (D + d_chunk - 1) / d_chunk), 128, 0, st>>>(ba);
            CKL();
        }
        CKR(prof_mark(ctx, st, ev, 1));
        CKR(launch_weights(ctx, A, P.weight_kind, P.radius, S.weights, b0, rows, st));
        MatchArgs ma = match_args(ctx, ref, nbrs, nn, S, b0, rows);
        ma.out_volume = (P.keep_cost_volume & 1) ? ctx->d_volume : nullptr;
        CKR(run_match(ctx, ma, st));
        CKR(prof_mark(ctx, st, ev, 2));
    }
    if (on_lane) {
        CK(cudaEventRecord(L->done, st));
        L->pending = true;
        if ((int)ctx->view_done.size() != ctx->V) {
            for (cudaEvent_t e : ctx->view_done)
                if (e) cudaEventDestroy(e);
            ctx->view_done.assign(ctx->V, nullptr);
        }
        if (!ctx->view_done[ref]) CK(cudaEventCreateWithFlags(&ctx->view_done[ref], cudaEventDisableTiming));
        CK(cudaEventRecord(ctx->view_done[ref], st));
    }
    return SR_OK;
}

int sr_set_profiling(sr_ctx *ctx, int on) {
    if (!ctx) return SR_ERR_INVALID;
    ctx->profiling = on != 0;
    return SR_OK;
}

// out[0] = build-stage ms, out[1] = match-stage ms (summed over all bands run since the last
// call), out[2] = number of build launches' bands, out[3] = number of match launches.
int sr_get_stage_ms(sr_ctx *ctx, double *out4) {
    if (!ctx || !out4) return SR_ERR_INVALID;
    CKR(enter(ctx));
    CK(cudaStreamSynchronize(ctx->stream));
    out4[0] = out4[1] = out4[2] = out4[3] = 0;
    for (size_t i = 0; i + 2 < ctx->prof_events.size(); i += 3) {
        float b = 0, m = 0;
        CK(cudaEventElapsedTime(&b, ctx->prof_events[i], ctx->prof_events[i + 1]));
        CK(cudaEventElapsedTime(&m, ctx->prof_events[i + 1], ctx->prof_events[i + 2]));
        out4[0] += b;
        out4[1] += m;
        out4[2] += 1;
        out4[3] += 1;
    }
    for (cudaEvent_t e : ctx->prof_events) cudaEventDestroy(e);
    ctx->prof_events.clear();
    return SR_OK;
}

int sr_get_build_stats(sr_ctx *ctx, uint64_t *out4) {
    if (!ctx || !out4) return SR_ERR_INVALID;
    if (!ctx->d_stats) return fail(ctx, SR_ERR_STATE, "build statistics are off (set SR_MATCH_STATS=1 before sr_ctx_create)");
    CKR(enter(ctx, false));
    CK(cudaStreamSynchronize(ctx->stream));
    CK(cudaMemcpy(out4, ctx->d_stats + 8, 4 * sizeof(uint64_t), cudaMemcpyDeviceToHost));
    return SR_OK;
}

// Debug counters of match_mvs_screen_kernel accumulated since context creation (SR_MATCH_STATS=1):
// out[0] pixels, [1] labels screened in FP32, [2] labels forced to FP64, [3] FP64 verifications,
// [4] pixels whose reference window is evaluated in FP64 only.
int sr_get_match_stats(sr_ctx *ctx, uint64_t *out8) {
    if (!ctx || !out8) return SR_ERR_INVALID;
    if (!ctx->d_stats) return fail(ctx, SR_ERR_STATE, "match statistics are off (set SR_MATCH_STATS=1 before sr_ctx_create)");
    CKR(enter(ctx, false));
    CK(cudaStreamSynchronize(ctx->stream));
    CK(cudaMemcpy(out8, ctx->d_stats, 8 * sizeof(uint64_t), cudaMemcpyDeviceToHost));
    return SR_OK;
}

static int ensure_rays(sr_ctx *ctx, int v) {
    ViewDev &d = ctx->views[v];
    const size_t n = (size_t)ctx->w * ctx->h;
    const double scale = ctx->params.image_scale;
    if (!d.rays) CK(cudaMalloc(&d.rays, n * 6 * 8));
    if (d.rays_scale != scale) {
        CKR(launch_rays(ctx, ctx->cams[v], 0, ctx->h, scale, d.rays, ctx->stream));
        d.rays_scale = scale;
    }
    return SR_OK;
}

// Curve-mode search (the reference's live path): rasterised epipolar curves as the candidate
// set, depth of a candidate = closest approach of the two viewing rays.
int sr_run_view_curve(sr_ctx *ctx, int ref, const int32_t *nbrs, int nn) {
    int r0, r1;
    CKR(check_run(ctx, ref, nbrs, nn, r0, r1));
    const sr_params &P = ctx->params;
    const bool mvs = (P.select_kind == SR_SELECT_MVS);
    if (P.keep_cost_volume & 1) return fail(ctx, SR_ERR_INVALID, "curve mode keeps no cost volume (candidates are not labels)");
    if (mvs && P.cost_kind != SR_COST_NCC_MVS) return fail(ctx, SR_ERR_INVALID, "multi-view curve search uses SR_COST_NCC_MVS");
    CKR(enter(ctx));
    cudaStream_t st = ctx->stream;
    Scratch &S = ctx->s;
    const int w = ctx->w, D = P.num_levels;
    ViewDev &A = ctx->views[ref];
    CKR(ensure_rays(ctx, ref));
    for (int j = 0; j < nn; ++j) CKR(ensure_rays(ctx, nbrs[j]));
    CKR(init_peaks(ctx, ref));  // keep_cost_volume & 2: the candidates' (ncc, z) pairs, through the all-FP64 kernel
    const size_t wn = (size_t)(2 * P.radius + 1) * (2 * P.radius + 1);
    const size_t per_row_w = wn * w * 8;

    auto curve_args = [&](int j, int b0, int rows) {
        CurveArgs ca;
        memset(&ca, 0, sizeof(ca));
        pair_fields(ca, ctx, ref, nbrs[j], A.rays, b0, rows, mvs);
        refr_pixel_map(ca.nbr, 0.0, P.image_scale, ca.Kn, ca.fxs, ca.cxs, ca.fys, ca.cys);
        ca.scale = P.image_scale;
        ca.nbr_mask = ctx->views[nbrs[j]].mask;
        return ca;
    };
    auto launch_curve = [&](const CurveArgs &ca, unsigned gx, bool masked) {
        if (ca.nbr.is_refractive) {
            if (masked) curve_build_kernel<true, true><<<gx, 128, 0, st>>>(ca);
            else curve_build_kernel<true, false><<<gx, 128, 0, st>>>(ca);
        } else {
            if (masked) curve_build_kernel<false, true><<<gx, 128, 0, st>>>(ca);
            else curve_build_kernel<false, false><<<gx, 128, 0, st>>>(ca);
        }
    };

    int cap = 2 * D + 64;  // planes per neighbour: curves are rarely longer than the label count
    int band = (int)std::min<size_t>((size_t)(r1 - r0), std::max<size_t>(1, ctx->tap_budget / ((size_t)nn * cap * w * 4 + per_row_w)));
    for (int b0 = r0; b0 < r1;) {
        if (ctx->cancel.load()) return fail(ctx, SR_ERR_CANCELLED, "cancelled");
        int rows = std::min(band, r1 - b0);
        int L = 1;
        cudaEvent_t ev[3] = {};
        CKR(prof_begin(ctx, st, ev));
        for (int attempt = 0;; ++attempt) {
            const size_t plane = (size_t)rows * w;
            CKR(grow(ctx, st, S.weights, S.weights_cap, per_row_w * rows));
            CKR(grow(ctx, st, S.taps, S.taps_cap, (size_t)nn * cap * plane * 4));
            CKR(ensure_scratch(ctx, 16));
            int32_t *d_max = (int32_t *)ctx->d_scratch;
            CK(cudaMemsetAsync(d_max, 0, 4, st));
            const unsigned gx = (unsigned)((plane + 127) / 128);
            for (int j = 0; j < nn; ++j) {
                CurveArgs ca = curve_args(j, b0, rows);
                ca.taps = S.taps + (size_t)j * cap * plane;
                ca.capacity = cap;
                ca.max_count = d_max;
                launch_curve(ca, gx, !ctx->views[nbrs[j]].all_white);
                CKL();
            }
            int32_t hmax = 0;
            CK(cudaMemcpyAsync(&hmax, d_max, 4, cudaMemcpyDeviceToHost, st));
            CK(cudaStreamSynchronize(st));
            L = std::max(1, (int)hmax);
            if (L <= cap) break;
            if (attempt >= 1) return fail(ctx, SR_ERR_STATE, "curve volume: inconsistent curve lengths");
            // the match kernels carry a candidate's position in 16 bits (queue entries, index maps)
            if (L > 65536) return fail(ctx, SR_ERR_INVALID, "an epipolar curve has more than 65536 candidates: narrow the depth range");
            cap = L;  // a longer curve than the volume holds: size the volume to it and fill again
            rows = (int)std::min<size_t>((size_t)rows, std::max<size_t>(1, ctx->tap_budget / ((size_t)nn * cap * w * 4 + per_row_w)));
        }
        CKR(prof_mark(ctx, st, ev, 1));
        CKR(launch_weights(ctx, A, P.weight_kind, P.radius, S.weights, b0, rows, st));
        MatchArgs ma = match_args(ctx, ref, nbrs, nn, S, b0, rows);
        ma.curve = 1;
        ma.raysL = A.rays;
        for (int j = 0; j < nn; ++j) ma.raysR[j] = ctx->views[nbrs[j]].rays;
        memcpy(ma.camR, ctx->cams[ref].R, sizeof(ma.camR));
        memcpy(ma.camT, ctx->cams[ref].t, sizeof(ma.camT));
        ma.D = L;
        ma.tap_planes = cap;
        ma.depth_up = 1;
        ma.use_screen = 1;  // (SR_MATCH_SCREEN does not apply to curve mode)
        CKR(run_match(ctx, ma, st));
        CKR(prof_mark(ctx, st, ev, 2));
        b0 += rows;
    }
    return SR_OK;
}

int sr_select_neighbours(sr_ctx *ctx, int max_nbrs, int32_t *out, int32_t *counts) {
    if (!ctx || !out || !counts || max_nbrs <= 0) return SR_ERR_INVALID;
    if (ctx->V == 0) return fail(ctx, SR_ERR_STATE, "sr_set_views has not been called");
    // Host-side control logic of MultiViewStereo::runTask (stereo/multiviewstereo.cpp:335-360):
    // V^2 dot products on the camera PODs; not part of the per-pixel path.
    for (int i = 0; i < ctx->V; ++i) {
        std::vector<std::pair<double, int>> nearViews;
        const sr_camera &a = ctx->cams[i];
        for (int j = 0; j < ctx->V; ++j) {
            if (i == j) continue;
            const sr_camera &b = ctx->cams[j];
            const double dp = a.prin_dir[0] * b.prin_dir[0] + a.prin_dir[1] * b.prin_dir[1] + a.prin_dir[2] * b.prin_dir[2];
            if (std::fabs(dp) > 0.2) {
                const double dx = a.C[0] - b.C[0], dy = a.C[1] - b.C[1], dz = a.C[2] - b.C[2];
                nearViews.push_back(std::make_pair(dx * dx + dy * dy + dz * dz, j));
            }
        }
        size_t end = nearViews.size();
        if ((size_t)max_nbrs < nearViews.size()) {
            std::sort(nearViews.begin(), nearViews.end());
            end = max_nbrs;
        }
        counts[i] = (int32_t)end;
        for (size_t k = 0; k < end; ++k) out[i * max_nbrs + k] = nearViews[k].second;
    }
    return SR_OK;
}

int sr_cross_check(sr_ctx *ctx, int two_view, double threshold) {
    if (!ctx) return SR_ERR_INVALID;
    if (ctx->V == 0 || !ctx->have_params) return fail(ctx, SR_ERR_STATE, "views/params not set");
    if (two_view && ctx->V != 2) return fail(ctx, SR_ERR_INVALID, "two-view cross-check needs exactly 2 views");
    CKR(enter(ctx));
    const size_t n = (size_t)ctx->w * ctx->h;
    // View by view, in place, in index order: view v sees the already-updated maps of views < v,
    // exactly as twoviewstereo.cpp:604-670 / multiviewstereo.cpp:427-431 do.
    for (int v = 0; v < ctx->V; ++v) {
        CrossArgs ca;
        ca.cams = ctx->d_cams;
        ca.depth_ptrs = ctx->d_depth_ptrs;
        ca.indexA = ctx->views[v].index;
        ca.viewA = v;
        ca.num_views = ctx->V;
        ca.w = ctx->w;
        ca.h = ctx->h;
        ca.scale = ctx->params.image_scale;
        ca.thresh = threshold;
        ca.two_view = two_view;
        cross_check_kernel<<<(unsigned)((n + 127) / 128), 128, 0, ctx->stream>>>(ca);
        CKL();
    }
    return SR_OK;
}

int sr_flush(sr_ctx *ctx) {
    if (!ctx) return SR_ERR_INVALID;
    return enter(ctx);
}
int sr_synchronize(sr_ctx *ctx) {
    if (!ctx) return SR_ERR_INVALID;
    CKR(enter(ctx));
    CK(cudaStreamSynchronize(ctx->stream));
    return SR_OK;
}

int sr_get_depth_index(sr_ctx *ctx, int view, int32_t *out) {
    CKR(check_view(ctx, view));
    return d2h(ctx, out, ctx->views[view].index, (size_t)ctx->w * ctx->h * 4, view);
}
int sr_get_depth(sr_ctx *ctx, int view, double *out) {
    CKR(check_view(ctx, view));
    return d2h(ctx, out, ctx->views[view].depth, (size_t)ctx->w * ctx->h * 8, view);
}
int sr_get_best_cost(sr_ctx *ctx, int view, double *out) {
    CKR(check_view(ctx, view));
    return d2h(ctx, out, ctx->views[view].best, (size_t)ctx->w * ctx->h * 8, view);
}
int sr_get_cost_volume(sr_ctx *ctx, float *out, size_t out_elems) {
    if (!ctx || !out) return SR_ERR_INVALID;
    if (ctx->vol_elems == 0) return fail(ctx, SR_ERR_STATE, "no cost volume kept (set keep_cost_volume and run)");
    if (out_elems < ctx->vol_elems) return fail(ctx, SR_ERR_INVALID, "output buffer too small");
    return d2h(ctx, out, ctx->d_volume, ctx->vol_elems * 4);
}
int sr_get_peaks(sr_ctx *ctx, int view, double *out) {
    CKR(check_view(ctx, view));
    if (!out) return SR_ERR_INVALID;
    if (ctx->peaks_view != view) return fail(ctx, SR_ERR_STATE, "no peak lists kept for this view (set keep_cost_volume |= 2 and run it)");
    return d2h_transposed(ctx, out, ctx->d_peaks, (size_t)ctx->w * ctx->h, 18);  // [9][2][pixel] -> [pixel][9][2]
}
int sr_set_depth(sr_ctx *ctx, int view, const double *depth) {
    CKR(check_view(ctx, view));
    CKR(enter(ctx));
    CK(cudaMemcpyAsync(ctx->views[view].depth, depth, (size_t)ctx->w * ctx->h * 8, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return SR_OK;
}
int sr_get_depth_image(sr_ctx *ctx, int view, int mvs, uint8_t *out) {
    CKR(check_view(ctx, view));
    CKR(check_params(ctx));
    if (!mvs) return fail(ctx, SR_ERR_INVALID, "two-view HSV depth image is produced by the host class (QColor semantics)");
    CKR(enter(ctx));  // the view may still be running on a lane
    const size_t n = (size_t)ctx->w * ctx->h;
    CKR(ensure_scratch(ctx, n * 4));
    depth_image_mvs_kernel<<<(unsigned)((n + 255) / 256), 256, 0, ctx->stream>>>(
        ctx->views[view].depth, ctx->views[view].mask, (int)n, ctx->params.min_depth, ctx->params.max_depth,
        (uchar4 *)ctx->d_scratch);
    CKL();
    return d2h(ctx, out, ctx->d_scratch, n * 4);
}

int sr_get_points(sr_ctx *ctx, int view, int64_t capacity, double *out_xyz, uint8_t *out_rgb, int32_t *out_pixel,
                  int64_t *out_count) {
    CKR(check_view(ctx, view));
    if (!out_count || capacity < 0 || (capacity > 0 && (!out_xyz || !out_rgb)))
        return fail(ctx, SR_ERR_INVALID, "sr_get_points: out_count, and out_xyz and out_rgb when capacity > 0, are required");
    CKR(check_params(ctx));
    if (!ctx->views[view].have_image) return fail(ctx, SR_ERR_STATE, "the view was given no image in sr_set_views");
    CKR(enter(ctx));  // the view may still be running on a lane
    const int h = ctx->h;
    PointsArgs pa;
    memset(&pa, 0, sizeof(pa));
    pa.cam = ctx->cams[view];
    pa.depth = ctx->views[view].depth;
    pa.rgba = ctx->views[view].rgba;
    pa.w = ctx->w;
    pa.h = h;
    pa.scale = ctx->params.image_scale;
    pa.min_depth = ctx->params.min_depth;
    // scratch: the row offsets; the points go to the output buffer
    CKR(ensure_scratch(ctx, (size_t)(h + 1) * sizeof(long long)));
    pa.offsets = (long long *)ctx->d_scratch;
    points_count_kernel<<<h, POINTS_THREADS, 0, ctx->stream>>>(pa);
    CKL();
    points_scan_kernel<<<1, POINTS_SCAN_THREADS, 0, ctx->stream>>>(pa.offsets, h);
    CKL();
    return fill_points(ctx, pa.offsets + h, capacity, out_count, "sr_get_points: capacity is smaller than the number of points",
                       out_xyz, out_rgb, out_pixel, 1, [&](double *xyz, int32_t *pixel, uint8_t *rgb) -> int {
                           pa.xyz = xyz;
                           pa.pixel = pixel;
                           pa.rgb = rgb;
                           points_write_kernel<<<h, POINTS_THREADS, 0, ctx->stream>>>(pa);
                           CKL();
                           return SR_OK;
                       });
}

int sr_fuse_points(sr_ctx *ctx, double max_dist, int min_views, int64_t capacity, double *out_xyz, uint8_t *out_rgb,
                   int32_t *out_source, int64_t *out_count) {
    if (!ctx) return SR_ERR_INVALID;
    if (!out_count || capacity < 0 || (capacity > 0 && (!out_xyz || !out_rgb)))
        return fail(ctx, SR_ERR_INVALID, "sr_fuse_points: out_count, and out_xyz and out_rgb when capacity > 0, are required");
    if (!(max_dist >= 0.0 && std::isfinite(max_dist)) || min_views < 0)
        return fail(ctx, SR_ERR_INVALID, "sr_fuse_points: max_dist must be finite and >= 0, min_views >= 0");
    if (ctx->V == 0) return fail(ctx, SR_ERR_STATE, "sr_set_views has not been called");
    CKR(check_params(ctx));
    for (const ViewDev &v : ctx->views)
        if (!v.have_image) return fail(ctx, SR_ERR_STATE, "sr_fuse_points: a view was given no image in sr_set_views");
    CKR(enter(ctx));  // a view may still be running on a lane
    const int rows = ctx->V * ctx->h;
    const size_t N = (size_t)ctx->V * ctx->w * ctx->h;
    FuseArgs fa;
    memset(&fa, 0, sizeof(fa));
    fa.cams = ctx->d_cams;
    fa.depth = ctx->d_depth_ptrs;
    fa.rgba = ctx->d_rgba_ptrs;
    fa.V = ctx->V;
    fa.w = ctx->w;
    fa.h = ctx->h;
    fa.scale = ctx->params.image_scale;
    fa.min_depth = ctx->params.min_depth;
    fa.max_dist = max_dist;
    fa.min_views = min_views;
    // scratch: [row offsets][fused xyz planes][support][rgbe]; the points go to the output buffer
    const size_t off_bytes = align256((size_t)(rows + 1) * sizeof(long long));
    CKR(ensure_scratch(ctx, off_bytes + N * (3 * sizeof(double) + sizeof(int32_t) + sizeof(uint32_t))));
    char *base = (char *)ctx->d_scratch;
    fa.offsets = (long long *)base;
    fa.fxyz = (double *)(base + off_bytes);
    fa.support = (int32_t *)(fa.fxyz + 3 * N);
    fa.rgbe = (uint32_t *)(fa.support + N);
    fuse_support_kernel<<<(unsigned)((N + FUSE_THREADS - 1) / FUSE_THREADS), FUSE_THREADS, 0, ctx->stream>>>(fa);
    CKL();
    fuse_emit_kernel<<<rows, POINTS_THREADS, 0, ctx->stream>>>(fa);
    CKL();
    points_scan_kernel<<<1, POINTS_SCAN_THREADS, 0, ctx->stream>>>(fa.offsets, rows);
    CKL();
    return fill_points(ctx, fa.offsets + rows, capacity, out_count, "sr_fuse_points: capacity is smaller than the number of points",
                       out_xyz, out_rgb, out_source, 2, [&](double *xyz, int32_t *source, uint8_t *rgb) -> int {
                           fa.xyz = xyz;
                           fa.source = source;
                           fa.rgb = rgb;
                           fuse_write_kernel<<<rows, POINTS_THREADS, 0, ctx->stream>>>(fa);
                           CKL();
                           return SR_OK;
                       });
}

void sr_mrf_params_default(sr_mrf_params *p) {
    if (!p) return;
    p->iterations = MRF_DEFAULT_ITERATIONS;
    p->unknown_cost = MRF_DEFAULT_UNKNOWN_COST;
    p->smooth_weight = MRF_DEFAULT_SMOOTH_WEIGHT;
    p->smooth_trunc = MRF_DEFAULT_SMOOTH_TRUNC;
    p->unknown_pair = MRF_DEFAULT_UNKNOWN_PAIR;
}

int sr_set_peaks(sr_ctx *ctx, int view, const double *peaks) {
    CKR(check_view(ctx, view));
    if (!peaks) return fail(ctx, SR_ERR_INVALID, "sr_set_peaks: peaks is null");
    const size_t n = (size_t)ctx->w * ctx->h;
    CKR(enter(ctx));
    ctx->peaks_view = -1;
    CKR(grow(ctx, ctx->stream, ctx->d_peaks, ctx->peaks_cap, n * 18 * 8));
    CKR(h2d_transposed(ctx, ctx->d_peaks, peaks, n, 18));  // [pixel][9][2] -> the device's [9][2][pixel]
    ctx->peaks_view = view;
    return SR_OK;
}

// A term of sr_mrf_params as the kernels use it: finite, >= 0, at most `cap`; +0 for a (signed) zero.
static bool mrf_term(double v, double cap, float &out) {
    if (!(v >= 0.0 && v <= cap)) return false;
    out = v == 0.0 ? 0.0f : (float)v;
    return true;
}

int sr_mrf_select(sr_ctx *ctx, int view, const sr_mrf_params *mp, double *out_energy) {
    CKR(check_view(ctx, view));
    if (!mp) return fail(ctx, SR_ERR_INVALID, "sr_mrf_select: params is null");
    CKR(check_params(ctx));
    if (ctx->peaks_view != view)
        return fail(ctx, SR_ERR_STATE, "no peak lists for this view (run it with keep_cost_volume |= 2, or sr_set_peaks)");
    const sr_params &P = ctx->params;
    const int w = ctx->w, h = ctx->h;
    const double step = (P.max_depth - P.min_depth) / (P.num_levels - 1.0);
    if (P.num_levels < 2 || !(step > 0.0 && std::isfinite(step)))
        return fail(ctx, SR_ERR_INVALID, "sr_mrf_select: needs num_levels >= 2 and max_depth > min_depth");
    if (!(P.ncc_threshold < 1.0 && std::isfinite(P.ncc_threshold)))
        return fail(ctx, SR_ERR_INVALID, "sr_mrf_select: ncc_threshold must be finite and < 1");
    if (std::max(P.row_begin, 0) > 0 || (P.row_end > 0 && P.row_end < h))
        return fail(ctx, SR_ERR_INVALID, "sr_mrf_select: the MRF needs the whole view (a row band is set in the params)");
    MrfArgs ma;
    memset(&ma, 0, sizeof(ma));
    const double cap = 1e30;
    if (mp->iterations < 0 || !mrf_term(mp->unknown_cost, cap, ma.du) || !mrf_term(mp->smooth_weight, cap, ma.weight) ||
        !mrf_term(mp->smooth_trunc, cap, ma.trunc) || !mrf_term(mp->unknown_pair, cap, ma.upair) ||
        !(mp->smooth_weight * mp->smooth_trunc <= cap))
            return fail(ctx, SR_ERR_INVALID, "sr_mrf_select: iterations must be >= 0 and every term finite, >= 0 and at most "
                                         "1e30 (smooth_weight * smooth_trunc too)");
    CKR(enter(ctx));
    const size_t n = (size_t)w * h;
    const unsigned blocks = (unsigned)((n + 255) / 256);
    // scratch: [messages 4*10*n][unary 9*n][z 9*n] floats, [labels n], [energy partials][energy]
    const size_t msg_bytes = (size_t)4 * MRF_L * n * sizeof(float), slot_bytes = (size_t)MRF_K * n * sizeof(float);
    const size_t lab_off = msg_bytes + 2 * slot_bytes, part_off = lab_off + align256(n);
    CKR(ensure_scratch(ctx, part_off + ((size_t)blocks + 1) * sizeof(double)));
    char *base = (char *)ctx->d_scratch;
    ViewDev &V = ctx->views[view];
    ma.mask = V.mask;
    ma.peaks = ctx->d_peaks;
    ma.msg = (float *)base;
    ma.unary = (float *)(base + msg_bytes);
    ma.zs = (float *)(base + msg_bytes + slot_bytes);
    ma.label = (uint8_t *)(base + lab_off);
    ma.partial = (double *)(base + part_off);
    ma.w = w;
    ma.h = h;
    mrf_prep_kernel<<<blocks, 256, 0, ctx->stream>>>(ma, 1.0 - P.ncc_threshold, step);
    CKL();
    CK(cudaMemsetAsync(ma.msg, 0, msg_bytes, ctx->stream));
    const dim3 sweep_grid((unsigned)(((w + 1) / 2 + MRF_THREADS - 1) / MRF_THREADS), (unsigned)h);
    for (int it = 0;; ++it) {
        if (ctx->cancel.load()) return fail(ctx, SR_ERR_CANCELLED, "cancelled");
        if (it == mp->iterations) break;
        for (int colour = 0; colour < 2; ++colour) {
            mrf_sweep_kernel<<<sweep_grid, MRF_THREADS, 0, ctx->stream>>>(ma, colour);
            CKL();
        }
    }
    mrf_label_kernel<<<blocks, 256, 0, ctx->stream>>>(ma, V.depth, V.best, V.index);
    CKL();
    if (!out_energy) return SR_OK;
    mrf_energy_kernel<<<blocks, 256, 0, ctx->stream>>>(ma);
    CKL();
    mrf_sum_kernel<<<1, MRF_SUM_THREADS, 0, ctx->stream>>>(ma.partial, (int)blocks, ma.partial + blocks);
    CKL();
    return d2h(ctx, out_energy, ma.partial + blocks, sizeof(double));
}

int sr_unproject_grid(sr_ctx *ctx, int view, double *out) {
    CKR(check_view(ctx, view));
    CKR(enter(ctx));
    const double scale = ctx->have_params ? ctx->params.image_scale : 1.0;
    CKR(launch_rays(ctx, ctx->cams[view], 0, ctx->h, scale, ctx->s.rays, ctx->stream));
    return d2h_transposed(ctx, out, ctx->s.rays, (size_t)ctx->w * ctx->h, 6);  // [6][h][w] -> [h][w][6]
}

int sr_project_points(sr_ctx *ctx, int view, int n, const double *xyz, double *out_xy, int32_t *out_ok) {
    CKR(check_view(ctx, view));
    if (n <= 0) return SR_OK;
    CKR(enter(ctx, false));
    CKR(ensure_scratch(ctx, (size_t)n * (24 + 16 + 4)));
    double *dx = (double *)ctx->d_scratch;
    double *dxy = dx + (size_t)3 * n;
    int32_t *dok = (int32_t *)(dxy + (size_t)2 * n);
    CK(cudaMemcpyAsync(dx, xyz, (size_t)n * 24, cudaMemcpyHostToDevice, ctx->stream));
    project_points_kernel<<<(n + 127) / 128, 128, 0, ctx->stream>>>(ctx->cams[view], n, dx, dxy, dok);
    CKL();
    CK(cudaMemcpyAsync(out_xy, dxy, (size_t)n * 16, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(out_ok, dok, (size_t)n * 4, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return SR_OK;
}

int sr_compute_weights(sr_ctx *ctx, int view, int kind, int radius, int n, const int32_t *cx, const int32_t *cy,
                       double *out) {
    CKR(check_view(ctx, view));
    if (n <= 0) return SR_OK;
    if (radius < 1 || radius > 64 || kind < 0 || kind > 1) return fail(ctx, SR_ERR_INVALID, "bad radius/kind");
    CKR(enter(ctx, false));
    const size_t wn = (size_t)(2 * radius + 1) * (2 * radius + 1);
    CKR(ensure_scratch(ctx, (size_t)n * 8 + (size_t)n * wn * 8));
    int32_t *dcx = (int32_t *)ctx->d_scratch;
    int32_t *dcy = dcx + n;
    double *dW = (double *)(dcy + n);
    CK(cudaMemcpyAsync(dcx, cx, (size_t)n * 4, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(dcy, cy, (size_t)n * 4, cudaMemcpyHostToDevice, ctx->stream));
    CKR(launch_weights(ctx, ctx->views[view], kind, radius, dW, 0, 0, ctx->stream, dcx, dcy, n));
    return d2h_transposed(ctx, out, dW, (size_t)n, wn);  // [tap][centre] -> [centre][row][col]
}

int sr_calibration_residuals_batch(sr_ctx *ctx, int num_models, int num_cams, const sr_camera *cams, int n,
                                   const int32_t *view_pairs, const double *pixels, double *out) {
    if (!ctx || !cams || num_models <= 0 || num_models > 65535 || num_cams <= 0 || n < 0 ||
        (n > 0 && (!view_pairs || !pixels || !out)))
        return SR_ERR_INVALID;
    if (n == 0) return SR_OK;
    for (int i = 0; i < 2 * n; ++i)
        if (view_pairs[i] < 0 || view_pairs[i] >= num_cams) return fail(ctx, SR_ERR_INVALID, "camera index out of range");
    CKR(enter(ctx, false));
    const size_t ncam = (size_t)num_models * num_cams;
    const size_t cam_bytes = align256(sizeof(sr_camera) * ncam);
    CKR(ensure_scratch(ctx, cam_bytes + (size_t)n * (32 + 8) + (size_t)num_models * n * 8));
    char *base = (char *)ctx->d_scratch;
    sr_camera *dc = (sr_camera *)base;
    double *dpix = (double *)(base + cam_bytes);
    double *dout = dpix + (size_t)4 * n;
    int32_t *dpairs = (int32_t *)(dout + (size_t)num_models * n);
    CK(cudaMemcpyAsync(dc, cams, sizeof(sr_camera) * ncam, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(dpix, pixels, (size_t)n * 32, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(dpairs, view_pairs, (size_t)n * 8, cudaMemcpyHostToDevice, ctx->stream));
    calibration_residual_kernel<<<dim3((unsigned)((n + 127) / 128), (unsigned)num_models), 128, 0, ctx->stream>>>(
        dc, num_cams, n, dpairs, dpix, dout);
    CKL();
    CK(cudaMemcpyAsync(out, dout, (size_t)num_models * n * 8, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return SR_OK;
}

int sr_calibration_residuals(sr_ctx *ctx, int num_cams, const sr_camera *cams, int n, const int32_t *view_pairs,
                             const double *pixels, double *out) {
    return sr_calibration_residuals_batch(ctx, 1, num_cams, cams, n, view_pairs, pixels, out);
}

// ---- multi-GPU ---------------------------------------------------------------------------
int sr_comm_unique_id(void *out128) {
    std::string err;
    if (!load_nccl(err)) return fail(nullptr, SR_ERR_NCCL, err);
    int r = g_nccl.GetUniqueId(out128);
    if (r != 0) return fail(nullptr, SR_ERR_NCCL, g_nccl.GetErrorString(r));
    return SR_OK;
}

int sr_comm_init(sr_ctx *ctx, const void *uid128, int rank, int nranks) {
    if (!ctx || !uid128 || nranks < 1 || rank < 0 || rank >= nranks) return SR_ERR_INVALID;
    std::string err;
    if (!load_nccl(err)) return fail(ctx, SR_ERR_NCCL, err);
    CKR(enter(ctx, false));
    Uid128 id;
    memcpy(id.b, uid128, 128);
    int r = g_nccl.CommInitRank(&ctx->comm, nranks, id, rank);
    if (r != 0) return fail(ctx, SR_ERR_NCCL, g_nccl.GetErrorString(r));
    ctx->rank = rank;
    ctx->nranks = nranks;
    return SR_OK;
}

// Broadcast pixels [off, off + cnt) of the depth, index and best maps of view d from rank `root`; an NCCL result.
static int bcast_maps(sr_ctx *ctx, ViewDev &d, size_t off, size_t cnt, int root) {
    int r = g_nccl.Broadcast(d.depth + off, d.depth + off, cnt * 8, NCCL_CHAR, root, ctx->comm, ctx->stream);
    if (r == 0) r = g_nccl.Broadcast(d.index + off, d.index + off, cnt * 4, NCCL_CHAR, root, ctx->comm, ctx->stream);
    if (r == 0) r = g_nccl.Broadcast(d.best + off, d.best + off, cnt * 8, NCCL_CHAR, root, ctx->comm, ctx->stream);
    return r;
}

// All-gather realised as one broadcast per view from its owner (views are whole buffers owned
// by exactly one rank, so a grouped broadcast moves each byte once over NVLink).
int sr_comm_allgather_views(sr_ctx *ctx, const int32_t *owner) {
    if (!ctx || !owner) return SR_ERR_INVALID;
    if (!ctx->comm) return fail(ctx, SR_ERR_STATE, "sr_comm_init has not been called");
    for (int v = 0; v < ctx->V; ++v)
        if (owner[v] < 0 || owner[v] >= ctx->nranks) return fail(ctx, SR_ERR_INVALID, "sr_comm_allgather_views: owner rank out of range");
    CKR(enter(ctx));
    const size_t n = (size_t)ctx->w * ctx->h;
    int r = g_nccl.GroupStart();
    for (int v = 0; v < ctx->V && r == 0; ++v) r = bcast_maps(ctx, ctx->views[v], 0, n, owner[v]);
    int r2 = g_nccl.GroupEnd();
    if (r == 0) r = r2;
    if (r != 0) return fail(ctx, SR_ERR_NCCL, g_nccl.GetErrorString(r));
    return SR_OK;
}

int sr_comm_allgather_rows(sr_ctx *ctx, int view, const int32_t *row_begin, const int32_t *row_end) {
    CKR(check_view(ctx, view));
    if (!ctx->comm) return fail(ctx, SR_ERR_STATE, "sr_comm_init has not been called");
    if (!row_begin || !row_end) return fail(ctx, SR_ERR_INVALID, "sr_comm_allgather_rows: null row ranges");
    for (int k = 0; k < ctx->nranks; ++k)
        if (row_begin[k] < 0 || row_begin[k] > row_end[k] || row_end[k] > ctx->h)
            return fail(ctx, SR_ERR_INVALID, "sr_comm_allgather_rows: need 0 <= row_begin <= row_end <= height for every rank");
    CKR(enter(ctx));
    ViewDev &d = ctx->views[view];
    int r = g_nccl.GroupStart();
    for (int k = 0; k < ctx->nranks && r == 0; ++k) {
        const size_t off = (size_t)row_begin[k] * ctx->w, cnt = (size_t)(row_end[k] - row_begin[k]) * ctx->w;
        if (cnt > 0) r = bcast_maps(ctx, d, off, cnt, k);
    }
    int r2 = g_nccl.GroupEnd();
    if (r == 0) r = r2;
    if (r != 0) return fail(ctx, SR_ERR_NCCL, g_nccl.GetErrorString(r));
    return SR_OK;
}

}  // extern "C"
