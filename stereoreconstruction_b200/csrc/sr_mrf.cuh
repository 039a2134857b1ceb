// sr_mrf.cuh — the MRF stage of the multiple-hypothesis multi-view stereo (sr_mrf_select): choose, for every
// in-mask pixel of one view, one of the K = 9 (ncc, depth) hypotheses of its peak list or "unknown", by min-sum
// loopy belief propagation over the 4-connected pixel grid on a checkerboard schedule (Felzenszwalb &
// Huttenlocher 2006).  The model is stated in include/sr_b200.h; tests/mrf_util.py restates it in NumPy.
//
//   mrf_prep_kernel   per pixel: FP32 unary D(k) and FP32 z(k) / step of the 9 slots from the FP64 lists
//   mrf_sweep_kernel  one thread per pixel of one colour ((x + y) & 1 == colour): the messages to its 4
//                     neighbours, written into each receiver's slot for that direction
//   mrf_label_kernel  per pixel: argmin of D + the four incoming messages; writes the view's maps
//   mrf_energy_kernel per pixel: unary + right and lower pairwise terms of the final labelling, summed in FP64
//                     to one partial per block
//   mrf_sum_kernel    one block: the partials summed in a fixed order
//
// Every FP32 operation of the sweep and labelling is an explicit round-to-nearest intrinsic, so the results do
// not depend on FMA contraction.  A slot of the receiver's mailbox has exactly one writer per half-sweep (its
// neighbour on that side), and a half-sweep reads only mailboxes of the colour it does not write: no atomics,
// no races, the same bits on every run.
#pragma once
#include <cfloat>
#include "sr_kernels.cuh"

namespace sr {

constexpr int MRF_K = 9;          // hypothesis slots of a peak list
constexpr int MRF_U = MRF_K;      // the unknown label
constexpr int MRF_L = MRF_K + 1;  // labels of a pixel
constexpr int MRF_THREADS = 128;
constexpr int MRF_SUM_THREADS = 1024;

// sr_mrf_params_default (the measurements behind them: DESIGN.md §7)
constexpr int MRF_DEFAULT_ITERATIONS = 16;
constexpr double MRF_DEFAULT_UNKNOWN_COST = 1.0;
constexpr double MRF_DEFAULT_SMOOTH_WEIGHT = 0.15;
constexpr double MRF_DEFAULT_SMOOTH_TRUNC = 6.0;
constexpr double MRF_DEFAULT_UNKNOWN_PAIR = 0.3;

// Message directions: msg[d] of a pixel holds what it received from its left (0), right (1), upper (2) and
// lower (3) neighbour.
struct MrfArgs {
    const uint8_t *mask;   // [h][w], 255 = in the model
    const double *peaks;   // [9][2][h*w] (ncc, depth)
    float *unary;          // [9][h*w] D(k); +INF for a slot that is no hypothesis
    float *zs;             // [9][h*w] z(k) / step; NaN for a slot that is no hypothesis
    float *msg;            // [4][10][h*w]
    uint8_t *label;        // [h*w] 0..8, or MRF_U
    double *partial;       // [blocks of mrf_energy_kernel]
    int w, h;
    float du;      // D(U) = unknown_cost
    float weight;  // smooth_weight
    float trunc;   // smooth_trunc
    float upair;   // V(k, U) = V(U, k)
};

__device__ __forceinline__ float finf() { return __int_as_float(0x7f800000); }
__device__ __forceinline__ float fnan() { return __int_as_float(0x7fffffff); }

// V(k, l) of two hypotheses, given their z / step.
__device__ __forceinline__ float mrf_vpair(const MrfArgs &a, float zk, float zl) {
    return __fmul_rn(a.weight, fminf(fabsf(__fsub_rn(zk, zl)), a.trunc));
}

// A slot is a hypothesis when its ncc and depth are finite and it is not the padding (0, -1).
// D(k) = max(0, (1 - ncc) / (1 - ncc_threshold)) and z / step are computed in FP64 and rounded to FP32 once
// (z / step clamped to the finite FP32 range first).
__global__ void __launch_bounds__(256) mrf_prep_kernel(const MrfArgs a, double one_minus_thr, double step) {
    const size_t n = (size_t)a.w * a.h;
    const size_t p = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n || a.mask[p] != 255) return;
#pragma unroll
    for (int k = 0; k < MRF_K; ++k) {
        const double c = a.peaks[(size_t)(2 * k) * n + p], z = a.peaks[(size_t)(2 * k + 1) * n + p];
        float d = finf(), s = fnan();
        if (isfinite(c) && isfinite(z) && !(c == 0.0 && z == -1.0)) {
            d = __double2float_rn(fmax(__ddiv_rn(__dsub_rn(1.0, c), one_minus_thr), 0.0));
            s = __double2float_rn(fmin(fmax(__ddiv_rn(z, step), -(double)FLT_MAX), (double)FLT_MAX));
        }
        a.unary[(size_t)k * n + p] = d;
        a.zs[(size_t)k * n + p] = s;
    }
}

// m(l) = min_k [D(k) + the incoming messages except the receiver's (left, right, up, down order) + V(k, l)],
// then min_l m(l) subtracted.  Entries for a receiver's non-hypothesis slots are 0 and take no part in the
// minimum; they never matter, as the receiver's D there is +INF.
__global__ void __launch_bounds__(MRF_THREADS) mrf_sweep_kernel(const MrfArgs a, int colour) {
    const int y = blockIdx.y;
    const int x = 2 * (int)(blockIdx.x * MRF_THREADS + threadIdx.x) + ((y + colour) & 1);
    if (x >= a.w) return;
    const int w = a.w;
    const size_t n = (size_t)w * a.h, p = (size_t)y * w + x;
    if (a.mask[p] != 255) return;
    float D[MRF_L], z[MRF_K], in[4][MRF_L];
#pragma unroll
    for (int k = 0; k < MRF_K; ++k) {
        D[k] = a.unary[(size_t)k * n + p];
        z[k] = a.zs[(size_t)k * n + p];
    }
    D[MRF_U] = a.du;
#pragma unroll
    for (int d = 0; d < 4; ++d)
#pragma unroll
        for (int l = 0; l < MRF_L; ++l) in[d][l] = a.msg[(size_t)(d * MRF_L + l) * n + p];
    const bool has[4] = {x > 0 && a.mask[p - 1] == 255, x + 1 < w && a.mask[p + 1] == 255,
                         y > 0 && a.mask[p - w] == 255, y + 1 < a.h && a.mask[p + w] == 255};
    const long long off[4] = {-1, 1, -(long long)w, (long long)w};
    const int slot[4] = {1, 0, 3, 2};  // the receiver hears this pixel from its right, left, lower, upper side
#pragma unroll
    for (int t = 0; t < 4; ++t) {
        if (!has[t]) continue;
        float S[MRF_L];
#pragma unroll
        for (int l = 0; l < MRF_L; ++l) {
            float s = D[l];
#pragma unroll
            for (int d = 0; d < 4; ++d)
                if (d != t) s = __fadd_rn(s, in[d][l]);
            S[l] = s;
        }
        float hmin = finf();  // min over the hypotheses k of S(k)
#pragma unroll
        for (int k = 0; k < MRF_K; ++k)
            if (z[k] == z[k]) hmin = fminf(hmin, S[k]);
        const size_t q = (size_t)((long long)p + off[t]);
        const float from_u = __fadd_rn(S[MRF_U], a.upair);
        float m[MRF_L];
        m[MRF_U] = fminf(S[MRF_U], __fadd_rn(hmin, a.upair));
        float mn = m[MRF_U];
        unsigned qhyp = 0;
#pragma unroll
        for (int l = 0; l < MRF_K; ++l) {
            const float zq = a.zs[(size_t)l * n + q];
            float v = from_u;
            if (zq == zq) {
                qhyp |= 1u << l;
#pragma unroll
                for (int k = 0; k < MRF_K; ++k)
                    if (z[k] == z[k]) v = fminf(v, __fadd_rn(S[k], mrf_vpair(a, z[k], zq)));
                mn = fminf(mn, v);
            }
            m[l] = v;
        }
        float *out = a.msg + (size_t)(slot[t] * MRF_L) * n + q;
#pragma unroll
        for (int l = 0; l < MRF_L; ++l)
            out[(size_t)l * n] = (l == MRF_U || ((qhyp >> l) & 1u)) ? __fsub_rn(m[l], mn) : 0.0f;
    }
}

// Belief b(k) = D(k) + from left + from right + from up + from down; the highest hypothesis slot wins a tie
// and U loses every tie.  Writes the view's maps: the chosen hypothesis's FP64 depth and ncc and its slot, or
// -1 / 0 / SR_INDEX_NONE for U (what the winner-take-all writes for a pixel without a candidate).
__global__ void __launch_bounds__(256) mrf_label_kernel(const MrfArgs a, double *depth, double *best, int32_t *index) {
    const size_t n = (size_t)a.w * a.h;
    const size_t p = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n || a.mask[p] != 255) return;
    auto belief = [&](int l, float d) {
#pragma unroll
        for (int dir = 0; dir < 4; ++dir) d = __fadd_rn(d, a.msg[(size_t)(dir * MRF_L + l) * n + p]);
        return d;
    };
    float b = belief(MRF_U, a.du);
    int lab = MRF_U;
#pragma unroll
    for (int k = 0; k < MRF_K; ++k) {
        const float zk = a.zs[(size_t)k * n + p];
        if (zk != zk) continue;
        const float bk = belief(k, a.unary[(size_t)k * n + p]);
        if (bk <= b) {
            b = bk;
            lab = k;
        }
    }
    a.label[p] = (uint8_t)lab;
    if (lab == MRF_U) {
        depth[p] = -1.0;
        best[p] = 0.0;
        index[p] = SR_INDEX_NONE;
    } else {
        depth[p] = a.peaks[(size_t)(2 * lab + 1) * n + p];
        best[p] = a.peaks[(size_t)(2 * lab) * n + p];
        index[p] = lab;
    }
}

__device__ __forceinline__ float mrf_pair_term(const MrfArgs &a, size_t n, size_t p, int lp, size_t q, int lq) {
    if (lp == MRF_U && lq == MRF_U) return 0.0f;
    if (lp == MRF_U || lq == MRF_U) return a.upair;
    return mrf_vpair(a, a.zs[(size_t)lp * n + p], a.zs[(size_t)lq * n + q]);
}

// Per in-mask pixel, in FP64: its unary term, plus the pairwise term of its edge to the right, plus that of its
// edge downwards (edges between two in-mask pixels only); summed over the block by a fixed tree.
__global__ void __launch_bounds__(256) mrf_energy_kernel(const MrfArgs a) {
    __shared__ double sh[256];
    const int w = a.w;
    const size_t n = (size_t)w * a.h;
    const size_t p = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    double e = 0.0;
    if (p < n && a.mask[p] == 255) {
        const int lp = a.label[p];
        const int x = (int)(p % w);
        e = (double)(lp == MRF_U ? a.du : a.unary[(size_t)lp * n + p]);
        if (x + 1 < w && a.mask[p + 1] == 255) e += (double)mrf_pair_term(a, n, p, lp, p + 1, a.label[p + 1]);
        if (p + w < n && a.mask[p + w] == 255) e += (double)mrf_pair_term(a, n, p, lp, p + w, a.label[p + w]);
    }
    sh[threadIdx.x] = e;
    __syncthreads();
    for (int s = 128; s > 0; s >>= 1) {
        if ((int)threadIdx.x < s) sh[threadIdx.x] += sh[threadIdx.x + s];
        __syncthreads();
    }
    if (threadIdx.x == 0) a.partial[blockIdx.x] = sh[0];
}

// out[0] = the sum of partial[0..count): each thread a strided run, then a fixed tree.
__global__ void __launch_bounds__(MRF_SUM_THREADS) mrf_sum_kernel(const double *partial, int count, double *out) {
    __shared__ double sh[MRF_SUM_THREADS];
    double s = 0.0;
    for (int i = threadIdx.x; i < count; i += MRF_SUM_THREADS) s += partial[i];
    sh[threadIdx.x] = s;
    __syncthreads();
    for (int k = MRF_SUM_THREADS / 2; k > 0; k >>= 1) {
        if ((int)threadIdx.x < k) sh[threadIdx.x] += sh[threadIdx.x + k];
        __syncthreads();
    }
    if (threadIdx.x == 0) out[0] = sh[0];
}

}  // namespace sr
