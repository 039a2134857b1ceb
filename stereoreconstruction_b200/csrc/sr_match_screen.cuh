// sr_match_screen.cuh — stages (2)+(3) for the MultiViewStereo selection rule, organised as an
// FP32 screening pass with an FP64 verification of the few labels that can win.  This file holds the
// error bars, the FP64 verification (verify_cost_mvs) and the kernel for the radii whose window is
// shared by a group of G > 1 lanes per pixel (r >= 3: LanesFor in sr_match_dispatch.cuh).  The
// thread-per-pixel radii (r <= 2) run the one-pass form of sr_screen2.cuh.
//
// What the reference computes per reference pixel (stereo/multiviewstereo.cpp:583-602,654-660):
// the weighted NCC (cost_ncc, :113-189) of every candidate, keeps those with ncc > 0.95 and
// returns the candidate that is largest under (ncc, depth) ordering.  Only the *winner* and its
// exact cost leave the kernel, so all but a handful of the D x N_nbr evaluations only need to be
// accurate enough to prove that they cannot be the winner:
//
//   screen (FP32)  ncc32 of every (label, neighbour) by the reference's own two-pass form
//                  t_i = w_i*g_i - meanR;  s3 = sum t_i^2;  s1 = sum dl_i*t_i;  ncc = s1/sqrt(s2*s3)
//                  on FP32 copies of the gray planes.  Each lane of a pixel's group holds every G-th
//                  tap of the window (weights, dl_i and the loaded taps in registers; dl_i is stored
//                  divided by sqrt(s2), rounded once from FP64, so ncc32 = s1 * rsqrt(s3)) and the
//                  partial sums meet in a shuffle butterfly.  Every screened value carries an error
//                  bar eps (SCREEN_EPS_*, by conditioning of the two windows); ill-conditioned windows
//                  and windows touching the neighbour's border are FORCEd into the verified set.
//   candidates     lower32 = max(threshold, max over labels of ncc32 - eps) is a proven lower
//                  bound of the winning ncc64, so a label can only win if ncc32 + eps >= lower32.
//                  Candidates live in a small per-pixel queue in shared memory; entries whose
//                  upper bound falls below a risen lower32 are evicted.
//   verify (FP64)  when a queue fills (and at the end) each lane group walks its pixel's queue in
//                  order and evaluates the candidates with the reference's exact two-pass tap filter
//                  in FP64, operation for operation (verify_cost_mvs / slow_cost), applying the
//                  reference's selection rule as it goes.  The result is the reference's winner, its
//                  depth and its FP64 cost; the screening precision never reaches the output.
//
// Consecutive labels whose projections truncate to the same integer tap have the same cost by
// construction; the queue keeps one entry per distinct tap (carrying the label the tie-break would
// pick).  The screen itself re-evaluates them: skipping only pays when all 32 lanes of a warp
// repeat at once, and the bookkeeping cost three live registers and ~5 % of the kernel.
#pragma once
#include <type_traits>
#include "sr_kernels.cuh"

namespace sr {

// Error bars of the screened ncc (|ncc32 - ncc64| <= eps), by conditioning of the two windows.
// With u = 2^-24: the two FFMA chains of s1 and s3 are <= 13 long (<= 13u relative each), and an
// input perturbation dt of the deviation vector t moves ncc by at most sqrt(1-ncc^2)*|dt|/|t|
// (<= 0.31 for ncc >= 0.95); |dt| <= sqrt(WN)*(2u*255 + 13u*|meanR|) ~ 6e-4 for a 5x5 window.
//   |t|^2 = s3 >= 100*WN (RMS deviation of 10 gray levels, the normal case): <= ~5e-6 -> TIGHT
//   s3 >= WN: <= ~4e-5 -> LOOSE;   below that the label is FORCEd into the verified set.
// SR_MATCH_STATS=1 records the largest |ncc32 - ncc64| actually seen on verified labels.
constexpr float SCREEN_EPS_TIGHT = 1e-5f;
constexpr float SCREEN_EPS_LOOSE = 2e-4f;
constexpr float SCREEN_FORCE = 3.0e38f;  // "must be verified in FP64" marker (|ncc| <= 1 otherwise)
constexpr int SCREEN_QCAP = 8;  // candidate queue entries per pixel

// Packed FP32 FMA of sm_100 (SASS FFMA2): two independent fused multiply-adds per issue slot.
__device__ __forceinline__ float2 fma2(float2 a, float2 b, float2 c) {
    unsigned long long ua, ub, uc, ud;
    asm("mov.b64 %0, {%1, %2};" : "=l"(ua) : "f"(a.x), "f"(a.y));
    asm("mov.b64 %0, {%1, %2};" : "=l"(ub) : "f"(b.x), "f"(b.y));
    asm("mov.b64 %0, {%1, %2};" : "=l"(uc) : "f"(c.x), "f"(c.y));
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(ud) : "l"(ua), "l"(ub), "l"(uc));
    float2 d;
    asm("mov.b64 {%0, %1}, %2;" : "=f"(d.x), "=f"(d.y) : "l"(ud));
    return d;
}

template <int G>
__device__ __forceinline__ float group_sum_f(float v, unsigned gmask) {
#pragma unroll
    for (int o = G / 2; o > 0; o >>= 1) v += __shfl_xor_sync(gmask, v, o);
    return v;
}

// cost_ncc of stereo/multiviewstereo.cpp:113-189 in FP64 for the common case "both windows
// inside their images, every tap active" — the reference's two passes, tap order and operation
// order (no FMA contraction: the library is built with -fmad=false), with the label-independent
// left-window quantities (meanL, sum of weights, s2) computed once per pixel in the same order.
// G == 1 is bit-identical to the reference; G > 1 sums the lanes' partial sums in a butterfly.
template <int R, int G>
__device__ __noinline__ double verify_cost_mvs(const MatchArgs &a, const double *__restrict__ gR, int x, int y, int tx,
                                               int ty, int pid, int sub, unsigned gmask, double meanL, double totW,
                                               double s2) {
    constexpr int WS = 2 * R + 1, WN = WS * WS;
    const int w = a.w;
    const size_t npix = (size_t)a.rows * w;
    const double *__restrict__ Wp = a.W + pid;
    const double *__restrict__ bl = a.grayL + ((size_t)y * w + x);
    const double *__restrict__ br = gR + ((size_t)ty * w + tx);
    double mR = 0.0;
#pragma unroll 5
    for (int k = sub; k < WN; k += G) {
        const int o = (k / WS - R) * w + (k % WS - R);
        mR += Wp[(size_t)k * npix] * br[o];
    }
    mR = group_sum<G>(mR, gmask) / totW;
    double q1 = 0.0, q3 = 0.0;
#pragma unroll 5
    for (int k = sub; k < WN; k += G) {
        const int o = (k / WS - R) * w + (k % WS - R);
        const double wt = Wp[(size_t)k * npix];
        const double pl = wt * bl[o] - meanL, pr = wt * br[o] - mR;
        q1 += pl * pr;
        q3 += pr * pr;
    }
    q1 = group_sum<G>(q1, gmask);
    q3 = group_sum<G>(q3, gmask);
    return (s2 * q3 < 1e-10) ? 0.0 : q1 / sqrt(s2 * q3);
}

// Threads per block: the kernel has no block-wide step, so a block is one warp and a slow warp
// (verification-heavy pixels) holds no other warp's slot.
constexpr int SCREEN_BLOCK = 32;
constexpr int SCREEN_MINBLOCKS = 8;  // resident blocks per SM the register allocation must allow (8 warps)

template <int R, int G, bool STATS>
__global__ void __launch_bounds__(SCREEN_BLOCK, SCREEN_MINBLOCKS) match_mvs_screen_kernel(const __grid_constant__ MatchArgs a) {
    static_assert(G > 1, "thread-per-pixel radii run match_mvs_screen2_kernel (sr_screen2.cuh)");
    constexpr int COST = SR_COST_NCC_MVS;
    constexpr int WS = 2 * R + 1;
    constexpr int WN = WS * WS;
    constexpr int TPL = (WN + G - 1) / G;
    constexpr int PIX_PER_BLOCK = SCREEN_BLOCK / G;
    __shared__ int32_t tap_ring[2][TAP_CHUNK][SCREEN_BLOCK];
    __shared__ int32_t q_lab[SCREEN_QCAP][SCREEN_BLOCK];  // (eps class << 30) | (neighbour << 16) | label
    __shared__ int32_t q_tap[SCREEN_QCAP][SCREEN_BLOCK];
    __shared__ float q_c32[SCREEN_QCAP][SCREEN_BLOCK];    // upper bound ncc32 + eps
    // Per-pixel state that only the verification step touches lives in shared memory, so that the
    // label loop keeps its registers for the window (w, dl, taps): exact left-window quantities
    // in the reference's summation order, and the verified winner so far.
    __shared__ double px_meanL[SCREEN_BLOCK], px_totW[SCREEN_BLOCK], px_s2[SCREEN_BLOCK], px_bestC[SCREEN_BLOCK];
    __shared__ int px_bestIdx[SCREEN_BLOCK];
    __shared__ double px_bestZ[SCREEN_BLOCK];  // curve mode: depth hypothesis of the verified winner
    __shared__ unsigned long long px_act[SCREEN_BLOCK];  // bit i: this lane's i-th tap is active (TPL <= 35)

    const int tid = threadIdx.x;
    const int lane = tid & 31;
    const int sub = tid % G;
    const unsigned gmask = (G == 32) ? 0xffffffffu : (((1u << G) - 1u) << (lane & ~(G - 1)));
    const int w = a.w, h = a.h;
    const int fp = a.pitch_f;
    const int npix_i = a.rows * w;
    const size_t npix = (size_t)npix_i;
    const int pid_raw = blockIdx.x * PIX_PER_BLOCK + tid / G;
    const bool in_band = pid_raw < npix_i;
    const int pid = in_band ? pid_raw : npix_i - 1;  // out-of-band lanes shadow the last pixel (no writes)
    const int x = pid % w, y = a.row0 + pid / w;
    const size_t pix = (size_t)y * w + x;
    // Lanes stay in the loops (warp-wide votes below); `alive` gates all work and all writes.
    const bool alive = in_band && a.maskL[pix] == 255;
    if (in_band && !alive && sub == 0) {  // multiviewstereo.cpp:559,565: masked-out pixels stay INF
        a.out_index[pix] = SR_INDEX_MASKED;
        a.out_depth[pix] = dinf();
        a.out_best[pix] = qnan();
    }

    // ---- reference-window invariants, FP64 (once per pixel) ----------------------------------
    // dlf carries 1/sqrt(s2): ncc32 = (sum dlf_i t_i) * rsqrt(s3), one rounding per element as before
    float wtf[TPL], dlf[TPL];
    bool all_slow = false, has_inactive = false;
    float inv_totWf = 0.0f, eps_pix = SCREEN_EPS_LOOSE;
    {
        double wt[TPL], gl[TPL];
        double totW = 0.0, SL = 0.0;
        int ninact = 0;
        unsigned long long actmask = 0ull;
#pragma unroll
        for (int i = 0; i < TPL; ++i) {
            const int k = sub + G * i;
            const int row = k / WS - R, col = k % WS - R;
            const int xl = x + col, yl = y + row;
            double g = qnan(), wv = 0.0;
            if (alive && k < WN && xl >= 0 && yl >= 0 && xl < w && yl < h) {
                g = a.grayL[(size_t)yl * w + xl];
                wv = a.W[(size_t)k * npix + pid];
            }
            const bool active = (g == g) && (wv > 1e-10);
            wt[i] = active ? wv : 0.0;
            gl[i] = active ? g : 0.0;
            if (active) {
                actmask |= 1ull << i;
                totW += wv;
                SL += wv * g;
            } else if (k < WN) {
                ++ninact;
            }
        }
        totW = group_sum<G>(totW, gmask);
        SL = group_sum<G>(SL, gmask);
        ninact = group_sum_i<G>(ninact, gmask);
        const double meanL = SL / totW;
        double s2 = 0.0;
#pragma unroll
        for (int i = 0; i < TPL; ++i) {
            const double dl = (wt[i] > 0.0) ? wt[i] * gl[i] - meanL : 0.0;
            s2 += dl * dl;
            wtf[i] = (float)wt[i];
            gl[i] = dl;
        }
        s2 = group_sum<G>(s2, gmask);
        const double rs2 = (s2 >= (double)WN && s2 < 1e30) ? 1.0 / sqrt(s2) : 0.0;  // otherwise all_slow: dlf unused
#pragma unroll
        for (int i = 0; i < TPL; ++i) dlf[i] = (float)(gl[i] * rs2);
        // An ill-conditioned reference side is evaluated only by the exact FP64 filter.  Inactive
        // taps (outside the image, weight <= 1e-10) carry w = dl = 0 through the screen and their
        // t_i is masked out of s3 (screen_one<true>, taken only by the warps that hold such a pixel).
        all_slow = !(totW >= 1e-10) || !(s2 >= (double)WN) || !(s2 < 1e30);
        has_inactive = ninact != 0;
        eps_pix = (s2 >= 100.0 * WN) ? SCREEN_EPS_TIGHT : SCREEN_EPS_LOOSE;
        inv_totWf = (float)(1.0 / totW);
        px_meanL[tid] = meanL;
        px_totW[tid] = totW;
        px_s2[tid] = s2;
        px_act[tid] = actmask;
        px_bestC[tid] = 0.0;
        px_bestIdx[tid] = SR_INDEX_NONE;
        px_bestZ[tid] = -1.0;
    }
    // keep the FP32 copies as values of their own (otherwise they are re-derived from the FP64
    // ones with an F2F / DSETP inside the label loop)
    asm volatile("" : "+f"(eps_pix), "+f"(inv_totWf));

    // ---- FP32 screening of one label: returns ncc32 or SCREEN_FORCE ---------------------------
    // Taps are processed in pairs (2p, 2p+1) with the packed FFMA2 (fma.rn.f32x2): the pair of
    // accumulators is the even/odd split a scalar version would use anyway, and the issue slots of
    // the window arithmetic halve (4 FFMA2 per two taps instead of 8 FFMA).
    auto screen_one = [&](const float *__restrict__ base, float &eps, auto masked_tag) -> float {
        constexpr bool MASKED = decltype(masked_tag)::value;
        constexpr int NP = TPL / 2;          // full pairs
        constexpr bool ODD = (TPL & 1) != 0; // one scalar tap left over
        float g[TPL];
#pragma unroll
        for (int i = 0; i < TPL; ++i) {
            const int k = sub + G * i;
            g[i] = 0.0f;
            if (k < WN) g[i] = base[(k / WS - R) * fp + (k % WS - R)];
        }
        // three independent accumulator pairs per sum: the dependent FFMA2 chains stay short
        float2 S1p[3] = {make_float2(0.0f, 0.0f), make_float2(0.0f, 0.0f), make_float2(0.0f, 0.0f)};
#pragma unroll
        for (int p = 0; p < NP; ++p)
            S1p[p % 3] = fma2(make_float2(wtf[2 * p], wtf[2 * p + 1]), make_float2(g[2 * p], g[2 * p + 1]), S1p[p % 3]);
        float S1s = ((S1p[0].x + S1p[0].y) + (S1p[1].x + S1p[1].y)) + (S1p[2].x + S1p[2].y);
        if (ODD) S1s = fmaf(wtf[TPL - 1], g[TPL - 1], S1s);
        const float S1 = group_sum_f<G>(S1s, gmask);
        const float mR = S1 * inv_totWf;
        const float2 nm = make_float2(-mR, -mR);
        float2 s3p[2] = {make_float2(0.0f, 0.0f), make_float2(0.0f, 0.0f)};
        float2 s1p[2] = {make_float2(0.0f, 0.0f), make_float2(0.0f, 0.0f)};
        unsigned long long actmask = 0ull;
        if (MASKED) actmask = px_act[tid];
        auto mask_of = [&](int i) -> int {  // 0 / ~0: tap i is active (bfe.s32 of one bit)
            const unsigned word = (i < 32) ? (unsigned)actmask : (unsigned)(actmask >> 32);
            int m;
            asm("bfe.s32 %0, %1, %2, 1;" : "=r"(m) : "r"(word), "r"(i & 31));
            return m;
        };
#pragma unroll
        for (int p = 0; p < NP; ++p) {
            float2 t = fma2(make_float2(wtf[2 * p], wtf[2 * p + 1]), make_float2(g[2 * p], g[2 * p + 1]), nm);
            if (MASKED) {  // inactive or padding tap -> 0, branch- and predicate-free
                t.x = __int_as_float(__float_as_int(t.x) & mask_of(2 * p));
                t.y = __int_as_float(__float_as_int(t.y) & mask_of(2 * p + 1));
            } else if (!ODD && p == NP - 1) {
                if (sub + G * (2 * p + 1) >= WN) t.y = 0.0f;  // padding tap of the last round
            }
            s3p[p & 1] = fma2(t, t, s3p[p & 1]);
            s1p[p & 1] = fma2(make_float2(dlf[2 * p], dlf[2 * p + 1]), t, s1p[p & 1]);
        }
        float s3s = (s3p[0].x + s3p[0].y) + (s3p[1].x + s3p[1].y);
        float s1s = (s1p[0].x + s1p[0].y) + (s1p[1].x + s1p[1].y);
        if (ODD) {
            float t = fmaf(wtf[TPL - 1], g[TPL - 1], -mR);
            if (MASKED) t = __int_as_float(__float_as_int(t) & mask_of(TPL - 1));
            else if (sub + G * (TPL - 1) >= WN) t = 0.0f;
            s3s = fmaf(t, t, s3s);
            s1s = fmaf(dlf[TPL - 1], t, s1s);
        }
        const float s3 = group_sum_f<G>(s3s, gmask);
        const float s1 = group_sum_f<G>(s1s, gmask);
        // ill-conditioned or non-finite neighbour window: FP64 decides
        if (!(s3 >= (float)WN) || !(s3 < 1e30f)) return SCREEN_FORCE;
        eps = (s3 >= 100.0f * WN) ? eps_pix : SCREEN_EPS_LOOSE;
        // s3 >= WN here: the flush-to-zero rsqrt needs no denormal fix-up (3 issue slots less)
        float rs;
        asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(rs) : "f"(s3));
        return s1 * rs;
    };

    // ---- exact state (FP64) and candidate queue -----------------------------------------------
    const bool depth_up = a.depth_up != 0;
    int n_verified = 0, n_forced = 0, n_screened = 0;  // STATS only
    int qn = 0;
    // lower32: a proven lower bound of the winning ncc64 (max over screened labels of ncc32 - eps,
    // never below the threshold): a label whose upper bound ncc32 + eps is below it cannot win.
    float lower32 = (float)a.ncc_threshold - 1e-6f;
    float max_err = 0.0f;  // STATS only
    int n_viol = 0;        // STATS only: verified labels outside their error bar (must stay 0)

    // Verification of the queued candidates: the lane group of a pixel walks its queue slot by slot.
    auto flush = [&]() {
        const int nmax = __reduce_max_sync(0xffffffffu, qn);
        // the pixel's coordinates are re-derived here (rare path) instead of living in registers
        // across the label loop
        const int pid = min((int)(blockIdx.x * PIX_PER_BLOCK + threadIdx.x / G), a.rows * a.w - 1);
        const int x = pid % a.w, y = a.row0 + pid / a.w;
        const size_t pix = (size_t)y * a.w + x;
        double bestC = px_bestC[tid];
        int bestIdx = px_bestIdx[tid];
        const double meanL_x = px_meanL[tid], totW_x = px_totW[tid], s2_x = px_s2[tid];
#pragma unroll 1
        for (int q = 0; q < nmax; ++q) {
            if (q < qn) {  // uniform within a pixel's lane group
                const int lab = q_lab[q][tid], tap = q_tap[q][tid];
                const int j = (lab >> 16) & 0xff, d = lab & 0xffff;
                const int tx = (int)(short)(tap & 0xffff), ty = (int)(short)((uint32_t)tap >> 16);
                const bool inside = tx >= R && ty >= R && tx < w - R && ty < h - R;
                const double cost = (inside && !all_slow && !has_inactive)
                                        ? verify_cost_mvs<R, G>(a, a.grayR[j], x, y, tx, ty, pid, sub, gmask, meanL_x, totW_x, s2_x)
                                        : slow_cost<R, G, COST>(a, a.grayR[j], x, y, tx, ty, pid, sub, gmask);
                if (STATS) ++n_verified;
                if (STATS && q_c32[q][tid] < 2.0f) {  // |ncc32 - ncc64| relative to its error bar
                    const float e = (lab >> 30) ? SCREEN_EPS_TIGHT : SCREEN_EPS_LOOSE;
                    const float c32 = q_c32[q][tid] - e;
                    const float err = fabsf((float)(cost - (double)c32));
                    max_err = fmaxf(max_err, err);
                    if (err > e) ++n_viol;
                }
                if (cost > a.ncc_threshold) {  // multiviewstereo.cpp:589-602,654-660
                    if (a.curve) {
                        // candidates are (ncc, z) pairs, the winner is the largest pair (:600-602,:654-660)
                        if (bestIdx == SR_INDEX_NONE || cost >= bestC) {
                            const double z = curve_depth(a.raysL, a.raysR[j], (size_t)w * h, pix, (size_t)ty * w + tx, a.camR, a.camT);
                            if (bestIdx == SR_INDEX_NONE || cost > bestC || z > px_bestZ[tid]) {
                                bestC = cost;
                                bestIdx = d;
                                px_bestZ[tid] = z;
                            }
                        }
                    } else {
                        const bool deeper = depth_up ? (d > bestIdx) : (d < bestIdx);
                        if (bestIdx == SR_INDEX_NONE || cost > bestC || (cost == bestC && deeper)) {
                            bestC = cost;
                            bestIdx = d;
                        }
                    }
                }
            }
        }
        qn = 0;
        px_bestC[tid] = bestC;
        px_bestIdx[tid] = bestIdx;
        // the verified maximum is a valid (and tighter) floor for the screen
        if (bestIdx != SR_INDEX_NONE) lower32 = fmaxf(lower32, (float)bestC - 1e-6f);
    };

    // ---- label sweep -------------------------------------------------------------------------
    const int D = a.D;
    const uint64_t pol = l2_evict_first_policy();
    // The tap stream: chunk k (TAP_CHUNK labels of one neighbour) lands in ring buffer k & 1 while
    // chunk k-1 is processed.  (jn, dn) is the next chunk to request.
    int jn = 0, dn = 0, bufn = 0;
    auto issue_next = [&]() {
        if (jn < a.num_nbrs && alive) {
            const int32_t *src = a.taps + ((size_t)jn * (a.tap_planes ? a.tap_planes : D) + dn) * npix + pid;
            const int nl = min(TAP_CHUNK, D - dn);
            for (int l = 0; l < nl; ++l) cp_async4(&tap_ring[bufn][l][tid], src + (size_t)l * npix, pol);
        }
        cp_async_commit();
        bufn ^= 1;
        dn += TAP_CHUNK;
        if (dn >= D) {
            dn = 0;
            ++jn;
        }
    };
    issue_next();

    int buf = 0;
    // The ring column of this thread as a shared-window address that the label loop increments (the
    // compiler otherwise re-derives it from %tid and the loop counters for every label: 7 issue slots).
    // Lanes without a pixel never request taps: their columns hold TAP_NONE from here on.
    if (!alive) {
        for (int l = 0; l < TAP_CHUNK; ++l) tap_ring[0][l][tid] = tap_ring[1][l][tid] = TAP_NONE;
    }
    const unsigned ring_base = (unsigned)__cvta_generic_to_shared(&tap_ring[0][0][tid]);
    constexpr unsigned RING_STEP = SCREEN_BLOCK * 4, RING_BUF = TAP_CHUNK * SCREEN_BLOCK * 4;
#pragma unroll 1
    for (int j = 0; j < a.num_nbrs; ++j) {
      const float *__restrict__ gRf = a.grayRf[j];
#pragma unroll 1
      for (int d0 = 0; d0 < D; d0 += TAP_CHUNK, buf ^= 1) {
        issue_next();
        cp_async_wait<1>();
        const int nl = min(TAP_CHUNK, D - d0);
        unsigned ra = ring_base + buf * RING_BUF;
#pragma unroll 1
        for (int l = 0; l < nl; ++l, ra += RING_STEP) {
            int32_t tap;
            asm volatile("ld.shared.b32 %0, [%1];" : "=r"(tap) : "r"(ra));
            if (tap != TAP_NONE) {
                // (Consecutive labels often share a tap; re-using the previous value only pays when all
                // 32 lanes repeat at once, which is rare, and costs three live registers: not done.
                // The queue below still keeps one entry per distinct tap.)
                float c32 = SCREEN_FORCE, eps = 0.0f;
                {
                    const int tx = (int)(short)(tap & 0xffff), ty = (int)(short)((uint32_t)tap >> 16);
                    // R <= t < dim - R as one unsigned comparison per coordinate
                    if (!all_slow && (unsigned)(tx - R) < (unsigned)a.win_w && (unsigned)(ty - R) < (unsigned)a.win_h) {
                        const float *base = gRf + ((size_t)ty * fp + tx);
                        c32 = has_inactive ? screen_one(base, eps, std::true_type{}) : screen_one(base, eps, std::false_type{});
                    }
                    if (STATS) {
                        if (c32 == SCREEN_FORCE) ++n_forced;
                        else ++n_screened;
                    }
                }
                const float ub = c32 + eps;  // FORCE stays FORCE
                if (ub >= lower32) {         // candidate
                    const int d = d0 + l;
                    const int lab = ((eps == SCREEN_EPS_TIGHT) ? (1 << 30) : 0) | (j << 16) | d;
                    if (qn > 0 && q_tap[qn - 1][tid] == tap && ((q_lab[qn - 1][tid] >> 16) & 0xff) == j) {
                        // equal cost by construction: the tie-break picks the deeper label (in curve
                        // mode the same pixel is the same (ncc, z) pair: nothing to add)
                        if (depth_up && !a.curve) q_lab[qn - 1][tid] = lab;
                    } else {
                        const float lb = c32 - eps;
                        if (c32 != SCREEN_FORCE && lb > lower32) {
                            // the bound rises: queued labels whose upper bound is below it cannot win
                            lower32 = lb;
                            int kept = 0;
                            for (int q = 0; q < qn; ++q) {
                                const float uq = q_c32[q][tid];
                                if (uq >= lower32) {
                                    if (kept != q) {
                                        q_c32[kept][tid] = uq;
                                        q_lab[kept][tid] = q_lab[q][tid];
                                        q_tap[kept][tid] = q_tap[q][tid];
                                    }
                                    ++kept;
                                }
                            }
                            qn = kept;
                        }
                        q_lab[qn][tid] = lab;
                        q_tap[qn][tid] = tap;
                        q_c32[qn][tid] = ub;
                        ++qn;
                    }
                }
            }
            if (__any_sync(0xffffffffu, qn == SCREEN_QCAP)) flush();
        }
      }
    }
    cp_async_wait<0>();
    flush();

    if (STATS && a.stats && alive && sub == 0) {
        atomicAdd(a.stats + 0, 1ull);
        atomicAdd(a.stats + 1, (unsigned long long)n_screened);
        atomicAdd(a.stats + 2, (unsigned long long)n_forced);
        atomicAdd(a.stats + 3, (unsigned long long)n_verified);
        if (all_slow) atomicAdd(a.stats + 4, 1ull);
        atomicAdd(a.stats + 6, (unsigned long long)n_viol);
        atomicMax(a.stats + 5, (unsigned long long)__float_as_uint(max_err));  // positive floats order as integers
    }
    if (alive && sub == 0) {
        const int bestIdx = px_bestIdx[tid];
        a.out_index[pix] = bestIdx;
        a.out_depth[pix] = (bestIdx >= 0) ? (a.curve ? px_bestZ[tid] : a.depth_table[bestIdx]) : -1.0;
        a.out_best[pix] = px_bestC[tid];
    }
}

}  // namespace sr
