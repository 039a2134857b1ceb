// sr_screen2.cuh — the thread-per-pixel (r <= 2) form of the FP32 screen / FP64 verify selection of
// sr_match_screen.cuh, reorganised so that the label loop is nothing but loads and window arithmetic.
//
//   * ONE-PASS window sums.  With p_i = w_i g_i (support weight x neighbour gray; w_i = 0 for the taps the
//     reference skips on the reference side, stereo/multiviewstereo.cpp:137-141), n_a active taps and
//     totW = sum w_i, the reference's two passes (:143-185) are algebraically
//         meanR = S1 / totW,                      S1 = sum p_i
//         s3 = sum_active (p_i - meanR)^2 = Q - meanR^2 (2 totW - n_a),      Q = sum p_i^2
//         s1 = sum dl_i (p_i - meanR)      = X - meanR * SDL,                 X = sum (dl_i w_i) g_i
//     so S1, Q and X are three independent accumulations over the taps: every loaded value is consumed
//     as it arrives (no second pass that has to wait for the mean), the window needs no registers of
//     its own beyond the loads in flight, and pixels with inactive taps need no special path at all.
//     What the mean-first form bought in conditioning is paid back by an error bar that follows the
//     cancellation kappa = Q / s3 of each label (see eps below) instead of two fixed classes.
//   * Candidate handling is deferred to the end of a 16-label chunk: the loop stores the label's upper
//     bound to a shared column, raises the lower bound and sets a bit in a per-lane mask; one warp vote
//     per CHUNK decides whether anybody has to look at the queue at all.  Queue overflow is resolved
//     there too (flush, then continue with the lane's remaining bits); entries a risen bound has made
//     hopeless are evicted when a queue fills and before a flush.
//   * The warps of a block own the rows of a 32-pixel-wide tile of the reference image.
//
// The rule that makes this exact is unchanged (sr_match_screen.cuh): a label is dropped only if its
// upper bound ncc32 + eps is below lower32, a proven lower bound of the winning FP64 cost; every label
// that survives is evaluated by the reference's own two-pass filter in FP64 and the reference's
// selection rule (stereo/multiviewstereo.cpp:589-602,654-660) picks the winner.
//
// Error bar of the one-pass value (u = 2^-24; all inputs rounded once from FP64: <= u each):
//   S1, Q, X are sums of <= 13 terms in two chains + a 3-add tree: <= 9 roundings per term.
//     |dS1| <= 11u S1 (all terms >= 0),   |dQ| <= 15u Q,   |dX| <= 11u sum|dl_i| p_i <= 11u sqrt(Q)  (|dl| = 1)
//   meanR: 13u relative;  meanR^2 (2 totW - n_a) = Q - s3, at most Q in magnitude when 2 totW > n_a
//     (otherwise nothing cancels):  |ds3| <= 46u Q
//   |meanR SDL| <= sqrt(n_a Q) |SDL| / totW:  |ds1| <= u sqrt(Q) (12 + 15 sigma),  sigma = |SDL| sqrt(n_a) / totW
//   ncc = s1 / sqrt(s3):  |dncc| <= |ds1| / sqrt(s3) + |ds3| / (2 s3) <= u [(12 + 15 sigma) sqrt(kappa) + 23 kappa]
//   with sqrt(kappa) <= (1 + kappa) / 2, a safety factor 1.5 and 3e-7 for rsqrt.approx and the last product:
//         eps = e0 + e1 * kappa,   e0 = 1.5u (6 + 7.5 sigma) + 3e-7,   e1 = 1.5u (29 + 7.5 sigma)
//   (per-pixel constants).  The first-order step needs |ds3| << s3: labels with eps > SCREEN_EPS_MAX, and
//   windows with s3 < WN (RMS deviation below one gray level), are FORCEd to FP64.
//   SR_MATCH_STATS=1 checks every verified label against its bar (outside_error_bar must stay 0).
#pragma once
#include "sr_match_screen.cuh"

namespace sr {

constexpr float SCREEN_EPS_MAX = 5e-3f;  // a wider error bar means FP64 decides
constexpr float SCREEN_SKIP = -2.0f;     // "no value": below every possible lower bound

// Shared memory of one screening warp.
template <bool STATS>
struct alignas(16) Screen2Smem {
    int32_t tap_ring[2][TAP_CHUNK][32];
    float ub_ring[TAP_CHUNK][32];    // ncc32 + eps of the chunk's labels (SCREEN_FORCE: FP64 decides)
    int32_t q_lab[SCREEN_QCAP][32];  // (neighbour << 16) | label
    int32_t q_tap[SCREEN_QCAP][32];
    float q_ub[SCREEN_QCAP][32];     // upper bound; after verification: high word of the FP64 cost
    double px_meanL[32], px_totW[32], px_s2[32], px_bestC[32], px_bestZ[32];
    int px_bestIdx[32];
    unsigned short v_ent[SCREEN_QCAP * 32];
    unsigned char px_flags[32];  // bit 0: all_slow, bit 1: has_inactive
    // SR_MATCH_STATS only: the labels' error bars, and what the verifications found
    float eps_ring[STATS ? TAP_CHUNK : 1][32], q_eps[STATS ? SCREEN_QCAP : 1][32], st_maxerr[STATS ? 32 : 1];
    int st_verified[STATS ? 32 : 1], st_viol[STATS ? 32 : 1];
};

// Register slot i of the window arrays holds window tap k = screen2_slot_tap<R>(i) (row-major k).  The
// 5x5 window starts with the centre 3x3 block and the tap left of it, then the rest in row-major order.
// The slot order is the order in which the FP32 window sums accumulate, so it fixes the screened values to
// the last bit (and the error bars were checked with it): keep it.
template <int R>
__host__ __device__ constexpr int screen2_slot_tap(int i) {
    if (R != 2) return i;
    constexpr int centre[10] = {6, 7, 8, 11, 12, 13, 16, 17, 18, 10};
    constexpr int rest[15] = {0, 1, 2, 3, 4, 5, 9, 14, 15, 19, 20, 21, 22, 23, 24};
    return i < 10 ? centre[i] : rest[i - 10];
}

__device__ __forceinline__ int32_t lds_b32(unsigned addr) {
    int32_t v;
    asm volatile("ld.shared.b32 %0, [%1];" : "=r"(v) : "r"(addr));
    return v;
}
__device__ __forceinline__ void sts_f32(unsigned addr, float v) { asm volatile("st.shared.f32 [%0], %1;" ::"r"(addr), "f"(v)); }

// ---- the rare paths: free functions with by-value arguments, so that the screening warp's register
// arrays (weights, dl) never have to be addressable ------------------------------------------------
struct Screen2Cold {
    int qn;
    float lower32;
};

// pixel of lane `o` (clamped into the band: out-of-band lanes shadow the last pixel, no writes)
__device__ __forceinline__ int screen2_pid(const MatchArgs &a, int first_pid, int o) { return min(first_pid + o, a.rows * a.w - 1); }

// exact evaluation of one queued candidate of lane `o` (FP64, the reference's filter)
template <int R, bool STATS>
__device__ __forceinline__ double screen2_exact_cost(const MatchArgs &a, const Screen2Smem<STATS> &sm, int first_pid, int o, int lab, int tap) {
    const int j = (lab >> 16) & 0xff;
    const int tx = tap & 0xffff, ty = (int)((uint32_t)tap >> 16);
    const int opid = screen2_pid(a, first_pid, o);
    const int ox = opid % a.w, oy = a.row0 + opid / a.w;
    const bool inside = (unsigned)(tx - R) < (unsigned)a.win_w && (unsigned)(ty - R) < (unsigned)a.win_h;
    return (inside && sm.px_flags[o] == 0)
               ? verify_cost_mvs<R, 1>(a, a.grayR[j], ox, oy, tx, ty, opid, 0, 0xffffffffu, sm.px_meanL[o], sm.px_totW[o], sm.px_s2[o])
               : slow_cost<R, 1, SR_COST_NCC_MVS>(a, a.grayR[j], ox, oy, tx, ty, opid, 0, 0xffffffffu);
}

template <bool STATS>
__device__ __forceinline__ void screen2_stats_verified(Screen2Smem<STATS> &sm, int lane, int o, int q, double cost) {
    if (!STATS) return;
    ++sm.st_verified[lane];
    if (sm.q_ub[q][o] < 2.0f) {  // |ncc32 - ncc64| relative to its error bar
        const float eb = sm.q_eps[q][o];
        const float c32 = sm.q_ub[q][o] - eb;
        const float err = fabsf((float)(cost - (double)c32));
        sm.st_maxerr[lane] = fmaxf(sm.st_maxerr[lane], err);
        if (err > eb) ++sm.st_viol[lane];
    }
}

// Queued labels whose upper bound has fallen below the (risen) lower bound cannot win.
template <bool STATS>
__device__ __forceinline__ int screen2_evict(Screen2Smem<STATS> &sm, int lane, int qn, float lower32) {
    int kept = 0;
    for (int q = 0; q < qn; ++q) {
        const float uq = sm.q_ub[q][lane];
        if (uq >= lower32) {
            if (kept != q) {
                sm.q_ub[kept][lane] = uq;
                sm.q_lab[kept][lane] = sm.q_lab[q][lane];
                sm.q_tap[kept][lane] = sm.q_tap[q][lane];
                if (STATS) sm.q_eps[kept][lane] = sm.q_eps[q][lane];
            }
            ++kept;
        }
    }
    return kept;
}

// Verification of the warp's queued candidates; returns the lane's new lower bound (its queue is empty
// afterwards).  Label mode: the entries are compacted into one list and dealt out one per lane, whoever
// owns them; every lane then applies the selection rule (multiviewstereo.cpp:589-602,654-660) to its
// own entries in order.  Curve mode: candidates are (ncc, z) pairs, z = closest approach of the two
// viewing rays (:583-588); each lane walks its own queue.
template <int R, bool STATS>
__device__ __noinline__ float screen2_flush(const MatchArgs &a, Screen2Smem<STATS> &sm, int lane, int first_pid, int qn, float lower32) {
    constexpr unsigned FULL = 0xffffffffu;
    qn = screen2_evict<STATS>(sm, lane, qn, lower32);
    double bestC = sm.px_bestC[lane];
    int bestIdx = sm.px_bestIdx[lane];
    if (a.curve) {
        const int w = a.w, h = a.h;
        const int pid = screen2_pid(a, first_pid, lane);
        const size_t pix = (size_t)(a.row0 + pid / w) * w + pid % w;
#pragma unroll 1
        for (int q = 0; q < qn; ++q) {
            const int lab = sm.q_lab[q][lane], tap = sm.q_tap[q][lane];
            const int j = (lab >> 16) & 0xff, d = lab & 0xffff;
            const double cost = screen2_exact_cost<R, STATS>(a, sm, first_pid, lane, lab, tap);
            screen2_stats_verified<STATS>(sm, lane, lane, q, cost);
            if (cost > a.ncc_threshold && (bestIdx == SR_INDEX_NONE || cost >= bestC)) {
                const int tx = tap & 0xffff, ty = (int)((uint32_t)tap >> 16);
                const double z = curve_depth(a.raysL, a.raysR[j], (size_t)w * h, pix, (size_t)ty * w + tx, a.camR, a.camT);
                if (bestIdx == SR_INDEX_NONE || cost > bestC || z > sm.px_bestZ[lane]) {
                    bestC = cost;
                    bestIdx = d;
                    sm.px_bestZ[lane] = z;
                }
            }
        }
    } else {
        unsigned short *ent = sm.v_ent;
        int incl = qn;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int v = __shfl_up_sync(FULL, incl, o);
            if (lane >= o) incl += v;
        }
        const int total = __shfl_sync(FULL, incl, 31);
        const int off = incl - qn;
        for (int q = 0; q < qn; ++q) ent[off + q] = (unsigned short)((lane << 8) | q);
        __syncwarp();
#pragma unroll 1
        for (int e = lane; e < total; e += 32) {
            const int o = ent[e] >> 8, q = ent[e] & 0xff;
            const int lab = sm.q_lab[q][o], tap = sm.q_tap[q][o];
            const double cost = screen2_exact_cost<R, STATS>(a, sm, first_pid, o, lab, tap);
            screen2_stats_verified<STATS>(sm, lane, o, q, cost);
            sm.q_tap[q][o] = __double2loint(cost);
            sm.q_ub[q][o] = __int_as_float(__double2hiint(cost));
        }
        __syncwarp();
        const bool depth_up = a.depth_up != 0;
        for (int q = 0; q < qn; ++q) {
            const double cost = __hiloint2double(__float_as_int(sm.q_ub[q][lane]), sm.q_tap[q][lane]);
            const int d = sm.q_lab[q][lane] & 0xffff;
            if (cost > a.ncc_threshold) {
                const bool deeper = depth_up ? (d > bestIdx) : (d < bestIdx);
                if (bestIdx == SR_INDEX_NONE || cost > bestC || (cost == bestC && deeper)) {
                    bestC = cost;
                    bestIdx = d;
                }
            }
        }
    }
    sm.px_bestC[lane] = bestC;
    sm.px_bestIdx[lane] = bestIdx;
    // the verified maximum is a valid (and tighter) floor for the screen
    if (bestIdx != SR_INDEX_NONE) lower32 = fmaxf(lower32, (float)bestC - 1e-6f);
    __syncwarp();  // the list and the queues are rewritten by the caller
    return lower32;
}

// End of a chunk: the lanes' marked labels (bits of `pend`, upper bounds in sm.ub_ring) go through the queue; a queue that is full even after eviction makes the warp flush.
template <int R, bool STATS>
__device__ __noinline__ Screen2Cold screen2_process_pending(const MatchArgs &a, Screen2Smem<STATS> &sm, int lane, int first_pid, int j, int d0,
                                                            int buf, int qn, unsigned pend, float lower32) {
    constexpr unsigned FULL = 0xffffffffu;
    const bool depth_up = a.depth_up != 0;
#pragma unroll 1
    for (;;) {
#pragma unroll 1
        while (pend) {
            if (qn == SCREEN_QCAP) {
                qn = screen2_evict<STATS>(sm, lane, qn, lower32);
                if (qn == SCREEN_QCAP) break;  // still full: the warp flushes
            }
            const int l = __ffs(pend) - 1;
            pend &= pend - 1;
            const float ub = sm.ub_ring[l][lane];  // ncc32 + eps, or SCREEN_FORCE
            if (!(ub >= lower32)) continue;        // the bound rose after this label was marked
            const int32_t tap = sm.tap_ring[buf][l][lane];
            const int lab = (j << 16) | (d0 + l);
            if (qn > 0 && sm.q_tap[qn - 1][lane] == tap && ((sm.q_lab[qn - 1][lane] >> 16) & 0xff) == j) {
                // equal cost by construction: the tie-break picks the deeper label (curve mode: the same
                // pixel is the same (ncc, z) pair, nothing to add)
                if (depth_up && !a.curve) sm.q_lab[qn - 1][lane] = lab;
            } else {
                sm.q_lab[qn][lane] = lab;
                sm.q_tap[qn][lane] = tap;
                sm.q_ub[qn][lane] = ub;
                if (STATS) sm.q_eps[qn][lane] = sm.eps_ring[l][lane];
                ++qn;
            }
        }
        if (!__any_sync(FULL, pend != 0u)) break;
        lower32 = screen2_flush<R, STATS>(a, sm, lane, first_pid, qn, lower32);
        qn = 0;
    }
    Screen2Cold r;
    r.qn = qn;
    r.lower32 = lower32;
    return r;
}

// One screening warp: 32 consecutive pixels of the band, one per lane.  PITCH: compile-time row pitch of
// the FP32 gray planes (0: run-time a.pitch_f).
template <int R, bool STATS, int PITCH>
struct Screener {
    static constexpr int WS = 2 * R + 1, WN = WS * WS;
    static constexpr unsigned FULL = 0xffffffffu;

    const MatchArgs &a;
    Screen2Smem<STATS> &sm;
    const int lane;
    // wtf: support weights w_i; c1f: dl_i w_i / sqrt(s2)
    float wtf[WN], c1f[WN];
    // k0 = 2 totW - n_a, k1 = SDL / sqrt(s2), error bar e0 + e1 * kappa
    float inv_totWf, k0, k1, e0, e1, lower32;
    int qn, my_win_w, first_pid;
    unsigned pend;
    bool alive;
    int n_forced, n_screened;  // STATS only

    __device__ __forceinline__ Screener(const MatchArgs &a_, Screen2Smem<STATS> &sm_, int lane_) : a(a_), sm(sm_), lane(lane_) {}

    // ---- per-pixel invariants in FP64, as sr_match_screen.cuh ---------------------------------
    // The warp's pixels are first_pid_ .. first_pid_ + nvalid - 1 of the band (lanes >= nvalid have none).
    __device__ __forceinline__ void init(int first_pid_, int nvalid) {
        first_pid = first_pid_;
        const int w = a.w, h = a.h;
        const size_t npix = (size_t)a.rows * w;
        const bool in_band = lane < nvalid;
        const int pid = screen2_pid(a, first_pid, lane);
        const int x = pid % w, y = a.row0 + pid / w;
        const size_t pix = (size_t)y * w + x;
        alive = in_band && a.maskL[pix] == 255;
        if (in_band && !alive) {  // multiviewstereo.cpp:559,565: masked-out pixels stay INF
            a.out_index[pix] = SR_INDEX_MASKED;
            a.out_depth[pix] = dinf();
            a.out_best[pix] = qnan();
        }
        double wt[WN], gl[WN];
        double totW = 0.0, SL = 0.0;
        int ninact = 0;
        // (the reference's summation order, row-major: these sums also feed the exact verification)
#pragma unroll
        for (int k = 0; k < WN; ++k) {
            const int row = k / WS - R, col = k % WS - R;
            const int xl = x + col, yl = y + row;
            double g = qnan(), wv = 0.0;
            if (alive && xl >= 0 && yl >= 0 && xl < w && yl < h) {
                g = a.grayL[(size_t)yl * w + xl];
                wv = a.W[(size_t)k * npix + pid];
            }
            const bool active = (g == g) && (wv > 1e-10);
            wt[k] = active ? wv : 0.0;
            gl[k] = active ? g : 0.0;
            if (active) {
                totW += wv;
                SL += wv * g;
            } else {
                ++ninact;
            }
        }
        const double meanL = SL / totW;
        double s2 = 0.0, SDL = 0.0;
#pragma unroll
        for (int k = 0; k < WN; ++k) {
            const double dl = (wt[k] > 0.0) ? wt[k] * gl[k] - meanL : 0.0;
            s2 += dl * dl;
            SDL += dl;
            gl[k] = dl;
        }
        const bool all_slow = !(totW >= 1e-10) || !(s2 >= (double)WN) || !(s2 < 1e30);
        const double rs2 = all_slow ? 0.0 : 1.0 / sqrt(s2);  // folded into c1f: ncc32 = s1 * rsqrt(s3)
#pragma unroll
        for (int i = 0; i < WN; ++i) {
            const int k = screen2_slot_tap<R>(i);
            wtf[i] = (float)wt[k];
            c1f[i] = (float)((gl[k] * rs2) * wt[k]);
        }
        const bool has_inactive = ninact != 0;
        inv_totWf = (float)(1.0 / totW);
        {
            const double na = (double)(WN - ninact);
            const double sigma = fabs(SDL * rs2) * sqrt(na) / totW;
            const double u = 5.9604644775390625e-8;  // 2^-24
            k0 = (float)(2.0 * totW - na);
            k1 = (float)(SDL * rs2);
            e0 = (float)(1.5 * u * (6.0 + 7.5 * sigma) + 3e-7);
            e1 = (float)(1.5 * u * (29.0 + 7.5 * sigma));
            if (!(e1 < 1.0f)) e1 = 1.0f;  // (all_slow pixels: unused)
        }
        // lanes that screen nothing (no pixel, or an ill-conditioned reference window that only the exact
        // filter may judge) see an empty interior: every evaluable tap of theirs is FORCEd
        my_win_w = (alive && !all_slow) ? a.win_w : 0;
        sm.px_meanL[lane] = meanL;
        sm.px_totW[lane] = totW;
        sm.px_s2[lane] = s2;
        sm.px_bestC[lane] = 0.0;
        sm.px_bestIdx[lane] = SR_INDEX_NONE;
        sm.px_bestZ[lane] = -1.0;
        sm.px_flags[lane] = (unsigned char)((all_slow ? 1 : 0) | (has_inactive ? 2 : 0));
        if (STATS) {
            sm.st_verified[lane] = sm.st_viol[lane] = 0;
            sm.st_maxerr[lane] = 0.0f;
        }
        // keep the FP32 constants as values of their own (not re-derived from FP64 inside the label loop)
        asm volatile("" : "+f"(inv_totWf), "+f"(k0), "+f"(k1), "+f"(e0), "+f"(e1));
        qn = 0;
        pend = 0u;
        lower32 = (float)a.ncc_threshold - 1e-6f;
        n_forced = n_screened = 0;
        if (STATS && alive && all_slow && a.stats) atomicAdd(a.stats + 4, 1ull);
        __syncwarp();
    }

    // ---- FP32 screen -----------------------------------------------------------------------------------
    // The (2R+1)^2 taps around element `idx` of the neighbour's FP32 plane.
    __device__ __forceinline__ void load_window(const float *__restrict__ gplane, int idx, float (&g)[WN]) const {
        const int fp = PITCH ? PITCH : a.pitch_f;
        const float *__restrict__ base = gplane + idx;
#pragma unroll
        for (int i = 0; i < WN; ++i) {
            const int k = screen2_slot_tap<R>(i);
            g[i] = base[(k / WS - R) * fp + (k % WS - R)];
        }
    }

    // One window: ub = ncc32 + eps (SCREEN_FORCE when FP64 has to decide), lb = ncc32 - eps (SCREEN_SKIP
    // then), eps (statistics).  The taps go in pairs through one FFMA2 accumulator pair per sum; the three
    // sums interleave, which keeps dependent FFMA2s three issue slots apart.
    __device__ __forceinline__ void eval_window(const float (&g)[WN], float &ub, float &lb, float &eps_out) const {
        constexpr int NP = WN / 2;  // WN is odd: NP pairs + one scalar tap
        const float2 zero = make_float2(0.0f, 0.0f);
        float2 S1p = zero, Qp = zero, Xp = zero;
#pragma unroll
        for (int p = 0; p < NP; ++p) {
            const float2 wv = make_float2(wtf[2 * p], wtf[2 * p + 1]), gv = make_float2(g[2 * p], g[2 * p + 1]);
            S1p = fma2(wv, gv, S1p);
            const float2 pv = fma2(wv, gv, zero);
            Qp = fma2(pv, pv, Qp);
            Xp = fma2(make_float2(c1f[2 * p], c1f[2 * p + 1]), gv, Xp);
        }
        float S1 = S1p.x + S1p.y, Q = Qp.x + Qp.y, X = Xp.x + Xp.y;
        {
            const float pl = wtf[WN - 1] * g[WN - 1];
            S1 += pl;
            Q = fmaf(pl, pl, Q);
            X = fmaf(c1f[WN - 1], g[WN - 1], X);
        }
        const float mR = S1 * inv_totWf;
        const float s3 = fmaf(-k0, mR * mR, Q);
        const float s1 = fmaf(-mR, k1, X);
        float rs;
        asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(rs) : "f"(s3));
        const float c32 = s1 * rs;
        const float eps = fmaf(Q * (rs * rs), e1, e0);  // e0 + e1 * kappa
        // ill-conditioned or non-finite neighbour window, or a bar too wide to be first order: FP64 decides
        const bool ok = (s3 >= (float)WN) && (eps <= SCREEN_EPS_MAX);
        eps_out = eps;
        lb = ok ? c32 - eps : SCREEN_SKIP;
        ub = ok ? c32 + eps : SCREEN_FORCE;
    }

    // Two windows at once, vectorised ACROSS the two labels: every FFMA2 carries tap i of both windows in its
    // two halves and the tap's weight as a scalar (broadcast) operand.  The sums of a label live in one half
    // of an accumulator, so there is no horizontal reduction, the 25th tap is not a scalar straggler, and the
    // whole tail (mean, s3, s1, kappa, error bar, bounds) is packed as well: ~58 FMA-pipe instructions per
    // label instead of ~77 (the loop's time is additive in them, DESIGN.md section 5).
    __device__ __forceinline__ void eval_window2(const float (&gA)[WN], const float (&gB)[WN], float (&ub)[2], float (&lb)[2],
                                                 float (&eps_out)[2]) const {
        const float2 zero = make_float2(0.0f, 0.0f);
        float2 S1 = zero, Q = zero, X = zero;
#pragma unroll
        for (int i = 0; i < WN; ++i) {
            const float2 gv = make_float2(gA[i], gB[i]);
            const float2 wv = make_float2(wtf[i], wtf[i]);
            S1 = fma2(gv, wv, S1);
            const float2 pv = fma2(gv, wv, zero);
            Q = fma2(pv, pv, Q);
            X = fma2(gv, make_float2(c1f[i], c1f[i]), X);
        }
        const float2 mR = fma2(S1, make_float2(inv_totWf, inv_totWf), zero);
        const float2 mR2 = fma2(mR, mR, zero);
        const float2 s3 = fma2(mR2, make_float2(-k0, -k0), Q);
        const float2 s1 = fma2(mR, make_float2(-k1, -k1), X);
        float2 rs;
        asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(rs.x) : "f"(s3.x));
        asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(rs.y) : "f"(s3.y));
        const float2 c32 = fma2(s1, rs, zero);
        const float2 kappa = fma2(Q, fma2(rs, rs, zero), zero);
        const float2 eps = fma2(kappa, make_float2(e1, e1), make_float2(e0, e0));  // e0 + e1 * kappa
        const float2 up = fma2(eps, make_float2(1.0f, 1.0f), c32), lo = fma2(eps, make_float2(-1.0f, -1.0f), c32);
        const bool okx = (s3.x >= (float)WN) && (eps.x <= SCREEN_EPS_MAX), oky = (s3.y >= (float)WN) && (eps.y <= SCREEN_EPS_MAX);
        eps_out[0] = eps.x;
        eps_out[1] = eps.y;
        lb[0] = okx ? lo.x : SCREEN_SKIP;
        lb[1] = oky ? lo.y : SCREEN_SKIP;
        ub[0] = okx ? up.x : SCREEN_FORCE;
        ub[1] = oky ? up.y : SCREEN_FORCE;
    }

    // NL = 1 or 2 windows at once (two: eval_window2).
    template <int NL>
    __device__ __forceinline__ void screen_n(const float *__restrict__ gplane, const int (&idx)[NL], float (&ub)[NL], float (&lb)[NL],
                                             float (&eps_out)[NL]) const {
        float g[NL][WN];
#pragma unroll
        for (int n = 0; n < NL; ++n) load_window(gplane, idx[n], g[n]);
        if (NL == 2) {
            float ub2[2], lb2[2], ep2[2];
            eval_window2(g[0], g[NL - 1], ub2, lb2, ep2);
#pragma unroll
            for (int n = 0; n < NL; ++n) {
                ub[n] = ub2[n];
                lb[n] = lb2[n];
                eps_out[n] = ep2[n];
            }
        } else {
#pragma unroll
            for (int n = 0; n < NL; ++n) eval_window(g[n], ub[n], lb[n], eps_out[n]);
        }
    }

    // A ring entry -> is its window interior to the neighbour image (then idx = its element index, else a
    // safe interior element).  MVS taps lie inside the image; TAP_NONE decodes to ty = 32768 (never interior).
    __device__ __forceinline__ bool decode_tap(int32_t tap, int &idx) const {
        const int fp = PITCH ? PITCH : a.pitch_f;
        const int tx = tap & 0xffff, ty = (int)((uint32_t)tap >> 16);
        const bool interior = (unsigned)(tx - R) < (unsigned)my_win_w && (unsigned)(ty - R) < (unsigned)a.win_h;
        idx = interior ? ty * fp + tx : R * fp + R;
        return interior;
    }
    // What a label's screen result does to the lane's state (ca: its slot of the upper-bound ring).
    __device__ __forceinline__ void commit_label(bool interior, int32_t tap, float ub, float lb, float eps, unsigned ca, unsigned bit, int l) {
        if (interior) {
            sts_f32(ca, ub);
            lower32 = fmaxf(lower32, lb);
            pend |= (ub >= lower32) ? bit : 0u;
            if (STATS) {
                sm.eps_ring[l][lane] = eps;
                if (ub == SCREEN_FORCE) ++n_forced;
                else ++n_screened;
            }
        } else if (tap != TAP_NONE && alive) {  // window on the neighbour's border / FP64-only pixel
            sts_f32(ca, SCREEN_FORCE);
            pend |= bit;
            if (STATS) ++n_forced;
        }
    }

    // NL consecutive labels of a chunk: ring entries at shared addresses ra, ra + 128, ...; `bit` = mask bit
    // of the first.  A lane with at least one interior label evaluates all NL (the others at a safe address,
    // result discarded).
    template <int NL>
    __device__ __forceinline__ void labels(const float *__restrict__ gplane, unsigned ra, unsigned ca, unsigned bit, int l) {
        int32_t tap[NL];
        int idx[NL];
        bool interior[NL], any = false;
#pragma unroll
        for (int n = 0; n < NL; ++n) {
            tap[n] = lds_b32(ra + 128u * n);
            interior[n] = decode_tap(tap[n], idx[n]);
            any = any || interior[n];
        }
        float ub[NL], lb[NL], eps[NL];
#pragma unroll
        for (int n = 0; n < NL; ++n) ub[n] = lb[n] = eps[n] = 0.0f;
        if (any) screen_n<NL>(gplane, idx, ub, lb, eps);
#pragma unroll
        for (int n = 0; n < NL; ++n) commit_label(interior[n], tap[n], ub[n], lb[n], eps[n], ca + 128u * n, bit << n, l + n);
    }

    // ---- one chunk of labels of neighbour j: taps in sm.tap_ring[buf][0..nl) -----------------------
    __device__ __forceinline__ void chunk(int j, int d0, int nl, int buf, const float *__restrict__ gplane) {
        unsigned ra = (unsigned)__cvta_generic_to_shared(&sm.tap_ring[buf][0][lane]);
        unsigned ca = (unsigned)__cvta_generic_to_shared(&sm.ub_ring[0][lane]);
        unsigned bit = 1u;
        int l = 0;
        // two labels per iteration (independent chains, eval_window2), then an odd last label on its own
#pragma unroll 1
        for (; l + 2 <= nl; l += 2, ra += 256u, ca += 256u, bit <<= 2) labels<2>(gplane, ra, ca, bit, l);
#pragma unroll 1
        for (; l < nl; ++l, ra += 128u, ca += 128u, bit <<= 1) labels<1>(gplane, ra, ca, bit, l);
        if (__any_sync(FULL, pend != 0u)) {
            const Screen2Cold r = screen2_process_pending<R, STATS>(a, sm, lane, first_pid, j, d0, buf, qn, pend, lower32);
            qn = r.qn;
            lower32 = r.lower32;
            pend = 0u;
        }
    }

    __device__ __forceinline__ void finish() {
        lower32 = screen2_flush<R, STATS>(a, sm, lane, first_pid, qn, lower32);
        qn = 0;
        if (STATS && a.stats && alive) {
            atomicAdd(a.stats + 0, 1ull);
            atomicAdd(a.stats + 1, (unsigned long long)n_screened);
            atomicAdd(a.stats + 2, (unsigned long long)n_forced);
        }
        if (STATS && a.stats) {  // verifications are counted by the lane that ran them
            atomicAdd(a.stats + 3, (unsigned long long)sm.st_verified[lane]);
            atomicAdd(a.stats + 6, (unsigned long long)sm.st_viol[lane]);
            atomicMax(a.stats + 5, (unsigned long long)__float_as_uint(sm.st_maxerr[lane]));  // positive floats order as integers
        }
        if (alive) {
            const int pid = screen2_pid(a, first_pid, lane);
            const size_t pix = (size_t)(a.row0 + pid / a.w) * a.w + pid % a.w;
            const int bestIdx = sm.px_bestIdx[lane];
            a.out_index[pix] = bestIdx;
            a.out_depth[pix] = (bestIdx >= 0) ? (a.curve ? sm.px_bestZ[lane] : a.depth_table[bestIdx]) : -1.0;
            a.out_best[pix] = sm.px_bestC[lane];
        }
    }
};

constexpr int SCREEN2_TILE_ROWS = 4;  // warps per block: a block owns a 32 x TILE_ROWS tile of reference pixels (measured: 4 < 8 < 1)
constexpr int SCREEN2_MINBLOCKS = 4;  // resident blocks per SM the register allocation must allow (x TILE_ROWS = 16 warps)

// Stand-alone form: the tap volume comes from HBM (label mode: build kernels; curve mode: the curve
// rasteriser) through the two-stage cp.async ring.  The warps of a block are independent (nothing is
// block-wide); they own the rows of a 32-pixel-wide tile so that their neighbour-image footprints overlap
// in L1 (adjacent reference rows project to adjacent neighbour rows).  grid = (ceil(w/32), ceil(rows/TR)).
template <int R, bool STATS, int PITCH>
__global__ void __launch_bounds__(32 * SCREEN2_TILE_ROWS, SCREEN2_MINBLOCKS) match_mvs_screen2_kernel(const __grid_constant__ MatchArgs a) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    Screen2Smem<STATS> &sm = reinterpret_cast<Screen2Smem<STATS> *>(smem_raw)[warp];
    const int x0 = blockIdx.x * 32, row = blockIdx.y * SCREEN2_TILE_ROWS + warp;  // row within the band
    const int nvalid = (row < a.rows) ? min(32, a.w - x0) : 0;
    const int first_pid = min(row, a.rows - 1) * a.w + x0;
    Screener<R, STATS, PITCH> S(a, sm, lane);
    S.init(first_pid, nvalid);
    const int D = a.D;
    const size_t npix = (size_t)a.rows * a.w;
    const int pid = screen2_pid(a, first_pid, lane);
    const uint64_t pol = l2_evict_first_policy();
    // lanes without a pixel never request taps: their columns hold TAP_NONE from here on
    if (!S.alive) {
        for (int l = 0; l < TAP_CHUNK; ++l) sm.tap_ring[0][l][lane] = sm.tap_ring[1][l][lane] = TAP_NONE;
    }
    int jn = 0, dn = 0, bufn = 0;
    auto issue_next = [&]() {
        if (jn < a.num_nbrs && S.alive) {
            const int32_t *src = a.taps + ((size_t)jn * (a.tap_planes ? a.tap_planes : D) + dn) * npix + pid;
            const int nl = min(TAP_CHUNK, D - dn);
            const unsigned dst = (unsigned)__cvta_generic_to_shared(&sm.tap_ring[bufn][0][lane]);
            if (nl == TAP_CHUNK) {  // whole chunk: ring offsets are immediates, the source a running pointer
#pragma unroll
                for (int l = 0; l < TAP_CHUNK; ++l, src += npix) cp_async4_saddr(dst + 128u * l, src, pol);
            } else {
                for (int l = 0; l < nl; ++l, src += npix) cp_async4_saddr(dst + 128u * l, src, pol);
            }
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
#pragma unroll 1
    for (int j = 0; j < a.num_nbrs; ++j) {
        const float *__restrict__ gplane = a.grayRf[j];
#pragma unroll 1
        for (int d0 = 0; d0 < D; d0 += TAP_CHUNK, buf ^= 1) {
            issue_next();
            cp_async_wait<1>();
            S.chunk(j, d0, min(TAP_CHUNK, D - d0), buf, gplane);
        }
    }
    cp_async_wait<0>();
    S.finish();
}

template <int R, bool STATS, int PITCH>
cudaError_t launch_screen2(const MatchArgs &a, cudaStream_t st) {
    auto kern = match_mvs_screen2_kernel<R, STATS, PITCH>;
    constexpr size_t smem = sizeof(Screen2Smem<STATS>) * SCREEN2_TILE_ROWS;
    if (smem > 48 * 1024) {  // (per device: set on every launch, it is cheap)
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
    }
    const dim3 grid((unsigned)((a.w + 31) / 32), (unsigned)((a.rows + SCREEN2_TILE_ROWS - 1) / SCREEN2_TILE_ROWS));
    kern<<<grid, 32 * SCREEN2_TILE_ROWS, smem, st>>>(a);
    return cudaGetLastError();
}

}  // namespace sr
