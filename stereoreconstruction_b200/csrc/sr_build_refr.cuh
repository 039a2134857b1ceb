// sr_build_refr.cuh — stage (1) for refractive target views: tap-volume build with the
// reprojection organised around the label sweep.
//
// What is computed per (reference pixel, depth label, neighbour view) is Camera::project of
// pointFromDepth (stereo/multiviewstereo.cpp:740-750,768-775; project/camera.cpp:95-138,380-419).
// How: every quantity is an affine function of the ray parameter t(depth) and is hoisted per
// (pixel, view):
//     t      = depth*tA + tB                       (Plane3d(normal, C + normal*depth) + intersect)
//     a      = a0 + t*a1                           (N . local,  local = R*P + t_cam = Ls + t*Ld)
//     radv   = R0 + t*R1                           (local - a*N, the in-plane offset from the axis)
//     Kradv  = KR0 + t*KR1                         (K applied to radv, K normalised when distorted)
// The reference's quartic (camera.cpp:110-116) in the ratio rho = x/r needs only r^2:
//     G(rho) = rho^2 (s^2 rr + hh) - n^2 s^2 (rho^2 rr + dd),   s = 1 - rho,  rr = |radv|^2
// It has exactly one root in [0,1] (the physical one, SURVEY §8a G4).  rho moves smoothly along
// the depth axis, so the start is the quadratic extrapolation of the three previous labels
// (error ~1e-8) and ONE FP64 Newton step on G lands at ~1e-15; the loop repeats the step until it
// is below 3e-8 (cold start: the first labels of a chunk), a safeguarded bisection/Newton on the
// un-squared equation is the fallback.  No square root, no FP32 excursion, no FP64<->FP32
// conversions (16/clk/SM on B200) on the label path: ~65 FP64 instructions + 2 MUFU per label.
#pragma once
#include "sr_kernels.cuh"

namespace sr {

struct BuildRefrArgs {
    sr_camera nbr;               // target view
    double Kn[9];                // K, or for a distorted view K with rows 0/1 normalised:
                                 //   (K.row0 - cx K.row2)/fx, (K.row1 - cy K.row2)/fy, K.row2
    double fxs, cxs, fys, cys;   // pixel = (fxs*xd + cxs, fys*yd + cys): scale and shift folded in
    double prin[3], C[3];        // reference view principal direction and centre
    const double *rays;          // [6][h][w] of the reference view
    const double *depth_table;   // [D]
    const uint8_t *ref_mask;
    const uint8_t *nbr_mask;     // null: every neighbour pixel is WHITE (no mask was given)
    int32_t *taps;               // [D][rows][w] for this neighbour
    int w, h, row0, rows, D, d_chunk;
    int mvs;
    unsigned long long *check;   // optional [4] (SR_MATCH_STATS=1): labels interpolated, guard fall-backs,
                                 // interpolated labels whose tap differs from the exact projection (must be 0)
};

// fmin(fmax(v, lo), hi) with the same results (a NaN comes out as lo) as two compare+select pairs.
// max.f64/min.f64 expand to 7 instructions each on sm_100a (NaN canonicalisation), and the compiler
// turns the C++ `v > lo ? v : lo` back into max.f64: hence PTX.  3 instructions per bound.
__device__ __forceinline__ double clamp_sel(double v, double lo, double hi) {
    double r;
    asm("{\n\t.reg .pred p;\n\t"
        "setp.gt.f64 p, %1, %2;\n\tselp.f64 %0, %1, %2, p;\n\t"
        "setp.lt.f64 p, %0, %3;\n\tselp.f64 %0, %0, %3, p;\n\t}"
        : "=&d"(r)
        : "d"(v), "d"(lo), "d"(hi));
    return r;
}

__device__ __forceinline__ double rcp_approx(double a) {  // ~2^-20 relative (MUFU.RCP64H)
    double r;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(a));
    return r;
}

// Per (reference pixel, refractive target view) state of the label sweep: the hoisted affine
// geometry, and the exact projection of one label.  Shared by the label-mode build below and the
// curve-mode rasteriser (sr_curve.cuh).
struct RefrProjector {
    double tA, tB, a0, a1, pd, dd, n1, n2, fxs, cxs, fys, cys;
    d3 R0, R1, KR0, KR1, KdN;
    const double *depth_table, *k;
    bool ray_ok, distorted;

    // Kn: K, or K with rows 0/1 normalised for a distorted view (see BuildRefrArgs)
    __device__ __forceinline__ void init(const sr_camera &nbr, const double *Kn, const double *prin_, const double *C_,
                                         d3 src, d3 dir, const double *table, double fxs_, double cxs_, double fys_,
                                         double cys_) {
        // pointFromDepth: plane through C + prin*depth with unit normal nrm; t = (dist*nn - ns)/nd
        const d3 prin = ld3(prin_);
        const d3 nrm = normalized(prin);
        const double nd = dot(nrm, dir);
        ray_ok = !(fabs(nd) < 1e-10);
        const double inv_nd = 1.0 / nd;
        const double nC = dot(nrm, ld3(C_)), npn = dot(nrm, prin), nn = dot(nrm, nrm), ns = dot(nrm, src);
        tA = npn * nn * inv_nd;
        tB = (nC * nn - ns) * inv_nd;
        if (!ray_ok) {  // a ray parallel to the depth planes has no point at any label: t = -1 fails the test in project()
            tA = 0.0;
            tB = -1.0;
        }
        // camera-local ray and its decomposition about the interface normal
        const d3 Ls = fmul3(nbr.R, src) + ld3(nbr.t), Ld = fmul3(nbr.R, dir);
        const d3 N = ld3(nbr.plane_n);
        a0 = fdot(N, Ls);
        a1 = fdot(N, Ld);
        R0 = faxpy(-a0, N, Ls);
        R1 = faxpy(-a1, N, Ld);
        KR0 = fmul3(Kn, R0);
        KR1 = fmul3(Kn, R1);
        pd = nbr.plane_d;
        KdN = fmul3(Kn, pd * N);
        dd = pd * pd;
        n1 = nbr.n;
        n2 = n1 * n1;
        distorted = nbr.is_distorted != 0;
        k = nbr.dist;
        depth_table = table;
        fxs = fxs_;
        cxs = cxs_;
        fys = fys_;
        cys = cys_;
    }

    // Exact projection of label d.  rho_guess in [0,1] or < 0 (paraxial start).  Outputs the
    // coordinate that is truncated (U,V) and the root rho.
    __device__ __forceinline__ bool project(int d, double rho_guess, double &U, double &V, double &rho_out) const {
        const double t = fma(depth_table[d], tA, tB);
        if (t < 1e-10) return false;  // (also every label of a ray with !ray_ok, see init)
        const d3 radv = faxpy(t, R1, R0);
        const double rr = fdot(radv, radv);
        if (!(rr > 0.0)) return false;  // on the axis dir = radv/r is NaN in the reference: no root is accepted
        const double av = fma(t, a1, a0);
        const double h = fabs(av) - pd, hh = h * h;
        double rho = (rho_guess >= 0.0) ? rho_guess : n1 * fabs(pd) / (fabs(h) + n1 * fabs(pd) + 1e-300);
        rho = clamp_sel(rho, 0.0, 1.0);
        // One Newton step on G: G/2 and G'/2 = rho*B + n^2 s A - rho s rr (rho + n^2 s) at rho; returns the
        // step and leaves the reciprocal of G'/2 in rinv.
        double rinv = 0.0;
        auto half_G = [&](double rho_, double &A, double &B, double &s) {
            s = 1.0 - rho_;
            const double p2 = rho_ * rho_, s2 = s * s;
            A = fma(p2, rr, dd);
            B = fma(s2, rr, hh);
            return 0.5 * fma(p2, B, -((n2 * s2) * A));
        };
        auto newton_step = [&](double rho_) {
            double A, B, s;
            const double hG = half_G(rho_, A, B, s);
            const double u = fma(n2, s, rho_);
            const double g2 = fma(n2 * s, A, fma(rho_, B, -(((rho_ * s) * rr) * u)));
            rinv = rcp_approx(g2);
            return hG * rinv;
        };
        bool conv = false;
        double step = newton_step(rho);
        rho -= step;
        if (fabs(step) <= 3e-8) {
            conv = true;
#if SR_BUILD_CHORD
        } else if (fabs(step) <= 1e-5) {
            // The usual case between anchors (the extrapolated start is ~1e-6 off): the error is now
            // ~1e-12, and a chord step with the SAME derivative takes it to ~1e-12 * (|step| + 2^-20),
            // below the rounding of rho, for half the FP64 instructions of a second full step.
            double A, B, s;
            step = half_G(rho, A, B, s) * rinv;
            rho -= step;
            conv = fabs(step) <= 3e-8;
#endif
        }
        if (!conv) {
#pragma unroll 1
            for (int it = 0; it < 7; ++it) {
                rho = clamp_sel(rho, 0.0, 1.0);
                step = newton_step(rho);
                rho -= step;
                if (fabs(step) <= 3e-8) {
                    conv = true;
                    break;
                }
            }
        }
        if (!conv || !(rho >= 0.0 && rho <= 1.0)) {
            const double r = sqrt(rr);
            rho = snell_root_robust(r, pd, h, n1, -1.0) / r;
        }
        if (!(rho == rho)) return false;
        rho_out = rho;
        // point on the interface = rho*radv + d*N (camera.cpp:127); K*point hoisted
        const d3 Kr = faxpy(t, KR1, KR0);
        const d3 p = faxpy(rho, Kr, KdN);
        const double iz = fast_rcp(p.z);
        double xn = p.x * iz, yn = p.y * iz;
        if (distorted) {  // camera.cpp:395-416 on normalised coordinates
            const double k0 = k[0], k1 = k[1], k2 = k[2], k3 = k[3], k4 = k[4];
            const double q2 = fma(xn, xn, yn * yn);
            const double cdist = fma(fma(fma(k4, q2, k1), q2, k0), q2, 1.0);
            const double xo = xn, yo = yn;
            xn = fma(xo, cdist, fma(2 * k2 * xo, yo, k3 * fma(2 * xo, xo, q2)));
            // camera.cpp:411-412: y's tangential term uses the already-distorted x
            yn = fma(yo, cdist, fma(k2, fma(2 * yo, yo, q2), 2 * k3 * xn * yo));
        }
        U = fma(fxs, xn, cxs);
        V = fma(fys, yn, cys);
        return true;
    }
};

// Labels between two anchors are not re-projected: the pixel coordinate (U,V)(label) is an
// analytic, slowly varying function of the label, so it is read off the cubic through the four
// surrounding ANCHOR labels (every BUILD_STRIDE-th label, projected exactly as above).  What
// must be exact is only trunc(U), trunc(V): the interpolated value is accepted when it is farther
// from the nearest integer than a guard, otherwise that label is projected exactly as well.
//   guard = |third difference| * L2(x)  +  0.1 * |fourth difference|  +  1e-6 px
// The first term is |cubic - quadratic|, the full error of the NEXT-LOWER-order interpolant (~100x
// the cubic's own error where the differences decay, each by ~BUILD_STRIDE*dDepth/Depth ~ 1e-2).
// The second bounds the cubic's own error, <= 0.0234 * |fourth difference| + higher orders, with a
// 4x margin; it is what protects the labels near a sign change of the third difference, where the
// first term vanishes (found with stride 8: 2 differing taps in 2.5e9 without it).  The fourth
// difference is the change of the third difference from one interval to the next.  With the guard
// ~1e-4 px a label falls back with probability ~4e-4.
#ifndef SR_BUILD_STRIDE
#define SR_BUILD_STRIDE 4
#endif
#ifndef SR_BUILD_CHORD  // second solver step between anchors as a chord step (A/B)
#define SR_BUILD_CHORD 1
#endif
#ifndef SR_BUILD_ONEGUARD  // one guard threshold per interval (the largest L2) instead of one per label (A/B)
#define SR_BUILD_ONEGUARD 1
#endif
constexpr int BUILD_STRIDE = SR_BUILD_STRIDE;

// What one label sweep needs to know: the target view, the reference view's geometry and where the
// tables are.  (Pointers may point into the kernel's parameter space.)
struct BuildSweep {
    const sr_camera *nbr;        // target view
    const double *Kn;            // see BuildRefrArgs::Kn
    double fxs, cxs, fys, cys;
    const double *prin, *C;      // reference view principal direction and centre
    const double *rays;          // [6][h][w] of the reference view
    const double *depth_table;   // [D]
    const uint8_t *nbr_mask;     // null: every neighbour pixel is WHITE
    int w, h, D;
    unsigned long long *check;   // see BuildRefrArgs::check
};

// MVS: the multi-view tap rule (tap inside the image and WHITE in the neighbour's mask);
// HAS_MASK: the neighbour has a mask plane (a.nbr_mask != null).  Compile-time so that the other
// variant's clamps, mask address arithmetic and loads do not occupy (predicated-off) issue slots.
// Labels [d0, d1) of reference pixel (x, y), d0 a multiple of BUILD_STRIDE; sink(d, tap) receives every
// one of them exactly once, in increasing d.
template <bool MVS, bool HAS_MASK, class Sink>
__device__ __forceinline__ void build_refr_sweep(const BuildSweep &a, int x, int y, int d0, int d1, Sink sink) {
    const size_t pix = (size_t)y * a.w + x;
    const size_t n = (size_t)a.w * a.h;
    const d3 src = {a.rays[pix], a.rays[n + pix], a.rays[2 * n + pix]};
    const d3 dir = {a.rays[3 * n + pix], a.rays[4 * n + pix], a.rays[5 * n + pix]};
    RefrProjector pj;
    pj.init(*a.nbr, a.Kn, a.prin, a.C, src, dir, a.depth_table, a.fxs, a.cxs, a.fys, a.cys);
    const int D = a.D;

    // trunc toward zero of a coordinate without the conversion pipe (F2I.F64 issues at 16
    // lanes/clk/SM): r = rint(|c|) through the 1.5*2^52 constant, whose sum carries the integer in
    // its low word; diff = |c| - r is exact and tells floor from rint.  Also returns |diff|, the
    // distance to the nearest integer (the guard test).  Valid for |c| < 2^31; callers clamp.
    auto trunc_magic = [](double c, double &dist) -> int {
        const double MAGIC = 6755399441055744.0;
        const double m = fabs(c) + MAGIC;
        const double diff = fabs(c) - (m - MAGIC);
        dist = fabs(diff);
        const int fl = __double2loint(m) + (__double2hiint(diff) >> 31);  // rint - [diff < 0]
        return (__double2hiint(c) < 0) ? -fl : fl;
    };

    constexpr int S = BUILD_STRIDE;
    // anchor window: labels (k-1)S, kS, (k+1)S, (k+2)S for the interval [kS, (k+1)S)
    double au[4], av_[4], ar[4];
    unsigned aok = 0, asane = 0;  // bit = slot: the anchor projected / is usable as a node of the cubic
    auto anchor = [&](int slot, int d, double guess) {
        bool ok = false;
        au[slot] = av_[slot] = ar[slot] = 0.0;
        if (d >= 0 && d < D) ok = pj.project(d, guess, au[slot], av_[slot], ar[slot]);
        // an anchor far outside any image (a projection near the camera plane) is not interpolated
        // through: the labels around it are projected exactly, and the cubic never leaves 2^31
        const bool sane = ok && fabs(au[slot]) + fabs(av_[slot]) < 1.0e6;
        aok = (aok & ~(1u << slot)) | ((unsigned)ok << slot);
        asane = (asane & ~(1u << slot)) | ((unsigned)sane << slot);
    };
    const int kfirst = d0 / S;
    anchor(0, (kfirst - 1) * S, -1.0);
    anchor(1, kfirst * S, (aok & 1) ? ar[0] : -1.0);
    anchor(2, (kfirst + 1) * S, ((aok & 3) == 3) ? fma(2.0, ar[1], -ar[0]) : ((aok & 2) ? ar[1] : -1.0));
    // Lagrange weights of the cubic through nodes -1,0,1,2 at x = s/S and of its top term L2(x)
    double lw[S][4], l2[S];
#pragma unroll
    for (int s = 1; s < S; ++s) {
        const double xq = (double)s / S;
        lw[s][0] = -xq * (xq - 1) * (xq - 2) / 6;
        lw[s][1] = (xq + 1) * (xq - 1) * (xq - 2) / 2;
        lw[s][2] = -(xq + 1) * xq * (xq - 2) / 2;
        lw[s][3] = (xq + 1) * xq * (xq - 1) / 6;
        l2[s] = fabs(lw[s][3]);
    }
    double d3u_prev = 0.0, d3v_prev = 0.0;  // signed third differences of the previous interval
    bool have_d3 = false;
    const double CL = 30000.0;  // beyond any image: |c| >= TAP_CLAMP is outside every window
#pragma unroll 1
    for (int kk = kfirst; kk * S < d1; ++kk) {
        {
            double g = -1.0;
            if ((aok & 7) == 7) g = fma(3.0, ar[2] - ar[1], ar[0]);
            else if ((aok & 6) == 6) g = fma(2.0, ar[2], -ar[1]);
            else if (aok & 4) g = ar[2];
            anchor(3, (kk + 2) * S, g);
        }
        const int db = kk * S;
        const bool full = (asane & 15) == 15;
        double d3u = 0.0, d3v = 0.0, d4u = 0.0, d4v = 0.0;
        if (full) {
            const double su = (au[3] - au[0]) - 3.0 * (au[2] - au[1]);  // signed third differences
            const double sv = (av_[3] - av_[0]) - 3.0 * (av_[2] - av_[1]);
            d3u = fabs(su);
            d3v = fabs(sv);
            // fourth difference = change of the third difference between consecutive intervals; the
            // first full interval of a sweep has no predecessor and takes |third difference| instead
            d4u = have_d3 ? fabs(su - d3u_prev) : d3u;
            d4v = have_d3 ? fabs(sv - d3v_prev) : d3v;
            d3u_prev = su;
            d3v_prev = sv;
        }
        have_d3 = full;
        const double g0u = fma(0.1, d4u, 1e-6), g0v = fma(0.1, d4v, 1e-6);  // label-independent part of the guard
#if SR_BUILD_ONEGUARD
        const double gmaxu = fma(0.0625, d3u, g0u), gmaxv = fma(0.0625, d3v, g0v);  // L2(x) <= L2(1/2) = 1/16
#endif
        // ---- stage 1: coordinates of the S labels of this interval (branch-free) ----
        int tx[S], ty[S];
        bool ok[S];
        unsigned need_exact = 0;  // bit s: label must be projected exactly
        {
            double du, dv;
            tx[0] = trunc_magic(clamp_sel(au[1], -CL, CL), du);
            ty[0] = trunc_magic(clamp_sel(av_[1], -CL, CL), dv);
            ok[0] = (aok & 2) != 0;
        }
#pragma unroll
        for (int s = 1; s < S; ++s) {
            const double U = fma(lw[s][0], au[0], fma(lw[s][1], au[1], fma(lw[s][2], au[2], lw[s][3] * au[3])));
            const double V = fma(lw[s][0], av_[0], fma(lw[s][1], av_[1], fma(lw[s][2], av_[2], lw[s][3] * av_[3])));
            ok[s] = true;
#if SR_BUILD_ONEGUARD
            double du, dv;
            tx[s] = trunc_magic(U, du);  // |U|,|V| < 2^31 when `full`; otherwise recomputed below
            ty[s] = trunc_magic(V, dv);
            const bool safe = full && du > gmaxu && dv > gmaxv;
#else
            double du, dv;
            tx[s] = trunc_magic(U, du);
            ty[s] = trunc_magic(V, dv);
            const bool safe = full && du > fma(l2[s], d3u, g0u) && dv > fma(l2[s], d3v, g0v);
#endif
            if (!safe && db + s < d1) need_exact |= 1u << s;
        }
        // ---- stage 2 (rare): labels too close to a pixel boundary, or without a full stencil ----
        if (a.check) {
#pragma unroll
            for (int s = 1; s < S; ++s) {
                if (db + s >= d1) continue;
                if (need_exact & (1u << s)) {
                    if (full) atomicAdd(a.check + 1, 1ull);
                    continue;
                }
                double Ue, Ve, re, du;
                const bool oke = pj.project(db + s, fma((double)s / S, ar[2] - ar[1], ar[1]), Ue, Ve, re);
                atomicAdd(a.check + 0, 1ull);
                if (!oke || trunc_magic(clamp_sel(Ue, -CL, CL), du) != tx[s] || trunc_magic(clamp_sel(Ve, -CL, CL), du) != ty[s])
                    atomicAdd(a.check + 2, 1ull);
            }
        }
        if (need_exact) {
#pragma unroll
            for (int s = 1; s < S; ++s) {
                if (need_exact & (1u << s)) {
                    double U = 0.0, V = 0.0, rho, du;
                    double g = -1.0;
                    if ((aok & 6) == 6) g = fma((double)s / S, ar[2] - ar[1], ar[1]);
                    ok[s] = pj.project(db + s, g, U, V, rho);
                    tx[s] = trunc_magic(clamp_sel(U, -CL, CL), du);
                    ty[s] = trunc_magic(clamp_sel(V, -CL, CL), du);
                }
            }
        }
        // ---- stage 3: neighbour-mask test (loads issued together), pack, store ----
        bool keep[S];
        uint8_t mk[S];
#pragma unroll
        for (int s = 0; s < S; ++s) {
            keep[s] = ok[s];
            mk[s] = 255;
            if (MVS) {  // multiviewstereo.cpp:787: only WHITE neighbour-mask pixels are candidates
                keep[s] = keep[s] && (unsigned)tx[s] < (unsigned)a.w && (unsigned)ty[s] < (unsigned)a.h;
                if (HAS_MASK && keep[s]) mk[s] = a.nbr_mask[(size_t)ty[s] * a.w + tx[s]];
            }
        }
#pragma unroll
        for (int s = 0; s < S; ++s) {
            const int d = db + s;
            if (d >= d1) break;
            int32_t tap = TAP_NONE;
            if (keep[s] && (!HAS_MASK || mk[s] == 255)) {
                int cx = tx[s], cy = ty[s];
                if (!MVS) {  // (with the MVS rule the tap is inside the image already)
                    cx = max(-TAP_CLAMP, min(TAP_CLAMP, cx));
                    cy = max(-TAP_CLAMP, min(TAP_CLAMP, cy));
                }
                tap = (int32_t)(((uint32_t)(cy & 0xffff) << 16) | (uint32_t)(cx & 0xffff));
            }
            sink(d, tap);
        }
#pragma unroll
        for (int i = 0; i < 3; ++i) {
            au[i] = au[i + 1];
            av_[i] = av_[i + 1];
            ar[i] = ar[i + 1];
        }
        aok >>= 1;
        asane >>= 1;
    }
}

__device__ __forceinline__ BuildSweep build_sweep_of(const BuildRefrArgs &a) {
    BuildSweep s;
    s.nbr = &a.nbr;
    s.Kn = a.Kn;
    s.fxs = a.fxs;
    s.cxs = a.cxs;
    s.fys = a.fys;
    s.cys = a.cys;
    s.prin = a.prin;
    s.C = a.C;
    s.rays = a.rays;
    s.depth_table = a.depth_table;
    s.nbr_mask = a.nbr_mask;
    s.w = a.w;
    s.h = a.h;
    s.D = a.D;
    s.check = a.check;
    return s;
}

// One thread per reference pixel of the band, blockIdx.y = chunk of labels; the taps go to the
// [D][rows][w] volume of this neighbour.  128 threads and the register allocation that implies (128
// registers, 4 blocks per SM) measured best: 160 registers / 3 blocks took 8.6 vs 7.95 ms per cfg4 view.
template <bool MVS, bool HAS_MASK>
__global__ void __launch_bounds__(128) build_refr_kernel(const __grid_constant__ BuildRefrArgs a) {
    const int pid = blockIdx.x * blockDim.x + threadIdx.x;
    if (pid >= a.rows * a.w) return;
    const int x = pid % a.w, y = a.row0 + pid / a.w;
    if (a.ref_mask[(size_t)y * a.w + x] != 255) return;  // the match kernels never read taps of masked-out pixels
    const size_t plane = (size_t)a.rows * a.w;
    const int d0 = blockIdx.y * a.d_chunk;  // d_chunk is a multiple of BUILD_STRIDE
    const int d1 = min(d0 + a.d_chunk, a.D);
    // the sweep hands over labels d0, d0+1, ... in order: a running pointer instead of a 64-bit multiply per label
    build_refr_sweep<MVS, HAS_MASK>(build_sweep_of(a), x, y, d0, d1,
                                    [p = a.taps + pid + (size_t)d0 * plane, plane](int, int32_t tap) mutable {
                                        *p = tap;
                                        p += plane;
                                    });
}

}  // namespace sr
