// sr_match_dispatch.cuh — (radius, cost) -> match_kernel<R,G,COST> instantiation.
// G (lanes cooperating on one pixel) is chosen so that the per-lane tap share (two FP64
// registers per tap) stays within the register file: ceil((2R+1)^2 / G) <= 35.
#pragma once
#include "sr_kernels.cuh"
#include "sr_match_screen.cuh"
#include "sr_screen2.cuh"

namespace sr {

template <int R> struct LanesFor { static constexpr int G = (R <= 2) ? 1 : (R == 3) ? 2 : (R <= 5) ? 4 : (R <= 7) ? 8 : (R <= 10) ? 16 : 32; };

// Radii with a compiled match kernel.  SR_FEW_RADII (the default build, capi.py) leaves out 6-12 to
// keep the nvcc time of the (radius x cost x pitch) instantiations in check.
#ifdef SR_FEW_RADII
inline bool match_supported(int r) { return (r >= 1 && r <= 5) || r == 16; }
#define SR_RADII_TEXT "1-5, 16 (build without -DSR_FEW_RADII for 6-8, 10, 12)"
#else
inline bool match_supported(int r) { return (r >= 1 && r <= 8) || r == 10 || r == 12 || r == 16; }
#define SR_RADII_TEXT "1-8, 10, 12, 16"
#endif

template <int R, int COST>
cudaError_t launch_match_rc(const MatchArgs &a, cudaStream_t st) {
    constexpr int G = LanesFor<R>::G;
    constexpr int PPB = 128 / G;
    const size_t npix = (size_t)a.rows * a.w;
    const unsigned grid = (unsigned)((npix + PPB - 1) / PPB);
    constexpr size_t smem = (G > 1) ? (size_t)PPB * (2 * R + 1) * (2 * R + 1) * sizeof(double) : 0;  // wstage
    if (smem > 0) {  // with the static tap ring the block can exceed 48 KB (r = 16): opt in
        const cudaError_t e = cudaFuncSetAttribute(match_kernel<R, G, COST>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
    }
    match_kernel<R, G, COST><<<grid, 128, smem, st>>>(a);
    return cudaGetLastError();
}

// MultiViewStereo selection with its own NCC and no kept cost volume: FP32 screen + FP64 verify.
template <int R>
cudaError_t launch_match_screen(const MatchArgs &a, cudaStream_t st) {
    constexpr int G = LanesFor<R>::G;  // (two lanes per pixel at r = 2 measured 1.7x slower: 35.8 vs 20.4 ms)
    if constexpr (G == 1) {  // thread-per-pixel radii: sr_screen2.cuh, the row pitch a compile-time constant
        if (a.stats) return launch_screen2<R, true, 0>(a, st);
        switch (a.pitch_f) {
            case 1024: return launch_screen2<R, false, 1024>(a, st);
            case 2048: return launch_screen2<R, false, 2048>(a, st);
            case 4096: return launch_screen2<R, false, 4096>(a, st);
            default: return launch_screen2<R, false, 0>(a, st);
        }
    } else {  // lane groups: sr_match_screen.cuh, one warp per block
        constexpr int PPB = SCREEN_BLOCK / G;
        const unsigned grid = (unsigned)(((size_t)a.rows * a.w + PPB - 1) / PPB);
        if (a.stats) match_mvs_screen_kernel<R, G, true><<<grid, SCREEN_BLOCK, 0, st>>>(a);
        else match_mvs_screen_kernel<R, G, false><<<grid, SCREEN_BLOCK, 0, st>>>(a);
        return cudaGetLastError();
    }
}

template <int R>
cudaError_t launch_match_r(int cost, const MatchArgs &a, cudaStream_t st) {
    if (cost == SR_COST_NCC_MVS && a.select_kind == SR_SELECT_MVS && !a.out_volume && !a.out_peaks && (a.use_screen || a.curve))
        return launch_match_screen<R>(a, st);
    switch (cost) {
        case SR_COST_NCC_TWOVIEW: return launch_match_rc<R, SR_COST_NCC_TWOVIEW>(a, st);
        case SR_COST_NCC_MVS: return launch_match_rc<R, SR_COST_NCC_MVS>(a, st);
        default: return launch_match_rc<R, SR_COST_SAD_TWOVIEW>(a, st);
    }
}

inline cudaError_t launch_match(int radius, int cost, const MatchArgs &a, cudaStream_t st) {
    switch (radius) {
        case 1: return launch_match_r<1>(cost, a, st);
        case 2: return launch_match_r<2>(cost, a, st);
        case 3: return launch_match_r<3>(cost, a, st);
        case 4: return launch_match_r<4>(cost, a, st);
        case 5: return launch_match_r<5>(cost, a, st);
#ifndef SR_FEW_RADII
        case 6: return launch_match_r<6>(cost, a, st);
        case 7: return launch_match_r<7>(cost, a, st);
        case 8: return launch_match_r<8>(cost, a, st);
        case 10: return launch_match_r<10>(cost, a, st);
        case 12: return launch_match_r<12>(cost, a, st);
#endif
        case 16: return launch_match_r<16>(cost, a, st);
        default: return cudaErrorInvalidValue;
    }
}

}  // namespace sr
