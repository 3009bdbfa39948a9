// The adaptive-moments iteration of shape_core.cuh on one warp: the lane loop that k_adaptive_moments (shape.cu) and k_metacal
// (metacal.cu) share.
//
// Lane l holds pixels l + 32k (k < 72) of its stamp in registers for every pass.  Because 32k mod 48 cycles through 0, 32, 16,
// the column and row of those pixels are compile-time patterns: for k = 3j the pixel is (r, c) = (2j, l), for k = 3j + 1 it is
// (2j, l + 32) on lanes 0-15 and (2j + 1, l - 16) on lanes 16-31, for k = 3j + 2 it is (2j + 1, l + 16).  Each lane sums its 72
// contributions in k order, an xor butterfly gives every lane the same six totals (fp32 addition commutes, so the bits agree
// across lanes), and every lane runs the same update: control flow is warp-uniform.  The summation order is fixed, so a stamp's
// result does not depend on where its pixels came from.  Device only (warp shuffles); tests/cpu/test_shape_core.cpp sums in the
// same order on the host.
#pragma once
#include "shape_core.cuh"

namespace gdshape {

constexpr int LANE_PIXELS = STAMP * STAMP / 32;     // 72
static_assert(LANE_PIXELS % 3 == 0, "pixel pattern");

// all 32 lanes call this with their pixels px[k] = stamp[lane + 32k]; every lane returns the status and holds the eight outputs
__device__ __forceinline__ int measure_warp(const float (&px)[LANE_PIXELS], int lane, float guess_sigma, float (&out)[8], int* passes) {
    const float c0 = (float)lane, c1 = (float)(lane < 16 ? lane + 32 : lane - 16), c2 = (float)(lane + 16);
    const float h1 = lane < 16 ? 0.0f : 1.0f;                             // row offset of the k = 3j + 1 pixels
    auto sums = [&](const Weight& w, const Quad& q) {
        Sums s = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
        const float dx0 = c0 - w.x0, dx1 = c1 - w.x0, dx2 = c2 - w.x0;
#pragma unroll
        for (int j = 0; j < LANE_PIXELS / 3; ++j) {
            add_pixel(s, q, dx0, (float)(2 * j) - w.y0, px[3 * j]);
            add_pixel(s, q, dx1, ((float)(2 * j) + h1) - w.y0, px[3 * j + 1]);
            add_pixel(s, q, dx2, (float)(2 * j + 1) - w.y0, px[3 * j + 2]);
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            s.a += __shfl_xor_sync(0xffffffffu, s.a, o);
            s.bx += __shfl_xor_sync(0xffffffffu, s.bx, o);
            s.by += __shfl_xor_sync(0xffffffffu, s.by, o);
            s.cxx += __shfl_xor_sync(0xffffffffu, s.cxx, o);
            s.cxy += __shfl_xor_sync(0xffffffffu, s.cxy, o);
            s.cyy += __shfl_xor_sync(0xffffffffu, s.cyy, o);
        }
        return s;
    };
    return measure(guess_sigma, sums, out, passes);
}

}  // namespace gdshape
