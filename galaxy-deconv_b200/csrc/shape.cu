// k_adaptive_moments: adaptive second moments of 48x48 stamps (the estimator of shape_core.cuh).
//
// One warp owns one stamp; 8 warps per 256-thread CTA.  Lane l loads pixels l + 32k (k < 72) once, coalesced, and keeps them in
// registers for every pass; gdshape::measure_warp (shape_warp.cuh) runs the passes, and a warp leaves as soon as its stamp stops.
// No shared memory, no block barrier.  The summation order is fixed per warp, so a stamp's result does not depend on the batch it
// is in.
#include "kernels.cuh"
#include "launch.cuh"
#include "shape_warp.cuh"

namespace gd {

constexpr int AM_WARPS = 8;
constexpr int AM_THREADS = 32 * AM_WARPS;
constexpr int AM_PER = gdshape::LANE_PIXELS;
static_assert(AM_PER * 32 == NPIX && STAMP == gdshape::STAMP, "pixel pattern");

__global__ void __launch_bounds__(AM_THREADS) k_adaptive_moments(const float* __restrict__ img, int batch, float guess_sigma,
                                                                 float* __restrict__ shape, int32_t* __restrict__ info) {
    const int lane = threadIdx.x & 31;
    const int stamp = blockIdx.x * AM_WARPS + (threadIdx.x >> 5);
    if (stamp >= batch) return;
    const float* src = img + (size_t)stamp * NPIX + lane;
    float px[AM_PER];
#pragma unroll
    for (int k = 0; k < AM_PER; ++k) px[k] = __ldcs(src + 32 * k);      // read once: evict-first
    float out[8];
    int passes;
    const int status = gdshape::measure_warp(px, lane, guess_sigma, out, &passes);
    if (lane == 0) {
        float* o = shape + (size_t)stamp * 8;
#pragma unroll
        for (int i = 0; i < 8; ++i) o[i] = out[i];
        info[(size_t)stamp * 2] = status;
        info[(size_t)stamp * 2 + 1] = passes;
    }
}

int launch_adaptive_moments(const float* img, int batch, float guess_sigma, float* shape, int32_t* info, cudaStream_t st) {
    if (batch <= 0) return GD_OK;
    k_adaptive_moments<<<(batch + AM_WARPS - 1) / AM_WARPS, AM_THREADS, 0, st>>>(img, batch, guess_sigma, shape, info);
    GD_LAUNCHED();
    return GD_OK;
}

}  // namespace gd
