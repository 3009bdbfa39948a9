// k_adaptive_moments: adaptive second moments of 48x48 stamps (the estimator of shape_core.cuh).
//
// One warp owns one stamp; 8 warps per 256-thread CTA.  Lane l loads pixels l + 32k (k < 72) once, coalesced, and keeps
// them in registers for every pass.  Because 32k mod 48 cycles through 0, 32, 16, the column and row of those pixels are
// compile-time patterns: for k = 3j the pixel is (r, c) = (2j, l), for k = 3j + 1 it is (2j, l + 32) on lanes 0-15 and
// (2j + 1, l - 16) on lanes 16-31, for k = 3j + 2 it is (2j + 1, l + 16).  Each lane sums its 72 contributions in k order,
// an xor butterfly gives every lane the same six totals (fp32 addition commutes, so the bits agree across lanes), and every
// lane runs the same update: control flow is warp-uniform, and a warp leaves as soon as its stamp stops.  No shared memory,
// no block barrier.  The summation order is fixed per warp, so a stamp's result does not depend on the batch it is in.
#include "kernels.cuh"
#include "launch.cuh"
#include "shape_core.cuh"

namespace gd {

constexpr int AM_WARPS = 8;
constexpr int AM_THREADS = 32 * AM_WARPS;
constexpr int AM_PER = NPIX / 32;          // 72 pixels per lane
static_assert(AM_PER % 3 == 0 && STAMP == gdshape::STAMP, "pixel pattern");

__global__ void __launch_bounds__(AM_THREADS) k_adaptive_moments(const float* __restrict__ img, int batch, float guess_sigma,
                                                                 float* __restrict__ shape, int32_t* __restrict__ info) {
    const int lane = threadIdx.x & 31;
    const int stamp = blockIdx.x * AM_WARPS + (threadIdx.x >> 5);
    if (stamp >= batch) return;
    const float* src = img + (size_t)stamp * NPIX + lane;
    float px[AM_PER];
#pragma unroll
    for (int k = 0; k < AM_PER; ++k) px[k] = __ldcs(src + 32 * k);      // read once: evict-first
    const float c0 = (float)lane, c1 = (float)(lane < 16 ? lane + 32 : lane - 16), c2 = (float)(lane + 16);
    const float h1 = lane < 16 ? 0.0f : 1.0f;                             // row offset of the k = 3j + 1 pixels
    auto sums = [&](const gdshape::Weight& w, const gdshape::Quad& q) {
        gdshape::Sums s = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
        const float dx0 = c0 - w.x0, dx1 = c1 - w.x0, dx2 = c2 - w.x0;
#pragma unroll
        for (int j = 0; j < AM_PER / 3; ++j) {
            gdshape::add_pixel(s, q, dx0, (float)(2 * j) - w.y0, px[3 * j]);
            gdshape::add_pixel(s, q, dx1, ((float)(2 * j) + h1) - w.y0, px[3 * j + 1]);
            gdshape::add_pixel(s, q, dx2, (float)(2 * j + 1) - w.y0, px[3 * j + 2]);
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
    float out[8];
    int passes;
    const int status = gdshape::measure(guess_sigma, sums, out, &passes);
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
