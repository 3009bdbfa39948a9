// The body of k_metacal (metacal.cu) and k_metacal_fixnoise (metacal_fixnoise.cu): metacalibration of 48x48 stamps (the images of
// metacal_core.cuh, the shapes of shape_core.cuh), with or without the fix-noise images of metacal_core.cuh.
//
// Persistent grid, one stamp per CTA pass, all in shared memory:
//   load   the stamp (and a per-stamp PSF) into shared memory
//   fwd    Fft48 column and row passes of the stamp (and of a per-stamp PSF) into planes 0 (and 1): the grid spectrum
//   factor (PSF only) one thread per (shear, half-plane target): the PSF's spectrum at the sheared frequency (the DTFT, or the
//          grid spectrum for noshear), normalised by its sum, turned into G~ / P.  With one PSF for the batch this runs once per
//          CTA, before the first stamp, and the table stays in shared memory.
//   shear  one thread per (shear, target): the stamp's spectrum at the sheared frequency (the DTFT: 48 column factors in
//          registers, stamp rows read from shared memory as broadcasts; noshear: the grid spectrum) times G~ / P -> plane j
//   noise  (fix-noise only) one thread per (shear, target): the noise field's DTFT at the opposite shear's frequency (noshear: at
//          k) times the phase and the factor of the rotated cell, added to the cell of plane j
//   inv    Fft48 inverse row and column passes of the five planes; each real image lands in its own plane
//   out    the five images to `images` (if given); warps 0..4 measure one image each with gdshape::measure_warp, as
//          k_adaptive_moments does, loading their 72 pixels per lane from shared memory.
// A stamp's arithmetic is the same whichever CTA it lands in and whether its PSF is broadcast or repeated (the factor table is
// made by the same code either way), so its result does not depend on its batch.
#pragma once
#include "gd_common.cuh"
#include "metacal_core.cuh"
#include "shape_warp.cuh"

namespace gd {

namespace mc = gdmetacal;

constexpr int MC_THREADS = 256;                                  // 2 CTAs per SM at 128 registers, no spills
constexpr int MC_ITEMS = mc::NIMG * mc::NTARGET;                 // 4 sheared x 1105 DTFT items first, then 1105 noshear
static_assert(mc::NIMG * mc::HALF <= MC_THREADS, "one inverse column item per thread");
static_assert(mc::NIMG <= MC_THREADS / 32, "one warp per image for the shapes");
static_assert(mc::STAMP == STAMP && gdshape::LANE_PIXELS * 32 == NPIX, "stamp size");

// planes, s_img, s_psf (with a PSF or fix-noise: the PSF, then the noise field), factor (with a PSF)
static size_t metacal_smem(bool psf, bool fix) {
    return (size_t)mc::NIMG * mc::PLANE * sizeof(float2) + (psf || fix ? 2 : 1) * NPIX * sizeof(float) +
           (psf ? (size_t)mc::NIMG * mc::NTARGET * sizeof(float2) : 0);
}

// G~ / P of every (shear, target) of the PSF in s_psf whose grid spectrum is in pplane -> factor [5][1105].  Ends with a barrier.
__device__ __forceinline__ void psf_factors(const float* s_psf, const float2* pplane, float2* factor, float delta, float sigma) {
    const float p0 = pplane[0].x;
#pragma unroll 1
    for (int it = threadIdx.x; it < MC_ITEMS; it += MC_THREADS) {
        const int j = it < 4 * mc::NTARGET ? 1 + it / mc::NTARGET : 0, t = j ? it - (j - 1) * mc::NTARGET : it - 4 * mc::NTARGET;
        const mc::Cell k = mc::target(t);
        const int u = mc::fftfreq(k.i);
        const float sgn = mc::centre_sign(k.v, k.i);
        float2 pt;
        if (j) {
            const float2 f = mc::sheared_freq(j, delta, u, k.v);
            pt = mc::dtft(s_psf, f.x, f.y);
        } else {
            const float2 g = pplane[k.v * mc::PROW + k.i];
            pt = make_float2(sgn * g.x, sgn * g.y);
        }
        factor[j * mc::NTARGET + t] = mc::psf_factor(pt, p0, mc::reconv(k.v, k.i, sigma));
    }
    __syncthreads();
}

// the fix-noise field of a stamp -> s_noise: the caller's noise, or sigma N(start + stamp, p) (metacal_core.cuh) with sigma
// noise_sigma[stamp * sigma_step]
__device__ __forceinline__ void load_noise(float* s_noise, const float* __restrict__ noise, const float* __restrict__ noise_sigma,
                                           int sigma_step, int64_t start, int64_t seed, int stamp) {
    if (noise) {
        const float* src = noise + (size_t)stamp * NPIX;
        for (int i = threadIdx.x; i < NPIX; i += MC_THREADS) s_noise[i] = __ldcs(src + i);
    } else {
        const float sig = __ldg(noise_sigma + stamp * sigma_step);
        const uint64_t idx = (uint64_t)start + (uint64_t)stamp;
        for (int i = threadIdx.x; i < NPIX; i += MC_THREADS) s_noise[i] = mc::fixnoise_pixel(idx, i, (uint64_t)seed, sig);
    }
}

// forward Fft48 passes of n images (img[0], img[1]) into planes (plane, plane + PLANE).  Ends with a barrier.
__device__ __forceinline__ void forward(const float* im0, const float* im1, int n, float2* planes) {
#pragma unroll 1
    for (int it = threadIdx.x; it < n * mc::HALF; it += MC_THREADS)
        mc::fwd_col(it < mc::HALF ? im0 : im1, it % mc::HALF, planes + (it / mc::HALF) * mc::PLANE);
    __syncthreads();
#pragma unroll 1
    for (int it = threadIdx.x; it < n * mc::HALF; it += MC_THREADS) mc::fwd_row(planes + (it / mc::HALF) * mc::PLANE, it % mc::HALF);
    __syncthreads();
}

// resident CTAs of `kernel` on the current device with `smem` bytes
static inline int metacal_grid_cap(const void* kernel, size_t smem) {
    int dev, sms, per_sm;
    GD_CUDA_CHECK(cudaGetDevice(&dev));
    GD_CUDA_CHECK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    GD_CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, MC_THREADS, smem));
    return sms * (per_sm > 0 ? per_sm : 1);
}

// How the body learns whether there is a PSF and whether it is per stamp: from the arguments (k_metacal), or at compile time
// (k_metacal_fixnoise, whose noise steps leave no registers for the flags).
enum { PSF_RUNTIME = -1, PSF_NONE = 0, PSF_ONE = 1, PSF_EACH = 2 };

// The body of both kernels.  FIX: the fix-noise images (metacal_core.cuh), with the noise field of each stamp in s_noise: the
// caller's `noise`, or generated from (seed, start + stamp) and its sigma.  s_noise is the PSF's slot, free once the factors are
// made: after the prologue for one PSF, after psf_factors for a per-stamp PSF.  Then, after the stamp's items, one item per
// (shear, target) adds the noise term to its cell.
// HAS_PSF is evaluated where it is used, as k_metacal always has
#define HAS_PSF (MODE == PSF_RUNTIME ? psf != nullptr : MODE != PSF_NONE)
template <bool FIX, int MODE>
__device__ __forceinline__ void metacal_stamps(const float* __restrict__ img, const float* __restrict__ psf, int psf_batch, int batch,
                                               float delta, float sigma, float guess_sigma, const float* __restrict__ noise,
                                               const float* __restrict__ noise_sigma, int sigma_step, int64_t start, int64_t seed,
                                               float* __restrict__ images, float* __restrict__ shape, int32_t* __restrict__ info) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float2* planes = reinterpret_cast<float2*>(smem_raw);                          // [5][PLANE]
    float* s_img = reinterpret_cast<float*>(planes + mc::NIMG * mc::PLANE);         // [2304]
    float* s_psf = s_img + NPIX;                                                    // [2304], with a PSF or fix-noise
    float2* factor = reinterpret_cast<float2*>(s_psf + NPIX);                       // [5][1105], with a PSF
    const int tid = threadIdx.x;
    const bool per_stamp_psf = MODE == PSF_RUNTIME ? psf && psf_batch > 1 : MODE == PSF_EACH;
    if (HAS_PSF && !per_stamp_psf) {                     // one PSF for the batch: its factors once per CTA
        for (int i = tid; i < NPIX; i += MC_THREADS) s_psf[i] = psf[i];
        __syncthreads();
        forward(s_psf, nullptr, 1, planes + mc::PLANE);
        psf_factors(s_psf, planes + mc::PLANE, factor, delta, sigma);
    }
    for (int stamp = blockIdx.x; stamp < batch; stamp += gridDim.x) {
        const float* src = img + (size_t)stamp * NPIX;
        for (int i = tid; i < NPIX; i += MC_THREADS) s_img[i] = __ldcs(src + i);
        if (per_stamp_psf) {
            const float* p = psf + (size_t)stamp * NPIX;
            for (int i = tid; i < NPIX; i += MC_THREADS) s_psf[i] = __ldcs(p + i);
        }
        if (FIX && !per_stamp_psf) load_noise(s_psf, noise, noise_sigma, sigma_step, start, seed, stamp);
        __syncthreads();                             // also: the previous stamp's shapes are done with the planes
        forward(s_img, s_psf, per_stamp_psf ? 2 : 1, planes);
        if (per_stamp_psf) psf_factors(s_psf, planes + mc::PLANE, factor, delta, sigma);
        if (FIX && per_stamp_psf) load_noise(s_psf, noise, noise_sigma, sigma_step, start, seed, stamp);   // read after a barrier
#pragma unroll 1
        for (int it = tid; it < MC_ITEMS; it += MC_THREADS) {
            const int j = it < 4 * mc::NTARGET ? 1 + it / mc::NTARGET : 0, t = j ? it - (j - 1) * mc::NTARGET : it - 4 * mc::NTARGET;
            const mc::Cell k = mc::target(t);
            const float sgn = mc::centre_sign(k.v, k.i);
            float2 spec;
            if (j) {
                const float2 f = mc::sheared_freq(j, delta, mc::fftfreq(k.i), k.v);
                spec = mc::dtft(s_img, f.x, f.y);
            } else {
                const float2 g = planes[k.v * mc::PROW + k.i];
                spec = make_float2(sgn * g.x, sgn * g.y);
            }
            planes[j * mc::PLANE + k.v * mc::PROW + k.i] =
                HAS_PSF ? mc::cell_value(spec, factor[j * mc::NTARGET + t], sgn) : mc::cell_value(spec, mc::reconv(k.v, k.i, sigma), sgn);
        }
        __syncthreads();
        if (FIX) {
#pragma unroll 1
            for (int it = tid; it < MC_ITEMS; it += MC_THREADS) {
                const int j = it < 4 * mc::NTARGET ? 1 + it / mc::NTARGET : 0, t = j ? it - (j - 1) * mc::NTARGET : it - 4 * mc::NTARGET;
                const mc::Cell k = mc::target(t);
                const float2 f = mc::sheared_freq(mc::opposite(j), delta, mc::fftfreq(k.i), k.v);
                const float2 term = mc::fixnoise_value(j, t, delta, sigma, mc::dtft(s_psf, f.x, f.y), HAS_PSF ? factor : nullptr);
                float2* cell = planes + j * mc::PLANE + k.v * mc::PROW + k.i;
                *cell = make_float2(cell->x + term.x, cell->y + term.y);
            }
            __syncthreads();
        }
#pragma unroll 1
        for (int it = tid; it < mc::NIMG * mc::HALF; it += MC_THREADS) mc::inv_row(planes + (it / mc::HALF) * mc::PLANE, it % mc::HALF);
        __syncthreads();
        {   // each image overwrites its own plane: every column item is read before any is stored
            const bool mine = tid < mc::NIMG * mc::HALF;
            const int ci = mine ? tid : 0;           // the idle threads load item 0 too: a uniform load keeps x out of local memory
            float2 x[mc::STAMP];
            mc::inv_col(planes + (ci / mc::HALF) * mc::PLANE, ci % mc::HALF, x);
            __syncthreads();
            if (mine) mc::inv_col_store(x, ci % mc::HALF, reinterpret_cast<float*>(planes + (ci / mc::HALF) * mc::PLANE));
            __syncthreads();
        }
        if (images) {
            float* dst = images + (size_t)stamp * mc::NIMG * NPIX;
            for (int i = tid; i < mc::NIMG * NPIX; i += MC_THREADS)
                __stcs(dst + i, reinterpret_cast<const float*>(planes + (i / NPIX) * mc::PLANE)[i % NPIX]);
        }
        const int w = tid >> 5, lane = tid & 31;
        if (w < mc::NIMG) {
            const float* im = reinterpret_cast<const float*>(planes + w * mc::PLANE) + lane;
            float px[gdshape::LANE_PIXELS];
#pragma unroll
            for (int k = 0; k < gdshape::LANE_PIXELS; ++k) px[k] = im[32 * k];
            float out[mc::NSHAPE];
            int passes;
            const int status = gdshape::measure_warp(px, lane, guess_sigma, out, &passes);
            if (lane == 0) {
                const size_t o = (size_t)stamp * mc::NIMG + w;
#pragma unroll
                for (int i = 0; i < mc::NSHAPE; ++i) shape[o * mc::NSHAPE + i] = out[i];
                info[o * 2] = status;
                info[o * 2 + 1] = passes;
            }
        }
    }
}

#undef HAS_PSF

}  // namespace gd
