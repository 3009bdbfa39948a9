// k_metacal: metacalibration of 48x48 stamps.  The body, its shared-memory layout and its steps are in metacal_stamps.cuh.
#include "kernels.cuh"
#include "launch.cuh"
#include "metacal_stamps.cuh"

namespace gd {

__global__ void __launch_bounds__(MC_THREADS, 2) k_metacal(const float* __restrict__ img, const float* __restrict__ psf, int psf_batch,
                                                           int batch, float delta, float sigma, float guess_sigma,
                                                           float* __restrict__ images, float* __restrict__ shape,
                                                           int32_t* __restrict__ info) {
    metacal_stamps<false, PSF_RUNTIME>(img, psf, psf_batch, batch, delta, sigma, guess_sigma, nullptr, nullptr, 0, 0, 0, images, shape, info);
}

int metacal_init() {
    GD_CUDA_CHECK(cudaFuncSetAttribute(k_metacal, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)metacal_smem(true, false)));
    return GD_OK;
}

int launch_metacal(const float* img, const float* psf, int psf_batch, int batch, float delta, float sigma, float guess_sigma,
                   float* images, float* shape, int32_t* info, cudaStream_t st) {
    if (batch <= 0) return GD_OK;
    const bool with_psf = psf != nullptr;
    static int grid_cap[2] = {0, 0};                 // resident CTAs on the device, without / with a PSF
    if (!grid_cap[with_psf]) {
        const int cap = metacal_grid_cap((const void*)k_metacal, metacal_smem(with_psf, false));
        if (cap < 0) return cap;
        grid_cap[with_psf] = cap;
    }
    k_metacal<<<batch < grid_cap[with_psf] ? batch : grid_cap[with_psf], MC_THREADS, metacal_smem(with_psf, false), st>>>(
        img, psf, psf_batch, batch, delta, sigma, guess_sigma, images, shape, info);
    GD_LAUNCHED();
    return GD_OK;
}

}  // namespace gd
