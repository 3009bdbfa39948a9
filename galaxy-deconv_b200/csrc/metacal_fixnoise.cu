// k_metacal_fixnoise: metacalibration of 48x48 stamps with the fix-noise correction (metacal_core.cuh), one instantiation per PSF
// form.  The body is k_metacal's (metacal_stamps.cuh); it is compiled apart from k_metacal, which keeps its own code.
#include "kernels.cuh"
#include "launch.cuh"
#include "metacal_stamps.cuh"

namespace gd {

template <int MODE>
__global__ void __launch_bounds__(MC_THREADS, 2)
    k_metacal_fixnoise(const float* __restrict__ img, const float* __restrict__ psf, int psf_batch, int batch, float delta, float sigma,
                       float guess_sigma, const float* __restrict__ noise, const float* __restrict__ noise_sigma, int sigma_step,
                       int64_t start, int64_t seed, float* __restrict__ images, float* __restrict__ shape, int32_t* __restrict__ info) {
    metacal_stamps<true, MODE>(img, psf, psf_batch, batch, delta, sigma, guess_sigma, noise, noise_sigma, sigma_step, start, seed, images,
                         shape, info);
}

int metacal_fixnoise_init() {
    GD_CUDA_CHECK(cudaFuncSetAttribute(k_metacal_fixnoise<PSF_NONE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)metacal_smem(false, true)));
    GD_CUDA_CHECK(cudaFuncSetAttribute(k_metacal_fixnoise<PSF_ONE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)metacal_smem(true, true)));
    GD_CUDA_CHECK(cudaFuncSetAttribute(k_metacal_fixnoise<PSF_EACH>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)metacal_smem(true, true)));
    return GD_OK;
}

int launch_metacal_fixnoise(const float* img, const float* psf, int psf_batch, int batch, float delta, float sigma, float guess_sigma,
                            const float* noise, const float* noise_sigma, int sigma_batch, int64_t start, int64_t seed, float* images,
                            float* shape, int32_t* info, cudaStream_t st) {
    if (batch <= 0) return GD_OK;
    const int mode = !psf ? PSF_NONE : psf_batch > 1 ? PSF_EACH : PSF_ONE;
    void (*const kernels[3])(const float*, const float*, int, int, float, float, float, const float*, const float*, int, int64_t, int64_t,
                             float*, float*, int32_t*) = {k_metacal_fixnoise<PSF_NONE>, k_metacal_fixnoise<PSF_ONE>, k_metacal_fixnoise<PSF_EACH>};
    static int grid_cap[3] = {0, 0, 0};              // resident CTAs on the device per PSF mode
    const size_t smem = metacal_smem(psf != nullptr, true);
    if (!grid_cap[mode]) {
        const int cap = metacal_grid_cap((const void*)kernels[mode], smem);
        if (cap < 0) return cap;
        grid_cap[mode] = cap;
    }
    kernels[mode]<<<batch < grid_cap[mode] ? batch : grid_cap[mode], MC_THREADS, smem, st>>>(
        img, psf, psf_batch, batch, delta, sigma, guess_sigma, noise, noise_sigma, sigma_batch > 1 ? 1 : 0, start, seed, images, shape, info);
    GD_LAUNCHED();
    return GD_OK;
}

}  // namespace gd
