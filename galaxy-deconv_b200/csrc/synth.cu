// k_synth: synthetic galaxy stamps on the device, the CUDA twin of gdsynth.make_batch (gdsynth.py; the conventions of
// the reference's generate_data.py:114-334 and utils/utils_data.py:26-40,100-101).
//
// One CTA owns one stamp.  Every value depends only on (seed, start + blockIdx.x), and the block reductions run in a
// fixed order, so a stamp's bits do not depend on the batch it is generated in.  Stages, each skipped when nothing
// that was asked for needs it:
//   1. galaxy: 4x4 mean of the oversampled Sersic profile (synth_core.cuh), clamped at 0      -> needed for gt / obs
//   2. flux scale snr * sigma / sqrt(sum g^2) -> gt; gt goes to the 96x96 forward transform
//   3. true PSF: Moffat, normalised to sum 1 (block reduction); written as psf / 16 unless a mismatch was asked for
//   4. obs = max(gt (*) psf, 0) + sigma * N(0,1): the product of the two spectra, shifted by the PSF centre, through
//      the inverse transform (the FG96 blocks of k_g_prologue), then alpha = mean(obs)
//   5. mismatched model PSF (psf_fwhm_err / psf_shear_err != 0), written as psf / 16
// The stamp lives in Z (packed row pairs) between stages; shared memory: Z + two half spectra + twiddles = 96 KB,
// two CTAs per SM.
#include <math.h>
#include "fft_block.cuh"
#include "kernels.cuh"
#include "launch.cuh"
#include "synth_core.cuh"

namespace gd {

using FS96 = Real2D<96, 8, 12, 48>;
constexpr int SPS = 50;                    // row pitch of the half spectra (>= 49)
constexpr int SY_THREADS = 256;
constexpr int SY_PER = NPIX / SY_THREADS;  // 9 pixels per thread
constexpr size_t SY_SMEM = (size_t)(24 * 96 + 2 * 96 * SPS + 96) * sizeof(float2) + 64;
static_assert(NPIX % SY_THREADS == 0, "pixels per thread");

struct SynthArgs {
    uint64_t start, seed;
    int mixed;
    float snr, fwhm_err, shear_err;
    float *obs, *psf, *alpha, *gt;
};

// Moffat PSF of stamp idx into v[] (this thread's pixels), normalised to sum 1
__device__ __forceinline__ void render_psf(const gdsyn::PsfParams& pp, float (&v)[SY_PER], float* red) {
    float s = 0.f;
#pragma unroll 1
    for (int e = 0; e < SY_PER; ++e) {
        const int i = threadIdx.x + e * SY_THREADS, r = i / STAMP, c = i - r * STAMP;
        v[e] = gdsyn::render_pixel([&](float dx, float dy) { return gdsyn::moffat_value(pp, dx, dy); }, r, c);
        s += v[e];
    }
    s = block_sum(s, red);
#pragma unroll
    for (int e = 0; e < SY_PER; ++e) v[e] = gdsyn::fdiv(v[e], s);
}

__device__ __forceinline__ void store_psf16(float* dst, const float (&v)[SY_PER]) {
#pragma unroll
    for (int e = 0; e < SY_PER; ++e) dst[threadIdx.x + e * SY_THREADS] = gdsyn::fmul(v[e], 1.0f / 16.0f);
}

__global__ void __launch_bounds__(SY_THREADS, 2) k_synth(const __grid_constant__ SynthArgs a) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float2* Z = reinterpret_cast<float2*>(smem_raw);
    float2* SG = Z + 24 * 96;
    float2* SP = SG + 96 * SPS;
    float2* tw = SP + 96 * SPS;
    float* red = reinterpret_cast<float*>(tw + 96);
    const uint64_t idx = a.start + blockIdx.x;
    const size_t o = (size_t)blockIdx.x * NPIX;
    const bool mismatch = a.fwhm_err != 0.f || a.shear_err != 0.f;
    const bool need_obs = a.obs || a.alpha;
    const bool need_gal = need_obs || a.gt;
    const bool need_true_psf = need_obs || (a.psf && !mismatch);
    float v[SY_PER];

    if (need_gal) {
        if (need_obs) fill_twiddles<96>(tw);
        const gdsyn::GalaxyParams gp = gdsyn::galaxy_params(idx, a.seed);
        float ss = 0.f;
#pragma unroll 1
        for (int e = 0; e < SY_PER; ++e) {
            const int i = threadIdx.x + e * SY_THREADS, r = i / STAMP, c = i - r * STAMP;
            v[e] = fmaxf(gdsyn::render_pixel([&](float dx, float dy) { return gdsyn::sersic_value(gp, dx, dy); }, r, c), 0.f);
            ss += gdsyn::fmul(v[e], v[e]);
        }
        ss = block_sum(ss, red);
        const float snr = a.mixed ? gdsyn::snr_mixed(idx, a.seed) : a.snr;
        const float scale = gdsyn::fdiv(gdsyn::fmul(snr, gdsyn::SIGMA), sqrtf(ss));
#pragma unroll
        for (int e = 0; e < SY_PER; ++e) {
            const int i = threadIdx.x + e * SY_THREADS, r = i / STAMP, c = i - r * STAMP;
            const float g = gdsyn::fmul(v[e], scale);
            if (a.gt) a.gt[o + i] = g;
            if (need_obs) zpix<96>(Z, r, c) = g;
        }
        if (need_obs) fwd2d<FS96, SPS>(Z, SG, tw);          // leading barrier: Z and tw complete; trailing: Z free again
    }
    if (need_true_psf) {
        render_psf(gdsyn::psf_params(idx, a.seed, false, 0.f, 0.f), v, red);
        if (a.psf && !mismatch) store_psf16(a.psf + o, v);
        if (need_obs) {
#pragma unroll
            for (int e = 0; e < SY_PER; ++e) {
                const int i = threadIdx.x + e * SY_THREADS, r = i / STAMP, c = i - r * STAMP;
                zpix<96>(Z, r, c) = v[e];
            }
            fwd2d<FS96, SPS>(Z, SP, tw);
            GD_PHASE(FS96::NH * 96, gdsyn::conv_shift_product<FS96>(w, SG, SP, SPS));
            inv2d<FS96, SPS>(SG, Z, tw);
            float sum = 0.f;
#pragma unroll
            for (int e = 0; e < SY_PER; ++e) {
                const int i = threadIdx.x + e * SY_THREADS, r = i / STAMP, c = i - r * STAMP;
                const float y = gdsyn::obs_pixel(zpix<96>(Z, r, c), idx, i, a.seed);
                if (a.obs) a.obs[o + i] = y;
                sum += y;
            }
            sum = block_sum(sum, red);
            if (a.alpha && threadIdx.x == 0) a.alpha[blockIdx.x] = gdsyn::fdiv(sum, (float)NPIX);
        }
    }
    if (a.psf && mismatch) {
        render_psf(gdsyn::psf_params(idx, a.seed, true, a.fwhm_err, a.shear_err), v, red);
        store_psf16(a.psf + o, v);
    }
}

int synth_init() {
    GD_CUDA_CHECK(cudaFuncSetAttribute(k_synth, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SY_SMEM));
    return GD_OK;
}

int launch_synth(int64_t start, int count, int64_t seed, int mixed, float snr, float fwhm_err, float shear_err, float* obs,
                 float* psf, float* alpha, float* gt, cudaStream_t st) {
    if (count <= 0) return GD_OK;
    SynthArgs a;
    a.start = (uint64_t)start;
    a.seed = (uint64_t)seed;
    a.mixed = mixed;
    a.snr = snr;
    a.fwhm_err = fwhm_err;
    a.shear_err = shear_err;
    a.obs = obs; a.psf = psf; a.alpha = alpha; a.gt = gt;
    k_synth<<<count, SY_THREADS, SY_SMEM, st>>>(a);
    GD_LAUNCHED();
    return GD_OK;
}

}  // namespace gd
