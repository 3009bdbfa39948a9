// Scalar math of the synthetic stamp generator (gdsynth.py), __host__ __device__.
//
// gdsynth.py stands in for the reference's GalSim pipeline (generate_data.py:114-334) and keeps its conventions:
// 48x48 stamps, 4x oversampled rendering followed by a 4x4 mean (utils/utils_data.py:26-40), Moffat PSF centred on
// pixel (24,24) normalised to sum 1, sigma = 19.04 ADU sky + read noise, g <- g * SNR * sigma / sqrt(sum g^2) and
// obs = max(g * psf, 0) + N(0, sigma^2), alpha = obs.mean() (utils/utils_data.py:100-101).
//
// Everything here follows gdsynth's fp32 expressions term by term, with the rounding points torch has: every
// elementwise torch op rounds once, so products that torch rounds before an add are rounded here too (fmul_rn & co.
// keep nvcc from contracting them into FMAs).  The hash is integer arithmetic and bit-identical to gdsynth's int64
// version (two's-complement wrap == uint64 wrap); the transcendentals (powf, expf, logf, cosf, sinf, atan2f) differ
// from torch's by a few ulp at most.  k_synth (synth.cu) and the host test tests/cpu/test_synth_core.cpp run this code.
#pragma once
#include <math.h>
#include <stdint.h>
#include "fft_core.cuh"

#ifndef GD_HD
#define GD_HD __host__ __device__ __forceinline__
#endif

namespace gdsyn {

constexpr int STAMP = 48;
constexpr int UPSAMPLE = 4;

// fp32 roundings of gdsynth's Python (double) constants, exactly as torch converts a Python scalar
constexpr float SIGMA = (float)19.036936954773942;        // sqrt(349.47 + (8.8*0.94/2.3)^2), generate_data.py:202
constexpr float PI_F = (float)3.141592653589793;
constexpr float TWO_PI_F = (float)6.283185307179586;       // 2.0 * math.pi
constexpr float THIRD_F = (float)0.3333333333333333;        // 1.0 / 3.0
constexpr float LOG20_F = (float)2.995732273553991;         // math.log(20.0)
constexpr float LOG15_F = (float)2.70805020110221;          // math.log(300.0) - math.log(20.0)

// ---- one rounding per torch op ----
GD_HD float fmul(float a, float b) {
#ifdef __CUDA_ARCH__
    return __fmul_rn(a, b);
#else
    return a * b;
#endif
}
GD_HD float fadd(float a, float b) {
#ifdef __CUDA_ARCH__
    return __fadd_rn(a, b);
#else
    return a + b;
#endif
}
GD_HD float fsub(float a, float b) {
#ifdef __CUDA_ARCH__
    return __fsub_rn(a, b);
#else
    return a - b;
#endif
}
GD_HD float fdiv(float a, float b) {
#ifdef __CUDA_ARCH__
    return __fdiv_rn(a, b);
#else
    return a / b;
#endif
}

// ---- counter-based hash (gdsynth.hashed_uniform) ----
constexpr uint64_t M1 = 0x9E3779B97F4A7C15ull;
constexpr uint64_t M2 = 0xBF58476D1CE4E5B9ull;
constexpr uint64_t M3 = 0x94D049BB133111EBull;

GD_HD uint64_t mix64(uint64_t x) {
    x = (x ^ (x >> 30)) * M2;
    x = (x ^ (x >> 27)) * M3;
    return x ^ (x >> 31);
}
// U[0,1) with 24 random bits from (seed, idx, stream)
GD_HD float hashed_uniform(uint64_t idx, int stream, uint64_t seed) {
    uint64_t x = idx * M1 + ((uint64_t)(stream + 1) * M2 + seed * M3);
    x = mix64(mix64(x) + (uint64_t)stream);
    return (float)(uint32_t)(x >> 40) * (1.0f / 16777216.0f);
}

// standard normal for noise key idx*4099 + j (gdsynth._hashed_normal on streams stream0 / stream0 + 1; obs noise: 40 / 41)
GD_HD float hashed_normal(uint64_t idx, int j, uint64_t seed, int stream0 = 40) {
    const uint64_t key = idx * 4099ull + (uint64_t)j;
    const float u1 = fmaxf(hashed_uniform(key, stream0, seed), 1.0f / 16777216.0f);
    const float u2 = hashed_uniform(key, stream0 + 1, seed);
    return fmul(sqrtf(fmul(-2.0f, logf(u1))), cosf(fmul(TWO_PI_F, u2)));
}

// ---- per-stamp parameters ----
struct GalaxyParams {
    // draws (streams 20-26)
    float n, re, e, th, x0, y0;
    int is_gauss;
    // derived
    float q, bn, inv_n, neg_bn, ct, st;
};

// gdsynth.make_galaxy: 50% Gaussian (Sersic n = 0.5), 50% Sersic n ~ U[0.5,4]; r_e ~ U[1.5,6] px, |e| ~ U[0,0.6],
// angle ~ U[0,pi), centroid offset ~ U[-1,1] px (generate_data.py:234-235)
GD_HD GalaxyParams galaxy_params(uint64_t idx, uint64_t seed) {
    GalaxyParams g;
    g.is_gauss = hashed_uniform(idx, 20, seed) < 0.5f;
    g.n = g.is_gauss ? 0.5f : fadd(0.5f, fmul(3.5f, hashed_uniform(idx, 21, seed)));
    g.re = fadd(1.5f, fmul(4.5f, hashed_uniform(idx, 22, seed)));
    g.e = fmul((float)0.6, hashed_uniform(idx, 23, seed));
    g.th = fmul(PI_F, hashed_uniform(idx, 24, seed));
    g.x0 = fsub(fmul(2.0f, hashed_uniform(idx, 25, seed)), 1.0f);
    g.y0 = fsub(fmul(2.0f, hashed_uniform(idx, 26, seed)), 1.0f);
    g.q = fdiv(fsub(1.0f, g.e), fadd(1.0f, g.e));
    // bn = 2n - 1/3 + 4/(405 n); torch evaluates 4.0/t as reciprocal(t) * 4, which equals 4/t in binary floating point
    g.bn = fadd(fsub(fmul(2.0f, g.n), THIRD_F), fdiv(4.0f, fmul(405.0f, g.n)));
    g.inv_n = fdiv(1.0f, g.n);
    g.neg_bn = -g.bn;
    g.ct = cosf(g.th);
    g.st = sinf(g.th);
    return g;
}

struct PsfParams {
    // draws (streams 10-13) and mismatch signs (streams 50 / 51; +-1, only set for a model PSF)
    float beta, fwhm, e0, th0, sg, sg2;
    // derived (after the optional FWHM / shear error)
    float e, th, q, a, neg_beta, ct, st;
};

// gdsynth.make_psf: Moffat, beta ~ U[2.5,4.5], FWHM ~ U[2.25,4.75] px, ellipticity 0.01-0.03 (generate_data.py:185,209).
// model = true: the mismatched model PSF of make_batch (FWHM error sg * fwhm_err arcsec, shear (sg, sg2) * shear_err,
// test_psf.py:237,242).
GD_HD PsfParams psf_params(uint64_t idx, uint64_t seed, bool model, float fwhm_err, float shear_err) {
    PsfParams p;
    p.beta = fadd(2.5f, fmul(2.0f, hashed_uniform(idx, 10, seed)));
    p.fwhm = fadd(2.25f, fmul(2.5f, hashed_uniform(idx, 11, seed)));
    p.e0 = fadd((float)0.01, fmul((float)0.02, hashed_uniform(idx, 12, seed)));
    p.th0 = fmul(PI_F, hashed_uniform(idx, 13, seed));
    p.sg = p.sg2 = 0.0f;
    float e1 = fmul(p.e0, cosf(fmul(2.0f, p.th0))), e2 = fmul(p.e0, sinf(fmul(2.0f, p.th0)));
    if (model) {
        p.sg = hashed_uniform(idx, 50, seed) < 0.5f ? -1.0f : 1.0f;
        p.sg2 = hashed_uniform(idx, 51, seed) < 0.5f ? -1.0f : 1.0f;
        p.fwhm = fadd(p.fwhm, fdiv(fmul(p.sg, fwhm_err), (float)0.2));
        e1 = fadd(e1, fmul(p.sg, shear_err));
        e2 = fadd(e2, fmul(p.sg2, shear_err));
    }
    p.e = fminf(fmaxf(sqrtf(fadd(fmul(e1, e1), fmul(e2, e2))), (float)1e-6), (float)0.9);
    p.th = fmul(0.5f, atan2f(e2, e1));
    p.q = fdiv(fsub(1.0f, p.e), fadd(1.0f, p.e));
    p.a = fdiv(p.fwhm, fmul(2.0f, sqrtf(fsub(powf(2.0f, fdiv(1.0f, p.beta)), 1.0f))));
    p.neg_beta = -p.beta;
    p.ct = cosf(p.th);
    p.st = sinf(p.th);
    return p;
}

// SNR of stamp idx in 'mixed' mode: log-uniform in [20, 300] (stream 30)
GD_HD float snr_mixed(uint64_t idx, uint64_t seed) {
    return expf(fadd(LOG20_F, fmul(LOG15_F, hashed_uniform(idx, 30, seed))));
}

// ---- profiles at one sub-pixel offset (dx, dy) from the centre of pixel (24,24), in stamp pixels ----
// area-preserving elliptical radius of gdsynth._rot_ellipse_radius
GD_HD float ellipse_radius(float ddx, float ddy, float ct, float st, float q) {
    const float xr = fadd(fmul(ddx, ct), fmul(ddy, st));
    const float yr = fadd(fmul(-ddx, st), fmul(ddy, ct));
    return sqrtf(fadd(fmul(fmul(xr, xr), q), fdiv(fmul(yr, yr), q)));
}
GD_HD float sersic_value(const GalaxyParams& g, float dx, float dy) {
    const float r = ellipse_radius(fsub(dx, g.x0), fsub(dy, g.y0), g.ct, g.st, g.q);
    return expf(fmul(g.neg_bn, fsub(powf(fadd(fdiv(r, g.re), (float)1e-12), g.inv_n), 1.0f)));
}
GD_HD float moffat_value(const PsfParams& p, float dx, float dy) {
    const float t = fdiv(ellipse_radius(dx, dy, p.ct, p.st, p.q), p.a);
    return powf(fadd(1.0f, fmul(t, t)), p.neg_beta);
}

// centre of oversampled row / column i in [0, 192): (i + 0.5) / 4 - 0.5 - 24 (exact in fp32)
GD_HD float sub_offset(int i) { return ((float)i + 0.5f) * 0.25f - 24.5f; }

// 4x4 mean of the oversampled grid over stamp pixel (r, c) (gdsynth._render)
template <class Fn> GD_HD float render_pixel(const Fn& fn, int r, int c) {
    float s = 0.0f;
#pragma unroll
    for (int sy = 0; sy < UPSAMPLE; ++sy) {
        const float dy = sub_offset(UPSAMPLE * r + sy);
#pragma unroll
        for (int sx = 0; sx < UPSAMPLE; ++sx) s = fadd(s, fn(sub_offset(UPSAMPLE * c + sx), dy));
    }
    return fmul(s, 1.0f / (UPSAMPLE * UPSAMPLE));
}

// ---- forward model (gdsynth.convolve_padded) ----
// With g and psf both placed at the corner of a zero-padded 96x96 grid, G*P is the spectrum of their full linear
// convolution f[m] = sum g[m'] psf[m - m'];  the stamp wants out[r] = f[r + 24] (PSF centre at pixel 24), a shift by
// 24 = N/4, i.e. a factor exp(+2 pi i 24 k / 96) = (+i)^(k1+k2) = (-i)^(3 (k1+k2)).  Item q of the 96 x 49 half
// spectrum (digit-swapped row slot s1, natural column k2; fft_core.cuh Real2D<96, ...>), in place in sg.
template <class F> GD_HD void conv_shift_product(int q, float2* sg, const float2* sp, int SP) {
    const int s1 = q / F::NH, k2 = q - s1 * F::NH;
    const float2 v = gdfft::cmul(sg[s1 * SP + k2], sp[s1 * SP + k2]);
    sg[s1 * SP + k2] = gdfft::mul_negi_pow(v, 3 * (F::L::freq(s1) + k2));
}

// obs pixel j of stamp idx from the unscaled inverse transform value `acc` (times 1/96^2): max(conv, 0) + sigma * N(0,1)
GD_HD float obs_pixel(float acc, uint64_t idx, int j, uint64_t seed) {
    const float conv = fmaxf(fmul(acc, 1.0f / (96.0f * 96.0f)), 0.0f);
    return fadd(conv, fmul(SIGMA, hashed_normal(idx, j, seed)));
}

}  // namespace gdsyn
