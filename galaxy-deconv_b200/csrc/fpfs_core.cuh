// FPFS shear estimation of a 48x48 stamp (Li, Li & Mandelbaum 2018, MNRAS 481, 4445), __host__ __device__.
//
// On the grid k = 2 pi (u, v) / 48 (u, v the fftfreq integers -24..23, kx along columns) with r^2 = sigma^2 |k|^2 and
// G = exp(-r^2/2), the deconvolved power D(k) = |I~(k)|^2 / P(k), P = |p~(k)|^2 / |p~(0)|^2 (cells with P < 1e-8 give 0; no PSF:
// P = 1), is projected on six shapelet modes, summed over all 2304 cells:
//   M00  = 1/(sigma sqrt(pi))    sum D G                      M40  = 1/(sigma sqrt(pi)) sum D (r^4 - 4 r^2 + 2)/2 G
//   M22c = 1/(sigma sqrt(2 pi))  sum D r^2 cos2phi G          M42c = -1/(sigma sqrt(6 pi)) sum D r^2 (3 - r^2) cos2phi G
// and M22s, M42s with sin2phi.  With w = M00 + C: e1 = -M22c/w, e2 = -M22s/w, e41 = -M42c/w, e42 = -M42s/w and the response
// R = (M00 - M40)/(sqrt(2) w) + sqrt(6)/2 (e1 e41 + e2 e42); the shear of one galaxy is e / R, of an ensemble sum e / sum R.
//
// The basis is separable: with a = (sigma kx)^2, b = (sigma ky)^2, r^2 = a + b, r^2 cos2phi = a - b, r^2 sin2phi =
// 2 (sigma kx)(sigma ky) and G = exp(-a/2) exp(-b/2), so a cell needs no division and no transcendental; the per-frequency
// factors (Axis) are tabulated once.  Every basis function is even in k and the power of a real image is too, so the sums run
// over the half spectrum ky = 0..24 (fft rows k1 = 0..24, all 48 kx): rows 1..23 stand for themselves and their mirror rows
// (weight 2), rows 0 and 24 contain their own mirror cells (weight 1).  One exception: the mirror of the Nyquist column
// (u = -24, v) is (u = -24, -v), whose sin2phi has the opposite sign, so in rows 1..23 the sin terms of that column cancel.
//
// k_fpfs (fpfs.cu) and the host test tests/cpu/test_fpfs_core.cpp run this code; a row's cells are added in kx index order
// 0..47 (row_sums), the 25 row sums in row order 0..24 (finish).
#pragma once
#include <cuda_runtime.h>
#include <math.h>

#ifndef GD_HD
#define GD_HD __host__ __device__ __forceinline__
#endif

namespace gdfpfs {

constexpr int STAMP = 48;
constexpr int ROWS = STAMP / 2 + 1;        // half-spectrum rows k1 = 0..24
constexpr int NMODES = 6;                  // M00, M22c, M22s, M40, M42c, M42s
constexpr int NELL = 3;                    // e1, e2, R
constexpr float PSF_FLOOR = 1e-8f;
constexpr float DEFAULT_SIGMA = 3.5f;      // max_k G / P <= ~1.6 over the gdsynth PSFs (FWHM 2.25-4.75 px)

// per-frequency factors of fft index i (0..47): s = sigma k, a = s^2, g = exp(-a/2) (16-byte aligned: one load per table entry)
struct alignas(16) Axis { float s, a, g; };
GD_HD Axis axis(int i, float sigma) {
    const int f = i < STAMP / 2 ? i : i - STAMP;
    const float s = sigma * (0.13089969389957472f * (float)f);        // 2 pi / 48
    const float a = s * s;
    return {s, a, expf(-0.5f * a)};
}

// the unnormalised sums of one row, or of the whole stamp: m40 holds sum D (r^4 - 4 r^2 + 2) G (the 1/2 is in finish)
struct Sums { float m00, m22c, m22s, m40, m42c, m42s; };

// one cell of a row whose ky factors are y (b = y.a, sy = y.s): d is the deconvolved power D; the row's g factor is applied
// by the caller once per row (row_scale).  nyq_sin = false drops the sin terms (the Nyquist column of rows 1..23).
GD_HD void add_cell(Sums& s, const Axis& x, const Axis& y, float d, bool nyq_sin = true) {
    const float v = x.g * d;
    const float r2 = x.a + y.a, c2 = x.a - y.a, t2 = nyq_sin ? 2.0f * x.s * y.s : 0.0f;
    const float h = 3.0f - r2;
    s.m00 += v;
    s.m22c += c2 * v;
    s.m22s += t2 * v;
    s.m40 += (r2 * (r2 - 4.0f) + 2.0f) * v;
    s.m42c += h * c2 * v;
    s.m42s += h * t2 * v;
}

// does row k1 keep the sin terms of its Nyquist column (rows 0 and 24 contain that column's mirror cells themselves)
GD_HD bool row_keeps_nyquist_sin(int k1) { return k1 == 0 || k1 == ROWS - 1; }
// G's ky factor times the half-spectrum weight of row k1
GD_HD float row_scale(int k1, const Axis& y) { return row_keeps_nyquist_sin(k1) ? y.g : 2.0f * y.g; }

// D of one cell: hh = |p~(k)|^2, h0 = |p~(0)|^2; 0 where the PSF power is below the floor
GD_HD float psf_factor(float hh, float h0) { return hh >= PSF_FLOOR * h0 ? h0 / hh : 0.0f; }

// The scaled sums of row k1 (ky factors y): d(u) is D at fft column u, xs[u] the kx factors; cells are added in order u = 0..47.
template <class DFn> GD_HD Sums row_sums(int k1, const Axis& y, const Axis* xs, const DFn& d) {
    Sums s = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int u = 0; u < STAMP; ++u) add_cell(s, xs[u], y, d(u), u != STAMP / 2 || row_keeps_nyquist_sin(k1));
    const float sc = row_scale(k1, y);
    return {s.m00 * sc, s.m22c * sc, s.m22s * sc, s.m40 * sc, s.m42c * sc, s.m42s * sc};
}

// The estimator from the 25 row sums (each already multiplied by row_scale), added in row order.  psf_ok = the PSF sums to a
// positive value (always true without a PSF).  modes [6] may be NULL; ell [3] = e1, e2, R.
GD_HD void finish(const Sums* rows, float sigma, float cnst, bool psf_ok, float* modes, float* ell) {
    Sums t = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    for (int k1 = 0; k1 < ROWS; ++k1) {
        t.m00 += rows[k1].m00;
        t.m22c += rows[k1].m22c;
        t.m22s += rows[k1].m22s;
        t.m40 += rows[k1].m40;
        t.m42c += rows[k1].m42c;
        t.m42s += rows[k1].m42s;
    }
    const float n0 = 0.56418958354775628f / sigma;       // 1/(sigma sqrt(pi))
    const float n2 = 0.39894228040143268f / sigma;       // 1/(sigma sqrt(2 pi))
    const float n4 = -0.23032943298089031f / sigma;      // -1/(sigma sqrt(6 pi))
    float m[NMODES] = {n0 * t.m00, n2 * t.m22c, n2 * t.m22s, 0.5f * n0 * t.m40, n4 * t.m42c, n4 * t.m42s};
    if (!psf_ok)
        for (int i = 0; i < NMODES; ++i) m[i] = NAN;
    if (modes)
        for (int i = 0; i < NMODES; ++i) modes[i] = m[i];
    const float w = m[0] + cnst;
    if (!(w > 0.0f)) {
        ell[0] = ell[1] = ell[2] = NAN;
        return;
    }
    const float iw = 1.0f / w;
    const float e1 = -m[1] * iw, e2 = -m[2] * iw, e41 = -m[4] * iw, e42 = -m[5] * iw;
    ell[0] = e1;
    ell[1] = e2;
    ell[2] = (m[0] - m[3]) * (0.70710678118654752f * iw) + 1.2247448713915890f * (e1 * e41 + e2 * e42);
}

}  // namespace gdfpfs
