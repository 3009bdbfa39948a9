// Metacalibration images of a 48x48 stamp (Huff & Mandelbaum 2017; Sheldon & Huff 2017), __host__ __device__.
//
// Pixel p = 48 r + c sits at X = c - 24, Y = r - 24; the grid frequencies are k = 2 pi (u, v) / 48 (u, v the fftfreq integers
// -24..23, kx along columns).  With I~(q) = sum_{r,c} I[r,c] exp(-i (qx X + qy Y)) (the same for the PSF p~), the shear
// A_g = [[1+g1, g2], [g2, 1-g1]] / sqrt(1 - g1^2 - g2^2) and the round reconvolution kernel G~(k) = exp(-sigma^2 |k|^2 / 2),
// image j of the five shears (0,0), (+d,0), (-d,0), (0,+d), (0,-d) has the spectrum
//   M_j(k) = I~(A_j k) G~(k) / P(A_j k),   P = p~ / p~(0)   (0 where |P|^2 < 1e-8; no PSF: P = 1; 0 on the Nyquist row and column)
// and the image is Re ifft2(M_j (-1)^(u+v)): the sign factor centres it at pixel (24, 24).
//
// M_j is Hermitian, so only the 1,105 half-plane targets are computed: row v = 0 with u = 0..23 and rows v = 1..23 with every
// u except the Nyquist column; row 0's cells u < 0 are their conjugate mirrors.  The noshear spectrum is on the grid and comes
// from the FFT (Fft48 column and row passes, as k_fpfs); the four sheared ones are off the grid and come from the direct DTFT
// (dtft below).  The spectra live in "planes" of 24 rows (v = 0..23; the Nyquist row is zero) of PROW float2, fft column order.
//
// Fix-noise (Sheldon & Huff 2017).  Metacalibration shears the stamp's noise with the galaxy, and adaptive moments respond to the
// sheared noise as to a shear.  With a second noise field n of the stamp's kind, fix-noise image j is
//   T_j(I) + rot^-1(T_j(rot n))
// where T_j maps a stamp to image j above (deconvolution, shear, reconvolution, floor, Nyquist rule and centring) and
// rot(a)[r][c] = a[c][47 - r] (numpy's rot90).  A quarter turn flips the sign of a shear, so the two noise fields are sheared in
// opposite senses and their spurious responses cancel; the images carry twice the noise variance of the stamp.  The second term
// folds into plane j:
//   rot(a)(X, Y) = a(-Y - 1, X), so FT[rot a](q) = exp(i qy) a~(R q) and, on the grid, FT[rot^-1 m](k) = exp(i kx) m~(R^-1 k),
//   with R (x, y) = (-y, x).  With R A_g R^-1 = A_-g and F_j(k) = G~(k) / P(A_j k) (G~ without a PSF; 0 where floored and on the
//   Nyquist row and column):
//     FT[rot^-1 T_j rot n](k) = exp(i (kx + qy)) n~(A_j' k) F_j(R^-1 k),   q = A_j R^-1 k
//   j' is the opposite shear (1p <-> 1m, 2p <-> 2m, noshear <-> noshear).  For noshear qy = -kx: the phase is 1.  R^-1 (u, v) =
//   (v, -u) maps the grid onto itself and the Nyquist row and column onto each other, so F_j(R^-1 k) of a target is the factor
//   of another target, or the conjugate of its mirror (F_j(-k) = conj F_j(k)); G~ is unchanged by it.
// So fix-noise needs one more DTFT per (shear, target), of n at A_j' k (noshear: at k), and no more planes or factors.  The
// generated field of stamp idx is n[p] = sigma N(idx, p), gdsynth._hashed_normal on streams 60 / 61 (gdsynth's draws use streams
// 10-51, so it is independent of the obs noise under any seed).
//
// k_metacal (metacal.cu), k_metacal_fixnoise (metacal_fixnoise.cu) and the host tests tests/cpu/test_metacal_core.cpp and
// tests/cpu/test_metacal_fixnoise_core.cpp run this code.
#pragma once
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>
#include "fft_core.cuh"
#include "synth_core.cuh"

#ifndef GD_HD
#define GD_HD __host__ __device__ __forceinline__
#endif

namespace gdmetacal {

using gdfft::Fft48;

constexpr int STAMP = 48;
constexpr int NPIX = STAMP * STAMP;
constexpr int HALF = STAMP / 2;              // 24: the centre pixel, and the fft index of the Nyquist frequency
constexpr int NIMG = 5;                      // noshear, 1p, 1m, 2p, 2m
constexpr int NTARGET = HALF + (HALF - 1) * (STAMP - 1);   // 24 + 23 * 47 = 1105 half-plane targets
constexpr int PROW = 50;                     // float2 per plane row (16-byte rows, conflict-free float4 reads as k_wiener48)
constexpr int PLANE = HALF * PROW;            // float2 per plane: rows v = 0..23
constexpr float PSF_FLOOR = 1e-8f;           // the floor of fpfs_core.cuh
constexpr float MAX_DELTA = 0.1f;
constexpr float MAX_SIGMA = 24.0f;
constexpr int NSHAPE = 8;                    // the record of gd_adaptive_moments
static_assert(NPIX * sizeof(float) <= PLANE * sizeof(float2), "an image fits in its plane");

GD_HD int fftfreq(int i) { return i < HALF ? i : i - STAMP; }

// target t (0..NTARGET-1) -> plane row v and fft column i
struct Cell { int v, i; };
GD_HD Cell target(int t) {
    if (t < HALF) return {0, t};
    const int s = t - HALF, j = s % (STAMP - 1);
    return {1 + s / (STAMP - 1), j < HALF ? j : j + 1};
}

// shear j of the five, applied to the integer frequencies (u, v): (fx, fy) = A_j (u, v) in cycles per 48 px
GD_HD float2 sheared_freq(int j, float delta, int u, int v) {
    const float g1 = j == 1 ? delta : j == 2 ? -delta : 0.0f, g2 = j == 3 ? delta : j == 4 ? -delta : 0.0f;
    const float n = 1.0f / sqrtf(1.0f - g1 * g1 - g2 * g2);
    const float fu = (float)u, fv = (float)v;
    return make_float2(((1.0f + g1) * fu + g2 * fv) * n, (g2 * fu + (1.0f - g1) * fv) * n);
}

// G~(k) of the reconvolution kernel at fft cell (v, i)
GD_HD float reconv(int v, int i, float sigma) {
    const float kx = 0.13089969389957472f * (float)fftfreq(i), ky = 0.13089969389957472f * (float)v;   // 2 pi / 48
    return expf(-0.5f * sigma * sigma * (kx * kx + ky * ky));
}

// (-1)^(u+v) of fft cell (v, i)
GD_HD float centre_sign(int v, int i) { return ((v + i) & 1) ? -1.0f : 1.0f; }

// exp(-2 pi i t) for a phase of t turns: t is reduced to [-1/2, 1/2] first, so the transcendental sees at most pi
GD_HD float2 expi_turns(float t) {
    t -= rintf(t);
    float s, c;
#ifdef __CUDA_ARCH__
    sincospif(2.0f * t, &s, &c);
#else
    const double a = 6.283185307179586 * (double)t;
    s = (float)sin(a);
    c = (float)cos(a);
#endif
    return make_float2(c, -s);
}

// I~(q) at q = 2 pi (fx, fy) / 48 of a stamp img [48][48] (16-byte aligned rows).  Order: each row's cells are added in four
// running sums over columns c = 4m + l (l = 0..3, m ascending), combined as (l0 + l1) + (l2 + l3); the row sums are added in row
// order.  The 48 column factors are formed once per target.
GD_HD float2 dtft(const float* __restrict__ img, float fx, float fy) {
    const float ax = fx * (1.0f / STAMP), ay = fy * (1.0f / STAMP);
    float cx[STAMP], sx[STAMP];                  // exp(-i qx X) = cx + i sx
#pragma unroll
    for (int c = 0; c < STAMP; ++c) {
        const float2 w = expi_turns(ax * (float)(c - HALF));
        cx[c] = w.x;
        sx[c] = w.y;
    }
    float re = 0.0f, im = 0.0f;
#pragma unroll 1
    for (int r = 0; r < STAMP; ++r) {
        const float4* row = reinterpret_cast<const float4*>(img + r * STAMP);
        float a[4] = {0.f, 0.f, 0.f, 0.f}, b[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int m = 0; m < STAMP / 4; ++m) {
            const float4 q = row[m];
            a[0] = fmaf(q.x, cx[4 * m], a[0]);     b[0] = fmaf(q.x, sx[4 * m], b[0]);
            a[1] = fmaf(q.y, cx[4 * m + 1], a[1]); b[1] = fmaf(q.y, sx[4 * m + 1], b[1]);
            a[2] = fmaf(q.z, cx[4 * m + 2], a[2]); b[2] = fmaf(q.z, sx[4 * m + 2], b[2]);
            a[3] = fmaf(q.w, cx[4 * m + 3], a[3]); b[3] = fmaf(q.w, sx[4 * m + 3], b[3]);
        }
        const float tr = (a[0] + a[1]) + (a[2] + a[3]), ti = (b[0] + b[1]) + (b[2] + b[3]);
        const float2 w = expi_turns(ay * (float)(r - HALF));                       // exp(-i qy Y)
        re = fmaf(tr, w.x, fmaf(-ti, w.y, re));
        im = fmaf(tr, w.y, fmaf(ti, w.x, im));
    }
    return make_float2(re, im);
}

// G~ / P for a PSF whose centred spectrum at the sheared frequency is pt and whose sum (its spectrum at 0) is p0
GD_HD float2 psf_factor(float2 pt, float p0, float gam) {
    const float px = pt.x / p0, py = pt.y / p0;
    const float h = px * px + py * py;
    if (h < PSF_FLOOR) return make_float2(0.0f, 0.0f);
    const float s = gam / h;
    return make_float2(px * s, -py * s);
}

// the plane value M_j (-1)^(u+v) of a cell: it = I~ (centred), f = G~ / P, sgn = centre_sign
GD_HD float2 cell_value(float2 it, float2 f, float sgn) {
    return make_float2(sgn * (it.x * f.x - it.y * f.y), sgn * (it.x * f.y + it.y * f.x));
}
// the same without a PSF (f = G~)
GD_HD float2 cell_value(float2 it, float gam, float sgn) { return make_float2(sgn * (it.x * gam), sgn * (it.y * gam)); }

// ---- FFT passes over one plane (fft_core.cuh's Fft48, one 48-point transform per call) ----

// forward column pass, c = 0..23: columns c and c + 24 of img [48][48] packed as one complex column, transformed, and split by
// Hermitian symmetry into rows v = 0..23 of the half spectrum (fft columns c and c + 24), as k_fpfs's column pass
GD_HD void fwd_col(const float* img, int c, float2* plane) {
    float2 v[STAMP];
#pragma unroll
    for (int n = 0; n < STAMP; ++n) v[n] = make_float2(img[n * STAMP + c], img[n * STAMP + c + HALF]);
    Fft48::run(v);
#pragma unroll
    for (int k = 0; k < HALF; ++k) {                 // W = A + iB: A(k) = (W(k) + conj W(-k)) / 2, B(k) = -i (W(k) - conj W(-k)) / 2
        const float2 p = v[Fft48::reg(k)], q = v[Fft48::reg((STAMP - k) % STAMP)];
        plane[k * PROW + c] = make_float2(0.5f * (p.x + q.x), 0.5f * (p.y - q.y));
        plane[k * PROW + c + HALF] = make_float2(0.5f * (p.y + q.y), 0.5f * (q.x - p.x));
    }
}

// forward row pass, v = 0..23, in place: the row's 48-point transform in fft column order
GD_HD void fwd_row(float2* plane, int v) {
    float2 x[STAMP];
    float4* row = reinterpret_cast<float4*>(plane + v * PROW);
#pragma unroll
    for (int c = 0; c < HALF; ++c) { const float4 q = row[c]; x[2 * c] = make_float2(q.x, q.y); x[2 * c + 1] = make_float2(q.z, q.w); }
    Fft48::run(x);
#pragma unroll
    for (int c = 0; c < HALF; ++c) {
        const float2 p = x[Fft48::reg(2 * c)], q = x[Fft48::reg(2 * c + 1)];
        row[c] = make_float4(p.x, p.y, q.x, q.y);
    }
}

// inverse row pass, v = 0..23, in place: the unscaled inverse transform along u of row v, with the Nyquist column 0 and, in row
// 0, the cells u < 0 the conjugates of u > 0 (only the half-plane targets were written)
GD_HD void inv_row(float2* plane, int v) {
    float2 x[STAMP];
    float4* row = reinterpret_cast<float4*>(plane + v * PROW);
#pragma unroll
    for (int c = 0; c < HALF; ++c) { const float4 q = row[c]; x[2 * c] = make_float2(q.x, -q.y); x[2 * c + 1] = make_float2(q.z, -q.w); }
    x[HALF] = make_float2(0.0f, 0.0f);
    if (v == 0) {
#pragma unroll
        for (int i = HALF + 1; i < STAMP; ++i) x[i] = make_float2(x[STAMP - i].x, -x[STAMP - i].y);
    }
    Fft48::run(x);                                   // idft(X) = conj(dft(conj X))
#pragma unroll
    for (int c = 0; c < HALF; ++c) {
        const float2 p = x[Fft48::reg(2 * c)], q = x[Fft48::reg(2 * c + 1)];
        row[c] = make_float4(p.x, -p.y, q.x, -q.y);
    }
}

// inverse column pass, c = 0..23, load and transform: rows v = 0..23 of the row-transformed plane at columns c and c + 24,
// packed as A + iB and extended to v = 24..47 by Hermitian symmetry (the Nyquist row is 0); on return x[Fft48::reg(r)] holds
// 2304 x pixel r of column c in its real part and -2304 x pixel r of column c + 24 in its imaginary part
GD_HD void inv_col(const float2* plane, int c, float2 (&x)[STAMP]) {
#pragma unroll
    for (int k = 0; k < HALF; ++k) {
        const float2 a = plane[k * PROW + c], b = plane[k * PROW + c + HALF];
        x[k] = make_float2(a.x - b.y, -(a.y + b.x));                               // conj(A + iB): idft = conj dft conj
        if (k) x[STAMP - k] = make_float2(a.x + b.y, a.y - b.x);                  // conj(conj A + i conj B)
    }
    x[HALF] = make_float2(0.0f, 0.0f);
    Fft48::run(x);
}
// inverse column pass, store: pixels of columns c and c + 24 of the real image img [48][48], scaled by 1/2304
GD_HD void inv_col_store(const float2 (&x)[STAMP], int c, float* img) {
    constexpr float S = 1.0f / NPIX;
#pragma unroll
    for (int r = 0; r < STAMP; ++r) {
        const float2 p = x[Fft48::reg(r)];
        img[r * STAMP + c] = p.x * S;
        img[r * STAMP + c + HALF] = -p.y * S;
    }
}

// ---- fix-noise ----
constexpr int FIXNOISE_STREAM = 60;              // streams 60 / 61

// pixel p of the generated fix-noise field of stamp idx: sigma N(idx, p); a non-finite sigma gives NaN (the stamp fails)
GD_HD float fixnoise_pixel(uint64_t idx, int p, uint64_t seed, float sigma) {
    return isfinite(sigma) ? gdsyn::fmul(sigma, gdsyn::hashed_normal(idx, p, seed, FIXNOISE_STREAM)) : NAN;
}

// the opposite shear j' of shear j: 1p <-> 1m, 2p <-> 2m, noshear itself
GD_HD int opposite(int j) { return j ? ((j & 1) ? j + 1 : j - 1) : 0; }

// the target whose factor is F_j(R^-1 k) for the target cell (v, u), R^-1 (u, v) = (v, -u): for u <= 0 the cell (v, -u) itself;
// for u > 0 it lies in the lower half plane and the target is its mirror (-v, u), whose factor is conjugated
struct RotTarget { int t; bool conj; };
GD_HD RotTarget rotated_target(int v, int u) {
    if (u <= 0) return {u == 0 ? v : HALF + (-u - 1) * (STAMP - 1) + v, false};
    return {HALF + (u - 1) * (STAMP - 1) + (v ? STAMP - 1 - v : 0), true};
}

// exp(i (kx + qy)), q = A_j R^-1 k, of the cell (v, u)
GD_HD float2 rotation_phase(int j, float delta, int u, int v) {
    const float2 q = sheared_freq(j, delta, v, -u);
    return expi_turns(-((float)u + q.y) * (1.0f / STAMP));
}

// the fix-noise term of target t of plane j: sgn exp(i (kx + qy)) n~(A_j' k) F_j(R^-1 k), with nt = n~(A_j' k) (centred);
// factor: the PSF's table [5][1105], or NULL (no PSF: F_j(R^-1 k) = G~(k))
GD_HD float2 fixnoise_value(int j, int t, float delta, float sigma, float2 nt, const float2* factor) {
    const Cell k = target(t);
    const int u = fftfreq(k.i);
    const float sgn = centre_sign(k.v, k.i);
    if (j) nt = gdfft::cmul(nt, rotation_phase(j, delta, u, k.v));
    if (!factor) return cell_value(nt, reconv(k.v, k.i, sigma), sgn);
    const RotTarget r = rotated_target(k.v, u);
    float2 f = factor[j * NTARGET + r.t];
    if (r.conj) f.y = -f.y;
    return cell_value(nt, f, sgn);
}

}  // namespace gdmetacal
