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
// k_metacal (metacal.cu) and the host test tests/cpu/test_metacal_core.cpp run this code.
#pragma once
#include <cuda_runtime.h>
#include <math.h>
#include "fft_core.cuh"

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

}  // namespace gdmetacal
