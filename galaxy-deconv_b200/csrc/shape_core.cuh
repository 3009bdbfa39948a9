// Adaptive second moments of a 48x48 stamp (Bernstein & Jarvis 2002; Hirata & Seljak 2003), __host__ __device__.
//
// The weight is an elliptical Gaussian w = exp(-rho^2/2), rho^2 = (Myy dx^2 - 2 Mxy dx dy + Mxx dy^2) / det(M) around
// (x0, y0), iterated until (x0, y0, M) reproduce the weighted centroid and twice the weighted central second moments of the
// image.  Pixel p = 48 r + c sits at x = c, y = r (the coordinates of k_moments).  Start: (24, 24), M = s^2 I.  One pass:
//   A = sum v, Bx = sum v dx, By = sum v dy, Cxx = sum v dx^2, Cxy = sum v dx dy, Cyy = sum v dy^2   with v = I w
//   !(A > 0) -> FLUX (NaN pixels land here);  mx = Bx/A, my = By/A, M' = 2 (C/A - m m^T), x0' = x0 + mx, y0' = y0 + my
//   M' not positive definite or tr M' > 2 * 24^2 (a weight wider than the stamp) -> MOMENTS;  |x0' - 24| or |y0' - 24| > 15
//   -> CENTROID;  converged when max|m| <= TOL sqrt(t) and max|M' - M| <= TOL t, t = tr M' / 2;  then (x0, y0, M) <- (x0', y0', M')
// and a converged pass stops with OK.  No convergence in MAX_PASSES passes -> MAXITER.  On OK the outputs are flux = 2A of the
// last pass (exact for an elliptical Gaussian: at the fixed point sum I w = F/2), x0, y0, Mxx, Mxy, Myy and the distortion
// e1 = (Mxx - Myy)/(Mxx + Myy), e2 = 2 Mxy/(Mxx + Myy); on any other status all eight are NaN.
//
// k_adaptive_moments (shape.cu) and the host test tests/cpu/test_shape_core.cpp run this code; they differ only in how the
// per-pixel contributions are summed.
#pragma once
#include <cuda_runtime.h>
#include <math.h>

#ifndef GD_HD
#define GD_HD __host__ __device__ __forceinline__
#endif

namespace gdshape {

constexpr int STAMP = 48;
constexpr float START = 24.0f;        // the pixel PSFs and galaxies are centred on
constexpr int MAX_PASSES = 100;
constexpr float TOL = 1e-5f;
constexpr float MAX_TRACE = 1152.0f;  // 2 * 24^2
constexpr float MAX_SHIFT = 15.0f;
constexpr float HALF_LOG2E = 0.7213475204444817f;   // log2(e) / 2

enum Status { OK = 0, MAXITER = 1, FLUX = 2, MOMENTS = 3, CENTROID = 4, RUNNING = -1 };

struct Weight { float x0, y0, mxx, mxy, myy; };
struct Sums { float a, bx, by, cxx, cxy, cyy; };
// exp(-rho^2 / 2) = exp2(qxx dx^2 + qxy dx dy + qyy dy^2): the quadratic form and -log2(e)/2 folded into three coefficients
struct Quad { float qxx, qxy, qyy; };

GD_HD Quad weight_quad(const Weight& w) {
    const float s = -HALF_LOG2E / (w.mxx * w.myy - w.mxy * w.mxy);
    return {s * w.myy, -2.0f * s * w.mxy, s * w.mxx};
}

// the six contributions of one pixel.  Written dy-outer so that, with dx fixed for a run of pixels, qxy dx and qxx dx^2 are
// common subexpressions and the exponent costs two FMAs per pixel.
GD_HD void add_pixel(Sums& s, const Quad& q, float dx, float dy, float img) {
    const float v = img * exp2f((q.qyy * dy + q.qxy * dx) * dy + q.qxx * dx * dx);
    const float vx = v * dx, vy = v * dy;
    s.a += v;
    s.bx += vx;
    s.by += vy;
    s.cxx += vx * dx;
    s.cxy += vx * dy;
    s.cyy += vy * dy;
}

// one pass's update from its six sums: RUNNING, or the status the stamp stops with (w is updated on RUNNING and OK)
GD_HD int step(Weight& w, const Sums& s) {
    if (!(s.a > 0.0f)) return FLUX;
    const float ia = 1.0f / s.a;
    const float mx = s.bx * ia, my = s.by * ia;
    const float mxx = 2.0f * (s.cxx * ia - mx * mx);
    const float mxy = 2.0f * (s.cxy * ia - mx * my);
    const float myy = 2.0f * (s.cyy * ia - my * my);
    if (!(mxx > 0.0f && myy > 0.0f && mxx * myy - mxy * mxy > 0.0f) || mxx + myy > MAX_TRACE) return MOMENTS;
    const float x0 = w.x0 + mx, y0 = w.y0 + my;
    if (fabsf(x0 - START) > MAX_SHIFT || fabsf(y0 - START) > MAX_SHIFT) return CENTROID;
    const float t = 0.5f * (mxx + myy);
    const bool done = fmaxf(fabsf(mx), fabsf(my)) <= TOL * sqrtf(t) &&
                      fmaxf(fmaxf(fabsf(mxx - w.mxx), fabsf(mxy - w.mxy)), fabsf(myy - w.myy)) <= TOL * t;
    w = {x0, y0, mxx, mxy, myy};
    return done ? OK : RUNNING;
}

// The whole iteration.  sums(w, q) returns the six sums of one pass with weight w (coefficients q).  Writes the eight output
// floats (flux, x0, y0, Mxx, Mxy, Myy, e1, e2) and the number of passes made; returns the status.
template <class SumFn> GD_HD int measure(float guess_sigma, const SumFn& sums, float* out, int* passes) {
    Weight w = {START, START, guess_sigma * guess_sigma, 0.0f, guess_sigma * guess_sigma};
    int status = RUNNING, n = 0;
    float a = 0.0f;
    while (status == RUNNING && n < MAX_PASSES) {
        const Sums s = sums(w, weight_quad(w));
        a = s.a;
        status = step(w, s);
        ++n;
    }
    *passes = n;
    if (status == RUNNING) status = MAXITER;
    if (status != OK) {
        for (int i = 0; i < 8; ++i) out[i] = NAN;
        return status;
    }
    const float tr = w.mxx + w.myy;
    out[0] = 2.0f * a;
    out[1] = w.x0;
    out[2] = w.y0;
    out[3] = w.mxx;
    out[4] = w.mxy;
    out[5] = w.myy;
    out[6] = (w.mxx - w.myy) / tr;
    out[7] = 2.0f * w.mxy / tr;
    return status;
}

}  // namespace gdshape
