// Per-stamp shared-memory FFT kernels: everything in the hot path that the reference does with torch.fft.
//   path G  (models/unrolled_admm_gaussian.py): k_g_prologue (:118-123 + init_l2 :111-115), k_g_xupdate
//           (XUpdateGaussian :89-93 fused with the dual update :145 and the denoiser-input scaling of :142)
//   path U  (models/Unrolled_ADMM.py): k_u_prologue (:181-196 + init_l2 :170-175), k_u_pre (V-update :207,
//           denoiser input :208), k_u_post (X-update :209 -> effective :315-319, duals :212-213)
//   solvers (models/Richard_Lucy.py:10-24, models/Wiener.py:10-20, models/Tikhonet.py:15-31)
// One CTA owns one stamp; the stamp, its spectrum and the PSF spectrum never leave shared memory inside a kernel.
//
// Index conventions (see fft_core.cuh): spectra are half spectra S[s1][k2], k2 natural in [0, N/2], s1 the
// digit-swapped slot of frequency k1 = freq(s1).  The reference's pad_double + ifftshift (path G) and
// psf_to_otf == roll(N/2) (path U / solvers) are pure phase factors on the spectrum of the image placed at the
// corner of the grid:  shift by 72 on a 96 grid -> (+i)^(k1+k2), shift by 24 on a 48 grid -> (-1)^(k1+k2).
#include <math.h>
#include "fft_block.cuh"
#include "launch.cuh"
#include "umma_ptx.cuh"

#include <cstdlib>
#include <mutex>
#include <vector>

namespace gd {

// =====================================================================================================
// Path G
// =====================================================================================================
using FG96 = Real2D<96, 8, 12, 48>;
constexpr int SPG = 50;
constexpr int G_THREADS = 256;
constexpr size_t G_SMEM_PRO = (size_t)(24 * 96 + 2 * 96 * SPG + 96) * sizeof(float2) + 64;
constexpr size_t G_SMEM_XUP = (size_t)(24 * 96 + 96 * SPG + 96) * sizeof(float2) + 64;

// y, psf -> Pc = (-i)^(k1+k2) conj(Hc) Yc, HtH = |Hc|^2 (workspace), z0 = init_l2, u = 0
__global__ void __launch_bounds__(G_THREADS) k_g_prologue(const float* __restrict__ y, const float* __restrict__ psf,
                                                          const float* __restrict__ alpha, float2* __restrict__ Pc,
                                                          float* __restrict__ HtH, float* __restrict__ z,
                                                          float* __restrict__ u, float* __restrict__ x) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float2* Z = reinterpret_cast<float2*>(smem_raw);
    float2* SY = Z + 24 * 96;
    float2* SH = SY + 96 * SPG;
    float2* tw = SH + 96 * SPG;
    const int b = blockIdx.x;
    const float* yb = y + (size_t)b * NPIX;
    const float* kb = psf + (size_t)b * NPIX;
    fill_twiddles<96>(tw);
    for (int i = threadIdx.x; i < 24 * 48; i += blockDim.x) {
        int j = i / 48, c = i - j * 48;
        Z[j * 96 + c] = make_float2(fmaxf(yb[(2 * j) * 48 + c], 0.f), fmaxf(yb[(2 * j + 1) * 48 + c], 0.f));   // :118
    }
    fwd2d<FG96, SPG>(Z, SY, tw);
    for (int i = threadIdx.x; i < 24 * 48; i += blockDim.x) {
        int j = i / 48, c = i - j * 48;
        Z[j * 96 + c] = make_float2(kb[(2 * j) * 48 + c], kb[(2 * j + 1) * 48 + c]);
    }
    fwd2d<FG96, SPG>(Z, SH, tw);
    const float ia = 1.0f / alpha[b];
    float2* Pb = Pc + (size_t)b * FG_SPEC;
    float* Hb = HtH + (size_t)b * FG_SPEC;
    for (int q = threadIdx.x; q < FG_SPEC; q += blockDim.x) {
        int s1 = q / FG_NH, k2 = q - s1 * FG_NH;
        float2 h = SH[s1 * SPG + k2], yy = SY[s1 * SPG + k2];
        float2 p = mul_negi_pow(cmul(cconj(h), yy), FG96::L::freq(s1) + k2);
        float hh = h.x * h.x + h.y * h.y;
        Pb[q] = p;
        Hb[q] = hh;
        float d = 1.0f / (hh + ia);                                                                           // :112-113
        SY[s1 * SPG + k2] = make_float2(p.x * d, p.y * d);
    }
    inv2d<FG96, SPG>(SY, Z, tw);
    const float sc = 1.0f / (96.f * 96.f);
    for (int i = threadIdx.x; i < NPIX; i += blockDim.x) {
        int r = i / 48, c = i - r * 48;
        z[(size_t)b * NPIX + i] = zpix<96>(Z, r, c) * sc;
        u[(size_t)b * NPIX + i] = 0.f;                                                                        // :130
        x[(size_t)b * NPIX + i] = 0.f;
    }
}

// iteration `it`:  u <- u + rho_{it-1} (x_prev - z)   (it > 0; the dual update of the previous iteration, :145)
//                  x <- crop(ifft((Pc + F(rho z - u)) / (rho + HtH)))                                    (:89-93)
//                  t <- (rho x + u) * 2^-e, tscale = 2^e                                   (denoiser input, :142)
__global__ void __launch_bounds__(G_THREADS) k_g_xupdate(const float2* __restrict__ Pc, const float* __restrict__ HtH,
                                                         const float* __restrict__ rho, int n_rho, int it,
                                                         const float* __restrict__ z, float* __restrict__ x,
                                                         float* __restrict__ u, float* __restrict__ t,
                                                         float* __restrict__ tscale) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float2* Z = reinterpret_cast<float2*>(smem_raw);
    float2* S = Z + 24 * 96;
    float2* tw = S + 96 * SPG;
    float* red = reinterpret_cast<float*>(tw + 96);
    const int b = blockIdx.x;
    const size_t o = (size_t)b * NPIX;
    const float r_now = rho[(size_t)b * n_rho + it];
    const float r_prev = it > 0 ? rho[(size_t)b * n_rho + it - 1] : 0.f;
    fill_twiddles<96>(tw);
    constexpr int PER = NPIX / G_THREADS;      // 9
    float ureg[PER];
#pragma unroll
    for (int e = 0; e < PER; ++e) {
        int i = threadIdx.x + e * G_THREADS;
        int r = i / 48, c = i - r * 48;
        float zz = z[o + i], uu = u[o + i];
        if (it > 0) uu = uu + r_prev * (x[o + i] - zz);
        ureg[e] = uu;
        zpix<96>(Z, r, c) = r_now * zz - uu;
    }
    fwd2d<FG96, SPG>(Z, S, tw);
    const float2* Pb = Pc + (size_t)b * FG_SPEC;
    const float* Hb = HtH + (size_t)b * FG_SPEC;
    for (int q = threadIdx.x; q < FG_SPEC; q += blockDim.x) {
        int s1 = q / FG_NH, k2 = q - s1 * FG_NH;
        float2 v = S[s1 * SPG + k2], p = Pb[q];
        float d = 1.0f / (r_now + Hb[q]);
        S[s1 * SPG + k2] = make_float2((p.x + v.x) * d, (p.y + v.y) * d);
    }
    inv2d<FG96, SPG>(S, Z, tw);
    const float sc = 1.0f / (96.f * 96.f);
    float tv[PER], amax = 0.f;
#pragma unroll
    for (int e = 0; e < PER; ++e) {
        int i = threadIdx.x + e * G_THREADS;
        int r = i / 48, c = i - r * 48;
        float xx = zpix<96>(Z, r, c) * sc;
        x[o + i] = xx;
        u[o + i] = ureg[e];
        tv[e] = r_now * xx + ureg[e];
        amax = fmaxf(amax, fabsf(tv[e]));
    }
    amax = block_max(amax, red);
    float inv;
    float s = pow2_scale(amax, &inv);
    if (threadIdx.x == 0) tscale[b] = s;
#pragma unroll
    for (int e = 0; e < PER; ++e) t[o + threadIdx.x + e * G_THREADS] = tv[e] * inv;
}

// analysis=True bookkeeping (:147-152): u_i = u + rho_i (x_i - z_i) written to the analysis buffer
__global__ void k_g_dual_out(const float* __restrict__ rho, int n_rho, int it, const float* __restrict__ x,
                             const float* __restrict__ z, const float* __restrict__ u, float* __restrict__ uo, int n) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    int b = i / NPIX;
    uo[i] = u[i] + rho[(size_t)b * n_rho + it] * (x[i] - z[i]);
}

// plain scaling of an arbitrary single-channel stamp batch for gd_resunet_forward
__global__ void __launch_bounds__(G_THREADS) k_scale_in(const float* __restrict__ in, float* __restrict__ t,
                                                        float* __restrict__ tscale) {
    __shared__ float red[G_THREADS / 32];
    const size_t o = (size_t)blockIdx.x * NPIX;
    float v[NPIX / G_THREADS], amax = 0.f;
#pragma unroll
    for (int e = 0; e < NPIX / G_THREADS; ++e) { v[e] = in[o + threadIdx.x + e * G_THREADS]; amax = fmaxf(amax, fabsf(v[e])); }
    amax = block_max(amax, red);
    float inv;
    float s = pow2_scale(amax, &inv);
    if (threadIdx.x == 0) tscale[blockIdx.x] = s;
#pragma unroll
    for (int e = 0; e < NPIX / G_THREADS; ++e) t[o + threadIdx.x + e * G_THREADS] = v[e] * inv;
}

__global__ void k_fill_rho(const float* __restrict__ src, int n_rho, float* __restrict__ rho, int batch) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < batch * n_rho) rho[i] = src[i % n_rho];
}

// =====================================================================================================
// 48x48 circular transforms: path U and the classical solvers
// =====================================================================================================
using FU48 = Real2D<48, 4, 12, 48>;
constexpr int SPU = 26;
constexpr int U_THREADS = 128;
constexpr int U_PER = NPIX / U_THREADS;        // 18
constexpr int ZU = 24 * 48;                    // float2 per packed stamp
constexpr int SU = 48 * SPU;                   // float2 per spectrum buffer

__device__ __forceinline__ void load_packed48(float2* Z, const float* __restrict__ src, float mul, bool clamp) {
    for (int i = threadIdx.x; i < ZU; i += blockDim.x) {
        int j = i / 48, c = i - j * 48;
        float a = src[(2 * j) * 48 + c], bb = src[(2 * j + 1) * 48 + c];
        if (clamp) { a = fmaxf(a, 0.f); bb = fmaxf(bb, 0.f); }
        Z[i] = make_float2(a * mul, bb * mul);
    }
}
__device__ __forceinline__ float sgn48(int s1, int k2) { return ((FU48::L::freq(s1) + k2) & 1) ? -1.f : 1.f; }

// H = fft2(roll(psf, 24, 24)) = (-1)^(k1+k2) Hc   (psf_to_otf, utils/utils_torch.py:79-92, same-size kernel)
__device__ __forceinline__ void otf48(const float* __restrict__ psf, float2* Z, float2* SH, const float2* tw) {
    load_packed48(Z, psf, 1.f, false);
    fwd2d<FU48, SPU>(Z, SH, tw);
    for (int q = threadIdx.x; q < FU_SPEC; q += blockDim.x) {
        int s1 = q / FU_NH, k2 = q - s1 * FU_NH;
        float sg = sgn48(s1, k2);
        float2 h = SH[s1 * SPU + k2];
        SH[s1 * SPU + k2] = make_float2(sg * h.x, sg * h.y);
    }
    __syncthreads();
}

// |L|^2 of the reference's 3x3 "Laplacian" pushed through psf_to_otf: the quadrant assignments broadcast and
// leave 7 non-zeros (SURVEY.md section 0.6):  (0,47)=(1,47)=(46,47)=(47,0)=(47,1)=(47,46)=1, (47,47)=-4.
__device__ __forceinline__ float lap_quirk_abs2(int k1, int k2, const float2* tw) {
    const int rr[7] = {0, 1, 46, 47, 47, 47, 47}, cc[7] = {47, 47, 47, 0, 1, 46, 47};
    const float vv[7] = {1.f, 1.f, 1.f, 1.f, 1.f, 1.f, -4.f};
    float re = 0.f, im = 0.f;
#pragma unroll
    for (int i = 0; i < 7; ++i) {
        float2 e = tw[(k1 * rr[i] + k2 * cc[i]) % 48];
        re += vv[i] * e.x; im += vv[i] * e.y;
    }
    return re * re + im * im;
}

constexpr size_t SOLVER_SMEM = (size_t)(ZU + 2 * SU + 48) * sizeof(float2) + (size_t)2 * NPIX * sizeof(float) + 64;
constexpr size_t SOLVER_SMEM_LIGHT = (size_t)(ZU + 2 * SU + 48) * sizeof(float2) + 64;   // Wiener / Tikhonov / conv_fft: no x, y copies -> 7 CTAs per SM

// kind: GD_SOLVER_* ; one CTA per stamp
__global__ void __launch_bounds__(U_THREADS) k_solver(int kind_flags, int n_iters, float lam, const float* __restrict__ y,
                                                      const float* __restrict__ psf, const float* __restrict__ alpha,
                                                      float* __restrict__ out) {
    const int kind = kind_flags & 0xff;
    const bool clamp_y = (kind_flags & 0x100) != 0;       // Tikhonet clamps y before its Tikhonov step (models/Tikhonet.py:43)
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float2* Z = reinterpret_cast<float2*>(smem_raw);
    float2* S = Z + ZU;
    float2* SH = S + SU;
    float2* tw = SH + SU;
    float* ys = reinterpret_cast<float*>(tw + 48);
    float* xs = ys + NPIX;
    const int b = blockIdx.x;
    const size_t o = (size_t)b * NPIX;
    fill_twiddles<48>(tw);
    __syncthreads();
    otf48(psf + o, Z, SH, tw);
    const float sc = 1.0f / (48.f * 48.f);
    if (kind == 0) {                                      // Richardson-Lucy, models/Richard_Lucy.py:10-24
        // conv_fft_batch(Ht, ones) = conj(H[0,0]) = sum(psf): loop-invariant (:22)
        const float div = SH[0].x;
        for (int i = threadIdx.x; i < NPIX; i += blockDim.x) { float v = fmaxf(y[o + i], 0.f); ys[i] = v; xs[i] = v; }
        __syncthreads();
        for (int it = 0; it < n_iters; ++it) {
            for (int i = threadIdx.x; i < ZU; i += blockDim.x) {
                int j = i / 48, c = i - j * 48;
                Z[i] = make_float2(xs[(2 * j) * 48 + c], xs[(2 * j + 1) * 48 + c]);
            }
            fwd2d<FU48, SPU>(Z, S, tw);
            for (int q = threadIdx.x; q < FU_SPEC; q += blockDim.x) {
                int idx = (q / FU_NH) * SPU + (q % FU_NH);
                S[idx] = cmul(S[idx], SH[idx]);
            }
            inv2d<FU48, SPU>(S, Z, tw);                    // Hx (unscaled)
            for (int i = threadIdx.x; i < ZU; i += blockDim.x) {
                int j = i / 48, c = i - j * 48;
                float2 hx = Z[i];
                Z[i] = make_float2(ys[(2 * j) * 48 + c] / (hx.x * sc), ys[(2 * j + 1) * 48 + c] / (hx.y * sc));   // :21
            }
            fwd2d<FU48, SPU>(Z, S, tw);
            for (int q = threadIdx.x; q < FU_SPEC; q += blockDim.x) {
                int idx = (q / FU_NH) * SPU + (q % FU_NH);
                S[idx] = cmul(S[idx], cconj(SH[idx]));
            }
            inv2d<FU48, SPU>(S, Z, tw);                    // num (unscaled)
            for (int i = threadIdx.x; i < ZU; i += blockDim.x) {
                int j = i / 48, c = i - j * 48;
                float2 nm = Z[i];
                int p0 = (2 * j) * 48 + c, p1 = p0 + 48;
                xs[p0] = xs[p0] * (nm.x * sc) / div;                                                        // :23
                xs[p1] = xs[p1] * (nm.y * sc) / div;
            }
            __syncthreads();
        }
        for (int i = threadIdx.x; i < NPIX; i += blockDim.x) out[o + i] = xs[i];
        return;
    }
    const float a = alpha[b];
    // Wiener: fftn(y) un-clamped, un-scaled (models/Wiener.py:16-18); Tikhonov: fftn(y/alpha) (models/Tikhonet.py:20)
    load_packed48(Z, y + o, kind == 1 ? 1.f : 1.0f / a, clamp_y);
    fwd2d<FU48, SPU>(Z, S, tw);
    for (int q = threadIdx.x; q < FU_SPEC; q += blockDim.x) {
        int s1 = q / FU_NH, k2 = q - s1 * FU_NH, idx = s1 * SPU + k2;
        float2 h = SH[idx];
        float hh = h.x * h.x + h.y * h.y;
        float div = kind == 1 ? hh + 350.f / a
                  : kind == 2 ? hh + lam
                              : hh + lam * lap_quirk_abs2(FU48::L::freq(s1), k2, tw);
        float2 n = cmul(cconj(h), S[idx]);
        S[idx] = make_float2(n.x / div, n.y / div);
    }
    inv2d<FU48, SPU>(S, Z, tw);
    for (int i = threadIdx.x; i < NPIX; i += blockDim.x) {
        int r = i / 48, c = i - r * 48;
        out[o + i] = zpix<48>(Z, r, c) * sc;
    }
}

// ---------------------------------------------------------------------------------------------------------------------------
// Wiener / Tikhonov with every 48-point transform in the REGISTERS of one thread (Fft48, fft_core.cuh): the phase-structured
// k_solver moves each element through shared memory ~15 times per stamp (5 phases per 2-D transform, 39 % of the wavefronts
// bank-conflict replays, 76 % of the shared-memory pipe) and spends 2.8 instructions per flop on index arithmetic
// (profiles/solver_r02.md).  Here a 2-D real transform is
//   P1   column pass: one thread = columns c and c+24 of y (or of psf) packed as ONE complex column, read straight from global
//        memory (coalesced), 48-point FFT in registers, split by Hermitian symmetry, rows k1 = 0..24 of the half spectrum -> smem
//   P23  row pass: one thread = row k1 of one stamp: FFT of the psf row, FFT of the y row, the pointwise solve
//        conj(H) Y / (|H|^2 + reg) (models/Wiener.py:16-19, models/Tikhonet.py:20-31), and the inverse row FFT
//   P4   inverse column pass: one thread = output columns n2 and n2+24 as one complex column (rows 25..47 by Hermitian symmetry),
//        stored straight to global memory (coalesced).
// Three shared-memory exchanges per stamp, all conflict-free (row stride 49 float2), no index arithmetic inside the transforms.
constexpr int W48_G = 5;                          // stamps per CTA pass: 25 rows x 5 = 125 row items on 128 threads
constexpr int W48_THREADS = 128;
constexpr int W48_ROW = 50;                       // float2 per spectrum row (48 + 2 pad): rows 16-byte aligned for 128-bit accesses,
                                                  // 100 words = 4 mod 32 keeps the 8 threads of a 128-bit wavefront on distinct banks
constexpr int W48_PLANE = 25 * W48_ROW;           // rows k1 = 0..24
constexpr size_t W48_SMEM = (size_t)W48_G * 2 * W48_PLANE * sizeof(float2) + (size_t)W48_PLANE * sizeof(float);

__global__ void __launch_bounds__(W48_THREADS, 2) k_wiener48(int kind_flags, float lam, const float* __restrict__ y,
                                                             const float* __restrict__ psf, const float* __restrict__ alpha,
                                                             float* __restrict__ out, int batch, const float* __restrict__ lap_abs2) {
    const int kind = kind_flags & 0xff;
    const bool clamp_y = (kind_flags & 0x100) != 0;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float2* buf = reinterpret_cast<float2*>(smem_raw);                  // [G][2][25][49]: plane 0 = y, plane 1 = psf
    float* lapS = reinterpret_cast<float*>(buf + W48_G * 2 * W48_PLANE);    // [25][49] |L|^2 of the Laplacian filter (kind 3)
    if (kind == 3)
        for (int i = threadIdx.x; i < 25 * 48; i += W48_THREADS) lapS[(i / 48) * W48_ROW + i % 48] = lap_abs2[i];
    for (int g0 = blockIdx.x * W48_G; g0 < batch; g0 += gridDim.x * W48_G) {
        const int ng = min(W48_G, batch - g0);
        {   // the next pass's stamps on their way into L2 while this pass computes (pass 0 reads them with plain loads)
            const int gn = g0 + gridDim.x * W48_G;
            if (threadIdx.x < 2 && gn < batch) {
                const int nn = min(W48_G, batch - gn);
                bulk_prefetch_l2((threadIdx.x ? psf : y) + (size_t)gn * NPIX, (uint32_t)(nn * NPIX * sizeof(float)));
            }
        }
        // Five passes of (load 48 values, FFT, store) through ONE inlined copy of the transform: with a copy per pass the kernel
        // is ~90 KB of straight-line code and stalls on instruction fetch more than on anything else (measured: 'no_instruction'
        // 1.09 warps per issue).  Pass 0 = P1, passes 1-3 = P23 (psf row, y row + solve, inverse row), pass 4 = P4.
#pragma unroll 1
        for (int pass = 0; pass < 5; ++pass) {
            const int per = pass == 0 ? 48 : pass == 4 ? 24 : 25;
#pragma unroll 1
            for (int it = threadIdx.x; it < ng * per; it += W48_THREADS) {
                const int s = it / per, j = it - s * per;
                float2* yplane = buf + (s * 2) * W48_PLANE;
                float2 v[48];
                if (pass == 0) {
                    const int im = j / 24, c = j - im * 24;
                    const float* src = (im ? psf : y) + (size_t)(g0 + s) * NPIX + c;
                    float mul = 1.f;
                    if (!im && kind != 1) mul = 1.0f / alpha[g0 + s];   // Tikhonov transforms y / alpha (Tikhonet.py:20), Wiener y itself
                    const bool cl = !im && clamp_y;
#pragma unroll
                    for (int n = 0; n < 48; ++n) {
                        float a = src[n * 48], b = src[n * 48 + 24];
                        if (cl) { a = fmaxf(a, 0.f); b = fmaxf(b, 0.f); }
                        v[n] = make_float2(a * mul, b * mul);
                    }
                } else if (pass < 4) {
                    const float4* row = reinterpret_cast<const float4*>(yplane + (pass == 1 ? W48_PLANE : 0) + j * W48_ROW);
#pragma unroll
                    for (int c = 0; c < 24; ++c) { const float4 q = row[c]; v[2 * c] = make_float2(q.x, q.y); v[2 * c + 1] = make_float2(q.z, q.w); }
                } else {
                    const float2* G = yplane + j;
#pragma unroll
                    for (int k1 = 0; k1 <= 24; ++k1) {                            // conj(Ga + i Gb)
                        const float2 ga = G[k1 * W48_ROW], gb = G[k1 * W48_ROW + 24];
                        v[k1] = make_float2(ga.x - gb.y, -(ga.y + gb.x));
                        if (k1 > 0 && k1 < 24) v[48 - k1] = make_float2(ga.x + gb.y, -(gb.x - ga.y));   // rows 48 - k1: conj(conj Ga + i conj Gb)
                    }
                }
                Fft48::run(v);
                if (pass == 0) {
                    const int im = j / 24, c = j - im * 24;
                    float2* plane = yplane + im * W48_PLANE + c;
#pragma unroll
                    for (int k = 0; k <= 24; ++k) {                           // W = A + iB, A and B real columns: A(k) = (W(k) + conj W(-k)) / 2
                        const float2 p = v[Fft48::reg(k)], q = v[Fft48::reg((48 - k) % 48)];
                        plane[k * W48_ROW] = make_float2(0.5f * (p.x + q.x), 0.5f * (p.y - q.y));
                        plane[k * W48_ROW + 24] = make_float2(0.5f * (p.y + q.y), 0.5f * (q.x - p.x));  // B(k) = -i (W(k) - conj W(-k)) / 2
                    }
                } else if (pass == 1) {
                    float4* hrow = reinterpret_cast<float4*>(yplane + W48_PLANE + j * W48_ROW);
#pragma unroll
                    for (int k2 = 0; k2 < 48; k2 += 2) {
                        const float2 p = v[Fft48::reg(k2)], q = v[Fft48::reg(k2 + 1)];
                        hrow[k2 / 2] = make_float4(p.x, p.y, q.x, q.y);
                    }
                } else if (pass == 2) {
                    float4* yrow = reinterpret_cast<float4*>(yplane + j * W48_ROW);
                    const float4* hrow = reinterpret_cast<const float4*>(yplane + W48_PLANE + j * W48_ROW);
                    const float a = alpha[g0 + s];
                    const float reg0 = kind == 1 ? 350.f / a : lam;
                    const float sg1 = (j & 1) ? -1.f : 1.f;                       // H = (-1)^(k1+k2) Hc (psf_to_otf's roll by 24, 24)
#pragma unroll
                    for (int k2 = 0; k2 < 48; k2 += 2) {
                        const float4 hq = hrow[k2 / 2];
                        float o[4];
#pragma unroll
                        for (int e = 0; e < 2; ++e) {
                            const float2 h = e ? make_float2(hq.z, hq.w) : make_float2(hq.x, hq.y), yy = v[Fft48::reg(k2 + e)];
                            const float hh = h.x * h.x + h.y * h.y;
                            const float div = kind == 3 ? hh + lam * lapS[j * W48_ROW + k2 + e] : hh + reg0;
                            const float2 n = cmul(cconj(h), yy);
                            const float f = (e ? -sg1 : sg1) / div;                  // k2 + e is odd exactly for e = 1
                            o[2 * e] = n.x * f; o[2 * e + 1] = -n.y * f;              // conj(X): inverse = conj(dft(conj X))
                        }
                        yrow[k2 / 2] = make_float4(o[0], o[1], o[2], o[3]);
                    }
                } else if (pass == 3) {
                    float4* yrow = reinterpret_cast<float4*>(yplane + j * W48_ROW);
#pragma unroll
                    for (int n2 = 0; n2 < 48; n2 += 2) {
                        const float2 p = v[Fft48::reg(n2)], q = v[Fft48::reg(n2 + 1)];
                        yrow[n2 / 2] = make_float4(p.x, -p.y, q.x, -q.y);
                    }
                } else {
                    float* dst = out + (size_t)(g0 + s) * NPIX + j;
                    const float sc = 1.0f / (48.f * 48.f);
#pragma unroll
                    for (int n1 = 0; n1 < 48; ++n1) {
                        const float2 g = v[Fft48::reg(n1)];
                        dst[n1 * 48] = g.x * sc;
                        dst[n1 * 48 + 24] = -g.y * sc;
                    }
                }
            }
            if (pass == 0 || pass >= 3) __syncthreads();          // passes 1-3 stay in one thread's own rows
        }
    }
}

// Richardson-Lucy (models/Richard_Lucy.py:10-24) on the same register-resident transforms: per iteration
//   Hx = irfft2(rfft2(x) H),  num = irfft2(rfft2(y / Hx) conj H),  x <- x num / div,   div = conj(H[0,0]) (:22, loop-invariant)
// With five stamps per CTA pass every thread owns ONE column item (columns c, c+24 of one stamp: 120 items) and ONE row item (row k1
// of one stamp's half spectrum: 125 items) for the whole loop, so an inverse column transform, the pointwise step in image space
// (y / Hx, or the x update) and the next forward column transform chain in one thread's registers, and so do a forward row
// transform, the multiplication by H or conj H and the inverse row transform.  Four barriers and 196 transforms per iteration;
// x lives in `out` (L2-resident between iterations), y is re-read from global memory, the planes are those of k_wiener48.
// The loop below runs ONE inlined copy of the transform; `kind` selects what happens before and after it.
__global__ void __launch_bounds__(W48_THREADS, 2) k_rl48(int n_iters, const float* __restrict__ y, const float* __restrict__ psf,
                                                         float* __restrict__ out, int batch) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float2* buf = reinterpret_cast<float2*>(smem_raw);                  // [G][2][25][ROW]: plane 0 = work, plane 1 = H (sign folded in)
    float* divS = reinterpret_cast<float*>(buf + W48_G * 2 * W48_PLANE);
    const int tid = threadIdx.x;
    const int sc_ = tid / 24, cc = tid - sc_ * 24;                      // column item
    const int sr = tid / 25, jr = tid - sr * 25;                        // row item
    const float sc = 1.0f / (48.f * 48.f);
    const int nsteps = n_iters > 0 ? 2 + 8 * n_iters : 3;               // 3 prologue steps + 8 per iteration - the last iteration's split
    for (int g0 = blockIdx.x * W48_G; g0 < batch; g0 += gridDim.x * W48_G) {
        const int ng = min(W48_G, batch - g0);
        const bool colv = tid < ng * 24, rowv = tid < ng * 25;
        float2* cplane = buf + (sc_ * 2) * W48_PLANE + cc;               // this thread's two columns of the work plane
        float2* wrow = buf + (sr * 2) * W48_PLANE + jr * W48_ROW;        // this thread's row of the work plane
        float2* hrow = wrow + W48_PLANE;
        const size_t co = colv ? (size_t)(g0 + sc_) * NPIX + cc : 0;
        float2 v[48];
        __syncthreads();                          // the previous pass is done with the planes
#pragma unroll 1
        for (int t = 0; t < nsteps; ++t) {
            const int kind = t < 3 ? t : 3 + ((t - 3) & 7);
            // kinds: 0 psf columns -> H plane | 1 H rows | 2 y columns -> work plane | 3 / 7 row: forward, times H / conj H
            //        4 / 8 row: inverse -> work plane | 5 column: inverse -> Hx, y / Hx | 9 column: inverse -> num, x update
            //        6 / 10 column: forward -> work plane
            const bool is_col = kind == 0 || kind == 2 || kind == 5 || kind == 6 || kind == 9 || kind == 10;
            if (is_col ? colv : rowv) {
                if (kind == 0 || kind == 2) {
                    const float* src = (kind == 0 ? psf : y) + co;
#pragma unroll
                    for (int n = 0; n < 48; ++n) {
                        float a = src[n * 48], b = src[n * 48 + 24];
                        if (kind == 2) { a = fmaxf(a, 0.f); b = fmaxf(b, 0.f); out[co + n * 48] = a; out[co + n * 48 + 24] = b; }   // x0 = y (:17)
                        v[n] = make_float2(a, b);
                    }
                } else if (kind == 1 || kind == 3 || kind == 7) {
                    const float4* row = reinterpret_cast<const float4*>(kind == 1 ? hrow : wrow);
#pragma unroll
                    for (int c = 0; c < 24; ++c) { const float4 q = row[c]; v[2 * c] = make_float2(q.x, q.y); v[2 * c + 1] = make_float2(q.z, q.w); }
                } else if (kind == 5 || kind == 9) {
#pragma unroll
                    for (int k1 = 0; k1 <= 24; ++k1) {                            // conj(Ga + i Gb), rows 48 - k1 by Hermitian symmetry
                        const float2 ga = cplane[k1 * W48_ROW], gb = cplane[k1 * W48_ROW + 24];
                        v[k1] = make_float2(ga.x - gb.y, -(ga.y + gb.x));
                        if (k1 > 0 && k1 < 24) v[48 - k1] = make_float2(ga.x + gb.y, -(gb.x - ga.y));
                    }
                }
                Fft48::run(v);
                if (kind == 0 || kind == 2 || kind == 6 || kind == 10) {
                    float2* plane = kind == 0 ? cplane + W48_PLANE : cplane;
#pragma unroll
                    for (int k = 0; k <= 24; ++k) {                           // split the packed pair of real columns
                        const float2 p = v[Fft48::reg(k)], q = v[Fft48::reg((48 - k) % 48)];
                        plane[k * W48_ROW] = make_float2(0.5f * (p.x + q.x), 0.5f * (p.y - q.y));
                        plane[k * W48_ROW + 24] = make_float2(0.5f * (p.y + q.y), 0.5f * (q.x - p.x));
                    }
                } else if (kind == 1) {
                    const float sg1 = (jr & 1) ? -1.f : 1.f;                      // H = (-1)^(k1+k2) Hc (psf_to_otf's roll by 24, 24)
                    float4* hr = reinterpret_cast<float4*>(hrow);
#pragma unroll
                    for (int k2 = 0; k2 < 48; k2 += 2) {
                        const float2 p = v[Fft48::reg(k2)], q = v[Fft48::reg(k2 + 1)];
                        hr[k2 / 2] = make_float4(sg1 * p.x, sg1 * p.y, -sg1 * q.x, -sg1 * q.y);
                    }
                    if (jr == 0) divS[sr] = v[Fft48::reg(0)].x;                   // conv_fft_batch(Ht, ones) = conj(H[0,0]) = sum(psf)
                } else if (kind == 3 || kind == 7) {
                    const float cj = kind == 7 ? -1.f : 1.f;                      // times H (Hx) or conj H (numerator)
                    const float4* hr = reinterpret_cast<const float4*>(hrow);
                    float2 w[48];
#pragma unroll
                    for (int k2 = 0; k2 < 48; k2 += 2) {
                        const float4 hq = hr[k2 / 2];
                        const float2 x0 = cmul(v[Fft48::reg(k2)], make_float2(hq.x, cj * hq.y));
                        const float2 x1 = cmul(v[Fft48::reg(k2 + 1)], make_float2(hq.z, cj * hq.w));
                        w[k2] = make_float2(x0.x, -x0.y); w[k2 + 1] = make_float2(x1.x, -x1.y);        // conjugate: inverse = conj(dft(conj X))
                    }
#pragma unroll
                    for (int k2 = 0; k2 < 48; ++k2) v[k2] = w[k2];
                } else if (kind == 4 || kind == 8) {
                    float4* wr = reinterpret_cast<float4*>(wrow);
#pragma unroll
                    for (int n2 = 0; n2 < 48; n2 += 2) {
                        const float2 p = v[Fft48::reg(n2)], q = v[Fft48::reg(n2 + 1)];
                        wr[n2 / 2] = make_float4(p.x, -p.y, q.x, -q.y);
                    }
                } else if (kind == 5) {
                    float2 w[48];
#pragma unroll
                    for (int n1 = 0; n1 < 48; ++n1) {
                        const float2 g = v[Fft48::reg(n1)];                       // Hx of columns c, c + 24 (unscaled; second one negated)
                        const float ya = fmaxf(y[co + n1 * 48], 0.f), yb = fmaxf(y[co + n1 * 48 + 24], 0.f);
                        // :21.  __fdividef (reciprocal + multiply, 2 ulp): the IEEE division's special-case subroutine is taken for
                        // every clamped-to-zero pixel and cost more than the transforms (measured: 307 M slow-path calls per launch)
                        w[n1] = make_float2(__fdividef(ya, g.x * sc), __fdividef(yb, -g.y * sc));
                    }
#pragma unroll
                    for (int n1 = 0; n1 < 48; ++n1) v[n1] = w[n1];
                } else {                                                          // kind 9
                    const float rdiv = sc / divS[sc_];                            // 1 / (2304 div): one division per thread and iteration
                    float2 w[48];
#pragma unroll
                    for (int n1 = 0; n1 < 48; ++n1) {
                        const float2 g = v[Fft48::reg(n1)];
                        const float xa = out[co + n1 * 48] * (g.x * rdiv), xb = out[co + n1 * 48 + 24] * (-g.y * rdiv);     // :23
                        out[co + n1 * 48] = xa; out[co + n1 * 48 + 24] = xb;
                        w[n1] = make_float2(xa, xb);
                    }
#pragma unroll
                    for (int n1 = 0; n1 < 48; ++n1) v[n1] = w[n1];
                }
            }
            if (kind == 0 || kind == 1 || kind == 2 || kind == 4 || kind == 6 || kind == 8 || kind == 10) __syncthreads();
        }
    }
}

// conv_fft_batch(H or conj(H), x), utils/utils_torch.py:46-50
__global__ void __launch_bounds__(U_THREADS) k_conv_fft(const float* __restrict__ x, const float* __restrict__ psf,
                                                        float* __restrict__ out, int adjoint) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float2* Z = reinterpret_cast<float2*>(smem_raw);
    float2* S = Z + ZU;
    float2* SH = S + SU;
    float2* tw = SH + SU;
    const size_t o = (size_t)blockIdx.x * NPIX;
    fill_twiddles<48>(tw);
    __syncthreads();
    otf48(psf + o, Z, SH, tw);
    load_packed48(Z, x + o, 1.f, false);
    fwd2d<FU48, SPU>(Z, S, tw);
    for (int q = threadIdx.x; q < FU_SPEC; q += blockDim.x) {
        int idx = (q / FU_NH) * SPU + (q % FU_NH);
        S[idx] = cmul(S[idx], adjoint ? cconj(SH[idx]) : SH[idx]);
    }
    inv2d<FU48, SPU>(S, Z, tw);
    for (int i = threadIdx.x; i < NPIX; i += blockDim.x) {
        int r = i / 48, c = i - r * 48;
        out[o + i] = zpix<48>(Z, r, c) * (1.0f / 2304.f);
    }
}

// psf_to_otf(ker, size) with the reference's signature and semantics (utils/utils_torch.py:79-92) for size = (B,1,48,48):
// `psf` = zeros(size) with the four quadrant assignments (centre = (kh + 1) / 2 for BOTH axes, each source block broadcast
// to centre x centre the way torch broadcasts a size-1 dimension, later assignments overwriting earlier ones -- for a 3x3 kernel
// this leaves the 7-non-zero array of SURVEY.md section 0.6), `otf` = fft2(psf) as the FULL 48x48 complex spectrum.
// kb = 1: one kernel shared by the batch (the reference's broadcasting assignment), kb = batch: one kernel per stamp.
__global__ void __launch_bounds__(U_THREADS) k_psf_to_otf(const float* __restrict__ ker, int kb, int kh, int kw, float* __restrict__ psf_out,
                                                          float2* __restrict__ otf_out) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float2* Z = reinterpret_cast<float2*>(smem_raw);
    float2* S = Z + ZU;
    float2* tw = S + 2 * SU;
    const int b = blockIdx.x;
    const float* kp = ker + (kb == 1 ? 0 : (size_t)b * kh * kw);
    const int ce = (kh + 1) / 2;
    fill_twiddles<48>(tw);
    for (int i = threadIdx.x; i < NPIX; i += blockDim.x) {
        const int r = i / 48, c = i - r * 48;
        const bool top = r < ce, bot = r >= 48 - ce, left = c < ce, right = c >= 48 - ce;
        float v = 0.f;
        // source block (rows r0.., cols c0.., shape sh x sw) of the LAST assignment that covers (r, c)
        int r0 = -1, c0 = 0, sh = 0, sw = 0, ri = 0, ci = 0;
        if (bot && right) { r0 = 0; c0 = 0; sh = ce; sw = ce; ri = r - (48 - ce); ci = c - (48 - ce); }
        else if (bot && left) { r0 = 0; c0 = ce; sh = ce; sw = kw - ce; ri = r - (48 - ce); ci = c; }
        else if (top && right) { r0 = ce; c0 = 0; sh = kh - ce; sw = ce; ri = r; ci = c - (48 - ce); }
        else if (top && left) { r0 = ce; c0 = ce; sh = kh - ce; sw = kw - ce; ri = r; ci = c; }
        if (r0 >= 0) v = kp[(r0 + (sh == 1 ? 0 : ri)) * kw + c0 + (sw == 1 ? 0 : ci)];
        psf_out[(size_t)b * NPIX + i] = v;
        zpix<48>(Z, r, c) = v;
    }
    fwd2d<FU48, SPU>(Z, S, tw);
    float2* ob = otf_out + (size_t)b * NPIX;
    for (int q = threadIdx.x; q < FU_SPEC; q += blockDim.x) {
        const int s1 = q / FU_NH, k2 = q - s1 * FU_NH, k1 = FU48::L::freq(s1);
        const float2 h = S[s1 * SPU + k2];
        ob[k1 * 48 + k2] = h;
        if (k2 > 0 && k2 < 24) ob[((48 - k1) % 48) * 48 + (48 - k2)] = cconj(h);      // Hermitian half the transform does not store
    }
}

// conv_fft_batch(H, x) with the reference's signature (utils/utils_torch.py:46-50): ifft2(fft2(x) * H).real for a FULL
// complex spectrum H [B][48][48].  x is real, so the real part of the inverse transform only sees the Hermitian part of H,
// Hs(k) = (H(k) + conj(H(-k))) / 2, which is what the half-spectrum transform multiplies by (exact for any H).
__global__ void __launch_bounds__(U_THREADS) k_conv_otf(const float2* __restrict__ H, int hb, const float* __restrict__ x, float* __restrict__ out) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float2* Z = reinterpret_cast<float2*>(smem_raw);
    float2* S = Z + ZU;
    float2* tw = S + 2 * SU;
    const size_t o = (size_t)blockIdx.x * NPIX;
    const float2* Hb = H + (hb == 1 ? 0 : o);
    fill_twiddles<48>(tw);
    load_packed48(Z, x + o, 1.f, false);
    fwd2d<FU48, SPU>(Z, S, tw);
    for (int q = threadIdx.x; q < FU_SPEC; q += blockDim.x) {
        const int s1 = q / FU_NH, k2 = q - s1 * FU_NH, k1 = FU48::L::freq(s1);
        const float2 a = Hb[k1 * 48 + k2], bq = Hb[((48 - k1) % 48) * 48 + (48 - k2) % 48];
        const float2 hs = make_float2(0.5f * (a.x + bq.x), 0.5f * (a.y - bq.y));
        S[s1 * SPU + k2] = cmul(S[s1 * SPU + k2], hs);
    }
    inv2d<FU48, SPU>(S, Z, tw);
    for (int i = threadIdx.x; i < NPIX; i += blockDim.x) {
        int r = i / 48, c = i - r * 48;
        out[o + i] = zpix<48>(Z, r, c) * (1.0f / 2304.f);
    }
}

// ---------------------------------------------------------------------------------------------------
// Path U.  Per-stamp state in the workspace: H (half spectrum, with the (-1)^k sign), x, z(=denoiser out),
// v, u1, u2, Hx.  The reference's three conv_fft_batch calls per iteration (:207,:209,:213) collapse to
// 4 transforms (SURVEY.md section 7): Hx = F^-1(H X) is produced by the same kernel that produces x.
// ---------------------------------------------------------------------------------------------------
constexpr size_t U_SMEM = (size_t)(ZU + 2 * SU + 48) * sizeof(float2) + (size_t)NPIX * sizeof(float) + 64;

// y (clamped, :181), H, rho -> x0 = init_l2 (:170-175), z = x0, v = y or y/alpha, u1 = u2 = 0, Hx0 = conv(H, x0)
__global__ void __launch_bounds__(U_THREADS) k_u_prologue(const float* __restrict__ y, const float* __restrict__ psf,
                                                          const float* __restrict__ alpha, int v0_over_alpha,
                                                          float2* __restrict__ Hw, float* __restrict__ x,
                                                          float* __restrict__ z, float* __restrict__ v,
                                                          float* __restrict__ u1, float* __restrict__ u2,
                                                          float* __restrict__ Hx) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float2* Z = reinterpret_cast<float2*>(smem_raw);
    float2* S = Z + ZU;
    float2* SH = S + SU;
    float2* tw = SH + SU;
    const int b = blockIdx.x;
    const size_t o = (size_t)b * NPIX;
    const float a = alpha[b], ia = 1.0f / a;
    const float sc = 1.0f / 2304.f;
    fill_twiddles<48>(tw);
    __syncthreads();
    otf48(psf + o, Z, SH, tw);
    float2* Hb = Hw + (size_t)b * FU_SPEC;
    for (int q = threadIdx.x; q < FU_SPEC; q += blockDim.x) Hb[q] = SH[(q / FU_NH) * SPU + (q % FU_NH)];
    // init_l2: rhs = fftn(conv_fft_batch(Ht, y/alpha)); the inner conv's ".real" is a no-op on a real signal up to
    // rounding, so rhs = conj(H) F(y/alpha) without the spatial round trip.
    load_packed48(Z, y + o, ia, true);
    fwd2d<FU48, SPU>(Z, S, tw);
    for (int q = threadIdx.x; q < FU_SPEC; q += blockDim.x) {
        int idx = (q / FU_NH) * SPU + (q % FU_NH);
        float2 h = SH[idx];
        float d = 1.0f / (h.x * h.x + h.y * h.y + ia);
        float2 n = cmul(cconj(h), S[idx]);
        S[idx] = make_float2(n.x * d, n.y * d);
    }
    inv2d<FU48, SPU>(S, Z, tw);
    for (int i = threadIdx.x; i < ZU; i += blockDim.x) {
        int j = i / 48, c = i - j * 48;
        float2 q = Z[i];
        q.x = fminf(fmaxf(q.x * sc, 0.f), 1.f);                                                               // :175
        q.y = fminf(fmaxf(q.y * sc, 0.f), 1.f);
        Z[i] = q;
        int p0 = (2 * j) * 48 + c, p1 = p0 + 48;
        x[o + p0] = q.x; x[o + p1] = q.y;
        z[o + p0] = q.x; z[o + p1] = q.y;                                                                     // :193
        float y0 = fmaxf(y[o + p0], 0.f), y1 = fmaxf(y[o + p1], 0.f);
        v[o + p0] = v0_over_alpha ? y0 * ia : y0;                                                             // :194 / :416
        v[o + p1] = v0_over_alpha ? y1 * ia : y1;
        u1[o + p0] = 0.f; u1[o + p1] = 0.f; u2[o + p0] = 0.f; u2[o + p1] = 0.f;
    }
    fwd2d<FU48, SPU>(Z, S, tw);
    for (int q = threadIdx.x; q < FU_SPEC; q += blockDim.x) {
        int idx = (q / FU_NH) * SPU + (q % FU_NH);
        S[idx] = cmul(S[idx], SH[idx]);
    }
    inv2d<FU48, SPU>(S, Z, tw);
    for (int i = threadIdx.x; i < NPIX; i += blockDim.x) {
        int r = i / 48, c = i - r * 48;
        Hx[o + i] = zpix<48>(Z, r, c) * sc;
    }
}

// elementwise: V-update (:207 with :322-328 / :335-336) and the scaled denoiser input x + u1 (:208)
__global__ void __launch_bounds__(G_THREADS) k_u_pre(int llh, const float* __restrict__ y, const float* __restrict__ alpha,
                                                     const float* __restrict__ rho, int n_rho, int n, int it,
                                                     const float* __restrict__ x, const float* __restrict__ u1,
                                                     const float* __restrict__ u2, const float* __restrict__ Hx,
                                                     float* __restrict__ v, float* __restrict__ t,
                                                     float* __restrict__ tscale) {
    __shared__ float red[G_THREADS / 32];
    const int b = blockIdx.x;
    const size_t o = (size_t)b * NPIX;
    const float a = alpha[b], rho2 = rho[(size_t)b * n_rho + n + it];
    float tv[NPIX / G_THREADS], amax = 0.f;
#pragma unroll
    for (int e = 0; e < NPIX / G_THREADS; ++e) {
        size_t i = o + threadIdx.x + e * G_THREADS;
        float yy = fmaxf(y[i], 0.f);
        float vt = Hx[i] + u2[i];
        float vv;
        if (llh == 1) {
            float t1 = rho2 * vt - a;
            vv = 0.5f * (1.0f / rho2) * (-t1 + sqrtf(t1 * t1 + 4.f * yy * rho2));
        } else {
            vv = (rho2 * vt + yy / a) / (1.f + rho2);
        }
        v[i] = vv;
        tv[e] = x[i] + u1[i];
        amax = fmaxf(amax, fabsf(tv[e]));
    }
    float inv = 1.f;
    if (tscale) {          // tscale == nullptr: unscaled denoiser input (XDenseUNet has BatchNorm shifts and biases: not homogeneous)
        amax = block_max(amax, red);
        float s = pow2_scale(amax, &inv);
        if (threadIdx.x == 0) tscale[b] = s;
    }
#pragma unroll
    for (int e = 0; e < NPIX / G_THREADS; ++e) t[o + threadIdx.x + e * G_THREADS] = tv[e] * inv;
}

// X-update (:315-319 effective), duals (:212-213); z is the denoiser output of this iteration
__global__ void __launch_bounds__(U_THREADS) k_u_post(const float2* __restrict__ Hw, const float* __restrict__ rho,
                                                      int n_rho, int n, int it, const float* __restrict__ z,
                                                      const float* __restrict__ v, float* __restrict__ x,
                                                      float* __restrict__ u1, float* __restrict__ u2,
                                                      float* __restrict__ Hx) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float2* Z = reinterpret_cast<float2*>(smem_raw);
    float2* S = Z + ZU;
    float2* SB = S + SU;
    float2* tw = SB + SU;
    const int b = blockIdx.x;
    const size_t o = (size_t)b * NPIX;
    const float rho1 = rho[(size_t)b * n_rho + it], rho2 = rho[(size_t)b * n_rho + n + it];
    const float sc = 1.0f / 2304.f;
    const float2* Hb = Hw + (size_t)b * FU_SPEC;
    fill_twiddles<48>(tw);
    // A = F(z - u1)
    for (int i = threadIdx.x; i < ZU; i += blockDim.x) {
        int j = i / 48, c = i - j * 48;
        size_t p0 = o + (2 * j) * 48 + c, p1 = p0 + 48;
        Z[i] = make_float2(z[p0] - u1[p0], z[p1] - u1[p1]);
    }
    fwd2d<FU48, SPU>(Z, S, tw);
    // B = F(v - u2)
    for (int i = threadIdx.x; i < ZU; i += blockDim.x) {
        int j = i / 48, c = i - j * 48;
        size_t p0 = o + (2 * j) * 48 + c, p1 = p0 + 48;
        Z[i] = make_float2(v[p0] - u2[p0], v[p1] - u2[p1]);
    }
    fwd2d<FU48, SPU>(Z, SB, tw);
    // X = (rho1 A + rho2 conj(H) B) / (rho1 |H|^2 + rho2);  S <- X, SB <- H X
    for (int q = threadIdx.x; q < FU_SPEC; q += blockDim.x) {
        int idx = (q / FU_NH) * SPU + (q % FU_NH);
        float2 h = Hb[q], A = S[idx], Bq = cmul(cconj(h), SB[idx]);
        float d = 1.0f / (rho1 * (h.x * h.x + h.y * h.y) + rho2);
        float2 X = make_float2((rho1 * A.x + rho2 * Bq.x) * d, (rho1 * A.y + rho2 * Bq.y) * d);
        S[idx] = X;
        SB[idx] = cmul(h, X);
    }
    inv2d<FU48, SPU>(S, Z, tw);
    for (int i = threadIdx.x; i < ZU; i += blockDim.x) {
        int j = i / 48, c = i - j * 48;
        size_t p0 = o + (2 * j) * 48 + c, p1 = p0 + 48;
        float x0 = Z[i].x * sc, x1 = Z[i].y * sc;
        x[p0] = x0; x[p1] = x1;
        u1[p0] = u1[p0] + x0 - z[p0];
        u1[p1] = u1[p1] + x1 - z[p1];
    }
    inv2d<FU48, SPU>(SB, Z, tw);
    for (int i = threadIdx.x; i < ZU; i += blockDim.x) {
        int j = i / 48, c = i - j * 48;
        size_t p0 = o + (2 * j) * 48 + c, p1 = p0 + 48;
        float h0 = Z[i].x * sc, h1 = Z[i].y * sc;
        Hx[p0] = h0; Hx[p1] = h1;
        u2[p0] = u2[p0] + h0 - v[p0];
        u2[p1] = u2[p1] + h1 - v[p1];
    }
}

__global__ void k_scale_by_alpha(float* __restrict__ out, const float* __restrict__ x, const float* __restrict__ alpha,
                                 int n, int use_alpha) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = use_alpha ? x[i] * alpha[i / NPIX] : x[i];
}

// ---------------------------------------------------------------------------------------------------
// moment ellipticities (utils/fit_ellipse.py:370-399 normalize_images, :467-548 compute_moments,
// utils/utils_test.py:92-96): one warp-group per stamp
// ---------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(U_THREADS) k_moments(const float* __restrict__ img, float* __restrict__ e12) {
    __shared__ float red[U_THREADS / 32];
    const size_t o = (size_t)blockIdx.x * NPIX;
    float v[U_PER], mn = INFINITY, mx = -INFINITY;
#pragma unroll
    for (int e = 0; e < U_PER; ++e) { v[e] = img[o + threadIdx.x + e * U_THREADS]; mn = fminf(mn, v[e]); mx = fmaxf(mx, v[e]); }
    mx = block_max(mx, red);
    mn = -block_max(-mn, red);
    const float dv = fmaxf(mx - mn, 1e-8f);
    float m00 = 0.f, sx = 0.f, sy = 0.f;
#pragma unroll
    for (int e = 0; e < U_PER; ++e) {
        int i = threadIdx.x + e * U_THREADS;
        float g = (v[e] - mn) / dv;
        v[e] = g;
        m00 += g; sx += g * (float)(i % 48); sy += g * (float)(i / 48);
    }
    m00 = block_sum(m00, red) + 1e-8f;
    const float cx = block_sum(sx, red) / m00, cy = block_sum(sy, red) / m00;
    float a20 = 0.f, a11 = 0.f, a02 = 0.f;
#pragma unroll
    for (int e = 0; e < U_PER; ++e) {
        int i = threadIdx.x + e * U_THREADS;
        float dx = (float)(i % 48) - cx, dy = (float)(i / 48) - cy;
        a20 += v[e] * dx * dx; a11 += v[e] * dx * dy; a02 += v[e] * dy * dy;
    }
    const float mu20 = block_sum(a20, red) / m00, mu11 = block_sum(a11, red) / m00, mu02 = block_sum(a02, red) / m00;
    if (threadIdx.x == 0) {
        e12[2 * blockIdx.x] = (mu20 - mu02) / (mu20 + mu02);
        e12[2 * blockIdx.x + 1] = 2.f * mu11 / (mu20 + mu02);
    }
}

// =====================================================================================================
// host launchers
// =====================================================================================================
template <class K> static int opt_in_smem(K kernel, size_t bytes) {
    GD_CUDA_CHECK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
    return GD_OK;
}

int fft_kernels_init() {
    int rc;
    if ((rc = opt_in_smem(k_g_prologue, G_SMEM_PRO))) return rc;
    if ((rc = opt_in_smem(k_g_xupdate, G_SMEM_XUP))) return rc;
    if ((rc = opt_in_smem(k_solver, SOLVER_SMEM))) return rc;
    if ((rc = opt_in_smem(k_wiener48, W48_SMEM))) return rc;
    if ((rc = opt_in_smem(k_rl48, W48_SMEM))) return rc;
    if ((rc = opt_in_smem(k_conv_fft, SOLVER_SMEM))) return rc;
    if ((rc = opt_in_smem(k_psf_to_otf, SOLVER_SMEM_LIGHT))) return rc;
    if ((rc = opt_in_smem(k_conv_otf, SOLVER_SMEM_LIGHT))) return rc;
    if ((rc = opt_in_smem(k_u_prologue, U_SMEM))) return rc;
    if ((rc = opt_in_smem(k_u_post, U_SMEM))) return rc;
    return GD_OK;
}

int launch_g_prologue(const float* y, const float* psf, const float* alpha, float2* Pc, float* HtH, float* z, float* u,
                      float* x, int batch, cudaStream_t st) {
    if (batch <= 0) return GD_OK;
    k_g_prologue<<<batch, G_THREADS, G_SMEM_PRO, st>>>(y, psf, alpha, Pc, HtH, z, u, x);
    GD_LAUNCHED();
    return GD_OK;
}
int launch_g_xupdate(const float2* Pc, const float* HtH, const float* rho, int n_rho, int it, const float* z, float* x,
                     float* u, float* t, float* tscale, int batch, cudaStream_t st) {
    if (batch <= 0) return GD_OK;
    k_g_xupdate<<<batch, G_THREADS, G_SMEM_XUP, st>>>(Pc, HtH, rho, n_rho, it, z, x, u, t, tscale);
    GD_LAUNCHED();
    return GD_OK;
}
int launch_g_dual_out(const float* rho, int n_rho, int it, const float* x, const float* z, const float* u, float* uo,
                      int batch, cudaStream_t st) {
    int n = batch * NPIX;
    if (n <= 0) return GD_OK;
    k_g_dual_out<<<(n + 255) / 256, 256, 0, st>>>(rho, n_rho, it, x, z, u, uo, n);
    GD_LAUNCHED();
    return GD_OK;
}
int launch_scale_in(const float* in, float* t, float* tscale, int batch, cudaStream_t st) {
    if (batch <= 0) return GD_OK;
    k_scale_in<<<batch, G_THREADS, 0, st>>>(in, t, tscale);
    GD_LAUNCHED();
    return GD_OK;
}
int launch_fill_rho(const float* src, int n_rho, float* rho, int batch, cudaStream_t st) {
    int n = batch * n_rho;
    if (n <= 0) return GD_OK;
    k_fill_rho<<<(n + 255) / 256, 256, 0, st>>>(src, n_rho, rho, batch);
    GD_LAUNCHED();
    return GD_OK;
}
// |L|^2 of the reference's Laplacian filter on the half spectrum k1 in [0, 25), k2 in [0, 48) (lap_quirk_abs2 above, in double)
static float* g_lap_abs2[16] = {nullptr};
static int lap_table(float** out) {
    int dev;
    GD_CUDA_CHECK(cudaGetDevice(&dev));
    if (dev < 0 || dev >= 16) { set_error("lap_table: device %d out of range", dev); return GD_ECUDA; }
    static std::mutex mu;
    std::lock_guard<std::mutex> lk(mu);
    if (!g_lap_abs2[dev]) {
        const int rr[7] = {0, 1, 46, 47, 47, 47, 47}, cc[7] = {47, 47, 47, 0, 1, 46, 47};
        const double vv[7] = {1, 1, 1, 1, 1, 1, -4};
        std::vector<float> h(25 * 48);
        for (int k1 = 0; k1 < 25; ++k1)
            for (int k2 = 0; k2 < 48; ++k2) {
                double re = 0, im = 0;
                for (int i = 0; i < 7; ++i) {
                    const double ph = -2.0 * 3.14159265358979323846 * ((k1 * rr[i] + k2 * cc[i]) % 48) / 48.0;
                    re += vv[i] * cos(ph); im += vv[i] * sin(ph);
                }
                h[k1 * 48 + k2] = (float)(re * re + im * im);
            }
        GD_CUDA_CHECK(cudaMalloc(&g_lap_abs2[dev], h.size() * sizeof(float)));
        GD_CUDA_CHECK(cudaMemcpy(g_lap_abs2[dev], h.data(), h.size() * sizeof(float), cudaMemcpyHostToDevice));
    }
    *out = g_lap_abs2[dev];
    return GD_OK;
}

// GDECONV_SOLVER48=0 restores the phase-structured k_solver for all classical solvers
static int solver48_mode() {
    static int m = -1;
    if (m < 0) { const char* e = getenv("GDECONV_SOLVER48"); m = e ? atoi(e) : 1; }
    return m;
}

int launch_solver(int kind, int n_iters, float lam, const float* y, const float* psf, const float* alpha, float* out,
                  int batch, cudaStream_t st) {
    if (batch <= 0) return GD_OK;
    if (solver48_mode()) {
        static int sms0 = 0;
        if (!sms0) {
            int dev;
            GD_CUDA_CHECK(cudaGetDevice(&dev));
            GD_CUDA_CHECK(cudaDeviceGetAttribute(&sms0, cudaDevAttrMultiProcessorCount, dev));
        }
        const int groups0 = (batch + W48_G - 1) / W48_G;
        if ((kind & 0xff) == 0) {
            k_rl48<<<groups0 < 2 * sms0 ? groups0 : 2 * sms0, W48_THREADS, W48_SMEM, st>>>(n_iters, y, psf, out, batch);
            GD_LAUNCHED();
            return GD_OK;
        }
    }
    if ((kind & 0xff) != 0 && solver48_mode()) {
        float* lap = nullptr;
        if ((kind & 0xff) == 3) { int rc = lap_table(&lap); if (rc != GD_OK) return rc; }
        static int sms = 0;
        if (!sms) {
            int dev;
            GD_CUDA_CHECK(cudaGetDevice(&dev));
            GD_CUDA_CHECK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
        }
        const int groups = (batch + W48_G - 1) / W48_G;
        k_wiener48<<<groups < 2 * sms ? groups : 2 * sms, W48_THREADS, W48_SMEM, st>>>(kind, lam, y, psf, alpha, out, batch, lap);
        GD_LAUNCHED();
        return GD_OK;
    }
    k_solver<<<batch, U_THREADS, (kind & 0xff) == 0 ? SOLVER_SMEM : SOLVER_SMEM_LIGHT, st>>>(kind, n_iters, lam, y, psf, alpha, out);
    GD_LAUNCHED();
    return GD_OK;
}
int launch_conv_fft(const float* x, const float* psf, float* out, int adjoint, int batch, cudaStream_t st) {
    if (batch <= 0) return GD_OK;
    k_conv_fft<<<batch, U_THREADS, SOLVER_SMEM_LIGHT, st>>>(x, psf, out, adjoint);
    GD_LAUNCHED();
    return GD_OK;
}
int launch_psf_to_otf(const float* ker, int kb, int kh, int kw, float* psf_out, float2* otf_out, int batch, cudaStream_t st) {
    if (batch <= 0) return GD_OK;
    k_psf_to_otf<<<batch, U_THREADS, SOLVER_SMEM_LIGHT, st>>>(ker, kb, kh, kw, psf_out, otf_out);
    GD_LAUNCHED();
    return GD_OK;
}
int launch_conv_otf(const float2* H, int hb, const float* x, float* out, int batch, cudaStream_t st) {
    if (batch <= 0) return GD_OK;
    k_conv_otf<<<batch, U_THREADS, SOLVER_SMEM_LIGHT, st>>>(H, hb, x, out);
    GD_LAUNCHED();
    return GD_OK;
}
int launch_u_prologue(const float* y, const float* psf, const float* alpha, int v0_over_alpha, float2* Hw, float* x,
                      float* z, float* v, float* u1, float* u2, float* Hx, int batch, cudaStream_t st) {
    if (batch <= 0) return GD_OK;
    k_u_prologue<<<batch, U_THREADS, U_SMEM, st>>>(y, psf, alpha, v0_over_alpha, Hw, x, z, v, u1, u2, Hx);
    GD_LAUNCHED();
    return GD_OK;
}
int launch_u_pre(int llh, const float* y, const float* alpha, const float* rho, int n_rho, int n, int it, const float* x,
                 const float* u1, const float* u2, const float* Hx, float* v, float* t, float* tscale, int batch,
                 cudaStream_t st) {
    if (batch <= 0) return GD_OK;
    k_u_pre<<<batch, G_THREADS, 0, st>>>(llh, y, alpha, rho, n_rho, n, it, x, u1, u2, Hx, v, t, tscale);
    GD_LAUNCHED();
    return GD_OK;
}
int launch_u_post(const float2* Hw, const float* rho, int n_rho, int n, int it, const float* z, const float* v, float* x,
                  float* u1, float* u2, float* Hx, int batch, cudaStream_t st) {
    if (batch <= 0) return GD_OK;
    k_u_post<<<batch, U_THREADS, U_SMEM, st>>>(Hw, rho, n_rho, n, it, z, v, x, u1, u2, Hx);
    GD_LAUNCHED();
    return GD_OK;
}
int launch_scale_by_alpha(float* out, const float* x, const float* alpha, int batch, int use_alpha, cudaStream_t st) {
    int n = batch * NPIX;
    if (n <= 0) return GD_OK;
    k_scale_by_alpha<<<(n + 255) / 256, 256, 0, st>>>(out, x, alpha, n, use_alpha);
    GD_LAUNCHED();
    return GD_OK;
}
int launch_moments(const float* img, float* e12, int batch, cudaStream_t st) {
    if (batch <= 0) return GD_OK;
    k_moments<<<batch, U_THREADS, 0, st>>>(img, e12);
    GD_LAUNCHED();
    return GD_OK;
}

}  // namespace gd
