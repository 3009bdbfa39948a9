// k_fpfs: FPFS shear estimation of 48x48 stamps (the estimator of fpfs_core.cuh) on the register-resident transforms of
// k_wiener48 (Fft48, fft_core.cuh).  Per pass over FP_G stamps:
//   P0  column pass: one thread = columns c and c+24 of the stamp (or of its PSF) packed as ONE complex column, read straight
//       from global memory, 48-point FFT in registers, split by Hermitian symmetry into rows k1 = 0..24 of the half spectrum
//   P1  PSF row pass (only with a PSF): one thread = row k1 of one PSF: FFT, |p~|^2 written back over the row; row 0 also
//       records p~(0) (the PSF's sum)
//   P2  stamp row pass: one thread = row k1 of one stamp: FFT, D = |I~|^2 (x |p~(0)|^2 / |p~|^2), the six weighted sums of the
//       row (gdfpfs::row_sums, kx factors from a per-CTA table) -> shared memory
//   fin one thread per stamp adds its 25 row sums in row order and forms the modes, e1, e2 and R (gdfpfs::finish).
// Each stamp's arithmetic is the same whichever slot, pass or CTA it lands in, so its result does not depend on its batch.
// With no PSF only the stamp is transformed and P1 is skipped.
#include "fft_core.cuh"
#include "fpfs_core.cuh"
#include "kernels.cuh"
#include "launch.cuh"
#include "umma_ptx.cuh"

namespace gd {

using gdfft::Fft48;
using gdfpfs::Axis;
using gdfpfs::ROWS;

constexpr int FP_G = 5;                           // stamps per CTA pass: 25 rows x 5 = 125 row items on 128 threads
constexpr int FP_THREADS = 128;
constexpr int FP_ROW = 50;                        // float2 per spectrum row, as k_wiener48 (16-byte rows, conflict-free)
constexpr int FP_PLANE = ROWS * FP_ROW;
static_assert(gdfpfs::STAMP == STAMP, "stamp size");

static size_t fpfs_smem(int planes) {
    return (size_t)FP_G * planes * FP_PLANE * sizeof(float2) + STAMP * sizeof(Axis) + (size_t)FP_G * ROWS * sizeof(gdfpfs::Sums) +
           FP_G * sizeof(float2);
}

__global__ void __launch_bounds__(FP_THREADS, 2) k_fpfs(const float* __restrict__ img, const float* __restrict__ psf, int psf_batch,
                                                        int batch, float sigma, float cnst, float* __restrict__ modes,
                                                        float* __restrict__ ell) {
    const int planes = psf ? 2 : 1;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    float2* buf = reinterpret_cast<float2*>(smem_raw);                                    // [G][planes][25][FP_ROW]
    Axis* xs = reinterpret_cast<Axis*>(buf + FP_G * planes * FP_PLANE);                    // kx factors by fft column
    gdfpfs::Sums* rs = reinterpret_cast<gdfpfs::Sums*>(xs + STAMP);                         // [G][25] row sums
    float2* p0 = reinterpret_cast<float2*>(rs + FP_G * ROWS);                              // [G] (p~(0), |p~(0)|^2)
    if (threadIdx.x < STAMP) xs[threadIdx.x] = gdfpfs::axis(threadIdx.x, sigma);
    const bool pf_img = ((uintptr_t)img & 15) == 0, pf_psf = psf && psf_batch > 1 && ((uintptr_t)psf & 15) == 0;
    for (int g0 = blockIdx.x * FP_G; g0 < batch; g0 += gridDim.x * FP_G) {
        const int ng = min(FP_G, batch - g0);
        {   // the next pass's stamps on their way into L2 while this pass computes
            const int gn = g0 + gridDim.x * FP_G;
            if (threadIdx.x < 2 && gn < batch && (threadIdx.x ? pf_psf : pf_img)) {
                const int nn = min(FP_G, batch - gn);
                bulk_prefetch_l2((threadIdx.x ? psf : img) + (size_t)gn * NPIX, (uint32_t)(nn * NPIX * sizeof(float)));
            }
        }
        // Three passes of (load 48 values, FFT, consume) through ONE inlined copy of the transform, as in k_wiener48.
#pragma unroll 1
        for (int pass = 0; pass < 3; ++pass) {
            if (pass == 1 && !psf) continue;                 // uniform over the CTA
            const int per = pass == 0 ? 24 * planes : ROWS;
#pragma unroll 1
            for (int it = threadIdx.x; it < ng * per; it += FP_THREADS) {
                const int s = it / per, j = it - s * per;
                float2* gplane = buf + (s * planes) * FP_PLANE;
                float2* pplane = gplane + FP_PLANE;           // only with a PSF
                float2 v[48];
                if (pass == 0) {
                    const int im = j / 24, c = j - im * 24;
                    const float* src = im ? psf + (size_t)(psf_batch == 1 ? 0 : g0 + s) * NPIX + c : img + (size_t)(g0 + s) * NPIX + c;
#pragma unroll
                    for (int n = 0; n < 48; ++n) v[n] = make_float2(src[n * 48], src[n * 48 + 24]);
                } else {
                    const float4* row = reinterpret_cast<const float4*>((pass == 1 ? pplane : gplane) + j * FP_ROW);
#pragma unroll
                    for (int c = 0; c < 24; ++c) { const float4 q = row[c]; v[2 * c] = make_float2(q.x, q.y); v[2 * c + 1] = make_float2(q.z, q.w); }
                }
                Fft48::run(v);
                if (pass == 0) {
                    const int im = j / 24, c = j - im * 24;
                    float2* plane = gplane + im * FP_PLANE + c;
#pragma unroll
                    for (int k = 0; k < ROWS; ++k) {                          // W = A + iB, A and B real columns: A(k) = (W(k) + conj W(-k)) / 2
                        const float2 p = v[Fft48::reg(k)], q = v[Fft48::reg((48 - k) % 48)];
                        plane[k * FP_ROW] = make_float2(0.5f * (p.x + q.x), 0.5f * (p.y - q.y));
                        plane[k * FP_ROW + 24] = make_float2(0.5f * (p.y + q.y), 0.5f * (q.x - p.x));  // B(k) = -i (W(k) - conj W(-k)) / 2
                    }
                } else if (pass == 1) {
                    float4* hrow = reinterpret_cast<float4*>(pplane + j * FP_ROW);          // |p~|^2 of columns 0..47 as floats
#pragma unroll
                    for (int u = 0; u < 48; u += 4) {
                        float h[4];
#pragma unroll
                        for (int e = 0; e < 4; ++e) { const float2 p = v[Fft48::reg(u + e)]; h[e] = p.x * p.x + p.y * p.y; }
                        hrow[u / 4] = make_float4(h[0], h[1], h[2], h[3]);
                    }
                    if (j == 0) { const float2 p = v[Fft48::reg(0)]; p0[s] = make_float2(p.x, p.x * p.x + p.y * p.y); }
                } else {
                    const Axis y = gdfpfs::axis(j, sigma);
                    gdfpfs::Sums r;
                    if (psf) {
                        const float* hrow = reinterpret_cast<const float*>(pplane + j * FP_ROW);
                        const float h0 = p0[s].y;
                        r = gdfpfs::row_sums(j, y, xs, [&](int u) {
                            const float2 p = v[Fft48::reg(u)];
                            return (p.x * p.x + p.y * p.y) * gdfpfs::psf_factor(hrow[u], h0);
                        });
                    } else {
                        r = gdfpfs::row_sums(j, y, xs, [&](int u) { const float2 p = v[Fft48::reg(u)]; return p.x * p.x + p.y * p.y; });
                    }
                    rs[s * ROWS + j] = r;
                }
            }
            __syncthreads();
        }
        if (threadIdx.x < ng) {
            const int s = threadIdx.x;
            const size_t o = (size_t)(g0 + s);
            gdfpfs::finish(rs + s * ROWS, sigma, cnst, !psf || p0[s].x > 0.0f, modes ? modes + o * gdfpfs::NMODES : nullptr,
                           ell + o * gdfpfs::NELL);
        }
        // fin needs no barrier of its own: the next pass writes p0 (P1) and rs (P2) only after P0's barrier
    }
}

int fpfs_init() {
    GD_CUDA_CHECK(cudaFuncSetAttribute(k_fpfs, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fpfs_smem(2)));
    return GD_OK;
}

int launch_fpfs(const float* img, const float* psf, int psf_batch, int batch, float sigma, float cnst, float* modes, float* ell,
                cudaStream_t st) {
    if (batch <= 0) return GD_OK;
    const int planes = psf ? 2 : 1;
    static int grid_cap[3] = {0, 0, 0};                // resident CTAs on the device, by planes
    if (!grid_cap[planes]) {
        int dev, sms, per_sm;
        GD_CUDA_CHECK(cudaGetDevice(&dev));
        GD_CUDA_CHECK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
        GD_CUDA_CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_fpfs, FP_THREADS, fpfs_smem(planes)));
        grid_cap[planes] = sms * (per_sm > 0 ? per_sm : 1);
    }
    const int groups = (batch + FP_G - 1) / FP_G;
    k_fpfs<<<groups < grid_cap[planes] ? groups : grid_cap[planes], FP_THREADS, fpfs_smem(planes), st>>>(img, psf, psf_batch, batch, sigma,
                                                                                                      cnst, modes, ell);
    GD_LAUNCHED();
    return GD_OK;
}

}  // namespace gd
