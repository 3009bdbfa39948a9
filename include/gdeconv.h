/* libgdeconv -- C ABI of the B200 (sm_100a) Galaxy-Deconv inference hot path.
 *
 * The reference (mbertagna/Galaxy-Deconv) has no FFI of its own: its boundary is the torch nn.Module surface
 * (SURVEY.md section 8b).  The Python modules under galaxy-deconv_b200/models/ keep that surface and bind the
 * entry points below with ctypes; each entry point names the reference code it replaces.  Plain pointers and
 * sizes only -- no torch types.  All device pointers must live on the device `gd_pack_weights` was given
 * (or the current device for the weight-free solvers); all work is stream-ordered on `stream`
 * (a cudaStream_t passed as void*), with no host synchronisation and no hidden device allocation.
 *
 * Return value: 0 on success, a negative GD_E* code otherwise; gd_last_error() holds the message
 * (thread-local).
 */
#ifndef GDECONV_H_
#define GDECONV_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GD_VERSION 100

#if defined(__GNUC__)
#define GD_API __attribute__((visibility("default")))
#else
#define GD_API
#endif

enum { GD_OK = 0, GD_EBADSHAPE = -1, GD_EBADDEVICE = -2, GD_ECUDA = -3, GD_EUNSUPPORTED = -4, GD_EWORKSPACE = -5 };

/* which unrolled-ADMM class the weights belong to */
enum { GD_ARCH_G = 0,  /* models/unrolled_admm_gaussian.py:96-152  UnrolledADMMGaussian, ResUNet nc 32..256  */
       GD_ARCH_U = 1   /* models/Unrolled_ADMM.py:153-215,371-442  Unrolled_ADMM(_Old),   ResUNet nc 64..512  */ };

/* arithmetic of the 34 inner ResUNet convolutions (head 1->C and tail C->1 are always fp32 CUDA-core) */
enum { GD_PREC_FP32_SIMT = 0,  /* fp32 FMA on CUDA cores: validation mode                                        */
       GD_PREC_FP16_UMMA = 1,  /* fp16 operands, fp32 accumulate, tcgen05.mma + TMEM: the product path            */
       GD_PREC_FP16_SIMT = 2   /* same fp16 rounding points as UMMA but CUDA-core FMAs: isolates descriptor bugs  */ };

/* likelihood of path U (models/Unrolled_ADMM.py:322-336) */
enum { GD_LLH_GAUSSIAN = 0, GD_LLH_POISSON = 1 };

/* classical solvers */
enum { GD_SOLVER_RL = 0,            /* models/Richard_Lucy.py:10-24                 */
       GD_SOLVER_WIENER = 1,        /* models/Wiener.py:10-20                       */
       GD_SOLVER_TIKHONOV_ID = 2,   /* models/Tikhonet.py:15-31, filter='Identity'  */
       GD_SOLVER_TIKHONOV_LAP = 3   /* models/Tikhonet.py:15-31, filter='Laplacian' */ };

/* One entry of a torch state_dict, as HOST fp32 memory (the weight ABI is the reference's state_dict key layout,
 * SURVEY.md section 8b: "Z.net.m_head.weight", "init.conv_layers.0.maxpool_conv.1.double_conv.0.weight", ...). */
typedef struct GdTensorDesc {
    const char* name;
    const float* data;
    int ndim;
    int64_t shape[4];
} GdTensorDesc;

typedef struct GdWeights GdWeights;   /* opaque, immutable after packing, shareable across streams */

GD_API int gd_version(void);
GD_API const char* gd_last_error(void);

/* Replaces nn.Module.load_state_dict + .to(device) for UnrolledADMMGaussian / Unrolled_ADMM(_Old)
 * (test.py:47-54): folds the SubNet BatchNorms, repacks every conv as a K-major tap-GEMM operand in the
 * chosen precision and uploads one blob to `device`.  Missing SubNet tensors are allowed when the matching
 * `rho*_iters` vectors are present (subnet=False). */
GD_API int gd_pack_weights(int arch, int n_iters, const GdTensorDesc* tensors, int n_tensors, int precision, int device,
                    GdWeights** out);
GD_API void gd_free_weights(GdWeights* w);

/* Workspace (caller-owned device memory) for processing up to `chunk` stamps at a time. */
GD_API size_t gd_workspace_bytes(int arch, int precision, int chunk);
/* Zeroes the activation halos and writes the header gd_admm_forward validates.  Once per workspace. */
GD_API int gd_workspace_init(void* workspace, size_t bytes, int arch, int precision, int chunk, void* stream);
/* Forgets an initialised workspace; call it before freeing the memory (a later allocation may reuse the address). */
GD_API void gd_workspace_release(void* workspace);

/* Replaces UnrolledADMMGaussian.forward (models/unrolled_admm_gaussian.py:117-152) for arch G and
 * Unrolled_ADMM.forward / Unrolled_ADMM_Old.forward (models/Unrolled_ADMM.py:177-215,396-442) for arch U.
 *   y, psf   [batch][48*48] fp32 device;  alpha [batch] fp32 device
 *   out      [batch][48*48] fp32 device: z_list[-1] (G) / x_list[-1] (U; times alpha for llh=Poisson)
 *   rho_out  optional [batch][n_rho] (n_rho = n_iters for G, 2*n_iters for U)
 *   analysis optional per-iteration state:
 *            G: [n_iters][3][batch][2304]  (x, z, u)                 (analysis=True lists, :147-152)
 *            U: [n_iters+1][5][batch][2304] (v, z, x, u1, u2), entry 0 = initial state (Old, :419-442)
 *   u_v0_over_alpha  path U only, bit flags: bit 0: initial v = y/alpha (Unrolled_ADMM_Old, :416) instead of y (:194);
 *                    bit 1: the result is multiplied by alpha for BOTH likelihoods (models/ADMMNet.py:129 -- with
 *                    rho1_iters = rho2_iters = 0.5 in the weights this entry point is ADMMNet.forward, :96-129)
 * Any `batch` >= 0 is accepted; it is processed in chunks of the workspace's `chunk`. */
GD_API int gd_admm_forward(const GdWeights* w, int llh, int u_v0_over_alpha, const float* y, const float* psf,
                    const float* alpha, float* out, float* rho_out, float* analysis, int batch, void* workspace,
                    size_t workspace_bytes, void* stream);

/* Replaces ResUNet.forward (models/ResUNet.py:26-42) on [batch][48*48] fp32 single-channel stamps
 * (the z-update of both ADMM classes); uses the same workspace as gd_admm_forward. */
GD_API int gd_resunet_forward(const GdWeights* w, const float* in, float* out, int batch, void* workspace,
                       size_t workspace_bytes, void* stream);

/* Replaces SubNet.forward (models/unrolled_admm_gaussian.py:61-71, models/Unrolled_ADMM.py:77-90):
 * rho_out [batch][n_rho]. */
GD_API int gd_subnet_forward(const GdWeights* w, const float* psf, const float* alpha, float* rho_out, int batch,
                      void* stream);

/* Replaces Richard_Lucy.forward / Wiener.forward / Tikhonov.forward (see GD_SOLVER_*), including the
 * psf_to_otf quirks of utils/utils_torch.py:79-92.  alpha may be NULL for RL; lam is Tikhonov's lambda. */
GD_API int gd_fft_solver(int kind, int n_iters, float lam, const float* y, const float* psf, const float* alpha, float* out,
                  int batch, void* stream);

/* Batched FFT plumbing of utils/utils_torch.py:46-50 (conv_fft_batch with H = psf_to_otf(psf)):
 * out = ifft2(fft2(x) * H).real, or with conj(H) when `adjoint`.  Used by the parity tests of the FFT core. */
GD_API int gd_conv_fft(const float* x, const float* psf, float* out, int adjoint, int batch, void* stream);

/* Replaces psf_to_otf(ker, size) (utils/utils_torch.py:79-92) for size = (batch,1,48,48), on the device (the reference builds
 * `psf` on the CPU and FFTs it there).  ker [ker_batch][kh][kw] fp32 with ker_batch = 1 (broadcast, e.g. the 3x3 Laplacian of
 * models/Tikhonet.py:26) or = batch; psf_out [batch][48*48] fp32 is the circularly shifted / broadcast kernel, otf_out
 * [batch][48*48] interleaved complex64 its FULL spectrum.  Kernel sizes torch could not broadcast are GD_EBADSHAPE. */
GD_API int gd_psf_to_otf(const float* ker, int ker_batch, int kh, int kw, float* psf_out, float* otf_out, int batch, void* stream);

/* Replaces conv_fft_batch(H, x) / the 4-D branch of conv_fft(H, x) (utils/utils_torch.py:35-50): out = ifft2(fft2(x) * H).real
 * for a full complex spectrum otf [otf_batch][48*48] (interleaved complex64, otf_batch = 1 or batch), x / out [batch][48*48]. */
GD_API int gd_conv_otf(const float* otf, int otf_batch, const float* x, float* out, int batch, void* stream);

/* Per-stamp moment ellipticities (utils/fit_ellipse.py:370-399,467-548 + utils/utils_test.py:92-96):
 * e12 [batch][2]. */
GD_API int gd_moments_e(const float* img, float* e12, int batch, void* stream);

/* XDenseUNet denoiser and the full Tikhonet / ShapeNet model (models/XDenseUNet.py:5-115, models/Tikhonet.py:34-47;
 * SURVEY.md section 8f #1).  `tensors` is a state_dict as for gd_pack_weights; `prefix` is prepended to the XDenseUNet key
 * names ("denoiser." for a Tikhonet state_dict, "" for a bare XDenseUNet).  The workspace needs no initialisation.
 * gd_tikhonet_forward = clamp(y) -> Tikhonov(filter, lam) -> XDenseUNet -> * alpha. */
typedef struct GdXDense GdXDense;
GD_API int gd_pack_xdense(const GdTensorDesc* tensors, int n_tensors, const char* prefix, int device, GdXDense** out);
GD_API void gd_free_xdense(GdXDense* x);
GD_API size_t gd_xdense_workspace_bytes(int chunk);
GD_API int gd_xdense_forward(const GdXDense* x, const float* in, float* out, int batch, void* workspace, size_t workspace_bytes,
                             int chunk, void* stream);
GD_API int gd_tikhonet_forward(const GdXDense* x, int filter, float lam, const float* y, const float* psf, const float* alpha,
                               float* out, int batch, void* workspace, size_t workspace_bytes, int chunk, void* stream);

/* Replaces Unrolled_ADMM(_Old).forward / ADMMNet.forward constructed with denoiser='XDenseUNet' (models/Unrolled_ADMM.py:142-151,163,
 * 360-369,381; models/ADMMNet.py:65-74,87): the path-U loop of gd_admm_forward with z = XDenseUNet(x + u1) as the Z-update (fp32, on
 * the unscaled input).  `w` is packed with gd_pack_weights(GD_ARCH_U, ...) from the same state_dict and carries the SubNet or the
 * rho parameters (a ResUNet is not needed); `x` is packed with gd_pack_xdense(prefix "Z.net.").  Arguments as gd_admm_forward
 * (`flags` = its u_v0_over_alpha word) plus the XDenseUNet workspace of gd_xdense_workspace_bytes(xd_chunk). */
GD_API int gd_admm_forward_xdense(const GdWeights* w, const GdXDense* x, int llh, int flags, const float* y, const float* psf,
                                  const float* alpha, float* out, float* rho_out, float* analysis, int batch, void* workspace,
                                  size_t workspace_bytes, void* xd_workspace, size_t xd_workspace_bytes, int xd_chunk, void* stream);

/* Synthetic galaxy stamps on the device: the CUDA twin of the generator module gdsynth.py (make_batch), which stands in for the
 * reference's GalSim pipeline (generate_data.py:114-334) and keeps its conventions: 48x48 stamps rendered 4x oversampled and
 * averaged 4x4 (utils/utils_data.py:26-40), Sersic galaxy, Moffat PSF centred on pixel (24,24), sky + read noise sigma = 19.04
 * ADU, flux scaled to the SNR, obs = max(gt (*) psf, 0) + N(0, sigma^2) and alpha = obs.mean() (utils/utils_data.py:100-101).
 * Stamp i of the batch is stamp `start + i` of the stream `seed`: its values depend only on (seed, start + i).
 *   snr_mode  GD_SYNTH_SNR_FIXED: every stamp at `snr` (> 0);  GD_SYNTH_SNR_MIXED: log-uniform in [20, 300] per stamp
 *   psf_fwhm_err (arcsec) / psf_shear_err: when either is non-zero, `psf` is the mismatched model PSF while obs was blurred
 *             with the true one (the PSF-mismatch sweep of test_psf.py:237,242)
 *   obs, psf, gt [count][48*48] fp32 device, alpha [count] fp32 device; `psf` sums to 1/16.  Any output may be NULL (not all):
 *             only the stages the requested outputs need run, so a psf-only call renders just the PSF. */
enum { GD_SYNTH_SNR_FIXED = 0, GD_SYNTH_SNR_MIXED = 1 };
GD_API int gd_synth_batch(int64_t start, int count, int64_t seed, int snr_mode, float snr, float psf_fwhm_err,
                          float psf_shear_err, float* obs, float* psf, float* alpha, float* gt, void* stream);

/* Adaptive second moments of each stamp (Bernstein & Jarvis 2002; Hirata & Seljak 2003; the estimator family of GalSim's
 * galsim.hsm.FindAdaptiveMom, without its step damping and bounds).  Pixel p = 48 r + c is at x = c, y = r.  The weight
 * w = exp(-rho^2/2), rho^2 = (Myy dx^2 - 2 Mxy dx dy + Mxx dy^2) / det(M) starts at (24, 24) with M = guess_sigma^2 I; each pass
 * sets the centroid to the weighted centroid and M to twice the weighted central second moments, until the centroid moves by
 * <= 1e-5 sqrt(t) and M by <= 1e-5 t (t = tr M / 2), at most 100 passes.  A stamp stops early with GD_SHAPE_FLUX when the
 * weighted flux is not positive (or NaN), GD_SHAPE_MOMENTS when M is not positive definite or tr M > 1152 px^2, and
 * GD_SHAPE_CENTROID when the centroid leaves the 15 px box around (24, 24).
 *   img    [batch][48*48] fp32 device;  guess_sigma in (0, 24] px (3 is a good start for galaxies of 1.5-6 px)
 *   shape  [batch][8] fp32 device: flux (= 2 x the weighted flux, exact for a Gaussian), x0, y0, Mxx, Mxy, Myy,
 *          e1 = (Mxx - Myy)/(Mxx + Myy), e2 = 2 Mxy/(Mxx + Myy) (the distortion of gd_moments_e); all NaN unless GD_SHAPE_OK
 *   info   [batch][2] int32 device: status (GD_SHAPE_*), number of passes made
 * A stamp's result does not depend on the batch it is measured in. */
enum { GD_SHAPE_OK = 0, GD_SHAPE_MAXITER = 1, GD_SHAPE_FLUX = 2, GD_SHAPE_MOMENTS = 3, GD_SHAPE_CENTROID = 4 };
GD_API int gd_adaptive_moments(const float* img, int batch, float guess_sigma, float* shape, int32_t* info, void* stream);

/* Test hook: one tap-GEMM layer of the denoiser on caller-packed operands (layouts of csrc/gd_common.cuh:
 * activations [Kt/CH][Ptot][CH], CH = 8 halves (fp16 modes) or 4 floats; weights as gd_pack_weights lays them out
 * for `precision`; out32 [N/4][Ptot][4] fp32).  ntaps = 9 (3x3, zero padding) or 1.  `geom7` receives
 * {H, W, Wp, S, base0, Ptot, M} for `batch` stamps of HxH pixels so the caller can pack/unpack. */
/* Largest `chunk` gd_workspace_bytes / gd_workspace_init accept: the kernels decode GEMM rows into (stamp, y, x) with a
 * multiply-shift division that is exact below 2^26 rows; larger chunks are rejected (GD_EBADSHAPE), never mis-decoded. */
GD_API int gd_max_chunk(void);
/* Test hook (host only): first n in [n_lo, n_hi) for which the kernels' multiply-shift n / d is wrong, or -1. */
GD_API long long gd_debug_divmagic(unsigned d, unsigned n_lo, unsigned n_hi);
GD_API int gd_debug_geom(int H, int batch, int* geom7);
GD_API int gd_debug_tapgemm(int precision, int H, int batch, int ntaps, int Kt, int N, int relu, const void* act,
                            const void* weights, float* out32, void* stream);

/* Live timing of the dominant kernel (k_conv_umma, the tcgen05 tap-GEMM): between begin and end every launch is
 * bracketed by CUDA events on its stream; end synchronises them and returns the summed device time (ms), the summed
 * ALGORITHMIC FLOPs (2*K*N per tap and valid output pixel) and the number of launches.  Not thread-safe. */
GD_API void gd_profile_begin(void);
GD_API int gd_profile_end(double* ms_total, double* flops_total, uint64_t* launches);

/* Number of kernel launches issued by this library since load (bench.py's gpu_launches claim). */
GD_API uint64_t gd_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* GDECONV_H_ */
