// Host-callable launchers of every kernel in libgdeconv (definitions in fft_kernels.cu, subnet.cu, conv_simt.cu,
// conv_umma.cu, synth.cu, shape.cu).  All are stream-ordered and return GD_OK or a negative GD_E* code.
#pragma once
#include "gd_common.cuh"
#include "subnet.cuh"

namespace gd {

int fft_kernels_init();
int ensure_device_init(int device);      // api.cu: once per device, opt-in shared memory sizes etc. of every kernel
int subnet_init();
int conv_umma_init();
void conv_profile_begin();
int conv_profile_end(double* ms_total, double* flops_total, unsigned long long* launches);
int conv_profile_mark(double flops, cudaStream_t st, cudaEvent_t* stop);
int conv_rb_init();
int conv_l1chain_init();
int launch_l1chain_down(const Geom& g0, const Geom& g1, int nb, const float* t, const float* head_w_host, const void* const* w4, const void* wdown,
                        float* skip32, void* x2_16, void* x2_lo, cudaStream_t st);
size_t l1chain_scratch_bytes();
int launch_l1chain_up(const Geom& g0, const Geom& g1, int nb, const void* x_in, const void* wup, const float* tail_w_host, const void* const* w4,
                      float* tail_part, void* scratch, cudaStream_t st);
int conv_l2chain_init();
size_t l2chain_scratch_bytes();
int launch_l2chain(int mode, const Geom& g1, const Geom& g2, int nb, const void* x_hi, const void* x_lo, const void* const* w4, const void* wdown,
                   float* skip3, void* x3_16, const void* a_coarse, const void* wup, void* scratch, const float* skip32, void* out16, cudaStream_t st);
bool conv_rb_supported(const ConvParams& p1, const ConvParams& p2);
int launch_conv_rb(const ConvParams& p1, const ConvParams& p2, cudaStream_t st);

int launch_g_prologue(const float* y, const float* psf, const float* alpha, float2* Pc, float* HtH, float* z, float* u,
                      float* x, int batch, cudaStream_t st);
int launch_g_xupdate(const float2* Pc, const float* HtH, const float* rho, int n_rho, int it, const float* z, float* x,
                     float* u, float* t, float* tscale, int batch, cudaStream_t st, const float* head_w_host = nullptr,
                     const Geom* g0 = nullptr, void* a16 = nullptr, float* tpad = nullptr);
int launch_g_dual_out(const float* rho, int n_rho, int it, const float* x, const float* z, const float* u, float* uo,
                      int batch, cudaStream_t st);
int launch_scale_in(const float* in, float* t, float* tscale, int batch, cudaStream_t st);
int launch_fill_rho(const float* src, int n_rho, float* rho, int batch, cudaStream_t st);
int launch_solver(int kind, int n_iters, float lam, const float* y, const float* psf, const float* alpha, float* out,
                  int batch, cudaStream_t st);
int launch_conv_fft(const float* x, const float* psf, float* out, int adjoint, int batch, cudaStream_t st);
int launch_psf_to_otf(const float* ker, int kb, int kh, int kw, float* psf_out, float2* otf_out, int batch, cudaStream_t st);
int launch_conv_otf(const float2* H, int hb, const float* x, float* out, int batch, cudaStream_t st);
int launch_u_prologue(const float* y, const float* psf, const float* alpha, int v0_over_alpha, float2* Hw, float* x,
                      float* z, float* v, float* u1, float* u2, float* Hx, int batch, cudaStream_t st);
int launch_u_pre(int llh, const float* y, const float* alpha, const float* rho, int n_rho, int n, int it, const float* x,
                 const float* u1, const float* u2, const float* Hx, float* v, float* t, float* tscale, int batch,
                 cudaStream_t st);
int launch_u_post(const float2* Hw, const float* rho, int n_rho, int n, int it, const float* z, const float* v, float* x,
                  float* u1, float* u2, float* Hx, int batch, cudaStream_t st);
int launch_scale_by_alpha(float* out, const float* x, const float* alpha, int batch, int use_alpha, cudaStream_t st);
int launch_moments(const float* img, float* e12, int batch, cudaStream_t st);
int launch_subnet(const SubnetParams& P, const float* psf, const float* alpha, float* rho, int batch, cudaStream_t st);
int synth_init();
int launch_synth(int64_t start, int count, int64_t seed, int mixed, float snr, float fwhm_err, float shear_err, float* obs,
                 float* psf, float* alpha, float* gt, cudaStream_t st);
int launch_adaptive_moments(const float* img, int batch, float guess_sigma, float* shape, int32_t* info, cudaStream_t st);

int launch_conv_simt(const ConvParams& p, int prec, cudaStream_t st);
int launch_conv_umma(const ConvParams& p, cudaStream_t st);
int launch_head(const float* t, const float* w, const float* w_host, int C0, const ConvParams& p, int batch, int prec, float* tpad, cudaStream_t st);
int launch_tail_gather(const float* P, int units, const Geom& g, const float* tscale, float* z, int batch, const float* tpad,
                       const float* G81_host, cudaStream_t st, int t_plain = 0);
int launch_tail(const float* x32, const float* w, int C0, const Geom& g, const float* tscale, float* z, int batch,
                cudaStream_t st);

}  // namespace gd
