// Shared definitions for libgdeconv (B200 / sm_100a): activation layouts, layer parameter blocks,
// error plumbing.  See DESIGN.md for the data layout in HBM.
#pragma once
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/gdeconv.h"

#ifndef GD_HD
#define GD_HD __host__ __device__ __forceinline__
#endif

namespace gd {

constexpr int STAMP = 48;
constexpr int NPIX = STAMP * STAMP;          // 2304
constexpr int FG = 96;                       // zero-padded grid of path G (pad_double, utils_torch.py:11-13)
constexpr int FG_NH = FG / 2 + 1;            // 49
constexpr int FG_SPEC = FG * FG_NH;          // half-spectrum elements per stamp (digit-swapped k1, natural k2)
constexpr int FU_NH = STAMP / 2 + 1;         // 25
constexpr int FU_SPEC = STAMP * FU_NH;       // 48x25 half spectrum of the circular 48x48 transforms
constexpr int MTILE = 128;                   // GEMM rows (pixels) per tile = tcgen05 M

enum Precision { PREC_FP32_SIMT = GD_PREC_FP32_SIMT, PREC_FP16_UMMA = GD_PREC_FP16_UMMA, PREC_FP16_SIMT = GD_PREC_FP16_SIMT };

// ---------------------------------------------------------------------------------------------------
// Activation layout ("padded-linear, channel-chunk-major").
//
// A feature map of C channels at resolution HxW for a chunk of B stamps is stored as
//     act[C / CH][Ptot][CH]          CH = 8 for fp16, 4 for fp32  (one 16-byte vector per pixel and chunk)
// where the pixel axis is a single linear index
//     row(b, y, x) = base0 + b*S + y*Wp + x,   Wp = W+1,  S = (H+1)*Wp,  base0 = Wp+1+64
// i.e. every image row is followed by ONE zero pixel and every stamp by ONE zero row; those zeros are shared
// by the neighbours on both sides, so the 3x3 tap (dy,dx) of ANY pixel is simply row + dy*Wp + dx and a conv
// is a GEMM whose A operand for tap t is the same buffer shifted by a constant number of 16-byte rows.
// Halo rows are never written (the buffer is zeroed once per forward), the GEMM computes garbage there and
// the epilogue drops it.  Overhead (H+1)(W+1)/(HW): 4 % at 48x48 ... 36 % at 6x6.
// ---------------------------------------------------------------------------------------------------
struct Geom {
    int H, W, Wp, S, base0, Ptot, M;          // M = B*S GEMM rows to compute
    uint32_t magS, shS, magW, shW;            // floor(n / S) = (n * magS) >> shS, floor(n / Wp) = (n * magW) >> shW
};

// Exact unsigned division of n < 2^26 by an invariant d through one 32x32->64 multiply (Granlund-Montgomery):
// with l = ceil(log2 d), shift = 26 + l and magic = ceil(2^shift / d) < 2^27, n * (magic*d - 2^shift) < 2^shift holds
// for every n < 2^26.  geom_rows_ok() is the gate: gd_workspace_bytes / gd_workspace_init reject a chunk whose GEMM rows (plus the
// tile and halo slack the kernels add) reach 2^26, gd_max_chunk() reports the largest admitted chunk, and
// tests/test_abi.py checks div_by_magic exhaustively over [0, 2^26) for every divisor the geometry uses.
constexpr uint32_t DIV_MAGIC_LIMIT = 1u << 26;
inline void div_magic(uint32_t d, uint32_t* magic, uint32_t* shift) {
    uint32_t l = 0;
    while ((1u << l) < d) ++l;
    *shift = 26 + l;
    *magic = (uint32_t)(((1ull << *shift) + d - 1) / d);
}
GD_HD uint32_t div_by_magic(uint32_t n, uint32_t magic, uint32_t shift) { return (uint32_t)(((unsigned long long)n * magic) >> shift); }

inline Geom make_geom(int H, int batch) {
    Geom g;
    // base0 >= Wp + 1 zero rows in front of the first stamp: the A window of k_conv_umma starts Wp + 1 rows before its first tile.
    // The 64 rows in front of them, like the 5 * MTILE rows at the end of Ptot, are slack that no kernel reads; removing either
    // would move every buffer offset and change gd_workspace_bytes and gd_max_chunk.
    g.H = H; g.W = H; g.Wp = H + 1; g.S = (H + 1) * (H + 1); g.base0 = g.Wp + 1 + 64;
    div_magic((uint32_t)g.S, &g.magS, &g.shS); div_magic((uint32_t)g.Wp, &g.magW, &g.shW);
    g.M = batch * g.S;
    int mt = ((g.M + MTILE - 1) / MTILE + 7) / 8 * 8;
    // the tiles rounded up to a multiple of 8 hold every work item of k_conv_umma (up to 4 tiles each); the base0 rows after them
    // hold the Wp + 1 rows its A window reaches past the last item
    g.Ptot = mt * MTILE + 2 * g.base0 + 5 * MTILE;
    return g;
}

// every row index a kernel may decode for a chunk of `batch` stamps at resolution H stays below the div_by_magic limit
inline bool geom_rows_ok(int H, long long batch) {
    const long long S = (long long)(H + 1) * (H + 1), M = batch * S;
    const long long mt = ((M + MTILE - 1) / MTILE + 7) / 8 * 8;
    return mt * MTILE + 2 * (H + 2 + 64) + 5 * MTILE < (long long)DIV_MAGIC_LIMIT;
}

GD_HD bool row_valid(int m, int S, int Wp, int H, int W, int M) {
    if (m >= M) return false;
    int r = m % S;
    return (r / Wp) < H && (r % Wp) < W;
}

// One conv / strided-conv / transposed-conv layer as a GEMM over taps (all layers of models/ResUNet.py:11-24
// except head and tail).  D[m, n] = sum_t sum_k A[m + off[t], t*? ...] -- see conv_simt.cu / conv_umma.cu.
struct ConvParams {
    Geom g;                   // geometry of the GEMM rows (level the accumulators live on)
    int ntaps;                // 9 (3x3) or 1 (k2s2 down on space-to-depth input, k2s2 up)
    int off[9];               // row offset per tap
    int Kt;                   // input channels per tap
    int N;                    // GEMM N (C_out, or 4*C_out for the transposed conv)
    const void* a;            // input activations  [Kt/CH][g.Ptot][CH]
    const void* w;            // weights, layout depends on the kernel (see pack.cu)
    int relu;
    // epilogue, all optional.  mode 0: outputs live on the GEMM-row level (C = N, Ptot = g.Ptot).
    const float* res32;       // += residual (fp32 stream)
    const float* skip32;      // += U-Net skip (fp32)
    float* out32;             // fp32 result [N/4][Ptot][4]
    void* out16;              // operand-precision copy for the next conv [N/CH][Ptot][CH]
    void* s2d;                // space-to-depth copy for the following k2s2 strided conv, coarse geometry gc
    // mode 1 (transposed conv): column n = tap*Cf + c scatters to fine pixel (2Y+dy, 2X+dx), geometry gf
    int mode;
    int Cf, Cf_log2;
    Geom gc;                  // coarse level (s2d target)
    Geom gf;                  // fine level (mode 1 target)
    // fp16 hi/lo residual stream (tcgen05 path).  A stream value x is kept as hi = rn16(x) -- which IS the fp16 operand copy
    // the next conv reads -- plus lo = rn16(x - hi) in a second fp16 buffer: 4 bytes per element written instead of 4 (fp32
    // stream) + 2 (operand copy), |x - (hi + lo)| <= 2^-22 |x|.  Layout of both: [N/8][Ptot][8] like every fp16 activation.
    const void* res_hi;       // += float(res_hi) + float(res_lo)   (instead of res32)
    const void* res_lo;
    void* out_lo;             // out16 receives hi, out_lo receives lo   (instead of out32)
    // head / tail fusion (tcgen05 path, level 0 only; conv_umma.cu EPI_HT).  The fp32 output of m_head (ResUNet.py:31)
    // is never stored: wherever it is consumed as a residual or as the final U-Net skip (ResUNet.py:39) the epilogue
    // recomputes it from the 1-channel padded-linear input `head_t` (9 FMAs per channel).  The last conv of m_up1 does
    // not store its 32-channel result either: it reduces it against the m_tail weights into 9 per-tap partial sums per
    // row, `tail_part[(n/32)*9 + tap][row]`, which k_tail_gather shifts and adds (4.5x fewer bytes than the stream).
    const float* head_t;      // [g.Ptot] fp32, zero halos
    const float* head_w;      // [9][N] fp32, HOST pointer: copied into the kernel parameters (constant bank) at launch
    float* tail_part;         // [(N/32)*9][g.Ptot] fp32
    const float* tail_w;      // [9][N] fp32, HOST pointer
};

// ---------------------------------------------------------------------------------------------------
// error plumbing (C ABI returns ints; message retrievable through gd_last_error())
// ---------------------------------------------------------------------------------------------------
void set_error(const char* fmt, ...);
#define GD_CUDA_CHECK(expr)                                                                         \
    do {                                                                                            \
        cudaError_t _e = (expr);                                                                    \
        if (_e != cudaSuccess) {                                                                    \
            gd::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
            return GD_ECUDA;                                                                    \
        }                                                                                           \
    } while (0)

// Makes `device` current for the scope and restores the caller's device on exit: the C-ABI entry points (and the free functions,
// which Python runs from __del__ at arbitrary points) must not change the current device of a multi-GPU process behind its back.
struct DeviceScope {
    int prev = -1;
    cudaError_t err = cudaSuccess;
    explicit DeviceScope(int device) {
        err = cudaGetDevice(&prev);
        if (err == cudaSuccess && prev != device) err = cudaSetDevice(device);
        else if (err == cudaSuccess) prev = -1;                      // nothing to restore
    }
    ~DeviceScope() { if (prev >= 0) cudaSetDevice(prev); }
    DeviceScope(const DeviceScope&) = delete;
    DeviceScope& operator=(const DeviceScope&) = delete;
};
#define GD_DEVICE_SCOPE(device)           \
    gd::DeviceScope _gd_dev_scope(device); \
    GD_CUDA_CHECK(_gd_dev_scope.err)

}  // namespace gd
