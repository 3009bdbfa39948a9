// CUDA-core convolution kernels.
//  * k_conv_simt<T>: the same tap-GEMM the tcgen05 kernel computes, on FP32 FMA units.  T = float is the
//    PREC_FP32_SIMT precision mode (bit-for-bit independent check of the layer graph against the oracle);
//    T = __half reads the very same fp16 buffers/rounding points as the tcgen05 path (PREC_FP16_SIMT), which
//    isolates tensor-core descriptor bugs from precision effects.
//  * k_head / k_tail: the 1->C and C->1 3x3 convs of models/ResUNet.py:11,24 in fp32 (SURVEY.md section 0.8:
//    these two layers dominate the rounding error, and are 0.2 % of the FLOPs).
#include "conv_epilogue.cuh"
#include "kernels.cuh"
#include "launch.cuh"

namespace gd {

constexpr int SIMT_KSLAB = 256;

template <typename T> __device__ __forceinline__ void load_vec(const T* p, float* a);
template <> __device__ __forceinline__ void load_vec<float>(const float* p, float* a) {
    float4 v = *reinterpret_cast<const float4*>(p);
    a[0] = v.x; a[1] = v.y; a[2] = v.z; a[3] = v.w;
}
template <> __device__ __forceinline__ void load_vec<__half>(const __half* p, float* a) {
    uint4 v = *reinterpret_cast<const uint4*>(p);
    const __half2* h = reinterpret_cast<const __half2*>(&v);
#pragma unroll
    for (int i = 0; i < 4; ++i) { float2 f = __half22float2(h[i]); a[2 * i] = f.x; a[2 * i + 1] = f.y; }
}

// weights: [tap][Kt][N] of T
template <typename T>
__global__ void __launch_bounds__(128) k_conv_simt(const ConvParams p) {
    constexpr int CH = ActT<T>::CH;
    __shared__ __align__(16) float wsm[SIMT_KSLAB * 16];
    const int m = blockIdx.x * MTILE + threadIdx.x;
    const int n0 = blockIdx.y * 16;
    const T* A = reinterpret_cast<const T*>(p.a);
    const T* Wt = reinterpret_cast<const T*>(p.w);
    const int row = p.g.base0 + m;
    float acc[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) acc[i] = 0.f;
    for (int tap = 0; tap < p.ntaps; ++tap) {
        for (int k0 = 0; k0 < p.Kt; k0 += SIMT_KSLAB) {
            const int kn = min(SIMT_KSLAB, p.Kt - k0);
            __syncthreads();
            for (int i = threadIdx.x; i < kn * 16; i += blockDim.x)
                wsm[i] = (float)Wt[((size_t)tap * p.Kt + k0 + (i >> 4)) * p.N + n0 + (i & 15)];
            __syncthreads();
            const T* ap = A + ((size_t)(k0 / CH) * p.g.Ptot + row + p.off[tap]) * CH;
            for (int kc = 0; kc < kn / CH; ++kc) {
                float a[CH];
                load_vec<T>(ap + (size_t)kc * p.g.Ptot * CH, a);
#pragma unroll
                for (int j = 0; j < CH; ++j) {
                    const float4* wr = reinterpret_cast<const float4*>(wsm + (kc * CH + j) * 16);
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        float4 w4 = wr[q];
                        acc[4 * q] = fmaf(a[j], w4.x, acc[4 * q]);
                        acc[4 * q + 1] = fmaf(a[j], w4.y, acc[4 * q + 1]);
                        acc[4 * q + 2] = fmaf(a[j], w4.z, acc[4 * q + 2]);
                        acc[4 * q + 3] = fmaf(a[j], w4.w, acc[4 * q + 3]);
                    }
                }
            }
        }
    }
    RowCtx rc = make_row_ctx(p, m);
    if (rc.valid) epilogue_store16<T>(p, rc, n0, acc);
}

// head: t [B][48*48] fp32 (already scaled per stamp) -> skip32 (fp32) + x16 (operand precision), C0 channels.
// weights w[tap][C0] fp32.
template <typename T>
__global__ void __launch_bounds__(128) k_head(const float* __restrict__ t, const float* __restrict__ w, int C0,
                                              ConvParams p, int batch, float* __restrict__ tpad) {
    extern __shared__ __align__(16) float wsm[];           // 9*C0
    for (int i = threadIdx.x; i < 9 * C0; i += blockDim.x) wsm[i] = w[i];
    __syncthreads();
    int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= batch * NPIX) return;
    int b = idx / NPIX, r = idx - b * NPIX, y = r / STAMP, x = r - y * STAMP;
    float in[9];
#pragma unroll
    for (int dy = -1; dy <= 1; ++dy)
#pragma unroll
        for (int dx = -1; dx <= 1; ++dx) {
            int yy = y + dy, xx = x + dx;
            in[(dy + 1) * 3 + dx + 1] = (yy >= 0 && yy < STAMP && xx >= 0 && xx < STAMP) ? t[(size_t)b * NPIX + yy * STAMP + xx] : 0.f;
        }
    RowCtx rc;
    rc.valid = true; rc.row = p.g.base0 + b * p.g.S + y * p.g.Wp + x; rc.crow = 0; rc.ctap = 0; rc.frow0 = 0;
    if (tpad) tpad[rc.row] = in[4];          // padded-linear copy of the input for the head-recomputing epilogues (EPI_HT)
    for (int n0 = 0; n0 < C0; n0 += 16) {
        float acc[16];
#pragma unroll
        for (int c = 0; c < 16; ++c) acc[c] = 0.f;
#pragma unroll
        for (int tp = 0; tp < 9; ++tp) {         // per channel: fma chain over the taps in order 0..8 (LDS.128 weight loads)
            const float4* w4 = reinterpret_cast<const float4*>(wsm + tp * C0 + n0);
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const float4 ww = w4[q];
                acc[4 * q] = fmaf(in[tp], ww.x, acc[4 * q]); acc[4 * q + 1] = fmaf(in[tp], ww.y, acc[4 * q + 1]);
                acc[4 * q + 2] = fmaf(in[tp], ww.z, acc[4 * q + 2]); acc[4 * q + 3] = fmaf(in[tp], ww.w, acc[4 * q + 3]);
            }
        }
        epilogue_store16<T>(p, rc, n0, acc);
    }
}

// tail: x32 [C0/4][Ptot][4] fp32 -> z [B][48*48] fp32, times the per-stamp power-of-two scale.
// Works in the padded-linear row space (the halo rows of the stream are zero, so there are no bounds checks): a CTA
// stages the window rows [m0 - Wp - 1, m0 + TAIL_ROWS + Wp + 1) of all C0/4 planes in shared memory with coalesced
// 16-byte loads (each element leaves L2 once instead of nine times through L1), then every thread reduces the 9 taps x
// C0 channels of its row from shared memory (conflict-free LDS.128) and writes its pixel if the row is a real one.
constexpr int TAIL_ROWS = 256;
__global__ void __launch_bounds__(TAIL_ROWS) k_tail(const float* __restrict__ x32, const float* __restrict__ w, int C0, Geom g,
                                                    const float* __restrict__ tscale, float* __restrict__ z, int batch) {
    extern __shared__ __align__(16) float tsm[];          // [9*C0 weights][C0/4 planes][win rows][4]
    float* wsm = tsm;
    const int halo = g.Wp + 1, win = TAIL_ROWS + 2 * halo, planes = C0 / 4;
    float4* xs = reinterpret_cast<float4*>(tsm + 9 * C0);
    for (int i = threadIdx.x; i < 9 * C0; i += blockDim.x) wsm[i] = w[i];
    const int m0 = blockIdx.x * TAIL_ROWS;
    const float4* src = reinterpret_cast<const float4*>(x32) + (g.base0 + m0 - halo);
    for (int i = threadIdx.x; i < planes * win; i += blockDim.x) {
        const int pl = i / win, r = i - pl * win;
        xs[i] = __ldg(src + (size_t)pl * g.Ptot + r);
    }
    __syncthreads();
    const int m = m0 + threadIdx.x;
    if (m >= g.M) return;
    const int b = (int)div_by_magic((uint32_t)m, g.magS, g.shS), r = m - b * g.S;
    const int y = (int)div_by_magic((uint32_t)r, g.magW, g.shW), x = r - y * g.Wp;
    if (y >= g.H || x >= g.W) return;
    float s = 0.f;
    const float4* row = xs + halo + threadIdx.x;
    for (int pl = 0; pl < planes; ++pl) {
#pragma unroll
        for (int t = 0; t < 9; ++t) {
            const float4 v = row[pl * win + (t / 3 - 1) * g.Wp + (t % 3 - 1)];
            const float4 wv = *reinterpret_cast<const float4*>(wsm + t * C0 + 4 * pl);
            s = fmaf(v.x, wv.x, s); s = fmaf(v.y, wv.y, s); s = fmaf(v.z, wv.z, s); s = fmaf(v.w, wv.w, s);
        }
    }
    z[(size_t)b * NPIX + y * STAMP + x] = s * tscale[b];
}

// Tail of the head/tail-fused tcgen05 path: the last conv of m_up1 left P[u*9 + tap][row] = sum_c w_tail[tap][c] * x[row][c]
// (32-channel unit u, x = the ResBlock output WITHOUT the U-Net skip x1); m_tail (ResUNet.py:39) of x + x1 is then
//     z[m] = sum_tap sum_u P[u*9 + tap][m + off(tap)]  +  tail(x1)[m],
// times the per-stamp power-of-two input scale.  Since x1 = m_head(t) is linear in the 1-channel input t, its tail is the
// 81-coefficient composite  tail(x1)[m] = sum_{tap2: m+off2 inside the stamp} sum_tap1 G[tap2][tap1] * t[m + off2 + off1],
// G = W_tail W_head^T (kernel parameters), evaluated here from the padded-linear copy of t (zero halos) instead of 288 FMAs
// per row in the conv epilogue.  Halo rows of P are never written.
// The zero padding of m_tail drops the taps t2 whose pixel lies outside the stamp, so the composite is one of NINE 5x5 stencils,
// chosen by whether the pixel sits on the first / last row and column; the host collapses G (81 coefficients) into them.
struct TailG { float g5[9 * 25]; };
__global__ void __launch_bounds__(256) k_tail_gather(const float* __restrict__ P, int units, Geom g, const float* __restrict__ tscale,
                                                     float* __restrict__ z, int batch, const float* __restrict__ tpad,
                                                     const __grid_constant__ TailG G, int t_plain) {
    __shared__ float g5s[9 * 25];
    if (threadIdx.x < 9 * 25) g5s[threadIdx.x] = G.g5[threadIdx.x];
    __syncthreads();
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= batch * NPIX) return;
    const int b = idx / NPIX, r = idx - b * NPIX, y = r / STAMP, x = r - y * STAMP;
    const int row = g.base0 + b * g.S + y * g.Wp + x;
    const float* src = P + row;
    float s = 0.f;
    for (int u = 0; u < units; ++u) {
#pragma unroll
        for (int t = 0; t < 9; ++t) s += __ldg(src + (size_t)(u * 9 + t) * g.Ptot + (t / 3 - 1) * g.Wp + (t % 3 - 1));
    }
    // (a leaner address / predicate computation -- 118 M instead of 199 M warp instructions -- needs 75 registers and is SLOWER,
    // 262 us against 234 us per 5000 stamps: the kernel is bound by bytes in flight, i.e. by resident threads)
    const float* c5 = g5s + ((y == 0 ? 0 : y == STAMP - 1 ? 2 : 1) * 3 + (x == 0 ? 0 : x == STAMP - 1 ? 2 : 1)) * 25;
    float a = 0.f;
#pragma unroll
    for (int dy = -2; dy <= 2; ++dy)
#pragma unroll
        for (int dx = -2; dx <= 2; ++dx) {
            const int yy = y + dy, xx = x + dx;
            // 5x5 neighbourhood of t (zero outside the stamp).  t_plain: `tpad` is the dense [B][48*48] denoiser input itself
            // (conv_l1chain.cu path: no padded-linear copy exists)
            const float tv = (yy >= 0 && yy < STAMP && xx >= 0 && xx < STAMP)
                                 ? (t_plain ? __ldg(tpad + (size_t)b * NPIX + yy * STAMP + xx) : __ldg(tpad + row + dy * g.Wp + dx)) : 0.f;
            a = fmaf(c5[(dy + 2) * 5 + dx + 2], tv, a);
        }
    s += a;
    z[idx] = s * tscale[b];
}

// ---- host launchers ----
int launch_conv_simt(const ConvParams& p, int prec, cudaStream_t st) {
    if (p.g.M <= 0) return GD_OK;
    dim3 grid((p.g.M + MTILE - 1) / MTILE, p.N / 16);
    if (prec == PREC_FP32_SIMT) k_conv_simt<float><<<grid, 128, 0, st>>>(p);
    else k_conv_simt<__half><<<grid, 128, 0, st>>>(p);
    GD_LAUNCHED();
    return GD_OK;
}

int launch_head(const float* t, const float* w, int C0, const ConvParams& p, int batch, int prec, float* tpad, cudaStream_t st) {
    int n = batch * NPIX, blocks = (n + 127) / 128;
    if (n <= 0) return GD_OK;
    if (prec == PREC_FP32_SIMT) k_head<float><<<blocks, 128, 9 * C0 * sizeof(float), st>>>(t, w, C0, p, batch, tpad);
    else k_head<__half><<<blocks, 128, 9 * C0 * sizeof(float), st>>>(t, w, C0, p, batch, tpad);
    GD_LAUNCHED();
    return GD_OK;
}

int launch_tail_gather(const float* P, int units, const Geom& g, const float* tscale, float* z, int batch, const float* tpad,
                       const float* G81_host, cudaStream_t st, int t_plain) {
    if (batch <= 0) return GD_OK;
    // G81[t2 * 9 + t1]: tail tap t2 (pixel p + t2) times head tap t1 (input p + t2 + t1).  Class (cy, cx): 0 = first row / column
    // (tap -1 falls outside and is dropped), 2 = last, 1 = interior.
    double acc[9 * 25] = {0};
    for (int cy = 0; cy < 3; ++cy)
        for (int cx = 0; cx < 3; ++cx)
            for (int t2 = 0; t2 < 9; ++t2) {
                const int ty = t2 / 3, tx = t2 % 3;
                if ((cy == 0 && ty == 0) || (cy == 2 && ty == 2) || (cx == 0 && tx == 0) || (cx == 2 && tx == 2)) continue;
                for (int t1 = 0; t1 < 9; ++t1)
                    acc[(cy * 3 + cx) * 25 + (ty + t1 / 3) * 5 + (tx + t1 % 3)] += (double)G81_host[t2 * 9 + t1];
            }
    TailG G;
    for (int i = 0; i < 9 * 25; ++i) G.g5[i] = (float)acc[i];
    k_tail_gather<<<(batch * NPIX + 255) / 256, 256, 0, st>>>(P, units, g, tscale, z, batch, tpad, G, t_plain);
    GD_LAUNCHED();
    return GD_OK;
}

int launch_tail(const float* x32, const float* w, int C0, const Geom& g, const float* tscale, float* z, int batch,
                cudaStream_t st) {
    if (batch <= 0) return GD_OK;
    Geom gg = g;
    gg.M = batch * g.S;
    const int blocks = (gg.M + TAIL_ROWS - 1) / TAIL_ROWS;
    const size_t smem = (size_t)9 * C0 * sizeof(float) + (size_t)(C0 / 4) * (TAIL_ROWS + 2 * (g.Wp + 1)) * 16;
    static bool attr_set = false;
    if (!attr_set) { GD_CUDA_CHECK(cudaFuncSetAttribute(k_tail, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024)); attr_set = true; }
    k_tail<<<blocks, TAIL_ROWS, smem, st>>>(x32, w, C0, gg, tscale, z, batch);
    GD_LAUNCHED();
    return GD_OK;
}

}  // namespace gd
