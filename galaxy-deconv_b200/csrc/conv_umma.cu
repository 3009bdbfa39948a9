// tcgen05 tap-GEMM convolution for the 34 inner layers of the ResUNet denoiser (models/ResUNet.py:12-23):
//     D[m, n] = sum_tap sum_k A[m + off[tap], k] * W[tap][k][n]        fp16 operands, fp32 accumulate in TMEM
// on the padded-linear activation layout of gd_common.cuh.  Because every image row / stamp is followed by a
// shared zero pixel / zero row, the A operand of tap (dy,dx) is the SAME buffer shifted by dy*Wp+dx rows of 16
// bytes.  A CTA therefore stages ONE window of 128*J + 2*(Wp+1) rows per K-slab in shared memory (bulk-async
// copies, one per 8-channel chunk) and feeds all 9 taps from it by moving the start address of the UMMA shared
// memory descriptor -- the activations cross L2->SMEM once, not nine times, and no im2col is ever materialised.
//
// Shared memory operand layout (both A and B): K-major, no swizzle ("interleaved") canonical layout,
//     [K/8 chunks][rows][8 halves]   core matrix = 8 consecutive rows x 16 bytes = 128 contiguous bytes
//     SBO (8-row group stride) = 128 B,  LBO (K-chunk stride) = rows * 16 B
// which is byte-for-byte the global layout of activations ([C/8][Ptot][8]) and packed weights
// ([tap][K/8][N][8]), so staging is plain 1-D cp.async.bulk (UBLKCP) with mbarrier complete_tx.
//
// Warp roles (416 threads, one persistent CTA per SM): warp 0 = bulk-copy producer; warps 1..4 = MMA issue, warp 1+j owns
// tile j of every item (warp 1 also allocates TMEM).  Several issuing warps are needed: ONE thread sustains only about one
// tcgen05.mma per ~57 cycles whatever the issue order (measured in round 2: a single warp issuing all J tiles interleaved
// lowered the N = 64 layers from 57 % to 45 % tensor-pipe activity, profiles/README_r02.md), below the 41..49-cycle MMAs of the
// narrow layers.  Warps 5..12 = epilogue (tcgen05.ld 32x32b -> fused ReLU / residual / skip / fp16 hi-lo stream /
// space-to-depth / pixel-shuffle scatter, conv_epilogue.cuh; residual loads are issued one item ahead).
// The 512 TMEM columns hold two accumulator stages, so the epilogue of work item i overlaps the MMAs of item i+1.
// Layers whose packed weights fit (<= 96 KB: levels 1-2 of the U-Net and all k2s2 layers) keep them resident in
// shared memory for the whole kernel; larger layers stream (slab, tap) weight stages through a 6-deep ring shared by a
// cluster of 4 CTAs (multicast bulk copies + multicast tcgen05.commit).
#include "conv_epilogue.cuh"
#include "kernels.cuh"
#include "launch.cuh"
#include "umma_ptx.cuh"

#include <cstdlib>
#include <cstring>
#include <map>
#include <mutex>
#include <utility>
#include <vector>

namespace gd {

struct UmmaCfg {
    int ncta;        // GEMM N per MMA (<= 128)
    int nslices;     // N / ncta
    int J;           // 128-row tiles per work item (J * ncta <= 256 TMEM columns per accumulator stage)
    int BK;          // channels per K-slab of the A ring
    int halo;        // Wp + 1 for 3x3, 0 for 1-tap layers
    int win_rows;    // 128 * J + 2 * halo
    int a_stage_bytes, a_stages;
    int b_resident;  // 1: all taps/K of the weights loaded once per CTA; 0: streamed per (slab, tap) through a ring
    int b_stage_bytes, b_stages, b_total_bytes;
    int items_m;     // ceil(tiles / J)
    int nsl_log2, nb32_log2;   // log2(nslices), log2(ncta / 32): both are powers of two
    int abl;         // diagnostic ablation bits (GDECONV_ABL): 1 = no weight streaming, 2 = no epilogue global traffic, 4 = no activation loads
    int late_pf;     // epilogue: all residual loads of the next item are issued after this item's last register use
    int cls;         // CTAs per cluster sharing every streamed weight stage by multicast (1 = no cluster)
    int aux_off;     // mode 1: byte offset of the 8 warp-private 4 KB transpose stages of epi_up_unit in dynamic shared memory
    size_t smem;
};

// EPI_HT: the fp32 m_head / m_tail weights travel as kernel parameters, so that every weight is an immediate
// constant-bank operand of its FFMA (no shared-memory loads on the epilogue's critical path: with two epilogue warps per
// scheduler their latency was fully exposed).  N = 128 / J for the two level-0 shapes (G: N = 32, J = 4; U: N = 64, J = 2).
template <int EPI, int N>
struct HtWeights { float head[EPI == EPI_HT ? 9 * N : 1], tail[EPI == EPI_HT ? 9 * N : 1]; };

// v[0..31] += m_head(t)[N0 .. N0+31]: 9 taps x 32 channels, weights straight from the constant bank
template <int N, int N0>
__device__ __forceinline__ void ht_head(const float* __restrict__ hw, const float* hcur, float* v) {
#pragma unroll
    for (int t = 0; t < 9; ++t)
#pragma unroll
        for (int k = 0; k < 32; ++k) v[k] = fmaf(hcur[t], hw[t * N + N0 + k], v[k]);
}
// 9 per-tap partial sums of m_tail over channels N0 .. N0+31 (four independent chains per tap)
template <int N, int N0>
__device__ __forceinline__ void ht_tail(const float* __restrict__ tw, const float* v, float* dst, size_t Ptot) {
#pragma unroll
    for (int t = 0; t < 9; ++t) {
        float s[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int k = 0; k < 32; ++k) s[k & 3] = fmaf(v[k], tw[t * N + N0 + k], s[k & 3]);
        dst[(size_t)t * Ptot] = (s[0] + s[1]) + (s[2] + s[3]);
    }
}

template <int J, int KK, int EPI>
__global__ void __launch_bounds__(UMMA_THREADS, 1) k_conv_umma(const ConvParams p, const UmmaCfg c,
                                                               const __grid_constant__ HtWeights<EPI, 128 / J> htw) {
    extern __shared__ __align__(128) unsigned char smem[];
    __shared__ __align__(8) uint64_t bars[2 * MAX_A_STAGES + 2 * MAX_B_STAGES + 5];
    __shared__ uint32_t tmem_slot;
    const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0), lane = threadIdx.x & 31;   // provably warp-uniform
    unsigned char* a_smem = smem;
    unsigned char* b_smem = smem + (size_t)c.a_stages * c.a_stage_bytes;
    const uint32_t bar0 = smem_u32(bars);
    auto a_full = [&](int s) { return bar0 + 8u * s; };
    auto a_empty = [&](int s) { return bar0 + 8u * (MAX_A_STAGES + s); };
    auto b_full = [&](int s) { return bar0 + 8u * (2 * MAX_A_STAGES + s); };
    auto b_empty = [&](int s) { return bar0 + 8u * (2 * MAX_A_STAGES + MAX_B_STAGES + s); };
    const uint32_t w_full = bar0 + 8u * (2 * MAX_A_STAGES + 2 * MAX_B_STAGES);
    auto acc_full = [&](int s) { return w_full + 8u * (1 + s); };
    auto acc_empty = [&](int s) { return w_full + 8u * (3 + s); };

    if (threadIdx.x == 0) {
        for (int s = 0; s < MAX_A_STAGES; ++s) { mbar_init(a_full(s), 1); mbar_init(a_empty(s), J); }
        for (int s = 0; s < MAX_B_STAGES; ++s) { mbar_init(b_full(s), 1); mbar_init(b_empty(s), J * c.cls); }
        mbar_init(w_full, 1);
        const int nu_all = J * (c.ncta / 32);
        for (int s = 0; s < 2; ++s) { mbar_init(acc_full(s), J); mbar_init(acc_empty(s), nu_all >= 2 ? EPI_WARPS : EPI_WARPS / 2); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_slot)), "r"(TMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    if (c.cls > 1) cluster_sync_all();             // the peers' barriers exist before anything is multicast to them
    tc_fence_after();
    const uint32_t tmem = tmem_slot;

    const int nslabs = p.Kt / c.BK;
    const int chunks = c.BK / 8;
    const int KC = p.Kt / 8;                       // K chunks per tap in the packed weights
    // Work distribution.  Iteration `it` of the kernel-wide list is (M-group it >> nsl_log2, N-slice it & (nslices-1)); the
    // CTAs of a cluster take the cls consecutive M-items of the group with the SAME slice, so they walk identical weight
    // stage sequences in lockstep (cls = 1: one item per iteration).  M-items past items_m are dummies: no A loads, nothing stored.
    const int cls = c.cls, rank = cls > 1 ? (int)cluster_ctarank() : 0;
    const int it0 = (int)blockIdx.x / cls, it_stride = (int)gridDim.x / cls;
    const int total_items = ((c.items_m + cls - 1) / cls) * c.nslices;
    const uint16_t cmask = (uint16_t)((1u << cls) - 1);
    auto item_m = [&](int it) { return (it >> c.nsl_log2) * cls + rank; };

    if (warp == 0) {
        // ===== producer: one thread issues every bulk copy =====
        if (lane == 0) {
            int as = 0, aph = 0, bs = 0, bph = 0;
            const unsigned char* act = reinterpret_cast<const unsigned char*>(p.a);
            const unsigned char* wts = reinterpret_cast<const unsigned char*>(p.w);
            if (c.b_resident) {
                mbar_expect_tx(w_full, (uint32_t)c.b_total_bytes);
                const uint32_t bdst = smem_u32(b_smem);
                for (int off = 0; off < c.b_total_bytes; off += 16384) {
                    const int n = c.b_total_bytes - off < 16384 ? c.b_total_bytes - off : 16384;
                    bulk_g2s(bdst + off, wts + off, (uint32_t)n, w_full);
                }
            }
            for (int item = it0; item < total_items; item += it_stride) {
                const int im = item_m(item), ns = item & (c.nslices - 1);
                const bool dummy = im >= c.items_m;
                const size_t row0 = (size_t)p.g.base0 + (size_t)im * J * MTILE - c.halo;
                for (int s = 0; s < nslabs; ++s) {
                    mbar_wait(a_empty(as), aph ^ 1);
                    if (((c.abl & 4) && aph) || dummy) {
                        mbar_arrive(a_full(as));                      // ablation: reuse whatever the stage holds
                    } else {
                        mbar_expect_tx(a_full(as), (uint32_t)c.a_stage_bytes);
                        const uint32_t adst = smem_u32(a_smem + (size_t)as * c.a_stage_bytes);
                        for (int ch = 0; ch < chunks; ++ch)
                            bulk_g2s(adst + (uint32_t)ch * c.win_rows * 16,
                                     act + ((size_t)(s * chunks + ch) * p.g.Ptot + row0) * 16, (uint32_t)c.win_rows * 16, a_full(as));
                    }
                    if (++as == c.a_stages) { as = 0; aph ^= 1; }
                    if (!c.b_resident) {
                        for (int tap = 0; tap < p.ntaps; ++tap) {
                            mbar_wait(b_empty(bs), bph ^ 1);
                            if ((c.abl & 1) && bph) {
                                mbar_arrive(b_full(bs));              // ablation: reuse whatever the stage holds
                            } else {
                                mbar_expect_tx(b_full(bs), (uint32_t)c.b_stage_bytes);
                                const uint32_t bdst = smem_u32(b_smem + (size_t)bs * c.b_stage_bytes);
                                if (cls == 1) {
                                    for (int ch = 0; ch < chunks; ++ch)
                                        bulk_g2s(bdst + (uint32_t)ch * c.ncta * 16,
                                                 wts + (((size_t)tap * KC + s * chunks + ch) * p.N + (size_t)ns * c.ncta) * 16,
                                                 (uint32_t)c.ncta * 16, b_full(bs));
                                } else {                        // this CTA fetches every cls-th chunk for the whole cluster
                                    for (int ch = rank; ch < chunks; ch += cls)
                                        bulk_g2s_mc(bdst + (uint32_t)ch * c.ncta * 16,
                                                    wts + (((size_t)tap * KC + s * chunks + ch) * p.N + (size_t)ns * c.ncta) * 16,
                                                    (uint32_t)c.ncta * 16, b_full(bs), cmask);
                                }
                            }
                            if (++bs == c.b_stages) { bs = 0; bph ^= 1; }
                        }
                    }
                }
            }
        }
    } else if (warp <= MMA_WARPS) {
      // ===== MMA issuers: warp 1+jw owns tile jw of every item (its own accumulator columns), so up to four warps on
      // four schedulers feed the tensor pipe in parallel -- a single warp's scalar issue loop (~20 instructions per MMA)
      // is slower than the 16..64-cycle MMAs of the narrow layers.  Each warp walks the (warp-uniform) loop nest as a
      // whole, one elected lane issues; stage/accumulator barriers expect one commit per MMA warp. =====
      const int jw = warp - 1;
      if (jw < J) {
        const uint32_t leader = lane == 0;
        int as = 0, aph = 0, bs = 0, bph = 0, acs = 0, accph = 0;
        const uint32_t idesc = instr_desc_f16(MTILE, c.ncta);
        const uint32_t a_lbo = (uint32_t)c.win_rows * 16;
        const uint32_t b_lbo = (uint32_t)(c.b_resident ? p.N : c.ncta) * 16;
        // descriptors are advanced by adding 16-byte units to their 14-bit start-address field
        const uint64_t a_desc0 = smem_desc(smem_u32(a_smem), a_lbo, 128);
        const uint64_t b_desc0 = smem_desc(smem_u32(b_smem), b_lbo, 128);
        const uint32_t a_stage_u = (uint32_t)c.a_stage_bytes >> 4, b_stage_u = (uint32_t)c.b_stage_bytes >> 4;
        const uint32_t a_kk = (2 * a_lbo) >> 4, b_kk = (2 * b_lbo) >> 4;
        const uint32_t ncta = (uint32_t)c.ncta;
        if (c.b_resident) mbar_wait(w_full, 0);
        for (int item = it0; item < total_items; item += it_stride) {
            const int ns = item & (c.nslices - 1);
            mbar_wait(acc_empty(acs), accph ^ 1);
            tc_fence_after();
            const uint32_t dcol = tmem + (uint32_t)(acs * ACC_STAGE_COLS);
            for (int s = 0; s < nslabs; ++s) {
                mbar_wait(a_full(as), aph);
                tc_fence_after();
                const uint64_t ad_s = a_desc0 + (uint64_t)((uint32_t)as * a_stage_u + (uint32_t)c.halo);
                for (int tap = 0; tap < p.ntaps; ++tap) {
                    uint64_t bd;
                    if (c.b_resident) {
                        bd = b_desc0 + (uint64_t)((uint32_t)((tap * KC + s * chunks) * p.N + ns * c.ncta));
                    } else {
                        mbar_wait(b_full(bs), bph);
                        tc_fence_after();
                        bd = b_desc0 + (uint64_t)((uint32_t)bs * b_stage_u);
                    }
                    const uint64_t ad_t = ad_s + (uint64_t)(int64_t)p.off[tap];
                    tc_mma_tap<1, KK>(dcol + (uint32_t)jw * ncta, ncta, ad_t + (uint64_t)(jw * MTILE), bd, a_kk, b_kk, idesc, (uint32_t)((s | tap) != 0));
                    if (!c.b_resident) {
                        if (cls == 1) tc_commit_pred(b_empty(bs), leader); else tc_commit_mc_pred(b_empty(bs), cmask);
                        if (++bs == c.b_stages) { bs = 0; bph ^= 1; }
                    }
                }
                tc_commit_pred(a_empty(as), leader);
                if (++as == c.a_stages) { as = 0; aph ^= 1; }
            }
            tc_commit_pred(acc_full(acs), leader);
            if (++acs == 2) { acs = 0; accph ^= 1; }
        }
      }
    } else {
        // ===== epilogue: warp e owns TMEM lanes 32*(warp%4) .. +31 and every second 32-column unit of an item.
        // Lean, specialised per layer kind (EPI): EPI_PLAIN = ReLU? + fp16 copy only (first conv of a ResBlock);
        // EPI_FULL = residual / skip / fp32 stream / fp16 copy / space-to-depth / pixel-shuffle.  The fp32 residual of
        // unit u of the NEXT item is requested as soon as the registers of unit u of this item have been consumed, so
        // its HBM latency hides behind the rest of this item and the wait for the next accumulator.
        const int e = warp - EPI_WARP0, q = warp & 3, half = e >> 2;
        const int nb32 = c.ncta / 32, nu = J * nb32;
        constexpr int UPW_MAX = 4;                       // units per warp and item: nu / 2 <= 4 (J * ncta <= 256)
        const int upw = nu >> 1;
        if (half < nu) {
            int acs = 0, accph = 0;
            const Geom& g = p.g;
            const uint32_t Ptot = (uint32_t)g.Ptot;
            constexpr int UPW_PREF = 2;                      // units per warp whose residual is prefetched one item ahead
            float add[EPI != EPI_PLAIN ? UPW_PREF : 1][32];
            // row decomposition of GEMM row m: validity + absolute row (+ s2d / pixel-shuffle targets via make_row_ctx)
            auto unit_of = [&](int i) { return nu == 1 ? 0 : half + 2 * i; };
            auto issue_res = [&](int item, int i) {
                if (EPI == EPI_PLAIN || (!p.res32 && !p.res_hi) || p.mode == 1 || i >= UPW_PREF || (c.abl & 2)) return;
                const int im = item_m(item), ns = item & (c.nslices - 1);
                const int uu = unit_of(i), j = uu >> c.nb32_log2, b = uu & (nb32 - 1);
                const int m = (im * J + j) * MTILE + q * 32 + lane;
                if (m >= g.M) return;
                float* d = add[EPI != EPI_PLAIN && i < UPW_PREF ? i : 0];
                if (p.res_hi) {                  // fp16 hi/lo stream: raw packed halves, decoded at use (d[0..15] = hi, d[16..31] = lo)
                    const size_t o = (size_t)((ns * c.ncta + b * 32) >> 3) * Ptot + (g.base0 + m);
                    const uint4* sh = reinterpret_cast<const uint4*>(p.res_hi) + o;
                    const uint4* sl = reinterpret_cast<const uint4*>(p.res_lo) + o;
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        const uint4 t = __ldg(sh + (size_t)k * Ptot), u = __ldg(sl + (size_t)k * Ptot);
                        d[4 * k] = __uint_as_float(t.x); d[4 * k + 1] = __uint_as_float(t.y); d[4 * k + 2] = __uint_as_float(t.z); d[4 * k + 3] = __uint_as_float(t.w);
                        d[16 + 4 * k] = __uint_as_float(u.x); d[17 + 4 * k] = __uint_as_float(u.y); d[18 + 4 * k] = __uint_as_float(u.z); d[19 + 4 * k] = __uint_as_float(u.w);
                    }
                    return;
                }
                const float4* src = reinterpret_cast<const float4*>(p.res32) + (size_t)((ns * c.ncta + b * 32) >> 2) * Ptot + (g.base0 + m);
#pragma unroll
                for (int k = 0; k < 8; ++k) {
                    float4 t = __ldg(src + (size_t)k * Ptot);
                    d[4 * k] = t.x; d[4 * k + 1] = t.y; d[4 * k + 2] = t.z; d[4 * k + 3] = t.w;
                }
            };
            int item = it0;
            if (item < total_items) {
#pragma unroll
                for (int i = 0; i < UPW_MAX; ++i)
                    if (i < upw || (nu == 1 && i == 0)) issue_res(item, i);
            }
            for (; item < total_items; item += it_stride) {
                const int im = item_m(item), ns = item & (c.nslices - 1);
                const int nitem = item + it_stride;
                mbar_wait(acc_full(acs), accph);
                tc_fence_after();
#pragma unroll
                for (int i = 0; i < UPW_MAX; ++i) {
                    if (!(i < upw || (nu == 1 && i == 0))) continue;
                    const int uu = unit_of(i), j = uu >> c.nb32_log2, b = uu & (nb32 - 1);
                    const int n0 = ns * c.ncta + b * 32;
                    const uint32_t taddr = tmem + ((uint32_t)(q * 32) << 16) + (uint32_t)(acs * ACC_STAGE_COLS + j * c.ncta + b * 32);
                    uint32_t r0[16], r1[16];
                    tc_ld16_nowait(taddr, r0);
                    tc_ld16_nowait(taddr + 16, r1);
                    const int m = (im * J + j) * MTILE + q * 32 + lane;
                    float v[32];
                    if (EPI == EPI_PLAIN) {
                        // validity only (no s2d / scatter targets needed)
                        const uint32_t bq = div_by_magic((uint32_t)m, g.magS, g.shS), r = (uint32_t)m - bq * (uint32_t)g.S;
                        const uint32_t y = div_by_magic(r, g.magW, g.shW), x = r - y * (uint32_t)g.Wp;
                        const bool valid = m < g.M && (int)y < g.H && (int)x < g.W && !(c.abl & 2);
                        tc_ld_wait16(r0);
                        tc_ld_wait16(r1);
                        if (valid) {
#pragma unroll
                            for (int k = 0; k < 16; ++k) { v[k] = __uint_as_float(r0[k]); v[16 + k] = __uint_as_float(r1[k]); }
                            if (p.relu) {
#pragma unroll
                                for (int k = 0; k < 32; ++k) v[k] = fmaxf(v[k], 0.f);
                            }
                            uint4* dst = reinterpret_cast<uint4*>(p.out16) + (size_t)(n0 >> 3) * Ptot + (g.base0 + m);
#pragma unroll
                            for (int k = 0; k < 4; ++k) dst[(size_t)k * Ptot] = pack8_half(v + 8 * k);
                        }
                    } else {
                        RowCtx rc = make_row_ctx(p, m);
                        if (c.abl & 2) rc.valid = false;
                        float hcur[9];
                        if constexpr (EPI == EPI_HT) {
                            if (p.head_t && m < g.M) {           // 3x3 neighbourhood of the 1-channel denoiser input
                                const float* tp = p.head_t + (g.base0 + m);
#pragma unroll
                                for (int t = 0; t < 9; ++t) hcur[t] = __ldg(tp + p.off[t]);
                            }
                        }
                        tc_ld_wait16(r0);
                        tc_ld_wait16(r1);
#pragma unroll
                        for (int k = 0; k < 16; ++k) { v[k] = __uint_as_float(r0[k]); v[16 + k] = __uint_as_float(r1[k]); }
                        if (p.relu) {
#pragma unroll
                            for (int k = 0; k < 32; ++k) v[k] = fmaxf(v[k], 0.f);
                        }
                        if (p.res_hi && p.mode == 0 && m < g.M && !(c.abl & 2)) {
                            if (i < UPW_PREF) {
                                const float* d = add[EPI != EPI_PLAIN && i < UPW_PREF ? i : 0];
#pragma unroll
                                for (int k = 0; k < 16; ++k) {
                                    const float2 f = hilo_pair(__float_as_uint(d[k]), __float_as_uint(d[16 + k]));
                                    v[2 * k] += f.x; v[2 * k + 1] += f.y;
                                }
                            } else {
                                const size_t o = (size_t)(n0 >> 3) * Ptot + (g.base0 + m);
                                const uint4* sh = reinterpret_cast<const uint4*>(p.res_hi) + o;
                                const uint4* sl = reinterpret_cast<const uint4*>(p.res_lo) + o;
#pragma unroll
                                for (int k = 0; k < 4; ++k) {
                                    const uint4 t = __ldg(sh + (size_t)k * Ptot), u = __ldg(sl + (size_t)k * Ptot);
                                    const float2 f0 = hilo_pair(t.x, u.x), f1 = hilo_pair(t.y, u.y), f2 = hilo_pair(t.z, u.z), f3 = hilo_pair(t.w, u.w);
                                    v[8 * k] += f0.x; v[8 * k + 1] += f0.y; v[8 * k + 2] += f1.x; v[8 * k + 3] += f1.y;
                                    v[8 * k + 4] += f2.x; v[8 * k + 5] += f2.y; v[8 * k + 6] += f3.x; v[8 * k + 7] += f3.y;
                                }
                            }
                        } else if (p.res32 && p.mode == 0 && m < g.M && !(c.abl & 2)) {
                            if (i < UPW_PREF) {
#pragma unroll
                                for (int k = 0; k < 32; ++k) v[k] += add[EPI != EPI_PLAIN && i < UPW_PREF ? i : 0][k];
                            } else {                        // units beyond the prefetch depth (streamed-weight layers): load at use
                                const float4* src = reinterpret_cast<const float4*>(p.res32) + (size_t)(n0 >> 2) * Ptot + (g.base0 + m);
#pragma unroll
                                for (int k = 0; k < 8; ++k) {
                                    float4 t = __ldg(src + (size_t)k * Ptot);
                                    v[4 * k] += t.x; v[4 * k + 1] += t.y; v[4 * k + 2] += t.z; v[4 * k + 3] += t.w;
                                }
                            }
                        }
                        if (!c.late_pf && nitem < total_items) issue_res(nitem, i);          // registers of unit i are free again
                        if constexpr (EPI == EPI_FULL) {
                            if (p.mode == 1) {                   // transposed conv: lane-paired pixel-shuffle stores
                                epi_up_unit(p, rc.valid, rc.frow0, n0, v, reinterpret_cast<float4*>(smem + c.aux_off) + e * 256);
                                continue;
                            }
                        }
                        if constexpr (EPI == EPI_HT) {
                            constexpr int HN = 128 / J;
                            if (p.head_t) {                      // + m_head(t)[n0 .. n0+31] (rows that are not stored may hold anything)
                                if (HN == 32 || n0 == 0) ht_head<HN, 0>(htw.head, hcur, v);
                                else ht_head<HN, HN == 32 ? 0 : 32>(htw.head, hcur, v);
                            }
                            if (p.tail_part) {                   // 9 per-tap partial sums of m_tail instead of the 32 channels
                                if (rc.valid) {
                                    float* dst = p.tail_part + (size_t)((n0 >> 5) * 9) * Ptot + rc.row;
                                    if (HN == 32 || n0 == 0) ht_tail<HN, 0>(htw.tail, v, dst, Ptot);
                                    else ht_tail<HN, HN == 32 ? 0 : 32>(htw.tail, v, dst, Ptot);
                                }
                                continue;
                            }
                        }
                        if (rc.valid) {
                            const EpiAddr a0 = epi_addr(p, rc, n0), a1 = epi_addr(p, rc, n0 + 16);
                            if (p.skip32) {
                                float sk[32];
                                epi_load16_one(p.skip32, a0, sk); epi_load16_one(p.skip32, a1, sk + 16);
#pragma unroll
                                for (int k = 0; k < 32; ++k) v[k] += sk[k];
                            }
                            epi_out16(p, rc, a0, n0, v);
                            epi_out16(p, rc, a1, n0 + 16, v + 16);
                        }
                    }
                }
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(acc_empty(acs));
                if (++acs == 2) { acs = 0; accph ^= 1; }
                // A warp has six load scoreboards: a prefetch issued between two units makes the second unit's first use of ITS
                // (long landed) registers wait for the new loads too.  So the next item's loads go out together, here.
                if (EPI != EPI_PLAIN && c.late_pf && nitem < total_items) {
#pragma unroll
                    for (int i = 0; i < UPW_MAX; ++i)
                        if (i < upw || (nu == 1 && i == 0)) issue_res(nitem, i);
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (c.cls > 1) cluster_sync_all();             // no CTA leaves while a peer may still multicast into it or signal its barriers
    if (warp == 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(TMEM_COLS) : "memory");
    }
}

static int g_num_sms = 0;
static int g_cluster = 4;
static int g_late_pf = -1;     // request the next item's residual after the LAST unit of this item (1) or after each unit (0);
                               // -1 (default): late for the streamed-weight layers (levels 3-4: 327 -> 297 us, 456 -> 396 us), early for
                               // the resident ones (level 1 tail conv: 708 vs 794 us), GDECONV_LATEPF overrides
static int g_bstages = 6;
constexpr int A_STAGES = 4;    // A ring depth: deeper rings measured slower everywhere (profiles/README_r01.md)
static int g_abl = 0;

// Optional per-launch timing of k_conv_umma with CUDA events on the launching stream (gd_profile_begin/end):
// bench.py uses it to measure the dominant kernel's average duration live for the roofline line.
struct ConvTiming {
    bool on = false;
    std::vector<cudaEvent_t> pool;
    size_t used = 0;
    std::vector<double> flops;
    cudaEvent_t get() {
        if (used == pool.size()) { cudaEvent_t e; cudaEventCreate(&e); pool.push_back(e); }
        return pool[used++];
    }
};
static ConvTiming g_timing;

void conv_profile_begin() { g_timing.on = true; g_timing.used = 0; g_timing.flops.clear(); }
int conv_profile_end(double* ms_total, double* flops_total, unsigned long long* launches) {
    g_timing.on = false;
    double ms = 0, fl = 0;
    for (size_t i = 0; i + 1 < g_timing.used; i += 2) {
        GD_CUDA_CHECK(cudaEventSynchronize(g_timing.pool[i + 1]));
        float t = 0;
        GD_CUDA_CHECK(cudaEventElapsedTime(&t, g_timing.pool[i], g_timing.pool[i + 1]));
        ms += t; fl += g_timing.flops[i / 2];
    }
    if (ms_total) *ms_total = ms;
    if (flops_total) *flops_total = fl;
    if (launches) *launches = g_timing.used / 2;
    return GD_OK;
}

// Timing hook for the other tcgen05 conv kernels (conv_l1chain.cu, conv_l2chain.cu): records the start event and returns the stop event to record.
int conv_profile_mark(double flops, cudaStream_t st, cudaEvent_t* stop) {
    *stop = nullptr;
    if (!g_timing.on) return GD_OK;
    cudaEvent_t e0 = g_timing.get();
    *stop = g_timing.get();
    g_timing.flops.push_back(flops);
    GD_CUDA_CHECK(cudaEventRecord(e0, st));
    return GD_OK;
}

int conv_umma_init() {
    int dev;
    GD_CUDA_CHECK(cudaGetDevice(&dev));
    GD_CUDA_CHECK(cudaDeviceGetAttribute(&g_num_sms, cudaDevAttrMultiProcessorCount, dev));
    if (const char* e = getenv("GDECONV_ABL")) g_abl = atoi(e);
    if (const char* e = getenv("GDECONV_LATEPF")) g_late_pf = atoi(e);
    if (const char* e = getenv("GDECONV_CLUSTER")) { g_cluster = atoi(e); if (g_cluster != 1 && g_cluster != 2 && g_cluster != 4) g_cluster = 4; }
    if (const char* e = getenv("GDECONV_BSTAGES")) { g_bstages = atoi(e); if (g_bstages < 2 || g_bstages > MAX_B_STAGES) g_bstages = 6; }
#define GD_UMMA_ATTR(J, KK)                                                                                                        \
    GD_CUDA_CHECK(cudaFuncSetAttribute(k_conv_umma<J, KK, EPI_PLAIN>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)UMMA_SMEM_MAX)); \
    GD_CUDA_CHECK(cudaFuncSetAttribute(k_conv_umma<J, KK, EPI_FULL>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)UMMA_SMEM_MAX))
    GD_UMMA_ATTR(1, 2); GD_UMMA_ATTR(2, 2); GD_UMMA_ATTR(4, 2); GD_UMMA_ATTR(1, 4); GD_UMMA_ATTR(2, 4); GD_UMMA_ATTR(4, 4);
#undef GD_UMMA_ATTR
    GD_CUDA_CHECK(cudaFuncSetAttribute(k_conv_umma<2, 2, EPI_HT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)UMMA_SMEM_MAX));
    return GD_OK;
}

static int make_cfg(const ConvParams& p, UmmaCfg* out) {
    UmmaCfg c;
    memset(&c, 0, sizeof(c));
    if (p.N % 32 || p.Kt % 16) { set_error("conv_umma: N=%d must be a multiple of 32 and K=%d of 16", p.N, p.Kt); return GD_EUNSUPPORTED; }
    c.ncta = p.N < 128 ? p.N : 128;
    if (p.N % c.ncta) { set_error("conv_umma: N=%d is not a multiple of %d", p.N, c.ncta); return GD_EUNSUPPORTED; }
    c.nslices = p.N / c.ncta;
    c.BK = (p.Kt % 64 == 0 && (size_t)p.ntaps * p.Kt * p.N * 2 > B_RESIDENT_MAX) ? 64 : 32;   // streamed weights: 64-channel slabs
    if (p.Kt % c.BK) { set_error("conv_umma: K=%d must be a multiple of 32", p.Kt); return GD_EUNSUPPORTED; }
    c.halo = p.ntaps == 9 ? p.g.Wp + 1 : 0;
    c.b_total_bytes = p.ntaps * p.Kt * p.N * 2;
    c.b_resident = (size_t)c.b_total_bytes <= B_RESIDENT_MAX;
    c.b_stage_bytes = c.ncta * c.BK * 2;
    c.b_stages = c.b_resident ? 0 : g_bstages;
    size_t b_region = c.b_resident ? (size_t)c.b_total_bytes : (size_t)c.b_stages * c.b_stage_bytes;
    if (p.head_t || p.tail_part) {                // EPI_HT (weights are kernel parameters)
        if (p.mode != 0 || p.ntaps != 9 || p.N != 64 || p.skip32 || p.s2d || (p.head_t && !p.head_w) || (p.tail_part && !p.tail_w)) {
            set_error("conv_umma: head/tail fusion needs a 3x3 level-0 layer with N = 64"); return GD_EUNSUPPORTED;
        }
    } else if (p.mode == 1) {
        c.aux_off = (int)((b_region + 127) / 128 * 128);
        b_region = (size_t)c.aux_off + (size_t)EPI_WARPS * 4096;
    }
    // resident weights: <= 128 accumulator columns per item (2 epilogue units per warp, fine-grained A ring, good tail
    // balance); streamed weights: 256 columns so that every weight stage is reused by twice as many rows
    c.J = (c.b_resident ? 128 : ACC_STAGE_COLS) / c.ncta;
    if (c.J > 4) c.J = 4;
    for (;; c.J >>= 1) {
        c.win_rows = MTILE * c.J + 2 * c.halo;
        c.a_stage_bytes = c.win_rows * c.BK * 2;
        if (b_region + 2 * (size_t)c.a_stage_bytes <= UMMA_SMEM_MAX || c.J == 1) break;
    }
    c.a_stages = (int)((UMMA_SMEM_MAX - b_region) / c.a_stage_bytes);
    if (c.a_stages > A_STAGES) c.a_stages = A_STAGES;
    if (c.a_stages < 2) { set_error("conv_umma: layer does not fit shared memory"); return GD_EUNSUPPORTED; }
    c.smem = (size_t)c.a_stages * c.a_stage_bytes + b_region;
    if (p.mode == 1) c.aux_off += c.a_stages * c.a_stage_bytes;     // relative to the start of dynamic smem
    const int tiles = (p.g.M + MTILE - 1) / MTILE;
    c.items_m = (tiles + c.J - 1) / c.J;
    c.abl = g_abl;
    c.cls = (!c.b_resident && (c.BK / 8) % g_cluster == 0) ? g_cluster : 1;
    c.late_pf = g_late_pf < 0 ? !c.b_resident : g_late_pf != 0;
    auto ilog2 = [](int v) { int l = 0; while ((1 << l) < v) ++l; return l; };
    c.nsl_log2 = ilog2(c.nslices); c.nb32_log2 = ilog2(c.ncta / 32);
    if ((1 << c.nsl_log2) != c.nslices || (1 << c.nb32_log2) != c.ncta / 32) { set_error("conv_umma: N=%d must split into power-of-two slices", p.N); return GD_EUNSUPPORTED; }
    *out = c;
    return GD_OK;
}

int launch_conv_umma(const ConvParams& p, cudaStream_t st) {
    if (p.g.M <= 0) return GD_OK;
    UmmaCfg c;
    int rc = make_cfg(p, &c);
    if (rc != GD_OK) return rc;
    if (!g_num_sms) { set_error("conv_umma: library not initialised"); return GD_ECUDA; }
    const int iters = ((c.items_m + c.cls - 1) / c.cls) * c.nslices;              // kernel-wide iteration list (see k_conv_umma)
    int grid = (iters < g_num_sms / c.cls ? iters : g_num_sms / c.cls) * c.cls;   // cls > 1: refined below by the cluster occupancy
    cudaEvent_t e1 = nullptr;
    if (g_timing.on) {
        cudaEvent_t e0 = g_timing.get();
        e1 = g_timing.get();
        // algorithmic FLOPs: 2*K*N per tap and VALID output pixel (halo rows of the padded-linear layout excluded)
        g_timing.flops.push_back(2.0 * (double)(p.g.M / p.g.S) * p.g.H * p.g.W * (double)p.N * p.Kt * p.ntaps);
        GD_CUDA_CHECK(cudaEventRecord(e0, st));
    }
    const int KK = c.BK / 16;
    const bool ht = p.head_t || p.tail_part;
    const bool plain = p.mode == 0 && !p.res32 && !p.res_hi && !p.out_lo && !p.skip32 && !p.out32 && !p.s2d && p.out16 && !ht;
    // Launch helper: plain launch, or (streamed weights) clusters of c.cls CTAs with as many clusters as can be co-resident
    auto go = [&](auto kern, auto hw) -> int {
        if (c.cls == 1) { kern<<<grid, UMMA_THREADS, c.smem, st>>>(p, c, hw); return GD_OK; }
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3((unsigned)grid); cfg.blockDim = dim3(UMMA_THREADS); cfg.dynamicSmemBytes = c.smem; cfg.stream = st;
        cudaLaunchAttribute at[1];
        at[0].id = cudaLaunchAttributeClusterDimension;
        at[0].val.clusterDim.x = (unsigned)c.cls; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
        cfg.attrs = at; cfg.numAttrs = 1;
        static std::map<std::pair<const void*, int>, int> max_clusters;      // per (kernel, cluster size)
        static std::mutex mu;
        int max_cl;
        {
            std::lock_guard<std::mutex> lk(mu);
            auto key = std::make_pair((const void*)kern, c.cls);
            auto it = max_clusters.find(key);
            if (it == max_clusters.end()) {
                int n = 0;
                cfg.gridDim = dim3((unsigned)(g_num_sms / c.cls * c.cls));
                GD_CUDA_CHECK(cudaOccupancyMaxActiveClusters(&n, kern, &cfg));
                if (n < 1) { set_error("conv_umma: no cluster of %d CTAs fits", c.cls); return GD_ECUDA; }
                it = max_clusters.emplace(key, n).first;
            }
            max_cl = it->second;
        }
        const int clusters = iters < max_cl ? iters : max_cl;
        cfg.gridDim = dim3((unsigned)(clusters * c.cls));
        GD_CUDA_CHECK(cudaLaunchKernelEx(&cfg, kern, p, c, hw));
        return GD_OK;
    };
#define GD_UMMA_GO(JJ, KKK)                                                                         \
    if (c.J == JJ && KK == KKK && !ht) {                                                            \
        int rc2;                                                                                    \
        if (plain) rc2 = go(k_conv_umma<JJ, KKK, EPI_PLAIN>, HtWeights<EPI_PLAIN, 128 / JJ>());     \
        else rc2 = go(k_conv_umma<JJ, KKK, EPI_FULL>, HtWeights<EPI_FULL, 128 / JJ>());             \
        if (rc2 != GD_OK) return rc2;                                                               \
    } else
#define GD_UMMA_GO_HT(JJ, KKK)                                                                      \
    if (c.J == JJ && KK == KKK && ht && p.N == 128 / JJ) {                                          \
        HtWeights<EPI_HT, 128 / JJ> hw;                                                             \
        memset(&hw, 0, sizeof(hw));                                                                 \
        if (p.head_t) memcpy(hw.head, p.head_w, sizeof(hw.head));                                   \
        if (p.tail_part) memcpy(hw.tail, p.tail_w, sizeof(hw.tail));                                \
        k_conv_umma<JJ, KKK, EPI_HT><<<grid, UMMA_THREADS, c.smem, st>>>(p, c, hw);                 \
    } else
    GD_UMMA_GO_HT(2, 2)
    GD_UMMA_GO(1, 2) GD_UMMA_GO(2, 2) GD_UMMA_GO(4, 2) GD_UMMA_GO(1, 4) GD_UMMA_GO(2, 4) GD_UMMA_GO(4, 4)
    { set_error("conv_umma: no kernel variant for J=%d, BK=%d", c.J, c.BK); return GD_EUNSUPPORTED; }
#undef GD_UMMA_GO
#undef GD_UMMA_GO_HT
    GD_LAUNCHED();
    if (e1) GD_CUDA_CHECK(cudaEventRecord(e1, st));
    return GD_OK;
}

}  // namespace gd
