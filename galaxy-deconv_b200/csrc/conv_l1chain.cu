// Level-0 chain kernels of the ResUNet denoiser (32 channels at 48x48, models/ResUNet.py:31-32 and :38-39), tcgen05 path:
//
//   DOWN:  x1 = m_head(t);  x = ResBlock(ResBlock(x1))                  -> space-to-depth copy for the m_down1 strided conv
//   UP:    x  = ResBlock(ResBlock(m_up1's transposed conv of the level-1 map))  -> per-tap m_tail partial sums (k_tail_gather)
//
// i.e. FOUR 3x3 convolutions (two `x + conv(ReLU(conv(x)))` blocks, models/resnet_basicblock.py:69-71) per launch with every
// intermediate on chip.  Why: at this level one conv per launch is HBM-bound (768 MB per 32-channel fp16 map of 5000 stamps), and
// even a kernel that runs one whole ResBlock per launch moves 3.1 GB per block for 0.3 ms of tensor work.  Here a work item is HALF A
// STAMP (24 output rows + the 4 rows of halo the four convs need = a 28-row window, 1372 rows of the padded-linear layout):
//   * the fp16 operand copies of the stream (X) and of ReLU(conv1) (T) live in shared memory, two buffers of 4 chunk planes
//     x 1428 rows x 16 B; planes are separated by 56 zero rows that are never written, which serve as the zero row above /
//     below the stamp and absorb the tap shifts of the first / last tile;
//   * the fp32 residual stream lives in TENSOR MEMORY (10 tiles x 32 columns): the second conv of a block adds its
//     accumulator to it in the epilogue (tcgen05.ld + tcgen05.st), nothing is rounded to fp16 on the residual path;
//   * conv accumulators: 2 stages x 3 tiles x 32 TMEM columns: the three tiles of a unit are issued by three warps in parallel
//     and the epilogue of a unit overlaps the MMAs of the next one;
//   * weights (18 KB per conv) stream through two shared-memory slots, one layer ahead.
// The halo is RECOMPUTED (layer l of a top item is valid on rows y < 27 - l, mirrored for bottom items): 41 tiles of MMA work per
// item for 36.75 tiles of output, no inter-CTA exchange.  Tiles are 128 consecutive padded-linear rows; a tile of layer l+1
// is issued as soon as the epilogues of the layer-l tiles under its 3x3 footprint have arrived (per-tile mbarriers), so the
// tensor pipe never drains at a layer boundary.
//
// Tried and rejected in round 2 (profiles/README_r02.md): concatenating the three dx taps of a kernel row along N (three N = 96 MMAs
// per K16 step on one A window instead of nine N = 32 ones, the epilogue adding the neighbouring lanes' partial sums by warp
// shuffles + a shared-memory exchange at warp boundaries).  Bit-for-bit the same results and a third of the A-operand fetches,
// but the epilogue grew to ~575 instructions per tile and warp (64 shuffles, 64 adds, hi/lo conversions of the then packed
// stream) and became the bound: 2.3 ms per launch instead of 1.5 ms.
//
// Warp roles (512 threads, one persistent CTA per SM):
//   warp 0      producer: weight slots; UP: the item's hi -> X and lo -> T windows; DOWN: 29 rows of t (bulk async copies)
//   warps 1-3   MMA issuers, warp 1 + j owns tile j of every 3-tile unit (one elected lane each, straight-line 18 MMAs); warp 1 allocates TMEM
//   warps 4-7   helpers (one per TMEM lane quarter): DOWN: x1 = m_head(t) in fp32 on CUDA cores -> X (fp16) + stream (TMEM);
//               UP: stream = hi + lo
//   warps 8-15  epilogue: two groups of four (one warp per lane quarter), alternating units
#include "conv_epilogue.cuh"
#include "kernels.cuh"
#include "launch.cuh"
#include "umma_ptx.cuh"

#include <cstdlib>
#include <cstring>

namespace gd {

constexpr int LC_C = 32;
constexpr int LC_WP = 49;                            // padded row length at 48x48
constexpr int LC_WIN_Y = 28;                         // image rows per item window
constexpr int LC_ROWS = LC_WIN_Y * LC_WP;            // 1372
constexpr int LC_GAP = 56;                           // zero rows between planes (>= Wp + 1)
constexpr int LC_PSTRIDE = LC_ROWS + LC_GAP;         // 1428
constexpr int LC_ACT_BYTES = (8 * LC_PSTRIDE + LC_GAP) * 16;    // 183,680: planes 0-3 = X, 4-7 = T
constexpr int LC_W_BYTES = 9 * LC_C * LC_C * 2;      // 18,432
constexpr int LC_TWIN_ROWS = 29;                     // image rows of the 1-channel input a DOWN item needs (window + 1 row of halo, clipped)
constexpr int LC_TWIN_BYTES = LC_TWIN_ROWS * STAMP * 4;          // 5,568
constexpr int LC_SMEM = LC_ACT_BYTES + 2 * LC_W_BYTES + 5632;   // 226,176
constexpr int LC_BOT_Y0 = 20;                        // first image row of a bottom item's window
constexpr int LC_BOT = LC_ROWS - 10 * MTILE;         // 92: first row of the 10-tile grid of a bottom item
constexpr int LC_OWN = 24 * LC_WP;                   // 1176 rows of final output per item
constexpr int LC_THREADS = (1 + 3 + 4 + 8) * 32;      // producer, LC_J MMA warps, 4 helpers, 8 epilogue warps
constexpr int LC_STREAM_TILES = 10;
constexpr int LC_J = 3;                              // tiles per MMA unit = MMA-issuing warps
constexpr int LC_ACC_COL = LC_STREAM_TILES * LC_C;   // 320: two accumulator stages of LC_J x 32 columns follow the stream (512 in all)
constexpr int LC_HEAD_TILES = 11;
// DOWN: the m_down1 strided conv (k2 s2, 32 -> 64 channels; models/resnet_basicblock.py:73-79) runs in the same kernel: the epilogue of
// the 4th conv writes the item's own 24 rows as a space-to-depth operand [16 chunks][304 coarse rows][8] over the (then idle) X
// planes, three M128 N64 K128 GEMM tiles follow, and their epilogue stores x2 = the level-1 skip (fp32) + its fp16 operand copy.
constexpr int LC_SR = 304;                           // rows per chunk plane of the space-to-depth operand (12 coarse rows x 25 = 300 used)
constexpr int LC_WD_BYTES = 4 * LC_C * 2 * LC_C * 2; // 16,384: packed strided-conv weights [16][64][8]
constexpr int LC_DN = 2 * LC_C;                      // 64 output channels
// UP: the m_up1 transposed conv (k2 s2, 64 -> 32 channels; models/resnet_basicblock.py:81-87) runs in the same kernel: the 14 coarse
// rows x 25 of the level-1 map the item needs are bulk-copied over the (then idle) first two T planes, three M128 N128 K64 GEMM
// tiles (N = 4 sub-pixels x 32 channels) go to TMEM columns [0, 384), and their epilogue scatters hi = rn16(x) into the X planes
// and lo = rn16(x - hi) into a per-CTA global scratch (L2-resident, 88 KB) from which the helpers build the fp32 stream
// -- the accumulator's lanes are coarse pixels, the stream's lanes fine rows, so the fp32 values have to change lanes somewhere.
constexpr int LC_AR = 352;                           // rows per chunk plane of the transposed conv's A operand (350 used)
constexpr int LC_A_BYTES = 8 * LC_AR * 16;           // 45,056
constexpr int LC_WU_BYTES = 2 * LC_C * 4 * LC_C * 2; // 16,384: packed transposed-conv weights [8][128][8], n = (dy*2+dx)*32 + co
constexpr int LC_SCRATCH_BYTES = LC_ROWS * 64;       // per CTA: lo halves of the transposed conv's output, [row][32] fp16

enum { LCB_W_FULL = 0, LCB_W_EMPTY = 2, LCB_ACC_FULL = 4, LCB_ACC_EMPTY = 6, LCB_X_FULL = 8, LCB_T_FULL = 9, LCB_X_FREE = 10,
       LCB_T_FREE = 11, LCB_ITEM_DONE = 12, LCB_X_READY = 13, LCB_TILE_DONE = LCB_X_READY + LC_HEAD_TILES, LCB_S_READY = LCB_TILE_DONE + 4 * 11,
       LCB_TWIN_FULL = LCB_S_READY + LC_STREAM_TILES, LCB_TWIN_EMPTY, LCB_DOWN_FULL, LCB_DOWN_EMPTY, LCB_CONVT_FULL, LCB_CONVT_DONE, LCB_COUNT };

struct L1ChainParams {
    int nb;                        // stamps
    Geom g0, g1;                   // level 0 (48x48) and level 1 (24x24) geometry of the chunk
    const float* t;                // DOWN: scaled denoiser input [nb][48*48]
    const void* x_in;              // UP: fp16 level-1 map (input of m_up1's transposed conv) [8][g1.Ptot][8]
    const void* wup;               // UP: packed transposed-conv weights [8][128][8]
    unsigned char* scratch;        // UP: gridDim.x * LC_SCRATCH_BYTES of global scratch (zero-initialised once: pad rows are never written)
    const void* w[4];              // packed 3x3 weights [tap][4][32][8]: block 1 conv 1, conv 2, block 2 conv 1, conv 2
    const void* wdown;             // DOWN: packed strided-conv weights [16][64][8] (K = (dy*2+dx)*32 + ci)
    float* skip32;                 // DOWN: x2 fp32 [16][g1.Ptot][4] (U-Net skip + residual of the next level)
    void* x2_16;                   // DOWN: x2 fp16 [8][g1.Ptot][8] (operand of the next conv)
    void* x2_lo;                   // DOWN, optional: rn16(x2 - fp16(x2)), same layout (lo half of the stream read by conv_l2chain.cu)
    float* tail_part;              // UP: [9][g0.Ptot] per-tap m_tail partial sums
};
struct L1ChainHT { float head[9 * LC_C], tail[9 * LC_C]; };

__device__ __forceinline__ int lc_ntiles(int L) { return L == 0 ? 11 : 10; }
// tile i of layer L (0..3) of a top (h = 0) / bottom (h = 1) item: first row r and the rows [wlo, whi) its epilogue writes
__device__ __forceinline__ void lc_tile(int L, int h, int i, int& r, int& wlo, int& whi) {
    if (h == 0) {
        if (L == 0 && i == 10) { r = 27 * LC_WP - MTILE; wlo = 10 * MTILE; whi = 27 * LC_WP; }      // overlaps tile 9: writes only the new rows
        else { r = MTILE * i; wlo = r; whi = r + MTILE; }
    } else {
        if (L == 0) {
            if (i == 0) { r = LC_WP; wlo = LC_WP; whi = LC_BOT; }
            else { r = LC_BOT + MTILE * (i - 1); wlo = r; whi = r + MTILE; }
        } else { r = LC_BOT + MTILE * i; wlo = r; whi = r + MTILE; }
    }
}
__device__ __forceinline__ int lc_tile_start(int L, int h, int i) { int r, a, b; lc_tile(L, h, i, r, a, b); return r; }
__device__ __forceinline__ int lc_stream_start(int h, int i) { return (h ? LC_BOT : 0) + MTILE * i; }
__device__ __forceinline__ int lc_head_start(int h, int j) { return (h ? LC_BOT - MTILE : 0) + MTILE * j; }

// 9 per-tap partial sums of m_tail over the 32 channels of one row (weights = constant-bank operands)
__device__ __forceinline__ void lc_tail(const float* __restrict__ tw, const float* v, float* dst, size_t Ptot) {
#pragma unroll
    for (int t = 0; t < 9; ++t) {
        float s[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int k = 0; k < 32; ++k) s[k & 3] = fmaf(v[k], tw[t * LC_C + k], s[k & 3]);
        dst[(size_t)t * Ptot] = (s[0] + s[1]) + (s[2] + s[3]);
    }
}

template <int MODE>      // 0 = DOWN, 1 = UP
__global__ void __launch_bounds__(LC_THREADS, 1) k_l1_chain(const L1ChainParams p, const __grid_constant__ L1ChainHT htw) {
    extern __shared__ __align__(128) unsigned char smem[];
    __shared__ __align__(8) uint64_t bars[LCB_COUNT];
    __shared__ uint32_t tmem_slot;
    const int warp = __shfl_sync(0xffffffffu, threadIdx.x >> 5, 0), lane = threadIdx.x & 31;
    unsigned char* w_smem = smem + LC_ACT_BYTES;
    const float* twin = reinterpret_cast<const float*>(smem + LC_ACT_BYTES + 2 * LC_W_BYTES);   // DOWN: rows [ylo, ylo + 29) of the item's stamp of t
    const uint32_t bar0 = smem_u32(bars);
    auto bar = [&](int i) { return bar0 + 8u * (uint32_t)i; };

    if (threadIdx.x == 0) {
        for (int s = 0; s < 2; ++s) {
            mbar_init(bar(LCB_W_FULL + s), 1); mbar_init(bar(LCB_W_EMPTY + s), LC_J);
            mbar_init(bar(LCB_ACC_FULL + s), LC_J); mbar_init(bar(LCB_ACC_EMPTY + s), 4);
        }
        mbar_init(bar(LCB_X_FULL), 1); mbar_init(bar(LCB_T_FULL), 1); mbar_init(bar(LCB_X_FREE), LC_J); mbar_init(bar(LCB_T_FREE), LC_J);
        mbar_init(bar(LCB_ITEM_DONE), 8);
        for (int j = 0; j < LC_HEAD_TILES; ++j) mbar_init(bar(LCB_X_READY + j), 4);
        for (int j = 0; j < 44; ++j) mbar_init(bar(LCB_TILE_DONE + j), 4);
        mbar_init(bar(LCB_DOWN_FULL), LC_J); mbar_init(bar(LCB_DOWN_EMPTY), 8);
        mbar_init(bar(LCB_CONVT_FULL), LC_J); mbar_init(bar(LCB_CONVT_DONE), 8);
        for (int j = 0; j < LC_STREAM_TILES; ++j) mbar_init(bar(LCB_S_READY + j), 4);
        mbar_init(bar(LCB_TWIN_FULL), 1); mbar_init(bar(LCB_TWIN_EMPTY), 4);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_slot)), "r"(TMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    {   // zero the activation planes once: the gaps and the pad pixels (x = 48) are never written afterwards
        uint4* z = reinterpret_cast<uint4*>(smem);
        for (int i = threadIdx.x; i < LC_ACT_BYTES / 16; i += blockDim.x) z[i] = make_uint4(0u, 0u, 0u, 0u);
        fence_proxy_async_smem();
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = tmem_slot;
    const int total_items = 2 * p.nb;
    const int n_my = total_items > (int)blockIdx.x ? (total_items - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x : 0;
    const uint32_t Ptot0 = (uint32_t)p.g0.Ptot;
    constexpr int NLAYERS = 5;                    // weight layers per item: DOWN: conv 0-3, strided conv; UP: transposed conv, conv 0-3
    constexpr int L0_IDX = MODE == 0 ? 0 : 1;     // position of conv 0 in that sequence
    unsigned char* scratch = MODE == 1 ? p.scratch + (size_t)blockIdx.x * LC_SCRATCH_BYTES : nullptr;
    // byte offset of row s of plane pl inside the activation region
    auto row_off = [](int pl, int s) { return (uint32_t)((pl * LC_PSTRIDE + LC_GAP + s) * 16); };

    // DOWN: x1 = m_head(t) of local row s of a top (h = 0) / bottom (h = 1) item from the t window in shared memory (zeros outside the
    // window / on pad pixels); weights are constant-bank operands
    auto head_row = [&](int h, int s, float* acc) -> bool {
        const int ylo = h ? LC_BOT_Y0 - 1 : 0;                   // first image row held by the t window
        const int yq = s >= 0 ? (s * 1338) >> 16 : 0, x = s - yq * LC_WP;
        const bool inimg = s >= 0 && s < LC_ROWS && x < STAMP;
        const int y = h * LC_BOT_Y0 + yq;
        float in[9];
#pragma unroll
        for (int dy = -1; dy <= 1; ++dy)
#pragma unroll
            for (int dx = -1; dx <= 1; ++dx) {
                const int yy = y + dy, xx = x + dx;
                in[(dy + 1) * 3 + dx + 1] = (inimg && yy >= 0 && yy < STAMP && xx >= 0 && xx < STAMP) ? twin[(yy - ylo) * STAMP + xx] : 0.f;
            }
#pragma unroll
        for (int c = 0; c < LC_C; ++c) acc[c] = 0.f;
#pragma unroll
        for (int tp = 0; tp < 9; ++tp)
#pragma unroll
            for (int c = 0; c < LC_C; ++c) acc[c] = fmaf(in[tp], htw.head[tp * LC_C + c], acc[c]);
        return inimg;
    };
    // DOWN, X fill: head tile j (128 rows) by the four warps of one set (q = TMEM-independent quarter index).  The space-to-depth
    // operand of the previous item overwrote pad pixels and inter-plane gaps of X, so from the second item on every row is rewritten
    // (zeros where there is no pixel).  The fill (~900 cycles per tile on the four helper warps) can no longer overlap the previous
    // item's last conv, because the strided conv's operand occupies X until then: measured, the in-kernel strided conv costs 0.33 ms
    // per launch and replaces a 0.45 ms launch + 1.5 GB of HBM traffic (sharing the fill with the epilogue warps was slower still).
    auto fill_x_tile = [&](int h, int k, int j, int q) {
        const int s = lc_head_start(h, j) + q * 32 + lane;
        float acc[LC_C];
        const bool inimg = head_row(h, s, acc);
        if (inimg || (k > 0 && s >= 0 && s < LC_PSTRIDE)) {
#pragma unroll
            for (int ch = 0; ch < 4; ++ch) *reinterpret_cast<uint4*>(smem + row_off(ch, s)) = pack8_half(acc + 8 * ch);
        }
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) mbar_arrive(bar(LCB_X_READY + j));
    };

    if (warp == 0) {
        // ===== producer =====
        if (lane == 0) {
            // weight layers of an item (NLAYERS = 5): layer counter Lc picks the slot.  idx = position in the item's sequence
            auto load_w = [&](int k, int idx, const void* srcp, uint32_t bytes) {
                const int Lc = NLAYERS * k + idx, slot = Lc & 1;
                mbar_wait(bar(LCB_W_EMPTY + slot), ((Lc >> 1) & 1) ^ 1);
                mbar_expect_tx(bar(LCB_W_FULL + slot), bytes);
                const uint32_t dst = smem_u32(w_smem) + (uint32_t)slot * LC_W_BYTES;
                const unsigned char* src = reinterpret_cast<const unsigned char*>(srcp);
                bulk_g2s(dst, src, bytes / 2, bar(LCB_W_FULL + slot));
                bulk_g2s(dst + bytes / 2, src + bytes / 2, bytes / 2, bar(LCB_W_FULL + slot));
            };
            for (int k = 0; k < n_my; ++k) {
                const int it = (int)blockIdx.x + k * (int)gridDim.x;
                if (MODE == 0) {       // 29 image rows of the 1-channel input: rows 0..28 (top item) or 19..47 (bottom item)
                    mbar_wait(bar(LCB_TWIN_EMPTY), (k & 1) ^ 1);
                    mbar_expect_tx(bar(LCB_TWIN_FULL), (uint32_t)LC_TWIN_BYTES);
                    bulk_g2s(smem_u32(twin), p.t + (size_t)(it >> 1) * NPIX + (size_t)((it & 1) ? (LC_BOT_Y0 - 1) * STAMP : 0), (uint32_t)LC_TWIN_BYTES,
                             bar(LCB_TWIN_FULL));
                    for (int L = 0; L < 4; ++L) load_w(k, L, p.w[L], (uint32_t)LC_W_BYTES);
                    load_w(k, 4, p.wdown, (uint32_t)LC_WD_BYTES);
                } else {
                    load_w(k, 0, p.wup, (uint32_t)LC_WU_BYTES);
                    // A operand of the transposed conv: coarse rows [0, 14) (top) / [10, 24) (bottom) of the stamp's level-1 map -> T planes
                    mbar_wait(bar(LCB_T_FREE), (k & 1) ^ 1);                     // the previous item's 4th conv has finished reading T
                    const size_t row0 = (size_t)p.g1.base0 + (size_t)(it >> 1) * p.g1.S + (size_t)((it & 1) ? 250 : 0);
                    mbar_expect_tx(bar(LCB_T_FULL), 8u * 350u * 16u);
#pragma unroll
                    for (int ch = 0; ch < 8; ++ch)
                        bulk_g2s(smem_u32(smem) + row_off(4, 0) + (uint32_t)(ch * LC_AR * 16),
                                 reinterpret_cast<const unsigned char*>(p.x_in) + ((size_t)ch * p.g1.Ptot + row0) * 16, 350u * 16u, bar(LCB_T_FULL));
                    for (int L = 0; L < 4; ++L) load_w(k, 1 + L, p.w[L], (uint32_t)LC_W_BYTES);
                }
            }
        }
    } else if (warp <= LC_J) {
        // ===== MMA issuers: warp 1 + jw owns tile jw of every unit (its own 32 accumulator columns of the stage).  Three warps,
        // because one thread sustains only about one tcgen05.mma per ~57 cycles (measured: a single issuing warp held this kernel
        // at 27 % tensor-pipe activity whatever the issue order) while an M128 N32 K16 MMA occupies the pipe for ~41. =====
        const int jw = warp - 1;
        const uint32_t idesc = instr_desc_f16(MTILE, LC_C);
        const uint64_t a_desc0 = smem_desc(smem_u32(smem), LC_PSTRIDE * 16, 128);
        const uint64_t w_desc0 = smem_desc(smem_u32(w_smem), LC_C * 16, 128);
        constexpr uint32_t A_KK = 2 * LC_PSTRIDE, W_KK = 2 * LC_C, W_TAP = 4 * LC_C;   // in 16-byte units
        uint32_t g = 0;                                   // running unit counter of this CTA (accumulator stage = g & 1)
        for (int k = 0; k < n_my; ++k) {
            const int it = (int)blockIdx.x + k * (int)gridDim.x, h = it & 1;
            const uint32_t kp = (uint32_t)(k & 1);
            if (MODE == 0) mbar_wait(bar(LCB_DOWN_EMPTY), kp ^ 1);       // the previous item's strided-conv accumulators have been read
            if (MODE == 1) {
                // ---- transposed conv: tile jw = coarse rows [128 jw, +128) of the item's window, D = 128 columns at 128 jw ----
                const int Lc = NLAYERS * k, slot = Lc & 1;
                mbar_wait(bar(LCB_ITEM_DONE), kp ^ 1);                   // TMEM (stream + accumulators) of the previous item is free
                mbar_wait(bar(LCB_W_FULL + slot), (Lc >> 1) & 1);
                mbar_wait(bar(LCB_T_FULL), kp);
                tc_fence_after();
                if (elect_one()) {
                    const uint32_t dd = tmem + (uint32_t)(jw * 4 * LC_C);
                    const uint64_t ad = smem_desc(smem_u32(smem) + row_off(4, 0), LC_AR * 16, 128) + (uint64_t)(uint32_t)(jw * MTILE);
                    const uint64_t bd = smem_desc(smem_u32(w_smem) + (uint32_t)slot * LC_W_BYTES, 4 * LC_C * 16, 128);
                    const uint32_t idu = instr_desc_f16(MTILE, 4 * LC_C);
#pragma unroll
                    for (int ks = 0; ks < 4; ++ks) {
                        if (ks == 0) tc_mma_f16(dd, ad, bd, idu, 0u);
                        else tc_mma_f16_acc(dd, ad + (uint64_t)(ks * 2 * LC_AR), bd + (uint64_t)(ks * 2 * 4 * LC_C), idu);
                    }
                    tc_commit(bar(LCB_CONVT_FULL));
                    tc_commit(bar(LCB_W_EMPTY + slot));
                }
                __syncwarp();
                mbar_wait(bar(LCB_CONVT_DONE), kp);                      // X holds hi(x), the accumulator columns have been read
            }
            for (int L = 0; L < 4; ++L) {
                const int Lc = NLAYERS * k + L0_IDX + L, slot = Lc & 1;
                mbar_wait(bar(LCB_W_FULL + slot), (Lc >> 1) & 1);
                const int n = lc_ntiles(L), nprev = L == 0 ? LC_HEAD_TILES : lc_ntiles(L - 1);
                const int src_pl = (L & 1) ? 4 : 0;       // conv 1 of a block reads X, conv 2 reads T
                int pw = 0;
                for (int u0 = 0; u0 < n; u0 += LC_J, ++g) {
                    const int i = u0 + jw;
                    const bool active = i < n;
                    const int r = active ? lc_tile_start(L, h, i) : 0;
                    // rows [r - 50, r + 178) of the input of the tile must be complete
                    if (active && !(MODE == 1 && L == 0)) {
                        while (pw < nprev && (L == 0 ? lc_head_start(h, pw) : lc_tile_start(L - 1, h, pw)) < r + MTILE + LC_WP + 1) {
                            mbar_wait(bar(L == 0 ? LCB_X_READY + pw : LCB_TILE_DONE + (L - 1) * 11 + pw), kp);
                            ++pw;
                        }
                    }
                    const uint32_t b = g & 1;
                    mbar_wait(bar(LCB_ACC_EMPTY + b), ((g >> 1) & 1) ^ 1);     // also orders an inactive warp's arrival behind the stage's previous phase
                    tc_fence_after();
                    if (elect_one()) {
                        if (active) {
                            const uint32_t d = tmem + (uint32_t)(LC_ACC_COL + b * (LC_J * LC_C) + jw * LC_C);
                            const uint64_t ad = a_desc0 + (uint64_t)(uint32_t)(src_pl * LC_PSTRIDE + LC_GAP + r);
                            const uint64_t wd = w_desc0 + (uint64_t)((uint32_t)slot * (LC_W_BYTES >> 4));
#pragma unroll
                            for (int tap = 0; tap < 9; ++tap) {
                                const uint64_t at = ad + (uint64_t)(int64_t)((tap / 3 - 1) * LC_WP + (tap % 3 - 1));
                                const uint64_t bt = wd + (uint64_t)(tap * W_TAP);
                                if (tap == 0) tc_mma_f16(d, at, bt, idesc, 0u); else tc_mma_f16_acc(d, at, bt, idesc);
                                tc_mma_f16_acc(d, at + A_KK, bt + W_KK, idesc);
                            }
                            tc_commit(bar(LCB_ACC_FULL + b));
                        } else {
                            mbar_arrive(bar(LCB_ACC_FULL + b));
                        }
                    }
                    __syncwarp();
                }
                if (elect_one()) {
                    tc_commit(bar(LCB_W_EMPTY + slot));
                    if (L == 2) tc_commit(bar(LCB_X_FREE));
                    if (L == 3) tc_commit(bar(LCB_T_FREE));
                }
                __syncwarp();
            }
            if (MODE == 0) {
                // ---- strided conv: tile jw = coarse rows [128 jw, +128) of the item, D = 64 columns at LC_ACC_COL + 64 jw ----
                const int Lc = NLAYERS * k + 4, slot = Lc & 1;
                mbar_wait(bar(LCB_W_FULL + slot), (Lc >> 1) & 1);
                for (int i = 0; i < lc_ntiles(3); ++i) mbar_wait(bar(LCB_TILE_DONE + 3 * 11 + i), kp);   // operand complete, accumulators drained
                tc_fence_after();
                if (elect_one()) {
                    const uint32_t dd = tmem + (uint32_t)(LC_ACC_COL + jw * LC_DN);
                    const uint64_t ad = smem_desc(smem_u32(smem) + row_off(0, 0), LC_SR * 16, 128) + (uint64_t)(uint32_t)(jw * MTILE);
                    const uint64_t bd = smem_desc(smem_u32(w_smem) + (uint32_t)slot * LC_W_BYTES, LC_DN * 16, 128);
                    const uint32_t idd = instr_desc_f16(MTILE, LC_DN);
#pragma unroll
                    for (int ks = 0; ks < 8; ++ks) {
                        if (ks == 0) tc_mma_f16(dd, ad, bd, idd, 0u);
                        else tc_mma_f16_acc(dd, ad + (uint64_t)(ks * 2 * LC_SR), bd + (uint64_t)(ks * 2 * LC_DN), idd);
                    }
                    tc_commit(bar(LCB_DOWN_FULL));
                    tc_commit(bar(LCB_W_EMPTY + slot));
                }
                __syncwarp();
            }
        }
    } else if (warp < LC_J + 5) {
        // ===== helpers =====
        // DOWN, phase A (as soon as the previous item's last reads of X are done, i.e. during its 4th conv): x1 = m_head(t) -> X (fp16);
        //       phase B (once the previous item's stream has been consumed): the same fp32 values -> stream (TMEM).  Recomputing the
        //       288 FMAs per row is cheaper than holding them, and neither phase is on the MMA warp's critical path.
        // UP:   stream = hi (X) + lo (T), which also releases T for the first conv's output.
        const int q = warp & 3;
        for (int k = 0; k < n_my; ++k) {
            const int it = (int)blockIdx.x + k * (int)gridDim.x, h = it & 1;
            const uint32_t kp = (uint32_t)(k & 1);
            if (MODE == 0) {
                mbar_wait(bar(LCB_DOWN_FULL), kp ^ 1);                   // the previous item's strided conv has finished reading the X planes
                mbar_wait(bar(LCB_TWIN_FULL), kp);
                if (k > 0) {                                             // gap rows below the window, which no head tile covers
                    const int s = LC_ROWS + q * 32 + lane;
                    if (s < LC_PSTRIDE) {
#pragma unroll
                        for (int ch = 0; ch < 4; ++ch) *reinterpret_cast<uint4*>(smem + row_off(ch, s)) = make_uint4(0u, 0u, 0u, 0u);
                    }
                }
                for (int j = 0; j < LC_HEAD_TILES; ++j) fill_x_tile(h, k, j, q);
                mbar_wait(bar(LCB_ITEM_DONE), kp ^ 1);                   // the previous item's stream has been consumed
                tc_fence_after();
                for (int i = 0; i < LC_STREAM_TILES; ++i) {
                    const int s = lc_stream_start(h, i) + q * 32 + lane;
                    float acc[LC_C];
                    head_row(h, s, acc);
                    const uint32_t taddr = tmem + ((uint32_t)(q * 32) << 16) + (uint32_t)(i * LC_C);
                    uint32_t u[LC_C];
#pragma unroll
                    for (int c = 0; c < LC_C; ++c) u[c] = __float_as_uint(acc[c]);
                    tc_st16(taddr, u); tc_st16(taddr + 16, u + 16);
                    tc_st_wait();
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(bar(LCB_S_READY + i));
                }
                __syncwarp();
                if (lane == 0) mbar_arrive(bar(LCB_TWIN_EMPTY));
            } else {
                mbar_wait(bar(LCB_CONVT_DONE), kp);                      // hi in X, lo in the scratch; TMEM columns of the stream are free
                tc_fence_after();
                for (int i = 0; i < LC_STREAM_TILES; ++i) {
                    const int s = lc_stream_start(h, i) + q * 32 + lane;
                    const uint4* lop = reinterpret_cast<const uint4*>(scratch + (size_t)s * 64);
                    uint32_t u[LC_C];
#pragma unroll
                    for (int ch = 0; ch < 4; ++ch) {
                        const uint4 hi = *reinterpret_cast<const uint4*>(smem + row_off(ch, s));
                        const uint4 lo = __ldcg(lop + ch);
                        const float2 f0 = hilo_pair(hi.x, lo.x), f1 = hilo_pair(hi.y, lo.y), f2 = hilo_pair(hi.z, lo.z), f3 = hilo_pair(hi.w, lo.w);
                        u[8 * ch] = __float_as_uint(f0.x); u[8 * ch + 1] = __float_as_uint(f0.y); u[8 * ch + 2] = __float_as_uint(f1.x); u[8 * ch + 3] = __float_as_uint(f1.y);
                        u[8 * ch + 4] = __float_as_uint(f2.x); u[8 * ch + 5] = __float_as_uint(f2.y); u[8 * ch + 6] = __float_as_uint(f3.x); u[8 * ch + 7] = __float_as_uint(f3.y);
                    }
                    const uint32_t taddr = tmem + ((uint32_t)(q * 32) << 16) + (uint32_t)(i * LC_C);
                    tc_st16(taddr, u); tc_st16(taddr + 16, u + 16);
                    tc_st_wait();
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(bar(LCB_S_READY + i));
                }
            }
        }
    } else {
        // ===== epilogue: group (warps 6-9 / 10-13) takes every second UNIT of the CTA-wide sequence; a warp walks the unit's tiles =====
        const int q = warp & 3, grp = (warp - (LC_J + 5)) >> 2;
        const uint32_t lane_base = (uint32_t)(q * 32) << 16;
        uint32_t g = 0;
        for (int k = 0; k < n_my; ++k) {
            const int it = (int)blockIdx.x + k * (int)gridDim.x, bst = it >> 1, h = it & 1;
            const uint32_t kp = (uint32_t)(k & 1);
            if (MODE == 1) {
                // ---- transposed-conv epilogue: warp (q, grp) takes sub-pixel row dy = grp (both dx) of coarse rows 128 j + 32 q + lane ----
                mbar_wait(bar(LCB_CONVT_FULL), kp);
                tc_fence_after();
                if (q == 0 && grp == 0) {
                    // the A operand overwrote pad pixels and gap rows of T planes 4-5 (bytes [0, 45056) from plane 4): restore the zeros
                    for (int i = lane; i < 128; i += 32) {
                        int pl, s;
                        if (i < 28) { pl = 4; s = i * LC_WP + STAMP; }
                        else if (i < 84) { pl = 4; s = LC_ROWS + (i - 28); }
                        else if (i < 112) { pl = 5; s = (i - 84) * LC_WP + STAMP; }
                        else { pl = 5; s = LC_ROWS + (i - 112); }
                        *reinterpret_cast<uint4*>(smem + row_off(pl, s)) = make_uint4(0u, 0u, 0u, 0u);
                    }
                }
                for (int j = 0; j < 3; ++j) {
                    const int cr = j * MTILE + q * 32 + lane, cy = cr / 25, cx = cr - cy * 25;
                    const bool valid = cr < 350 && cx < 24;
#pragma unroll
                    for (int dx = 0; dx < 2; ++dx) {
                        const uint32_t a = tmem + lane_base + (uint32_t)(j * 4 * LC_C + (grp * 2 + dx) * LC_C);
                        uint32_t d0[16], d1[16];
                        tc_ld16_nowait(a, d0); tc_ld16_nowait(a + 16, d1);
                        const int s = (2 * cy + grp) * LC_WP + 2 * cx + dx;
                        tc_ld_wait16(d0); tc_ld_wait16(d1);
                        if (valid) {
                            float v[LC_C];
#pragma unroll
                            for (int c = 0; c < 16; ++c) { v[c] = __uint_as_float(d0[c]); v[16 + c] = __uint_as_float(d1[c]); }
                            uint4* lop = reinterpret_cast<uint4*>(scratch + (size_t)s * 64);
#pragma unroll
                            for (int ch = 0; ch < 4; ++ch) {
                                uint4 hi, lo;
                                split8_hilo(v + 8 * ch, hi, lo);
                                *reinterpret_cast<uint4*>(smem + row_off(ch, s)) = hi;
                                __stcg(lop + ch, lo);
                            }
                        }
                    }
                }
                tc_fence_before();
                fence_proxy_async_smem();
                __threadfence_block();
                __syncwarp();
                if (lane == 0) mbar_arrive(bar(LCB_CONVT_DONE));
            }
            for (int L = 0; L < 4; ++L) {
                const int n = lc_ntiles(L);
                for (int u0 = 0; u0 < n; u0 += LC_J, ++g) {
                    if ((int)(g & 1) != grp) continue;
                    const int nj = n - u0 < LC_J ? n - u0 : LC_J;
                    const uint32_t b = g & 1;
                    mbar_wait(bar(LCB_ACC_FULL + b), (g >> 1) & 1);
                    tc_fence_after();
                    for (int j = 0; j < nj; ++j) {
                        const int i = u0 + j;
                        int r, wlo, whi;
                        lc_tile(L, h, i, r, wlo, whi);
                        const uint32_t acc_addr = tmem + lane_base + (uint32_t)(LC_ACC_COL + b * (LC_J * LC_C) + j * LC_C);
                        const uint32_t st_addr = tmem + lane_base + (uint32_t)(i * LC_C);     // layers 1, 3 run on the stream grid
                        uint32_t r0[16], r1[16], s0[16], s1[16];
                        tc_ld16_nowait(acc_addr, r0);
                        tc_ld16_nowait(acc_addr + 16, r1);
                        if (L == 1) { mbar_wait(bar(LCB_S_READY + i), kp); tc_fence_after(); }   // the helpers have filled this stream tile
                        if (L & 1) { tc_ld16_nowait(st_addr, s0); tc_ld16_nowait(st_addr + 16, s1); }
                        const int s = r + q * 32 + lane;
                        const int yq = (s * 1338) >> 16, x = s - yq * LC_WP;       // s / 49 exactly for 0 <= s < 2400
                        const bool inimg = s < LC_ROWS && x < STAMP;
                        const bool wr = inimg && s >= wlo && s < whi;
                        tc_ld_wait16(r0);
                        tc_ld_wait16(r1);
                        if (L & 1) { tc_ld_wait16(s0); tc_ld_wait16(s1); }
                        if (j == nj - 1) {               // every accumulator of the unit has been read: the MMA warp may reuse the stage
                            tc_fence_before();
                            __syncwarp();
                            if (lane == 0) mbar_arrive(bar(LCB_ACC_EMPTY + b));
                        }
                        float v[LC_C];
#pragma unroll
                        for (int c = 0; c < 16; ++c) { v[c] = __uint_as_float(r0[c]); v[16 + c] = __uint_as_float(r1[c]); }
                        if (!(L & 1)) {
                            // first conv of a block: ReLU -> fp16 -> T
                            if (wr) {
#pragma unroll
                                for (int c = 0; c < LC_C; ++c) v[c] = fmaxf(v[c], 0.f);
#pragma unroll
                                for (int ch = 0; ch < 4; ++ch) *reinterpret_cast<uint4*>(smem + row_off(4 + ch, s)) = pack8_half(v + 8 * ch);
                            }
                            fence_proxy_async_smem();
                            __syncwarp();
                            if (lane == 0) mbar_arrive(bar(LCB_TILE_DONE + L * 11 + i));
                        } else {
#pragma unroll
                            for (int c = 0; c < 16; ++c) { v[c] += __uint_as_float(s0[c]); v[16 + c] += __uint_as_float(s1[c]); }
                            if (L == 1) {
                                // second conv of block 1: stream += acc (TMEM), fp16 copy -> X
                                uint32_t u[LC_C];
#pragma unroll
                                for (int c = 0; c < LC_C; ++c) u[c] = __float_as_uint(v[c]);
                                tc_st16(st_addr, u); tc_st16(st_addr + 16, u + 16);
                                if (wr) {
#pragma unroll
                                    for (int ch = 0; ch < 4; ++ch) *reinterpret_cast<uint4*>(smem + row_off(ch, s)) = pack8_half(v + 8 * ch);
                                }
                                tc_st_wait();
                                tc_fence_before();
                                fence_proxy_async_smem();
                                __syncwarp();
                                if (lane == 0) mbar_arrive(bar(LCB_TILE_DONE + L * 11 + i));
                            } else {
                                // second conv of block 2: the item's own 24 rows leave the SM (UP) / become the strided conv's operand (DOWN)
                                const bool own = wr && (h ? s >= LC_ROWS - LC_OWN : s < LC_OWN);
                                if (MODE == 0) mbar_wait(bar(LCB_X_FREE), kp);      // conv 3 has finished reading the X planes the operand overwrites
                                if (own) {
                                    const int y = h * LC_BOT_Y0 + yq;
                                    if (MODE == 0) {
                                        // space-to-depth operand of the strided conv: K chunk = (dy*2+dx)*4 + ch, row = coarse pixel of the item
                                        const int yl = yq - (h ? LC_WIN_Y - 24 : 0);
                                        const int cr = (yl >> 1) * 25 + (x >> 1), ctap = ((yl & 1) << 1) | (x & 1);
                                        unsigned char* dst = smem + row_off(0, 0) + (uint32_t)((ctap * 4 * LC_SR + cr) * 16);
#pragma unroll
                                        for (int ch = 0; ch < 4; ++ch) *reinterpret_cast<uint4*>(dst + ch * LC_SR * 16) = pack8_half(v + 8 * ch);
                                    } else {
                                        float* dst = p.tail_part + ((size_t)p.g0.base0 + (size_t)bst * p.g0.S + (size_t)(y * LC_WP + x));
                                        lc_tail(htw.tail, v, dst, Ptot0);
                                    }
                                }
                                if (MODE == 0) {
                                    fence_proxy_async_smem();
                                    __syncwarp();
                                    if (lane == 0) mbar_arrive(bar(LCB_TILE_DONE + L * 11 + i));
                                }
                            }
                        }
                    }
                }
            }
            if (MODE == 0) {
                // ---- strided-conv epilogue: warp (q, grp) stores channels [32 grp, +32) of coarse rows 128 j + 32 q + lane, j = 0..2 ----
                mbar_wait(bar(LCB_DOWN_FULL), kp);
                tc_fence_after();
                const Geom& g1 = p.g1;
                for (int j = 0; j < 3; ++j) {
                    const uint32_t a = tmem + lane_base + (uint32_t)(LC_ACC_COL + j * LC_DN + grp * 32);
                    uint32_t d0[16], d1[16];
                    tc_ld16_nowait(a, d0); tc_ld16_nowait(a + 16, d1);
                    const int cr = j * MTILE + q * 32 + lane, cx = cr % 25;
                    tc_ld_wait16(d0); tc_ld_wait16(d1);
                    if (j == 2) {                    // every accumulator column of the strided conv has been read
                        tc_fence_before();
                        __syncwarp();
                        if (lane == 0) mbar_arrive(bar(LCB_DOWN_EMPTY));
                    }
                    if (cr < 300 && cx < 24) {
                        const size_t row = (size_t)g1.base0 + (size_t)bst * g1.S + (size_t)(h * 300 + cr);
                        float4* o32 = reinterpret_cast<float4*>(p.skip32) + (size_t)(grp * 8) * g1.Ptot + row;
                        uint4* o16 = reinterpret_cast<uint4*>(p.x2_16) + (size_t)(grp * 4) * g1.Ptot + row;
                        float v[32];
#pragma unroll
                        for (int c = 0; c < 16; ++c) { v[c] = __uint_as_float(d0[c]); v[16 + c] = __uint_as_float(d1[c]); }
#pragma unroll
                        for (int c4 = 0; c4 < 8; ++c4) o32[(size_t)c4 * g1.Ptot] = make_float4(v[4 * c4], v[4 * c4 + 1], v[4 * c4 + 2], v[4 * c4 + 3]);
#pragma unroll
                        for (int c8 = 0; c8 < 4; ++c8) {
                            uint4 hi8, lo8;
                            split8_hilo(v + 8 * c8, hi8, lo8);
                            o16[(size_t)c8 * g1.Ptot] = hi8;
                            if (p.x2_lo) (reinterpret_cast<uint4*>(p.x2_lo) + (size_t)(grp * 4) * g1.Ptot + row)[(size_t)c8 * g1.Ptot] = lo8;
                        }
                    }
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(bar(LCB_ITEM_DONE));
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(TMEM_COLS) : "memory");
    }
}

static int g_lc_sms = 0;

int conv_l1chain_init() {
    int dev;
    GD_CUDA_CHECK(cudaGetDevice(&dev));
    GD_CUDA_CHECK(cudaDeviceGetAttribute(&g_lc_sms, cudaDevAttrMultiProcessorCount, dev));
    GD_CUDA_CHECK(cudaFuncSetAttribute(k_l1_chain<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, LC_SMEM));
    GD_CUDA_CHECK(cudaFuncSetAttribute(k_l1_chain<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, LC_SMEM));
    return GD_OK;
}

static int l1chain_launch(int mode, const L1ChainParams& p, const float* head_w, const float* tail_w, cudaStream_t st) {
    if (p.nb <= 0) return GD_OK;
    if (!g_lc_sms) { set_error("conv_l1chain: library not initialised"); return GD_ECUDA; }
    if (p.g0.Wp != LC_WP || p.g0.base0 < LC_WP + 1 || p.g1.Wp != 25) { set_error("conv_l1chain: needs the 48x48 / 24x24 geometries"); return GD_EUNSUPPORTED; }
    L1ChainHT hw;
    memset(&hw, 0, sizeof(hw));
    if (head_w) memcpy(hw.head, head_w, sizeof(hw.head));
    if (tail_w) memcpy(hw.tail, tail_w, sizeof(hw.tail));
    const int items = 2 * p.nb, grid = items < g_lc_sms ? items : g_lc_sms;
    cudaEvent_t e1 = nullptr;
    double flops = 4.0 * 2.0 * (double)p.nb * NPIX * (double)LC_C * LC_C * 9;            // four 3x3 convs, valid pixels
    flops += 2.0 * (double)p.nb * (NPIX / 4) * (4.0 * LC_C) * LC_DN;                     // + the k2s2 strided (DOWN) / transposed (UP) conv
    { int rc = conv_profile_mark(flops, st, &e1); if (rc != GD_OK) return rc; }
    if (mode == 0) k_l1_chain<0><<<grid, LC_THREADS, LC_SMEM, st>>>(p, hw);
    else k_l1_chain<1><<<grid, LC_THREADS, LC_SMEM, st>>>(p, hw);
    GD_LAUNCHED();
    if (e1) GD_CUDA_CHECK(cudaEventRecord(e1, st));
    return GD_OK;
}

int launch_l1chain_down(const Geom& g0, const Geom& g1, int nb, const float* t, const float* head_w_host, const void* const* w4, const void* wdown,
                        float* skip32, void* x2_16, void* x2_lo, cudaStream_t st) {
    L1ChainParams p;
    memset(&p, 0, sizeof(p));
    p.nb = nb; p.g0 = g0; p.g1 = g1; p.t = t; p.wdown = wdown; p.skip32 = skip32; p.x2_16 = x2_16; p.x2_lo = x2_lo;
    for (int i = 0; i < 4; ++i) p.w[i] = w4[i];
    if (!t || !head_w_host || !wdown || !skip32 || !x2_16) { set_error("conv_l1chain: down needs t, the head / strided-conv weights and the x2 outputs"); return GD_EBADSHAPE; }
    return l1chain_launch(0, p, head_w_host, nullptr, st);
}

size_t l1chain_scratch_bytes() { return (size_t)160 * LC_SCRATCH_BYTES; }     // one region per CTA of the persistent grid (<= 160 SMs)

int launch_l1chain_up(const Geom& g0, const Geom& g1, int nb, const void* x_in, const void* wup, const float* tail_w_host, const void* const* w4,
                      float* tail_part, void* scratch, cudaStream_t st) {
    L1ChainParams p;
    memset(&p, 0, sizeof(p));
    p.nb = nb; p.g0 = g0; p.g1 = g1; p.x_in = x_in; p.wup = wup; p.tail_part = tail_part; p.scratch = reinterpret_cast<unsigned char*>(scratch);
    for (int i = 0; i < 4; ++i) p.w[i] = w4[i];
    if (!x_in || !wup || !tail_w_host || !tail_part || !scratch) { set_error("conv_l1chain: up needs the level-1 map, the transposed-conv / tail weights, tail_part and the scratch"); return GD_EBADSHAPE; }
    if (g_lc_sms > 160) { set_error("conv_l1chain: scratch is sized for 160 CTAs"); return GD_EUNSUPPORTED; }
    return l1chain_launch(1, p, nullptr, tail_w_host, st);
}

}  // namespace gd
