// C ABI of libgdeconv (include/gdeconv.h): weight packing, workspace layout, the ResUNet layer graph and the
// unrolled-ADMM drivers.  Host code only; every kernel lives in fft_kernels.cu / subnet.cu / conv_*.cu.
#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/gdeconv.h"
#include "kernels.cuh"
#include "launch.cuh"

namespace gd {

std::atomic<unsigned long long> g_launches{0};

static thread_local char g_err[512] = "";
void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

#define GD_FAIL(code, ...)           \
    do {                             \
        gd::set_error(__VA_ARGS__);  \
        return (code);               \
    } while (0)
#define GD_TRY(expr)                 \
    do {                             \
        int _rc = (expr);            \
        if (_rc != GD_OK) return _rc; \
    } while (0)

static size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// ---------------------------------------------------------------------------------------------------
// weights
// ---------------------------------------------------------------------------------------------------
struct ConvW { const void* w; };

}  // namespace gd

struct GdWeights {
    int arch, n_iters, n_rho, precision, device;
    int nc[4];
    int has_resunet, has_subnet, has_rho_param;
    void* blob;                       // one device allocation
    size_t blob_bytes;
    const float* head;                // [9][C0] fp32
    const float* tail;                // [9][C0] fp32
    float head_h[9 * 64], tail_h[9 * 64];   // host copies (C0 <= 64): kernel-parameter weights of the head/tail-fused epilogue
    float tail_head_g[81];                  // G[tap2][tap1] = sum_c tail[tap2][c] * head[tap1][c]: m_tail(m_head(t)) as one 1-channel stencil
    const void* down_rb[3][2][2];     // down stage L, ResBlock, conv  (3x3, C_L -> C_L)
    const void* down[3];              // k2s2 strided conv C_L -> C_{L+1}
    const void* body_rb[2][2];
    const void* up[3];                // k2s2 transposed conv C_{L+1} -> C_L (index = fine level L)
    const void* up_rb[3][2][2];
    const void* up1_plain;            // C1 = 64: m_up2's transposed conv in the same plain order (conv_l2chain.cu)
    const void* up0_plain;            // C0 = 32, tcgen05 path: m_up1's transposed conv with plain column order n = (dy*2+dx)*C0 + co (conv_l1chain.cu)
    gd::SubnetParams sub;
    const float* rho_param;           // [n_rho] when subnet=False
};

namespace gd {

struct Finder {
    std::map<std::string, const GdTensorDesc*> m;
    Finder(const GdTensorDesc* t, int n) {
        for (int i = 0; i < n; ++i)
            if (t[i].name && t[i].data) m[t[i].name] = &t[i];
    }
    const GdTensorDesc* get(const std::string& key) const {
        auto it = m.find(key);
        return it == m.end() ? nullptr : it->second;
    }
    // ResUNet tensors are looked up as "Z.net.<key>" (ADMM classes) or "<key>" (a bare ResUNet state_dict)
    const GdTensorDesc* net(const std::string& key) const {
        const GdTensorDesc* t = get("Z.net." + key);
        return t ? t : get(key);
    }
};

static bool shape_is(const GdTensorDesc* t, int64_t a, int64_t b, int64_t c, int64_t d) {
    return t && t->ndim == 4 && t->shape[0] == a && t->shape[1] == b && t->shape[2] == c && t->shape[3] == d;
}

struct Blob {
    std::vector<unsigned char> host;
    size_t reserve(size_t bytes) {
        size_t off = align_up(host.size(), 256);
        host.resize(off + bytes, 0);
        return off;
    }
};

// element writer in the operand precision
static void put_elem(unsigned char* base, size_t idx, float v, int prec) {
    if (prec == PREC_FP32_SIMT) reinterpret_cast<float*>(base)[idx] = v;
    else reinterpret_cast<__half*>(base)[idx] = __float2half_rn(v);
}
static size_t elem_size(int prec) { return prec == PREC_FP32_SIMT ? 4 : 2; }

// B[tap][k][n] -> blob in the layout the conv kernel of `prec` wants:
//   SIMT: [tap][Kt][N];   UMMA: [tap][Kt/8][N][8]  (K-major, one 16-byte vector per (n, 8 channels))
static size_t pack_tapgemm(Blob& bl, int ntaps, int Kt, int N, int prec, const std::vector<float>& B) {
    size_t off = bl.reserve((size_t)ntaps * Kt * N * elem_size(prec));
    unsigned char* base = bl.host.data() + off;
    for (int t = 0; t < ntaps; ++t)
        for (int k = 0; k < Kt; ++k)
            for (int n = 0; n < N; ++n) {
                float v = B[((size_t)t * Kt + k) * N + n];
                size_t idx = prec == PREC_FP16_UMMA ? (((size_t)t * (Kt / 8) + k / 8) * N + n) * 8 + (k % 8)
                                                    : ((size_t)t * Kt + k) * N + n;
                put_elem(base, idx, v, prec);
            }
    return off;
}

// Conv2d weight [Co][Ci][3][3] -> B[tap = ky*3+kx][ci][co]      (models/resnet_basicblock.py:21-56, mode 'C')
static int pack_conv3(Blob& bl, const GdTensorDesc* t, int C, int prec, size_t* off, const char* what) {
    if (!shape_is(t, C, C, 3, 3)) GD_FAIL(GD_EBADSHAPE, "weight %s: missing or not (%d,%d,3,3)", what, C, C);
    std::vector<float> B((size_t)9 * C * C);
    for (int co = 0; co < C; ++co)
        for (int ci = 0; ci < C; ++ci)
            for (int tp = 0; tp < 9; ++tp) B[((size_t)tp * C + ci) * C + co] = t->data[((size_t)co * C + ci) * 9 + tp];
    *off = pack_tapgemm(bl, 9, C, C, prec, B);
    return GD_OK;
}
// strided Conv2d k2 s2 [Co][Ci][2][2] -> one tap, K = (dy*2+dx)*Ci + ci     (resnet_basicblock.py:73-79)
static int pack_down(Blob& bl, const GdTensorDesc* t, int Ci, int Co, int prec, size_t* off, const char* what) {
    if (!shape_is(t, Co, Ci, 2, 2)) GD_FAIL(GD_EBADSHAPE, "weight %s: missing or not (%d,%d,2,2)", what, Co, Ci);
    std::vector<float> B((size_t)4 * Ci * Co);
    for (int co = 0; co < Co; ++co)
        for (int ci = 0; ci < Ci; ++ci)
            for (int tp = 0; tp < 4; ++tp) B[((size_t)tp * Ci + ci) * Co + co] = t->data[((size_t)co * Ci + ci) * 4 + tp];
    *off = pack_tapgemm(bl, 1, 4 * Ci, Co, prec, B);
    return GD_OK;
}
// ConvTranspose2d k2 s2 [Ci][Co][2][2] -> one tap, N = (dy*2+dx)*Co + co    (resnet_basicblock.py:81-87)
static int pack_up(Blob& bl, const GdTensorDesc* t, int Ci, int Co, int prec, size_t* off, const char* what) {
    if (!shape_is(t, Ci, Co, 2, 2)) GD_FAIL(GD_EBADSHAPE, "weight %s: missing or not (%d,%d,2,2)", what, Ci, Co);
    std::vector<float> B((size_t)Ci * 4 * Co);
    for (int ci = 0; ci < Ci; ++ci)
        for (int co = 0; co < Co; ++co)
            for (int tp = 0; tp < 4; ++tp) {
                // tcgen05 path: columns ordered for the lane-paired stores of epi_up_unit (conv_epilogue.cuh)
                const int dy = tp >> 1, dx = tp & 1;
                const int n = prec == PREC_FP16_UMMA ? dy * 2 * Co + (co / 16) * 32 + ((co % 16) / 4) * 8 + dx * 4 + (co % 4) : tp * Co + co;
                B[(size_t)ci * 4 * Co + n] = t->data[((size_t)ci * Co + co) * 4 + tp];
            }
    *off = pack_tapgemm(bl, 1, Ci, 4 * Co, prec, B);
    return GD_OK;
}

// the same transposed conv for the level-0 chain kernel: plain column order n = (dy*2+dx)*Co + co
static int pack_up_plain(Blob& bl, const GdTensorDesc* t, int Ci, int Co, size_t* off, const char* what) {
    if (!shape_is(t, Ci, Co, 2, 2)) GD_FAIL(GD_EBADSHAPE, "weight %s: missing or not (%d,%d,2,2)", what, Ci, Co);
    std::vector<float> B((size_t)Ci * 4 * Co);
    for (int ci = 0; ci < Ci; ++ci)
        for (int co = 0; co < Co; ++co)
            for (int tp = 0; tp < 4; ++tp) B[(size_t)ci * 4 * Co + tp * Co + co] = t->data[((size_t)ci * Co + co) * 4 + tp];
    *off = pack_tapgemm(bl, 1, Ci, 4 * Co, PREC_FP16_UMMA, B);
    return GD_OK;
}

static size_t pack_f32(Blob& bl, const float* src, size_t n) {
    size_t off = bl.reserve(n * sizeof(float));
    memcpy(bl.host.data() + off, src, n * sizeof(float));
    return off;
}

}  // namespace gd

using namespace gd;

extern "C" int gd_version(void) { return GD_VERSION; }
extern "C" const char* gd_last_error(void) { return g_err; }
extern "C" uint64_t gd_launch_count(void) { return g_launches.load(); }

static int init_once(int device) {
    static std::atomic<unsigned> done{0};                 // bit per device
    if (device < 0 || device >= 32) GD_FAIL(GD_EBADDEVICE, "device %d out of range", device);
    if (done.load() & (1u << device)) return GD_OK;
    cudaDeviceProp prop;
    GD_CUDA_CHECK(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10) GD_FAIL(GD_EBADDEVICE, "libgdeconv is built for sm_100a only; device %d is sm_%d%d", device, prop.major, prop.minor);
    GD_TRY(fft_kernels_init());
    GD_TRY(subnet_init());
    GD_TRY(conv_umma_init());
    GD_TRY(conv_rb_init());
    GD_TRY(conv_l1chain_init());
    GD_TRY(conv_l2chain_init());
    GD_TRY(synth_init());
    done.fetch_or(1u << device);
    return GD_OK;
}

// for the entry points that live in other translation units (xdense.cu): the device's kernels get their launch attributes here
namespace gd { int ensure_device_init(int device) { return init_once(device); } }

extern "C" int gd_pack_weights(int arch, int n_iters, const GdTensorDesc* tensors, int n_tensors, int precision,
                               int device, GdWeights** out) {
    if (!out) GD_FAIL(GD_EBADSHAPE, "gd_pack_weights: out is NULL");
    *out = nullptr;
    if (arch != GD_ARCH_G && arch != GD_ARCH_U) GD_FAIL(GD_EUNSUPPORTED, "unknown arch %d", arch);
    if (precision < 0 || precision > 2) GD_FAIL(GD_EUNSUPPORTED, "unknown precision mode %d", precision);
    if (n_iters < 0 || n_iters > 64) GD_FAIL(GD_EBADSHAPE, "n_iters %d out of range", n_iters);
    GD_DEVICE_SCOPE(device);
    GD_TRY(init_once(device));
    Finder F(tensors, n_tensors);
    GdWeights W;
    memset(&W, 0, sizeof(W));
    W.arch = arch; W.n_iters = n_iters; W.precision = precision; W.device = device;
    W.n_rho = arch == GD_ARCH_G ? n_iters : 2 * n_iters;
    Blob bl;
    std::map<const void**, size_t> fix;      // pointer slot -> blob offset
    auto slot = [&](const void** p, size_t off) { fix[p] = off; };

    // ---- ResUNet (models/ResUNet.py:7-24); channel widths are read from the head conv ----
    const GdTensorDesc* th = F.net("m_head.weight");
    if (th) {
        if (th->ndim != 4 || th->shape[1] != 1 || th->shape[2] != 3 || th->shape[3] != 3 || th->shape[0] % 16 || th->shape[0] > 256)
            GD_FAIL(GD_EBADSHAPE, "m_head.weight must be (C0,1,3,3) with C0 a multiple of 16, <= 256");
        const int C0 = (int)th->shape[0];
        for (int L = 0; L < 4; ++L) W.nc[L] = C0 << L;
        W.has_resunet = 1;
        {   // head [C0][1][3][3] -> [tap][C0]; tail [1][C0][3][3] -> [tap][C0]
            std::vector<float> h((size_t)9 * C0), tl((size_t)9 * C0);
            const GdTensorDesc* tt = F.net("m_tail.weight");
            if (!shape_is(tt, 1, C0, 3, 3)) GD_FAIL(GD_EBADSHAPE, "m_tail.weight: missing or not (1,%d,3,3)", C0);
            for (int c = 0; c < C0; ++c)
                for (int tp = 0; tp < 9; ++tp) { h[(size_t)tp * C0 + c] = th->data[(size_t)c * 9 + tp]; tl[(size_t)tp * C0 + c] = tt->data[(size_t)c * 9 + tp]; }
            if (C0 <= 64) { memcpy(W.head_h, h.data(), h.size() * sizeof(float)); memcpy(W.tail_h, tl.data(), tl.size() * sizeof(float)); }
            for (int t2 = 0; t2 < 9; ++t2)
                for (int t1 = 0; t1 < 9; ++t1) {
                    double a = 0;
                    for (int c = 0; c < C0; ++c) a += (double)tl[(size_t)t2 * C0 + c] * (double)h[(size_t)t1 * C0 + c];
                    W.tail_head_g[t2 * 9 + t1] = (float)a;
                }
            slot((const void**)&W.head, pack_f32(bl, h.data(), h.size()));
            slot((const void**)&W.tail, pack_f32(bl, tl.data(), tl.size()));
        }
        char key[128];
        size_t off;
        for (int L = 0; L < 3; ++L) {
            const int C = W.nc[L];
            for (int blk = 0; blk < 2; ++blk)
                for (int j = 0; j < 2; ++j) {
                    snprintf(key, sizeof key, "m_down%d.%d.res.%d.weight", L + 1, blk, 2 * j);
                    GD_TRY(pack_conv3(bl, F.net(key), C, precision, &off, key));
                    slot(&W.down_rb[L][blk][j], off);
                    snprintf(key, sizeof key, "m_up%d.%d.res.%d.weight", L + 1, blk + 1, 2 * j);
                    GD_TRY(pack_conv3(bl, F.net(key), C, precision, &off, key));
                    slot(&W.up_rb[L][blk][j], off);
                }
            snprintf(key, sizeof key, "m_down%d.2.weight", L + 1);
            GD_TRY(pack_down(bl, F.net(key), C, 2 * C, precision, &off, key));
            slot(&W.down[L], off);
            snprintf(key, sizeof key, "m_up%d.0.weight", L + 1);
            GD_TRY(pack_up(bl, F.net(key), 2 * C, C, precision, &off, key));
            slot(&W.up[L], off);
            if (L == 0 && C == 32 && precision == PREC_FP16_UMMA) { GD_TRY(pack_up_plain(bl, F.net(key), 2 * C, C, &off, key)); slot(&W.up0_plain, off); }
            if (L == 1 && C == 64 && precision == PREC_FP16_UMMA) { GD_TRY(pack_up_plain(bl, F.net(key), 2 * C, C, &off, key)); slot(&W.up1_plain, off); }
        }
        for (int blk = 0; blk < 2; ++blk)
            for (int j = 0; j < 2; ++j) {
                snprintf(key, sizeof key, "m_body.%d.res.%d.weight", blk, 2 * j);
                GD_TRY(pack_conv3(bl, F.net(key), W.nc[3], precision, &off, key));
                slot(&W.body_rb[blk][j], off);
            }
    }

    // ---- SubNet (unrolled_admm_gaussian.py:43-71 / Unrolled_ADMM.py:59-90): fold BN(eval) into the convs ----
    if (F.get("init.mlp.0.weight")) {
        const int cin[4] = {1, 4, 8, 16}, cout[4] = {4, 8, 16, 16};
        char key[160];
        for (int s = 0; s < 4; ++s)
            for (int j = 0; j < 2; ++j) {
                const int Ci = j == 0 ? cin[s] : cout[s], Co = cout[s];
                const char* names[6] = {"weight", "bias", "weight", "bias", "running_mean", "running_var"};
                const GdTensorDesc* t[6];
                for (int q = 0; q < 6; ++q) {
                    snprintf(key, sizeof key, "init.conv_layers.%d.maxpool_conv.1.double_conv.%d.%s", s, (q < 2 ? 0 : 1) + 3 * j, names[q]);
                    t[q] = F.get(key);
                    if (!t[q]) GD_FAIL(GD_EBADSHAPE, "missing SubNet tensor %s", key);
                }
                if (!shape_is(t[0], Co, Ci, 3, 3)) GD_FAIL(GD_EBADSHAPE, "SubNet conv %d.%d has the wrong shape", s, j);
                std::vector<float> w((size_t)Co * Ci * 9 + Co);
                for (int co = 0; co < Co; ++co) {
                    const float sc = t[2]->data[co] / sqrtf(t[5]->data[co] + 1e-5f);      // nn.BatchNorm2d eps
                    for (int i = 0; i < Ci * 9; ++i) w[(size_t)i * Co + co] = t[0]->data[(size_t)co * Ci * 9 + i] * sc;   // [ci][tap][co]
                    w[(size_t)Co * Ci * 9 + co] = (t[1]->data[co] - t[4]->data[co]) * sc + t[3]->data[co];
                }
                slot((const void**)&W.sub.conv[2 * s + j], pack_f32(bl, w.data(), w.size()));
            }
        const GdTensorDesc *l1w = F.get("init.mlp.0.weight"), *l1b = F.get("init.mlp.0.bias"), *l2w = F.get("init.mlp.2.weight"),
                           *l2b = F.get("init.mlp.2.bias"), *l3w = F.get("init.mlp.4.weight"), *l3b = F.get("init.mlp.4.bias");
        if (!l1w || !l1b || !l2w || !l2b || !l3w || !l3b) GD_FAIL(GD_EBADSHAPE, "missing SubNet mlp tensor");
        if (l1w->ndim != 2 || l1w->shape[0] != 64 || l1w->shape[1] != 1025 || l2w->shape[0] != 64 || l2w->shape[1] != 64 ||
            l3w->ndim != 2 || l3w->shape[1] != 64 || l3w->shape[0] != W.n_rho)
            GD_FAIL(GD_EBADSHAPE, "SubNet mlp shapes must be (64,1025),(64,64),(%d,64)", W.n_rho);
        slot((const void**)&W.sub.l1w, pack_f32(bl, l1w->data, 64 * 1025));
        slot((const void**)&W.sub.l1b, pack_f32(bl, l1b->data, 64));
        slot((const void**)&W.sub.l2w, pack_f32(bl, l2w->data, 64 * 64));
        slot((const void**)&W.sub.l2b, pack_f32(bl, l2b->data, 64));
        slot((const void**)&W.sub.l3w, pack_f32(bl, l3w->data, (size_t)W.n_rho * 64));
        slot((const void**)&W.sub.l3b, pack_f32(bl, l3b->data, W.n_rho));
        W.sub.n_out = W.n_rho;
        W.has_subnet = 1;
    } else if (arch == GD_ARCH_G && F.get("rho_iters")) {
        const GdTensorDesc* r = F.get("rho_iters");
        if (r->ndim != 1 || r->shape[0] != n_iters) GD_FAIL(GD_EBADSHAPE, "rho_iters must have shape (%d,)", n_iters);
        slot((const void**)&W.rho_param, pack_f32(bl, r->data, n_iters));
        W.has_rho_param = 1;
    } else if (arch == GD_ARCH_U && F.get("rho1_iters") && F.get("rho2_iters")) {
        const GdTensorDesc *r1 = F.get("rho1_iters"), *r2 = F.get("rho2_iters");
        if (r1->ndim != 1 || r1->shape[0] != n_iters || r2->ndim != 1 || r2->shape[0] != n_iters)
            GD_FAIL(GD_EBADSHAPE, "rho1_iters/rho2_iters must have shape (%d,)", n_iters);
        std::vector<float> r(2 * n_iters);
        memcpy(r.data(), r1->data, n_iters * sizeof(float));
        memcpy(r.data() + n_iters, r2->data, n_iters * sizeof(float));
        slot((const void**)&W.rho_param, pack_f32(bl, r.data(), r.size()));
        W.has_rho_param = 1;
    }
    if (!W.has_resunet && !W.has_subnet && !W.has_rho_param)
        GD_FAIL(GD_EBADSHAPE, "state_dict holds neither ResUNet (m_head.weight) nor SubNet (init.mlp.0.weight) nor rho parameter tensors");

    W.blob_bytes = align_up(bl.host.size(), 256);
    bl.host.resize(W.blob_bytes, 0);
    GD_CUDA_CHECK(cudaMalloc(&W.blob, W.blob_bytes));
    cudaError_t e = cudaMemcpy(W.blob, bl.host.data(), W.blob_bytes, cudaMemcpyHostToDevice);
    if (e != cudaSuccess) { cudaFree(W.blob); GD_FAIL(GD_ECUDA, "weight upload failed: %s", cudaGetErrorString(e)); }
    GdWeights* res = new GdWeights(W);
    // the slots recorded above point into the local W; rebase them onto the heap copy
    for (auto& kv : fix) {
        const void** p = (const void**)((unsigned char*)res + ((unsigned char*)kv.first - (unsigned char*)&W));
        *p = (unsigned char*)res->blob + kv.second;
    }
    *out = res;
    return GD_OK;
}

extern "C" void gd_free_weights(GdWeights* w) {
    if (!w) return;
    {
        gd::DeviceScope scope(w->device);
        cudaFree(w->blob);
    }
    delete w;
}

// ---------------------------------------------------------------------------------------------------
// workspace
// ---------------------------------------------------------------------------------------------------
namespace gd {

struct WsHeader { uint32_t magic; int arch, prec, chunk; uint64_t bytes; };
constexpr uint32_t WS_MAGIC = 0x47444332u;   // "GDC2"

struct Ws {
    size_t total;
    int C[4];
    Geom g[4];
    // ADMM state
    float *rho, *tscale, *z, *x, *u, *t;       // path G: z,x,u ; path U: + v,u2,Hx (u == u1)
    float *v, *u2, *Hx;
    float2* spec;                              // G: Pc [chunk][96*49]; U: H [chunk][48*25]
    float* HtH;                                // G only
    // ResUNet activations
    float *skip32[4], *p32a[4], *p32b[4];
    void *a16[4], *t16[4], *d16[4], *lo16[4];   // lo16: fp16 correction planes of the hi/lo residual stream (hi = a16 / t16)
    void* lc_scratch;                          // conv_l1chain.cu UP: per-CTA lo halves of the transposed conv's output
    float *tpad, *tail_part;                   // head/tail fusion (conv_umma.cu EPI_HT): padded-linear input, per-tap tail sums
};

static Ws ws_layout(unsigned char* base, int arch, int prec, int chunk) {
    Ws w;
    memset(&w, 0, sizeof(w));
    size_t off = 256;
    auto take = [&](size_t bytes) { unsigned char* p = base + off; off = align_up(off + bytes, 256); return (void*)p; };
    const int C0 = arch == GD_ARCH_G ? 32 : 64;
    const size_t es = elem_size(prec);
    const int nrho = 128;                       // >= 2 * max n_iters
    w.rho = (float*)take((size_t)chunk * nrho * 4);
    w.tscale = (float*)take((size_t)chunk * 4);
    const size_t img = (size_t)chunk * NPIX * 4;
    w.z = (float*)take(img); w.x = (float*)take(img); w.u = (float*)take(img); w.t = (float*)take(img);
    if (arch == GD_ARCH_G) {
        w.spec = (float2*)take((size_t)chunk * FG_SPEC * 8);
        w.HtH = (float*)take((size_t)chunk * FG_SPEC * 4);
    } else {
        w.v = (float*)take(img); w.u2 = (float*)take(img); w.Hx = (float*)take(img);
        w.spec = (float2*)take((size_t)chunk * FU_SPEC * 8);
    }
    for (int L = 0; L < 4; ++L) {
        w.C[L] = C0 << L;
        w.g[L] = make_geom(STAMP >> L, chunk);
        const size_t n = (size_t)w.C[L] * w.g[L].Ptot;
        w.skip32[L] = (float*)take(n * 4);
        w.p32a[L] = (float*)take(n * 4);
        if (L < 3) w.p32b[L] = (float*)take(n * 4);
        w.a16[L] = take(n * es);
        w.t16[L] = take(n * es);
        w.lo16[L] = take(n * es);
        if (L > 0) w.d16[L] = take((size_t)2 * n * es);        // 4*C_{L-1} = 2*C_L channels
    }
    w.lc_scratch = C0 == 32 ? take(l1chain_scratch_bytes() > l2chain_scratch_bytes() ? l1chain_scratch_bytes() : l2chain_scratch_bytes()) : nullptr;
    w.tpad = (float*)take((size_t)w.g[0].Ptot * 4);
    w.tail_part = (float*)take((size_t)(C0 / 16) * 9 * w.g[0].Ptot * 4);   // 32-channel units (conv_umma.cu) or 16-channel halves (conv_rb.cu)
    w.total = off;
    return w;
}

// Host-side registry of initialised workspaces (keyed by device pointer): validating a workspace costs a map lookup,
// never a device read-back, so the forward path stays free of host synchronisation.
static std::mutex g_ws_mu;
static std::map<const void*, WsHeader> g_ws_reg;

static int ws_check(void* workspace, size_t bytes, const GdWeights* W, Ws* ws, int* chunk) {
    if (!workspace) GD_FAIL(GD_EWORKSPACE, "workspace is NULL");
    WsHeader h;
    {
        std::lock_guard<std::mutex> lk(g_ws_mu);
        auto it = g_ws_reg.find(workspace);
        if (it == g_ws_reg.end()) GD_FAIL(GD_EWORKSPACE, "workspace was not initialised with gd_workspace_init");
        h = it->second;
    }
    if (h.arch != W->arch || h.prec != W->precision) GD_FAIL(GD_EWORKSPACE, "workspace was initialised for arch %d / precision %d, weights are %d / %d", h.arch, h.prec, W->arch, W->precision);
    *ws = ws_layout((unsigned char*)workspace, h.arch, h.prec, h.chunk);
    if (ws->total > bytes) GD_FAIL(GD_EWORKSPACE, "workspace holds %zu bytes, chunk %d needs %zu", bytes, h.chunk, ws->total);
    if (W->has_resunet && W->nc[0] != ws->C[0]) GD_FAIL(GD_EUNSUPPORTED, "ResUNet width %d does not match arch %d (expects %d)", W->nc[0], W->arch, ws->C[0]);
    *chunk = h.chunk;
    return GD_OK;
}

// ---------------------------------------------------------------------------------------------------
// ResUNet layer graph (models/ResUNet.py:26-42) on one chunk of `nb` stamps: t (scaled input) -> zout
// ---------------------------------------------------------------------------------------------------
static ConvParams conv_base(const Geom& g, int nb) {
    ConvParams p;
    memset(&p, 0, sizeof(p));
    p.g = g;
    p.g.M = nb * g.S;
    return p;
}
static ConvParams conv3(const Geom& g, int nb, int C, const void* a, const void* w, int relu) {
    ConvParams p = conv_base(g, nb);
    p.ntaps = 9;
    for (int ky = 0; ky < 3; ++ky)
        for (int kx = 0; kx < 3; ++kx) p.off[ky * 3 + kx] = (ky - 1) * g.Wp + (kx - 1);
    p.Kt = C; p.N = C; p.a = a; p.w = w; p.relu = relu;
    return p;
}

static int run_conv(const ConvParams& p, int prec, cudaStream_t st) {
    return prec == PREC_FP16_UMMA ? launch_conv_umma(p, st) : launch_conv_simt(p, prec, st);
}

// Head/tail fusion of the tcgen05 path (GDECONV_FUSE_HT=0 restores the stored fp32 head output and the k_tail kernel).
static int g_fuse_ht = -1;
static int fuse_ht_mode() {
    if (g_fuse_ht < 0) {
        const char* e = getenv("GDECONV_FUSE_HT");
        g_fuse_ht = e ? atoi(e) : 1;
    }
    return g_fuse_ht;
}
// Fused ResBlock kernel at the 32-channel level (conv_rb.cu); GDECONV_FUSE_RB=0 restores one launch per conv.
static int g_fuse_rb = -1;
static int fuse_rb_mode() {
    if (g_fuse_rb < 0) {
        const char* e = getenv("GDECONV_FUSE_RB");
        g_fuse_rb = e ? atoi(e) : 1;
    }
    return g_fuse_rb;
}
// fp16 hi/lo residual stream on the tcgen05 path (ConvParams::res_hi); GDECONV_HILO=0 restores the fp32 stream buffers.
static int g_hilo = -1;
static int hilo_mode() {
    if (g_hilo < 0) {
        const char* e = getenv("GDECONV_HILO");
        g_hilo = e ? atoi(e) : 1;
    }
    return g_hilo;
}
// m_tail(x1) as an 81-coefficient stencil of the denoiser input in k_tail_gather (GDECONV_TAILG=0: recompute x1 in the conv epilogue)
static int g_tailg = -1;
static int tail_g_mode() {
    if (g_tailg < 0) {
        const char* e = getenv("GDECONV_TAILG");
        g_tailg = e ? atoi(e) : 1;
    }
    return g_tailg;
}
// m_head fused into k_g_xupdate (path G, tcgen05, C0 = 32, head/tail fusion); GDECONV_XHEAD=0: separate k_head32 launch
static int g_xhead = -1;
static int xhead_mode() {
    if (g_xhead < 0) {
        const char* e = getenv("GDECONV_XHEAD");
        g_xhead = e ? atoi(e) : 1;
    }
    return g_xhead;
}
// Level-0 chain kernels (conv_l1chain.cu): m_head + the two ResBlocks of m_down1, and the two ResBlocks of m_up1 + the m_tail partial
// sums, each as ONE launch with the intermediates in shared / tensor memory.  GDECONV_L1CHAIN=0 restores one launch per layer pair.
static int g_l1chain = -1;
static int l1chain_mode() {
    if (g_l1chain < 0) {
        const char* e = getenv("GDECONV_L1CHAIN");
        g_l1chain = e ? atoi(e) : 1;
    }
    return g_l1chain;
}
static int g_fuse_ht_fwd();
static bool l1chain_applies(const GdWeights* W) {
    return l1chain_mode() && W->precision == PREC_FP16_UMMA && W->nc[0] == 32 && g_fuse_ht_fwd() && hilo_mode() && tail_g_mode();
}
// Level-1 chain kernel (conv_l2chain.cu): the two ResBlocks of m_down2 resp. m_up2 as one launch each.  GDECONV_L2CHAIN=0 restores the
// per-conv launches at that level.
static int g_l2chain = -1;
static int l2chain_mode() {
    if (g_l2chain < 0) {
        const char* e = getenv("GDECONV_L2CHAIN");
        g_l2chain = e ? atoi(e) : 1;
    }
    return g_l2chain;
}
static bool l2chain_applies(const GdWeights* W) {
    return l2chain_mode() && l1chain_applies(W) && W->nc[1] == 64 && W->up1_plain;
}
static bool xhead_applies(const GdWeights* W) {
    return xhead_mode() && W->precision == PREC_FP16_UMMA && W->nc[0] == 32 && g_fuse_ht_fwd() && !l1chain_applies(W);
}

static int resunet_chunk(const GdWeights* W, const Ws& ws, const float* t, const float* tscale, float* zout, int nb,
                         cudaStream_t st, bool head_done = false) {
    const int prec = W->precision;
    const Geom* g = ws.g;
    const int* C = ws.C;
    // every activation buffer has 16-byte rows, so stamps [s0, ...) of level L start s0 * S_L * 16 bytes into each plane
    auto at = [&](const void* base, int L, int s0) -> unsigned char* {
        return base ? (unsigned char*)base + (size_t)s0 * g[L].S * 16 : nullptr;
    };
    // tcgen05 path: x1 is never stored in fp32; its consumers recompute it from tpad (ConvParams::head_t)
    const bool fuse = prec == PREC_FP16_UMMA && fuse_ht_mode() && C[0] <= 64;
    const bool hilo = prec == PREC_FP16_UMMA && hilo_mode();
    const bool l1chain = l1chain_applies(W);      // level 0 runs in the two chain kernels: no separate head launch, no level-0 fp32 buffers
    const bool l2chain = l2chain_applies(W);      // the ResBlock pairs of level 1 run in one chain launch each
    if (!l1chain) {   // head (ResUNet.py:31): x1 = conv(t)  -> skip32[0] (fp32) + a16[0]
        ConvParams p = conv_base(g[0], nb);
        p.N = C[0]; p.out32 = fuse ? nullptr : ws.skip32[0]; p.out16 = ws.a16[0];
        if (!(head_done && fuse))
            GD_TRY(launch_head(t, W->head, C[0] <= 64 ? W->head_h : nullptr, C[0], p, nb, prec, fuse ? ws.tpad : nullptr, st));
    }
    auto at4 = [&](float* base, int s0) -> float* { return base + (size_t)s0 * g[0].S; };    // 4-byte rows of level 0
    // one ResBlock (resnet_basicblock.py:69-71) on stamps [s0, s0+n): stream + conv(relu(conv(stream))) -> two layers
    // fp16 input of the next resblock() call; nullptr = ws.a16[L].  The fused ResBlock kernel (conv_rb.cu) must not write its
    // fp16 output over its own input (neighbouring work items still read it as halo), so pairs ping-pong a16 <-> t16.
    const void* rb_in16 = nullptr;
    auto rb_params = [&](int L, int s0, int n, const void* const* w2, const float* res, const float* skip, float* out32,
                         void* out16, void* s2d, ConvParams* out) {
        const void* in16 = rb_in16 ? rb_in16 : ws.a16[L];
        void* mid16 = in16 == ws.t16[L] ? ws.a16[L] : ws.t16[L];          // intermediate ReLU(conv1(x)) (unfused launches only)
        out[0] = conv3(g[L], n, C[L], at(in16, L, s0), w2[0], 1);
        out[0].out16 = at(mid16, L, s0);
        out[1] = conv3(g[L], n, C[L], at(mid16, L, s0), w2[1], 0);
        out[1].res32 = (const float*)at(res, L, s0); out[1].skip32 = (const float*)at(skip, L, s0);
        out[1].out32 = (float*)at(out32, L, s0); out[1].out16 = at(out16, L, s0);
        if (s2d) { out[1].s2d = at(s2d, L + 1, s0); out[1].gc = g[L + 1]; out[1].gc.M = n * g[L + 1].S; }
    };
    // head/tail fusion hooks for the second conv of the next resblock() call (level 0, consumed once)
    bool ht_res_is_head = false, ht_skip_is_head = false, ht_tail = false, ht_drop_skip = false;
    auto resblock = [&](int L, int s0, int n, const void* const* w2, const float* res, const float* skip, float* out32,
                        void* out16, void* s2d) -> int {
        ConvParams p[2];
        rb_params(L, s0, n, w2, res, skip, out32, out16, s2d, p);
        if (ht_res_is_head || ht_skip_is_head) {
            p[1].head_t = at4(ws.tpad, s0); p[1].head_w = W->head_h;
            if (ht_res_is_head) p[1].res32 = nullptr; else p[1].skip32 = nullptr;
        }
        if (ht_drop_skip) p[1].skip32 = nullptr;          // the U-Net skip x1 enters through the composite stencil of k_tail_gather
        if (ht_tail) { p[1].tail_part = at4(ws.tail_part, s0); p[1].tail_w = W->tail_h; p[1].out32 = nullptr; p[1].out16 = nullptr; }
        ht_res_is_head = ht_skip_is_head = ht_tail = ht_drop_skip = false;
        rb_in16 = nullptr;
        if (hilo) {           // stream values travel as fp16 hi (= the ResBlock's fp16 input / output) + fp16 lo
            auto is_stream = [&](const float* q) {
                return q && (q == (const float*)at(ws.p32a[L], L, s0) || (L < 3 && q == (const float*)at(ws.p32b[L], L, s0)));
            };
            if (is_stream(p[1].res32)) { p[1].res_hi = p[0].a; p[1].res_lo = at(ws.lo16[L], L, s0); p[1].res32 = nullptr; }
            if (is_stream(p[1].out32) && p[1].out16) { p[1].out_lo = at(ws.lo16[L], L, s0); p[1].out32 = nullptr; }
        }
        // fused kernel, except (mode 1) for the two ResBlocks whose epilogue recomputes m_head / reduces against m_tail: those
        // FMA-heavy epilogues are faster on the eight 32-channel epilogue warps of conv_umma.cu (profiles/README);
        // GDECONV_FUSE_RB=2 fuses them too
        if (prec == PREC_FP16_UMMA && fuse_rb_mode() && conv_rb_supported(p[0], p[1]) &&
            (fuse_rb_mode() >= 2 || (!p[1].tail_part && !p[1].head_t)))
            return launch_conv_rb(p[0], p[1], st);
        if (p[0].a == p[0].out16 || p[1].a == p[1].out16) GD_FAIL(GD_EUNSUPPORTED, "resblock: in-place fp16 buffers need the fused kernel");
        GD_TRY(run_conv(p[0], prec, st));
        return run_conv(p[1], prec, st);
    };
    // two consecutive ResBlocks of one level: one chained launch when all four layers' weights fit in shared memory
    auto resblock_pair = [&](int L, int s0, int n, const void* const* wa, const void* const* wb, const float* res_a, float* out32_a,
                             void* out16_a, const float* res_b, const float* skip_b, float* out32_b, void* out16_b, void* s2d_b) -> int {
        const bool last_l0 = fuse && L == 0 && skip_b != nullptr;       // second ResBlock of m_up1: + x1, then m_tail
        const bool first_ht = fuse && L == 0 && res_a == ws.skip32[0];        // first ResBlock of m_down1: residual = x1
        if (first_ht) ht_res_is_head = true;
        // the first ResBlock writes its fp16 output to t16 when it runs in the fused kernel (no in-place halo race)
        const bool pingpong = prec == PREC_FP16_UMMA && fuse_rb_mode() && C[L] == 32 && out16_a == ws.a16[L] &&
                              (fuse_rb_mode() >= 2 || !first_ht);
        GD_TRY(resblock(L, s0, n, wa, res_a, nullptr, out32_a, pingpong ? ws.t16[L] : out16_a, nullptr));
        if (last_l0) { ht_skip_is_head = !tail_g_mode(); ht_tail = true; ht_drop_skip = tail_g_mode() != 0; }
        if (pingpong) rb_in16 = ws.t16[L];
        return resblock(L, s0, n, wb, res_b, skip_b, out32_b, out16_b, s2d_b);
    };
    auto down_stage = [&](int L, int s0, int n) -> int {          // m_down{L+1} (ResUNet.py:32-34)
        if (L == 0 && l1chain) {
            const void* w4[4] = {W->down_rb[0][0][0], W->down_rb[0][0][1], W->down_rb[0][1][0], W->down_rb[0][1][1]};
            // ... and the k2s2 strided conv of m_down1 (its space-to-depth operand never leaves shared memory)
            return launch_l1chain_down(g[0], g[1], n, t + (size_t)s0 * NPIX, W->head_h, w4, W->down[0], (float*)at(ws.skip32[1], 1, s0),
                                       at(ws.a16[1], 1, s0), l2chain ? at(ws.lo16[1], 1, s0) : nullptr, st);
        }
        if (L == 1 && l2chain) {
            const void* w4[4] = {W->down_rb[1][0][0], W->down_rb[1][0][1], W->down_rb[1][1][0], W->down_rb[1][1][1]};
            // ... and the k2s2 strided conv of m_down2 (its space-to-depth operand never leaves shared memory)
            return launch_l2chain(0, g[1], g[2], n, at(ws.a16[1], 1, s0), at(ws.lo16[1], 1, s0), w4, W->down[1], (float*)at(ws.skip32[2], 2, s0),
                                  at(ws.a16[2], 2, s0), nullptr, nullptr, nullptr, nullptr, nullptr, st);
        } else
            GD_TRY(resblock_pair(L, s0, n, W->down_rb[L][0], W->down_rb[L][1], ws.skip32[L], ws.p32a[L], ws.a16[L], ws.p32a[L], nullptr,
                                 nullptr, nullptr, ws.d16[L + 1]));
        ConvParams p = conv_base(g[L + 1], n);         // k2s2 strided conv as a 1-tap GEMM on the space-to-depth copy
        p.ntaps = 1; p.off[0] = 0; p.Kt = 4 * C[L]; p.N = C[L + 1]; p.a = at(ws.d16[L + 1], L + 1, s0); p.w = W->down[L];
        p.out32 = (float*)at(ws.skip32[L + 1], L + 1, s0); p.out16 = at(ws.a16[L + 1], L + 1, s0);
        return run_conv(p, prec, st);
    };
    auto up_stage = [&](int L, int s0, int n) -> int {            // m_up{L+1} (ResUNet.py:36-38)
        if (L == 0 && l1chain) {          // transposed conv + both ResBlocks + m_tail partial sums in one launch
            const void* w4[4] = {W->up_rb[0][0][0], W->up_rb[0][0][1], W->up_rb[0][1][0], W->up_rb[0][1][1]};
            return launch_l1chain_up(g[0], g[1], n, at(ws.a16[1], 1, s0), W->up0_plain, W->tail_h, w4, at4(ws.tail_part, s0), ws.lc_scratch, st);
        }
        if (L == 1 && l2chain) {          // transposed conv + both ResBlocks + U-Net skip in one launch
            const void* w4[4] = {W->up_rb[1][0][0], W->up_rb[1][0][1], W->up_rb[1][1][0], W->up_rb[1][1][1]};
            return launch_l2chain(1, g[1], g[2], n, nullptr, nullptr, w4, nullptr, nullptr, nullptr, at(ws.a16[2], 2, s0), W->up1_plain, ws.lc_scratch,
                                  (const float*)at(ws.skip32[1], 1, s0), at(ws.a16[1], 1, s0), st);
        }
        ConvParams p = conv_base(g[L + 1], n);         // k2s2 transposed conv: GEMM on the coarse level, scatter to fine
        p.ntaps = 1; p.off[0] = 0; p.Kt = C[L + 1]; p.N = 4 * C[L]; p.a = at(ws.a16[L + 1], L + 1, s0); p.w = W->up[L];
        p.mode = 1; p.Cf = C[L]; p.Cf_log2 = 0; while ((1 << p.Cf_log2) < p.Cf) ++p.Cf_log2; p.gf = g[L]; p.gf.M = n * g[L].S;
        p.out32 = (float*)at(ws.p32a[L], L, s0); p.out16 = at(ws.a16[L], L, s0);
        if (hilo) { p.out_lo = at(ws.lo16[L], L, s0); p.out32 = nullptr; }
        GD_TRY(run_conv(p, prec, st));
        if (L > 0) return resblock_pair(L, s0, n, W->up_rb[L][0], W->up_rb[L][1], ws.p32a[L], ws.p32b[L], ws.a16[L], ws.p32b[L],
                                        ws.skip32[L], nullptr, ws.a16[L], nullptr);
        return resblock_pair(L, s0, n, W->up_rb[L][0], W->up_rb[L][1], ws.p32a[L], ws.p32b[L], ws.a16[L], ws.p32b[L], ws.skip32[L],
                             ws.p32a[L], nullptr, nullptr);
    };
    GD_TRY(down_stage(0, 0, nb));
    GD_TRY(down_stage(1, 0, nb));
    GD_TRY(down_stage(2, 0, nb));
    // m_body (ResUNet.py:35) and the skip x + x4 (:36)
    GD_TRY(resblock(3, 0, nb, W->body_rb[0], ws.skip32[3], nullptr, ws.p32a[3], ws.a16[3], nullptr));
    GD_TRY(resblock(3, 0, nb, W->body_rb[1], ws.p32a[3], ws.skip32[3], nullptr, ws.a16[3], nullptr));
    GD_TRY(up_stage(2, 0, nb));
    GD_TRY(up_stage(1, 0, nb));
    GD_TRY(up_stage(0, 0, nb));
    // tail (ResUNet.py:39): conv(x + x1), times the per-stamp input scale
    if (l1chain) return launch_tail_gather(ws.tail_part, 1, g[0], tscale, zout, nb, t, W->tail_head_g, st, 1);
    if (fuse) return launch_tail_gather(ws.tail_part, (fuse_rb_mode() >= 2 && C[0] == 32) ? 2 : C[0] / 32, g[0], tscale, zout, nb,
                                        ws.tpad, tail_g_mode() ? W->tail_head_g : nullptr, st);
    return launch_tail(ws.p32a[0], W->tail, C[0], g[0], tscale, zout, nb, st);
}

static int g_fuse_ht_fwd() { return fuse_ht_mode(); }

static int rho_chunk(const GdWeights* W, const Ws& ws, const float* psf, const float* alpha, int nb, cudaStream_t st) {
    if (W->has_subnet) return launch_subnet(W->sub, psf, alpha, ws.rho, nb, st);
    if (W->has_rho_param) return launch_fill_rho(W->rho_param, W->n_rho, ws.rho, nb, st);
    GD_FAIL(GD_EBADSHAPE, "weights hold neither a SubNet nor rho parameters");
}

static int copy_f32(float* dst, const float* src, size_t n, cudaStream_t st) {
    GD_CUDA_CHECK(cudaMemcpyAsync(dst, src, n * sizeof(float), cudaMemcpyDeviceToDevice, st));
    return GD_OK;
}

}  // namespace gd

extern "C" int gd_max_chunk(void) {
    // largest chunk whose level-0 GEMM rows (2401 per stamp + tile/halo slack) stay below the 2^26 limit of div_by_magic
    int lo = 1, hi = 1 << 20;
    while (lo < hi) { const int mid = lo + (hi - lo + 1) / 2; if (geom_rows_ok(STAMP, mid)) lo = mid; else hi = mid - 1; }
    return lo;
}

extern "C" long long gd_debug_divmagic(unsigned d, unsigned n_lo, unsigned n_hi) {
    // host-side exhaustive check of the multiply-shift division the kernels decode rows with; -1 = exact on [n_lo, n_hi)
    uint32_t magic, shift;
    div_magic(d, &magic, &shift);
    for (unsigned n = n_lo; n < n_hi; ++n)
        if (div_by_magic(n, magic, shift) != n / d) return (long long)n;
    return -1;
}

extern "C" size_t gd_workspace_bytes(int arch, int precision, int chunk) {
    if ((arch != GD_ARCH_G && arch != GD_ARCH_U) || precision < 0 || precision > 2 || chunk < 1) return 0;
    if (!geom_rows_ok(STAMP, chunk)) return 0;            // row decode (div_by_magic) is only exact below 2^26 rows
    return ws_layout(nullptr, arch, precision, chunk).total;
}

extern "C" int gd_workspace_init(void* workspace, size_t bytes, int arch, int precision, int chunk, void* stream) {
    cudaStream_t st = (cudaStream_t)stream;
    size_t need = gd_workspace_bytes(arch, precision, chunk);
    if (!need) GD_FAIL(GD_EBADSHAPE, "bad workspace parameters (arch %d, precision %d, chunk %d; the largest chunk is %d stamps)", arch, precision, chunk, gd_max_chunk());
    if (!workspace || bytes < need) GD_FAIL(GD_EWORKSPACE, "workspace of %zu bytes is smaller than the %zu needed for chunk %d", bytes, need, chunk);
    GD_CUDA_CHECK(cudaMemsetAsync(workspace, 0, need, st));
    WsHeader h = {WS_MAGIC, arch, precision, chunk, (uint64_t)need};
    GD_CUDA_CHECK(cudaMemcpyAsync(workspace, &h, sizeof(h), cudaMemcpyHostToDevice, st));
    GD_CUDA_CHECK(cudaStreamSynchronize(st));
    std::lock_guard<std::mutex> lk(g_ws_mu);
    g_ws_reg[workspace] = h;
    return GD_OK;
}

// Forgets a workspace registered by gd_workspace_init (call before freeing its memory: the allocator may hand the same address to
// an unrelated buffer, which must not pass gd_admm_forward's workspace check).
extern "C" void gd_workspace_release(void* workspace) {
    std::lock_guard<std::mutex> lk(g_ws_mu);
    g_ws_reg.erase(workspace);
}

extern "C" int gd_resunet_forward(const GdWeights* W, const float* in, float* out, int batch, void* workspace,
                                  size_t workspace_bytes, void* stream) {
    cudaStream_t st = (cudaStream_t)stream;
    if (!W || !W->has_resunet) GD_FAIL(GD_EBADSHAPE, "weights hold no ResUNet");
    if (batch < 0 || (batch && (!in || !out))) GD_FAIL(GD_EBADSHAPE, "gd_resunet_forward: bad batch or NULL buffers");
    GD_DEVICE_SCOPE(W->device);
    Ws ws; int chunk;
    GD_TRY(ws_check(workspace, workspace_bytes, W, &ws, &chunk));
    for (int c0 = 0; c0 < batch; c0 += chunk) {
        const int nb = batch - c0 < chunk ? batch - c0 : chunk;
        GD_TRY(launch_scale_in(in + (size_t)c0 * NPIX, ws.t, ws.tscale, nb, st));
        GD_TRY(resunet_chunk(W, ws, ws.t, ws.tscale, out + (size_t)c0 * NPIX, nb, st));
    }
    return GD_OK;
}

extern "C" int gd_subnet_forward(const GdWeights* W, const float* psf, const float* alpha, float* rho_out, int batch,
                                 void* stream) {
    if (!W || !W->has_subnet) GD_FAIL(GD_EBADSHAPE, "weights hold no SubNet");
    if (batch < 0 || (batch && (!psf || !alpha || !rho_out))) GD_FAIL(GD_EBADSHAPE, "gd_subnet_forward: bad batch or NULL buffers");
    GD_DEVICE_SCOPE(W->device);
    return launch_subnet(W->sub, psf, alpha, rho_out, batch, (cudaStream_t)stream);
}

// Path U on one chunk (models/Unrolled_ADMM.py:177-215, :396-442; models/ADMMNet.py:97-129) with the Z-update supplied by the caller:
// `zupdate` maps the denoiser input ws.t (scaled by ws.tscale when `scaled`) to ws.z.  `analysis` points at this chunk's first stamp.
template <class ZUpdate>
static int admm_u_chunk(const GdWeights* W, const Ws& ws, int llh, int flags, const float* yc, const float* kc, const float* ac, float* outc,
                        float* analysis, size_t plane, int nb, cudaStream_t st, bool scaled, ZUpdate zupdate) {
    const int n = W->n_iters, nr = W->n_rho;
    const size_t ni = (size_t)nb * NPIX;
    float* u1 = ws.u;
    GD_TRY(launch_u_prologue(yc, kc, ac, flags & 1, ws.spec, ws.x, ws.z, ws.v, u1, ws.u2, ws.Hx, nb, st));
    auto dump = [&](int slot) -> int {
        if (!analysis) return GD_OK;
        float* A = analysis + (size_t)slot * 5 * plane;
        const float* src[5] = {ws.v, ws.z, ws.x, u1, ws.u2};
        for (int q = 0; q < 5; ++q) GD_TRY(copy_f32(A + q * plane, src[q], ni, st));
        return GD_OK;
    };
    GD_TRY(dump(0));
    for (int it = 0; it < n; ++it) {
        GD_TRY(launch_u_pre(llh, yc, ac, ws.rho, nr, n, it, ws.x, u1, ws.u2, ws.Hx, ws.v, ws.t, scaled ? ws.tscale : nullptr, nb, st));
        GD_TRY(zupdate());
        GD_TRY(launch_u_post(ws.spec, ws.rho, nr, n, it, ws.z, ws.v, ws.x, u1, ws.u2, ws.Hx, nb, st));
        GD_TRY(dump(it + 1));
    }
    return launch_scale_by_alpha(outc, ws.x, ac, nb, llh == GD_LLH_POISSON || (flags & 2), st);     // Unrolled_ADMM.py:215 / ADMMNet.py:129
}

extern "C" int gd_admm_forward(const GdWeights* W, int llh, int u_v0_over_alpha, const float* y, const float* psf,
                               const float* alpha, float* out, float* rho_out, float* analysis, int batch,
                               void* workspace, size_t workspace_bytes, void* stream) {
    cudaStream_t st = (cudaStream_t)stream;
    if (!W || !W->has_resunet) GD_FAIL(GD_EBADSHAPE, "weights hold no ResUNet");
    if (batch < 0 || (batch && (!y || !psf || !alpha || !out))) GD_FAIL(GD_EBADSHAPE, "gd_admm_forward: bad batch or NULL buffers");
    if (llh != GD_LLH_GAUSSIAN && llh != GD_LLH_POISSON) GD_FAIL(GD_EUNSUPPORTED, "unknown likelihood %d", llh);
    GD_DEVICE_SCOPE(W->device);
    Ws ws; int chunk;
    GD_TRY(ws_check(workspace, workspace_bytes, W, &ws, &chunk));
    const int n = W->n_iters, nr = W->n_rho;
    const size_t plane = (size_t)batch * NPIX;
    for (int c0 = 0; c0 < batch; c0 += chunk) {
        const int nb = batch - c0 < chunk ? batch - c0 : chunk;
        const size_t o = (size_t)c0 * NPIX, ni = (size_t)nb * NPIX;
        const float *yc = y + o, *kc = psf + o, *ac = alpha + c0;
        GD_TRY(rho_chunk(W, ws, kc, ac, nb, st));
        if (rho_out) GD_TRY(copy_f32(rho_out + (size_t)c0 * nr, ws.rho, (size_t)nb * nr, st));
        if (W->arch == GD_ARCH_G) {
            GD_TRY(launch_g_prologue(yc, kc, ac, ws.spec, ws.HtH, ws.z, ws.u, ws.x, nb, st));
            if (n == 0) GD_TRY(copy_f32(out + o, ws.z, ni, st));
            for (int it = 0; it < n; ++it) {
                const bool xh = xhead_applies(W);
                if (xh) GD_TRY(launch_g_xupdate(ws.spec, ws.HtH, ws.rho, nr, it, ws.z, ws.x, ws.u, ws.t, ws.tscale, nb, st, W->head_h, &ws.g[0], ws.a16[0], ws.tpad));
                else GD_TRY(launch_g_xupdate(ws.spec, ws.HtH, ws.rho, nr, it, ws.z, ws.x, ws.u, ws.t, ws.tscale, nb, st));
                float* zdst = it == n - 1 ? out + o : ws.z;
                GD_TRY(resunet_chunk(W, ws, ws.t, ws.tscale, zdst, nb, st, xh));
                if (analysis) {
                    float* A = analysis + (size_t)it * 3 * plane + o;
                    GD_TRY(copy_f32(A, ws.x, ni, st));
                    GD_TRY(copy_f32(A + plane, zdst, ni, st));
                    GD_TRY(launch_g_dual_out(ws.rho, nr, it, ws.x, zdst, ws.u, A + 2 * plane, nb, st));
                }
            }
        } else {
            GD_TRY(admm_u_chunk(W, ws, llh, u_v0_over_alpha, yc, kc, ac, out + o, analysis ? analysis + o : nullptr, plane, nb, st, true,
                                [&]() { return resunet_chunk(W, ws, ws.t, ws.tscale, ws.z, nb, st); }));
        }
    }
    return GD_OK;
}

// Unrolled_ADMM / ADMMNet with denoiser='XDenseUNet' (models/Unrolled_ADMM.py:142-151,163; models/ADMMNet.py:65-74,87): the path-U loop of
// gd_admm_forward with the Z-update z = XDenseUNet(x + u1) run by csrc/xdense.cu in fp32 on the UNSCALED input.  `W` carries the SubNet or
// the rho parameters only (packed from the same state_dict; it need not hold a ResUNet), `X` the packed XDenseUNet.
extern "C" int gd_admm_forward_xdense(const GdWeights* W, const GdXDense* X, int llh, int flags, const float* y, const float* psf,
                                      const float* alpha, float* out, float* rho_out, float* analysis, int batch, void* workspace,
                                      size_t workspace_bytes, void* xd_workspace, size_t xd_workspace_bytes, int xd_chunk, void* stream) {
    cudaStream_t st = (cudaStream_t)stream;
    if (!W || !X) GD_FAIL(GD_EBADSHAPE, "gd_admm_forward_xdense: NULL weights");
    if (W->arch != GD_ARCH_U) GD_FAIL(GD_EUNSUPPORTED, "the XDenseUNet denoiser exists for Unrolled_ADMM / ADMMNet (arch U) only");
    if (batch < 0 || (batch && (!y || !psf || !alpha || !out))) GD_FAIL(GD_EBADSHAPE, "gd_admm_forward_xdense: bad batch or NULL buffers");
    if (llh != GD_LLH_GAUSSIAN && llh != GD_LLH_POISSON) GD_FAIL(GD_EUNSUPPORTED, "unknown likelihood %d", llh);
    GD_DEVICE_SCOPE(W->device);
    Ws ws; int chunk;
    GD_TRY(ws_check(workspace, workspace_bytes, W, &ws, &chunk));
    const int nr = W->n_rho;
    const size_t plane = (size_t)batch * NPIX;
    for (int c0 = 0; c0 < batch; c0 += chunk) {
        const int nb = batch - c0 < chunk ? batch - c0 : chunk;
        const size_t o = (size_t)c0 * NPIX;
        GD_TRY(rho_chunk(W, ws, psf + o, alpha + c0, nb, st));
        if (rho_out) GD_TRY(copy_f32(rho_out + (size_t)c0 * nr, ws.rho, (size_t)nb * nr, st));
        GD_TRY(admm_u_chunk(W, ws, llh, flags, y + o, psf + o, alpha + c0, out + o, analysis ? analysis + o : nullptr, plane, nb, st, false,
                            [&]() { return gd_xdense_forward(X, ws.t, ws.z, nb, xd_workspace, xd_workspace_bytes, xd_chunk, stream); }));
    }
    return GD_OK;
}

extern "C" int gd_fft_solver(int kind, int n_iters, float lam, const float* y, const float* psf, const float* alpha,
                             float* out, int batch, void* stream) {
    if (kind < 0 || kind > 3) GD_FAIL(GD_EUNSUPPORTED, "unknown solver kind %d", kind);
    if (batch < 0 || (batch && (!y || !psf || !out))) GD_FAIL(GD_EBADSHAPE, "gd_fft_solver: bad batch or NULL buffers");
    if (kind != GD_SOLVER_RL && batch && !alpha) GD_FAIL(GD_EBADSHAPE, "gd_fft_solver: alpha is required for Wiener/Tikhonov");
    if (kind == GD_SOLVER_RL && n_iters < 0) GD_FAIL(GD_EBADSHAPE, "gd_fft_solver: n_iters < 0");
    int dev;
    GD_CUDA_CHECK(cudaGetDevice(&dev));
    GD_TRY(init_once(dev));
    return launch_solver(kind, n_iters, lam, y, psf, alpha, out, batch, (cudaStream_t)stream);
}

extern "C" int gd_conv_fft(const float* x, const float* psf, float* out, int adjoint, int batch, void* stream) {
    if (batch < 0 || (batch && (!x || !psf || !out))) GD_FAIL(GD_EBADSHAPE, "gd_conv_fft: bad batch or NULL buffers");
    int dev;
    GD_CUDA_CHECK(cudaGetDevice(&dev));
    GD_TRY(init_once(dev));
    return launch_conv_fft(x, psf, out, adjoint, batch, (cudaStream_t)stream);
}

extern "C" int gd_psf_to_otf(const float* ker, int ker_batch, int kh, int kw, float* psf_out, float* otf_out, int batch, void* stream) {
    if (batch < 0 || (batch && (!ker || !psf_out || !otf_out))) GD_FAIL(GD_EBADSHAPE, "gd_psf_to_otf: bad batch or NULL buffers");
    if (kh < 1 || kw < 1 || kh > STAMP || kw > STAMP) GD_FAIL(GD_EBADSHAPE, "gd_psf_to_otf: kernel %dx%d does not fit a 48x48 stamp", kh, kw);
    if (ker_batch != 1 && ker_batch != batch) GD_FAIL(GD_EBADSHAPE, "gd_psf_to_otf: kernel batch %d must be 1 or %d", ker_batch, batch);
    // the reference's slice assignments only broadcast a source dimension of 1 or `centre` (anything else raises in torch)
    const int ce = (kh + 1) / 2;
    if ((kh - ce != 1 && kh - ce != ce) || (kw - ce != 1 && kw - ce != ce) || 2 * ce > STAMP)
        GD_FAIL(GD_EBADSHAPE, "gd_psf_to_otf: a %dx%d kernel cannot be broadcast by the reference's quadrant assignment", kh, kw);
    int dev;
    GD_CUDA_CHECK(cudaGetDevice(&dev));
    GD_TRY(init_once(dev));
    return launch_psf_to_otf(ker, ker_batch, kh, kw, psf_out, reinterpret_cast<float2*>(otf_out), batch, (cudaStream_t)stream);
}

extern "C" int gd_conv_otf(const float* otf, int otf_batch, const float* x, float* out, int batch, void* stream) {
    if (batch < 0 || (batch && (!otf || !x || !out))) GD_FAIL(GD_EBADSHAPE, "gd_conv_otf: bad batch or NULL buffers");
    if (otf_batch != 1 && otf_batch != batch) GD_FAIL(GD_EBADSHAPE, "gd_conv_otf: OTF batch %d must be 1 or %d", otf_batch, batch);
    int dev;
    GD_CUDA_CHECK(cudaGetDevice(&dev));
    GD_TRY(init_once(dev));
    return launch_conv_otf(reinterpret_cast<const float2*>(otf), otf_batch, x, out, batch, (cudaStream_t)stream);
}

extern "C" int gd_moments_e(const float* img, float* e12, int batch, void* stream) {
    if (batch < 0 || (batch && (!img || !e12))) GD_FAIL(GD_EBADSHAPE, "gd_moments_e: bad batch or NULL buffers");
    return launch_moments(img, e12, batch, (cudaStream_t)stream);
}

extern "C" int gd_synth_batch(int64_t start, int count, int64_t seed, int snr_mode, float snr, float psf_fwhm_err,
                              float psf_shear_err, float* obs, float* psf, float* alpha, float* gt, void* stream) {
    if (count < 0) GD_FAIL(GD_EBADSHAPE, "gd_synth_batch: count %d < 0", count);
    if (!obs && !psf && !alpha && !gt) GD_FAIL(GD_EBADSHAPE, "gd_synth_batch: every output is NULL");
    if (snr_mode != GD_SYNTH_SNR_FIXED && snr_mode != GD_SYNTH_SNR_MIXED)
        GD_FAIL(GD_EBADSHAPE, "gd_synth_batch: unknown snr_mode %d", snr_mode);
    if (snr_mode == GD_SYNTH_SNR_FIXED && !(snr > 0.f && isfinite(snr)))
        GD_FAIL(GD_EBADSHAPE, "gd_synth_batch: snr must be positive and finite in fixed mode, got %g", (double)snr);
    if (start < 0 || start > INT64_MAX - count) GD_FAIL(GD_EBADSHAPE, "gd_synth_batch: stamp range [%lld, +%d) out of range", (long long)start, count);
    if (!isfinite(psf_fwhm_err) || !isfinite(psf_shear_err)) GD_FAIL(GD_EBADSHAPE, "gd_synth_batch: non-finite PSF error");
    if (count == 0) return GD_OK;
    int dev;
    GD_CUDA_CHECK(cudaGetDevice(&dev));
    GD_TRY(init_once(dev));
    return launch_synth(start, count, seed, snr_mode == GD_SYNTH_SNR_MIXED, snr, psf_fwhm_err, psf_shear_err, obs, psf, alpha, gt,
                        (cudaStream_t)stream);
}

extern "C" int gd_adaptive_moments(const float* img, int batch, float guess_sigma, float* shape, int32_t* info, void* stream) {
    if (batch < 0) GD_FAIL(GD_EBADSHAPE, "gd_adaptive_moments: batch %d < 0", batch);
    if (batch && (!img || !shape || !info)) GD_FAIL(GD_EBADSHAPE, "gd_adaptive_moments: NULL buffer for a batch of %d", batch);
    if (!(isfinite(guess_sigma) && guess_sigma > 0.f && guess_sigma <= 24.f))
        GD_FAIL(GD_EBADSHAPE, "gd_adaptive_moments: guess_sigma must be finite and in (0, 24] px, got %g", (double)guess_sigma);
    if (batch == 0) return GD_OK;
    int dev;
    GD_CUDA_CHECK(cudaGetDevice(&dev));
    GD_TRY(init_once(dev));
    return launch_adaptive_moments(img, batch, guess_sigma, shape, info, (cudaStream_t)stream);
}

extern "C" int gd_debug_geom(int H, int batch, int* geom7) {
    if (H < 1 || batch < 1 || !geom7) GD_FAIL(GD_EBADSHAPE, "gd_debug_geom: bad arguments");
    Geom g = make_geom(H, batch);
    const int v[7] = {g.H, g.W, g.Wp, g.S, g.base0, g.Ptot, g.M};
    memcpy(geom7, v, sizeof(v));
    return GD_OK;
}

extern "C" int gd_debug_tapgemm(int precision, int H, int batch, int ntaps, int Kt, int N, int relu, const void* act,
                                const void* weights, float* out32, void* stream) {
    if (precision < 0 || precision > 2 || (ntaps != 1 && ntaps != 9) || !act || !weights || !out32 || batch < 1)
        GD_FAIL(GD_EBADSHAPE, "gd_debug_tapgemm: bad arguments");
    int dev;
    GD_CUDA_CHECK(cudaGetDevice(&dev));
    GD_TRY(init_once(dev));
    Geom g = make_geom(H, batch);
    ConvParams p = ntaps == 9 ? conv3(g, batch, Kt, act, weights, relu) : conv_base(g, batch);
    if (ntaps == 1) { p.ntaps = 1; p.off[0] = 0; p.a = act; p.w = weights; p.relu = relu; }
    p.Kt = Kt; p.N = N; p.out32 = out32;
    return run_conv(p, precision, (cudaStream_t)stream);
}

extern "C" void gd_profile_begin(void) { conv_profile_begin(); }
extern "C" int gd_profile_end(double* ms_total, double* flops_total, uint64_t* launches) {
    unsigned long long n = 0;
    int rc = conv_profile_end(ms_total, flops_total, &n);
    if (launches) *launches = n;
    return rc;
}
