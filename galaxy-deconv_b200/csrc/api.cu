// C ABI of libgdeconv (include/gdeconv.h): weight packing, workspace layout, the ResUNet layer graph and the
// unrolled-ADMM drivers.  Host code only; every kernel lives in fft_kernels.cu / subnet.cu / conv_*.cu.
#include <array>
#include <atomic>
#include <cstdarg>
#include <cstdio>
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
// paired: columns ordered for the lane-paired stores of epi_up_unit (conv_epilogue.cuh), the order k_conv_umma's transposed
// conv writes; the chain kernels (conv_l1chain.cu, conv_l2chain.cu) and the SIMT kernel read the plain order
static int pack_up(Blob& bl, const GdTensorDesc* t, int Ci, int Co, int prec, bool paired, size_t* off, const char* what) {
    if (!shape_is(t, Ci, Co, 2, 2)) GD_FAIL(GD_EBADSHAPE, "weight %s: missing or not (%d,%d,2,2)", what, Ci, Co);
    std::vector<float> B((size_t)Ci * 4 * Co);
    for (int ci = 0; ci < Ci; ++ci)
        for (int co = 0; co < Co; ++co)
            for (int tp = 0; tp < 4; ++tp) {
                const int dy = tp >> 1, dx = tp & 1;
                const int n = paired ? dy * 2 * Co + (co / 16) * 32 + ((co % 16) / 4) * 8 + dx * 4 + (co % 4) : tp * Co + co;
                B[(size_t)ci * 4 * Co + n] = t->data[((size_t)ci * Co + co) * 4 + tp];
            }
    *off = pack_tapgemm(bl, 1, Ci, 4 * Co, prec, B);
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
    GD_TRY(conv_l1chain_init());
    GD_TRY(conv_l2chain_init());
    GD_TRY(synth_init());
    GD_TRY(fpfs_init());
    GD_TRY(metacal_init());
    GD_TRY(metacal_fixnoise_init());
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
            // tcgen05 path: on path G (C0 = 32) m_up1 and m_up2 run inside the chain kernels
            const bool paired = precision == PREC_FP16_UMMA && !(C0 == 32 && L < 2);
            GD_TRY(pack_up(bl, F.net(key), 2 * C, C, precision, paired, &off, key));
            slot(&W.up[L], off);
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
    // per-tap m_tail partial sums: k_conv_umma writes C0 / 32 units of 9 planes, k_l1_chain one unit.  The C0 / 16 units allocated
    // are twice that; shrinking them would change what gd_workspace_bytes reports.
    w.tail_part = (float*)take((size_t)(C0 / 16) * 9 * w.g[0].Ptot * 4);
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

// Two graphs, chosen by the precision mode:
//   * fp16_umma, the tcgen05 graph.  The fp32 output x1 of m_head is never stored: the conv epilogues that consume it recompute it
//     from the padded-linear input copy tpad (ConvParams::head_t), and m_tail runs as per-tap partial sums (ConvParams::tail_part)
//     that k_tail_gather shifts and adds, with m_tail(x1) as an 81-coefficient stencil of t.  The residual stream travels as fp16
//     hi/lo: the fp32 stream buffers p32a / p32b are replaced by hi = the fp16 operand copy a16 and lo = lo16.  On path G
//     (C0 = 32) levels 0 and 1 run in the chain kernels (conv_l1chain.cu, conv_l2chain.cu), one launch per stage.
//   * fp32_simt / fp16_simt, the validation graph: one launch per layer, fp32 stream buffers, k_head and k_tail.
static int resunet_chunk(const GdWeights* W, const Ws& ws, const float* t, const float* tscale, float* zout, int nb, cudaStream_t st) {
    const int prec = W->precision;
    const Geom* g = ws.g;
    const int* C = ws.C;
    const bool fused = prec == PREC_FP16_UMMA;
    const bool chain = fused && C[0] == 32;
    // one ResBlock (resnet_basicblock.py:69-71) on ws.a16[L]: conv + ReLU -> ws.t16[L], conv + res (+ skip) -> out32 / out16 / s2d
    auto resblock_params = [&](int L, const void* const* w2, const float* res, const float* skip, float* out32, void* out16, void* s2d,
                               ConvParams* p) {
        p[0] = conv3(g[L], nb, C[L], ws.a16[L], w2[0], 1);
        p[0].out16 = ws.t16[L];
        p[1] = conv3(g[L], nb, C[L], ws.t16[L], w2[1], 0);
        p[1].res32 = res; p[1].skip32 = skip; p[1].out32 = out32; p[1].out16 = out16;
        if (s2d) { p[1].s2d = s2d; p[1].gc = g[L + 1]; p[1].gc.M = nb * g[L + 1].S; }
        if (fused) {
            auto is_stream = [&](const float* q) { return q && (q == ws.p32a[L] || q == ws.p32b[L]); };
            if (is_stream(p[1].res32)) { p[1].res_hi = p[0].a; p[1].res_lo = ws.lo16[L]; p[1].res32 = nullptr; }
            if (is_stream(p[1].out32) && p[1].out16) { p[1].out_lo = ws.lo16[L]; p[1].out32 = nullptr; }
        }
    };
    auto run_pair = [&](const ConvParams* p) -> int {
        GD_TRY(run_conv(p[0], prec, st));
        return run_conv(p[1], prec, st);
    };
    auto resblock = [&](int L, const void* const* w2, const float* res, const float* skip, float* out32, void* out16, void* s2d) -> int {
        ConvParams p[2];
        resblock_params(L, w2, res, skip, out32, out16, s2d, p);
        return run_pair(p);
    };
    auto w4 = [](const void* const (*rb)[2]) -> std::array<const void*, 4> { return {rb[0][0], rb[0][1], rb[1][0], rb[1][1]}; };

    // m_head (ResUNet.py:31): x1 = conv(t) -> skip32[0] (fp32, validation graph) + a16[0]; tpad (tcgen05 graph)
    if (!chain) {
        ConvParams p = conv_base(g[0], nb);
        p.N = C[0]; p.out32 = fused ? nullptr : ws.skip32[0]; p.out16 = ws.a16[0];
        GD_TRY(launch_head(t, W->head, C[0], p, nb, prec, fused ? ws.tpad : nullptr, st));
    }
    // m_down1..3 (ResUNet.py:32-34): two ResBlocks, then the k2s2 strided conv as a 1-tap GEMM on the space-to-depth copy
    for (int L = 0; L < 3; ++L) {
        if (chain && L == 0) {          // m_head + both ResBlocks + the strided conv (its operand never leaves shared memory)
            GD_TRY(launch_l1chain_down(g[0], g[1], nb, t, W->head_h, w4(W->down_rb[0]).data(), W->down[0], ws.skip32[1], ws.a16[1],
                                       ws.lo16[1], st));
            continue;
        }
        if (chain && L == 1) {          // both ResBlocks + the strided conv
            GD_TRY(launch_l2chain(0, g[1], g[2], nb, ws.a16[1], ws.lo16[1], w4(W->down_rb[1]).data(), W->down[1], ws.skip32[2], ws.a16[2],
                                  nullptr, nullptr, nullptr, nullptr, nullptr, st));
            continue;
        }
        ConvParams p[2];
        resblock_params(L, W->down_rb[L][0], ws.skip32[L], nullptr, ws.p32a[L], ws.a16[L], nullptr, p);
        if (fused && L == 0) { p[1].res32 = nullptr; p[1].head_t = ws.tpad; p[1].head_w = W->head_h; }     // residual x1, recomputed
        GD_TRY(run_pair(p));
        GD_TRY(resblock(L, W->down_rb[L][1], ws.p32a[L], nullptr, nullptr, nullptr, ws.d16[L + 1]));
        ConvParams d = conv_base(g[L + 1], nb);
        d.ntaps = 1; d.off[0] = 0; d.Kt = 4 * C[L]; d.N = C[L + 1]; d.a = ws.d16[L + 1]; d.w = W->down[L];
        d.out32 = ws.skip32[L + 1]; d.out16 = ws.a16[L + 1];
        GD_TRY(run_conv(d, prec, st));
    }
    // m_body (ResUNet.py:35) and the skip x + x4 (:36)
    GD_TRY(resblock(3, W->body_rb[0], ws.skip32[3], nullptr, ws.p32a[3], ws.a16[3], nullptr));
    GD_TRY(resblock(3, W->body_rb[1], ws.p32a[3], ws.skip32[3], nullptr, ws.a16[3], nullptr));
    // m_up3..1 (ResUNet.py:36-38): the k2s2 transposed conv (GEMM on the coarse level, scattered to the fine one), two ResBlocks,
    // the U-Net skip
    for (int L = 2; L >= 0; --L) {
        if (chain && L == 1) {          // transposed conv + both ResBlocks + U-Net skip
            GD_TRY(launch_l2chain(1, g[1], g[2], nb, nullptr, nullptr, w4(W->up_rb[1]).data(), nullptr, nullptr, nullptr, ws.a16[2], W->up[1],
                                  ws.lc_scratch, ws.skip32[1], ws.a16[1], st));
            continue;
        }
        if (chain && L == 0) {          // transposed conv + both ResBlocks + the m_tail partial sums
            GD_TRY(launch_l1chain_up(g[0], g[1], nb, ws.a16[1], W->up[0], W->tail_h, w4(W->up_rb[0]).data(), ws.tail_part, ws.lc_scratch, st));
            continue;
        }
        ConvParams u = conv_base(g[L + 1], nb);
        u.ntaps = 1; u.off[0] = 0; u.Kt = C[L + 1]; u.N = 4 * C[L]; u.a = ws.a16[L + 1]; u.w = W->up[L];
        u.mode = 1; u.Cf = C[L]; u.Cf_log2 = 0; while ((1 << u.Cf_log2) < u.Cf) ++u.Cf_log2; u.gf = g[L]; u.gf.M = nb * g[L].S;
        u.out32 = ws.p32a[L]; u.out16 = ws.a16[L];
        if (fused) { u.out_lo = ws.lo16[L]; u.out32 = nullptr; }
        GD_TRY(run_conv(u, prec, st));
        GD_TRY(resblock(L, W->up_rb[L][0], ws.p32a[L], nullptr, ws.p32b[L], ws.a16[L], nullptr));
        if (L > 0) {
            GD_TRY(resblock(L, W->up_rb[L][1], ws.p32b[L], ws.skip32[L], nullptr, ws.a16[L], nullptr));
        } else if (fused) {             // + x1 enters through the stencil of k_tail_gather; the result only feeds m_tail
            ConvParams p[2];
            resblock_params(0, W->up_rb[0][1], ws.p32b[0], nullptr, nullptr, nullptr, nullptr, p);
            p[1].tail_part = ws.tail_part; p[1].tail_w = W->tail_h;
            GD_TRY(run_pair(p));
        } else {
            GD_TRY(resblock(0, W->up_rb[0][1], ws.p32b[0], ws.skip32[0], ws.p32a[0], nullptr, nullptr));
        }
    }
    // m_tail (ResUNet.py:39): conv(x + x1), times the per-stamp input scale
    if (chain) return launch_tail_gather(ws.tail_part, 1, g[0], tscale, zout, nb, t, W->tail_head_g, st, 1);
    if (fused) return launch_tail_gather(ws.tail_part, C[0] / 32, g[0], tscale, zout, nb, ws.tpad, W->tail_head_g, st);
    return launch_tail(ws.p32a[0], W->tail, C[0], g[0], tscale, zout, nb, st);
}

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
                GD_TRY(launch_g_xupdate(ws.spec, ws.HtH, ws.rho, nr, it, ws.z, ws.x, ws.u, ws.t, ws.tscale, nb, st));
                float* zdst = it == n - 1 ? out + o : ws.z;
                GD_TRY(resunet_chunk(W, ws, ws.t, ws.tscale, zdst, nb, st));
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

extern "C" int gd_fpfs(const float* img, const float* psf, int psf_batch, int batch, float sigma, float cnst, float* modes, float* ell,
                       void* stream) {
    if (batch < 0) GD_FAIL(GD_EBADSHAPE, "gd_fpfs: batch %d < 0", batch);
    if (batch && (!img || !ell)) GD_FAIL(GD_EBADSHAPE, "gd_fpfs: NULL img or ell for a batch of %d", batch);
    if (psf ? !(psf_batch == 1 || (psf_batch == batch && batch > 0)) : psf_batch != 0)
        GD_FAIL(GD_EBADSHAPE, "gd_fpfs: psf_batch %d with %s psf for a batch of %d (NULL psf <=> 0; otherwise 1 or the batch)", psf_batch,
                psf ? "a" : "a NULL", batch);
    if (!(sigma > 0.f && sigma <= 24.f)) GD_FAIL(GD_EBADSHAPE, "gd_fpfs: sigma must be in (0, 24] px, got %g", (double)sigma);
    if (!(isfinite(cnst) && cnst >= 0.f)) GD_FAIL(GD_EBADSHAPE, "gd_fpfs: const must be finite and >= 0, got %g", (double)cnst);
    if (batch == 0) return GD_OK;
    int dev;
    GD_CUDA_CHECK(cudaGetDevice(&dev));
    GD_TRY(init_once(dev));
    return launch_fpfs(img, psf, psf_batch, batch, sigma, cnst, modes, ell, (cudaStream_t)stream);
}

extern "C" int gd_metacal(const float* img, const float* psf, int psf_batch, int batch, float delta, float reconv_sigma,
                          float guess_sigma, float* images, float* shape, int32_t* info, void* stream) {
    if (batch < 0) GD_FAIL(GD_EBADSHAPE, "gd_metacal: batch %d < 0", batch);
    if (!shape || !info) GD_FAIL(GD_EBADSHAPE, "gd_metacal: NULL shape or info");
    if (batch && !img) GD_FAIL(GD_EBADSHAPE, "gd_metacal: NULL img for a batch of %d", batch);
    if (psf ? !(psf_batch == 1 || (psf_batch == batch && batch > 0)) : psf_batch != 0)
        GD_FAIL(GD_EBADSHAPE, "gd_metacal: psf_batch %d with %s psf for a batch of %d (NULL psf <=> 0; otherwise 1 or the batch)",
                psf_batch, psf ? "a" : "a NULL", batch);
    if (!(delta > 0.f && delta <= 0.1f)) GD_FAIL(GD_EBADSHAPE, "gd_metacal: delta must be in (0, 0.1], got %g", (double)delta);
    if (!(isfinite(reconv_sigma) && reconv_sigma > 0.f && reconv_sigma <= 24.f))
        GD_FAIL(GD_EBADSHAPE, "gd_metacal: reconv_sigma must be finite and in (0, 24] px, got %g", (double)reconv_sigma);
    if (!(isfinite(guess_sigma) && guess_sigma > 0.f && guess_sigma <= 24.f))
        GD_FAIL(GD_EBADSHAPE, "gd_metacal: guess_sigma must be finite and in (0, 24] px, got %g", (double)guess_sigma);
    if (batch == 0) return GD_OK;
    int dev;
    GD_CUDA_CHECK(cudaGetDevice(&dev));
    GD_TRY(init_once(dev));
    return launch_metacal(img, psf, psf_batch, batch, delta, reconv_sigma, guess_sigma, images, shape, info, (cudaStream_t)stream);
}

extern "C" int gd_metacal_fixnoise(const float* img, const float* psf, int psf_batch, int batch, float delta, float reconv_sigma,
                                   float guess_sigma, const float* noise, const float* noise_sigma, int sigma_batch, int64_t start,
                                   int64_t seed, float* images, float* shape, int32_t* info, void* stream) {
    if (batch < 0) GD_FAIL(GD_EBADSHAPE, "gd_metacal_fixnoise: batch %d < 0", batch);
    if (!shape || !info) GD_FAIL(GD_EBADSHAPE, "gd_metacal_fixnoise: NULL shape or info");
    if (batch && !img) GD_FAIL(GD_EBADSHAPE, "gd_metacal_fixnoise: NULL img for a batch of %d", batch);
    if (psf ? !(psf_batch == 1 || (psf_batch == batch && batch > 0)) : psf_batch != 0)
        GD_FAIL(GD_EBADSHAPE, "gd_metacal_fixnoise: psf_batch %d with %s psf for a batch of %d (NULL psf <=> 0; otherwise 1 or the batch)",
                psf_batch, psf ? "a" : "a NULL", batch);
    if (!(delta > 0.f && delta <= 0.1f)) GD_FAIL(GD_EBADSHAPE, "gd_metacal_fixnoise: delta must be in (0, 0.1], got %g", (double)delta);
    if (!(isfinite(reconv_sigma) && reconv_sigma > 0.f && reconv_sigma <= 24.f))
        GD_FAIL(GD_EBADSHAPE, "gd_metacal_fixnoise: reconv_sigma must be finite and in (0, 24] px, got %g", (double)reconv_sigma);
    if (!(isfinite(guess_sigma) && guess_sigma > 0.f && guess_sigma <= 24.f))
        GD_FAIL(GD_EBADSHAPE, "gd_metacal_fixnoise: guess_sigma must be finite and in (0, 24] px, got %g", (double)guess_sigma);
    if (!noise == !noise_sigma) GD_FAIL(GD_EBADSHAPE, "gd_metacal_fixnoise: exactly one of noise and noise_sigma must be given");
    if (noise_sigma ? !(sigma_batch == 1 || (sigma_batch == batch && batch > 0)) : sigma_batch != 0)
        GD_FAIL(GD_EBADSHAPE, "gd_metacal_fixnoise: sigma_batch %d with %s noise_sigma for a batch of %d (NULL <=> 0; otherwise 1 or the batch)",
                sigma_batch, noise_sigma ? "a" : "a NULL", batch);
    if (start < 0 || start > INT64_MAX - batch)
        GD_FAIL(GD_EBADSHAPE, "gd_metacal_fixnoise: stamp range [%lld, +%d) out of range", (long long)start, batch);
    if (batch == 0) return GD_OK;
    int dev;
    GD_CUDA_CHECK(cudaGetDevice(&dev));
    GD_TRY(init_once(dev));
    return launch_metacal_fixnoise(img, psf, psf_batch, batch, delta, reconv_sigma, guess_sigma, noise, noise_sigma, sigma_batch, start, seed,
                                   images, shape, info, (cudaStream_t)stream);
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
