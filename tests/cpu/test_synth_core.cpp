// Host harness of galaxy-deconv_b200/csrc/synth_core.cuh: runs the scalar math of k_synth on the CPU and writes raw fp32
// arrays that tests/test_synth_device.py compares with gdsynth.py.
//
//   test_synth_core DIR SEED SNR FWHM_ERR SHEAR_ERR       (SNR <= 0: 'mixed')
//     reads  DIR/triples.i64  [T][3] (idx, stream, seed)   ->  DIR/uniform.f32  [T]
//            DIR/index.i64    [M]    stamp indices         ->  DIR/gal_params.f32 [M][9], DIR/psf_params.f32 [M][13],
//                                                              DIR/galaxy.f32, psf.f32, model_psf.f32, gt.f32, obs.f32 [M][2304],
//                                                              DIR/alpha.f32 [M]
// The per-stamp pipeline mirrors k_synth stage by stage, sums in the same order, including the 96x96 transforms of
// fft_core.cuh and the shifted spectrum product, so the forward model is checked here without a GPU.
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <string>
#include <vector>
#include "synth_core.cuh"
using namespace gdsyn;

static std::vector<char> slurp(const std::string& path) {
    std::vector<char> b;
    FILE* f = fopen(path.c_str(), "rb");
    if (!f) { fprintf(stderr, "cannot open %s\n", path.c_str()); exit(2); }
    char buf[65536];
    size_t n;
    while ((n = fread(buf, 1, sizeof(buf), f)) > 0) b.insert(b.end(), buf, buf + n);
    fclose(f);
    return b;
}
static void dump(const std::string& path, const std::vector<float>& v) {
    FILE* f = fopen(path.c_str(), "wb");
    if (!f || fwrite(v.data(), sizeof(float), v.size(), f) != v.size()) { fprintf(stderr, "cannot write %s\n", path.c_str()); exit(2); }
    fclose(f);
}

constexpr int NPIX = STAMP * STAMP;
using F = gdfft::Real2D<96, 8, 12, 48>;
constexpr int SP = 50;

// Z (packed row pairs of a 48x48 image at the corner of the 96 grid) -> S (half spectrum)
static void fwd(std::vector<float2>& Z, std::vector<float2>& S, const std::vector<float2>& tw) {
    for (int w = 0; w < F::F1_ITEMS; ++w) F::F1(w, Z.data(), tw.data());
    for (int w = 0; w < F::F2_ITEMS; ++w) F::F2(w, Z.data());
    for (int w = 0; w < F::F3_ITEMS; ++w) F::F3(w, Z.data(), S.data(), SP);
    for (int w = 0; w < F::F4_ITEMS; ++w) F::F4(w, S.data(), SP, tw.data());
    for (int w = 0; w < F::F5_ITEMS; ++w) F::F5(w, S.data(), SP);
}
static void inv(std::vector<float2>& S, std::vector<float2>& Z, const std::vector<float2>& tw) {
    for (int w = 0; w < F::I1_ITEMS; ++w) F::I1(w, S.data(), SP, tw.data());
    for (int w = 0; w < F::I2_ITEMS; ++w) F::I2(w, S.data(), SP);
    for (int w = 0; w < F::I3_ITEMS; ++w) F::I3(w, S.data(), SP, Z.data());
    for (int w = 0; w < F::I4_ITEMS; ++w) F::I4(w, Z.data(), tw.data());
    for (int w = 0; w < F::I5_ITEMS; ++w) F::I5(w, Z.data());
}
static float& zpix(std::vector<float2>& Z, int r, int c) { return (r & 1) ? Z[(r >> 1) * 96 + c].y : Z[(r >> 1) * 96 + c].x; }

// the summation order of k_synth: 256 threads each add pixels t, t+256, ... in turn, then block_sum (fft_block.cuh): an xor
// butterfly inside each warp and the 8 warp sums added in order.  (A plain running sum over 2304 pixels would be ~100x less
// accurate than either torch's or the kernel's.)
static float block_order_sum(const float* x) {
    constexpr int T = 256;
    float v[T];
    for (int t = 0; t < T; ++t) {
        v[t] = 0.f;
        for (int i = t; i < NPIX; i += T) v[t] += x[i];
    }
    for (int o = 16; o > 0; o >>= 1) {
        float n[T];
        for (int t = 0; t < T; ++t) n[t] = v[t] + v[t ^ o];
        for (int t = 0; t < T; ++t) v[t] = n[t];
    }
    float r = v[0];
    for (int w = 1; w < T / 32; ++w) r += v[32 * w];
    return r;
}

static std::vector<float> render_psf(const PsfParams& pp) {
    std::vector<float> v(NPIX);
    for (int i = 0; i < NPIX; ++i) v[i] = render_pixel([&](float dx, float dy) { return moffat_value(pp, dx, dy); }, i / STAMP, i % STAMP);
    const float s = block_order_sum(v.data());
    for (auto& x : v) x = fdiv(x, s);
    return v;
}

int main(int argc, char** argv) {
    if (argc != 6) { fprintf(stderr, "usage: %s DIR SEED SNR FWHM_ERR SHEAR_ERR\n", argv[0]); return 2; }
    const std::string dir = argv[1];
    const uint64_t seed = (uint64_t)strtoll(argv[2], nullptr, 10);
    const float snr_fixed = strtof(argv[3], nullptr), fwhm_err = strtof(argv[4], nullptr), shear_err = strtof(argv[5], nullptr);

    std::vector<char> tb = slurp(dir + "/triples.i64");
    const int64_t* tr = reinterpret_cast<const int64_t*>(tb.data());
    const size_t T = tb.size() / (3 * sizeof(int64_t));
    std::vector<float> uni(T);
    for (size_t t = 0; t < T; ++t) uni[t] = hashed_uniform((uint64_t)tr[3 * t], (int)tr[3 * t + 1], (uint64_t)tr[3 * t + 2]);
    dump(dir + "/uniform.f32", uni);

    std::vector<char> ib = slurp(dir + "/index.i64");
    const int64_t* ix = reinterpret_cast<const int64_t*>(ib.data());
    const size_t M = ib.size() / sizeof(int64_t);
    std::vector<float> gpar, ppar, gal, psf, model, gt, obs, alpha;
    std::vector<float2> tw(96), Z(24 * 96), SG(96 * SP), SPc(96 * SP);
    for (int m = 0; m < 96; ++m) tw[m] = make_float2((float)cos(2 * M_PI * m / 96), (float)-sin(2 * M_PI * m / 96));
    for (size_t s = 0; s < M; ++s) {
        const uint64_t idx = (uint64_t)ix[s];
        const GalaxyParams gp = galaxy_params(idx, seed);
        const PsfParams pt = psf_params(idx, seed, false, 0.f, 0.f), pm = psf_params(idx, seed, true, fwhm_err, shear_err);
        const float snr = snr_fixed > 0.f ? snr_fixed : snr_mixed(idx, seed);
        for (float v : {gp.n, gp.re, gp.e, gp.th, gp.x0, gp.y0, (float)gp.is_gauss, gp.q, gp.bn}) gpar.push_back(v);
        for (float v : {pt.beta, pt.fwhm, pt.e0, pt.th0, pt.e, pt.th, pt.a, pm.fwhm, pm.sg, pm.sg2, pm.e, pm.th, snr}) ppar.push_back(v);
        // galaxy, flux scale
        std::vector<float> g(NPIX), g2(NPIX);
        for (int i = 0; i < NPIX; ++i) {
            g[i] = fmaxf(render_pixel([&](float dx, float dy) { return sersic_value(gp, dx, dy); }, i / STAMP, i % STAMP), 0.f);
            g2[i] = fmul(g[i], g[i]);
        }
        gal.insert(gal.end(), g.begin(), g.end());
        const float scale = fdiv(fmul(snr, SIGMA), sqrtf(block_order_sum(g2.data())));
        for (auto& v : g) v = fmul(v, scale);
        gt.insert(gt.end(), g.begin(), g.end());
        const std::vector<float> p = render_psf(pt), pmod = render_psf(pm);
        psf.insert(psf.end(), p.begin(), p.end());
        model.insert(model.end(), pmod.begin(), pmod.end());
        // forward model + noise
        for (auto& v : Z) v = make_float2(NAN, NAN);
        for (int i = 0; i < NPIX; ++i) zpix(Z, i / STAMP, i % STAMP) = g[i];
        fwd(Z, SG, tw);
        for (auto& v : Z) v = make_float2(NAN, NAN);
        for (int i = 0; i < NPIX; ++i) zpix(Z, i / STAMP, i % STAMP) = p[i];
        fwd(Z, SPc, tw);
        for (int q = 0; q < F::NH * 96; ++q) conv_shift_product<F>(q, SG.data(), SPc.data(), SP);
        inv(SG, Z, tw);
        const size_t o0 = obs.size();
        for (int i = 0; i < NPIX; ++i) obs.push_back(obs_pixel(zpix(Z, i / STAMP, i % STAMP), idx, i, seed));
        alpha.push_back(fdiv(block_order_sum(obs.data() + o0), (float)NPIX));
    }
    dump(dir + "/gal_params.f32", gpar);
    dump(dir + "/psf_params.f32", ppar);
    dump(dir + "/galaxy.f32", gal);
    dump(dir + "/psf.f32", psf);
    dump(dir + "/model_psf.f32", model);
    dump(dir + "/gt.f32", gt);
    dump(dir + "/obs.f32", obs);
    dump(dir + "/alpha.f32", alpha);
    printf("%zu uniforms, %zu stamps OK\n", T, M);
    return 0;
}
