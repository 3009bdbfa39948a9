// Host harness of the fix-noise path of galaxy-deconv_b200/csrc/metacal_core.cuh: makes the five fix-noise images of
// k_metacal_fixnoise on the CPU.
//
//   test_metacal_fixnoise_core DIR DELTA RECONV_SIGMA START SEED
//     reads  DIR/stamps.f32 [N][48*48], if present DIR/psf.f32 [1 or N][48*48], and either DIR/noise.f32 [N][48*48] (the caller's
//            field) or DIR/sigma.f32 [1 or N] (the field generated for stamps START .. START + N - 1 under SEED)
//     writes DIR/images.f32 [N][5][48*48] (noshear, 1p, 1m, 2p, 2m), DIR/field.f32 [N][48*48] (the field used) and
//            DIR/uniform.f32 [N][2][64] (the stream-60 and stream-61 uniforms of pixels 0..63 of each generated field)
//
// Every step is the kernel's, in the kernel's order: the stamp's planes as tests/cpu/test_metacal_core.cpp makes them, then one
// item per (shear, target) adding the noise term to its cell.
#include <cstdio>
#include <cstdlib>
#include <string>
#include <vector>
#include "metacal_core.cuh"
using namespace gdmetacal;

static bool slurp(const std::string& path, std::vector<float>& out) {
    FILE* f = fopen(path.c_str(), "rb");
    if (!f) return false;
    float buf[16384];
    size_t n;
    while ((n = fread(buf, sizeof(float), 16384, f)) > 0) out.insert(out.end(), buf, buf + n);
    fclose(f);
    return true;
}

static bool dump(const std::string& path, const std::vector<float>& v) {
    FILE* f = fopen(path.c_str(), "wb");
    const bool ok = f && fwrite(v.data(), sizeof(float), v.size(), f) == v.size();
    if (f) fclose(f);
    return ok;
}

static void psf_factors(const float* ppix, const float2* pplane, float2* factor, float delta, float sigma) {
    const float p0 = pplane[0].x;
    for (int j = 0; j < NIMG; ++j)
        for (int t = 0; t < NTARGET; ++t) {
            const Cell k = target(t);
            const float sgn = centre_sign(k.v, k.i);
            float2 pt;
            if (j) {
                const float2 f = sheared_freq(j, delta, fftfreq(k.i), k.v);
                pt = dtft(ppix, f.x, f.y);
            } else {
                const float2 g = pplane[k.v * PROW + k.i];
                pt = make_float2(sgn * g.x, sgn * g.y);
            }
            factor[j * NTARGET + t] = psf_factor(pt, p0, reconv(k.v, k.i, sigma));
        }
}

static void forward(const float* img, float2* plane) {
    for (int c = 0; c < HALF; ++c) fwd_col(img, c, plane);
    for (int v = 0; v < HALF; ++v) fwd_row(plane, v);
}

int main(int argc, char** argv) {
    if (argc != 6) { fprintf(stderr, "usage: %s DIR DELTA RECONV_SIGMA START SEED\n", argv[0]); return 2; }
    const std::string dir = argv[1];
    const float delta = strtof(argv[2], nullptr), sigma = strtof(argv[3], nullptr);
    const uint64_t start = (uint64_t)strtoll(argv[4], nullptr, 10), seed = (uint64_t)strtoll(argv[5], nullptr, 10);
    std::vector<float> stamps, psf, noise, sig;
    if (!slurp(dir + "/stamps.f32", stamps)) { fprintf(stderr, "cannot open stamps\n"); return 2; }
    const bool has_psf = slurp(dir + "/psf.f32", psf);
    const bool caller = slurp(dir + "/noise.f32", noise);
    if (!caller && !slurp(dir + "/sigma.f32", sig)) { fprintf(stderr, "neither noise nor sigma\n"); return 2; }
    const size_t N = stamps.size() / NPIX, P = psf.size() / NPIX;
    std::vector<float> out(N * NIMG * NPIX), field(N * NPIX), uni;
    alignas(16) static float2 planes[NIMG * PLANE];
    alignas(16) static float s_img[NPIX], s_psf[NPIX], s_noise[NPIX];
    static float2 factor[NIMG * NTARGET];
    for (size_t s = 0; s < N; ++s) {
        for (int i = 0; i < NPIX; ++i) s_img[i] = stamps[s * NPIX + i];
        if (caller) {
            for (int i = 0; i < NPIX; ++i) s_noise[i] = noise[s * NPIX + i];
        } else {
            const uint64_t idx = start + s;
            const float sg = sig[sig.size() == 1 ? 0 : s];
            for (int i = 0; i < NPIX; ++i) s_noise[i] = fixnoise_pixel(idx, i, seed, sg);
            for (int st = 0; st < 2; ++st)
                for (int i = 0; i < 64; ++i) uni.push_back(gdsyn::hashed_uniform(idx * 4099ull + (uint64_t)i, FIXNOISE_STREAM + st, seed));
        }
        for (int i = 0; i < NPIX; ++i) field[s * NPIX + i] = s_noise[i];
        if (has_psf && (P > 1 || s == 0)) {
            for (int i = 0; i < NPIX; ++i) s_psf[i] = psf[(P == 1 ? 0 : s) * NPIX + i];
            forward(s_psf, planes + PLANE);
            psf_factors(s_psf, planes + PLANE, factor, delta, sigma);
        }
        forward(s_img, planes);
        for (int j = 1; j <= NIMG; ++j) {            // the kernel's item order: shears 1..4, then noshear
            const int jj = j % NIMG;
            for (int t = 0; t < NTARGET; ++t) {
                const Cell k = target(t);
                const float sgn = centre_sign(k.v, k.i);
                float2 spec;
                if (jj) {
                    const float2 f = sheared_freq(jj, delta, fftfreq(k.i), k.v);
                    spec = dtft(s_img, f.x, f.y);
                } else {
                    const float2 g = planes[k.v * PROW + k.i];
                    spec = make_float2(sgn * g.x, sgn * g.y);
                }
                planes[jj * PLANE + k.v * PROW + k.i] =
                    has_psf ? cell_value(spec, factor[jj * NTARGET + t], sgn) : cell_value(spec, reconv(k.v, k.i, sigma), sgn);
            }
        }
        for (int jj = 0; jj < NIMG; ++jj)            // the noise terms: each cell is written by one item, in any order
            for (int t = 0; t < NTARGET; ++t) {
                const Cell k = target(t);
                const float2 f = sheared_freq(opposite(jj), delta, fftfreq(k.i), k.v);
                const float2 term = fixnoise_value(jj, t, delta, sigma, dtft(s_noise, f.x, f.y), has_psf ? factor : nullptr);
                float2& cell = planes[jj * PLANE + k.v * PROW + k.i];
                cell = make_float2(cell.x + term.x, cell.y + term.y);
            }
        for (int j = 0; j < NIMG; ++j) {
            float2* plane = planes + j * PLANE;
            for (int v = 0; v < HALF; ++v) inv_row(plane, v);
            static float2 x[HALF][STAMP];
            for (int c = 0; c < HALF; ++c) inv_col(plane, c, x[c]);
            for (int c = 0; c < HALF; ++c) inv_col_store(x[c], c, &out[(s * NIMG + j) * NPIX]);
        }
    }
    if (!dump(dir + "/images.f32", out) || !dump(dir + "/field.f32", field) || !dump(dir + "/uniform.f32", uni)) {
        fprintf(stderr, "cannot write outputs\n");
        return 2;
    }
    printf("%zu stamps OK\n", N);
    return 0;
}
