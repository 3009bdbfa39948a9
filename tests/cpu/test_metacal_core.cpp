// Host harness of galaxy-deconv_b200/csrc/metacal_core.cuh: makes the five metacalibration images of k_metacal on the CPU.
//
//   test_metacal_core DIR DELTA RECONV_SIGMA
//     reads  DIR/stamps.f32 [N][48*48] and, if present, DIR/psf.f32 [1 or N][48*48]
//     writes DIR/images.f32 [N][5][48*48] (noshear, 1p, 1m, 2p, 2m)
//
// Every step is the kernel's, in the kernel's order: the forward column and row passes into planes 0 (stamp) and 1 (PSF), the
// PSF factors G~ / P of every (shear, target), the sheared spectra (the DTFT) and the noshear one (the grid spectrum) times
// their factors, then the inverse row and column passes of the five planes.
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

// the factor table of one PSF (ppix) whose grid spectrum is in pplane
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
    if (argc != 4) { fprintf(stderr, "usage: %s DIR DELTA RECONV_SIGMA\n", argv[0]); return 2; }
    const std::string dir = argv[1];
    const float delta = strtof(argv[2], nullptr), sigma = strtof(argv[3], nullptr);
    std::vector<float> stamps, psf;
    if (!slurp(dir + "/stamps.f32", stamps)) { fprintf(stderr, "cannot open stamps\n"); return 2; }
    const bool has_psf = slurp(dir + "/psf.f32", psf);
    const size_t N = stamps.size() / NPIX, P = psf.size() / NPIX;
    std::vector<float> out(N * NIMG * NPIX);
    alignas(16) static float2 planes[NIMG * PLANE];
    alignas(16) static float s_img[NPIX], s_psf[NPIX];
    static float2 factor[NIMG * NTARGET];
    for (size_t s = 0; s < N; ++s) {
        for (int i = 0; i < NPIX; ++i) s_img[i] = stamps[s * NPIX + i];
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
        for (int j = 0; j < NIMG; ++j) {
            float2* plane = planes + j * PLANE;
            for (int v = 0; v < HALF; ++v) inv_row(plane, v);
            static float2 x[HALF][STAMP];
            for (int c = 0; c < HALF; ++c) inv_col(plane, c, x[c]);
            for (int c = 0; c < HALF; ++c) inv_col_store(x[c], c, &out[(s * NIMG + j) * NPIX]);
        }
    }
    FILE* f = fopen((dir + "/images.f32").c_str(), "wb");
    if (!f || fwrite(out.data(), sizeof(float), out.size(), f) != out.size()) { fprintf(stderr, "cannot write images\n"); return 2; }
    fclose(f);
    printf("%zu stamps OK\n", N);
    return 0;
}
