// Host harness of galaxy-deconv_b200/csrc/fpfs_core.cuh with the Fft48 transform of fft_core.cuh: runs the FPFS estimator of
// k_fpfs on the CPU.
//
//   test_fpfs_core DIR SIGMA CONST
//     reads  DIR/stamps.f32 [N][48*48] and, if present, DIR/psf.f32 [1 or N][48*48]
//     writes DIR/modes.f32 [N][6] (M00, M22c, M22s, M40, M42c, M42s) and DIR/ell.f32 [N][3] (e1, e2, R)
//
// Every step is the kernel's: the column pass packs columns c and c + 24 into one complex column and splits the transform by
// Hermitian symmetry into rows 0..24, the row pass transforms each row, and gdfpfs::row_sums / gdfpfs::finish add the cells
// and the rows in the kernel's order.
#include <cstdio>
#include <cstdlib>
#include <string>
#include <vector>
#include "fft_core.cuh"
#include "fpfs_core.cuh"
using namespace gdfpfs;
using gdfft::Fft48;

constexpr int NPIX = STAMP * STAMP;

static bool slurp(const std::string& path, std::vector<float>& out) {
    FILE* f = fopen(path.c_str(), "rb");
    if (!f) return false;
    float buf[16384];
    size_t n;
    while ((n = fread(buf, sizeof(float), 16384, f)) > 0) out.insert(out.end(), buf, buf + n);
    fclose(f);
    return true;
}
static void dump(const std::string& path, const std::vector<float>& v) {
    FILE* f = fopen(path.c_str(), "wb");
    if (!f || fwrite(v.data(), sizeof(float), v.size(), f) != v.size()) { fprintf(stderr, "cannot write %s\n", path.c_str()); exit(2); }
    fclose(f);
}

// the half spectrum [25][48] of one image: column pass then row pass, as k_fpfs passes P0 and P1/P2
static void half_spectrum(const float* x, float2 (*S)[STAMP]) {
    float2 plane[ROWS][STAMP];
    for (int c = 0; c < 24; ++c) {
        float2 v[48];
        for (int n = 0; n < 48; ++n) v[n] = make_float2(x[n * 48 + c], x[n * 48 + c + 24]);
        Fft48::run(v);
        for (int k = 0; k < ROWS; ++k) {
            const float2 p = v[Fft48::reg(k)], q = v[Fft48::reg((48 - k) % 48)];
            plane[k][c] = make_float2(0.5f * (p.x + q.x), 0.5f * (p.y - q.y));
            plane[k][c + 24] = make_float2(0.5f * (p.y + q.y), 0.5f * (q.x - p.x));
        }
    }
    for (int k = 0; k < ROWS; ++k) {
        float2 v[48];
        for (int c = 0; c < 48; ++c) v[c] = plane[k][c];
        Fft48::run(v);
        for (int u = 0; u < 48; ++u) S[k][u] = v[Fft48::reg(u)];
    }
}

int main(int argc, char** argv) {
    if (argc != 4) { fprintf(stderr, "usage: %s DIR SIGMA CONST\n", argv[0]); return 2; }
    const std::string dir = argv[1];
    const float sigma = strtof(argv[2], nullptr), cnst = strtof(argv[3], nullptr);
    std::vector<float> stamps, psf;
    if (!slurp(dir + "/stamps.f32", stamps)) { fprintf(stderr, "cannot open stamps\n"); return 2; }
    const bool has_psf = slurp(dir + "/psf.f32", psf);
    const size_t N = stamps.size() / NPIX, P = psf.size() / NPIX;
    Axis xs[STAMP];
    for (int u = 0; u < STAMP; ++u) xs[u] = axis(u, sigma);
    std::vector<float> modes(N * NMODES), ell(N * NELL);
    static float2 S[ROWS][STAMP], H[ROWS][STAMP];
    for (size_t s = 0; s < N; ++s) {
        half_spectrum(&stamps[s * NPIX], S);
        float hh[ROWS][STAMP], h0 = 1.f, p0 = 1.f;
        if (has_psf) {
            half_spectrum(&psf[(P == 1 ? 0 : s) * NPIX], H);
            for (int k = 0; k < ROWS; ++k)
                for (int u = 0; u < STAMP; ++u) hh[k][u] = H[k][u].x * H[k][u].x + H[k][u].y * H[k][u].y;
            p0 = H[0][0].x;
            h0 = H[0][0].x * H[0][0].x + H[0][0].y * H[0][0].y;
        }
        Sums rows[ROWS];
        for (int k = 0; k < ROWS; ++k) {
            const float2* y = S[k];
            const float* h = hh[k];
            rows[k] = row_sums(k, axis(k, sigma), xs, [&](int u) {
                const float pw = y[u].x * y[u].x + y[u].y * y[u].y;
                return has_psf ? pw * psf_factor(h[u], h0) : pw;
            });
        }
        finish(rows, sigma, cnst, !has_psf || p0 > 0.0f, &modes[s * NMODES], &ell[s * NELL]);
    }
    dump(dir + "/modes.f32", modes);
    dump(dir + "/ell.f32", ell);
    printf("%zu stamps OK\n", N);
    return 0;
}
