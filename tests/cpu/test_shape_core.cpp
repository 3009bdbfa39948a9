// Host harness of galaxy-deconv_b200/csrc/shape_core.cuh: runs the adaptive-moments iteration of k_adaptive_moments on the CPU.
//
//   test_shape_core DIR GUESS_SIGMA
//     reads  DIR/stamps.f32 [N][48*48]  ->  DIR/shape.f32 [N][8] (flux, x0, y0, Mxx, Mxy, Myy, e1, e2), DIR/info.i32 [N][2] (status, passes)
//
// The pixels are visited serially, but their contributions are summed in the kernel's order: lane l of a warp adds pixels
// l + 32k for k = 0..71 in turn, then an xor butterfly combines the 32 lane sums.
#include <cstdio>
#include <cstdlib>
#include <string>
#include <vector>
#include "shape_core.cuh"
using namespace gdshape;

constexpr int NPIX = STAMP * STAMP;

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
template <class T> static void dump(const std::string& path, const std::vector<T>& v) {
    FILE* f = fopen(path.c_str(), "wb");
    if (!f || fwrite(v.data(), sizeof(T), v.size(), f) != v.size()) { fprintf(stderr, "cannot write %s\n", path.c_str()); exit(2); }
    fclose(f);
}

static Sums warp_order_sums(const float* img, const Weight& w, const Quad& q) {
    Sums lane[32];
    for (int l = 0; l < 32; ++l) {
        lane[l] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
        for (int p = l; p < NPIX; p += 32) add_pixel(lane[l], q, (float)(p % STAMP) - w.x0, (float)(p / STAMP) - w.y0, img[p]);
    }
    for (int o = 16; o > 0; o >>= 1) {
        Sums nx[32];
        for (int l = 0; l < 32; ++l) {
            const Sums &a = lane[l], &b = lane[l ^ o];
            nx[l] = {a.a + b.a, a.bx + b.bx, a.by + b.by, a.cxx + b.cxx, a.cxy + b.cxy, a.cyy + b.cyy};
        }
        for (int l = 0; l < 32; ++l) lane[l] = nx[l];
    }
    return lane[0];
}

int main(int argc, char** argv) {
    if (argc != 3) { fprintf(stderr, "usage: %s DIR GUESS_SIGMA\n", argv[0]); return 2; }
    const std::string dir = argv[1];
    const float guess_sigma = strtof(argv[2], nullptr);
    std::vector<char> sb = slurp(dir + "/stamps.f32");
    const float* stamps = reinterpret_cast<const float*>(sb.data());
    const size_t N = sb.size() / (NPIX * sizeof(float));
    std::vector<float> shape(N * 8);
    std::vector<int> info(N * 2);
    for (size_t s = 0; s < N; ++s) {
        const float* img = stamps + s * NPIX;
        int passes = 0;
        info[2 * s] = measure(guess_sigma, [&](const Weight& w, const Quad& q) { return warp_order_sums(img, w, q); }, &shape[8 * s], &passes);
        info[2 * s + 1] = passes;
    }
    dump(dir + "/shape.f32", shape);
    dump(dir + "/info.i32", info);
    printf("%zu stamps OK\n", N);
    return 0;
}
