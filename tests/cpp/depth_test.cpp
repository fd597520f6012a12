// acm::render_depth / acm::depth_to_points through include/acm.hpp on the Kannala-Brandt sample camera.  argv[1]: binary
// input = R (9 doubles, row-major), t (3), n (1 double), xyz (3n); argv[2]: binary output = range (W*H floats), index (W*H
// uint32), back-projected points of that range image (3*W*H doubles), status (W*H bytes).  Needs a GPU; prints
// "DEPTH_TEST_OK".
#include <array>
#include <cstdio>
#include <limits>
#include <vector>

#include "acm.hpp"

using namespace acm;

int main(int argc, char** argv) {
    if (argc != 3) { std::fprintf(stderr, "usage: depth_test in.bin out.bin\n"); return 2; }
    std::FILE* f = std::fopen(argv[1], "rb");
    if (!f) return 2;
    std::array<double, 9> R;
    std::array<double, 3> t;
    double nd = 0.0;
    if (std::fread(R.data(), sizeof(double), 9, f) != 9 || std::fread(t.data(), sizeof(double), 3, f) != 3 || std::fread(&nd, sizeof(double), 1, f) != 1)
        return 2;
    const size_t n = (size_t)nd;
    std::vector<double> xyz(3 * n);
    if (std::fread(xyz.data(), sizeof(double), 3 * n, f) != 3 * n) return 2;
    std::fclose(f);

    Context ctx(0);
    KannalaBrandtModel kb = KannalaBrandtModel::create({190.97847715128717, 190.9733070521226, 254.93170605935475, 256.8974428996504,
                                                        0.0034823894022493434, 0.0007150348452162257, -0.0020532361418706202,
                                                        0.00020293673591811182});
    kb.resolution = {512, 512};
    kb.bind(ctx);
    const DepthImage img = render_depth(kb, R, t, xyz.data(), n);
    const DepthPoints back = depth_to_points(kb, R, t, img.range.data());
    try {
        render_depth(kb, R, {std::numeric_limits<double>::infinity(), 0.0, 0.0}, xyz.data(), n);
        std::fprintf(stderr, "non-finite t accepted\n");
        return 1;
    } catch (const CameraModelError& e) {
        if (std::string(e.what()).find("non-finite") == std::string::npos) { std::fprintf(stderr, "message: %s\n", e.what()); return 1; }
    }
    std::FILE* o = std::fopen(argv[2], "wb");
    if (!o) return 2;
    std::fwrite(img.range.data(), sizeof(float), img.range.size(), o);
    std::fwrite(img.index.data(), sizeof(uint32_t), img.index.size(), o);
    std::fwrite(back.points.data(), sizeof(double), back.points.size(), o);
    std::fwrite(back.status.data(), 1, back.status.size(), o);
    std::fclose(o);
    std::printf("DEPTH_TEST_OK\n");
    return 0;
}
