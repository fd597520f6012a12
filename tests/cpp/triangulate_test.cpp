// acm::triangulate through include/acm.hpp: the Kannala-Brandt sample camera (first) and the Double Sphere sample camera
// (second).  argv[1]: binary input = R (9 doubles, row-major), t (3), n (1 double), uv1 (2n), uv2 (2n); argv[2]: binary output =
// points (3n), errors (2n), status (n bytes).  Needs a GPU; prints "TRIANGULATE_TEST_OK".
#include <array>
#include <cstdio>
#include <vector>

#include "acm.hpp"

using namespace acm;

int main(int argc, char** argv) {
    if (argc != 3) { std::fprintf(stderr, "usage: triangulate_test in.bin out.bin\n"); return 2; }
    std::FILE* f = std::fopen(argv[1], "rb");
    if (!f) return 2;
    std::array<double, 9> R;
    std::array<double, 3> t;
    double nd = 0.0;
    if (std::fread(R.data(), sizeof(double), 9, f) != 9 || std::fread(t.data(), sizeof(double), 3, f) != 3 || std::fread(&nd, sizeof(double), 1, f) != 1)
        return 2;
    const size_t n = (size_t)nd;
    std::vector<double> uv1(2 * n), uv2(2 * n);
    if (std::fread(uv1.data(), sizeof(double), 2 * n, f) != 2 * n || std::fread(uv2.data(), sizeof(double), 2 * n, f) != 2 * n) return 2;
    std::fclose(f);

    Context ctx(0);
    KannalaBrandtModel kb = KannalaBrandtModel::create({190.97847715128717, 190.9733070521226, 254.93170605935475, 256.8974428996504,
                                                        0.0034823894022493434, 0.0007150348452162257, -0.0020532361418706202,
                                                        0.00020293673591811182});
    kb.resolution = {512, 512};
    DoubleSphereModel ds = DoubleSphereModel::create({348.112754378549, 347.1109973814674, 365.8121721753254, 249.3555778487899,
                                                      0.5657413673629862, -0.24425190195168348});
    ds.resolution = {752, 480};
    kb.bind(ctx);
    ds.bind(ctx);
    const Triangulation tri = triangulate(kb, ds, R, t, uv1.data(), uv2.data(), n);
    try {
        triangulate(kb, ds, R, {0.0, 0.0, 0.0}, uv1.data(), uv2.data(), n);
        std::fprintf(stderr, "t = 0 accepted\n");
        return 1;
    } catch (const CameraModelError& e) {
        if (std::string(e.what()).find("translation is zero") == std::string::npos) { std::fprintf(stderr, "message: %s\n", e.what()); return 1; }
    }
    std::FILE* o = std::fopen(argv[2], "wb");
    if (!o) return 2;
    std::fwrite(tri.points.data(), sizeof(double), 3 * n, o);
    std::fwrite(tri.errors.data(), sizeof(double), 2 * n, o);
    std::fwrite(tri.status.data(), 1, n, o);
    std::fclose(o);
    std::printf("TRIANGULATE_TEST_OK\n");
    return 0;
}
