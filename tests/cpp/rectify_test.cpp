// acm::stereo_rectify through include/acm.hpp (host only, runs without a GPU): R1 = R2 R, R2 t on the x axis, and a
// translation of zero raised as an error.  argv[1..12]: R (row-major) then t; prints R1, R2, baseline and vertical.
#include <cmath>
#include <cstdio>
#include <cstdlib>

#include "acm.hpp"

int main(int argc, char** argv) {
    if (argc != 13) { std::fprintf(stderr, "usage: rectify_test r00 .. r22 tx ty tz\n"); return 2; }
    std::array<double, 9> R;
    std::array<double, 3> t;
    for (int i = 0; i < 9; ++i) R[i] = std::strtod(argv[1 + i], nullptr);
    for (int i = 0; i < 3; ++i) t[i] = std::strtod(argv[10 + i], nullptr);
    const acm::StereoRectification s = acm::stereo_rectify(R, t);
    double dev = 0.0;
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j) {
            double r2r = 0.0;
            for (int k = 0; k < 3; ++k) r2r += s.R2[3 * i + k] * R[3 * k + j];
            dev = std::fmax(dev, std::fabs(r2r - s.R1[3 * i + j]));
        }
    if (dev > 1e-13) { std::fprintf(stderr, "R1 != R2 R: %g\n", dev); return 1; }
    try {
        acm::stereo_rectify(R, {0.0, 0.0, 0.0});
        std::fprintf(stderr, "t = 0 accepted\n");
        return 1;
    } catch (const acm::CameraModelError& e) {
        if (std::string(e.what()).find("translation is zero") == std::string::npos) { std::fprintf(stderr, "message: %s\n", e.what()); return 1; }
    }
    for (double v : s.R1) std::printf("%.17g ", v);
    for (double v : s.R2) std::printf("%.17g ", v);
    std::printf("%.17g %d\nRECTIFY_TEST_OK\n", s.baseline, s.vertical ? 1 : 0);
    return 0;
}
