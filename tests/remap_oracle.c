/*
 * remap_oracle.c -- CPU oracle of the camera-to-camera remap (test infrastructure only).
 *
 * The reference has no such function: the remap is a composition of its own functions, and this
 * file composes the oracle's restatements of them (oracle/acm_oracle.h) in the same way.  Output
 * pixel (u, v) of the output camera's grid (integer coordinates as f64, undistort.rs:35-37):
 *   ray = out.unproject((u, v))   -- with its pixel-bounds test
 *   src = in.project(ray)         -- if that is Ok
 *   interpolate_pixel(in_frame, src, interp) (undistort.rs:51-105)   -- if that is Ok; black otherwise.
 * Built with the oracle's flags (-O2 -ffp-contract=off -fno-fast-math) together with its sources.
 */
#include <math.h>
#include <stdlib.h>
#include <string.h>

#include "acm_oracle.h"

void orc_remap_map(const orc_model* in, const orc_model* out, double* src_xy) {
    for (uint32_t v = 0; v < out->height; ++v)
        for (uint32_t u = 0; u < out->width; ++u) {
            const double uv[2] = {(double)u, (double)v};
            double ray[3], p[2] = {NAN, NAN};
            if (orc_unproject(out, uv, ray) != ORC_OK || orc_project(in, ray, p) != ORC_OK) p[0] = p[1] = NAN;
            src_xy[2 * ((size_t)v * out->width + u)] = p[0];
            src_xy[2 * ((size_t)v * out->width + u) + 1] = p[1];
        }
}

/* undistort.rs:51-105, as oracle/acm_oracle_util.c states it (that copy is file-local there).  Pinned by
 * tests/test_oracle_remap.py: orc_remap_apply_map(orc_undistort_map(...)) == orc_undistort_rgb8 byte for byte. */
static int interpolate_pixel(const uint8_t* img, unsigned W, unsigned H, double x, double y, int interp, uint8_t rgb[3]) {
    if (interp == 0) {
        /* x.round() as i32: saturating cast, NaN -> 0 */
        double rx = round(x), ry = round(y);
        int u = isnan(rx) ? 0 : (rx >= 2147483647.0 ? 2147483647 : (rx <= -2147483648.0 ? (-2147483647 - 1) : (int)rx));
        int v = isnan(ry) ? 0 : (ry >= 2147483647.0 ? 2147483647 : (ry <= -2147483648.0 ? (-2147483647 - 1) : (int)ry));
        if (u >= 0 && u < (int)W && v >= 0 && v < (int)H) {
            const uint8_t* p = img + 3 * ((size_t)v * W + (size_t)u);
            rgb[0] = p[0]; rgb[1] = p[1]; rgb[2] = p[2];
            return 1;
        }
        return 0;
    }
    double x0 = floor(x), y0 = floor(y);
    double x1 = x0 + 1.0, y1 = y0 + 1.0;
    if (x0 < 0.0 || x1 >= (double)W || y0 < 0.0 || y1 >= (double)H) return 0;
    if (isnan(x0) || isnan(y0)) return 0;
    unsigned x0u = (unsigned)x0, y0u = (unsigned)y0, x1u = (unsigned)x1, y1u = (unsigned)y1;
    const uint8_t* p00 = img + 3 * ((size_t)y0u * W + x0u);
    const uint8_t* p10 = img + 3 * ((size_t)y0u * W + x1u);
    const uint8_t* p01 = img + 3 * ((size_t)y1u * W + x0u);
    const uint8_t* p11 = img + 3 * ((size_t)y1u * W + x1u);
    double wx = x - x0, wy = y - y0, wx_inv = 1.0 - wx, wy_inv = 1.0 - wy;
    for (int c = 0; c < 3; ++c) {
        double val = (double)p00[c] * wx_inv * wy_inv + (double)p10[c] * wx * wy_inv + (double)p01[c] * wx_inv * wy + (double)p11[c] * wx * wy;
        double r = round(val);
        r = r < 0.0 ? 0.0 : (r > 255.0 ? 255.0 : r);
        rgb[c] = (uint8_t)r;
    }
    return 1;
}

/* interpolate_pixel driven by a given map (Wo x Ho entries of (x, y), NaN = no sample) on a Wi x Hi input */
void orc_remap_apply_map(const double* src_xy, uint32_t Wo, uint32_t Ho, const uint8_t* img_in, uint32_t Wi, uint32_t Hi, int interp,
                         uint8_t* img_out) {
    memset(img_out, 0, (size_t)3 * Wo * Ho); /* RgbImage::new => black */
    for (size_t i = 0; i < (size_t)Wo * Ho; ++i) {
        const double x = src_xy[2 * i], y = src_xy[2 * i + 1];
        if (isnan(x) || isnan(y)) continue;
        interpolate_pixel(img_in, Wi, Hi, x, y, interp, img_out + 3 * i);
    }
}

void orc_remap_rgb8(const orc_model* in, const orc_model* out, const uint8_t* img_in, uint8_t* img_out, int interp) {
    double* map = (double*)malloc(sizeof(double) * 2 * (size_t)out->width * out->height);
    orc_remap_map(in, out, map);
    orc_remap_apply_map(map, out->width, out->height, img_in, in->width, in->height, interp, img_out);
    free(map);
}
