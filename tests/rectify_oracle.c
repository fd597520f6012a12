/*
 * rectify_oracle.c -- CPU oracle of the rotated camera-to-camera remap (test infrastructure only).
 *
 * Output pixel (u, v) of the output camera's grid:
 *   ray_o = out.unproject((u, v))                                  -- with its pixel-bounds test
 *   ray_i[k] = (R[0][k] * x + R[1][k] * y) + R[2][k] * z            -- R^T ray_o, R row-major with x_out = R x_in
 *   src = in.project(ray_i)                                        -- if the unproject is Ok
 * NaN where a step fails.  Built with the oracle's flags together with its sources and remap_oracle.c, whose
 * orc_remap_apply_map turns the map into frame bytes.
 */
#include <math.h>
#include <stdlib.h>

#include "acm_oracle.h"

void orc_remap_apply_map(const double* src_xy, uint32_t Wo, uint32_t Ho, const uint8_t* img_in, uint32_t Wi, uint32_t Hi, int interp,
                         uint8_t* img_out);

void orc_remap_map_rotated(const orc_model* in, const orc_model* out, const double R[9], double* src_xy) {
    for (uint32_t v = 0; v < out->height; ++v)
        for (uint32_t u = 0; u < out->width; ++u) {
            const double uv[2] = {(double)u, (double)v};
            double ro[3], ri[3], p[2] = {NAN, NAN};
            if (orc_unproject(out, uv, ro) == ORC_OK) {
                for (int k = 0; k < 3; ++k) ri[k] = (R[k] * ro[0] + R[3 + k] * ro[1]) + R[6 + k] * ro[2];
                if (orc_project(in, ri, p) != ORC_OK) p[0] = p[1] = NAN;
            }
            src_xy[2 * ((size_t)v * out->width + u)] = p[0];
            src_xy[2 * ((size_t)v * out->width + u) + 1] = p[1];
        }
}

void orc_remap_rgb8_rotated(const orc_model* in, const orc_model* out, const double R[9], const uint8_t* img_in, uint8_t* img_out,
                            int interp) {
    double* map = (double*)malloc(sizeof(double) * 2 * (size_t)out->width * out->height);
    orc_remap_map_rotated(in, out, R, map);
    orc_remap_apply_map(map, out->width, out->height, img_in, in->width, in->height, interp, img_out);
    free(map);
}
