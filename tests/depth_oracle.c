/*
 * depth_oracle.c -- CPU oracle of acm_render_depth / acm_depth_to_points (test infrastructure only).
 *
 * The reference has no depth images: this composes the oracle's restatements of its functions (oracle/acm_oracle.h) --
 * orc_project_nobounds and orc_unproject -- with the transform, nearest-pixel rounding, range and z-buffer key that
 * include/acm.h documents, in the same separately rounded operation order as the kernels
 * (apex_camera_models_b200/csrc/acm_depth.cu).  The render is a sequential minimum of the keys.
 * Built with the oracle's flags (-O2 -ffp-contract=off -fno-fast-math) together with its sources.
 */
#include <math.h>
#include <stdlib.h>
#include <string.h>

#include "acm_oracle.h"

enum { DEPTH_OK = 0, DEPTH_EMPTY = 1, DEPTH_UNPROJECT = 2 };

static void rigid_apply(const double R[9], const double t[3], const double X[3], double Y[3]) {
    for (int i = 0; i < 3; ++i) Y[i] = ((R[3 * i] * X[0] + R[3 * i + 1] * X[1]) + R[3 * i + 2] * X[2]) + t[i];
}

static uint32_t f32_bits(float f) {
    uint32_t b;
    memcpy(&b, &f, 4);
    return b;
}

/* The pixel (r*W + c) and key of point X, or -1 when it is not drawn; uv receives the projection (NaN when it fails). */
long long orc_depth_key1(const orc_model* m, const double R[9], const double t[3], const double X[3], uint32_t i, double uv[2],
                         uint64_t* key) {
    double Q[3];
    rigid_apply(R, t, X, Q);
    if (orc_project_nobounds(m, Q, uv) != ORC_OK) { uv[0] = uv[1] = NAN; return -1; }
    const double rx = round(uv[0]), ry = round(uv[1]);
    if (!(rx >= 0.0 && rx < (double)m->width && ry >= 0.0 && ry < (double)m->height)) return -1;
    const double range = sqrt((Q[0] * Q[0] + Q[1] * Q[1]) + Q[2] * Q[2]);
    if (!(range > 0.0 && range < INFINITY)) return -1;
    *key = ((uint64_t)f32_bits((float)range) << 32) | (uint64_t)i;
    return (long long)ry * (long long)m->width + (long long)rx;
}

/* n AoS points -> W*H range (f32) and index images: empty pixels hold range bits 0xFFFFFFFF and index UINT32_MAX.
 * uv (optional, 2n): each point's projection, NaN where project fails. */
void orc_render_depth(const orc_model* m, const double R[9], const double t[3], const double* xyz, size_t n, float* range,
                      uint32_t* index, double* uv) {
    const size_t npix = (size_t)m->width * m->height;
    uint64_t* keys = (uint64_t*)malloc((npix ? npix : 1) * sizeof(uint64_t));
    for (size_t p = 0; p < npix; ++p) keys[p] = ~(uint64_t)0;
    for (size_t i = 0; i < n; ++i) {
        double puv[2];
        uint64_t key = 0;
        const long long p = orc_depth_key1(m, R, t, xyz + 3 * i, (uint32_t)i, puv, &key);
        if (uv) { uv[2 * i] = puv[0]; uv[2 * i + 1] = puv[1]; }
        if (p >= 0 && key < keys[p]) keys[p] = key;
    }
    for (size_t p = 0; p < npix; ++p) {
        const uint32_t hi = (uint32_t)(keys[p] >> 32);
        memcpy(range + p, &hi, 4);
        index[p] = (uint32_t)keys[p];
    }
    free(keys);
}

/* W*H range image -> W*H AoS points (NaN where status != OK) and status */
void orc_depth_to_points(const orc_model* m, const double R[9], const double t[3], const float* range, double* xyz, uint8_t* status) {
    const size_t W = m->width, npix = (size_t)m->width * m->height;
    for (size_t p = 0; p < npix; ++p) {
        double* X = xyz + 3 * p;
        X[0] = X[1] = X[2] = NAN;
        const float d = range[p];
        if (!(d > 0.0f && d < INFINITY)) { status[p] = DEPTH_EMPTY; continue; }
        const double uv[2] = {(double)(p % W), (double)(p / W)};
        double ray[3], q[3];
        if (orc_unproject(m, uv, ray) != ORC_OK) { status[p] = DEPTH_UNPROJECT; continue; }
        const double dd = (double)d;
        for (int k = 0; k < 3; ++k) q[k] = ray[k] * dd - t[k];
        for (int k = 0; k < 3; ++k) X[k] = (R[k] * q[0] + R[3 + k] * q[1]) + R[6 + k] * q[2];
        status[p] = DEPTH_OK;
    }
}
