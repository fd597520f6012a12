/*
 * triangulate_oracle.c -- CPU oracle of acm_triangulate (test infrastructure only).
 *
 * The reference has no triangulation: this composes the oracle's restatements of its functions (oracle/acm_oracle.h) --
 * orc_unproject, orc_project_nobounds and orc_project_point_jacobian -- with the midpoint and Levenberg-Marquardt steps
 * and constants that include/acm.h documents, in the same separately rounded operation order as the kernel
 * (apex_camera_models_b200/csrc/acm_triangulate.cu).  x_cam2 = R x_cam1 + t, R row-major.
 * Built with the oracle's flags (-O2 -ffp-contract=off -fno-fast-math) together with its sources.
 */
#include <math.h>
#include <string.h>

#include "acm_oracle.h"

enum { TRI_OK = 0, TRI_UNPROJECT_FIRST = 1, TRI_UNPROJECT_SECOND = 2, TRI_PARALLEL = 3, TRI_BEHIND = 4, TRI_PROJECT = 5 };
#define TRI_PARALLEL_EPS 1e-12
#define TRI_LAMBDA0 1e-3
#define TRI_LAMBDA_FACTOR 10.0
#define TRI_STEP_TOL 1e-12

typedef struct {
    const orc_model *a, *b;
    const double* R;
    const double* t;
    double u1, v1, u2, v2;
} pair_t;

static void to_second(const pair_t* P, const double X[3], double Y[3]) {
    for (int i = 0; i < 3; ++i) Y[i] = ((P->R[3 * i] * X[0] + P->R[3 * i + 1] * X[1]) + P->R[3 * i + 2] * X[2]) + P->t[i];
}

static int residuals(const pair_t* P, const double X[3], double r[4], double* cost) {
    double p[2], q[2], Y[3];
    if (orc_project_nobounds(P->a, X, p) != ORC_OK) return 0;
    to_second(P, X, Y);
    if (orc_project_nobounds(P->b, Y, q) != ORC_OK) return 0;
    r[0] = p[0] - P->u1; r[1] = p[1] - P->v1; r[2] = q[0] - P->u2; r[3] = q[1] - P->v2;
    *cost = ((r[0] * r[0] + r[1] * r[1]) + r[2] * r[2]) + r[3] * r[3];
    return 1;
}

static int damped_solve(const double H[6], const double g[3], double lambda, double d[3]) {
    const double a00 = H[0] + lambda * H[0], a11 = H[3] + lambda * H[3], a22 = H[5] + lambda * H[5];
    if (!(a00 > 0.0)) return 0;
    const double l00 = sqrt(a00);
    const double l10 = H[1] / l00, l20 = H[2] / l00;
    const double p11 = a11 - l10 * l10;
    if (!(p11 > 0.0)) return 0;
    const double l11 = sqrt(p11);
    const double l21 = (H[4] - l20 * l10) / l11;
    const double p22 = (a22 - l20 * l20) - l21 * l21;
    if (!(p22 > 0.0)) return 0;
    const double l22 = sqrt(p22);
    const double y0 = -g[0] / l00;
    const double y1 = (-g[1] - l10 * y0) / l11;
    const double y2 = ((-g[2] - l20 * y0) - l21 * y1) / l22;
    d[2] = y2 / l22;
    d[1] = (y1 - l21 * d[2]) / l11;
    d[0] = ((y0 - l10 * d[1]) - l20 * d[2]) / l00;
    return 1;
}

int orc_triangulate1(const orc_model* a, const orc_model* b, const double R[9], const double t[3], const double uv1[2], const double uv2[2],
                     int max_iterations, double X[3], double err[2]) {
    X[0] = X[1] = X[2] = err[0] = err[1] = NAN;
    const pair_t P = {a, b, R, t, uv1[0], uv1[1], uv2[0], uv2[1]};
    double d1[3], d2[3], e[3], c2[3], Xm[3];
    if (orc_unproject(a, uv1, d1) != ORC_OK) return TRI_UNPROJECT_FIRST;
    if (orc_unproject(b, uv2, d2) != ORC_OK) return TRI_UNPROJECT_SECOND;
    for (int k = 0; k < 3; ++k) {
        e[k] = (R[k] * d2[0] + R[3 + k] * d2[1]) + R[6 + k] * d2[2];
        c2[k] = -((R[k] * t[0] + R[3 + k] * t[1]) + R[6 + k] * t[2]);
    }
    const double bb = (d1[0] * e[0] + d1[1] * e[1]) + d1[2] * e[2];
    const double p = (d1[0] * c2[0] + d1[1] * c2[1]) + d1[2] * c2[2];
    const double q = (e[0] * c2[0] + e[1] * c2[1]) + e[2] * c2[2];
    const double den = 1.0 - bb * bb;
    if (den <= TRI_PARALLEL_EPS) return TRI_PARALLEL;
    const double s1 = (p - bb * q) / den, s2 = (bb * p - q) / den;
    if (s1 <= 0.0 || s2 <= 0.0) return TRI_BEHIND;
    for (int k = 0; k < 3; ++k) Xm[k] = 0.5 * ((s1 * d1[k] + c2[k]) + s2 * e[k]);
    double r[4], cost;
    if (!residuals(&P, Xm, r, &cost)) return TRI_PROJECT;

    double lambda = TRI_LAMBDA0, H[6], g[3];
    int fresh = 0;
    for (int it = 0; it < max_iterations; ++it) {
        if (!fresh) {
            double J[4][3], ja[6], jb[6], Y[3], uv[2];
            orc_project_point_jacobian(a, Xm, uv, ja);
            to_second(&P, Xm, Y);
            orc_project_point_jacobian(b, Y, uv, jb);
            for (int k = 0; k < 3; ++k) { J[0][k] = ja[k]; J[1][k] = ja[3 + k]; }
            for (int row = 0; row < 2; ++row)
                for (int k = 0; k < 3; ++k) J[2 + row][k] = (jb[3 * row] * R[k] + jb[3 * row + 1] * R[3 + k]) + jb[3 * row + 2] * R[6 + k];
            int h = 0;
            for (int i = 0; i < 3; ++i) {
                g[i] = ((J[0][i] * r[0] + J[1][i] * r[1]) + J[2][i] * r[2]) + J[3][i] * r[3];
                for (int c = i; c < 3; ++c) H[h++] = ((J[0][i] * J[0][c] + J[1][i] * J[1][c]) + J[2][i] * J[2][c]) + J[3][i] * J[3][c];
            }
            fresh = 1;
        }
        double d[3], Xt[3], rt[4], ct = 0.0;
        int accept = damped_solve(H, g, lambda, d);
        if (accept) {
            for (int k = 0; k < 3; ++k) Xt[k] = Xm[k] + d[k];
            accept = residuals(&P, Xt, rt, &ct) && ct < cost;
        }
        if (!accept) { lambda = lambda * TRI_LAMBDA_FACTOR; continue; }
        memcpy(Xm, Xt, sizeof(Xm));
        memcpy(r, rt, sizeof(r));
        cost = ct;
        lambda = lambda / TRI_LAMBDA_FACTOR;
        fresh = 0;
        const double dmax = fmax(fabs(d[0]), fmax(fabs(d[1]), fabs(d[2])));
        const double xmax = fmax(fabs(Xm[0]), fmax(fabs(Xm[1]), fabs(Xm[2])));
        if (dmax <= TRI_STEP_TOL * fmax(1.0, xmax)) break;
    }
    memcpy(X, Xm, sizeof(Xm));
    err[0] = sqrt(r[0] * r[0] + r[1] * r[1]);
    err[1] = sqrt(r[2] * r[2] + r[3] * r[3]);
    return TRI_OK;
}

/* n pairs, AoS in (uvuv..) and out (xyz.., e1 e2 ..); nthreads > 1: OpenMP over the pairs */
void orc_triangulate(const orc_model* a, const orc_model* b, const double R[9], const double t[3], const double* uv1, const double* uv2,
                     size_t n, int max_iterations, double* xyz, double* err, uint8_t* status, int nthreads) {
    (void)nthreads;
#ifdef _OPENMP
#pragma omp parallel for schedule(static) num_threads(nthreads > 0 ? nthreads : 1)
#endif
    for (long long i = 0; i < (long long)n; ++i)
        status[i] = (uint8_t)orc_triangulate1(a, b, R, t, uv1 + 2 * i, uv2 + 2 * i, max_iterations, xyz + 3 * i, err + 2 * i);
}

/* the cost 0.5 * sum r^2 and the 4 residuals at X (for the checks against scipy); returns 0 when X does not project */
int orc_triangulate_residuals(const orc_model* a, const orc_model* b, const double R[9], const double t[3], const double uv1[2],
                              const double uv2[2], const double X[3], double r[4]) {
    const pair_t P = {a, b, R, t, uv1[0], uv1[1], uv2[0], uv2[1]};
    double cost;
    return residuals(&P, X, r, &cost);
}
