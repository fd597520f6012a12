/*
 * acm_oracle_solver.c -- CPU ORACLE. TEST INFRASTRUCTURE ONLY (see acm_oracle.h).
 *
 * Residuals, analytic parameter Jacobians, dense normal equations and a Levenberg-Marquardt
 * loop.  In the reference these live in the un-vendored crate apex-solver "0.1.5"
 * (ref: Cargo.toml:28; call sites bin/camera_converter.rs:378-420 and its five clones), so
 * this file restates the *published model derivatives* (SURVEY.md Appendix A) and a textbook
 * LM (Nielsen damping, Jacobi scaling, box projection) -- PARITY UNPINNED at that boundary.
 * Also: the in-tree linear_estimation of every model.
 */
#include "acm_oracle.h"
#include <math.h>
#include <stdlib.h>
#include <string.h>

#define EPS 2.220446049250313e-16
#define SQRT_EPS 1.4901161193847656e-08
#define PRECISION 1e-3

/* 2xP Jacobian of the projection w.r.t. [fx,fy,cx,cy,dist...] (README-era compute_jacobian;
 * ref doc-comments double_sphere.rs:326-332 "2x6", kannala_brandt.rs:309-313 "2x8") */
int orc_project_jacobian(const orc_model* m, const double X[3], double uv[2], double* J) {
    const int P = m->n_params;
    int st = orc_project_nobounds(m, X, uv);
    memset(J, 0, sizeof(double) * 2 * (size_t)P);
    if (st != ORC_OK) return st;
    const double fx = m->p[0], fy = m->p[1], cx = m->p[2], cy = m->p[3];
    const double x = X[0], y = X[1], z = X[2];
    double* Ju = J;
    double* Jv = J + P;
    /* common intrinsics block: u = fx*mx + cx  =>  du/dfx = mx, du/dcx = 1 */
    double mx = 0.0, my = 0.0;
    (void)cx; (void)cy;
    Ju[2] = 1.0; Jv[3] = 1.0;
    switch (m->model) {
    case ORC_PINHOLE: mx = x / z; my = y / z; break;
    case ORC_RADTAN: {
        double xp = x / z, yp = y / z;
        double rho = xp * xp + yp * yp;
        const double k1 = m->p[4], k2 = m->p[5], p1 = m->p[6], p2 = m->p[7], k3 = m->p[8];
        double rad = 1.0 + k1 * rho + k2 * rho * rho + k3 * rho * rho * rho;
        mx = xp * rad + 2.0 * p1 * xp * yp + p2 * (rho + 2.0 * xp * xp);
        my = yp * rad + p1 * (rho + 2.0 * yp * yp) + 2.0 * p2 * xp * yp;
        Ju[4] = fx * xp * rho;            Jv[4] = fy * yp * rho;
        Ju[5] = fx * xp * rho * rho;      Jv[5] = fy * yp * rho * rho;
        Ju[6] = fx * 2.0 * xp * yp;       Jv[6] = fy * (rho + 2.0 * yp * yp);
        Ju[7] = fx * (rho + 2.0 * xp * xp); Jv[7] = fy * 2.0 * xp * yp;
        Ju[8] = fx * xp * rho * rho * rho; Jv[8] = fy * yp * rho * rho * rho;
        break;
    }
    case ORC_KB: {
        double r = sqrt(x * x + y * y);
        double th = atan2(r, z);
        double xr = (r < EPS) ? 0.0 : x / r, yr = (r < EPS) ? 0.0 : y / r;
        double t2 = th * th, t3 = t2 * th, t5 = t3 * t2, t7 = t5 * t2, t9 = t7 * t2;
        Ju[4] = fx * t3 * xr; Jv[4] = fy * t3 * yr;
        Ju[5] = fx * t5 * xr; Jv[5] = fy * t5 * yr;
        Ju[6] = fx * t7 * xr; Jv[6] = fy * t7 * yr;
        Ju[7] = fx * t9 * xr; Jv[7] = fy * t9 * yr;
        double thd = th + m->p[4] * t3 + m->p[5] * t5 + m->p[6] * t7 + m->p[7] * t9;
        mx = thd * xr; my = thd * yr;
        break;
    }
    case ORC_UCM: {
        double alpha = m->p[4];
        double d = sqrt(x * x + y * y + z * z);
        double den = alpha * d + (1.0 - alpha) * z;
        Ju[4] = -fx * x * (d - z) / (den * den);
        Jv[4] = -fy * y * (d - z) / (den * den);
        mx = x / den; my = y / den;
        break;
    }
    case ORC_EUCM: {
        double alpha = m->p[4], beta = m->p[5];
        double rr = x * x + y * y;
        double d = sqrt(beta * rr + z * z);
        double den = alpha * d + (1.0 - alpha) * z;
        double dden_da = d - z;
        double dden_db = alpha * rr / (2.0 * d);
        Ju[4] = -fx * x * dden_da / (den * den); Jv[4] = -fy * y * dden_da / (den * den);
        Ju[5] = -fx * x * dden_db / (den * den); Jv[5] = -fy * y * dden_db / (den * den);
        mx = x / den; my = y / den;
        break;
    }
    case ORC_DS: {
        double alpha = m->p[4], xi = m->p[5];
        double rr = x * x + y * y;
        double d1 = sqrt(rr + z * z);
        double g = xi * d1 + z;
        double d2 = sqrt(rr + g * g);
        double den = alpha * d2 + (1.0 - alpha) * g;
        double dden_da = d2 - g;
        double dden_dxi = alpha * g * d1 / d2 + (1.0 - alpha) * d1;
        Ju[4] = -fx * x * dden_da / (den * den);  Jv[4] = -fy * y * dden_da / (den * den);
        Ju[5] = -fx * x * dden_dxi / (den * den); Jv[5] = -fy * y * dden_dxi / (den * den);
        mx = x / den; my = y / den;
        break;
    }
    case ORC_FOV: {
        double w = m->p[4];
        double r2 = x * x + y * y, r = sqrt(r2);
        double t = tan(w / 2.0);
        double drd, rd;
        if (r2 < SQRT_EPS) {
            rd = 2.0 * t / w;
            drd = (1.0 + t * t) / w - 2.0 * t / (w * w);
        } else {
            double a = atan2(2.0 * t * r, z);
            double da = z * r * (1.0 + t * t) / (4.0 * t * t * r2 + z * z);
            rd = a / (r * w);
            drd = da / (r * w) - a / (r * w * w);
        }
        Ju[4] = fx * x * drd; Jv[4] = fy * y * drd;
        mx = x * rd; my = y * rd;
        break;
    }
    default: return ORC_NUMERICAL;
    }
    Ju[0] = mx; Jv[1] = my;
    return ORC_OK;
}

/* denominator of the unified family and its derivatives w.r.t. the distortion parameters */
static int unified_den(const orc_model* m, const double X[3], double* den, double dd[2]) {
    const double x = X[0], y = X[1], z = X[2];
    switch (m->model) {
    case ORC_UCM: {
        double alpha = m->p[4];
        double d = sqrt(x * x + y * y + z * z);
        *den = alpha * d + (1.0 - alpha) * z; dd[0] = d - z; dd[1] = 0.0; return 1;
    }
    case ORC_EUCM: {
        double alpha = m->p[4], beta = m->p[5];
        double rr = x * x + y * y;
        double d = sqrt(beta * rr + z * z);
        *den = alpha * d + (1.0 - alpha) * z; dd[0] = d - z; dd[1] = alpha * rr / (2.0 * d); return 2;
    }
    case ORC_DS: {
        double alpha = m->p[4], xi = m->p[5];
        double rr = x * x + y * y;
        double d1 = sqrt(rr + z * z);
        double g = xi * d1 + z;
        double d2 = sqrt(rr + g * g);
        *den = alpha * d2 + (1.0 - alpha) * g;
        dd[0] = d2 - g; dd[1] = alpha * g * d1 / d2 + (1.0 - alpha) * d1; return 2;
    }
    default: return 0;
    }
}

int orc_residual_jacobian(const orc_model* m, int kind, const double X[3], const double uv_obs[2], double r[2], double* J) {
    const int P = m->n_params;
    if (kind == ORC_RES_ALGEBRAIC) {
        /* r_x = fx*x - (u_obs-cx)*den  (the system the in-tree linear_estimation solves:
         * ref double_sphere.rs:253-257, ucm.rs:221-231, eucm.rs:247-257) */
        double uvp[2];
        int st = orc_project_nobounds(m, X, uvp);
        memset(J, 0, sizeof(double) * 2 * (size_t)P);
        r[0] = r[1] = 0.0;
        double den, dd[2];
        int nd = unified_den(m, X, &den, dd);
        if (nd == 0) return ORC_NUMERICAL; /* no algebraic form for this model */
        if (st != ORC_OK) return st;
        const double fx = m->p[0], fy = m->p[1], cx = m->p[2], cy = m->p[3];
        double du = uv_obs[0] - cx, dv = uv_obs[1] - cy;
        r[0] = fx * X[0] - du * den;
        r[1] = fy * X[1] - dv * den;
        double* Jx = J; double* Jy = J + P;
        Jx[0] = X[0]; Jx[2] = den;
        Jy[1] = X[1]; Jy[3] = den;
        for (int k = 0; k < nd; ++k) { Jx[4 + k] = -du * dd[k]; Jy[4 + k] = -dv * dd[k]; }
        return ORC_OK;
    }
    double uvp[2];
    int st = orc_project_jacobian(m, X, uvp, J);
    if (st != ORC_OK) { r[0] = r[1] = 0.0; return st; }
    r[0] = uvp[0] - uv_obs[0];
    r[1] = uvp[1] - uv_obs[1];
    return ORC_OK;
}

/* batch forms of the two Jacobians over AoS points, mirroring orc_project_batch: uv (n x 2), status (n) and
 * J row-major per point -- (n x 2 x P) for the parameter Jacobian, (n x 2 x 3) for the point Jacobian */
void orc_project_jacobian_batch(const orc_model* m, const double* xyz, size_t n, double* uv, double* J, uint8_t* status, int nthreads) {
    const size_t P = (size_t)m->n_params;
    (void)nthreads;
#ifdef _OPENMP
#pragma omp parallel for schedule(static) num_threads(nthreads > 0 ? nthreads : 1)
#endif
    for (long long i = 0; i < (long long)n; ++i)
        status[i] = (uint8_t)orc_project_jacobian(m, xyz + 3 * i, uv + 2 * i, J + 2 * P * (size_t)i);
}

void orc_project_point_jacobian_batch(const orc_model* m, const double* xyz, size_t n, double* uv, double* J, uint8_t* status, int nthreads) {
    (void)nthreads;
#ifdef _OPENMP
#pragma omp parallel for schedule(static) num_threads(nthreads > 0 ? nthreads : 1)
#endif
    for (long long i = 0; i < (long long)n; ++i)
        status[i] = (uint8_t)orc_project_point_jacobian(m, xyz + 3 * i, uv + 2 * i, J + 6 * (size_t)i);
}

/* Dense path: materialise r and J for the chunk, then form J^T J and J^T r.  This is what the
 * reference's generic solver does (SURVEY.md 8a row a18) and is the timed CPU baseline. */
static void linearize_chunk(const orc_model* m, int kind, const double* xyz, const double* uv, size_t n,
                            double* H, double* g, double* cost, uint64_t* nvalid) {
    const int P = m->n_params;
    const size_t CH = 4096;
    double* J = (double*)malloc(sizeof(double) * 2 * CH * (size_t)P);
    double* r = (double*)malloc(sizeof(double) * 2 * CH);
    memset(H, 0, sizeof(double) * (size_t)P * P);
    memset(g, 0, sizeof(double) * (size_t)P);
    double c = 0.0; uint64_t nv = 0;
    for (size_t base = 0; base < n; base += CH) {
        size_t cnt = (n - base < CH) ? n - base : CH;
        for (size_t i = 0; i < cnt; ++i) {
            int st = orc_residual_jacobian(m, kind, xyz + 3 * (base + i), uv + 2 * (base + i), r + 2 * i, J + 2 * i * P);
            if (st == ORC_OK) ++nv;
            else { r[2 * i] = r[2 * i + 1] = 0.0; memset(J + 2 * i * P, 0, sizeof(double) * 2 * (size_t)P); }
        }
        for (size_t row = 0; row < 2 * cnt; ++row) {
            const double* Jr = J + row * P;
            double rr = r[row];
            c += rr * rr;
            for (int a = 0; a < P; ++a) {
                double ja = Jr[a];
                g[a] += ja * rr;
                for (int b = a; b < P; ++b) H[a * P + b] += ja * Jr[b];
            }
        }
    }
    for (int a = 0; a < P; ++a) for (int b = 0; b < a; ++b) H[a * P + b] = H[b * P + a];
    *cost = 0.5 * c; *nvalid = nv;
    free(J); free(r);
}

int orc_linearize(const orc_model* m, int kind, const double* xyz, const double* uv, size_t n,
                  double* H, double* g, double* cost, uint64_t* n_valid, int nthreads) {
    const int P = m->n_params;
    if (kind == ORC_RES_ALGEBRAIC && !(m->model == ORC_UCM || m->model == ORC_EUCM || m->model == ORC_DS)) return -1;
    if (nthreads <= 1) { linearize_chunk(m, kind, xyz, uv, n, H, g, cost, n_valid); return 0; }
    double* Hs = (double*)calloc((size_t)nthreads * P * P, sizeof(double));
    double* gs = (double*)calloc((size_t)nthreads * P, sizeof(double));
    double* cs = (double*)calloc((size_t)nthreads, sizeof(double));
    uint64_t* ns = (uint64_t*)calloc((size_t)nthreads, sizeof(uint64_t));
#ifdef _OPENMP
#pragma omp parallel for schedule(static, 1) num_threads(nthreads)
#endif
    for (int t = 0; t < nthreads; ++t) {
        size_t lo = n * (size_t)t / (size_t)nthreads, hi = n * (size_t)(t + 1) / (size_t)nthreads;
        linearize_chunk(m, kind, xyz + 3 * lo, uv + 2 * lo, hi - lo, Hs + (size_t)t * P * P, gs + (size_t)t * P, cs + t, ns + t);
    }
    memset(H, 0, sizeof(double) * (size_t)P * P); memset(g, 0, sizeof(double) * (size_t)P);
    *cost = 0.0; *n_valid = 0;
    for (int t = 0; t < nthreads; ++t) {
        for (int k = 0; k < P * P; ++k) H[k] += Hs[(size_t)t * P * P + k];
        for (int k = 0; k < P; ++k) g[k] += gs[(size_t)t * P + k];
        *cost += cs[t]; *n_valid += ns[t];
    }
    free(Hs); free(gs); free(cs); free(ns);
    return 0;
}

/* ------------------------------------------------------------------ LM --------------- */
void orc_lm_default_config(orc_lm_config* c) {
    /* ref: bin/camera_converter.rs:410-415 */
    c->max_iterations = 100; c->cost_tolerance = 1e-6; c->parameter_tolerance = 1e-8; c->gradient_tolerance = 1e-6;
    c->lambda0 = 1e-3; c->invalid_penalty = 0.0;
}

/* divisions hoisted into reciprocals of the diagonal (same arithmetic as the device step) */
static int chol_solve(int P, const double* A, const double* b, double* x) {
    double L[81], inv[9];
    for (int i = 0; i < P; ++i) {
        for (int j = 0; j <= i; ++j) {
            double s = A[i * P + j];
            for (int k = 0; k < j; ++k) s -= L[i * P + k] * L[j * P + k];
            if (i == j) { if (!(s > 0.0)) return 0; L[i * P + i] = sqrt(s); inv[i] = 1.0 / L[i * P + i]; }
            else L[i * P + j] = s * inv[j];
        }
    }
    double yv[9];
    for (int i = 0; i < P; ++i) { double s = b[i]; for (int k = 0; k < i; ++k) s -= L[i * P + k] * yv[k]; yv[i] = s * inv[i]; }
    for (int i = P - 1; i >= 0; --i) { double s = yv[i]; for (int k = i + 1; k < P; ++k) s -= L[k * P + i] * x[k]; x[i] = s * inv[i]; }
    return 1;
}

static double clampd(double v, double lo, double hi) { return v < lo ? lo : (v > hi ? hi : v); }

int orc_lm_solve(const orc_model* m_init, int kind, const double* xyz, const double* uv, size_t n,
                 const double* lower, const double* upper, const orc_lm_config* cfg, double* out_params,
                 orc_lm_result* res, int nthreads) {
    orc_model m = *m_init;
    const int P = m.n_params;
    double x[9], xt[9], H[81], g[9], Ht[81], gt[9], A[81], gs[9], s[9], dx[9], D[9];
    for (int i = 0; i < P; ++i) x[i] = clampd(m.p[i], lower ? lower[i] : -INFINITY, upper ? upper[i] : INFINITY);
    double cost, cost_t; uint64_t nv, nvt;
    memcpy(m.p, x, sizeof(double) * P);
    if (orc_linearize(&m, kind, xyz, uv, n, H, g, &cost, &nv, nthreads) != 0) return -1;
    cost += (double)(n - nv) * cfg->invalid_penalty * cfg->invalid_penalty;
    res->initial_cost = cost; res->passes = 1; res->iterations = 0; res->status = 3;
    double lambda = cfg->lambda0, nu = 2.0;
    while (res->iterations < cfg->max_iterations) {
        res->iterations++;
        for (int i = 0; i < P; ++i) { double d = sqrt(H[i * P + i]); D[i] = (d > 1e-300) ? 1.0 / d : 1.0; } /* D holds 1/sqrt(H_ii) */
        for (int i = 0; i < P; ++i) {
            for (int j = 0; j < P; ++j) A[i * P + j] = H[i * P + j] * D[i] * D[j];
            A[i * P + i] += lambda;
            gs[i] = -g[i] * D[i];
        }
        if (!chol_solve(P, A, gs, s)) { lambda *= nu; nu *= 2.0; if (lambda > 1e30) { res->status = 4; break; } continue; }
        double xnorm = 0.0, dnorm = 0.0;
        for (int i = 0; i < P; ++i) {
            xt[i] = clampd(x[i] + s[i] * D[i], lower ? lower[i] : -INFINITY, upper ? upper[i] : INFINITY);
            dx[i] = xt[i] - x[i];
            xnorm += x[i] * x[i]; dnorm += dx[i] * dx[i];
        }
        xnorm = sqrt(xnorm); dnorm = sqrt(dnorm);
        double pred = 0.0;
        for (int i = 0; i < P; ++i) {
            double hd = 0.0;
            for (int j = 0; j < P; ++j) hd += H[i * P + j] * dx[j];
            pred -= dx[i] * (g[i] + 0.5 * hd);
        }
        memcpy(m.p, xt, sizeof(double) * P);
        orc_linearize(&m, kind, xyz, uv, n, Ht, gt, &cost_t, &nvt, nthreads);
        cost_t += (double)(n - nvt) * cfg->invalid_penalty * cfg->invalid_penalty;
        res->passes++;
        int small_step = dnorm <= cfg->parameter_tolerance * (xnorm + cfg->parameter_tolerance);
        if (pred > 0.0 && cost_t < cost) {
            double rho = (cost - cost_t) / pred;
            double dcost = cost - cost_t, cost_old = cost;
            memcpy(x, xt, sizeof(double) * P); memcpy(H, Ht, sizeof(double) * P * P); memcpy(g, gt, sizeof(double) * P);
            cost = cost_t; nv = nvt;
            double q = 2.0 * rho - 1.0, f = 1.0 - q * q * q;
            lambda *= (f > 1.0 / 3.0) ? f : 1.0 / 3.0; nu = 2.0;
            if (lambda < 1e-15) lambda = 1e-15;
            double gmax = 0.0; for (int i = 0; i < P; ++i) if (fabs(g[i]) > gmax) gmax = fabs(g[i]);
            if (dcost <= cfg->cost_tolerance * cost_old) { res->status = 0; break; }
            if (small_step) { res->status = 1; break; }
            if (gmax <= cfg->gradient_tolerance) { res->status = 2; break; }
        } else {
            if (small_step) { res->status = 1; break; }
            lambda *= nu; nu *= 2.0;
            if (lambda > 1e30) { res->status = 4; break; }
        }
    }
    memcpy(out_params, x, sizeof(double) * P);
    res->final_cost = cost; res->n_valid = nv;
    return 0;
}

/* ------------------------------------------------------------------ linear estimation - */
/* Least squares via one-sided Jacobi SVD with nalgebra's SVD::solve(b, eps) semantics:
 * singular values <= eps are dropped (ref: double_sphere.rs:261-262 eps 1e-10,
 * kannala_brandt.rs:262-263 eps f64::EPSILON, rad_tan.rs:213-214 eps 1e-10). */
static void svd_solve(double* A, size_t mrows, int k, const double* b, double eps, double* x) {
    double V[16];
    for (int i = 0; i < k; ++i) for (int j = 0; j < k; ++j) V[i * k + j] = (i == j);
    for (int sweep = 0; sweep < 60; ++sweep) {
        int rotated = 0;
        for (int p = 0; p < k - 1; ++p) for (int q = p + 1; q < k; ++q) {
            double al = 0, be = 0, ga = 0;
            for (size_t i = 0; i < mrows; ++i) { double ap = A[i * k + p], aq = A[i * k + q]; al += ap * ap; be += aq * aq; ga += ap * aq; }
            if (fabs(ga) <= 1e-16 * sqrt(al * be) || ga == 0.0) continue;
            rotated = 1;
            double zeta = (be - al) / (2.0 * ga);
            double t = (zeta >= 0 ? 1.0 : -1.0) / (fabs(zeta) + sqrt(1.0 + zeta * zeta));
            double c = 1.0 / sqrt(1.0 + t * t), s = c * t;
            for (size_t i = 0; i < mrows; ++i) { double ap = A[i * k + p], aq = A[i * k + q]; A[i * k + p] = c * ap - s * aq; A[i * k + q] = s * ap + c * aq; }
            for (int i = 0; i < k; ++i) { double vp = V[i * k + p], vq = V[i * k + q]; V[i * k + p] = c * vp - s * vq; V[i * k + q] = s * vp + c * vq; }
        }
        if (!rotated) break;
    }
    for (int j = 0; j < k; ++j) x[j] = 0.0;
    for (int j = 0; j < k; ++j) {
        double s2 = 0, ub = 0;
        for (size_t i = 0; i < mrows; ++i) { s2 += A[i * k + j] * A[i * k + j]; ub += A[i * k + j] * b[i]; }
        double sig = sqrt(s2);
        if (sig > eps) { double coef = ub / (sig * sig); for (int i = 0; i < k; ++i) x[i] += V[i * k + j] * coef; }
    }
}

int orc_linear_estimation(orc_model* m, const double* xyz, const double* uv, size_t n) {
    const double fx = m->p[0], fy = m->p[1], cx = m->p[2], cy = m->p[3];
    switch (m->model) {
    case ORC_UCM: case ORC_EUCM: case ORC_DS: {
        /* ref: double_sphere.rs:225-290, ucm.rs:200-258, eucm.rs:216-288 */
        if (m->model == ORC_EUCM) { if (n < 1) return -2; m->p[5] = 1.0; }
        double* A = (double*)calloc(2 * n + 1, sizeof(double));
        double* b = (double*)calloc(2 * n + 1, sizeof(double));
        for (size_t i = 0; i < n; ++i) {
            double x = xyz[3 * i], y = xyz[3 * i + 1], z = xyz[3 * i + 2], u = uv[2 * i], v = uv[2 * i + 1];
            double d = sqrt(x * x + y * y + z * z);
            double u_cx = u - cx, v_cy = v - cy;
            A[2 * i] = u_cx * (d - z); A[2 * i + 1] = v_cy * (d - z);
            b[2 * i] = (fx * x) - (u_cx * z); b[2 * i + 1] = (fy * y) - (v_cy * z);
        }
        double alpha;
        svd_solve(A, 2 * n, 1, b, 1e-10, &alpha);
        free(A); free(b);
        if (m->model == ORC_DS) {
            m->p[5] = 0.0;
            if (alpha <= 0.0) alpha = 0.01; else if (alpha > 1.0) alpha = 1.0;
            m->p[4] = alpha;
            if (!(alpha > 0.0 && alpha <= 1.0)) return -3; /* validate_params */
        } else if (m->model == ORC_UCM) {
            if (alpha <= 0.0) alpha = 0.01;
            m->p[4] = alpha;
            if (!isfinite(alpha)) return -3;
        } else {
            if (alpha <= 0.0) alpha = 0.01; else if (alpha > 2.0) alpha = 2.0;
            m->p[4] = alpha;
            if (!isfinite(alpha)) return -3;
        }
        return 0;
    }
    case ORC_KB: { /* ref: kannala_brandt.rs:164-272 */
        if (n < 4) return -2;
        double* A = (double*)calloc(2 * n * 4, sizeof(double));
        double* b = (double*)calloc(2 * n, sizeof(double));
        for (size_t i = 0; i < n; ++i) {
            double xw = xyz[3 * i], yw = xyz[3 * i + 1], zw = xyz[3 * i + 2], u = uv[2 * i], v = uv[2 * i + 1];
            if (zw <= EPS) continue;
            double rw = sqrt(xw * xw + yw * yw);
            double th = atan2(rw, zw);
            double t2 = th * th, t3 = t2 * th, t5 = t3 * t2, t7 = t5 * t2, t9 = t7 * t2;
            for (int rrow = 0; rrow < 2; ++rrow) { double* a = A + (2 * i + rrow) * 4; a[0] = t3; a[1] = t5; a[2] = t7; a[3] = t9; }
            double x_r = (rw < EPS) ? 0.0 : xw / rw, y_r = (rw < EPS) ? 0.0 : yw / rw;
            if (fabs(fx * x_r) < EPS && fabs(x_r) > EPS) { free(A); free(b); return -4; }
            if (fabs(fy * y_r) < EPS && fabs(y_r) > EPS) { free(A); free(b); return -4; }
            if (fabs(x_r) > EPS) b[2 * i] = (u - cx) / (fx * x_r) - th;
            else b[2 * i] = (fabs(u - cx) < EPS) ? -th : 0.0;
            if (fabs(y_r) > EPS) b[2 * i + 1] = (v - cy) / (fy * y_r) - th;
            else b[2 * i + 1] = (fabs(v - cy) < EPS) ? -th : 0.0;
        }
        double k[4];
        svd_solve(A, 2 * n, 4, b, EPS, k);
        free(A); free(b);
        for (int j = 0; j < 4; ++j) m->p[4 + j] = k[j];
        return 0;
    }
    case ORC_RADTAN: { /* ref: rad_tan.rs:153-234 */
        if (n < 3) return -2;
        double* A = (double*)calloc(2 * n * 3, sizeof(double));
        double* b = (double*)calloc(2 * n, sizeof(double));
        for (size_t i = 0; i < n; ++i) {
            double x = xyz[3 * i], y = xyz[3 * i + 1], z = xyz[3 * i + 2], u = uv[2 * i], v = uv[2 * i + 1];
            double xn = x / z, yn = y / z;
            double r2 = xn * xn + yn * yn, r4 = r2 * r2, r6 = r4 * r2;
            double uu = fx * xn + cx, vu = fy * yn + cy;
            double* a0 = A + (2 * i) * 3; double* a1 = A + (2 * i + 1) * 3;
            a0[0] = fx * xn * r2; a0[1] = fx * xn * r4; a0[2] = fx * xn * r6;
            a1[0] = fy * yn * r2; a1[1] = fy * yn * r4; a1[2] = fy * yn * r6;
            b[2 * i] = u - uu; b[2 * i + 1] = v - vu;
        }
        double k[3];
        svd_solve(A, 2 * n, 3, b, 1e-10, k);
        free(A); free(b);
        m->p[4] = k[0]; m->p[5] = k[1]; m->p[6] = 0.0; m->p[7] = 0.0; m->p[8] = k[2];
        return 0;
    }
    case ORC_FOV: { /* ref: fov.rs:153-251 -- grid search w = i/100, i in [10,300) */
        if (n < 2) return -2;
        double best_w = 1.0, best_err = INFINITY;
        for (int iw = 10; iw < 300; ++iw) {
            double w = (double)iw / 100.0;
            double sum = 0.0; long cnt = 0;
            for (size_t i = 0; i < n; ++i) {
                double x = xyz[3 * i], y = xyz[3 * i + 1], z = xyz[3 * i + 2];
                double r2 = x * x + y * y, r = sqrt(r2);
                double t = tan(w / 2.0);
                double a = atan2(2.0 * t * r, z);
                double rd = (r2 < SQRT_EPS) ? 2.0 * t / w : a / (r * w);
                double mx = x * rd, my = y * rd;
                double up = fx * mx + cx, vp = fy * my + cy;
                double du = up - uv[2 * i], dv = vp - uv[2 * i + 1];
                double e = sqrt(du * du + dv * dv);
                if (isfinite(e)) { sum += e; cnt++; }
            }
            if (cnt > 0) { double avg = sum / (double)cnt; if (avg < best_err) { best_err = avg; best_w = w; } }
        }
        double w = best_w;
        if (w <= EPS) w = 0.01; else if (w > 3.0) w = 3.0;
        m->p[4] = w;
        return 0;
    }
    default: return -1; /* Pinhole has no linear_estimation */
    }
}

/* 2x3 Jacobian of the projection w.r.t. the 3-D point (the "Jacobian matrix (2x3)" of the README-era
 * `project(&p, compute_jacobian)`, stale trait doc reference src/camera/mod.rs:246-252).  The reference
 * tree holds no code for it (SURVEY.md Appendix A: derived there, third column of the table); pinned by
 * mpmath 50-digit differences of the model definitions (tests/golden/mpmath_point_jacobians.json) and by
 * central differences of orc_project.  Jx row-major: [du/dx du/dy du/dz dv/dx dv/dy dv/dz].
 * Status = the geometric validity of the projection (no image-bounds test); Jx = 0 when it fails.
 * KB at r < EPS (the reference returns the principal point there): the analytic limit on the axis, fx/z.
 * FOV at r^2 < sqrt(EPS): the derivative of the reference's near-axis branch mx = x * (2 tan(w/2) / w). */
int orc_project_point_jacobian(const orc_model* m, const double X[3], double uv[2], double Jx[6]) {
    int st = orc_project_nobounds(m, X, uv);
    memset(Jx, 0, 6 * sizeof(double));
    if (st != ORC_OK) return st;
    const double fx = m->p[0], fy = m->p[1];
    const double x = X[0], y = X[1], z = X[2];
    double* Ju = Jx;
    double* Jv = Jx + 3;
    switch (m->model) {
    case ORC_PINHOLE: {
        Ju[0] = fx / z; Ju[2] = -fx * x / (z * z);
        Jv[1] = fy / z; Jv[2] = -fy * y / (z * z);
        break;
    }
    case ORC_RADTAN: {
        const double k1 = m->p[4], k2 = m->p[5], p1 = m->p[6], p2 = m->p[7], k3 = m->p[8];
        double a = x / z, b = y / z;
        double rho = a * a + b * b;
        double rad = 1.0 + k1 * rho + k2 * rho * rho + k3 * rho * rho * rho;
        double drad = k1 + 2.0 * k2 * rho + 3.0 * k3 * rho * rho;  /* d rad / d rho */
        /* D = d(xd, yd) / d(a, b) */
        double d00 = rad + a * drad * 2.0 * a + 2.0 * p1 * b + p2 * (2.0 * a + 4.0 * a);
        double d01 = a * drad * 2.0 * b + 2.0 * p1 * a + p2 * 2.0 * b;
        double d10 = b * drad * 2.0 * a + p1 * 2.0 * a + 2.0 * p2 * b;
        double d11 = rad + b * drad * 2.0 * b + p1 * (2.0 * b + 4.0 * b) + 2.0 * p2 * a;
        /* d(a, b) / dX = [[1/z, 0, -x/z^2], [0, 1/z, -y/z^2]] */
        double iz = 1.0 / z, ax = -a * iz, bx = -b * iz;
        Ju[0] = fx * d00 * iz; Ju[1] = fx * d01 * iz; Ju[2] = fx * (d00 * ax + d01 * bx);
        Jv[0] = fy * d10 * iz; Jv[1] = fy * d11 * iz; Jv[2] = fy * (d10 * ax + d11 * bx);
        break;
    }
    case ORC_KB: {
        double r2 = x * x + y * y, r = sqrt(r2);
        double th = atan2(r, z);
        double t2 = th * th;
        double thd = th * (1.0 + t2 * (m->p[4] + t2 * (m->p[5] + t2 * (m->p[6] + t2 * m->p[7]))));
        double dthd = 1.0 + t2 * (3.0 * m->p[4] + t2 * (5.0 * m->p[5] + t2 * (7.0 * m->p[6] + t2 * 9.0 * m->p[7])));
        if (r < EPS) {  /* on the axis: u - cx -> fx * x / z */
            Ju[0] = fx / z; Jv[1] = fy / z;
            break;
        }
        double rho2 = r2 + z * z;
        double thx = x * z / (r * rho2), thy = y * z / (r * rho2), thz = -r / rho2;
        double xr = x / r, yr = y / r, ir = 1.0 / r;
        /* u - cx = fx * thd * x / r */
        Ju[0] = fx * (dthd * thx * xr + thd * (ir - x * x / (r2 * r)));
        Ju[1] = fx * (dthd * thy * xr - thd * x * y / (r2 * r));
        Ju[2] = fx * dthd * thz * xr;
        Jv[0] = fy * (dthd * thx * yr - thd * x * y / (r2 * r));
        Jv[1] = fy * (dthd * thy * yr + thd * (ir - y * y / (r2 * r)));
        Jv[2] = fy * dthd * thz * yr;
        break;
    }
    case ORC_UCM: case ORC_EUCM: case ORC_DS: {
        /* u - cx = fx * x / den:  grad u = fx * (e_x / den - x * grad den / den^2) */
        const double alpha = m->p[4];
        double den, gd[3];
        if (m->model == ORC_UCM) {
            double d = sqrt(x * x + y * y + z * z);
            den = alpha * d + (1.0 - alpha) * z;
            gd[0] = alpha * x / d; gd[1] = alpha * y / d; gd[2] = alpha * z / d + (1.0 - alpha);
        } else if (m->model == ORC_EUCM) {
            const double beta = m->p[5];
            double d = sqrt(beta * (x * x + y * y) + z * z);
            den = alpha * d + (1.0 - alpha) * z;
            gd[0] = alpha * beta * x / d; gd[1] = alpha * beta * y / d; gd[2] = alpha * z / d + (1.0 - alpha);
        } else {
            const double xi = m->p[5];
            double rr = x * x + y * y;
            double d1 = sqrt(rr + z * z);
            double g = xi * d1 + z;
            double d2 = sqrt(rr + g * g);
            den = alpha * d2 + (1.0 - alpha) * g;
            double gg[3] = {xi * x / d1, xi * y / d1, xi * z / d1 + 1.0};
            double gd2[3] = {(x + g * gg[0]) / d2, (y + g * gg[1]) / d2, g * gg[2] / d2};
            for (int k = 0; k < 3; ++k) gd[k] = alpha * gd2[k] + (1.0 - alpha) * gg[k];
        }
        double id = 1.0 / den, id2 = id * id;
        for (int k = 0; k < 3; ++k) {
            Ju[k] = fx * ((k == 0 ? id : 0.0) - x * gd[k] * id2);
            Jv[k] = fy * ((k == 1 ? id : 0.0) - y * gd[k] * id2);
        }
        break;
    }
    case ORC_FOV: {
        const double w = m->p[4];
        double t = tan(w / 2.0);
        double r2 = x * x + y * y;
        if (r2 < SQRT_EPS) {  /* the reference's near-axis branch (fov.rs:299-301): mx = x * (2t/w), a constant factor, no z */
            double rd = 2.0 * t / w;
            Ju[0] = fx * rd; Jv[1] = fy * rd;   /* the derivative of what project() evaluates there */
            break;
        }
        double r = sqrt(r2);
        double s = 2.0 * t * r;
        double a = atan2(s, z);
        double q = s * s + z * z;
        double rd = a / (r * w);
        /* grad a = (2t z / q) grad r + (0, 0, -s / q);  grad r = (x/r, y/r, 0) */
        double ar = 2.0 * t * z / q;              /* da/dr */
        double rdr = (ar - a / r) / (r * w);      /* d rd / d r */
        double rdz = (-s / q) / (r * w);          /* d rd / d z */
        double gx = rdr * x / r, gy = rdr * y / r;
        Ju[0] = fx * (rd + x * gx); Ju[1] = fx * x * gy; Ju[2] = fx * x * rdz;
        Jv[0] = fy * y * gx; Jv[1] = fy * (rd + y * gy); Jv[2] = fy * y * rdz;
        break;
    }
    default: return -1;
    }
    return ORC_OK;
}
