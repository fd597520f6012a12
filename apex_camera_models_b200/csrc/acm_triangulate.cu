// Triangulation of matched pixels of a calibrated camera pair (beyond the reference; composed of its functions): the two
// IEEE unprojects, the closest-approach midpoint in the first camera's frame, optionally refined by a damped Gauss-Newton
// (Levenberg-Marquardt) solve on the four pixel residuals with the analytic 2x3 point Jacobians.  The semantics, status
// order and constants are those of include/acm.h (acm_triangulate); tests/triangulate_oracle.c states the same steps on
// the CPU.
//
// Compiled with -fmad=false like acm_exact.cu: unproject<true> / project are bit-identical to the oracle's only without
// contraction, and the midpoint keeps the same separately rounded operations, so the midpoint points of the arithmetic-only
// models (Pinhole, RadTan, UCM, EUCM, Double Sphere) are bit-identical to the oracle's.
//
// One streaming kernel over independent pairs, one template instantiation per (first, second) model pair (49).  The
// rotation, translation and iteration cap are uniform kernel arguments.  Inputs and outputs are addressed with a stride so
// that the device form (SoA point buffers, stride 1) and the host form (AoS staging, strides 2 and 3) run the same kernel.
#include <cmath>
#include <cstring>

#include "acm_models.cuh"
#include "acm_pointjac.cuh"

struct TriRig {
    double R[9];  // row-major, x_cam2 = R x_cam1 + t
    double t[3];
};

struct TriIO {
    const double *u1, *v1, *u2, *v2;
    size_t in_stride;    // doubles between consecutive pairs of each input component
    double *x, *y, *z;
    size_t xyz_stride;
    double *e1, *e2;     // e1 == nullptr: no errors
    size_t err_stride;
    uint8_t* st;         // nullptr: no status
};

template <int M1, int M2> struct TriPair {
    const CamParams& ca;
    const CamParams& cb;
    const TriRig& g;
    double u1, v1, u2, v2;

    __device__ __forceinline__ void to_second(const double* X, double* Y) const { acm_rigid_apply(g.R, g.t, X, Y); }
    // the four pixel residuals at X; false when X does not project (geometric validity) into both cameras
    __device__ __forceinline__ bool residuals(const double* X, double* r, double& cost) const {
        double pu, pv, qu, qv, Y[3];
        if (CamModel<M1>::template project<false>(ca, X[0], X[1], X[2], pu, pv) != ACM_POINT_OK) return false;
        to_second(X, Y);
        if (CamModel<M2>::template project<false>(cb, Y[0], Y[1], Y[2], qu, qv) != ACM_POINT_OK) return false;
        r[0] = pu - u1; r[1] = pv - v1; r[2] = qu - u2; r[3] = qv - v2;
        cost = ((r[0] * r[0] + r[1] * r[1]) + r[2] * r[2]) + r[3] * r[3];
        return true;
    }
};

// (H + lambda diag(H)) d = -g by a 3x3 Cholesky factorisation; H packed as H00 H01 H02 H11 H12 H22.  false when a pivot is
// not positive (the trial is then rejected).
__device__ __forceinline__ bool tri_damped_solve(const double* H, const double* gr, double lambda, double* d) {
    const double a00 = H[0] + lambda * H[0], a11 = H[3] + lambda * H[3], a22 = H[5] + lambda * H[5];
    if (!(a00 > 0.0)) return false;
    const double l00 = sqrt(a00);
    const double l10 = H[1] / l00, l20 = H[2] / l00;
    const double p11 = a11 - l10 * l10;
    if (!(p11 > 0.0)) return false;
    const double l11 = sqrt(p11);
    const double l21 = (H[4] - l20 * l10) / l11;
    const double p22 = (a22 - l20 * l20) - l21 * l21;
    if (!(p22 > 0.0)) return false;
    const double l22 = sqrt(p22);
    const double y0 = -gr[0] / l00;
    const double y1 = (-gr[1] - l10 * y0) / l11;
    const double y2 = ((-gr[2] - l20 * y0) - l21 * y1) / l22;
    d[2] = y2 / l22;
    d[1] = (y1 - l21 * d[2]) / l11;
    d[0] = ((y0 - l10 * d[1]) - l20 * d[2]) / l00;
    return true;
}

template <int M1, int M2>
__device__ __forceinline__ int tri_one(const TriPair<M1, M2>& P, const LinParams& la, const LinParams& lb, const double* c2, int max_iterations,
                                       double* X, double& e1, double& e2) {
    const TriRig& g = P.g;
    double d1[3], d2[3];
    if (CamModel<M1>::template unproject<true>(P.ca, P.u1, P.v1, d1[0], d1[1], d1[2]) != ACM_POINT_OK) return ACM_TRI_UNPROJECT_FIRST;
    if (CamModel<M2>::template unproject<true>(P.cb, P.u2, P.v2, d2[0], d2[1], d2[2]) != ACM_POINT_OK) return ACM_TRI_UNPROJECT_SECOND;
    double e[3];  // d2' = R^T d2
    acm_rot_t(g.R, d2, e);
    const double b = (d1[0] * e[0] + d1[1] * e[1]) + d1[2] * e[2];
    const double p = (d1[0] * c2[0] + d1[1] * c2[1]) + d1[2] * c2[2];
    const double q = (e[0] * c2[0] + e[1] * c2[1]) + e[2] * c2[2];
    const double den = 1.0 - b * b;
    if (den <= ACM_TRI_PARALLEL_EPS) return ACM_TRI_PARALLEL;
    const double s1 = (p - b * q) / den, s2 = (b * p - q) / den;
    if (s1 <= 0.0 || s2 <= 0.0) return ACM_TRI_BEHIND;
#pragma unroll
    for (int k = 0; k < 3; ++k) X[k] = 0.5 * ((s1 * d1[k] + c2[k]) + s2 * e[k]);
    double r[4], cost;
    if (!P.residuals(X, r, cost)) return ACM_TRI_PROJECT;

    double lambda = ACM_TRI_LAMBDA0;
    double H[6], gr[3];
    bool fresh = false;  // H, gr belong to the current X
#pragma unroll 1
    for (int it = 0; it < max_iterations; ++it) {
        if (!fresh) {
            double J[4][3], jb[6], Y[3];
            PointJac<M1>::eval(la, X[0], X[1], X[2], J[0], J[1]);
            P.to_second(X, Y);
            PointJac<M2>::eval(lb, Y[0], Y[1], Y[2], jb, jb + 3);
#pragma unroll
            for (int row = 0; row < 2; ++row)
#pragma unroll
                for (int k = 0; k < 3; ++k)
                    J[2 + row][k] = (jb[3 * row] * g.R[k] + jb[3 * row + 1] * g.R[3 + k]) + jb[3 * row + 2] * g.R[6 + k];
            int h = 0;
#pragma unroll
            for (int a = 0; a < 3; ++a) {
                gr[a] = ((J[0][a] * r[0] + J[1][a] * r[1]) + J[2][a] * r[2]) + J[3][a] * r[3];
#pragma unroll
                for (int c = a; c < 3; ++c) H[h++] = ((J[0][a] * J[0][c] + J[1][a] * J[1][c]) + J[2][a] * J[2][c]) + J[3][a] * J[3][c];
            }
            fresh = true;
        }
        double d[3], Xt[3], rt[4], ct;
        bool accept = tri_damped_solve(H, gr, lambda, d);
        if (accept) {
#pragma unroll
            for (int k = 0; k < 3; ++k) Xt[k] = X[k] + d[k];
            accept = P.residuals(Xt, rt, ct) && ct < cost;
        }
        if (!accept) { lambda = lambda * ACM_TRI_LAMBDA_FACTOR; continue; }
#pragma unroll
        for (int k = 0; k < 3; ++k) X[k] = Xt[k];
#pragma unroll
        for (int k = 0; k < 4; ++k) r[k] = rt[k];
        cost = ct;
        lambda = lambda / ACM_TRI_LAMBDA_FACTOR;
        fresh = false;
        const double dmax = fmax(fabs(d[0]), fmax(fabs(d[1]), fabs(d[2])));
        const double xmax = fmax(fabs(X[0]), fmax(fabs(X[1]), fabs(X[2])));
        if (dmax <= ACM_TRI_STEP_TOL * fmax(1.0, xmax)) break;
    }
    e1 = sqrt(r[0] * r[0] + r[1] * r[1]);
    e2 = sqrt(r[2] * r[2] + r[3] * r[3]);
    return ACM_TRI_OK;
}

template <int M1, int M2>
__global__ void __launch_bounds__(256) triangulate_kernel(const __grid_constant__ CamParams ca, const __grid_constant__ CamParams cb,
                                                          const __grid_constant__ LinParams la, const __grid_constant__ LinParams lb,
                                                          const __grid_constant__ TriRig g, const __grid_constant__ TriIO io, int max_iterations,
                                                          size_t n) {
    double c2[3];  // c2 = -R^T t, the second camera's centre in the first camera's frame (same order as d2')
    acm_rot_t(g.R, g.t, c2);
#pragma unroll
    for (int k = 0; k < 3; ++k) c2[k] = -c2[k];
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const size_t j = i * io.in_stride;
        const TriPair<M1, M2> P{ca, cb, g, __ldcs(io.u1 + j), __ldcs(io.v1 + j), __ldcs(io.u2 + j), __ldcs(io.v2 + j)};
        double X[3], e1, e2;
        const int st = tri_one<M1, M2>(P, la, lb, c2, max_iterations, X, e1, e2);
        if (st != ACM_TRI_OK) X[0] = X[1] = X[2] = e1 = e2 = acm_nan();
        const size_t o = i * io.xyz_stride;
        __stcs(io.x + o, X[0]); __stcs(io.y + o, X[1]); __stcs(io.z + o, X[2]);
        if (io.e1) { __stcs(io.e1 + i * io.err_stride, e1); __stcs(io.e2 + i * io.err_stride, e2); }
        if (io.st) __stcs(io.st + i, (unsigned char)st);
    }
}

template <int M1>
static int32_t launch_triangulate(acm_ctx* ctx, const CamParams& ca, const CamParams& cb, const LinParams& la, const LinParams& lb,
                                  const TriRig& g, const TriIO& io, int max_iterations, size_t n) {
    const int grid = grid_for(ctx, n, 256, 8);
    ACM_DISPATCH_MODEL(cb.model, (triangulate_kernel<M1, M><<<grid, 256, 0, ctx->stream>>>(ca, cb, la, lb, g, io, max_iterations, n)))
    ACM_CHECK_LAUNCH(ctx);
    return ACM_OK;
}

// argument checks shared by both forms; fills the rig
static int32_t check_pair(acm_ctx* ctx, const acm_camera* first, const acm_camera* second, const double* R, const double* t, int32_t max_iterations,
                          TriRig* g) {
    ACM_REQUIRE(ctx, first && second, "triangulate: null camera");
    ACM_REQUIRE(ctx, max_iterations >= 0, "triangulate: max_iterations must be >= 0");
    int32_t rc = acm_check_rotation(ctx, R, "triangulate");
    if (rc) return rc;
    ACM_REQUIRE(ctx, t, "triangulate: null translation");
    ACM_REQUIRE(ctx, std::isfinite(t[0]) && std::isfinite(t[1]) && std::isfinite(t[2]), "triangulate: translation has a non-finite entry");
    ACM_REQUIRE(ctx, !(t[0] == 0.0 && t[1] == 0.0 && t[2] == 0.0), "triangulate: translation is zero (no baseline: every pair is parallel)");
    std::memcpy(g->R, R, sizeof(g->R));
    std::memcpy(g->t, t, sizeof(g->t));
    return ACM_OK;
}

static int32_t run(acm_ctx* ctx, const acm_camera* first, const acm_camera* second, const TriRig& g, const TriIO& io, int32_t max_iterations,
                   size_t n) {
    CamParams ca, cb;
    int32_t rc = acm_make_cam_params(ctx, first, &ca);
    if (!rc) rc = acm_make_cam_params(ctx, second, &cb);
    if (rc) return rc;
    if (n == 0) return ACM_OK;
    LinParams la, lb;
    make_lin_params(first, &la);
    make_lin_params(second, &lb);
    ACM_DISPATCH_MODEL(ca.model, return launch_triangulate<M>(ctx, ca, cb, la, lb, g, io, max_iterations, n))
    return ACM_OK;
}

extern "C" int32_t acm_triangulate(acm_ctx* ctx, const acm_camera* first, const acm_camera* second, const double R[9], const double t[3],
                                   const acm_points* uv1, const acm_points* uv2, int32_t max_iterations, acm_points* xyz, double* d_err,
                                   uint8_t* d_status) {
    ACM_ENTER(ctx);
    TriRig g;
    int32_t rc = check_pair(ctx, first, second, R, t, max_iterations, &g);
    if (rc) return rc;
    ACM_REQUIRE(ctx, uv1 && uv2 && xyz, "triangulate: null point buffer");
    ACM_REQUIRE(ctx, uv1->dim == 2 && uv2->dim == 2 && xyz->dim == 3, "triangulate: uv1 / uv2 must have dim 2 and xyz dim 3");
    ACM_REQUIRE(ctx, uv1->n == uv2->n && xyz->n == uv1->n, "triangulate: uv1, uv2 and xyz must hold the same number of points");
    ACM_REQUIRE(ctx, uv1->dtype == ACM_F64 && uv2->dtype == ACM_F64 && xyz->dtype == ACM_F64, "triangulate: f64 point buffers required");
    const size_t n = uv1->n;
    TriIO io{comp<double>(uv1, 0), comp<double>(uv1, 1), comp<double>(uv2, 0), comp<double>(uv2, 1), 1,
             comp<double>(xyz, 0), comp<double>(xyz, 1), comp<double>(xyz, 2), 1,
             d_err, d_err ? d_err + n : nullptr, 1, d_status};
    return run(ctx, first, second, g, io, max_iterations, n);
}

// Host form: the AoS buffers are copied as they are into the context's scratch arena and the kernel reads and writes them
// with AoS strides, so a call is copies and ONE kernel, and its bytes equal the device form's.
extern "C" int32_t acm_triangulate_host(acm_ctx* ctx, const acm_camera* first, const acm_camera* second, const double R[9], const double t[3],
                                        const double* uv1_aos, const double* uv2_aos, size_t n, int32_t max_iterations, double* xyz_aos,
                                        double* err, uint8_t* status) {
    ACM_ENTER(ctx);
    TriRig g;
    int32_t rc = check_pair(ctx, first, second, R, t, max_iterations, &g);
    if (rc) return rc;
    ACM_REQUIRE(ctx, n == 0 || (uv1_aos && uv2_aos && xyz_aos), "triangulate: null point buffer");
    // scratch layout in doubles: uv1 [0, 2n), uv2 [2n, 4n), xyz [4n, 7n), err [7n, 9n), then n status bytes
    const size_t bytes = 9 * n * sizeof(double) + n;
    if (n) {
        rc = acm_ensure_scratch(ctx, bytes);
        if (rc) return rc;
    }
    double* d = static_cast<double*>(ctx->d_scratch);
    uint8_t* d_st = reinterpret_cast<uint8_t*>(d + 9 * n);
    if (n) {
        ACM_CUDA(ctx, cudaMemcpyAsync(d, uv1_aos, 2 * n * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
        ACM_CUDA(ctx, cudaMemcpyAsync(d + 2 * n, uv2_aos, 2 * n * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    }
    TriIO io{d, d + 1, d + 2 * n, d + 2 * n + 1, 2, d + 4 * n, d + 4 * n + 1, d + 4 * n + 2, 3,
             err ? d + 7 * n : nullptr, d + 7 * n + 1, 2, status ? d_st : nullptr};
    rc = run(ctx, first, second, g, io, max_iterations, n);
    if (rc || n == 0) return rc;
    ACM_CUDA(ctx, cudaMemcpyAsync(xyz_aos, d + 4 * n, 3 * n * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    if (err) ACM_CUDA(ctx, cudaMemcpyAsync(err, d + 7 * n, 2 * n * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    if (status) ACM_CUDA(ctx, cudaMemcpyAsync(status, d_st, n, cudaMemcpyDeviceToHost, ctx->stream));
    ACM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return ACM_OK;
}
