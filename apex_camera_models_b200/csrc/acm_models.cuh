// Device math of the seven camera models: project / unproject with the reference's validity
// tests, evaluated in IEEE binary64 in the reference's operation order.  The translation
// unit that includes this header for the project / unproject / undistort kernels is compiled
// with -fmad=false: Rust never contracts a*b+c, and the status masks (and remap indices) must
// be bit-exact.  Per-model line references are to /root/reference/src/camera/<model>.rs.
#pragma once
#include "acm_internal.cuh"
#include "acm_math.cuh"

#define ACM_EPS 2.220446049250313e-16        // f64::EPSILON
#define ACM_SQRT_EPS 1.4901161193847656e-08  // f64::EPSILON.sqrt() == 2^-26
#define ACM_PRECISION 1e-3

__device__ __forceinline__ double acm_nan() { return __longlong_as_double(0x7ff8000000000000LL); }

__device__ __forceinline__ bool acm_outside(const CamParams& c, double u, double v) {
    // mod.rs:157-166, :194-206 -- half-open [0,W) x [0,H)
    return u < 0.0 || u >= c.W || v < 0.0 || v >= c.H;
}

// Rigid transforms with R row-major, every operation separately rounded in the including unit (-fmad=false there):
//   acm_rigid_apply:  Y = R X + t,   Y[i] = ((R[i][0] X0 + R[i][1] X1) + R[i][2] X2) + t[i]
//   acm_rot_t:        Y = R^T X,     Y[k] = (R[0][k] X0 + R[1][k] X1) + R[2][k] X2
__device__ __forceinline__ void acm_rigid_apply(const double* R, const double* t, const double* X, double* Y) {
#pragma unroll
    for (int i = 0; i < 3; ++i) Y[i] = ((R[3 * i] * X[0] + R[3 * i + 1] * X[1]) + R[3 * i + 2] * X[2]) + t[i];
}
__device__ __forceinline__ void acm_rot_t(const double* R, const double* X, double* Y) {
#pragma unroll
    for (int k = 0; k < 3; ++k) Y[k] = (R[k] * X[0] + R[3 + k] * X[1]) + R[6 + k] * X[2];
}

// The nearest-pixel rule of undistort.rs:79-90: rx = round(sx), ry = round(sy) (half away from zero); true when the pixel lies
// inside [0,W) x [0,H) (NaN fails).  `as i32` saturates in the reference; anything outside [0,W) fails the guard either way.
__device__ __forceinline__ bool acm_nearest_pixel(double sx, double sy, int W, int H, double& rx, double& ry) {
    rx = round(sx); ry = round(sy);
    return rx >= 0.0 && rx < (double)W && ry >= 0.0 && ry < (double)H;
}

// nalgebra normalize(): n = sqrt((x*x + y*y) + z*z), each component divided by n
__device__ __forceinline__ void acm_normalize_ieee(double x, double y, double z, double& ox, double& oy, double& oz) {
    double n = sqrt(x * x + y * y + z * z);
    ox = x / n; oy = y / n; oz = z / n;
}

// --- exact decisions, fast tails -----------------------------------------------------------
// unproject has two kinds of arithmetic.  Everything a validity test (or a branch between two
// formulas) depends on is evaluated exactly as the reference does -- separately rounded IEEE
// operations in the reference's order -- so the status bytes are bit-exact.  Three rewrites there
// are bit-IDENTICAL, not approximations: (u - cx) / fx through acm_div_by() with the host's RN(1/fx);
// RadTan's four divisions by one determinant through ONE IEEE reciprocal + acm_div_by(); and
// `sqrt(s) < t` / `sqrt(s) > t` as `s < S` / `s > S'` with the exact double thresholds of the
// correctly rounded sqrt.  What follows the last test only has to meet the 1e-9 relative bar of the
// values; there the IEEE divisions and square roots (three divisions in normalize() alone) become a
// MUFU-seeded reciprocal / rsqrt (<= 2 ulp, acm_math.cuh).  unproject<true> keeps IEEE tails: sample_points uses it, so the
// correspondences handed to the solver stay bit-identical to the reference's for the arithmetic-only models.
template <bool IEEE>
__device__ __forceinline__ void acm_normalize(double x, double y, double z, double& ox, double& oy, double& oz) {
    if (IEEE) { acm_normalize_ieee(x, y, z, ox, oy, oz); return; }
    const double inv = acm_rsqrt(__fma_rn(z, z, __fma_rn(y, y, __dmul_rn(x, x))));
    ox = x * inv; oy = y * inv; oz = z * inv;
}
template <bool IEEE> __device__ __forceinline__ double acm_tail_div(double a, double b) { return IEEE ? a / b : a * acm_rcp(b); }
template <bool IEEE> __device__ __forceinline__ double acm_tail_sqrt(double a) {
    if (IEEE) return sqrt(a);
    double inv;
    return acm_sqrt_inv(a, inv);
}

// (u - cx) / fx, (v - cy) / fy: bit-identical to the IEEE division (see acm_div_by)
__device__ __forceinline__ double acm_mx(const CamParams& c, double u) {
    const double a = u - c.cx;
    return c.fast_div ? acm_div_by(a, c.fx, c.ifx) : a / c.fx;
}
__device__ __forceinline__ double acm_my(const CamParams& c, double v) {
    const double a = v - c.cy;
    return c.fast_div ? acm_div_by(a, c.fy, c.ify) : a / c.fy;
}
#define ACM_SQRT_LT_1EM6 0x1.19799812dea10p-40  // sqrt(s) <  1e-6   <=>  s <  this   (correctly rounded sqrt)
#define ACM_SQRT_GT_1EM6 0x1.19799812dea11p-40  // sqrt(s) >  1e-6   <=>  s >  this
#define ACM_SQRT_GT_2M26 0x1.0000000000001p-52  // sqrt(s) >  2^-26  <=>  s >  this

template <int M> struct CamModel;

// ---- Pinhole (pinhole.rs:165-182, :228-246) ----------------------------------------------
template <> struct CamModel<ACM_MODEL_PINHOLE> {
    template <bool BOUNDS, bool FAST = false>
    static __device__ __forceinline__ int project(const CamParams& c, double x, double y, double z, double& u, double& v) {
        if (z < ACM_SQRT_EPS) return ACM_POINT_AT_CAMERA_CENTER;
        u = c.fx * x / z + c.cx;
        v = c.fy * y / z + c.cy;
        if (BOUNDS && acm_outside(c, u, v)) return ACM_PROJECTION_OUTSIDE_IMAGE;
        return ACM_POINT_OK;
    }
    template <bool IEEE = false>
    static __device__ __forceinline__ int unproject(const CamParams& c, double u, double v, double& rx, double& ry, double& rz) {
        if (acm_outside(c, u, v)) return ACM_POINT_IS_OUTSIDE_IMAGE;
        double mx = acm_mx(c, u), my = acm_my(c, v);
        double r2 = mx * mx + my * my;
        double ninv = 1.0 / sqrt(1.0 + r2);   // IEEE: the kernel is HBM-bound either way, and the values stay bit-identical
        rx = mx * ninv; ry = my * ninv; rz = ninv;
        return ACM_POINT_OK;
    }
};

// ---- RadTan (rad_tan.rs:302-348, :401-524), d = [k1,k2,p1,p2,k3] ---------------------------
template <> struct CamModel<ACM_MODEL_RADTAN> {
    template <bool BOUNDS, bool FAST = false>
    static __device__ __forceinline__ int project(const CamParams& c, double x, double y, double z, double& u, double& v) {
        if (z < ACM_SQRT_EPS) return ACM_POINT_AT_CAMERA_CENTER;
        const double k1 = c.d[0], k2 = c.d[1], p1 = c.d[2], p2 = c.d[3], k3 = c.d[4];
        double xp = x / z, yp = y / z;
        double r2 = xp * xp + yp * yp;
        double r4 = r2 * r2;
        double r6 = r4 * r2;
        double rad = 1.0 + k1 * r2 + k2 * r4 + k3 * r6;
        double xd = xp * rad + 2.0 * p1 * xp * yp + p2 * (r2 + 2.0 * xp * xp);
        double yd = yp * rad + p1 * (r2 + 2.0 * yp * yp) + 2.0 * p2 * xp * yp;
        u = c.fx * xd + c.cx;
        v = c.fy * yd + c.cy;
        if (BOUNDS && acm_outside(c, u, v)) return ACM_PROJECTION_OUTSIDE_IMAGE;
        return ACM_POINT_OK;
    }
    // Contracted form of the Newton loop below (rad_tan.rs:440-515) for cameras that pass the host-side gate
    // (CamParams::fast_newton, acm_make_cam_params): Horner / FMA evaluation of the distortion and of its 2x2 Jacobian
    // (the terms shared, ~50 FP64 instructions per step instead of ~106 separately rounded ones) and one MUFU-seeded
    // reciprocal of the determinant instead of an IEEE division + four quotients.
    // The reference returns the iterate at which one of its two tests fires -- `error.norm() < 1e-6` before a step,
    // `delta.norm() < 1e-6` after it -- so that iterate (typically two steps from the start, ~1e-9 from the root) IS the
    // result, and a different stopping decision would move it by up to 1e-6.  The contracted iterates track the IEEE
    // ones to a few 1e-15 (a Newton step contracts perturbations), which moves the two squared norms by <= ~1e-7
    // relative near their threshold (the error is a difference of O(1) quantities, |e| ~ 1e-6 there).  Every decision
    // is therefore taken with a guard band of 1e-5 relative around 1e-12; a value inside the band, a determinant that
    // is not clearly non-zero, a non-finite intermediate or the 100th iteration all return -1 ("ambiguous") and the
    // caller redoes the point with the IEEE loop.  ~2e-5 of the decisions land in a band; a warp with such a point pays
    // the IEEE loop once.  Status bytes stay bit-exact, rays agree with the reference's iterate to ~1e-14.
    // (Iterating the two points of a packet in ONE loop -- two independent chains per trip -- measured SLOWER, 2146 vs
    // 2628 GB/s on the same box: the selects that freeze a finished point cost more than the second chain hides.)
    static __device__ __forceinline__ int unproject_newton_fast(const CamParams& c, double tx, double ty, double& px, double& py) {
        const double k1 = c.d[0], k2 = c.d[1], p1 = c.d[2], p2 = c.d[3], k3 = c.d[4];
        const double k2x2 = k2 + k2, k3x3 = 3.0 * k3, p1x2 = p1 + p1, p2x2 = p2 + p2, p1x6 = 6.0 * p1, p2x6 = 6.0 * p2;  // kernel-invariant
        const double T = 1e-12, BAND = 1e-17;   // threshold of the squared norms, half-width of the guard band
        px = tx; py = ty;
#pragma unroll 1
        for (int it = 0; it < 100; ++it) {
            const double x = px, y = py;
            const double r2 = __fma_rn(x, x, __dmul_rn(y, y));
            const double rad = __fma_rn(r2, __fma_rn(r2, __fma_rn(r2, k3, k2), k1), 1.0);
            const double xy = __dmul_rn(x, y), x2 = __dadd_rn(x, x), y2 = __dadd_rn(y, y);
            const double ex = __fma_rn(x, rad, __fma_rn(p1x2, xy, __fma_rn(p2, __fma_rn(x2, x, r2), -tx)));
            const double ey = __fma_rn(y, rad, __fma_rn(p1, __fma_rn(y2, y, r2), __fma_rn(p2x2, xy, -ty)));
            const double e2 = __fma_rn(ex, ex, __dmul_rn(ey, ey));
            if (!(fabs(e2 - T) > BAND)) return -1;      // inside the band, or NaN
            if (e2 < T) return ACM_POINT_OK;             // error.norm() < 1e-6
            const double common = __fma_rn(r2, __fma_rn(r2, k3x3, k2x2), k1);
            const double dx_ = __dmul_rn(common, x2), dy_ = __dmul_rn(common, y2);   // d(rad)/dx, d(rad)/dy
            const double cross = __fma_rn(p1x2, x, __dmul_rn(p2x2, y));
            const double j00 = __fma_rn(x, dx_, __fma_rn(p1x2, y, __fma_rn(p2x6, x, rad)));
            const double j01 = __fma_rn(x, dy_, cross);
            const double j10 = __fma_rn(y, dx_, cross);
            const double j11 = __fma_rn(y, dy_, __fma_rn(p1x6, y, __fma_rn(p2x2, x, rad)));
            const double a = __dmul_rn(j00, j11), b = __dmul_rn(j10, j01);
            const double det = __dsub_rn(a, b);
            if (!(fabs(det) > 1e-9 * (fabs(a) + fabs(b)))) return -1;   // det == 0.0 of the reference cannot be decided here (or NaN)
            const double idet = acm_rcp(det);
            const double dx = __dmul_rn(__fma_rn(j11, ex, -__dmul_rn(j01, ey)), idet);
            const double dy = __dmul_rn(__fma_rn(j00, ey, -__dmul_rn(j10, ex)), idet);
            px = __dsub_rn(px, dx); py = __dsub_rn(py, dy);
            const double d2 = __fma_rn(dx, dx, __dmul_rn(dy, dy));
            if (!(fabs(d2 - T) > BAND)) return -1;
            if (d2 < T) return ACM_POINT_OK;             // delta.norm() < 1e-6
        }
        return -1;   // 100 steps without a stop: let the IEEE loop give the verdict
    }

    template <bool IEEE = false>
    static __device__ int unproject(const CamParams& c, double u, double v, double& rx, double& ry, double& rz) {
        if (acm_outside(c, u, v)) return ACM_POINT_IS_OUTSIDE_IMAGE;
        const double k1 = c.d[0], k2 = c.d[1], p1 = c.d[2], p2 = c.d[3], k3 = c.d[4];
        const double tx = acm_mx(c, u), ty = acm_my(c, v);
        double px = tx, py = ty;
        if (!IEEE && c.fast_newton) {
            if (unproject_newton_fast(c, tx, ty, px, py) == ACM_POINT_OK) {
                acm_normalize<false>(px, py, 1.0, rx, ry, rz);
                return ACM_POINT_OK;
            }
            px = tx; py = ty;   // ambiguous: the reference's own arithmetic decides
        }
        for (int it = 0; it < 100; ++it) {
            double x = px, y = py;
            double r2 = x * x + y * y;
            double r4 = r2 * r2;
            double r6 = r4 * r2;
            double rad = 1.0 + k1 * r2 + k2 * r4 + k3 * r6;
            double xe = x * rad + 2.0 * p1 * x * y + p2 * (r2 + 2.0 * x * x);
            double ye = y * rad + p1 * (r2 + 2.0 * y * y) + 2.0 * p2 * x * y;
            double ex = xe - tx, ey = ye - ty;
            if (ex * ex + ey * ey < ACM_SQRT_LT_1EM6) break;   // error.norm() < 1e-6, rad_tan.rs:460
            double dr_dx = 2.0 * x, dr_dy = 2.0 * y;
            double common = k1 + 2.0 * k2 * r2 + 3.0 * k3 * r4;
            double drad_dx = common * dr_dx, drad_dy = common * dr_dy;
            double j00 = rad + x * drad_dx + 2.0 * p1 * y + p2 * (dr_dx + 4.0 * x);
            double j01 = x * drad_dy + 2.0 * p1 * x + p2 * (dr_dy);
            double j10 = y * drad_dx + p1 * (dr_dx) + 2.0 * p2 * y;
            double j11 = rad + y * drad_dy + p1 * (dr_dy + 4.0 * y) + 2.0 * p2 * x;
            double det = j00 * j11 - j10 * j01;   // nalgebra Matrix2::try_inverse
            if (det == 0.0) return ACM_POINT_NUMERICAL_ERROR;
            double i00, i01, i10, i11;
            if (acm_exp_ok(det)) {   // one IEEE reciprocal, four bit-identical quotients
                const double idet = 1.0 / det;
                i00 = acm_div_by(j11, det, idet); i01 = acm_div_by(-j01, det, idet);
                i10 = acm_div_by(-j10, det, idet); i11 = acm_div_by(j00, det, idet);
            } else { i00 = j11 / det; i01 = -j01 / det; i10 = -j10 / det; i11 = j00 / det; }
            double dx = i00 * ex + i01 * ey;
            double dy = i10 * ex + i11 * ey;
            px -= dx; py -= dy;
            if (dx * dx + dy * dy < ACM_SQRT_LT_1EM6) break;   // delta.norm() < 1e-6, rad_tan.rs:500
            if (it == 99) return ACM_POINT_NUMERICAL_ERROR;
        }
        acm_normalize<IEEE>(px, py, 1.0, rx, ry, rz);
        return ACM_POINT_OK;
    }
};

// ---- Kannala-Brandt (kannala_brandt.rs:340-394, :445-562), d = [k1..k4] ---------------------
template <> struct CamModel<ACM_MODEL_KANNALA_BRANDT> {
    template <bool BOUNDS, bool FAST = false>
    static __device__ __forceinline__ int project(const CamParams& c, double x, double y, double z, double& u, double& v) {
        if (z < 0.0) return ACM_POINT_IS_OUTSIDE_IMAGE;
        else if (z < ACM_EPS) return ACM_POINT_AT_CAMERA_CENTER;
        // FAST (batch project / round trip only; undistort and the statistics keep the IEEE form): nothing after the two
        // z tests is a status decision, so sqrt + the two divisions by r become one coupled sqrt / rsqrt (<= 2 ulp);
        // the r < EPS branch is taken exactly on r2 (sqrt(s) < 2^-52  <=>  s < 2^-104 for the correctly rounded root)
        const double r2 = x * x + y * y;
        double ir = 0.0;
        const double r = FAST ? acm_sqrt_inv(r2, ir) : sqrt(r2);
        double th = acm_atan2_q1(r, z);  // r >= 0, z >= EPS: first quadrant (<= 1.5 ulp, see acm_math.cuh)
        double t2 = th * th;
        double t3 = t2 * th;
        double t5 = t3 * t2;
        double t7 = t5 * t2;
        double t9 = t7 * t2;
        double thd = th + c.d[0] * t3 + c.d[1] * t5 + c.d[2] * t7 + c.d[3] * t9;
        double xr, yr;
        if (FAST) { const bool axis = r2 < 0x1.0p-104; xr = axis ? 0.0 : x * ir; yr = axis ? 0.0 : y * ir; }
        else if (r < ACM_EPS) { xr = 0.0; yr = 0.0; } else { xr = x / r; yr = y / r; }
        u = c.fx * thd * xr + c.cx;
        v = c.fy * thd * yr + c.cy;
        return ACM_POINT_OK;  // no image-bounds test in the reference
    }
    template <bool IEEE = false>
    static __device__ int unproject(const CamParams& c, double u, double v, double& rx, double& ry, double& rz) {
        if (c.has_resolution && acm_outside(c, u, v)) return ACM_POINT_IS_OUTSIDE_IMAGE;
        const double k1 = c.d[0], k2 = c.d[1], k3 = c.d[2], k4 = c.d[3];
        double mx = acm_mx(c, u), my = acm_my(c, v);
        if (!IEEE && c.fast_newton) {
            // The host proved (Kantorovich bound in acm_make_cam_params) that Newton's method converges for every ru in
            // (1e-6, pi/2] of this camera: the reference's loop returns Ok for every such pixel and its iterate lies within
            // ~1e-12 of the root.  The only status decisions left are ru > 1e-6 and ru > 0, taken exactly on r2; the iteration
            // itself runs contracted (Horner FMAs, one reciprocal per step), ~17 instead of ~35 FP64 instructions per step.
            const double r2 = mx * mx + my * my;
            if (r2 == r2) {   // NaN pixels keep the reference's fmin(NaN, pi/2) path below
                if (!(r2 > ACM_SQRT_GT_1EM6)) {
                    if (r2 > 0.0) return ACM_POINT_NUMERICAL_ERROR;   // 0 < ru <= 1e-6 (kannala_brandt.rs:521-527)
                    rx = 0.0; ry = 0.0; rz = 1.0;                      // ru == 0: theta = 0, the optical axis
                    return ACM_POINT_OK;
                }
                double irs;
                const double rs = acm_sqrt_inv(r2, irs);
                const double half_pi = 3.14159265358979323846 / 2.0;
                const bool clamp = rs > half_pi;
                const double ru_f = clamp ? half_pi : rs, iru = clamp ? 1.0 / half_pi : irs;
                const double k3x = 3.0 * k1, k5x = 5.0 * k2, k7x = 7.0 * k3, k9x = 9.0 * k4;
                double th = ru_f;
#pragma unroll 1
                for (int i = 0; i < 10; ++i) {
                    const double t2 = __dmul_rn(th, th);
                    const double P = __fma_rn(t2, __fma_rn(t2, __fma_rn(t2, __fma_rn(t2, k4, k3), k2), k1), 1.0);
                    const double f = __fma_rn(th, P, -ru_f);
                    const double fp = __fma_rn(t2, __fma_rn(t2, __fma_rn(t2, __fma_rn(t2, k9x, k7x), k5x), k3x), 1.0);
                    const double delta = __dmul_rn(f, acm_rcp(fp));
                    th = __dsub_rn(th, delta);
                    if (fabs(delta) < 1e-6) break;
                }
                double st, ct;
                if (th >= 0.0 && th <= 1.8) acm_sincos_small(th, st, ct); else sincos(th, &st, &ct);
                rx = st * (mx * iru); ry = st * (my * iru); rz = ct;
                // (mx, my) / ru is a unit vector unless ru was clamped to pi/2 (kannala_brandt.rs:466): only then does the
                // reference's normalize() change more than the last bits
                if (clamp) acm_normalize<false>(rx, ry, rz, rx, ry, rz);
                return ACM_POINT_OK;
            }
        }
        double ru = sqrt(mx * mx + my * my);   // IEEE: ru enters the Newton iteration and its convergence tests
        ru = fmin(ru, 3.14159265358979323846 / 2.0);
        double th = ru;
        bool converged = true;
        if (ru > 1e-6) {
            for (int i = 0; i < 10; ++i) {
                double t2 = th * th, t4 = t2 * t2, t6 = t4 * t2, t8 = t4 * t4;
                double a1 = k1 * t2, a2 = k2 * t4, a3 = k3 * t6, a4 = k4 * t8;
                double f = th * (1.0 + a1 + a2 + a3 + a4) - ru;
                double fp = 1.0 + (3.0 * a1) + (5.0 * a2) + (7.0 * a3) + (9.0 * a4);
                if (fabs(fp) < ACM_EPS) { converged = false; break; }
                double delta = f / fp;
                th -= delta;
                if (fabs(delta) < 1e-6) break;
                if (i == 9) converged = false;
            }
        } else {
            if (ru > 0.0) converged = false; else th = 0.0;
        }
        if (!converged) return ACM_POINT_NUMERICAL_ERROR;
        double xc, yc;
        if (IEEE) {
            if (fabs(ru) < ACM_EPS) { xc = 0.0; yc = 0.0; } else { xc = mx / ru; yc = my / ru; }
        } else {
            const double iru = acm_rcp(ru);
            const bool axis = fabs(ru) < ACM_EPS;
            xc = axis ? 0.0 : mx * iru; yc = axis ? 0.0 : my * iru;
        }
        double st, ct;
        sincos(th, &st, &ct);
        acm_normalize<IEEE>(st * xc, st * yc, ct, rx, ry, rz);
        return ACM_POINT_OK;
    }
};

// ---- UCM (ucm.rs:297-316, :337-367, :154-161, :177-184), d = [alpha] -------------------------
// k0 = w of check_proj_condition, k1 = gamma*gamma/(2*alpha-1), k2 = xi = alpha/gamma
template <> struct CamModel<ACM_MODEL_UCM> {
    template <bool BOUNDS, bool FAST = false>
    static __device__ __forceinline__ int project(const CamParams& c, double x, double y, double z, double& u, double& v) {
        const double alpha = c.d[0];
        double d = sqrt(x * x + y * y + z * z);
        double den = alpha * d + (1.0 - alpha) * z;
        bool cond = z > -c.k0 * d;
        if (den < ACM_PRECISION || !cond) return ACM_POINT_IS_OUTSIDE_IMAGE;
        u = c.fx * (x / den) + c.cx;
        v = c.fy * (y / den) + c.cy;
        return ACM_POINT_OK;
    }
    template <bool IEEE = false>
    static __device__ __forceinline__ int unproject(const CamParams& c, double u, double v, double& rx, double& ry, double& rz) {
        const double alpha = c.d[0];
        double gamma = 1.0 - alpha;
        double xi = c.k2;
        double mx = acm_mx(c, u) * gamma, my = acm_my(c, v) * gamma;
        double r2 = mx * mx + my * my;
        double den = 1.0 - r2;
        bool cond = (alpha > 0.5) ? (r2 <= c.k1) : true;
        if (den < ACM_PRECISION || !cond) return ACM_POINT_IS_OUTSIDE_IMAGE;
        double num = xi + acm_tail_sqrt<IEEE>(1.0 + (1.0 - xi * xi) * r2);
        double coeff = acm_tail_div<IEEE>(num, den);
        acm_normalize<IEEE>(coeff * mx, coeff * my, coeff - xi, rx, ry, rz);
        return ACM_POINT_OK;
    }
};

// ---- EUCM (eucm.rs:328-347, :368-398, :167-177, :194-200), d = [alpha,beta] -------------------
// k0 = (alpha-1)/(2*alpha-1), k1 = 1/beta*(2*alpha-1)  (the reference's precedence, kept)
template <> struct CamModel<ACM_MODEL_EUCM> {
    template <bool BOUNDS, bool FAST = false>
    static __device__ __forceinline__ int project(const CamParams& c, double x, double y, double z, double& u, double& v) {
        const double alpha = c.d[0], beta = c.d[1];
        double d = sqrt(beta * (x * x + y * y) + z * z);
        double den = alpha * d + (1.0 - alpha) * z;
        bool cond = true;
        if (alpha > 0.5) { if (z < den * c.k0) cond = false; }
        if (den < ACM_PRECISION || !cond) return ACM_POINT_IS_OUTSIDE_IMAGE;
        u = c.fx * (x / den) + c.cx;
        v = c.fy * (y / den) + c.cy;
        return ACM_POINT_OK;
    }
    template <bool IEEE = false>
    static __device__ __forceinline__ int unproject(const CamParams& c, double u, double v, double& rx, double& ry, double& rz) {
        const double alpha = c.d[0], beta = c.d[1];
        double mx = acm_mx(c, u), my = acm_my(c, v);
        double r2 = mx * mx + my * my;
        double gamma = 1.0 - alpha;
        double num = 1.0 - r2 * alpha * alpha * beta;
        double det = 1.0 - (alpha - gamma) * beta * r2;
        bool cond = !(alpha > 0.5 && r2 > c.k1);
        if (det < ACM_PRECISION || !cond) return ACM_POINT_IS_OUTSIDE_IMAGE;
        double den = gamma + alpha * acm_tail_sqrt<IEEE>(det);
        double mz = acm_tail_div<IEEE>(num, den);
        acm_normalize<IEEE>(mx, my, mz, rx, ry, rz);
        return ACM_POINT_OK;
    }
};

// ---- Double Sphere (double_sphere.rs:361-390, :436-476, :177-184, :200-209), d = [alpha,xi] ---
// k0 = w2, k1 = 1/(2*alpha-1)
template <> struct CamModel<ACM_MODEL_DOUBLE_SPHERE> {
    template <bool BOUNDS, bool FAST = false>
    static __device__ __forceinline__ int project(const CamParams& c, double x, double y, double z, double& u, double& v) {
        const double alpha = c.d[0], xi = c.d[1];
        double r2 = (x * x) + (y * y);
        double d1 = sqrt(r2 + (z * z));
        double g = xi * d1 + z;
        double d2 = sqrt(r2 + g * g);
        double den = alpha * d2 + (1.0 - alpha) * g;
        bool cond = z > -c.k0 * d1;
        if (den < ACM_PRECISION || !cond) return ACM_POINT_IS_OUTSIDE_IMAGE;
        u = c.fx * (x / den) + c.cx;
        v = c.fy * (y / den) + c.cy;
        return ACM_POINT_OK;
    }
    template <bool IEEE = false>
    static __device__ __forceinline__ int unproject(const CamParams& c, double u, double v, double& rx, double& ry, double& rz) {
        const double alpha = c.d[0], xi = c.d[1];
        double gamma = 1.0 - alpha;
        double mx = acm_mx(c, u), my = acm_my(c, v);
        double r2 = (mx * mx) + (my * my);
        bool cond = true;
        if (alpha > 0.5) { if (r2 > c.k1) cond = false; }
        if (alpha != 0.0 && !cond) return ACM_POINT_IS_OUTSIDE_IMAGE;
        // mz feeds the last validity test (den < PRECISION).  The fast quotient is within 4 ulp, so den is
        // within ~1e-15 relative of the reference's; only inside a 1e-12 band around the threshold (never
        // reached with 0 < alpha <= 1, where r2 < 1e-3 implies mz ~ 1) is mz redone with IEEE operations.
        const double mz_num = 1.0 - alpha * alpha * r2, mz_arg = 1.0 - (2.0 * alpha - 1.0) * r2;
        double mz = acm_tail_div<IEEE>(mz_num, alpha * acm_tail_sqrt<IEEE>(mz_arg) + gamma);
        double mz2 = mz * mz;
        double den = mz2 + r2;
        if (!IEEE && fabs(den - ACM_PRECISION) < 1e-12) {
            mz = mz_num / (alpha * sqrt(mz_arg) + gamma);
            mz2 = mz * mz;
            den = mz2 + r2;
        }
        if (den < ACM_PRECISION) return ACM_POINT_IS_OUTSIDE_IMAGE;
        double num = mz * xi + acm_tail_sqrt<IEEE>(mz2 + (1.0 - xi * xi) * r2);
        double coeff = acm_tail_div<IEEE>(num, den);
        acm_normalize<IEEE>(coeff * mx, coeff * my, coeff * mz - xi, rx, ry, rz);
        return ACM_POINT_OK;
    }
};

// ---- FOV (fov.rs:284-316, :336-363), d = [w]; k0 = tan(w/2) from the host's libm -------------
template <> struct CamModel<ACM_MODEL_FOV> {
    template <bool BOUNDS, bool FAST = false>
    static __device__ __forceinline__ int project(const CamParams& c, double x, double y, double z, double& u, double& v) {
        const double w = c.d[0];
        if (z < ACM_SQRT_EPS) return ACM_POINT_AT_CAMERA_CENTER;
        double r2 = x * x + y * y;
        double t = c.k0;
        double rd;
        if (r2 < ACM_SQRT_EPS) rd = 2.0 * t / w;
        else if (FAST) {   // values only behind the branch: coupled sqrt / rsqrt and a reciprocal of w instead of sqrt + division
            double ir;
            const double r = acm_sqrt_inv(r2, ir);
            rd = acm_atan2_q1(2.0 * t * r, z) * (ir * acm_rcp(w));
        } else { const double r = sqrt(r2); rd = acm_atan2_q1(2.0 * t * r, z) / (r * w); }  // 2*t*r >= 0, z >= sqrt(EPS)
        double mx = x * rd, my = y * rd;
        u = c.fx * mx + c.cx;
        v = c.fy * my + c.cy;
        return ACM_POINT_OK;
    }
    template <bool IEEE = false>
    static __device__ __forceinline__ int unproject(const CamParams& c, double u, double v, double& rx, double& ry, double& rz) {
        const double w = c.d[0];
        double mul2 = c.k0 * 2.0;
        double mx = acm_mx(c, u), my = acm_my(c, v);
        double r2 = mx * mx + my * my;
        double x, y;
        if (IEEE) {
            double rd = sqrt(r2);
            if (mul2 > ACM_SQRT_EPS && rd > ACM_SQRT_EPS) {
                double s, co;
                sincos(rd * w, &s, &co);
                double ru = s / (rd * mul2);
                x = mx * ru / co; y = my * ru / co;
            } else { x = mx; y = my; }
        }
        // the branch (two formulas that do NOT agree at the seam, fov.rs:349-357) is decided exactly:
        // sqrt(r2) > sqrt(EPS)  <=>  r2 > ACM_SQRT_GT_2M26; the values behind it need 1e-9 only
        else if (mul2 > ACM_SQRT_EPS && r2 > ACM_SQRT_GT_2M26) {
            double ird;
            const double rd = acm_sqrt_inv(r2, ird);
            double s, co;
            const double arg = rd * w;
            if (arg >= 0.0 && arg <= 1.8) acm_sincos_small(arg, s, co); else sincos(arg, &s, &co);
            const double k = s * ird * acm_rcp(mul2 * co);   // (sin / (rd mul2)) / cos
            x = mx * k; y = my * k;
        } else { x = mx; y = my; }
        acm_normalize<IEEE>(x, y, 1.0, rx, ry, rz);
        return ACM_POINT_OK;
    }
};

// Runtime model id -> compile-time specialisation.
#define ACM_DISPATCH_MODEL(model_id, ...)                                                     \
    switch (model_id) {                                                                       \
        case ACM_MODEL_PINHOLE: { constexpr int M = ACM_MODEL_PINHOLE; __VA_ARGS__; break; }  \
        case ACM_MODEL_RADTAN: { constexpr int M = ACM_MODEL_RADTAN; __VA_ARGS__; break; }    \
        case ACM_MODEL_KANNALA_BRANDT: { constexpr int M = ACM_MODEL_KANNALA_BRANDT; __VA_ARGS__; break; } \
        case ACM_MODEL_UCM: { constexpr int M = ACM_MODEL_UCM; __VA_ARGS__; break; }          \
        case ACM_MODEL_EUCM: { constexpr int M = ACM_MODEL_EUCM; __VA_ARGS__; break; }        \
        case ACM_MODEL_DOUBLE_SPHERE: { constexpr int M = ACM_MODEL_DOUBLE_SPHERE; __VA_ARGS__; break; } \
        case ACM_MODEL_FOV: { constexpr int M = ACM_MODEL_FOV; __VA_ARGS__; break; }          \
        default: return acm_fail(ctx, ACM_ERR_INVALID_ARG, "unknown camera model id %d", (int)(model_id)); \
    }

