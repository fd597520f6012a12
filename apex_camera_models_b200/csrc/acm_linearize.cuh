// Fused residual + analytic Jacobian + J^T J / J^T r accumulation (one streaming pass).
//
// This replaces `*CameraParamsFactor::linearize` + the solver's J^T J of apex-solver at the
// call sites reference bin/camera_converter.rs:378-420 (and clones).  The Jacobian is never
// materialised: every thread keeps the normal equations of its points in registers.
//
// Sparsity (SURVEY.md Appendix A): the u-row touches only {fx, cx, dist..}, the v-row only
// {fy, cy, dist..}.  Per row we therefore carry a short vector a = [a_f, a_c, a_d0, a_d1, ..].
// For the PIXEL residual a_c == 1 exactly, so H[c,c] is the valid-point count and every
// product with a_c is a plain add (UNIT_C = true).
//
// Accumulator layout (flat, all indices compile-time => registers):
//   HFF[2]  H[fx,fx], H[fy,fy]          HFC[2]  H[fx,cx], H[fy,cy]      HCC[2] H[cx,cx], H[cy,cy]
//   HFD[2][ND]  H[f*,d_k]               HCD[2][ND]  H[c*,d_k]           HDD[ND(ND+1)/2]
//   GF[2] GC[2] GD[ND]   COST   COUNT
#pragma once
#include <type_traits>
#include "acm_internal.cuh"
#include "acm_math.cuh"

#define LIN_EPS 2.220446049250313e-16
#define LIN_SQRT_EPS 1.4901161193847656e-08
#define LIN_PRECISION 1e-3

// ---------------------------------------------------------------------------------------
// Branch-free f64 reciprocal / rsqrt / sqrt for the solver kernels.  The CUDA library versions
// carry a slow-path CALL for special operands inside the streaming loop, which stops the
// compiler from interleaving the two points a thread owns.  Here: MUFU seed (rcp.approx /
// rsqrt.approx, ~2^-23) + two Newton steps in FMA arithmetic => <= 2 ulp for normal operands;
// 0, inf and NaN propagate to NaN/inf and are rejected by the validity compares downstream.
// (Only used where the tolerance is 1e-9 relative -- never in the bit-exact project kernels.)
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ double fast_rcp(double a) { return acm_rcp(a); }
// sqrt(a) with 1/sqrt(a) as a by-product.
// REFINE_INV = false: one Newton step on the seed (inv accurate to ~2^-44, enough for a Jacobian
// entry), then a Heron correction with the exact fma residual, which squares the error: s <= 1 ulp.
// REFINE_INV = true (inv feeds a residual): two coupled Goldschmidt iterations on g ~ sqrt(a),
// h ~ 1/(2 sqrt(a)) -- r = 1/2 - g h, g += g r, h += h r -- take both from 2^-23 to full precision in
// 2 DMUL + 6 DFMA + 1 DADD (the separate Newton + Heron form needed 11).
template <bool REFINE_INV = false>
__device__ __forceinline__ double fast_sqrt(double a, double& inv) {
    double y;
    asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(a));
    if (REFINE_INV) {
        double g = a * y, h = 0.5 * y;
        double r = fma(-g, h, 0.5);
        g = fma(g, r, g); h = fma(h, r, h);
        r = fma(-g, h, 0.5);
        g = fma(g, r, g); h = fma(h, r, h);
        inv = h + h;
        return g;
    }
    const double h = 0.5 * a;
    y = y * fma(-h, y * y, 1.5);
    double s = a * y;
    double r = fma(-s, s, a);
    inv = REFINE_INV ? y * fma(-h, y * y, 1.5) : y;
    return fma(r, 0.5 * y, s);
}

__device__ __forceinline__ double fast_atan2_q1(double a, double b) { return acm_atan2_q1<false>(a, b); }

template <int ND> struct AccLayout {
    static constexpr int HFF = 0, HFC = 2, HCC = 4, HFD = 6, HCD = 6 + 2 * ND, HDD = 6 + 4 * ND;
    static constexpr int GF = HDD + ND * (ND + 1) / 2, GC = GF + 2, GD = GC + 2, COST = GD + ND, COUNT = COST + 1;
    static constexpr int N = COUNT + 1;
    __host__ __device__ static constexpr int tri(int j, int k) { return j * ND - j * (j - 1) / 2 + (k - j); }  // j <= k
};

// Parameters as the kernels see them (plain doubles; derived constants recomputed on device
// when the parameters come from the device-resident LM state).
struct LinParams {
    double fx, fy, cx, cy;
    double d[5];
    double k0;  // validity constant: UCM w, EUCM (a-1)/(2a-1), DS w2, FOV tan(w/2)
};

__host__ __device__ inline void lin_derive(int model, LinParams& p) {
    const double alpha = p.d[0];
    switch (model) {
        case ACM_MODEL_UCM: p.k0 = (alpha <= 0.5) ? alpha / (1.0 - alpha) : (1.0 - alpha) / alpha; break;
        case ACM_MODEL_EUCM: p.k0 = (alpha - 1.0) / (2.0 * alpha - 1.0); break;
        case ACM_MODEL_DOUBLE_SPHERE: {
            const double xi = p.d[1];
            double w1 = (alpha <= 0.5) ? alpha / (1.0 - alpha) : (1.0 - alpha) / alpha;
            p.k0 = (w1 + xi) / sqrt(2.0 * w1 * xi + xi * xi + 1.0);
            break;
        }
        case ACM_MODEL_FOV: p.k0 = tan(p.d[0] / 2.0); break;
        default: p.k0 = 0.0; break;
    }
}

// LinParams of a camera block on the host (acm_solver.cu's passes and Jacobian kernels, acm_triangulate.cu)
static inline void make_lin_params(const acm_camera* cam, LinParams* p) {
    memset(p, 0, sizeof(*p));
    p->fx = cam->params[0]; p->fy = cam->params[1]; p->cx = cam->params[2]; p->cy = cam->params[3];
    for (int i = 4; i < cam->n_params; ++i) p->d[i - 4] = cam->params[i];
    lin_derive(cam->model, *p);
}

// ---------------------------------------------------------------------------------------
// Per-model residual + Jacobian rows.  eval() returns validity (the model's geometric test,
// no image-bounds test: the factor has no resolution) and fills
//   ru, rv            residuals
//   au[2+ND], av[2+ND] non-zero Jacobian entries of the two rows (a[1] ignored when UNIT_C)
// ---------------------------------------------------------------------------------------
template <int M, int KIND> struct Lin;

template <> struct Lin<ACM_MODEL_PINHOLE, ACM_RESIDUAL_PIXEL> {
    static constexpr int ND = 0; static constexpr bool UNIT_C = true;
    static __device__ __forceinline__ bool eval(const LinParams& p, double x, double y, double z, double u, double v,
                                                double& ru, double& rv, double* au, double* av) {
        double iz = fast_rcp(z);
        double mx = x * iz, my = y * iz;
        ru = fma(p.fx, mx, p.cx) - u; rv = fma(p.fy, my, p.cy) - v;
        au[0] = mx; av[0] = my; au[1] = av[1] = 1.0;
        return z >= LIN_SQRT_EPS;
    }
};

template <> struct Lin<ACM_MODEL_RADTAN, ACM_RESIDUAL_PIXEL> {
    static constexpr int ND = 5; static constexpr bool UNIT_C = true;
    static __device__ __forceinline__ bool eval(const LinParams& p, double x, double y, double z, double u, double v,
                                                double& ru, double& rv, double* au, double* av) {
        const double k1 = p.d[0], k2 = p.d[1], p1 = p.d[2], p2 = p.d[3], k3 = p.d[4];
        double iz = fast_rcp(z);
        double xp = x * iz, yp = y * iz;
        double rho = xp * xp + yp * yp, rho2 = rho * rho, rho3 = rho2 * rho;
        double rad = 1.0 + k1 * rho + k2 * rho2 + k3 * rho3;
        double xy2 = 2.0 * xp * yp;
        double tx = rho + 2.0 * xp * xp, ty = rho + 2.0 * yp * yp;
        double mx = xp * rad + p1 * xy2 + p2 * tx;
        double my = yp * rad + p1 * ty + p2 * xy2;
        ru = fma(p.fx, mx, p.cx) - u; rv = fma(p.fy, my, p.cy) - v;
        double fxx = p.fx * xp, fyy = p.fy * yp;
        au[0] = mx; av[0] = my; au[1] = av[1] = 1.0;
        au[2] = fxx * rho;  av[2] = fyy * rho;    // k1
        au[3] = fxx * rho2; av[3] = fyy * rho2;   // k2
        au[4] = p.fx * xy2; av[4] = p.fy * ty;    // p1
        au[5] = p.fx * tx;  av[5] = p.fy * xy2;   // p2
        au[6] = fxx * rho3; av[6] = fyy * rho3;   // k3
        return z >= LIN_SQRT_EPS;
    }
};

template <> struct Lin<ACM_MODEL_KANNALA_BRANDT, ACM_RESIDUAL_PIXEL> {
    static constexpr int ND = 4; static constexpr bool UNIT_C = true;
    static __device__ __forceinline__ bool eval(const LinParams& p, double x, double y, double z, double u, double v,
                                                double& ru, double& rv, double* au, double* av) {
        const bool ok = z >= LIN_EPS;  // z < 0 and 0 <= z < EPS both fail (kannala_brandt.rs:345-351)
        double ir;
        double r = fast_sqrt<true>(x * x + y * y, ir);
        const bool on_axis = !(r >= LIN_EPS);  // also catches r = NaN from x = y = 0
        r = on_axis ? 0.0 : r;
        double th = fast_atan2_q1(r, ok ? z : 1.0);
        double xr = on_axis ? 0.0 : x * ir, yr = on_axis ? 0.0 : y * ir;
        double t2 = th * th, t3 = t2 * th, t5 = t3 * t2, t7 = t5 * t2, t9 = t7 * t2;
        double thd = th + p.d[0] * t3 + p.d[1] * t5 + p.d[2] * t7 + p.d[3] * t9;
        double mx = thd * xr, my = thd * yr;
        ru = fma(p.fx, mx, p.cx) - u; rv = fma(p.fy, my, p.cy) - v;
        double fxr = p.fx * xr, fyr = p.fy * yr;
        au[0] = mx; av[0] = my; au[1] = av[1] = 1.0;
        au[2] = fxr * t3; av[2] = fyr * t3;
        au[3] = fxr * t5; av[3] = fyr * t5;
        au[4] = fxr * t7; av[4] = fyr * t7;
        au[5] = fxr * t9; av[5] = fyr * t9;
        return ok;
    }
};

// Unified family: den and d(den)/d(dist) are shared by both residual kinds.
template <int M> struct Unified;
template <> struct Unified<ACM_MODEL_UCM> {
    static constexpr int ND = 1;
    static __device__ __forceinline__ bool den(const LinParams& p, double x, double y, double z, double& den, double* dd) {
        const double alpha = p.d[0];
        double id;
        double d = fast_sqrt(x * x + y * y + z * z, id);
        den = alpha * d + (1.0 - alpha) * z;
        dd[0] = d - z;
        return (den >= LIN_PRECISION) && (z > -p.k0 * d);
    }
};
template <> struct Unified<ACM_MODEL_EUCM> {
    static constexpr int ND = 2;
    static __device__ __forceinline__ bool den(const LinParams& p, double x, double y, double z, double& den, double* dd) {
        const double alpha = p.d[0], beta = p.d[1];
        double rr = x * x + y * y;
        double q = beta * rr + z * z;
        double id;
        double d = fast_sqrt(q, id);
        den = alpha * d + (1.0 - alpha) * z;
        dd[0] = d - z;
        dd[1] = 0.5 * alpha * rr * id;
        bool cond = true;
        if (alpha > 0.5) cond = !(z < den * p.k0);
        return (den >= LIN_PRECISION) && cond;
    }
};
template <> struct Unified<ACM_MODEL_DOUBLE_SPHERE> {
    static constexpr int ND = 2;
    static __device__ __forceinline__ bool den(const LinParams& p, double x, double y, double z, double& den, double* dd) {
        const double alpha = p.d[0], xi = p.d[1];
        double rr = x * x + y * y;
        double id1;
        double d1 = fast_sqrt(rr + z * z, id1);
        double g = fma(xi, d1, z);
        double q = fma(g, g, rr);
        double id2;
        double d2 = fast_sqrt(q, id2);
        double oma = 1.0 - alpha;
        den = alpha * d2 + oma * g;
        dd[0] = d2 - g;
        dd[1] = d1 * fma(alpha * g, id2, oma);
        return (den >= LIN_PRECISION) && (z > -p.k0 * d1);
    }
};

template <int M> struct LinUnifiedPixel {
    static constexpr int ND = Unified<M>::ND; static constexpr bool UNIT_C = true;
    static __device__ __forceinline__ bool eval(const LinParams& p, double x, double y, double z, double u, double v,
                                                double& ru, double& rv, double* au, double* av) {
        double den, dd[2];
        const bool ok = Unified<M>::den(p, x, y, z, den, dd);
        double inv = fast_rcp(den);
        double mx = x * inv, my = y * inv;
        ru = fma(p.fx, mx, p.cx) - u; rv = fma(p.fy, my, p.cy) - v;
        double cu = -(p.fx * mx) * inv, cv = -(p.fy * my) * inv;  // d(u)/d(den), d(v)/d(den)
        au[0] = mx; av[0] = my; au[1] = av[1] = 1.0;
#pragma unroll
        for (int k = 0; k < ND; ++k) { au[2 + k] = cu * dd[k]; av[2 + k] = cv * dd[k]; }
        return ok;
    }
};
template <int M> struct LinUnifiedAlgebraic {
    static constexpr int ND = Unified<M>::ND; static constexpr bool UNIT_C = false;
    static __device__ __forceinline__ bool eval(const LinParams& p, double x, double y, double z, double u, double v,
                                                double& ru, double& rv, double* au, double* av) {
        double den, dd[2];
        const bool ok = Unified<M>::den(p, x, y, z, den, dd);
        double du = u - p.cx, dv = v - p.cy;
        ru = p.fx * x - du * den; rv = p.fy * y - dv * den;
        au[0] = x; av[0] = y; au[1] = den; av[1] = den;
#pragma unroll
        for (int k = 0; k < ND; ++k) { au[2 + k] = -du * dd[k]; av[2 + k] = -dv * dd[k]; }
        return ok;
    }
};
template <> struct Lin<ACM_MODEL_UCM, ACM_RESIDUAL_PIXEL> : LinUnifiedPixel<ACM_MODEL_UCM> {};
template <> struct Lin<ACM_MODEL_EUCM, ACM_RESIDUAL_PIXEL> : LinUnifiedPixel<ACM_MODEL_EUCM> {};
template <> struct Lin<ACM_MODEL_DOUBLE_SPHERE, ACM_RESIDUAL_PIXEL> : LinUnifiedPixel<ACM_MODEL_DOUBLE_SPHERE> {};
template <> struct Lin<ACM_MODEL_UCM, ACM_RESIDUAL_ALGEBRAIC> : LinUnifiedAlgebraic<ACM_MODEL_UCM> {};
template <> struct Lin<ACM_MODEL_EUCM, ACM_RESIDUAL_ALGEBRAIC> : LinUnifiedAlgebraic<ACM_MODEL_EUCM> {};
template <> struct Lin<ACM_MODEL_DOUBLE_SPHERE, ACM_RESIDUAL_ALGEBRAIC> : LinUnifiedAlgebraic<ACM_MODEL_DOUBLE_SPHERE> {};

template <> struct Lin<ACM_MODEL_FOV, ACM_RESIDUAL_PIXEL> {
    static constexpr int ND = 1; static constexpr bool UNIT_C = true;
    static __device__ __forceinline__ bool eval(const LinParams& p, double x, double y, double z, double u, double v,
                                                double& ru, double& rv, double* au, double* av) {
        // branch-free: the r2 < sqrt(EPS) case (fov.rs:203-207, constant rd) is a select at the end
        const bool ok = z >= LIN_SQRT_EPS;
        z = ok ? z : 1.0;
        const double w = p.d[0], t = p.k0;
        const double iw = fast_rcp(w), t2 = 2.0 * t, tt1 = fma(t, t, 1.0);   // loop-invariant
        const double r2 = x * x + y * y;
        const bool small = r2 < LIN_SQRT_EPS;
        const double r2s = small ? 1.0 : r2;
        double ir;
        const double r = fast_sqrt<true>(r2s, ir);
        const double a = fast_atan2_q1(t2 * r, z);
        const double da = z * r * tt1 * fast_rcp(fma(t2 * t2, r2s, z * z));
        const double irw = iw * ir;
        double rd = a * irw;
        double drd = (da - a * iw) * irw;
        rd = small ? t2 * iw : rd;
        drd = small ? (tt1 - t2 * iw) * iw : drd;
        double mx = x * rd, my = y * rd;
        ru = fma(p.fx, mx, p.cx) - u; rv = fma(p.fy, my, p.cy) - v;
        au[0] = mx; av[0] = my; au[1] = av[1] = 1.0;
        au[2] = p.fx * x * drd; av[2] = p.fy * y * drd;
        return ok;
    }
};

// ---------------------------------------------------------------------------------------
// rank-2 update of the packed normal equations with the two sparse rows
// ---------------------------------------------------------------------------------------
// Invalid points are folded in branch-free: every factor is replaced by an exact 0 (a select,
// never a multiplication by zero, so NaN/inf of a rejected point cannot leak).
template <int ND, bool UNIT_C>
__device__ __forceinline__ void lin_accumulate_masked(double* acc, bool ok, double ru, double rv, double* au, double* av) {
    ru = ok ? ru : 0.0; rv = ok ? rv : 0.0;
#pragma unroll
    for (int k = 0; k < 2 + ND; ++k) { au[k] = ok ? au[k] : 0.0; av[k] = ok ? av[k] : 0.0; }
    using L = AccLayout<ND>;
    acc[L::HFF + 0] = fma(au[0], au[0], acc[L::HFF + 0]);
    acc[L::HFF + 1] = fma(av[0], av[0], acc[L::HFF + 1]);
    acc[L::GF + 0] = fma(au[0], ru, acc[L::GF + 0]);
    acc[L::GF + 1] = fma(av[0], rv, acc[L::GF + 1]);
    if (UNIT_C) {
        acc[L::HFC + 0] += au[0];
        acc[L::HFC + 1] += av[0];
        acc[L::GC + 0] += ru;
        acc[L::GC + 1] += rv;
    } else {
        acc[L::HFC + 0] = fma(au[0], au[1], acc[L::HFC + 0]);
        acc[L::HFC + 1] = fma(av[0], av[1], acc[L::HFC + 1]);
        acc[L::HCC + 0] = fma(au[1], au[1], acc[L::HCC + 0]);
        acc[L::HCC + 1] = fma(av[1], av[1], acc[L::HCC + 1]);
        acc[L::GC + 0] = fma(au[1], ru, acc[L::GC + 0]);
        acc[L::GC + 1] = fma(av[1], rv, acc[L::GC + 1]);
    }
#pragma unroll
    for (int k = 0; k < ND; ++k) {
        acc[L::HFD + k] = fma(au[0], au[2 + k], acc[L::HFD + k]);
        acc[L::HFD + ND + k] = fma(av[0], av[2 + k], acc[L::HFD + ND + k]);
        if (UNIT_C) {
            acc[L::HCD + k] += au[2 + k];
            acc[L::HCD + ND + k] += av[2 + k];
        } else {
            acc[L::HCD + k] = fma(au[1], au[2 + k], acc[L::HCD + k]);
            acc[L::HCD + ND + k] = fma(av[1], av[2 + k], acc[L::HCD + ND + k]);
        }
        acc[L::GD + k] = fma(au[2 + k], ru, fma(av[2 + k], rv, acc[L::GD + k]));
#pragma unroll
        for (int j = 0; j <= k; ++j)
            acc[L::HDD + L::tri(j, k)] = fma(au[2 + j], au[2 + k], fma(av[2 + j], av[2 + k], acc[L::HDD + L::tri(j, k)]));
    }
    acc[L::COST] = fma(ru, ru, fma(rv, rv, acc[L::COST]));
    acc[L::COUNT] += ok ? 1.0 : 0.0;
}

// Reduced accumulator vector -> dense symmetric H (P x P), g, cost, count.
// FULL = false (the LM step): only the structurally non-zero entries of the UPPER triangle are written -- the caller zeroed H
// once and mirrors while it copies -- so the serial part of the step is ~25 independent load/store pairs (__restrict__ lets
// the loads run ahead of the stores) instead of P^2 zero stores, the fill and P(P-1)/2 dependent load-store mirrors.
template <int ND, bool UNIT_C, bool FULL = true>
__host__ __device__ inline void lin_unpack(const double* __restrict__ r, double* __restrict__ H, double* __restrict__ g, double* __restrict__ cost, double* __restrict__ count) {  // params not needed
    using L = AccLayout<ND>;
    constexpr int P = 4 + ND;
    if (FULL) for (int i = 0; i < P * P; ++i) H[i] = 0.0;
    const double cnt = r[L::COUNT];
    H[0 * P + 0] = r[L::HFF]; H[1 * P + 1] = r[L::HFF + 1];
    H[0 * P + 2] = r[L::HFC]; H[1 * P + 3] = r[L::HFC + 1];
    H[2 * P + 2] = UNIT_C ? cnt : r[L::HCC]; H[3 * P + 3] = UNIT_C ? cnt : r[L::HCC + 1];
    for (int k = 0; k < ND; ++k) {
        H[0 * P + 4 + k] = r[L::HFD + k]; H[1 * P + 4 + k] = r[L::HFD + ND + k];
        H[2 * P + 4 + k] = r[L::HCD + k]; H[3 * P + 4 + k] = r[L::HCD + ND + k];
        for (int j = 0; j <= k; ++j) H[(4 + j) * P + 4 + k] = r[L::HDD + L::tri(j, k)];
        g[4 + k] = r[L::GD + k];
    }
    g[0] = r[L::GF]; g[1] = r[L::GF + 1]; g[2] = r[L::GC]; g[3] = r[L::GC + 1];
    if (FULL) for (int a = 0; a < P; ++a) for (int b = 0; b < a; ++b) H[a * P + b] = H[b * P + a];
    *cost = 0.5 * r[L::COST];
    *count = cnt;
}

// ---------------------------------------------------------------------------------------
// LinOps<M, KIND>: what the streaming kernel, the LM step and the host unpack use.
// Generic: per-model eval() + the sparse rank-2 update above.
// ---------------------------------------------------------------------------------------
template <int M, int KIND> struct LinOps {
    using E = Lin<M, KIND>;
    static constexpr int ND = E::ND, P = 4 + ND;
    using L = AccLayout<ND>;
    static constexpr int NACC = L::N, COST = L::COST, COUNT = L::COUNT;
    static __device__ __forceinline__ void point(double* acc, const LinParams& p, double x, double y, double z, double u, double v) {
        double ru, rv, au[2 + ND], av[2 + ND];
        const bool ok = E::eval(p, x, y, z, u, v, ru, rv, au, av);
        lin_accumulate_masked<ND, E::UNIT_C>(acc, ok, ru, rv, au, av);
    }
    // `x` = the parameter vector the pass was evaluated at (unused here: fx, fy are folded in during the pass)
    template <bool FULL = true>
    __host__ __device__ static void unpack(const double* __restrict__ r, const double* __restrict__ x, double* __restrict__ H, double* __restrict__ g, double* __restrict__ cost, double* __restrict__ count) {
        (void)x;
        lin_unpack<ND, E::UNIT_C, FULL>(r, H, g, cost, count);
    }
};

// Kannala-Brandt: J_u[k_i] = fx*xr*theta^(2i+1), J_v[k_i] = fy*yr*theta^(2i+1), so every product
// with a distortion column factors through the odd powers t_k = theta^(2k+3):
//   H[f,d_k] = sum (m*f*r) t_k      H[c,d_k] = sum (f*r) t_k      g[d_k] = sum (fxr*ru + fyr*rv) t_k
//   H[d_j,d_k] = sum (fxr^2 + fyr^2) theta^(2(j+k)+6)  -> depends on j+k only: 7 power sums S_m
// 48 accumulate instructions per point instead of 63, 37 accumulators instead of 45.
template <> struct LinOps<ACM_MODEL_KANNALA_BRANDT, ACM_RESIDUAL_PIXEL> {
    static constexpr int ND = 4, P = 8;
    static constexpr int HFF = 0, HFC = 2, GF = 4, GC = 6, HFD = 8, HCD = 16, S = 24, GD = 31, COST = 35, COUNT = 36, NACC = 37;
    static __device__ __forceinline__ void point(double* acc, const LinParams& p, double x, double y, double z, double u, double v) {
        const bool ok = z >= LIN_EPS;  // kannala_brandt.rs:345-351
        double ir;
        double r = fast_sqrt<true>(x * x + y * y, ir);
        const bool on_axis = !(r >= LIN_EPS);
        r = on_axis ? 0.0 : r;
        const double th = fast_atan2_q1(r, ok ? z : 1.0);
        const double xr = on_axis ? 0.0 : x * ir, yr = on_axis ? 0.0 : y * ir;
        const double t2 = th * th, t3 = t2 * th, t5 = t3 * t2, t7 = t5 * t2, t9 = t7 * t2;
        const double thd = fma(p.d[3], t9, fma(p.d[2], t7, fma(p.d[1], t5, fma(p.d[0], t3, th))));
        double mx = thd * xr, my = thd * yr;
        double ru = fma(p.fx, mx, p.cx) - u, rv = fma(p.fy, my, p.cy) - v;
        double fxr = p.fx * xr, fyr = p.fy * yr;
        mx = ok ? mx : 0.0; my = ok ? my : 0.0; ru = ok ? ru : 0.0; rv = ok ? rv : 0.0; fxr = ok ? fxr : 0.0; fyr = ok ? fyr : 0.0;
        acc[HFF] = fma(mx, mx, acc[HFF]); acc[HFF + 1] = fma(my, my, acc[HFF + 1]);
        acc[HFC] += mx; acc[HFC + 1] += my;
        acc[GF] = fma(mx, ru, acc[GF]); acc[GF + 1] = fma(my, rv, acc[GF + 1]);
        acc[GC] += ru; acc[GC + 1] += rv;
        const double t[4] = {t3, t5, t7, t9};
        const double a = mx * fxr, b = my * fyr, c = fma(fxr, ru, fyr * rv), w = fma(fxr, fxr, fyr * fyr);
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            acc[HFD + k] = fma(a, t[k], acc[HFD + k]);
            acc[HFD + 4 + k] = fma(b, t[k], acc[HFD + 4 + k]);
            acc[HCD + k] = fma(fxr, t[k], acc[HCD + k]);
            acc[HCD + 4 + k] = fma(fyr, t[k], acc[HCD + 4 + k]);
            acc[GD + k] = fma(c, t[k], acc[GD + k]);
        }
        const double wt3 = w * t3, wt9 = w * t9;
        acc[S + 0] = fma(wt3, t3, acc[S + 0]);  // theta^6
        acc[S + 1] = fma(wt3, t5, acc[S + 1]);  // theta^8
        acc[S + 2] = fma(wt3, t7, acc[S + 2]);  // theta^10
        acc[S + 3] = fma(wt3, t9, acc[S + 3]);  // theta^12
        acc[S + 4] = fma(wt9, t5, acc[S + 4]);  // theta^14
        acc[S + 5] = fma(wt9, t7, acc[S + 5]);  // theta^16
        acc[S + 6] = fma(wt9, t9, acc[S + 6]);  // theta^18
        acc[COST] = fma(ru, ru, fma(rv, rv, acc[COST]));
        acc[COUNT] += ok ? 1.0 : 0.0;
    }
    template <bool FULL = true>
    __host__ __device__ static void unpack(const double* __restrict__ r, const double* __restrict__ x, double* __restrict__ H, double* __restrict__ g, double* __restrict__ cost, double* __restrict__ count) {
        (void)x;
        if (FULL) for (int i = 0; i < P * P; ++i) H[i] = 0.0;
        const double cnt = r[COUNT];
        H[0 * P + 0] = r[HFF]; H[1 * P + 1] = r[HFF + 1];
        H[0 * P + 2] = r[HFC]; H[1 * P + 3] = r[HFC + 1];
        H[2 * P + 2] = cnt; H[3 * P + 3] = cnt;
        for (int k = 0; k < 4; ++k) {
            H[0 * P + 4 + k] = r[HFD + k]; H[1 * P + 4 + k] = r[HFD + 4 + k];
            H[2 * P + 4 + k] = r[HCD + k]; H[3 * P + 4 + k] = r[HCD + 4 + k];
            for (int j = 0; j <= k; ++j) H[(4 + j) * P + 4 + k] = r[S + j + k];
            g[4 + k] = r[GD + k];
        }
        g[0] = r[GF]; g[1] = r[GF + 1]; g[2] = r[GC]; g[3] = r[GC + 1];
        if (FULL) for (int a = 0; a < P; ++a) for (int b = 0; b < a; ++b) H[a * P + b] = H[b * P + a];
        *cost = 0.5 * r[COST];
        *count = cnt;
    }
};

// RadTan (parameter order k1, k2, p1, p2, k3): the radial columns are J_u[k_i] = fx*x'*rho^i,
// J_v[k_i] = fy*y'*rho^i (i = 1, 2, 3), so -- as for Kannala-Brandt -- every product with a radial
// column factors through the powers of rho and H[k_i,k_j] depends on i+j only (5 power sums instead
// of 6 x 2 FMAs).  The tangential columns J_u[p1] = 2 fx x'y', J_u[p2] = fx (rho + 2x'^2),
// J_v[p1] = fy (rho + 2y'^2), J_v[p2] = 2 fy x'y' are accumulated as raw moments of
// xy = x'y', tx = rho + 2x'^2, ty = rho + 2y'^2; the constant factors (fx, 2fx, fy, 2fy and their
// products) are applied once in unpack() from the parameter vector the pass was evaluated at.
// 97 FP64 instructions per point instead of 112; invalid points are folded in by zeroing x', y' and
// the residuals (4 selects), which zeroes every term except the count.
template <> struct LinOps<ACM_MODEL_RADTAN, ACM_RESIDUAL_PIXEL> {
    static constexpr int ND = 5, P = 9;
    static constexpr int HFF = 0, HFC = 2, GF = 4, GC = 6, HFK = 8 /*[2][3]*/, HFP = 14 /*mx*xy, mx*tx, my*ty, my*xy*/, HCK = 18 /*[2][3]*/,
                         HCP = 24 /*xy, tx, ty*/, GK = 27 /*[3]*/, GP = 30 /*xy*ru, tx*ru, ty*rv, xy*rv*/, SKK = 34 /*rho^2..rho^6*/,
                         SKP = 39 /*[2][3]*/, PP = 45 /*xy^2, tx^2, ty^2, xy*tx, xy*ty*/, COST = 50, COUNT = 51, NACC = 52;
    static __device__ __forceinline__ void point(double* acc, const LinParams& p, double x, double y, double z, double u, double v) {
        const double k1 = p.d[0], k2 = p.d[1], k3 = p.d[4];
        const double p1x2 = p.d[2] + p.d[2], p2x2 = p.d[3] + p.d[3];            // loop-invariant
        const double fx2 = p.fx + p.fx, fy2 = p.fy + p.fy;                      // loop-invariant
        const bool ok = z >= LIN_SQRT_EPS;  // rad_tan.rs:307-309
        const double iz = fast_rcp(z);
        double xp = x * iz, yp = y * iz;
        xp = ok ? xp : 0.0; yp = ok ? yp : 0.0;
        const double xx = xp * xp, xy = xp * yp;
        const double rho = fma(yp, yp, xx), rho2 = rho * rho, rho3 = rho2 * rho;
        const double rad = fma(k3, rho3, fma(k2, rho2, fma(k1, rho, 1.0)));
        const double tx = fma(2.0, xx, rho), ty = fma(4.0, rho, -tx);           // rho + 2x'^2, rho + 2y'^2
        const double mx = fma(p.d[3], tx, fma(p1x2, xy, xp * rad));
        const double my = fma(p2x2, xy, fma(p.d[2], ty, yp * rad));
        double ru = fma(p.fx, mx, p.cx - u), rv = fma(p.fy, my, p.cy - v);
        ru = ok ? ru : 0.0; rv = ok ? rv : 0.0;
        acc[HFF] = fma(mx, mx, acc[HFF]); acc[HFF + 1] = fma(my, my, acc[HFF + 1]);
        acc[HFC] += mx; acc[HFC + 1] += my;
        acc[GF] = fma(mx, ru, acc[GF]); acc[GF + 1] = fma(my, rv, acc[GF + 1]);
        acc[GC] += ru; acc[GC + 1] += rv;
        const double X = p.fx * xp, Y = p.fy * yp;
        const double a = mx * X, b = my * Y, c = fma(X, ru, Y * rv), w = fma(X, X, Y * Y);
        const double e1 = fma(xy, fx2 * X, ty * (p.fy * Y));   // J_u[k]J_u[p1] + J_v[k]J_v[p1] without the rho power
        const double e2 = fma(tx, p.fx * X, xy * (fy2 * Y));   // ... p2
        const double r[3] = {rho, rho2, rho3};
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            acc[HFK + k] = fma(a, r[k], acc[HFK + k]);
            acc[HFK + 3 + k] = fma(b, r[k], acc[HFK + 3 + k]);
            acc[HCK + k] = fma(X, r[k], acc[HCK + k]);
            acc[HCK + 3 + k] = fma(Y, r[k], acc[HCK + 3 + k]);
            acc[GK + k] = fma(c, r[k], acc[GK + k]);
            acc[SKP + k] = fma(e1, r[k], acc[SKP + k]);
            acc[SKP + 3 + k] = fma(e2, r[k], acc[SKP + 3 + k]);
        }
        const double wr = w * rho, wr3 = wr * rho2;
        acc[SKK + 0] = fma(wr, rho, acc[SKK + 0]);    // rho^2
        acc[SKK + 1] = fma(wr, rho2, acc[SKK + 1]);   // rho^3
        acc[SKK + 2] = fma(wr, rho3, acc[SKK + 2]);   // rho^4
        acc[SKK + 3] = fma(wr3, rho2, acc[SKK + 3]);  // rho^5
        acc[SKK + 4] = fma(wr3, rho3, acc[SKK + 4]);  // rho^6
        acc[HFP + 0] = fma(mx, xy, acc[HFP + 0]); acc[HFP + 1] = fma(mx, tx, acc[HFP + 1]);
        acc[HFP + 2] = fma(my, ty, acc[HFP + 2]); acc[HFP + 3] = fma(my, xy, acc[HFP + 3]);
        acc[HCP + 0] += xy; acc[HCP + 1] += tx; acc[HCP + 2] += ty;
        acc[GP + 0] = fma(xy, ru, acc[GP + 0]); acc[GP + 1] = fma(tx, ru, acc[GP + 1]);
        acc[GP + 2] = fma(ty, rv, acc[GP + 2]); acc[GP + 3] = fma(xy, rv, acc[GP + 3]);
        acc[PP + 0] = fma(xy, xy, acc[PP + 0]); acc[PP + 1] = fma(tx, tx, acc[PP + 1]); acc[PP + 2] = fma(ty, ty, acc[PP + 2]);
        acc[PP + 3] = fma(xy, tx, acc[PP + 3]); acc[PP + 4] = fma(xy, ty, acc[PP + 4]);
        acc[COST] = fma(ru, ru, fma(rv, rv, acc[COST]));
        acc[COUNT] += ok ? 1.0 : 0.0;
    }
    // parameter index of k1, k2, p1, p2, k3 = 4, 5, 6, 7, 8; radial power i = 1, 2, 3 <-> k1, k2, k3
    template <bool FULL = true>
    __host__ __device__ static void unpack(const double* __restrict__ r, const double* __restrict__ x, double* __restrict__ H, double* __restrict__ g, double* __restrict__ cost, double* __restrict__ count) {
        const double fx = x[0], fy = x[1];
        const int KI[3] = {4, 5, 8};
        if (FULL) for (int i = 0; i < P * P; ++i) H[i] = 0.0;
        const double cnt = r[COUNT];
        H[0 * P + 0] = r[HFF]; H[1 * P + 1] = r[HFF + 1];
        H[0 * P + 2] = r[HFC]; H[1 * P + 3] = r[HFC + 1];
        H[2 * P + 2] = cnt; H[3 * P + 3] = cnt;
        for (int i = 0; i < 3; ++i) {
            H[0 * P + KI[i]] = r[HFK + i]; H[1 * P + KI[i]] = r[HFK + 3 + i];
            H[2 * P + KI[i]] = r[HCK + i]; H[3 * P + KI[i]] = r[HCK + 3 + i];
            g[KI[i]] = r[GK + i];
            for (int j = i; j < 3; ++j) H[KI[i] * P + KI[j]] = r[SKK + i + j];
            // radial x tangential; (k1|k2, p*) sit above the diagonal, (p*, k3) too
            const int lo1 = KI[i] < 6 ? KI[i] : 6, hi1 = KI[i] < 6 ? 6 : KI[i];
            const int lo2 = KI[i] < 7 ? KI[i] : 7, hi2 = KI[i] < 7 ? 7 : KI[i];
            H[lo1 * P + hi1] = r[SKP + i];
            H[lo2 * P + hi2] = r[SKP + 3 + i];
        }
        H[0 * P + 6] = 2.0 * fx * r[HFP + 0]; H[0 * P + 7] = fx * r[HFP + 1];
        H[1 * P + 6] = fy * r[HFP + 2];       H[1 * P + 7] = 2.0 * fy * r[HFP + 3];
        H[2 * P + 6] = 2.0 * fx * r[HCP + 0]; H[2 * P + 7] = fx * r[HCP + 1];
        H[3 * P + 6] = fy * r[HCP + 2];       H[3 * P + 7] = 2.0 * fy * r[HCP + 0];
        g[6] = 2.0 * fx * r[GP + 0] + fy * r[GP + 2];
        g[7] = fx * r[GP + 1] + 2.0 * fy * r[GP + 3];
        H[6 * P + 6] = 4.0 * fx * fx * r[PP + 0] + fy * fy * r[PP + 2];
        H[6 * P + 7] = 2.0 * fx * fx * r[PP + 3] + 2.0 * fy * fy * r[PP + 4];
        H[7 * P + 7] = fx * fx * r[PP + 1] + 4.0 * fy * fy * r[PP + 0];
        g[0] = r[GF]; g[1] = r[GF + 1]; g[2] = r[GC]; g[3] = r[GC + 1];
        if (FULL) for (int a = 0; a < P; ++a) for (int b = 0; b < a; ++b) H[a * P + b] = H[b * P + a];
        *cost = 0.5 * r[COST];
        *count = cnt;
    }
};

// ---------------------------------------------------------------------------------------
// Double Sphere, pixel residual (the headline kernel): 68 FP64 instructions per point instead of the generic 77.
//
// Precision budget.  The residual needs full precision: near the minimiser ru, rv are ~0.01 px, and an error of 2^-46 in
// 1/den or d1 moves fx*mx by ~1e-11 px, a cost error of ~1e-9 relative.  So:
//   * everything that feeds ru, rv or the validity tests stays within a few ulp: d1 and d2 (<= 1 ulp, a Heron step with
//     the exact fma residual), g (one fma, as before), den, 1/den (<= 1 ulp), mx and my (one product each);
//   * quantities that only feed Jacobian columns may carry ~2^-44 relative error: h ~ 1/(2 d2) (one Goldschmidt step, the
//     same order as the one Newton step of the generic form's 1/d2), hence dd1, cu and cv;
//   * dd0 = d2 - g keeps its form (the oracle computes it so, and it cancels for points near the axis).
// Where the instructions went (generic form -> this one, per point):
//   * d1 = sqrt(x^2 + y^2 + z^2): 8 -> 5.  Seed s ~ 1/sqrt(a), h0 = s/2 by an exponent decrement (an integer add, off the
//     FP64 pipe; s is normal, or inf / 0 / NaN for a degenerate point, whose g0 = a s is then NaN as before), one coupled
//     Goldschmidt step on g ~ sqrt(a) only, then Heron with h0: its error is ~1.5 e0^3 (e0 the seed's) before the last
//     rounding, far under 2^-53, so d1 is within 1 ulp.
//   * d2 = sqrt(g^2 + x^2 + y^2): 8 -> 6, the same with h refined too; h feeds dd1 = d1 (1 + alpha (2 g h - 1)), written
//     so that no loop-invariant 1 - alpha or 2 alpha is recomputed in the loop (the one-pass kernel reads alpha from the
//     constant bank, and ptxas rematerialises such values rather than keep them in registers).
//   * den = alpha d2 + (1 - alpha) g = g + alpha dd0: 2 -> 1 (dd0 is needed anyway).  Correctly rounded when g >= d2/2 (dd0
//     is then exact, Sterbenz); otherwise an absolute error of ~1 ulp of max(d2, |g|), as in the two-product form.
//   * 1/den: one Newton step with the cubic term, r (1 + e + e^2), e = 1 - den r: error e^3 ~ 2^-66 before the last
//     rounding, <= 1 ulp, in 3 fma instead of 4.
//   * accumulation: every distortion entry is cu dd_k or cv dd_k (cu = d(u)/d(den)), so the products with them factor:
//       H[f,d_k] = sum (mx cu) dd_k   H[c,d_k] = sum cu dd_k   g[d_k] = sum (cu ru + cv rv) dd_k
//       H[d_j,d_k] = sum (cu^2 + cv^2) dd_j dd_k
//     30 FP64 instructions instead of 33 with the count: the valid points are counted in an int in the loop
//     (point(acc, count, ...)) that the kernel converts once, exactly.
// Invalid points are folded in by selects on mx, my, ru, rv, cu, cv and both dd_k: a rejected point can carry NaN in any of
// them, and every accumulated term is a product of those.
// ---------------------------------------------------------------------------------------
// y * 2^e for a normal y and a normal result, by an integer add to the exponent field instead of a DMUL.
__device__ __forceinline__ double lin_scale2(double y, int e) { return __hiloint2double(__double2hiint(y) + (e << 20), __double2loint(y)); }

template <> struct LinOps<ACM_MODEL_DOUBLE_SPHERE, ACM_RESIDUAL_PIXEL> {
    static constexpr int ND = 2, P = 6;
    static constexpr bool INT_COUNT = true;
    // HFD / HCD: u-row d0, u-row d1, v-row d0, v-row d1; HDD: d0 d0, d0 d1, d1 d1
    static constexpr int HFF = 0, HFC = 2, GF = 4, GC = 6, HFD = 8, HCD = 12, GD = 16, HDD = 18, COST = 21, COUNT = 22, NACC = 23;
    static __device__ __forceinline__ void point(double* acc, int& count, const LinParams& p, double x, double y, double z, double u, double v) {
        const double alpha = p.d[0], xi = p.d[1];
        const double nk0 = -p.k0;
        const double rr = fma(y, y, x * x);
        const double a1 = fma(z, z, rr);
        double s, h, g, r;
        asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(s) : "d"(a1));
        h = lin_scale2(s, -1); g = a1 * s;
        r = fma(-g, h, 0.5);
        g = fma(g, r, g);
        const double d1 = fma(fma(-g, g, a1), h, g);
        const double gz = fma(xi, d1, z);
        const double q = fma(gz, gz, rr);
        asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(s) : "d"(q));
        h = lin_scale2(s, -1); g = q * s;
        r = fma(-g, h, 0.5);
        g = fma(g, r, g); h = fma(h, r, h);
        const double d2 = fma(fma(-g, g, q), h, g);
        double dd0 = d2 - gz;
        const double den = fma(alpha, dd0, gz);
        double dd1 = d1 * fma(alpha, fma(gz, lin_scale2(h, 1), -1.0), 1.0);   // d1 (1 - alpha + alpha g / d2)
        const bool ok = (den >= LIN_PRECISION) && (z > nk0 * d1);
        double inv;
        asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(inv) : "d"(den));
        const double e = fma(-den, inv, 1.0);
        inv = fma(inv, fma(e, e, e), inv);
        double mx = x * inv, my = y * inv;
        double ru = fma(p.fx, mx, p.cx) - u, rv = fma(p.fy, my, p.cy) - v;
        double cu = -(p.fx * mx) * inv, cv = -(p.fy * my) * inv;   // d(u)/d(den), d(v)/d(den)
        mx = ok ? mx : 0.0; my = ok ? my : 0.0; ru = ok ? ru : 0.0; rv = ok ? rv : 0.0;
        cu = ok ? cu : 0.0; cv = ok ? cv : 0.0; dd0 = ok ? dd0 : 0.0; dd1 = ok ? dd1 : 0.0;
        acc[HFF] = fma(mx, mx, acc[HFF]); acc[HFF + 1] = fma(my, my, acc[HFF + 1]);
        acc[HFC] += mx; acc[HFC + 1] += my;
        acc[GF] = fma(mx, ru, acc[GF]); acc[GF + 1] = fma(my, rv, acc[GF + 1]);
        acc[GC] += ru; acc[GC + 1] += rv;
        const double a = mx * cu, b = my * cv, c = fma(cu, ru, cv * rv), w = fma(cu, cu, cv * cv);
        const double dd[2] = {dd0, dd1};
#pragma unroll
        for (int k = 0; k < 2; ++k) {
            acc[HFD + k] = fma(a, dd[k], acc[HFD + k]);
            acc[HFD + 2 + k] = fma(b, dd[k], acc[HFD + 2 + k]);
            acc[HCD + k] = fma(cu, dd[k], acc[HCD + k]);
            acc[HCD + 2 + k] = fma(cv, dd[k], acc[HCD + 2 + k]);
            acc[GD + k] = fma(c, dd[k], acc[GD + k]);
        }
        const double wd0 = w * dd0, wd1 = w * dd1;
        acc[HDD + 0] = fma(wd0, dd0, acc[HDD + 0]);
        acc[HDD + 1] = fma(wd0, dd1, acc[HDD + 1]);
        acc[HDD + 2] = fma(wd1, dd1, acc[HDD + 2]);
        acc[COST] = fma(ru, ru, fma(rv, rv, acc[COST]));
        count += ok;
    }
    template <bool FULL = true>
    __host__ __device__ static void unpack(const double* __restrict__ r, const double* __restrict__ x, double* __restrict__ H, double* __restrict__ g, double* __restrict__ cost, double* __restrict__ count) {
        (void)x;
        if (FULL) for (int i = 0; i < P * P; ++i) H[i] = 0.0;
        const double cnt = r[COUNT];
        H[0 * P + 0] = r[HFF]; H[1 * P + 1] = r[HFF + 1];
        H[0 * P + 2] = r[HFC]; H[1 * P + 3] = r[HFC + 1];
        H[2 * P + 2] = cnt; H[3 * P + 3] = cnt;
        for (int k = 0; k < 2; ++k) {
            H[0 * P + 4 + k] = r[HFD + k]; H[1 * P + 4 + k] = r[HFD + 2 + k];
            H[2 * P + 4 + k] = r[HCD + k]; H[3 * P + 4 + k] = r[HCD + 2 + k];
            g[4 + k] = r[GD + k];
        }
        H[4 * P + 4] = r[HDD]; H[4 * P + 5] = r[HDD + 1]; H[5 * P + 5] = r[HDD + 2];
        g[0] = r[GF]; g[1] = r[GF + 1]; g[2] = r[GC]; g[3] = r[GC + 1];
        if (FULL) for (int a = 0; a < P; ++a) for (int b = 0; b < a; ++b) H[a * P + b] = H[b * P + a];
        *cost = 0.5 * r[COST];
        *count = cnt;
    }
};

// What the streaming kernel calls per point: ops.point(acc, ...), or ops.point(acc, count, ...) for the specialisations
// that count valid points in an int (INT_COUNT = true); the kernel stores that count into acc[COUNT] once after its loop.
template <class Ops, class = void> struct LinIntCount { static constexpr bool value = false; };
template <class Ops> struct LinIntCount<Ops, std::void_t<decltype(Ops::INT_COUNT)>> { static constexpr bool value = Ops::INT_COUNT; };
template <class Ops>
__device__ __forceinline__ void lin_point(double* acc, int& count, const LinParams& p, double x, double y, double z, double u, double v) {
    if constexpr (LinIntCount<Ops>::value) Ops::point(acc, count, p, x, y, z, u, v);
    else Ops::point(acc, p, x, y, z, u, v);
}
