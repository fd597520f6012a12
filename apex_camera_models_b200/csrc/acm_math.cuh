// Branch-free f64 helpers shared by every translation unit.  Written with explicit __fma_rn /
// __dmul_rn / __dadd_rn intrinsics so that they compile to the same instructions with and without
// -fmad=false.
#pragma once
#include <cuda_runtime.h>

// 1/a for normal finite a: MUFU seed (~2^-23) + two Newton steps => <= 1 ulp.
__device__ __forceinline__ double acm_rcp(double a) {
    double r;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(a));
    double e = __fma_rn(-a, r, 1.0);
    r = __fma_rn(r, e, r);
    e = __fma_rn(-a, r, 1.0);
    return __fma_rn(r, e, r);
}

// 1/sqrt(a) for normal finite a > 0: MUFU seed + two Newton steps => <= 2 ulp.
__device__ __forceinline__ double acm_rsqrt(double a) {
    double y;
    asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(a));
    const double h = __dmul_rn(0.5, a);
    y = __dmul_rn(y, __fma_rn(-h, __dmul_rn(y, y), 1.5));
    return __dmul_rn(y, __fma_rn(-h, __dmul_rn(y, y), 1.5));
}

// sqrt(a) (<= 1 ulp) and 1/sqrt(a) (<= 2 ulp) together: two coupled Goldschmidt iterations on
// g ~ sqrt(a), h ~ 1/(2 sqrt(a)):  r = 1/2 - g h,  g += g r,  h += h r.  2 DMUL + 6 DFMA + 1 DADD.
// a = 0 returns 0 (inv = NaN is never used then); a < 0 and NaN give NaN like sqrt().
__device__ __forceinline__ double acm_sqrt_inv(double a, double& inv) {
    double y;
    asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(a));
    double g = __dmul_rn(a, y), h = __dmul_rn(0.5, y);
    double r = __fma_rn(-g, h, 0.5);
    g = __fma_rn(g, r, g); h = __fma_rn(h, r, h);
    r = __fma_rn(-g, h, 0.5);
    g = __fma_rn(g, r, g); h = __fma_rn(h, r, h);
    inv = __dadd_rn(h, h);
    return a == 0.0 ? 0.0 : g;
}

// Correctly rounded a / b from the correctly rounded reciprocal ib = RN(1/b) (Markstein: q = RN(a ib)
// is within 1 ulp of a/b, the fma residual r = a - q b is exact, and RN(q + r ib) is then the correctly
// rounded quotient): 3 FP64 instructions and no slow-path call instead of ~10 + a branch.  The result is
// BIT-IDENTICAL to a / b, so it may feed the bit-exact validity tests.  Valid while nothing under- or
// overflows: the caller guarantees 2^-100 <= |b| <= 2^100 (host flag CamParams::fast_div, or
// acm_exp_ok(b)); numerators outside [2^-895, 2^897] -- including 0, whose sign the fma chain would
// lose -- take the IEEE division (an integer test on the exponent field, off the FP64 pipe).
// Checked against a / b on 1e9 random and adversarial (near-tie, all-ones mantissa) operand pairs on the CPU.
__device__ __forceinline__ bool acm_exp_ok(double b) {  // 2^-100 <= |b| < 2^101
    const unsigned e = ((unsigned)__double2hiint(b) >> 20) & 0x7ffu;
    return e - 923u <= 200u;
}
__device__ __forceinline__ double acm_div_by(double a, double b, double ib) {
    const unsigned e = ((unsigned)__double2hiint(a) >> 20) & 0x7ffu;
    if (e - 128u >= 1792u) return a / b;
    const double q = __dmul_rn(a, ib);
    const double r = __fma_rn(-q, b, a);
    return __fma_rn(r, ib, q);
}

// sin and cos for 0 <= x <= ~1.8 (the Newton root of the Kannala-Brandt unprojection): x > pi/4 is reflected to
// y = pi/2 - x (two-term pi/2), then the classic minimax kernels on [-pi/4, pi/4] (degree 13 / 14, < 1 ulp).
// ~24 FP64 instructions, no branch, no slow path; used only behind the last validity test.
static __constant__ double ACM_SINCOS_C[12] = {
    -1.66666666666666324348e-01, 8.33333333332248946124e-03, -1.98412698298579493134e-04,
    2.75573137070700676789e-06, -2.50507602534068634195e-08, 1.58969099521155010221e-10,
    4.16666666666666019037e-02, -1.38888888888741095749e-03, 2.48015872894767294178e-05,
    -2.75573143513906633035e-07, 2.08757232129817482790e-09, -1.13596475577881948265e-11};
__device__ __forceinline__ void acm_sincos_small(double x, double& s, double& c) {
    const bool refl = x > 0.78539816339744828;
    const double y = refl ? __dadd_rn(__dsub_rn(1.5707963267948966, x), 6.123233995736766e-17) : x;
    const double z = __dmul_rn(y, y);
    double ps = ACM_SINCOS_C[5], pc = ACM_SINCOS_C[11];
#pragma unroll
    for (int k = 4; k >= 0; --k) { ps = __fma_rn(ps, z, ACM_SINCOS_C[k]); pc = __fma_rn(pc, z, ACM_SINCOS_C[6 + k]); }
    const double sy = __fma_rn(__dmul_rn(y, z), ps, y);                                   // y + y^3 S(z)
    const double cy = __fma_rn(__dmul_rn(z, z), pc, __fma_rn(-0.5, z, 1.0));              // 1 - z/2 + z^2 C(z)
    s = refl ? cy : sy;
    c = refl ? sy : cy;
}

// atan2(a, b) for a >= 0, b > 0 (first quadrant: all that the fisheye models need).  Two argument
// reductions share ONE reciprocal -- swap so that t = num/den <= 1, then
// atan(t) = pi/4 + atan((num-den)/(num+den)) above tan(pi/8) -- leaving |t| <= sqrt(2)-1, where a
// degree-10 polynomial in t^2 (Chebyshev-node fit computed with mpmath at 60 digits, approximation
// error 6.9e-17 relative) is evaluated by Horner.  Total error <= ~1.5 ulp, like the CUDA library's
// atan2 (2 ulp), in ~25 FP64 instructions with no branch and no slow-path call.
// Operands whose magnitude would push the MUFU seed into its flush-to-zero range take the library
// function (a branch that is practically never taken; GUARD = false drops it for the solver kernels,
// whose streaming loop must stay one basic block and whose inputs are sane by construction).
// The coefficients live in the constant bank: DFMA then reads them as c[bank][offset] operands,
// whereas 64-bit literals are re-materialised (two UMOV / IMAD.MOV each) inside the streaming loops.
static __constant__ double ACM_ATAN_C[14] = {
    2.11353731576932463e-02, -4.34805221571646222e-02, 5.68834922680901064e-02, -6.64023393042940807e-02,
    7.68995349630685748e-02, -9.09077307480841423e-02, 1.11111061804559458e-01, -1.42857141809764665e-01,
    1.99999999988551114e-01, -3.33333333333284410e-01,
    0.41421356237309503 /* tan(pi/8) */, 0.78539816339744828 /* pi/4 */, 1.5707963267948966 /* pi/2 */, 0.0};

template <bool GUARD = true>
__device__ __forceinline__ double acm_atan2_q1(double a, double b) {
    const bool swap = a > b;
    const double num = swap ? b : a, den = swap ? a : b;
    if (GUARD && !(den > 1e-280 && den < 1e280)) return atan2(a, b);
    const bool hi = num > __dmul_rn(ACM_ATAN_C[10], den);
    const double n2 = hi ? __dsub_rn(num, den) : num;
    const double d2 = hi ? __dadd_rn(num, den) : den;
    const double t = __dmul_rn(n2, acm_rcp(d2));
    const double s = __dmul_rn(t, t);
    // Horner: an Estrin split (depth 4 instead of 9, +2 instructions) measured 4 % SLOWER in the KB / FOV linearize
    // kernels (same-box A/B): with two points per thread and 12 warps per SM the chain is already hidden.
    double q = ACM_ATAN_C[0];
#pragma unroll
    for (int k = 1; k < 10; ++k) q = __fma_rn(q, s, ACM_ATAN_C[k]);
    double at = __fma_rn(__dmul_rn(t, s), q, t);
    at = hi ? __dadd_rn(ACM_ATAN_C[11], at) : at;
    return swap ? __dsub_rn(ACM_ATAN_C[12], at) : at;
}
