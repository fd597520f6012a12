// Batched project / unproject / undistort / synthetic-input kernels.
// Compiled with -fmad=false so that every +,-,*,/,sqrt is a separately rounded IEEE binary64
// operation exactly as in the reference (Rust never fuses): status masks and remap indices
// are bit-exact, f64 coordinates differ from the reference only through the <= 2 ulp device
// atan2 / sin / cos.
//
// Data movement (HBM-bound kernels): SoA components, one 16-byte vector load per component
// per thread (2 f64 or 4 f32 points), grid-stride loop over a grid of sm_count * k blocks.
#include <stdlib.h>

#include <cmath>
#include <cstring>
#include <new>
#include <type_traits>

#include <cuda.h>

#include "acm_models.cuh"

// ---------------------------------------------------------------------------------------
// 16-byte packets of points
// ---------------------------------------------------------------------------------------
template <typename T> struct Vec;
template <> struct Vec<double> {
    static constexpr int N = 2;
    using type = double2;
    static __device__ __forceinline__ void unpack(const double2& v, double* o) { o[0] = v.x; o[1] = v.y; }
    static __device__ __forceinline__ double2 pack(const double* o) { return make_double2(o[0], o[1]); }
};
template <> struct Vec<float> {
    static constexpr int N = 4;
    using type = float4;
    static __device__ __forceinline__ void unpack(const float4& v, double* o) { o[0] = v.x; o[1] = v.y; o[2] = v.z; o[3] = v.w; }
    static __device__ __forceinline__ float4 pack(const double* o) { return make_float4((float)o[0], (float)o[1], (float)o[2], (float)o[3]); }
};

template <typename V> __device__ __forceinline__ V ld_stream(const V* p) { return __ldcs(p); }
template <typename V> __device__ __forceinline__ void st_stream(V* p, const V& v) { __stcs(p, v); }

template <int NV> struct StatusVec;
template <> struct StatusVec<2> {
    static __device__ __forceinline__ void store(uint8_t* p, const int* s) {
        __stcs(reinterpret_cast<uchar2*>(p), make_uchar2((uint8_t)s[0], (uint8_t)s[1]));
    }
};
template <> struct StatusVec<4> {
    static __device__ __forceinline__ void store(uint8_t* p, const int* s) {
        __stcs(reinterpret_cast<uchar4*>(p), make_uchar4((uint8_t)s[0], (uint8_t)s[1], (uint8_t)s[2], (uint8_t)s[3]));
    }
};

// ---------------------------------------------------------------------------------------
// project: xyz -> uv + status
// ---------------------------------------------------------------------------------------
// Streaming variant per (kernel, model), chosen by same-box A/B on 100 M f64 points (scripts/ab_pu.sh).
// PIPE = software-pipelined: the packet of the next iteration is in flight while this one is evaluated, with
// __launch_bounds__(256, 3) so that the extra registers do not cost a resident block (uncapped, the pipelined
// kernels grew to 70-100 registers and lost 5-10 %).  ncu had these kernels on long_scoreboard with DRAM at
// 60-70 % of its peak.  GB/s plain -> pipelined (same box): project RadTan 5808 -> 6165, KB 5308 -> 5760,
// DS 6000 -> 6130 (Pinhole, UCM, EUCM, FOV are at 5.8-6.5 TB/s plain and lose 2-5 % pipelined); unproject
// DS 5125 -> 5590, UCM 5680 -> 5930, EUCM 5625 -> 5850, Pinhole 5730 -> 5935, FOV 5280 -> 5470 (KB, RadTan: Newton
// loops, unchanged); round trip DS 4500 -> 5220, Pinhole 5815 -> 6025 (the others are not faster pipelined).
// The plain variants keep an unspecified minimum block count: `__launch_bounds__(256, 1)` lets ptxas grow them
// past 64 registers, which costs a resident block and 10-15 %.
enum { PU_PROJECT = 0, PU_UNPROJECT = 1, PU_ROUND_TRIP = 2 };
template <int KERNEL, int M> struct PuStream { static constexpr bool PIPE = false; };
template <> struct PuStream<PU_PROJECT, ACM_MODEL_RADTAN> { static constexpr bool PIPE = true; };
template <> struct PuStream<PU_PROJECT, ACM_MODEL_KANNALA_BRANDT> { static constexpr bool PIPE = true; };
template <> struct PuStream<PU_PROJECT, ACM_MODEL_DOUBLE_SPHERE> { static constexpr bool PIPE = true; };
template <int M> struct PuStream<PU_UNPROJECT, M> { static constexpr bool PIPE = M != ACM_MODEL_RADTAN; };
template <> struct PuStream<PU_ROUND_TRIP, ACM_MODEL_PINHOLE> { static constexpr bool PIPE = true; };
template <> struct PuStream<PU_ROUND_TRIP, ACM_MODEL_DOUBLE_SPHERE> { static constexpr bool PIPE = true; };
template <int M, typename T, bool BOUNDS>
__global__ void __launch_bounds__(256, (PuStream<PU_PROJECT, M>::PIPE ? 3 : 0)) project_kernel(const __grid_constant__ CamParams c, const T* __restrict__ X,
                                                      const T* __restrict__ Y, const T* __restrict__ Z, T* __restrict__ U,
                                                      T* __restrict__ V, uint8_t* __restrict__ S, size_t n) {
    using VT = typename Vec<T>::type;
    constexpr int NV = Vec<T>::N;
    const size_t npk = n / NV;
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    constexpr bool PIPE = PuStream<PU_PROJECT, M>::PIPE;
    const VT* X4 = reinterpret_cast<const VT*>(X); const VT* Y4 = reinterpret_cast<const VT*>(Y); const VT* Z4 = reinterpret_cast<const VT*>(Z);
    auto packet = [&](size_t p, const VT& vx, const VT& vy, const VT& vz) {
        double x[NV], y[NV], z[NV], u[NV], v[NV];
        int s[NV];
        Vec<T>::unpack(vx, x);
        Vec<T>::unpack(vy, y);
        Vec<T>::unpack(vz, z);
#pragma unroll
        for (int k = 0; k < NV; ++k) {
            u[k] = v[k] = acm_nan();
            double uu, vv;
            s[k] = CamModel<M>::template project<BOUNDS, true>(c, x[k], y[k], z[k], uu, vv);
            if (s[k] == ACM_POINT_OK) { u[k] = uu; v[k] = vv; }
        }
        st_stream(reinterpret_cast<VT*>(U) + p, Vec<T>::pack(u));
        st_stream(reinterpret_cast<VT*>(V) + p, Vec<T>::pack(v));
        if (S) StatusVec<NV>::store(S + p * NV, s);
    };
    if constexpr (PIPE) {
        size_t p = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
        VT px, py, pz;
        if (p < npk) { px = ld_stream(X4 + p); py = ld_stream(Y4 + p); pz = ld_stream(Z4 + p); }
        while (p < npk) {
            const size_t pn = p + stride;
            VT nx = px, ny = py, nz = pz;
            if (pn < npk) { nx = ld_stream(X4 + pn); ny = ld_stream(Y4 + pn); nz = ld_stream(Z4 + pn); }
            packet(p, px, py, pz);
            px = nx; py = ny; pz = nz; p = pn;
        }
    } else {
        for (size_t p = (size_t)blockIdx.x * blockDim.x + threadIdx.x; p < npk; p += stride)
            packet(p, ld_stream(X4 + p), ld_stream(Y4 + p), ld_stream(Z4 + p));
    }
    // ragged tail (n not a multiple of the packet width)
    const size_t t = npk * NV + (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t < n) {
        double uu, vv;
        int st = CamModel<M>::template project<BOUNDS, true>(c, (double)X[t], (double)Y[t], (double)Z[t], uu, vv);
        if (st != ACM_POINT_OK) uu = vv = acm_nan();
        U[t] = (T)uu; V[t] = (T)vv;
        if (S) S[t] = (uint8_t)st;
    }
}

// ---------------------------------------------------------------------------------------
// unproject: uv -> ray + status
// ---------------------------------------------------------------------------------------
// resident 256-thread blocks per SM the unproject kernel is compiled for (register cap): 3 with the pipelined stream; the Newton
// models are bound by the latency of their dependent chains: RadTan gains 2.6 % from a 4th block (64 registers), Kannala-Brandt
// nothing (profiles/r02_ab_unproj_occ.log)
template <int M> struct UnprojBounds { static constexpr int MINB = PuStream<PU_UNPROJECT, M>::PIPE ? 3 : 0; };
template <> struct UnprojBounds<ACM_MODEL_RADTAN> { static constexpr int MINB = 4; };
template <> struct UnprojBounds<ACM_MODEL_KANNALA_BRANDT> { static constexpr int MINB = 3; };
template <int M, typename T, bool IEEE = false>
__global__ void __launch_bounds__(256, UnprojBounds<M>::MINB) unproject_kernel(const __grid_constant__ CamParams c, const T* __restrict__ U,
                                                        const T* __restrict__ V, T* __restrict__ X, T* __restrict__ Y,
                                                        T* __restrict__ Z, uint8_t* __restrict__ S, size_t n) {
    using VT = typename Vec<T>::type;
    constexpr int NV = Vec<T>::N;
    const size_t npk = n / NV;
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    constexpr bool PIPE = PuStream<PU_UNPROJECT, M>::PIPE;
    const VT* U4 = reinterpret_cast<const VT*>(U); const VT* V4 = reinterpret_cast<const VT*>(V);
    auto packet = [&](size_t p, const VT& vu, const VT& vv) {
        double u[NV], v[NV], x[NV], y[NV], z[NV];
        int s[NV];
        Vec<T>::unpack(vu, u);
        Vec<T>::unpack(vv, v);
#pragma unroll
        for (int k = 0; k < NV; ++k) {
            x[k] = y[k] = z[k] = acm_nan();
            double rx, ry, rz;
            s[k] = CamModel<M>::template unproject<IEEE>(c, u[k], v[k], rx, ry, rz);
            if (s[k] == ACM_POINT_OK) { x[k] = rx; y[k] = ry; z[k] = rz; }
        }
        st_stream(reinterpret_cast<VT*>(X) + p, Vec<T>::pack(x));
        st_stream(reinterpret_cast<VT*>(Y) + p, Vec<T>::pack(y));
        st_stream(reinterpret_cast<VT*>(Z) + p, Vec<T>::pack(z));
        if (S) StatusVec<NV>::store(S + p * NV, s);
    };
    if constexpr (PIPE) {
        size_t p = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
        VT pu, pv;
        if (p < npk) { pu = ld_stream(U4 + p); pv = ld_stream(V4 + p); }
        while (p < npk) {
            const size_t pn = p + stride;
            VT nu = pu, nv = pv;
            if (pn < npk) { nu = ld_stream(U4 + pn); nv = ld_stream(V4 + pn); }
            packet(p, pu, pv);
            pu = nu; pv = nv; p = pn;
        }
    } else {
        for (size_t p = (size_t)blockIdx.x * blockDim.x + threadIdx.x; p < npk; p += stride)
            packet(p, ld_stream(U4 + p), ld_stream(V4 + p));
    }
    const size_t t = npk * NV + (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t < n) {
        double rx, ry, rz;
        int st = CamModel<M>::template unproject<IEEE>(c, (double)U[t], (double)V[t], rx, ry, rz);
        if (st != ACM_POINT_OK) rx = ry = rz = acm_nan();
        X[t] = (T)rx; Y[t] = (T)ry; Z[t] = (T)rz;
        if (S) S[t] = (uint8_t)st;
    }
}

template <int M, typename T>
static int32_t launch_project(acm_ctx* ctx, const CamParams& c, const acm_points* xyz, acm_points* uv, uint8_t* st) {
    const size_t n = xyz->n;
    if (n == 0) return ACM_OK;
    constexpr int NV = Vec<T>::N;
    int grid = grid_for(ctx, n / NV + NV, 256, 8);
    project_kernel<M, T, true><<<grid, 256, 0, ctx->stream>>>(c, comp<T>(xyz, 0), comp<T>(xyz, 1), comp<T>(xyz, 2),
                                                                comp<T>(uv, 0), comp<T>(uv, 1), st, n);
    ACM_CHECK_LAUNCH(ctx);
    return ACM_OK;
}

template <int M, typename T, bool IEEE = false>
static int32_t launch_unproject(acm_ctx* ctx, const CamParams& c, const acm_points* uv, acm_points* xyz, uint8_t* st) {
    const size_t n = uv->n;
    if (n == 0) return ACM_OK;
    constexpr int NV = Vec<T>::N;
    int grid = grid_for(ctx, n / NV + NV, 256, 8);
    unproject_kernel<M, T, IEEE><<<grid, 256, 0, ctx->stream>>>(c, comp<T>(uv, 0), comp<T>(uv, 1), comp<T>(xyz, 0),
                                                           comp<T>(xyz, 1), comp<T>(xyz, 2), st, n);
    ACM_CHECK_LAUNCH(ctx);
    return ACM_OK;
}

// ---------------------------------------------------------------------------------------
// fused round trip: xyz -> uv -> ray (BASELINE config 2)
// ---------------------------------------------------------------------------------------
template <int M, typename T>
__global__ void __launch_bounds__(256, (PuStream<PU_ROUND_TRIP, M>::PIPE ? 3 : 0)) round_trip_kernel(const __grid_constant__ CamParams c, const T* __restrict__ X, const T* __restrict__ Y,
                                                         const T* __restrict__ Z, T* __restrict__ U, T* __restrict__ V, T* __restrict__ RX,
                                                         T* __restrict__ RY, T* __restrict__ RZ, uint8_t* __restrict__ SP,
                                                         uint8_t* __restrict__ SU, size_t n) {
    using VT = typename Vec<T>::type;
    constexpr int NV = Vec<T>::N;
    const size_t npk = n / NV;
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    auto one = [&](double x, double y, double z, double& u, double& v, double& rx, double& ry, double& rz, int& sp, int& su) {
        u = v = rx = ry = rz = acm_nan();
        double uu, vv;
        sp = CamModel<M>::template project<true, true>(c, x, y, z, uu, vv);
        su = sp;
        if (sp == ACM_POINT_OK) {
            u = uu; v = vv;
            if (sizeof(T) == 4) { uu = (double)(float)uu; vv = (double)(float)vv; }  // what the two-kernel path would read back
            double ax, ay, az;
            su = CamModel<M>::unproject(c, uu, vv, ax, ay, az);
            if (su == ACM_POINT_OK) { rx = ax; ry = ay; rz = az; }
        }
    };
    constexpr bool PIPE = PuStream<PU_ROUND_TRIP, M>::PIPE;
    const VT* X4 = reinterpret_cast<const VT*>(X); const VT* Y4 = reinterpret_cast<const VT*>(Y); const VT* Z4 = reinterpret_cast<const VT*>(Z);
    auto packet = [&](size_t p, const VT& vx, const VT& vy, const VT& vz) {
        double x[NV], y[NV], z[NV], u[NV], v[NV], rx[NV], ry[NV], rz[NV];
        int sp[NV], su[NV];
        Vec<T>::unpack(vx, x);
        Vec<T>::unpack(vy, y);
        Vec<T>::unpack(vz, z);
#pragma unroll
        for (int k = 0; k < NV; ++k) one(x[k], y[k], z[k], u[k], v[k], rx[k], ry[k], rz[k], sp[k], su[k]);
        st_stream(reinterpret_cast<VT*>(U) + p, Vec<T>::pack(u));
        st_stream(reinterpret_cast<VT*>(V) + p, Vec<T>::pack(v));
        st_stream(reinterpret_cast<VT*>(RX) + p, Vec<T>::pack(rx));
        st_stream(reinterpret_cast<VT*>(RY) + p, Vec<T>::pack(ry));
        st_stream(reinterpret_cast<VT*>(RZ) + p, Vec<T>::pack(rz));
        if (SP) StatusVec<NV>::store(SP + p * NV, sp);
        if (SU) StatusVec<NV>::store(SU + p * NV, su);
    };
    if constexpr (PIPE) {
        size_t p = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
        VT px, py, pz;
        if (p < npk) { px = ld_stream(X4 + p); py = ld_stream(Y4 + p); pz = ld_stream(Z4 + p); }
        while (p < npk) {
            const size_t pn = p + stride;
            VT nx = px, ny = py, nz = pz;
            if (pn < npk) { nx = ld_stream(X4 + pn); ny = ld_stream(Y4 + pn); nz = ld_stream(Z4 + pn); }
            packet(p, px, py, pz);
            px = nx; py = ny; pz = nz; p = pn;
        }
    } else {
        for (size_t p = (size_t)blockIdx.x * blockDim.x + threadIdx.x; p < npk; p += stride)
            packet(p, ld_stream(X4 + p), ld_stream(Y4 + p), ld_stream(Z4 + p));
    }
    const size_t t = npk * NV + (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t < n) {
        double u, v, rx, ry, rz; int sp, su;
        one((double)X[t], (double)Y[t], (double)Z[t], u, v, rx, ry, rz, sp, su);
        U[t] = (T)u; V[t] = (T)v; RX[t] = (T)rx; RY[t] = (T)ry; RZ[t] = (T)rz;
        if (SP) SP[t] = (uint8_t)sp;
        if (SU) SU[t] = (uint8_t)su;
    }
}

template <int M, typename T>
static int32_t launch_round_trip(acm_ctx* ctx, const CamParams& c, const acm_points* xyz, acm_points* uv, acm_points* ray, uint8_t* sp, uint8_t* su) {
    const size_t n = xyz->n;
    if (n == 0) return ACM_OK;
    constexpr int NV = Vec<T>::N;
    int grid = grid_for(ctx, n / NV + NV, 256, 8);
    round_trip_kernel<M, T><<<grid, 256, 0, ctx->stream>>>(c, comp<T>(xyz, 0), comp<T>(xyz, 1), comp<T>(xyz, 2), comp<T>(uv, 0), comp<T>(uv, 1),
                                                            comp<T>(ray, 0), comp<T>(ray, 1), comp<T>(ray, 2), sp, su, n);
    ACM_CHECK_LAUNCH(ctx);
    return ACM_OK;
}

extern "C" int32_t acm_project_unproject(acm_ctx* ctx, const acm_camera* cam, const acm_points* xyz, acm_points* uv, acm_points* ray,
                                         uint8_t* d_status_project, uint8_t* d_status_unproject) {
    ACM_ENTER(ctx);
    ACM_REQUIRE(ctx, cam && xyz && uv && ray, "acm_project_unproject: null argument");
    ACM_REQUIRE(ctx, xyz->dim == 3 && uv->dim == 2 && ray->dim == 3, "acm_project_unproject: xyz / ray must have dim 3 and uv dim 2");
    ACM_REQUIRE(ctx, xyz->n == uv->n && xyz->n == ray->n, "acm_project_unproject: point counts differ");
    ACM_REQUIRE(ctx, xyz->dtype == uv->dtype && xyz->dtype == ray->dtype, "acm_project_unproject: dtypes differ");
    CamParams c;
    int32_t rc = acm_make_cam_params(ctx, cam, &c);
    if (rc) return rc;
    if (xyz->dtype == ACM_F64) { ACM_DISPATCH_MODEL(cam->model, return (launch_round_trip<M, double>(ctx, c, xyz, uv, ray, d_status_project, d_status_unproject))) }
    else { ACM_DISPATCH_MODEL(cam->model, return (launch_round_trip<M, float>(ctx, c, xyz, uv, ray, d_status_project, d_status_unproject))) }
    return ACM_OK;
}

extern "C" int32_t acm_project(acm_ctx* ctx, const acm_camera* cam, const acm_points* xyz, acm_points* uv, uint8_t* d_status) {
    ACM_ENTER(ctx);
    ACM_REQUIRE(ctx, cam && xyz && uv, "acm_project: null argument");
    ACM_REQUIRE(ctx, xyz->dim == 3 && uv->dim == 2, "acm_project: xyz must have dim 3 and uv dim 2");
    ACM_REQUIRE(ctx, xyz->n == uv->n, "acm_project: point counts differ");
    ACM_REQUIRE(ctx, xyz->dtype == uv->dtype, "acm_project: dtypes of input and output differ");
    CamParams c;
    int32_t rc = acm_make_cam_params(ctx, cam, &c);
    if (rc) return rc;
    if (xyz->dtype == ACM_F64) { ACM_DISPATCH_MODEL(cam->model, return (launch_project<M, double>(ctx, c, xyz, uv, d_status))) }
    else { ACM_DISPATCH_MODEL(cam->model, return (launch_project<M, float>(ctx, c, xyz, uv, d_status))) }
    return ACM_OK;
}

extern "C" int32_t acm_unproject(acm_ctx* ctx, const acm_camera* cam, const acm_points* uv, acm_points* xyz, uint8_t* d_status) {
    ACM_ENTER(ctx);
    ACM_REQUIRE(ctx, cam && xyz && uv, "acm_unproject: null argument");
    ACM_REQUIRE(ctx, xyz->dim == 3 && uv->dim == 2, "acm_unproject: xyz must have dim 3 and uv dim 2");
    ACM_REQUIRE(ctx, xyz->n == uv->n, "acm_unproject: point counts differ");
    ACM_REQUIRE(ctx, xyz->dtype == uv->dtype, "acm_unproject: dtypes of input and output differ");
    CamParams c;
    int32_t rc = acm_make_cam_params(ctx, cam, &c);
    if (rc) return rc;
    if (uv->dtype == ACM_F64) { ACM_DISPATCH_MODEL(cam->model, return (launch_unproject<M, double>(ctx, c, uv, xyz, d_status))) }
    else { ACM_DISPATCH_MODEL(cam->model, return (launch_unproject<M, float>(ctx, c, uv, xyz, d_status))) }
    return ACM_OK;
}

// unproject with IEEE arithmetic to the end (what sample_points uses): statuses as acm_unproject, values
// bit-identical to the reference for the arithmetic-only models (Pinhole, RadTan, UCM, EUCM, Double Sphere)
extern "C" int32_t acm_unproject_ieee(acm_ctx* ctx, const acm_camera* cam, const acm_points* uv, acm_points* xyz, uint8_t* d_status) {
    ACM_ENTER(ctx);
    ACM_REQUIRE(ctx, cam && xyz && uv, "acm_unproject_ieee: null argument");
    ACM_REQUIRE(ctx, xyz->dim == 3 && uv->dim == 2, "acm_unproject_ieee: xyz must have dim 3 and uv dim 2");
    ACM_REQUIRE(ctx, xyz->n == uv->n, "acm_unproject_ieee: point counts differ");
    ACM_REQUIRE(ctx, xyz->dtype == ACM_F64 && uv->dtype == ACM_F64, "acm_unproject_ieee: f64 buffers required");
    CamParams c;
    int32_t rc = acm_make_cam_params(ctx, cam, &c);
    if (rc) return rc;
    ACM_DISPATCH_MODEL(cam->model, return (launch_unproject<M, double, true>(ctx, c, uv, xyz, d_status)))
    return ACM_OK;
}

// ---------------------------------------------------------------------------------------
// Small-batch host form (what a scalar `CameraModel::project(&p)` / `unproject(&uv)` of the trait binds): the points
// sit in mapped pinned host memory in nalgebra's AoS order, one kernel reads them over PCIe and writes the results
// (AoS) and the status bytes straight back -- one launch and one stream synchronisation per call, no allocation, no
// staging copy on the device.  Same device functions as the batch kernels, hence the same bits.
// ---------------------------------------------------------------------------------------
template <int M, bool PROJECT>
__device__ __forceinline__ void small_map_point(const CamParams& c, const double* __restrict__ in, double* __restrict__ out, uint8_t* __restrict__ S, int i);

// done_flag (optional, single-block launches only): after every result of the block is written, thread 0 publishes `seq`
// there (mapped host memory); the host spins on it instead of paying a stream synchronisation (~8 us of driver time).
template <int M, bool PROJECT>
__global__ void __launch_bounds__(128) small_map_kernel(const __grid_constant__ CamParams c, const double* __restrict__ in, double* __restrict__ out,
                                                        uint8_t* __restrict__ S, int n, unsigned long long* done_flag, unsigned long long seq) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) small_map_point<M, PROJECT>(c, in, out, S, i);
    if (done_flag) {
        __threadfence_system();
        __syncthreads();
        if (threadIdx.x == 0) { *reinterpret_cast<volatile unsigned long long*>(done_flag) = seq; __threadfence_system(); }
    }
}

template <int M, bool PROJECT>
__device__ __forceinline__ void small_map_point(const CamParams& c, const double* __restrict__ in, double* __restrict__ out, uint8_t* __restrict__ S, int i) {
    int st;
    if (PROJECT) {
        double u, v;
        st = CamModel<M>::template project<true, true>(c, in[3 * i], in[3 * i + 1], in[3 * i + 2], u, v);
        if (st != ACM_POINT_OK) u = v = acm_nan();
        out[2 * i] = u; out[2 * i + 1] = v;
    } else {
        double x, y, z;
        st = CamModel<M>::template unproject<false>(c, in[2 * i], in[2 * i + 1], x, y, z);
        if (st != ACM_POINT_OK) x = y = z = acm_nan();
        out[3 * i] = x; out[3 * i + 1] = y; out[3 * i + 2] = z;
    }
    S[i] = (uint8_t)st;
}

int32_t acm_small_map(acm_ctx* ctx, const acm_camera* cam, const double* d_in, double* d_out, uint8_t* d_status, int n, bool is_project,
                      unsigned long long* d_done_flag, unsigned long long seq) {
    CamParams c;
    int32_t rc = acm_make_cam_params(ctx, cam, &c);
    if (rc) return rc;
    const int grid = (n + 127) / 128;
    if (grid > 1) d_done_flag = nullptr;   // the flag protocol is for one block
    if (is_project) { ACM_DISPATCH_MODEL(cam->model, (small_map_kernel<M, true><<<grid, 128, 0, ctx->stream>>>(c, d_in, d_out, d_status, n, d_done_flag, seq))) }
    else { ACM_DISPATCH_MODEL(cam->model, (small_map_kernel<M, false><<<grid, 128, 0, ctx->stream>>>(c, d_in, d_out, d_status, n, d_done_flag, seq))) }
    ACM_CHECK_LAUNCH(ctx);
    return ACM_OK;
}

// ---------------------------------------------------------------------------------------
// undistort_image: per output pixel  ray = ((u-cx_t)/fx_t, (v-cy_t)/fy_t, 1) -> project ->
// bilinear / nearest sample (undistort.rs:33-46, :51-105).  Remap plans: the same sample at a
// source coordinate computed once per plan (acm_remap_plan below).
// ---------------------------------------------------------------------------------------
struct Tap {
    int ok;        // sample exists
    int off00;     // byte offset of p00 in a frame
    double wx, wy; // bilinear weights (unused for nearest)
};

__device__ __forceinline__ Tap make_tap(double sx, double sy, int status, int W, int H, int interp) {
    Tap t; t.ok = 0; t.off00 = 0; t.wx = 0.0; t.wy = 0.0;
    if (status != ACM_POINT_OK) return t;
    if (isnan(sx) || isnan(sy)) return t;
    if (interp == ACM_INTERP_NEAREST) {
        double rx = round(sx), ry = round(sy);
        // `as i32` saturates; anything outside [0,W) fails the guard either way
        if (rx >= 0.0 && rx < (double)W && ry >= 0.0 && ry < (double)H) { t.ok = 1; t.off00 = 3 * ((int)ry * W + (int)rx); }
        return t;
    }
    double x0 = floor(sx), y0 = floor(sy);
    double x1 = x0 + 1.0, y1 = y0 + 1.0;
    if (x0 < 0.0 || x1 >= (double)W || y0 < 0.0 || y1 >= (double)H) return t;
    t.ok = 1;
    t.off00 = 3 * ((int)y0 * W + (int)x0);
    t.wx = sx - x0; t.wy = sy - y0;
    return t;
}

__device__ __forceinline__ uint8_t blend(uint8_t p00, uint8_t p10, uint8_t p01, uint8_t p11, double wx, double wy, double wxi, double wyi) {
    double val = (double)p00 * wxi * wyi + (double)p10 * wx * wyi + (double)p01 * wxi * wy + (double)p11 * wx * wy;
    double r = round(val);  // f64::round: half away from zero
    r = fmin(fmax(r, 0.0), 255.0);
    return (uint8_t)r;
}

// ---------------------------------------------------------------------------------------
// Per-pixel work of the TMA and gather kernels below.  Byte-exact by construction:
//  * The reference blends in f64 (undistort.rs:92-99) and rounds half away from zero.  Here the
//    four tap weights are quantised once per output pixel to 24-bit fixed point
//    (W_i = rn(w_i * 2^24), sum <= 2^24 + 2, so sum p_i W_i fits 32 bits).
//    |S / 2^24 - sum p_i w_i| <= 4 * 255 * 2^-25 = 3.04e-5 and the f64 evaluation order of the
//    reference moves the value by < 1e-12, so whenever the fractional part of S + 0.5 is farther
//    than E = 640 / 2^24 = 3.8e-5 from an integer both round to the same byte.  Otherwise
//    (probability 7.6e-5 per channel) the pixel is redone with the reference's exact f64
//    expression, as are pixels with a weight of exactly 1.
//  * Instruction diet (the first gather kernel was issue-bound at 151 instr/pixel): each 6-byte tap
//    run is three aligned 32-bit words + two PRMT with a per-pixel selector; five more PRMT gather the
//    four taps of each channel into one register; the blend is S = (dp2a(hi16) << 8) + dp4a(lo8) + 2^23
//    per channel: the upper 16 bits of the weights pairwise through dp2a, the low byte plane through dp4a.
// Thread <-> pixel mapping: a warp owns a 32-wide, 4-tall output patch, lane = x.  Neighbouring
// lanes then read neighbouring source pixels (3 bytes apart), so one warp-wide 32-bit load touches
// ~4 sectors instead of the ~17 of a "4 consecutive pixels per thread" mapping (ncu: the first
// mapping was bound by L1 sector look-ups, 444 M per 8 frames).
// ---------------------------------------------------------------------------------------
constexpr uint32_t UND_TIE_E = 640u;

// One output pixel, set up once and reused for every frame.
struct FixedTap {
    Tap t;
    uint32_t sel;            // PRMT selector of the sample's bytes in its 4-byte-aligned window
    uint32_t wlo, w01, w23;  // 24-bit weights, tap order [00, 10, 01, 11]: low byte plane for dp4a, upper 16 bits pairwise
                             // for dp2a.  All zero without a sample: the blend is then 2^23 >> 24 = 0 (black) and can never
                             // look like a tie, so the frame loops need no per-pixel mode test.
    bool slow;               // bilinear with a weight of exactly 1: always takes the exact f64 expression
};

// The tap of a source coordinate (sx, sy) on a W x H input, `st` the status of the step that produced it.  The model source
// below calls it per launch, remap_pack_kernel once per plan: both give the same bits.
template <bool NEAREST>
__device__ __forceinline__ FixedTap tap_from_coord(double sx, double sy, int st, int W, int H) {
    FixedTap p;
    p.t = make_tap(sx, sy, st, W, H, NEAREST ? ACM_INTERP_NEAREST : ACM_INTERP_BILINEAR);
    const double wxi = 1.0 - p.t.wx, wyi = 1.0 - p.t.wy;
    uint32_t w00 = __double2uint_rn(wxi * wyi * 16777216.0), w10 = __double2uint_rn(p.t.wx * wyi * 16777216.0);
    uint32_t w01 = __double2uint_rn(wxi * p.t.wy * 16777216.0), w11 = __double2uint_rn(p.t.wx * p.t.wy * 16777216.0);
    if (!p.t.ok) w00 = w10 = w01 = w11 = 0u;
    p.slow = !NEAREST && ((w00 | w10 | w01 | w11) >> 24) != 0u;
    p.wlo = (w00 & 0xFF) | ((w10 & 0xFF) << 8) | ((w01 & 0xFF) << 16) | ((w11 & 0xFF) << 24);
    p.w01 = ((w00 >> 8) & 0xFFFF) | (((w10 >> 8) & 0xFFFF) << 16);
    p.w23 = ((w01 >> 8) & 0xFFFF) | (((w11 >> 8) & 0xFFFF) << 16);
    p.sel = 0x3210u + 0x1111u * (uint32_t)(p.t.off00 & 3);
    return p;
}

// Where the frame kernels get their taps.  W x H is the output grid.
//  * ModelSrc<M>: undistort_image computes each pixel's source coordinate per launch (the ray through the target pinhole,
//    then CamModel<M>::project, undistort.rs:33-46); input and output grids are the camera's.  undistort_map_kernel
//    writes the same coordinates out.
//  * PlanSrc: an acm_remap_plan's record (remap_pack_kernel) per pixel on any Wi x Hi input.  The plan's f64 map is read
//    only where the f64 weights are needed: by the byte kernel and by the rare exact re-blend.
// coord(): source coordinate and status; tap(): FixedTap; in_w / in_h: the input grid.
template <int M> struct ModelSrc {
    static constexpr bool PLAN = false;
    CamParams c;
    double tfx, tfy, tcx, tcy;  // target intrinsics
    __device__ __forceinline__ int in_w(int W) const { return W; }
    __device__ __forceinline__ int in_h(int H) const { return H; }
    __device__ __forceinline__ int coord(int uo, int vo, int W, int H, double& sx, double& sy) const {
        const double xn = ((double)uo - tcx) / tfx;  // outside the branch: the 4 pixels of a lane share it
        sx = 0.0; sy = 0.0;
        int st = ACM_POINT_IS_OUTSIDE_IMAGE;
        if (uo < W && vo < H) {
            const double yn = ((double)vo - tcy) / tfy;
            st = CamModel<M>::template project<true>(c, xn, yn, 1.0, sx, sy);
        }
        return st;
    }
    template <bool NEAREST> __device__ __forceinline__ FixedTap tap(int uo, int vo, int W, int H) const {
        double sx, sy;
        const int st = coord(uo, vo, W, H, sx, sy);
        return tap_from_coord<NEAREST>(sx, sy, st, W, H);
    }
};

// Plan record, one per output pixel (16 B): x = input pixel index of the tap (bits 0-29; 3 * Wi * Hi < 2^31) | slow << 30 |
// valid << 31, then wlo, w01, w23 of FixedTap.
struct PlanSrc {
    static constexpr bool PLAN = true;
    const uint4* rec;
    const double2* map;  // (sx, sy) per output pixel, NaN where there is no sample
    int Wi, Hi;
    __device__ __forceinline__ int in_w(int) const { return Wi; }
    __device__ __forceinline__ int in_h(int) const { return Hi; }
    __device__ __forceinline__ int coord(int uo, int vo, int W, int H, double& sx, double& sy) const {
        sx = 0.0; sy = 0.0;
        if (uo >= W || vo >= H) return ACM_POINT_IS_OUTSIDE_IMAGE;
        const double2 s = __ldg(map + (size_t)vo * W + uo);
        sx = s.x; sy = s.y;
        return ACM_POINT_OK;  // NaN: make_tap finds no sample
    }
    template <bool NEAREST> __device__ __forceinline__ FixedTap tap(int uo, int vo, int W, int H) const {
        FixedTap p;
        uint4 r = make_uint4(0u, 0u, 0u, 0u);
        if (uo < W && vo < H) r = __ldg(rec + (size_t)vo * W + uo);
        p.t.ok = (int)(r.x >> 31);
        p.t.off00 = 3 * (int)(r.x & 0x3FFFFFFFu);
        p.t.wx = 0.0; p.t.wy = 0.0;  // the exact re-blend takes them from the map (exact_w)
        p.slow = ((r.x >> 30) & 1u) != 0u;
        p.wlo = r.y; p.w01 = r.z; p.w23 = r.w;
        p.sel = 0x3210u + 0x1111u * (uint32_t)(p.t.off00 & 3);
        return p;
    }
    // the reference's bilinear weights (undistort.rs:94): wx = x - floor(x), wy = y - floor(y)
    __device__ __forceinline__ void exact_w(int uo, int vo, int W, double& wx, double& wy) const {
        const double2 s = __ldg(map + (size_t)vo * W + uo);
        wx = s.x - floor(s.x); wy = s.y - floor(s.y);
    }
};

// f64 map -> plan records, with the quantisation of the frame kernels (tap_from_coord).  Model-independent.
template <bool NEAREST>
__global__ void __launch_bounds__(256) remap_pack_kernel(const double2* __restrict__ map, uint4* __restrict__ rec, size_t n, int Wi, int Hi) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const double2 s = map[i];
    const FixedTap p = tap_from_coord<NEAREST>(s.x, s.y, ACM_POINT_OK, Wi, Hi);
    rec[i] = make_uint4((uint32_t)(p.t.off00 / 3) | ((uint32_t)p.slow << 30) | ((uint32_t)p.t.ok << 31), p.wlo, p.w01, p.w23);
}

// nearest: the sample is the pixel itself (undistort.rs:79-90), byte by byte from global memory; returns [R G B 0]
__device__ __forceinline__ uint32_t nearest_px(const uint8_t* p) { return __ldg(p) | (__ldg(p + 1) << 8) | ((uint32_t)__ldg(p + 2) << 16); }

// the reference's f64 expression for one pixel, p = its p00 in global memory; returns [R G B 0]
__device__ __forceinline__ uint32_t blend_exact_px(const uint8_t* p, int row_stride, double wx, double wy) {
    const uint8_t* q = p + row_stride;
    const double wxi = 1.0 - wx, wyi = 1.0 - wy;
    const uint32_t r = blend(__ldg(p), __ldg(p + 3), __ldg(q), __ldg(q + 3), wx, wy, wxi, wyi);
    const uint32_t g = blend(__ldg(p + 1), __ldg(p + 4), __ldg(q + 1), __ldg(q + 4), wx, wy, wxi, wyi);
    const uint32_t b = blend(__ldg(p + 2), __ldg(p + 5), __ldg(q + 2), __ldg(q + 5), wx, wy, wxi, wyi);
    return r | (g << 8) | (b << 16);
}

// Generic byte kernel (any width and alignment): one thread owns 4 horizontally adjacent output pixels: it finds their
// source coordinates once, then loops over the frames of the batch, gathers the taps through the read-only path, blends
// with the reference's f64 expression and stages the 12 output bytes in shared memory so that the block writes the row
// segment with 16-byte coalesced stores where the output allows.
template <class Src>
__global__ void __launch_bounds__(256) undistort_kernel(const __grid_constant__ Src source, const uint8_t* __restrict__ in,
                                                        uint8_t* __restrict__ out, int W, int H, size_t n_frames, int interp) {
    // block = 256 threads x 4 pixels = 1024 pixels of one image row (W is padded by the guard)
    __shared__ __align__(16) uint8_t sm[256 * 12];
    const int row = blockIdx.y;
    const int px0 = (blockIdx.x * 256 + threadIdx.x) * 4;
    const int Wi = source.in_w(W), Hi = source.in_h(H);
    const size_t in_frame_bytes = (size_t)Wi * Hi * 3, frame_bytes = (size_t)W * H * 3;
    Tap taps[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        double sx, sy;
        const int st = source.coord(px0 + k, row, W, H, sx, sy);
        taps[k] = make_tap(sx, sy, st, Wi, Hi, interp);
    }
    const int row_stride = 3 * Wi;  // input
    const int seg_px = min(1024, W - blockIdx.x * 1024);  // pixels of this block's segment
    const int seg_bytes = seg_px * 3;
    const size_t seg_off = ((size_t)row * W + (size_t)blockIdx.x * 1024) * 3;
    const bool vec_ok = ((seg_off & 15) == 0) && ((frame_bytes & 15) == 0) && ((reinterpret_cast<uintptr_t>(out) & 15) == 0);
    for (size_t f = 0; f < n_frames; ++f) {
        const uint8_t* src = in + f * in_frame_bytes;
        uint32_t px[4];  // [R G B 0] per pixel
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const uint8_t* p = src + taps[k].off00;
            px[k] = !taps[k].ok                     ? 0u
                    : interp == ACM_INTERP_NEAREST ? nearest_px(p)
                                                    : blend_exact_px(p, row_stride, taps[k].wx, taps[k].wy);
        }
        // the 12 bytes of the four pixels as three words
        uint32_t* smw = reinterpret_cast<uint32_t*>(sm) + threadIdx.x * 3;
        smw[0] = px[0] | (px[1] << 24);
        smw[1] = (px[1] >> 8) | (px[2] << 16);
        smw[2] = (px[2] >> 16) | (px[3] << 8);
        __syncthreads();
        uint8_t* dst = out + f * frame_bytes + seg_off;
        if (vec_ok) {
            const int nvec = seg_bytes >> 4;
            if ((int)threadIdx.x < nvec) __stcs(reinterpret_cast<uint4*>(dst) + threadIdx.x, reinterpret_cast<const uint4*>(sm)[threadIdx.x]);
            for (int b = (nvec << 4) + threadIdx.x; b < seg_bytes; b += 256) dst[b] = sm[b];
        } else {
            for (int b = threadIdx.x; b < seg_bytes; b += 256) dst[b] = sm[b];
        }
        __syncthreads();
    }
}

// Bilinear blend from the aligned 12-byte windows of the two tap rows (a0..a2, b0..b2) with the selector and weights
// of setup_tap.  Returns [R G B 0] and in `tz` the distance of the three channel sums to a rounding tie (see tie_bits).
__device__ __forceinline__ uint32_t blend_fixed(uint32_t a0, uint32_t a1, uint32_t a2, uint32_t b0, uint32_t b1, uint32_t b2, uint32_t sel,
                                                uint32_t wlo, uint32_t w01, uint32_t w23, uint32_t& tz) {
    const uint32_t A = __byte_perm(a0, a1, sel), B = __byte_perm(a1, a2, sel);         // [r0 g0 b0 r1] [g1 b1 . .]
    const uint32_t A2 = __byte_perm(b0, b1, sel), B2 = __byte_perm(b1, b2, sel);
    const uint32_t PR = __byte_perm(A, A2, 0x7430);                                    // [r00 r10 r01 r11]
    const uint32_t T0 = __byte_perm(A, B, 0x5241), T1 = __byte_perm(A2, B2, 0x5241);   // [g0 g1 b0 b1]
    const uint32_t PG = __byte_perm(T0, T1, 0x5410), PB = __byte_perm(T0, T1, 0x7632);
    const uint32_t sr = (__dp2a_hi(w23, PR, __dp2a_lo(w01, PR, 0u)) << 8) + __dp4a(PR, wlo, 1u << 23);
    const uint32_t sg = (__dp2a_hi(w23, PG, __dp2a_lo(w01, PG, 0u)) << 8) + __dp4a(PG, wlo, 1u << 23);
    const uint32_t sb = (__dp2a_hi(w23, PB, __dp2a_lo(w01, PB, 0u)) << 8) + __dp4a(PB, wlo, 1u << 23);
    // distance of the 24-bit fraction to a rounding tie, scaled by 2^8 so that the 32-bit wrap does the
    // masking: ((s + E) mod 2^24) < 2E  <=>  (s * 2^8 + E * 2^8) mod 2^32 < 2E * 2^8
    tz = min(min(sr * 256u + UND_TIE_E * 256u, sg * 256u + UND_TIE_E * 256u), sb * 256u + UND_TIE_E * 256u);
    return __byte_perm(__byte_perm(sr, sg, 0x4473), sb, 0x4710);                       // [sr.3 sg.3 sb.3 .]
}

// bit k: pixel k of blend_fixed is too close to a rounding tie and must be redone exactly
__device__ __forceinline__ uint32_t tie_bits(const uint32_t tz[4]) {
    uint32_t bits = 0u;
    if (min(min(tz[0], tz[1]), min(tz[2], tz[3])) < 2u * UND_TIE_E * 256u) {
#pragma unroll
        for (int k = 0; k < 4; ++k) bits |= (tz[k] < 2u * UND_TIE_E * 256u ? 1u : 0u) << k;
    }
    return bits;
}

// nearest: the sample is the pixel itself (undistort.rs:79-90), 3 bytes out of two aligned words
__device__ __forceinline__ uint32_t pick_nearest(uint32_t a0, uint32_t a1, uint32_t sel) { return __byte_perm(a0, a1, sel) & 0xFFFFFFu; }

// Stores a finished patch: px[k] = [R G B .] of this lane's pixel in row k.  The 96 output bytes of a patch row are
// exchanged with two shuffles so that lane j < 24 stores word j (bytes of pixels 4j/3 and 4j/3 + 1) at dst + 4j.
// dst: word 0 of row 0 plus 4 * lane; n_rows: rows this lane stores.
__device__ __forceinline__ void store_patch(const uint32_t px[4], uint8_t* dst, int row_stride, int n_rows) {
    const int lane = threadIdx.x & 31, src_lane = (4 * lane) / 3;
    const uint32_t out_sel = (lane % 3 == 0) ? 0x4210u : (lane % 3 == 1) ? 0x5421u : 0x6542u;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const uint32_t pa = __shfl_sync(0xffffffffu, px[k], src_lane);
        const uint32_t pb = __shfl_sync(0xffffffffu, px[k], (src_lane + 1) & 31);
        if (k < n_rows) __stcs(reinterpret_cast<uint32_t*>(dst + (size_t)k * row_stride), __byte_perm(pa, pb, out_sel));
    }
}

// ---------------------------------------------------------------------------------------
// Gather path (Wi % 4 == 0 and W % 4 == 0, 4-byte aligned frames; W x H the output, Wi x Hi the input grid): the taps come from global memory through L1, 3 x LDG.32 per tap row
// (2 for nearest).  With list == nullptr the grid covers the image: block = 64 x 16 pixels, warp w owns the patch at
// (w & 1, w >> 1).  Otherwise the warps stride over the patches the TMA kernel below listed (source box larger than its
// tile).
// ---------------------------------------------------------------------------------------
template <class Src, bool NEAREST>
__global__ void __launch_bounds__(256, 3) undistort_gather_kernel(const __grid_constant__ Src source, const uint8_t* __restrict__ in,
                                                               uint8_t* __restrict__ out, int W, int H, size_t n_frames,
                                                               const uint32_t* __restrict__ list, const uint32_t* __restrict__ list_count) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int Wi = source.in_w(W), Hi = source.in_h(H);
    const size_t in_frame_bytes = (size_t)Wi * Hi * 3, frame_bytes = (size_t)W * H * 3;
    const int in_stride = 3 * Wi, row_stride = 3 * W;
    const uint32_t npx = (uint32_t)(W + 31) / 32u;
    const uint32_t n = list ? *list_count : 1u;  // whole image: one patch per warp, the stride ends the loop
    for (uint32_t e = list ? blockIdx.x * 8u + warp : 0u; e < n; e += gridDim.x * 8u) {
        const int x0 = list ? (int)(list[e] % npx) * 32 : blockIdx.x * 64 + (warp & 1) * 32;
        const int y0 = list ? (int)(list[e] / npx) * 4 : blockIdx.y * 16 + (warp >> 1) * 4;
        FixedTap tap[4];
        int offa[4];  // aligned window of the taps
        uint32_t valid = 0u, slow = 0u;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            tap[k] = source.template tap<NEAREST>(x0 + lane, y0 + k, W, H);
            // a window that would read past the end of the frame (the last frame's end for the last pixels) is not read:
            // the pixel takes the exact path
            const bool exact = tap[k].slow || (tap[k].t.ok && (size_t)tap[k].t.off00 + (size_t)in_stride + 16 > in_frame_bytes);
            valid |= (uint32_t)tap[k].t.ok << k;
            slow |= (uint32_t)exact << k;
            // pixels without a sample or taken exactly load from offset 0 (always inside the frame): the tap loads of a
            // thread are issued back to back, ahead of any math or branch
            offa[k] = (tap[k].t.ok && !exact) ? (tap[k].t.off00 & ~3) : 0;
        }
        const int valid_px = min(32, W - x0);  // multiple of 4 because W % 4 == 0
        const int n_rows = (lane < 24 && 4 * lane + 3 < 3 * valid_px) ? min(4, H - y0) : 0;  // rows this lane stores
        uint8_t* dst = out + ((size_t)y0 * W + x0) * 3 + 4 * lane;
        for (size_t f = 0; f < n_frames; ++f, dst += frame_bytes) {
            const uint8_t* src = in + f * in_frame_bytes;
            uint32_t px[4];  // [R G B .] per pixel
            uint32_t redo = slow;
            if (NEAREST) {
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const uint32_t* r0 = reinterpret_cast<const uint32_t*>(src + offa[k]);
                    px[k] = ((valid >> k) & 1u) ? pick_nearest(__ldg(r0), __ldg(r0 + 1), tap[k].sel) : 0u;
                }
            } else {
                uint32_t ta[4][3], tb[4][3], tz[4];
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const uint32_t* r0 = reinterpret_cast<const uint32_t*>(src + offa[k]);
                    const uint32_t* r1 = reinterpret_cast<const uint32_t*>(src + offa[k] + in_stride);
                    ta[k][0] = __ldg(r0); ta[k][1] = __ldg(r0 + 1); ta[k][2] = __ldg(r0 + 2);
                    tb[k][0] = __ldg(r1); tb[k][1] = __ldg(r1 + 1); tb[k][2] = __ldg(r1 + 2);
                }
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    px[k] = blend_fixed(ta[k][0], ta[k][1], ta[k][2], tb[k][0], tb[k][1], tb[k][2], tap[k].sel, tap[k].wlo, tap[k].w01,
                                        tap[k].w23, tz[k]);
                }
                redo |= tie_bits(tz);
            }
            if (redo) {  // rare: these pixels byte by byte from global memory, bilinear with the reference's f64 expression
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    if ((redo >> k) & 1u) {
                        const uint8_t* p = src + tap[k].t.off00;
                        double wx = tap[k].t.wx, wy = tap[k].t.wy;
                        if constexpr (Src::PLAN) { if (!NEAREST) source.exact_w(x0 + lane, y0 + k, W, wx, wy); }
                        px[k] = NEAREST ? nearest_px(p) : blend_exact_px(p, in_stride, wx, wy);
                    }
                }
            }
            store_patch(px, dst, row_stride, n_rows);
        }
    }
}

// ---------------------------------------------------------------------------------------
// TMA path (Wi % 16 == 0, 16-byte aligned input; W % 4 == 0, 4-byte aligned output): the gathers above are bound by load latency and L1
// sector look-ups (ncu: long_scoreboard 4.6 per issue, 60 % of the LSU wavefront budget).  Here
// every warp stages the SOURCE BOX of its 32 x 4 output patch -- UND_BOX_W bytes x UND_BOX_ROWS
// rows, found once from the taps -- in shared memory with one `cp.async.bulk.tensor.3d` per frame
// (tensor = [frame][row][byte] over the input batch), UND_STAGES frames ahead through a ring of
// mbarriers.  The taps then come from shared memory at loop-invariant offsets, so the frame loop
// has no global loads and no address arithmetic left.  The warp is producer and consumer of its
// own ring, hence no "empty" barriers: the shuffles that exchange the finished pixels order every
// lane's tile reads before lane 0 re-arms the stage.  Patches whose box does not fit are appended
// to a list and handled by `undistort_gather_kernel`.
// ---------------------------------------------------------------------------------------
constexpr int UND_BOX_W = 128;
constexpr int UND_BOX_ROWS = 10;  // tallest box (the shared-memory tile holds this many rows)
constexpr int UND_MIN_ROWS = 4;   // one tensor map per box height UND_MIN_ROWS .. UND_BOX_ROWS: a warp fetches only the rows it needs
// Round 2, same-box A/B (4096^2, 32 frames): 4 stages x 1 frame 39.2 / 23.9 us per frame (bilinear / nearest), 2 stages x 2
// frames 38.4 / 21.6 (one barrier wait and one re-arm per two frames), 3 x 2 and 6 x 1 slower (shared memory costs a resident
// block).  Addressing the output rows as a warp-uniform frame base + 32-bit lane offsets instead of a per-lane pointer
// that is advanced per frame cost 18 % in the bilinear kernel (46.3 us) -- kept out.
constexpr int UND_STAGES = 2;  // ring depth in stages
constexpr int UND_FPS = 2;     // frames per stage: one TMA box {UND_BOX_W, rows, UND_FPS}, one barrier wait and one re-arm per UND_FPS frames

struct UndMaps { CUtensorMap m[UND_BOX_ROWS - UND_MIN_ROWS + 1]; };

__device__ __forceinline__ uint32_t und_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void und_mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void und_mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool und_mbar_try_wait(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    asm volatile("{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}"
                 : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
    return ok != 0;
}
__device__ __forceinline__ void und_tma_load_3d(uint32_t dst, const void* map, uint32_t bar, int c0, int c1, int c2) {
    asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
                 ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1), "r"(c2) : "memory");
}

template <class Src, bool NEAREST>
__global__ void __launch_bounds__(256, 3) undistort_tma_kernel(const __grid_constant__ Src source, const __grid_constant__ UndMaps in_maps,
                                                            const uint8_t* __restrict__ in, uint8_t* __restrict__ out, int W, int H,
                                                            int n_frames, uint32_t* __restrict__ list, uint32_t* __restrict__ list_count) {
    constexpr int TILE = UND_FPS * UND_BOX_W * UND_BOX_ROWS;   // one stage = UND_FPS frames of the box
    // dynamic shared memory: tiles[8 warps][STAGES][TILE] | mbarriers[8][STAGES] | wx[4][256] | wy[4][256]
    // (the f64 weights are only read by the rare exact re-blend; keeping them out of registers is what
    // lets three blocks stay resident; a plan source takes them from its map instead)
    extern __shared__ __align__(128) uint8_t und_smem[];
    uint8_t* const tiles = und_smem;
    unsigned long long* const bars = reinterpret_cast<unsigned long long*>(und_smem + 8 * UND_STAGES * TILE);
    double* const s_wx = reinterpret_cast<double*>(und_smem + 8 * UND_STAGES * TILE + 8 * UND_STAGES * 8);
    double* const s_wy = s_wx + 4 * 256;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int x0 = blockIdx.x * 64 + (warp & 1) * 32;        // patch origin
    const int y0 = blockIdx.y * 16 + (warp >> 1) * 4;
    if (x0 >= W || y0 >= H) return;                          // warp-uniform; nothing block-wide follows
    const int Wi = source.in_w(W), Hi = source.in_h(H);
    const size_t in_frame_bytes = (size_t)Wi * Hi * 3, frame_bytes = (size_t)W * H * 3;
    const int in_stride = 3 * Wi, row_stride = 3 * W;
    int off[4];
    uint32_t sel[4], wlo[4], w01[4], w23[4];
    uint32_t valid = 0u, slow = 0u;
    int bx_min = 0x7fffffff, bx_max = -1, by_min = 0x7fffffff, by_max = -1;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const FixedTap p = source.template tap<NEAREST>(x0 + lane, y0 + k, W, H);
        off[k] = p.t.off00; sel[k] = p.sel; wlo[k] = p.wlo; w01[k] = p.w01; w23[k] = p.w23;
        if (!NEAREST && !Src::PLAN) { s_wx[k * 256 + threadIdx.x] = p.t.wx; s_wy[k * 256 + threadIdx.x] = p.t.wy; }
        slow |= (uint32_t)p.slow << k;
        if (p.t.ok) {
            valid |= 1u << k;
            const int ty = p.t.off00 / in_stride, tb = p.t.off00 - ty * in_stride;
            bx_min = min(bx_min, tb); bx_max = max(bx_max, tb + (NEAREST ? 2 : 5));
            by_min = min(by_min, ty); by_max = max(by_max, ty + (NEAREST ? 0 : 1));
        }
    }
    bx_min = __reduce_min_sync(0xffffffffu, bx_min); bx_max = __reduce_max_sync(0xffffffffu, bx_max);
    by_min = __reduce_min_sync(0xffffffffu, by_min); by_max = __reduce_max_sync(0xffffffffu, by_max);
    const bool any_valid = bx_max >= 0;
    const int box_x = any_valid ? (bx_min & ~15) : 0, box_y = any_valid ? by_min : 0;
    // the aligned 12-byte window of the right-most tap may reach 3 bytes past bx_max
    if (any_valid && (bx_max + 3 - box_x >= UND_BOX_W || by_max - box_y >= UND_BOX_ROWS)) {
        if (lane == 0) list[atomicAdd(list_count, 1u)] = (uint32_t)(y0 >> 2) * ((uint32_t)(W + 31) / 32u) + (uint32_t)(x0 >> 5);
        return;
    }
    const uint32_t tile0 = und_smem_u32(tiles + warp * UND_STAGES * TILE), bar0 = und_smem_u32(bars + warp * UND_STAGES);
    const int box_rows = any_valid ? max(by_max - box_y + 1, UND_MIN_ROWS) : UND_MIN_ROWS;
    const CUtensorMap* const in_map = &in_maps.m[box_rows - UND_MIN_ROWS];
    const uint32_t frame_stride = (uint32_t)(box_rows * UND_BOX_W);   // the box is stored densely: frame h of a stage starts at h * rows * 128
    const uint32_t box_bytes = UND_FPS * frame_stride;
    uint32_t so[4];  // shared-memory address of the aligned tap window in stage 0
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int ty = off[k] / in_stride, tb = off[k] - ty * in_stride;
        so[k] = tile0 + (((valid >> k) & 1u) ? (uint32_t)((ty - box_y) * UND_BOX_W + ((tb - box_x) & ~3)) : 0u);
    }
    const int valid_px = min(32, W - x0);                     // multiple of 4 because W % 4 == 0
    const int n_rows = (lane < 24 && 4 * lane + 3 < 3 * valid_px) ? min(4, H - y0) : 0;  // rows this lane stores
    if (lane == 0) {
#pragma unroll
        for (int sidx = 0; sidx < UND_STAGES; ++sidx) und_mbar_init(bar0 + 8 * sidx, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        if (any_valid) {
#pragma unroll
            for (int sidx = 0; sidx < UND_STAGES; ++sidx) {
                if (sidx * UND_FPS < n_frames) {   // a box that reaches past the last frame is zero-filled and still counts in full
                    und_mbar_expect_tx(bar0 + 8 * sidx, box_bytes);
                    und_tma_load_3d(tile0 + sidx * TILE, in_map, bar0 + 8 * sidx, box_x, box_y, sidx * UND_FPS);
                }
            }
        }
    }
    __syncwarp();
    int stage = 0;
    uint32_t parity = 0;
    const long long t_begin = clock64();
    uint8_t* dst = out + ((size_t)y0 * W + x0) * 3 + 4 * lane;
    for (int f0 = 0; f0 < n_frames; f0 += UND_FPS) {
        const uint32_t stage_off = (uint32_t)(stage * TILE);
        if (any_valid) {
            const uint32_t bar = bar0 + 8 * stage;
            int spins = 0;
            while (!und_mbar_try_wait(bar, parity)) {
                // a lost TMA must not hang the GPU: give up after ~2 s
                if ((++spins & 255) == 0 && clock64() - t_begin > 4000000000LL) __trap();
            }
        }
#pragma unroll
        for (int h = 0; h < UND_FPS; ++h) {
            const int f = f0 + h;
            if (f >= n_frames) break;
            uint32_t px[4] = {0u, 0u, 0u, 0u};  // [R G B .] per pixel
            if (any_valid) {
                const uint32_t tile_off = stage_off + (uint32_t)h * frame_stride;
                uint32_t redo = slow;
                if (NEAREST) {
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        uint32_t a0, a1;
                        const uint32_t addr = so[k] + tile_off;
                        asm volatile("ld.shared.u32 %0, [%2];\n ld.shared.u32 %1, [%2+4];" : "=r"(a0), "=r"(a1) : "r"(addr));
                        px[k] = ((valid >> k) & 1u) ? pick_nearest(a0, a1, sel[k]) : 0u;
                    }
                } else {
                    uint32_t tz[4];
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        uint32_t a0, a1, a2, b0, b1, b2;
                        const uint32_t addr = so[k] + tile_off;
                        asm volatile("ld.shared.u32 %0, [%6];\n ld.shared.u32 %1, [%6+4];\n ld.shared.u32 %2, [%6+8];\n"
                                     "ld.shared.u32 %3, [%6+128];\n ld.shared.u32 %4, [%6+132];\n ld.shared.u32 %5, [%6+136];"
                                     : "=r"(a0), "=r"(a1), "=r"(a2), "=r"(b0), "=r"(b1), "=r"(b2) : "r"(addr));
                        px[k] = blend_fixed(a0, a1, a2, b0, b1, b2, sel[k], wlo[k], w01[k], w23[k], tz[k]);
                    }
                    redo |= tie_bits(tz);
                }
                if (redo) {  // rare: redo these pixels with the reference's f64 expression from global memory
                    const uint8_t* src = in + (size_t)f * in_frame_bytes;
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        if ((redo >> k) & 1u) {
                            // rebuild the byte offset of p00 from the tile address and the byte selector
                            const uint32_t rel = so[k] - tile0;
                            const int o00 = (box_y + (int)(rel / UND_BOX_W)) * in_stride + box_x + (int)(rel % UND_BOX_W) + (int)(sel[k] & 3u);
                            double wx, wy;
                            if constexpr (Src::PLAN) source.exact_w(x0 + lane, y0 + k, W, wx, wy);
                            else { wx = s_wx[k * 256 + threadIdx.x]; wy = s_wy[k * 256 + threadIdx.x]; }
                            px[k] = blend_exact_px(src + o00, in_stride, wx, wy);
                        }
                    }
                }
            }
            store_patch(px, dst, row_stride, n_rows);
            dst += frame_bytes;
        }
        // every lane's tile reads of this stage have been consumed by the shuffles above
        if (any_valid && lane == 0 && f0 + UND_STAGES * UND_FPS < n_frames) {
            und_mbar_expect_tx(bar0 + 8 * stage, box_bytes);
            und_tma_load_3d(tile0 + stage * TILE, in_map, bar0 + 8 * stage, box_x, box_y, f0 + UND_STAGES * UND_FPS);
        }
        if (++stage == UND_STAGES) { stage = 0; parity ^= 1u; }
    }
}

template <int M>
__global__ void __launch_bounds__(256) undistort_map_kernel(const __grid_constant__ ModelSrc<M> source, double* __restrict__ src_xy, int W,
                                                            int H) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (size_t)W * H) return;
    const int uo = (int)(i % W), vo = (int)(i / W);
    double sx, sy;
    const int st = source.coord(uo, vo, W, H, sx, sy);
    if (st != ACM_POINT_OK) sx = sy = acm_nan();
    reinterpret_cast<double2*>(src_xy)[i] = make_double2(sx, sy);
}

// Tensor map over the input batch as [frame][row][byte] (u8), box = UND_BOX_W bytes x UND_BOX_ROWS rows of
// one frame.  cuTensorMapEncodeTiled comes from the driver through the runtime's entry-point query, so
// libacm does not link against libcuda.  Returns false when the driver refuses (the caller then uses
// the gather kernel).
static bool make_frame_tensor_map(CUtensorMap* map, const uint8_t* d_in, int W, int H, size_t n_frames, int box_rows) {
    typedef CUresult (*EncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                 const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
    static EncodeFn encode = nullptr;
    static bool looked_up = false;
    if (!looked_up) {
        looked_up = true;
        void* fn = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
            encode = reinterpret_cast<EncodeFn>(fn);
        else
            cudaGetLastError();
    }
    if (!encode) return false;
    const cuuint64_t gdim[3] = {(cuuint64_t)3 * W, (cuuint64_t)H, (cuuint64_t)n_frames};
    const cuuint64_t gstride[2] = {(cuuint64_t)3 * W, (cuuint64_t)3 * W * H};  // bytes, dims 1 and 2
    const cuuint32_t box[3] = {UND_BOX_W, (cuuint32_t)box_rows, UND_FPS};
    const cuuint32_t estride[3] = {1, 1, 1};
    return encode(map, CU_TENSOR_MAP_DATA_TYPE_UINT8, 3, const_cast<uint8_t*>(d_in), gdim, gstride, box, estride, CU_TENSOR_MAP_INTERLEAVE_NONE,
                  CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// A camera whose frames the frame kernels read or write: resolution set, one frame under 2 GiB (the kernels address a frame
// with int offsets).  `who` names the entry point in the messages, `side` the camera ("input " / "output " / "").  With t
// given, it receives the target pinhole of undistort_image: `target`, or the camera's own intrinsics.
static int32_t check_frame_camera(acm_ctx* ctx, const acm_camera* cam, const char* who, const char* side, const double* target = nullptr,
                                  double* t = nullptr) {
    if (!cam) return acm_fail(ctx, ACM_ERR_INVALID_ARG, "%s: null %scamera", who, side);
    if (cam->width == 0 || cam->height == 0)
        return acm_fail(ctx, ACM_ERR_INVALID_ARG, "%s: %scamera resolution must be set (frames have the camera's resolution)", who, side);
    if ((uint64_t)cam->width * cam->height * 3 >= 0x7fffffffULL)
        return acm_fail(ctx, ACM_ERR_INVALID_ARG, "%s: %sframe larger than 2 GiB is not supported", who, side);
    if (t)
        for (int i = 0; i < 4; ++i) t[i] = target ? target[i] : cam->params[i];
    return ACM_OK;
}

// n_frames Wi x Hi input frames -> W x H output frames through the frame kernel the path rule picks (DESIGN 4.3): the TMA
// kernel, then the gather over the patches whose source box does not fit its tile, when Wi % 16 == 0, W % 4 == 0, the input
// is 16-byte and the output 4-byte aligned, n_frames < 2^31 and the driver encodes the tensor maps; the gather over the whole
// image when Wi % 4 == 0, W % 4 == 0 and both buffers are 4-byte aligned; the byte kernel otherwise.
template <class Src>
static int32_t launch_frames(acm_ctx* ctx, const Src& source, int Wi, int Hi, int W, int H, const uint8_t* d_in, uint8_t* d_out,
                             size_t n_frames, int32_t interpolation) {
    const uintptr_t in_addr = reinterpret_cast<uintptr_t>(d_in), out_addr = reinterpret_cast<uintptr_t>(d_out);
    if (Wi % 4 != 0 || W % 4 != 0 || (in_addr & 3) != 0 || (out_addr & 3) != 0) {
        undistort_kernel<Src><<<dim3((W + 1023) / 1024, H), 256, 0, ctx->stream>>>(source, d_in, d_out, W, H, n_frames, interpolation);
        ACM_CHECK_LAUNCH(ctx);
        return ACM_OK;
    }
    UndMaps maps;
    bool tma = Wi % 16 == 0 && (in_addr & 15) == 0 && n_frames < 0x7fffffffULL;
    for (int r = UND_MIN_ROWS; tma && r <= UND_BOX_ROWS; ++r) tma = make_frame_tensor_map(&maps.m[r - UND_MIN_ROWS], d_in, Wi, Hi, n_frames, r);
    // the TMA kernel's leftover list in the context's scratch: [count] at d_count, patch ids (one per 32 x 4 output patch
    // at most) from d_count + 64
    uint32_t* d_count = nullptr;
    if (tma) {
        const size_t n_patches = (size_t)((W + 31) / 32) * (size_t)((H + 3) / 4);
        const int32_t rc = acm_ensure_scratch(ctx, 256 + n_patches * sizeof(uint32_t));
        if (rc) return rc;
        d_count = static_cast<uint32_t*>(ctx->d_scratch);
        ACM_CUDA(ctx, cudaMemsetAsync(d_count, 0, sizeof(uint32_t), ctx->stream));
    }
    const dim3 patch_grid((W + 63) / 64, (H + 15) / 16);  // block = 64 x 16 output pixels
    const auto launch = [&](auto nearest) -> int32_t {
        constexpr bool NEAREST = decltype(nearest)::value;
        if (tma) {
            constexpr int smem = 8 * UND_STAGES * UND_FPS * UND_BOX_W * UND_BOX_ROWS + 8 * UND_STAGES * 8 + 2 * 4 * 256 * 8;
            uint32_t* const d_list = d_count + 64;
            cudaFuncSetAttribute(undistort_tma_kernel<Src, NEAREST>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
            undistort_tma_kernel<Src, NEAREST><<<patch_grid, 256, smem, ctx->stream>>>(source, maps, d_in, d_out, W, H, (int)n_frames, d_list,
                                                                                     d_count);
            ACM_CHECK_LAUNCH(ctx);
            undistort_gather_kernel<Src, NEAREST><<<ctx->sm_count * 3, 256, 0, ctx->stream>>>(source, d_in, d_out, W, H, n_frames, d_list,
                                                                                              d_count);
        } else {
            undistort_gather_kernel<Src, NEAREST><<<patch_grid, 256, 0, ctx->stream>>>(source, d_in, d_out, W, H, n_frames, nullptr, nullptr);
        }
        ACM_CHECK_LAUNCH(ctx);
        return ACM_OK;
    };
    return interpolation == ACM_INTERP_NEAREST ? launch(std::true_type{}) : launch(std::false_type{});
}

// Host frames through the device: a device copy of both batches, in_bytes up, run(d_in, d_out) on the context's stream,
// out_bytes down, synchronise, free.
template <class Run>
static int32_t frames_through_device(acm_ctx* ctx, const uint8_t* frames_in, size_t in_bytes, uint8_t* frames_out, size_t out_bytes, Run run) {
    uint8_t *d_in = nullptr, *d_out = nullptr;
    int32_t rc = acm_device_malloc(ctx, reinterpret_cast<void**>(&d_in), in_bytes);
    if (!rc) rc = acm_device_malloc(ctx, reinterpret_cast<void**>(&d_out), out_bytes);
    if (!rc) {
        const cudaError_t e = cudaMemcpyAsync(d_in, frames_in, in_bytes, cudaMemcpyHostToDevice, ctx->stream);
        if (e != cudaSuccess) rc = acm_fail(ctx, ACM_ERR_CUDA, "H2D failed: %s", cudaGetErrorString(e));
    }
    if (!rc) rc = run(d_in, d_out);
    if (!rc) {
        cudaError_t e = cudaMemcpyAsync(frames_out, d_out, out_bytes, cudaMemcpyDeviceToHost, ctx->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
        if (e != cudaSuccess) rc = acm_fail(ctx, ACM_ERR_CUDA, "D2H failed: %s", cudaGetErrorString(e));
    }
    cudaStreamSynchronize(ctx->stream);
    if (d_in) cudaFree(d_in);
    if (d_out) cudaFree(d_out);
    return rc;
}

extern "C" int32_t acm_undistort_rgb8(acm_ctx* ctx, const acm_camera* cam, const double* target_intrinsics, const uint8_t* d_in,
                                      uint8_t* d_out, size_t n_frames, int32_t interpolation) {
    ACM_ENTER(ctx);
    double t[4];
    int32_t rc = check_frame_camera(ctx, cam, "undistort", "", target_intrinsics, t);
    if (rc) return rc;
    ACM_REQUIRE(ctx, d_in && d_out, "undistort: null frame buffer");
    ACM_REQUIRE(ctx, interpolation == ACM_INTERP_NEAREST || interpolation == ACM_INTERP_BILINEAR, "undistort: unknown interpolation");
    if (n_frames == 0) return ACM_OK;
    CamParams c;
    rc = acm_make_cam_params(ctx, cam, &c);
    if (rc) return rc;
    const int W = (int)cam->width, H = (int)cam->height;
    ACM_DISPATCH_MODEL(cam->model, return launch_frames(ctx, ModelSrc<M>{c, t[0], t[1], t[2], t[3]}, W, H, W, H, d_in, d_out, n_frames, interpolation))
    return ACM_OK;
}

extern "C" int32_t acm_undistort_rgb8_host(acm_ctx* ctx, const acm_camera* cam, const double* target_intrinsics, const uint8_t* frames_in,
                                           uint8_t* frames_out, size_t n_frames, int32_t interpolation) {
    ACM_ENTER(ctx);
    const int32_t rc = check_frame_camera(ctx, cam, "undistort_host", "");
    if (rc) return rc;
    ACM_REQUIRE(ctx, n_frames == 0 || (frames_in && frames_out), "undistort_host: null frame buffer");
    if (n_frames == 0) return ACM_OK;
    const size_t bytes = (size_t)cam->width * cam->height * 3 * n_frames;
    return frames_through_device(ctx, frames_in, bytes, frames_out, bytes, [&](const uint8_t* d_in, uint8_t* d_out) {
        return acm_undistort_rgb8(ctx, cam, target_intrinsics, d_in, d_out, n_frames, interpolation);
    });
}

static int32_t launch_undistort_map(acm_ctx* ctx, const CamParams& c, const double* t, double* d_src_xy, int W, int H) {
    const int grid = (int)(((size_t)W * H + 255) / 256);
    ACM_DISPATCH_MODEL(c.model, (undistort_map_kernel<M><<<grid, 256, 0, ctx->stream>>>(ModelSrc<M>{c, t[0], t[1], t[2], t[3]}, d_src_xy, W, H)))
    ACM_CHECK_LAUNCH(ctx);
    return ACM_OK;
}

extern "C" int32_t acm_undistort_map(acm_ctx* ctx, const acm_camera* cam, const double* target_intrinsics, double* d_src_xy) {
    ACM_ENTER(ctx);
    double t[4];
    int32_t rc = check_frame_camera(ctx, cam, "undistort", "", target_intrinsics, t);
    if (rc) return rc;
    ACM_REQUIRE(ctx, d_src_xy, "undistort_map: null output");
    CamParams c;
    rc = acm_make_cam_params(ctx, cam, &c);
    if (rc) return rc;
    return launch_undistort_map(ctx, c, t, d_src_xy, (int)cam->width, (int)cam->height);
}

// ---------------------------------------------------------------------------------------
// Remap between two camera models (beyond the reference, composed of its functions): output pixel (u, v) of the output
// camera's grid -> ray = output.unproject((u, v)) (with its pixel-bounds test) -> src = input.project(ray) -> the
// interpolate_pixel of undistort.rs:51-105 on the input frame; black where a step fails.  Both steps keep their IEEE
// forms (unproject<true> as acm_unproject_ieee, the non-FAST project<true> as undistort), so the map of the five
// arithmetic-only models is bit-identical to the oracle's.
// A rotated map (stereo rectification; OpenCV's R1 / R2) puts ray_in = R^T ray_out between the two steps, with R taking
// input-camera coordinates to output-camera ones (x_out = R x_in).  The rotation is a uniform kernel argument, not a
// template axis, so the 49 instantiations stay 49; unrotated launches skip it and run the operations they always ran.
// ---------------------------------------------------------------------------------------
struct Rot3 {
    double r[9];  // row-major
};

template <int MI, int MO>
__global__ void __launch_bounds__(256) remap_map_kernel(const __grid_constant__ CamParams ci, const __grid_constant__ CamParams co,
                                                        const __grid_constant__ Rot3 R, int rotated, double* __restrict__ src_xy,
                                                        int W, int H) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (size_t)W * H) return;
    const int uo = (int)(i % W), vo = (int)(i / W);
    double x, y, z, sx, sy;
    int st = CamModel<MO>::template unproject<true>(co, (double)uo, (double)vo, x, y, z);
    if (rotated && st == ACM_POINT_OK) {  // ray_in[k] = (R[0][k] x + R[1][k] y) + R[2][k] z, each operation rounded (-fmad=false)
        const double* r = R.r;
        const double xi = (r[0] * x + r[3] * y) + r[6] * z;
        const double yi = (r[1] * x + r[4] * y) + r[7] * z;
        const double zi = (r[2] * x + r[5] * y) + r[8] * z;
        x = xi; y = yi; z = zi;
    }
    if (st == ACM_POINT_OK) st = CamModel<MI>::template project<true>(ci, x, y, z, sx, sy);
    if (st != ACM_POINT_OK) sx = sy = acm_nan();
    reinterpret_cast<double2*>(src_xy)[i] = make_double2(sx, sy);
}

template <int MO>
static int32_t launch_remap_map(acm_ctx* ctx, const CamParams& ci, const CamParams& co, const Rot3& R, int rotated, double* d_src_xy,
                                int W, int H) {
    const int grid = (int)(((size_t)W * H + 255) / 256);
    ACM_DISPATCH_MODEL(ci.model, (remap_map_kernel<M, MO><<<grid, 256, 0, ctx->stream>>>(ci, co, R, rotated, d_src_xy, W, H)))
    ACM_CHECK_LAUNCH(ctx);
    return ACM_OK;
}

// R must be a proper rotation: finite entries, max |R R^T - I| <= 1e-9, det R > 0.  ctx may be null (acm_stereo_rectify).
static int32_t check_rotation(acm_ctx* ctx, const double* R, const char* who) {
    if (!R) return acm_fail(ctx, ACM_ERR_INVALID_ARG, "%s: null rotation", who);
    for (int k = 0; k < 9; ++k)
        if (!std::isfinite(R[k])) return acm_fail(ctx, ACM_ERR_INVALID_ARG, "%s: rotation has a non-finite entry", who);
    double dev = 0.0;
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j) {
            const double d = R[3 * i] * R[3 * j] + R[3 * i + 1] * R[3 * j + 1] + R[3 * i + 2] * R[3 * j + 2] - (i == j ? 1.0 : 0.0);
            dev = std::fmax(dev, std::fabs(d));
        }
    if (!(dev <= 1e-9)) return acm_fail(ctx, ACM_ERR_INVALID_ARG, "%s: rotation is not orthonormal (max |R R^T - I| = %.3g > 1e-9)", who, dev);
    const double det = R[0] * (R[4] * R[8] - R[5] * R[7]) - R[1] * (R[3] * R[8] - R[5] * R[6]) + R[2] * (R[3] * R[7] - R[4] * R[6]);
    if (det < 0.0) return acm_fail(ctx, ACM_ERR_INVALID_ARG, "%s: rotation is a reflection (det R < 0)", who);
    return ACM_OK;
}

// source coordinates of every pixel of output_cam's grid: the remap map of input_cam -> output_cam, rotated by R unless it is
// null (R checked by the caller)
static int32_t remap_map(acm_ctx* ctx, const acm_camera* input_cam, const acm_camera* output_cam, const double* R, double* d_src_xy) {
    CamParams ci, co;
    int32_t rc = acm_make_cam_params(ctx, input_cam, &ci);
    if (!rc) rc = acm_make_cam_params(ctx, output_cam, &co);
    if (rc) return rc;
    Rot3 rot{};
    if (R) std::memcpy(rot.r, R, sizeof(rot.r));
    const int W = (int)output_cam->width, H = (int)output_cam->height;
    ACM_DISPATCH_MODEL(co.model, return launch_remap_map<M>(ctx, ci, co, rot, R != nullptr, d_src_xy, W, H))
    return ACM_OK;
}

static int32_t remap_map_entry(acm_ctx* ctx, const acm_camera* input_cam, const acm_camera* output_cam, const double* R, double* d_src_xy) {
    int32_t rc = check_frame_camera(ctx, input_cam, "remap", "input ");
    if (!rc) rc = check_frame_camera(ctx, output_cam, "remap", "output ");
    if (rc) return rc;
    ACM_REQUIRE(ctx, d_src_xy, "remap_map: null output");
    return remap_map(ctx, input_cam, output_cam, R, d_src_xy);
}

extern "C" int32_t acm_remap_map(acm_ctx* ctx, const acm_camera* input_cam, const acm_camera* output_cam, double* d_src_xy) {
    ACM_ENTER(ctx);
    return remap_map_entry(ctx, input_cam, output_cam, nullptr, d_src_xy);
}

extern "C" int32_t acm_remap_map_rotated(acm_ctx* ctx, const acm_camera* input_cam, const acm_camera* output_cam, const double R[9],
                                         double* d_src_xy) {
    ACM_ENTER(ctx);
    const int32_t rc = check_rotation(ctx, R, "remap_map");
    if (rc) return rc;
    return remap_map_entry(ctx, input_cam, output_cam, R, d_src_xy);
}

// A plan: the f64 map (16 B per output pixel, read by the byte kernel and the exact re-blend) and the packed records
// (16 B per output pixel, read by the TMA and gather kernels): 32 B per output pixel, 537 MB for a 4096 x 4096 output.
struct acm_remap_plan {
    acm_ctx* ctx;
    int Wi, Hi, Wo, Ho;
    int32_t interpolation;
    double2* d_map;
    uint4* d_rec;
};

static int32_t launch_remap_pack(acm_ctx* ctx, acm_remap_plan* p) {
    const size_t n = (size_t)p->Wo * p->Ho;
    const int grid = (int)((n + 255) / 256);
    if (p->interpolation == ACM_INTERP_NEAREST) remap_pack_kernel<true><<<grid, 256, 0, ctx->stream>>>(p->d_map, p->d_rec, n, p->Wi, p->Hi);
    else remap_pack_kernel<false><<<grid, 256, 0, ctx->stream>>>(p->d_map, p->d_rec, n, p->Wi, p->Hi);
    ACM_CHECK_LAUNCH(ctx);
    return ACM_OK;
}

static void free_plan(acm_remap_plan* p) {
    if (p->d_map) cudaFree(p->d_map);
    if (p->d_rec) cudaFree(p->d_rec);
    delete p;
}

// R: null, or a checked rotation with output_cam != null
static int32_t create_plan(acm_ctx* ctx, const acm_camera* input_cam, const acm_camera* output_cam, const double* target_intrinsics,
                           const double* R, int32_t interpolation, acm_remap_plan** out) {
    ACM_REQUIRE(ctx, !(output_cam && target_intrinsics), "remap_plan: give either an output camera or target intrinsics, not both");
    double t[4];
    int32_t rc = check_frame_camera(ctx, input_cam, "remap", "input ", target_intrinsics, t);
    if (!rc && output_cam) rc = check_frame_camera(ctx, output_cam, "remap", "output ");
    if (rc) return rc;
    ACM_REQUIRE(ctx, interpolation == ACM_INTERP_NEAREST || interpolation == ACM_INTERP_BILINEAR, "remap_plan: unknown interpolation");
    CamParams ci;
    rc = acm_make_cam_params(ctx, input_cam, &ci);
    if (rc) return rc;
    acm_remap_plan* p = new (std::nothrow) acm_remap_plan{ctx, (int)input_cam->width, (int)input_cam->height, 0, 0, interpolation, nullptr,
                                                          nullptr};
    if (!p) return acm_fail(ctx, ACM_ERR_CUDA, "remap_plan: out of host memory");
    const acm_camera* const grid_cam = output_cam ? output_cam : input_cam;
    p->Wo = (int)grid_cam->width; p->Ho = (int)grid_cam->height;
    const size_t n = (size_t)p->Wo * p->Ho;
    rc = acm_device_malloc(ctx, reinterpret_cast<void**>(&p->d_map), n * sizeof(double2));
    if (!rc) rc = acm_device_malloc(ctx, reinterpret_cast<void**>(&p->d_rec), n * sizeof(uint4));
    if (!rc && output_cam) {
        rc = remap_map(ctx, input_cam, output_cam, R, reinterpret_cast<double*>(p->d_map));
    } else if (!rc) {  // undistort_image semantics: the map of acm_undistort_map
        rc = launch_undistort_map(ctx, ci, t, reinterpret_cast<double*>(p->d_map), p->Wo, p->Ho);
    }
    if (!rc) rc = launch_remap_pack(ctx, p);
    if (rc) {
        cudaStreamSynchronize(ctx->stream);  // no kernel may still write to the buffers that are freed
        free_plan(p);
        return rc;
    }
    *out = p;
    return ACM_OK;
}

extern "C" int32_t acm_remap_plan_create(acm_ctx* ctx, const acm_camera* input_cam, const acm_camera* output_cam,
                                         const double* target_intrinsics, int32_t interpolation, acm_remap_plan** out) {
    ACM_ENTER(ctx);
    ACM_REQUIRE(ctx, out, "remap_plan: null output");
    *out = nullptr;
    return create_plan(ctx, input_cam, output_cam, target_intrinsics, nullptr, interpolation, out);
}

extern "C" int32_t acm_remap_plan_create_rotated(acm_ctx* ctx, const acm_camera* input_cam, const acm_camera* output_cam,
                                                 const double R[9], int32_t interpolation, acm_remap_plan** out) {
    ACM_ENTER(ctx);
    ACM_REQUIRE(ctx, out, "remap_plan: null output");
    *out = nullptr;
    ACM_REQUIRE(ctx, output_cam, "remap_plan: a rotated plan needs an output camera (a Pinhole camera gives undistort_image's view)");
    const int32_t rc = check_rotation(ctx, R, "remap_plan");
    if (rc) return rc;
    return create_plan(ctx, input_cam, output_cam, nullptr, R, interpolation, out);
}

extern "C" int32_t acm_remap_plan_destroy(acm_ctx* ctx, acm_remap_plan* plan) {
    ACM_ENTER(ctx);
    if (!plan) return ACM_OK;
    ACM_REQUIRE(ctx, plan->ctx == ctx, "remap_plan: the plan belongs to another context");
    ACM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    free_plan(plan);
    return ACM_OK;
}

extern "C" int32_t acm_remap_rgb8(acm_ctx* ctx, const acm_remap_plan* plan, const uint8_t* d_in, uint8_t* d_out, size_t n_frames) {
    ACM_ENTER(ctx);
    ACM_REQUIRE(ctx, plan, "remap: null plan");
    ACM_REQUIRE(ctx, plan->ctx == ctx, "remap: the plan belongs to another context");
    ACM_REQUIRE(ctx, d_in && d_out, "remap: null frame buffer");
    if (n_frames == 0) return ACM_OK;
    return launch_frames(ctx, PlanSrc{plan->d_rec, plan->d_map, plan->Wi, plan->Hi}, plan->Wi, plan->Hi, plan->Wo, plan->Ho, d_in, d_out,
                         n_frames, plan->interpolation);
}

extern "C" int32_t acm_remap_rgb8_host(acm_ctx* ctx, const acm_remap_plan* plan, const uint8_t* frames_in, uint8_t* frames_out,
                                       size_t n_frames) {
    ACM_ENTER(ctx);
    ACM_REQUIRE(ctx, plan, "remap_host: null plan");
    ACM_REQUIRE(ctx, plan->ctx == ctx, "remap_host: the plan belongs to another context");
    ACM_REQUIRE(ctx, n_frames == 0 || (frames_in && frames_out), "remap_host: null frame buffer");
    if (n_frames == 0) return ACM_OK;
    return frames_through_device(ctx, frames_in, (size_t)plan->Wi * plan->Hi * 3 * n_frames, frames_out, (size_t)plan->Wo * plan->Ho * 3 * n_frames,
                                 [&](const uint8_t* d_in, uint8_t* d_out) { return acm_remap_rgb8(ctx, plan, d_in, d_out, n_frames); });
}

// ---------------------------------------------------------------------------------------
// Stereo rectification (host only): the rotation part of OpenCV's cvStereoRectify (Bouguet).  Its R1 / R2 feed
// acm_remap_plan_create_rotated with one pinhole camera shared by both views.
// ---------------------------------------------------------------------------------------
// Rodrigues vector -> matrix: R = cos t I + (1 - cos t)/t^2 w w^T + (sin t / t) [w]x with t = |w|.  1 - cos t is taken as
// 2 sin^2(t/2) and the ratios are formed before squaring, so tiny angles keep every digit; w = 0 gives I exactly.
static void rodrigues_matrix(const double w[3], double R[9]) {
    const double t = std::sqrt(w[0] * w[0] + w[1] * w[1] + w[2] * w[2]);
    double a = 1.0, b = 0.5, c = 1.0;  // sin t / t, (1 - cos t) / t^2, cos t
    if (t > 0.0) {
        const double h = std::sin(0.5 * t) / t;
        a = std::sin(t) / t;
        b = 2.0 * h * h;
        c = std::cos(t);
    }
    R[0] = c + b * w[0] * w[0];         R[1] = b * w[0] * w[1] - a * w[2];  R[2] = b * w[0] * w[2] + a * w[1];
    R[3] = b * w[1] * w[0] + a * w[2];  R[4] = c + b * w[1] * w[1];         R[5] = b * w[1] * w[2] - a * w[0];
    R[6] = b * w[2] * w[0] - a * w[1];  R[7] = b * w[2] * w[1] + a * w[0];  R[8] = c + b * w[2] * w[2];
}

// Rodrigues matrix -> vector of a rotation.  s = vee(R - R^T)/2 = sin t k, c = (trace R - 1)/2, t = atan2(|s|, c).  For c >= 0
// the axis is s / |s| and w = s t/|s|, which tends to s as t -> 0: unlike OpenCV's Rodrigues, which returns 0 below
// sin t = 1e-5, a 1e-9 rad rotation keeps its 1e-9.  For c < 0 (t > 90 degrees, |s| -> 0 towards 180) the axis comes from
// the symmetric part, (R + R^T)/2 - c I = (1 - c) k k^T, through its largest diagonal entry (k_i^2 >= 1/3), signed to
// agree with s.
static void rodrigues_vector(const double R[9], double w[3]) {
    const double s[3] = {0.5 * (R[7] - R[5]), 0.5 * (R[2] - R[6]), 0.5 * (R[3] - R[1])};
    const double sn = std::sqrt(s[0] * s[0] + s[1] * s[1] + s[2] * s[2]);
    const double c = 0.5 * (R[0] + R[4] + R[8] - 1.0);
    const double t = std::atan2(sn, c);
    if (c >= 0.0) {
        const double f = sn > 0.0 ? t / sn : 1.0;
        for (int j = 0; j < 3; ++j) w[j] = s[j] * f;
        return;
    }
    int i = R[4] > R[0] ? 1 : 0;
    if (R[8] > R[4 * i]) i = 2;
    const double d = 1.0 - c;
    double k[3];
    k[i] = std::sqrt(std::fmax((R[4 * i] - c) / d, 0.0));
    for (int j = 0; j < 3; ++j)
        if (j != i) k[j] = 0.5 * (R[3 * i + j] + R[3 * j + i]) / (d * k[i]);
    const double sign = k[0] * s[0] + k[1] * s[1] + k[2] * s[2] < 0.0 ? -1.0 : 1.0;
    for (int j = 0; j < 3; ++j) w[j] = sign * t * k[j];
}

// C = A B (transpose_b: A B^T), 3 x 3 row-major
static void mat3_mul(const double* A, const double* B, bool transpose_b, double* C) {
    for (int i = 0; i < 3; ++i)
        for (int j = 0; j < 3; ++j) {
            double acc = 0.0;
            for (int k = 0; k < 3; ++k) acc += A[3 * i + k] * (transpose_b ? B[3 * j + k] : B[3 * k + j]);
            C[3 * i + j] = acc;
        }
}

static void mat3_vec(const double* A, const double* x, double* y) {
    for (int i = 0; i < 3; ++i) y[i] = A[3 * i] * x[0] + A[3 * i + 1] * x[1] + A[3 * i + 2] * x[2];
}

extern "C" int32_t acm_stereo_rectify(const double R[9], const double t[3], double R1[9], double R2[9], double* baseline,
                                      int32_t* vertical) {
    if (!t || !R1 || !R2 || !baseline || !vertical) return acm_fail(nullptr, ACM_ERR_INVALID_ARG, "stereo_rectify: null argument");
    const int32_t rc = check_rotation(nullptr, R, "stereo_rectify");
    if (rc) return rc;
    if (!std::isfinite(t[0]) || !std::isfinite(t[1]) || !std::isfinite(t[2]))
        return acm_fail(nullptr, ACM_ERR_INVALID_ARG, "stereo_rectify: translation has a non-finite entry");
    if (t[0] == 0.0 && t[1] == 0.0 && t[2] == 0.0)
        return acm_fail(nullptr, ACM_ERR_INVALID_ARG, "stereo_rectify: translation is zero (no baseline)");
    // half the relative rotation each way brings both cameras to the same orientation
    double om[3], r_r[9], tp[3];
    rodrigues_vector(R, om);
    for (int j = 0; j < 3; ++j) om[j] *= -0.5;
    rodrigues_matrix(om, r_r);
    mat3_vec(r_r, t, tp);
    // then one common rotation takes the baseline t' onto the x axis (or the y axis when the pair is stacked vertically)
    const int idx = std::fabs(tp[0]) > std::fabs(tp[1]) ? 0 : 1;
    const double c = tp[idx], nt = std::sqrt(tp[0] * tp[0] + tp[1] * tp[1] + tp[2] * tp[2]);
    double uu[3] = {0.0, 0.0, 0.0};
    uu[idx] = c > 0.0 ? 1.0 : -1.0;
    double ww[3] = {tp[1] * uu[2] - tp[2] * uu[1], tp[2] * uu[0] - tp[0] * uu[2], tp[0] * uu[1] - tp[1] * uu[0]};
    const double nw = std::sqrt(ww[0] * ww[0] + ww[1] * ww[1] + ww[2] * ww[2]);
    if (nw > 0.0) {
        const double f = std::acos(std::fmin(std::fabs(c) / nt, 1.0)) / nw;
        for (int j = 0; j < 3; ++j) ww[j] *= f;
    }
    double wR[9], t2[3];
    rodrigues_matrix(ww, wR);
    mat3_mul(wR, r_r, true, R1);
    mat3_mul(wR, r_r, false, R2);
    mat3_vec(R2, t, t2);
    *baseline = t2[idx];
    *vertical = idx;
    return ACM_OK;
}

// ---------------------------------------------------------------------------------------
// Synthetic inputs (SURVEY.md section 8d): counter-based splitmix64, transcendental-free so
// that the host oracle reproduces them bit for bit.
// ---------------------------------------------------------------------------------------
__host__ __device__ __forceinline__ uint64_t splitmix64(uint64_t x) {
    x += 0x9E3779B97F4A7C15ULL;
    uint64_t z = x;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ULL;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBULL;
    return z ^ (z >> 31);
}
__device__ __forceinline__ double unit01(uint64_t seed, uint64_t i, uint64_t k) {
    return (double)(splitmix64(seed + 3ULL * i + k) >> 11) * 0x1.0p-53;
}

template <typename T>
__global__ void __launch_bounds__(256) synth_points3_kernel(uint64_t seed, uint64_t i0, double cos_max, int adversarial,
                                                            T* __restrict__ X, T* __restrict__ Y, T* __restrict__ Z, size_t n) {
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t k = (size_t)blockIdx.x * blockDim.x + threadIdx.x; k < n; k += stride) {
        uint64_t i = i0 + k;
        double u0 = unit01(seed, i, 0), u1 = unit01(seed, i, 1), u2 = unit01(seed, i, 2);
        double c = 1.0 - u0 * (1.0 - cos_max);
        double s = sqrt((1.0 - c) * (1.0 + c));
        double t = 4.0 * u1;
        int q = (int)t;
        double f = t - (double)q;
        double a = 1.0 - f, b = f;
        double nrm = sqrt(a * a + b * b);
        a = a / nrm; b = b / nrm;
        double ca, sa;
        switch (q & 3) { case 0: ca = a; sa = b; break; case 1: ca = -b; sa = a; break; case 2: ca = -a; sa = -b; break; default: ca = b; sa = -a; break; }
        double rho = 0.5 + 9.5 * u2;
        double rs = rho * s;
        double x = rs * ca, y = rs * sa, z = rho * c;
        if (adversarial && (i & 63ULL) == 63ULL) {
            switch ((i >> 6) % 6ULL) {
                case 0: x = 0.0; y = 0.0; z = 0.0; break;
                case 1: x = 0.1; y = 0.2; z = -1.0; break;
                case 2: x = 0.0; y = 0.0; z = 1e-9; break;
                case 3: x = 0.0; y = 0.0; z = 1.0; break;
                case 4: x = 1e-3; y = 0.0; z = 0x1.0p-26; break;
                default: x = 1e-3; y = 0.0; z = 0x1.fffffffffffffp-27; break;
            }
        }
        X[k] = (T)x; Y[k] = (T)y; Z[k] = (T)z;
    }
}

template <typename T>
__global__ void __launch_bounds__(256) synth_pixels_kernel(uint64_t seed, uint64_t i0, double W, double H, T* __restrict__ U,
                                                           T* __restrict__ V, size_t n) {
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t k = (size_t)blockIdx.x * blockDim.x + threadIdx.x; k < n; k += stride) {
        uint64_t i = i0 + k;
        U[k] = (T)(W * unit01(seed, i, 0));
        V[k] = (T)(H * unit01(seed, i, 1));
    }
}

__global__ void __launch_bounds__(256) synth_bytes_kernel(uint64_t seed, uint64_t i0, uint8_t* __restrict__ out, size_t n) {
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    // 4 bytes per thread-iteration when aligned
    const size_t n4 = n / 4;
    for (size_t k = (size_t)blockIdx.x * blockDim.x + threadIdx.x; k < n4; k += stride) {
        uint64_t i = i0 + 4 * k;
        uint32_t w = (uint32_t)(splitmix64(seed + i) & 0xFF) | ((uint32_t)(splitmix64(seed + i + 1) & 0xFF) << 8) |
                     ((uint32_t)(splitmix64(seed + i + 2) & 0xFF) << 16) | ((uint32_t)(splitmix64(seed + i + 3) & 0xFF) << 24);
        reinterpret_cast<uint32_t*>(out)[k] = w;
    }
    size_t t = n4 * 4 + (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t < n) out[t] = (uint8_t)(splitmix64(seed + i0 + t) & 0xFF);
}

extern "C" int32_t acm_synth_points3(acm_ctx* ctx, uint64_t seed, size_t first_index, double cos_theta_max, int32_t adversarial, acm_points* xyz) {
    ACM_ENTER(ctx);
    ACM_REQUIRE(ctx, xyz && xyz->dim == 3, "synth_points3: need a dim-3 buffer");
    if (xyz->n == 0) return ACM_OK;
    int grid = grid_for(ctx, xyz->n, 256, 8);
    if (xyz->dtype == ACM_F64)
        synth_points3_kernel<double><<<grid, 256, 0, ctx->stream>>>(seed, first_index, cos_theta_max, adversarial, comp<double>(xyz, 0), comp<double>(xyz, 1), comp<double>(xyz, 2), xyz->n);
    else
        synth_points3_kernel<float><<<grid, 256, 0, ctx->stream>>>(seed, first_index, cos_theta_max, adversarial, comp<float>(xyz, 0), comp<float>(xyz, 1), comp<float>(xyz, 2), xyz->n);
    ACM_CHECK_LAUNCH(ctx);
    return ACM_OK;
}

extern "C" int32_t acm_synth_pixels(acm_ctx* ctx, uint64_t seed, size_t first_index, double width, double height, acm_points* uv) {
    ACM_ENTER(ctx);
    ACM_REQUIRE(ctx, uv && uv->dim == 2, "synth_pixels: need a dim-2 buffer");
    if (uv->n == 0) return ACM_OK;
    int grid = grid_for(ctx, uv->n, 256, 8);
    if (uv->dtype == ACM_F64)
        synth_pixels_kernel<double><<<grid, 256, 0, ctx->stream>>>(seed, first_index, width, height, comp<double>(uv, 0), comp<double>(uv, 1), uv->n);
    else
        synth_pixels_kernel<float><<<grid, 256, 0, ctx->stream>>>(seed, first_index, width, height, comp<float>(uv, 0), comp<float>(uv, 1), uv->n);
    ACM_CHECK_LAUNCH(ctx);
    return ACM_OK;
}

extern "C" int32_t acm_synth_bytes(acm_ctx* ctx, uint64_t seed, size_t first_index, uint8_t* d_out, size_t n) {
    ACM_ENTER(ctx);
    ACM_REQUIRE(ctx, d_out || n == 0, "synth_bytes: null output");
    if (n == 0) return ACM_OK;
    ACM_REQUIRE(ctx, ((uintptr_t)d_out & 3) == 0, "synth_bytes: output must be 4-byte aligned");
    int grid = grid_for(ctx, n / 4 + 4, 256, 8);
    synth_bytes_kernel<<<grid, 256, 0, ctx->stream>>>(seed, first_index, d_out, n);
    ACM_CHECK_LAUNCH(ctx);
    return ACM_OK;
}
