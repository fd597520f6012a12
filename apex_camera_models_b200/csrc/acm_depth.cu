// Depth images (beyond the reference; composed of its functions): a point cloud rendered into a z-buffered range image of
// one camera, and a range image back-projected into per-pixel points.  The semantics are those of include/acm.h
// (acm_render_depth, acm_depth_to_points); tests/depth_oracle.c states the same steps on the CPU.
//
// Compiled with -fmad=false like acm_exact.cu: the transform, project<false>, the nearest-pixel rounding and the range are
// then the oracle's separately rounded operations, so the images of the arithmetic-only models (Pinhole, RadTan, UCM, EUCM,
// Double Sphere) are byte-identical to the oracle's, and so are their back-projected points (unproject<true>).
//
// Render = a scatter: every drawn point does one 64-bit atomicMin of its key into a per-pixel key image in the context's
// scratch arena.  The key orders by f32 range, then by point index, so the minimum is the same whatever order the atomics
// land in.  A resolve pass splits the keys into the range and index images.
#include <cmath>
#include <cstring>

#include "acm_models.cuh"

struct DepthRig {
    double R[9];  // row-major, x_cam = R x + t
    double t[3];
};

template <int M>
__global__ void __launch_bounds__(256) render_depth_kernel(const __grid_constant__ CamParams c, const __grid_constant__ DepthRig g,
                                                           const double* __restrict__ X, const double* __restrict__ Y,
                                                           const double* __restrict__ Z, size_t in_stride, size_t n,
                                                           unsigned long long* __restrict__ keys, int W, int H) {
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const size_t j = i * in_stride;
        const double P[3] = {__ldcs(X + j), __ldcs(Y + j), __ldcs(Z + j)};
        double Q[3], u, v;
        acm_rigid_apply(g.R, g.t, P, Q);
        if (CamModel<M>::template project<false>(c, Q[0], Q[1], Q[2], u, v) != ACM_POINT_OK) continue;
        double rx, ry;
        if (!acm_nearest_pixel(u, v, W, H, rx, ry)) continue;
        const double range = sqrt((Q[0] * Q[0] + Q[1] * Q[1]) + Q[2] * Q[2]);
        if (!(range > 0.0 && range < INFINITY)) continue;
        const unsigned long long key = ((unsigned long long)__float_as_uint(__double2float_rn(range)) << 32) | (unsigned long long)i;
        atomicMin(keys + ((size_t)ry * (size_t)W + (size_t)rx), key);
    }
}

// key -> (f32 range, index); the empty key splits into range bits 0xFFFFFFFF (a NaN) and index UINT32_MAX
__global__ void __launch_bounds__(256) depth_resolve_kernel(const unsigned long long* __restrict__ keys, float* __restrict__ range,
                                                            uint32_t* __restrict__ index, size_t npix) {
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t p = (size_t)blockIdx.x * blockDim.x + threadIdx.x; p < npix; p += stride) {
        const unsigned long long k = __ldcs(keys + p);
        __stcs(range + p, __uint_as_float((uint32_t)(k >> 32)));
        __stcs(index + p, (uint32_t)k);
    }
}

template <int M>
__global__ void __launch_bounds__(256) depth_to_points_kernel(const __grid_constant__ CamParams c, const __grid_constant__ DepthRig g,
                                                              const float* __restrict__ range, double* __restrict__ X,
                                                              double* __restrict__ Y, double* __restrict__ Z,
                                                              uint8_t* __restrict__ st, int W, size_t npix) {
    const size_t p = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= npix) return;
    const float d = __ldcs(range + p);
    double P[3] = {acm_nan(), acm_nan(), acm_nan()};
    int s = ACM_DEPTH_EMPTY;
    if (d > 0.0f && d < INFINITY) {
        double ray[3];
        s = CamModel<M>::template unproject<true>(c, (double)(p % (size_t)W), (double)(p / (size_t)W), ray[0], ray[1], ray[2]) == ACM_POINT_OK
                ? ACM_DEPTH_OK : ACM_DEPTH_UNPROJECT;
        if (s == ACM_DEPTH_OK) {
            const double dd = (double)d;
            double q[3];
#pragma unroll
            for (int k = 0; k < 3; ++k) q[k] = ray[k] * dd - g.t[k];
            acm_rot_t(g.R, q, P);
        }
    }
    __stcs(X + p, P[0]); __stcs(Y + p, P[1]); __stcs(Z + p, P[2]);
    if (st) __stcs(st + p, (unsigned char)s);
}

// checks shared by every entry point: camera with a resolution, rotation, finite translation; fills the rig
static int32_t check_depth_args(acm_ctx* ctx, const acm_camera* cam, const double* R, const double* t, const char* who, DepthRig* g) {
    if (!cam) return acm_fail(ctx, ACM_ERR_INVALID_ARG, "%s: null camera", who);
    if (cam->width == 0 || cam->height == 0)
        return acm_fail(ctx, ACM_ERR_INVALID_ARG, "%s: camera resolution must be set (the image has the camera's resolution)", who);
    if (cam->width > 0x7fffffffu || cam->height > 0x7fffffffu || (uint64_t)cam->width * cam->height > (1ull << 40))
        return acm_fail(ctx, ACM_ERR_INVALID_ARG, "%s: camera width and height must be below 2^31 and the image at most 2^40 pixels", who);
    int32_t rc = acm_check_rotation(ctx, R, who);
    if (rc) return rc;
    if (!t) return acm_fail(ctx, ACM_ERR_INVALID_ARG, "%s: null translation", who);
    if (!(std::isfinite(t[0]) && std::isfinite(t[1]) && std::isfinite(t[2])))
        return acm_fail(ctx, ACM_ERR_INVALID_ARG, "%s: translation has a non-finite entry", who);
    std::memcpy(g->R, R, sizeof(g->R));
    std::memcpy(g->t, t, sizeof(g->t));
    return ACM_OK;
}

static int32_t check_render_n(acm_ctx* ctx, size_t n) {
    ACM_REQUIRE(ctx, n < 0xffffffffull, "render_depth: n must be below 2^32 - 1 (point indices are 32-bit keys)");
    return ACM_OK;
}

// keys (W*H, scratch) <- all ones; render n points read with stride in_stride; resolve into range / index
static int32_t render(acm_ctx* ctx, const acm_camera* cam, const DepthRig& g, const double* X, const double* Y, const double* Z,
                      size_t in_stride, size_t n, unsigned long long* keys, float* range, uint32_t* index) {
    CamParams c;
    int32_t rc = acm_make_cam_params(ctx, cam, &c);
    if (rc) return rc;
    const int W = (int)cam->width, H = (int)cam->height;
    const size_t npix = (size_t)W * (size_t)H;
    ACM_CUDA(ctx, cudaMemsetAsync(keys, 0xFF, npix * sizeof(unsigned long long), ctx->stream));
    if (n) {
        const int grid = grid_for(ctx, n, 256, 8);
        ACM_DISPATCH_MODEL(c.model, (render_depth_kernel<M><<<grid, 256, 0, ctx->stream>>>(c, g, X, Y, Z, in_stride, n, keys, W, H)))
        ACM_CHECK_LAUNCH(ctx);
    }
    depth_resolve_kernel<<<grid_for(ctx, npix, 256, 8), 256, 0, ctx->stream>>>(keys, range, index, npix);
    ACM_CHECK_LAUNCH(ctx);
    return ACM_OK;
}

extern "C" int32_t acm_render_depth(acm_ctx* ctx, const acm_camera* cam, const double R[9], const double t[3], const acm_points* xyz,
                                    float* d_range, uint32_t* d_index) {
    ACM_ENTER(ctx);
    DepthRig g;
    int32_t rc = check_depth_args(ctx, cam, R, t, "render_depth", &g);
    if (rc) return rc;
    ACM_REQUIRE(ctx, xyz && d_range && d_index, "render_depth: null buffer");
    ACM_REQUIRE(ctx, xyz->dim == 3 && xyz->dtype == ACM_F64, "render_depth: xyz must be a dim-3 f64 buffer");
    rc = check_render_n(ctx, xyz->n);
    if (rc) return rc;
    rc = acm_ensure_scratch(ctx, (size_t)cam->width * cam->height * sizeof(unsigned long long));
    if (rc) return rc;
    return render(ctx, cam, g, comp<double>(xyz, 0), comp<double>(xyz, 1), comp<double>(xyz, 2), 1, xyz->n,
                  static_cast<unsigned long long*>(ctx->d_scratch), d_range, d_index);
}

// Host form: the AoS points are copied as they are into the scratch arena behind the key image and the render kernel reads
// them with stride 3; range and index are resolved into the arena and copied back.  Same kernels, same bytes.
extern "C" int32_t acm_render_depth_host(acm_ctx* ctx, const acm_camera* cam, const double R[9], const double t[3], const double* xyz_aos,
                                         size_t n, float* range, uint32_t* index) {
    ACM_ENTER(ctx);
    DepthRig g;
    int32_t rc = check_depth_args(ctx, cam, R, t, "render_depth", &g);
    if (rc) return rc;
    rc = check_render_n(ctx, n);
    if (rc) return rc;
    ACM_REQUIRE(ctx, (n == 0 || xyz_aos) && range && index, "render_depth: null buffer");
    // scratch layout: keys [0, 8P), points [8P, 8P + 24n), range (4P bytes), index (4P bytes)
    const size_t npix = (size_t)cam->width * cam->height;
    rc = acm_ensure_scratch(ctx, 16 * npix + 24 * n);
    if (rc) return rc;
    unsigned long long* keys = static_cast<unsigned long long*>(ctx->d_scratch);
    double* pts = reinterpret_cast<double*>(keys + npix);
    float* d_range = reinterpret_cast<float*>(pts + 3 * n);
    uint32_t* d_index = reinterpret_cast<uint32_t*>(d_range + npix);
    if (n) ACM_CUDA(ctx, cudaMemcpyAsync(pts, xyz_aos, 3 * n * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    rc = render(ctx, cam, g, pts, pts + 1, pts + 2, 3, n, keys, d_range, d_index);
    if (rc) return rc;
    ACM_CUDA(ctx, cudaMemcpyAsync(range, d_range, npix * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
    ACM_CUDA(ctx, cudaMemcpyAsync(index, d_index, npix * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
    ACM_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return ACM_OK;
}

extern "C" int32_t acm_depth_to_points(acm_ctx* ctx, const acm_camera* cam, const double R[9], const double t[3], const float* d_range,
                                       acm_points* xyz, uint8_t* d_status) {
    ACM_ENTER(ctx);
    DepthRig g;
    int32_t rc = check_depth_args(ctx, cam, R, t, "depth_to_points", &g);
    if (rc) return rc;
    ACM_REQUIRE(ctx, d_range && xyz, "depth_to_points: null buffer");
    const size_t npix = (size_t)cam->width * cam->height;
    ACM_REQUIRE(ctx, xyz->dim == 3 && xyz->dtype == ACM_F64, "depth_to_points: xyz must be a dim-3 f64 buffer");
    ACM_REQUIRE(ctx, xyz->n == npix, "depth_to_points: xyz must hold width * height points");
    CamParams c;
    rc = acm_make_cam_params(ctx, cam, &c);
    if (rc) return rc;
    const int grid = (int)((npix + 255) / 256);
    ACM_DISPATCH_MODEL(c.model, (depth_to_points_kernel<M><<<grid, 256, 0, ctx->stream>>>(c, g, d_range, comp<double>(xyz, 0), comp<double>(xyz, 1),
                                                                                          comp<double>(xyz, 2), d_status, (int)cam->width, npix)))
    ACM_CHECK_LAUNCH(ctx);
    return ACM_OK;
}
