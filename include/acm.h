/*
 * acm.h -- C ABI of the B200-native hot path of apex-camera-models (libacm.so).
 *
 * This is the drop-in boundary: a Rust host crate (rust/acm-sys, see INTEGRATION.md) binds
 * exactly these symbols to re-create the reference's `CameraModel` trait surface
 * (reference src/camera/mod.rs:241-340), the per-model `linear_estimation`, the README-era
 * `*OptimizationCost::{linear_estimation, optimize}` facade (reference README.md:70-81) and the
 * two util hot loops (`undistort_image`, `sample_points`, `compute_reprojection_error`).
 *
 * Conventions
 *   - Every function returns an int32_t status: 0 = ACM_OK, negative = error; the text of the
 *     last error on a context is acm_last_error(ctx).  Nothing here aborts or throws.
 *   - Per-point results carry a uint8_t status that is the reference's `CameraModelError`
 *     variant (src/camera/mod.rs:79-113), so the host can rebuild the exact `Err(..)`.
 *     Outputs of failed points are NaN.
 *   - Host point buffers are nalgebra's memory order: Matrix3xX<f64> = xyzxyz..., Matrix2xX<f64>
 *     = uvuv...; device point buffers are SoA (`acm_points`).  Camera parameters are
 *     [fx, fy, cx, cy, distortion...] in the reference's struct order.
 *   - A context is bound to one CUDA device and one stream; calls on one context are issued
 *     by one host thread at a time.  Functions named *_host and the solver entry points are
 *     synchronous; the device-buffer entry points only enqueue work (acm_ctx_sync waits).
 *   - There is no CPU fallback: without a CUDA device acm_ctx_create fails with
 *     ACM_ERR_NO_DEVICE.
 */
#ifndef ACM_H
#define ACM_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define ACM_ABI_VERSION 2

/* CameraModelEnum (reference src/camera/mod.rs:37-46); ids fixed by SURVEY.md section 8b */
enum {
    ACM_MODEL_PINHOLE = 0,        /* pinhole.rs         P = 4 */
    ACM_MODEL_RADTAN = 1,         /* rad_tan.rs         P = 9  [k1,k2,p1,p2,k3] */
    ACM_MODEL_KANNALA_BRANDT = 2, /* kannala_brandt.rs  P = 8  [k1..k4] */
    ACM_MODEL_UCM = 3,            /* ucm.rs             P = 5  [alpha] */
    ACM_MODEL_EUCM = 4,           /* eucm.rs            P = 6  [alpha,beta] */
    ACM_MODEL_DOUBLE_SPHERE = 5,  /* double_sphere.rs   P = 6  [alpha,xi] */
    ACM_MODEL_FOV = 6             /* fov.rs             P = 5  [w] */
};
#define ACM_MAX_PARAMS 9

/* per-point status == CameraModelError variant (reference src/camera/mod.rs:79-113) */
enum {
    ACM_POINT_OK = 0,
    ACM_POINT_IS_OUTSIDE_IMAGE = 1,      /* PointIsOutSideImage */
    ACM_POINT_AT_CAMERA_CENTER = 2,      /* PointAtCameraCenter */
    ACM_PROJECTION_OUTSIDE_IMAGE = 3,    /* ProjectionOutSideImage */
    ACM_POINT_NUMERICAL_ERROR = 4        /* NumericalError(..) */
};

/* call status */
enum {
    ACM_OK = 0,
    ACM_ERR_INVALID_ARG = -1,
    ACM_ERR_CUDA = -2,
    ACM_ERR_NCCL = -3,
    ACM_ERR_INVALID_PARAMS = -4,          /* CameraModelError::InvalidParams */
    ACM_ERR_NUMERICAL = -5,               /* CameraModelError::NumericalError */
    ACM_ERR_NO_DEVICE = -6,
    ACM_ERR_ZERO_PROJECTION_POINTS = -7,  /* UtilError::ZeroProjectionPoints */
    ACM_ERR_FOCAL_LENGTH = -8,            /* CameraModelError::FocalLengthMustBePositive */
    ACM_ERR_PRINCIPAL_POINT = -9,         /* CameraModelError::PrincipalPointMustBeFinite */
    ACM_ERR_PEER = -10                    /* NVLink peer exchange timed out / was aborted by a peer: re-attach the peers */
};

enum { ACM_F64 = 0, ACM_F32 = 1 };
/* residual minimised by the optimiser (the reference's factor lives in apex-solver, unpinned):
 * PIXEL = project(X) - uv;  ALGEBRAIC = f*x - (u-c)*denominator (UCM / EUCM / Double Sphere) */
enum { ACM_RESIDUAL_PIXEL = 0, ACM_RESIDUAL_ALGEBRAIC = 1 };
/* util::InterpolationMethod (reference src/util/undistort.rs:8-12) */
enum { ACM_INTERP_NEAREST = 0, ACM_INTERP_BILINEAR = 1 };

/* Intrinsics + Resolution + distortion of one model (reference src/camera/mod.rs:52-73) */
typedef struct acm_camera {
    int32_t model;
    uint32_t width, height;
    int32_t n_params;
    double params[ACM_MAX_PARAMS];
} acm_camera;

typedef struct acm_ctx acm_ctx;
typedef struct acm_points acm_points;

/* ---- context ------------------------------------------------------------------------- */
/* cuda_stream: a cudaStream_t to enqueue on, or NULL for a stream owned by the context */
int32_t acm_ctx_create(int32_t device, void* cuda_stream, acm_ctx** out);
int32_t acm_ctx_destroy(acm_ctx* ctx);
int32_t acm_ctx_sync(acm_ctx* ctx);
const char* acm_last_error(const acm_ctx* ctx); /* ctx may be NULL: last error of a failed create */
int32_t acm_abi_version(void);
/* device facts used to size grids: {sm_count, l2_bytes, max_smem_per_block, cc_major*10+cc_minor} */
int32_t acm_ctx_device_info(const acm_ctx* ctx, int64_t info[4]);
/* CUDA-event stopwatch on the context's stream */
int32_t acm_timer_start(acm_ctx* ctx);
int32_t acm_timer_stop(acm_ctx* ctx, float* elapsed_ms); /* waits for the stop event */
/* number of kernels this context has launched since creation (bench "gpu_launches") */
uint64_t acm_ctx_kernel_launches(const acm_ctx* ctx);

/* ---- camera parameter blocks (pure host logic, no device needed) ---------------------- */
int32_t acm_n_params(int32_t model);
/* `new(&DVector)` of every model: length check for all; Pinhole/RadTan also validate
 * (reference pinhole.rs:81-104, rad_tan.rs:107-137; the others do not: double_sphere.rs:133-160) */
int32_t acm_camera_new(int32_t model, const double* params, size_t n, acm_camera* out, char* msg, size_t msg_len);
/* CameraModel::validate_params; msg receives the reference's message, e.g. "alpha must be in (0, 1]" */
int32_t acm_validate_params(const acm_camera* cam, char* msg, size_t msg_len);

/* ---- raw device / pinned memory for hosts without a CUDA binding ----------------------- */
int32_t acm_device_alloc(acm_ctx* ctx, size_t bytes, void** out);
int32_t acm_device_free(acm_ctx* ctx, void* p);
int32_t acm_host_alloc_pinned(acm_ctx* ctx, size_t bytes, void** out);
int32_t acm_host_free_pinned(acm_ctx* ctx, void* p);
int32_t acm_memcpy_h2d(acm_ctx* ctx, void* dst, const void* src, size_t bytes); /* async on ctx stream */
int32_t acm_memcpy_d2h(acm_ctx* ctx, void* dst, const void* src, size_t bytes); /* async on ctx stream */
int32_t acm_memcpy_d2d(acm_ctx* ctx, void* dst, const void* src, size_t bytes); /* async on ctx stream */
int32_t acm_memset_d(acm_ctx* ctx, void* dst, int value, size_t bytes);

/* ---- device point buffers (SoA, components 256-byte aligned) --------------------------- */
int32_t acm_points_create(acm_ctx* ctx, int32_t dim /*2|3*/, size_t n, int32_t dtype, acm_points** out);
int32_t acm_points_destroy(acm_ctx* ctx, acm_points* p);
size_t acm_points_len(const acm_points* p);
int32_t acm_points_dim(const acm_points* p);
int32_t acm_points_dtype(const acm_points* p);
void* acm_points_component(const acm_points* p, int32_t c); /* device pointer of component c */
/* nalgebra MatrixNxX<f64> memory (AoS) <-> device SoA; converts to the buffer's dtype */
int32_t acm_points_upload_aos_f64(acm_ctx* ctx, acm_points* p, const double* host_aos, size_t n);
int32_t acm_points_download_aos_f64(acm_ctx* ctx, const acm_points* p, double* host_aos, size_t n);

/* ---- CameraModel::project / unproject, batched (reference src/camera/<model>.rs) -------- */
/* xyz (dim 3) -> uv (dim 2) + status; dtypes of in/out must match (f64, or f32 I/O with f64 math) */
int32_t acm_project(acm_ctx* ctx, const acm_camera* cam, const acm_points* xyz, acm_points* uv, uint8_t* d_status);
int32_t acm_unproject(acm_ctx* ctx, const acm_camera* cam, const acm_points* uv, acm_points* xyz, uint8_t* d_status);
/* acm_unproject keeps every validity decision in the reference's IEEE arithmetic (status bytes bit-exact) and
 * evaluates what follows the last decision with <= 2 ulp reciprocals (values within ~1e-15 relative).  This form
 * stays IEEE to the end: the values are bit-identical to the reference's for the arithmetic-only models
 * (Pinhole, RadTan, UCM, EUCM, Double Sphere); f64 buffers only.  util::sample_points uses it. */
int32_t acm_unproject_ieee(acm_ctx* ctx, const acm_camera* cam, const acm_points* uv, acm_points* xyz, uint8_t* d_status);
/* Kannala-Brandt: acm_unproject replaces the reference's Newton loop (kannala_brandt.rs:470-520) by a contracted one
 * (FMA + reciprocal) for cameras whose coefficients pass a host-side convergence proof (Kantorovich bound over every
 * ru in (1e-6, pi/2]: the reference's loop provably returns Ok and its iterate lies within ~1e-12 of the root); other
 * cameras keep the IEEE loop.  Returns 1 / 0 for "contracted" / "IEEE", negative for an invalid camera block. */
int32_t acm_camera_fast_unproject(const acm_camera* cam);
/* BASELINE config 2, fused: project, then unproject the projected pixel, in one pass (66 B/pt f64
 * instead of 82 for the two kernels).  ray/status_unproject of a point whose projection failed are
 * NaN / the projection's status. */
int32_t acm_project_unproject(acm_ctx* ctx, const acm_camera* cam, const acm_points* xyz, acm_points* uv, acm_points* ray,
                              uint8_t* d_status_project, uint8_t* d_status_unproject);
/* project with the README-era `compute_jacobian = true`: also writes the 2xP Jacobian w.r.t. the
 * camera parameters as 2P device rows of n doubles, d_jac[(r*P + k)*n + i] (r = 0 for u, 1 for v);
 * validity is the model's geometric test only (no image-bounds test) */
int32_t acm_project_jacobian(acm_ctx* ctx, const acm_camera* cam, const acm_points* xyz, acm_points* uv,
                             double* d_jac, uint8_t* d_status);
/* project with the 2x3 Jacobian w.r.t. the 3-D POINT (the trait doc's "Jacobian matrix (2x3)", reference
 * src/camera/mod.rs:246-252): d_jac = six rows of n doubles du/dx, du/dy, du/dz, dv/dx, dv/dy, dv/dz (0 where the
 * projection fails; status = geometric validity, no image-bounds test, like acm_project_jacobian) */
int32_t acm_project_point_jacobian(acm_ctx* ctx, const acm_camera* cam, const acm_points* xyz, acm_points* uv, double* d_jac,
                                   uint8_t* d_status);
/* synchronous host-buffer forms (pageable or pinned AoS f64 in, AoS f64 + status out) */
int32_t acm_project_host(acm_ctx* ctx, const acm_camera* cam, const double* xyz_aos, size_t n, double* uv_aos, uint8_t* status);
int32_t acm_unproject_host(acm_ctx* ctx, const acm_camera* cam, const double* uv_aos, size_t n, double* xyz_aos, uint8_t* status);

/* ---- fused residual + analytic Jacobian + J^T J / J^T r ------------------------------- */
typedef struct acm_normal_equations {
    int32_t n_params;
    double H[ACM_MAX_PARAMS * ACM_MAX_PARAMS]; /* P x P row-major, symmetric, full */
    double g[ACM_MAX_PARAMS];                  /* J^T r */
    double cost;                               /* 0.5 * sum r^2 over valid points */
    uint64_t n_valid;
} acm_normal_equations;
/* one streaming pass over the resident points; only the normal equations leave the GPU.  If a
 * communicator is attached (acm_comm_init_rank) the result is the sum over all ranks. */
int32_t acm_linearize(acm_ctx* ctx, const acm_camera* cam, int32_t residual_kind, const acm_points* xyz,
                      const acm_points* uv, acm_normal_equations* out);
/* enqueue only: the pass (and the all-reduce) without the device->host read; for benchmarks */
int32_t acm_linearize_async(acm_ctx* ctx, const acm_camera* cam, int32_t residual_kind, const acm_points* xyz,
                            const acm_points* uv);
/* host-buffer form: uploads AoS correspondences (chunked, overlapped with the kernel), one pass */
int32_t acm_linearize_host(acm_ctx* ctx, const acm_camera* cam, int32_t residual_kind, const double* xyz_aos,
                           const double* uv_aos, size_t n, acm_normal_equations* out);

/* ---- Levenberg-Marquardt (replaces apex_solver::optimizer::levenberg_marquardt at the call
 *      sites reference bin/camera_converter.rs:378-420, :513-557, :652-698, :794-832, :925-965,
 *      :1058-1096) --------------------------------------------------------------------------- */
typedef struct acm_lm_config {
    int32_t max_iterations;      /* 100   (camera_converter.rs:411) */
    double cost_tolerance;       /* 1e-6  (:412) relative cost decrease */
    double parameter_tolerance;  /* 1e-8  (:413) */
    double gradient_tolerance;   /* 1e-6  (:414) max-norm of J^T r */
    double lambda0;              /* initial damping (1e-3) */
    double invalid_penalty;      /* residual given to invalid points; 0 = skipped */
    int32_t check_every;         /* NCCL path only: iterations enqueued between host polls of the done flag (4) */
} acm_lm_config;
typedef struct acm_lm_result {
    int32_t status;      /* 0 cost tol, 1 parameter tol, 2 gradient tol, 3 max iterations, 4 stalled */
    int32_t iterations;
    int32_t passes;      /* streaming passes over the points */
    double initial_cost, final_cost;
    uint64_t n_valid;
    double elapsed_ms;   /* host wall time of the solve */
    double device_ms;    /* device time of the solve: first pass to last LM step (device_ms / passes = per-iteration device time) */
} acm_lm_result;
int32_t acm_lm_default_config(acm_lm_config* cfg);
/* lower / upper: per-parameter box (Problem::set_variable_bounds), NULL = unbounded */
int32_t acm_lm_solve(acm_ctx* ctx, const acm_camera* init, int32_t residual_kind, const acm_points* xyz,
                     const acm_points* uv, const double* lower, const double* upper, const acm_lm_config* cfg,
                     double* out_params, acm_lm_result* result);

/* ---- inherent linear_estimation of each model (reference double_sphere.rs:225-290,
 *      ucm.rs:200-258, eucm.rs:216-288, kannala_brandt.rs:164-272, rad_tan.rs:153-234,
 *      fov.rs:153-251); updates the distortion part of *cam ---------------------------------- */
int32_t acm_linear_estimation(acm_ctx* ctx, acm_camera* cam, const acm_points* xyz, const acm_points* uv);

/* ---- util hot loops -------------------------------------------------------------------- */
/* util::undistort_image (reference src/util/undistort.rs:14-105) on a batch of RGB8 frames
 * (interleaved, row-major, W*H*3 bytes each, W x H = camera resolution); target = {fx,fy,cx,cy}
 * or NULL for the camera's own intrinsics */
int32_t acm_undistort_rgb8(acm_ctx* ctx, const acm_camera* cam, const double* target_intrinsics,
                           const uint8_t* d_frames_in, uint8_t* d_frames_out, size_t n_frames, int32_t interpolation);
int32_t acm_undistort_rgb8_host(acm_ctx* ctx, const acm_camera* cam, const double* target_intrinsics,
                                const uint8_t* frames_in, uint8_t* frames_out, size_t n_frames, int32_t interpolation);
/* the remap itself: source coordinates of every output pixel, d_src_xy[2*(v*W+u)+{0,1}], NaN
 * where the projection fails */
int32_t acm_undistort_map(acm_ctx* ctx, const acm_camera* cam, const double* target_intrinsics, double* d_src_xy);

/* ---- remap plans: RGB8 frames from one camera model to another (beyond the reference) -----
 * Output pixel (u, v) on the output camera's grid: ray = output.unproject((u, v)), then
 * src = input.project(ray), then undistort.rs's interpolate_pixel on the input frame; black where a
 * step fails.  Input frames have the input camera's resolution, output frames the output camera's.
 * A plan computes the source coordinates once and keeps 32 bytes per output pixel on the device
 * (537 MB for a 4096 x 4096 output); every acm_remap_rgb8 call then only reads them.
 * output_cam != NULL: camera-to-camera remap (target_intrinsics must be NULL).
 * output_cam == NULL: undistort_image semantics of input_cam with target_intrinsics (NULL = own), so the
 * plan's output is byte-identical to acm_undistort_rgb8.  interpolation is fixed per plan.  A plan
 * belongs to the context that created it. */
typedef struct acm_remap_plan acm_remap_plan;
int32_t acm_remap_plan_create(acm_ctx* ctx, const acm_camera* input_cam, const acm_camera* output_cam,
                              const double* target_intrinsics, int32_t interpolation, acm_remap_plan** out);
int32_t acm_remap_plan_destroy(acm_ctx* ctx, acm_remap_plan* plan);
/* n_frames frames, Wi*Hi*3 bytes each in, Wo*Ho*3 bytes each out; n_frames == 0 is a no-op */
int32_t acm_remap_rgb8(acm_ctx* ctx, const acm_remap_plan* plan, const uint8_t* d_frames_in, uint8_t* d_frames_out, size_t n_frames);
int32_t acm_remap_rgb8_host(acm_ctx* ctx, const acm_remap_plan* plan, const uint8_t* frames_in, uint8_t* frames_out, size_t n_frames);
/* the remap map itself: d_src_xy[2*(v*Wo+u)+{0,1}] over the output camera's grid, NaN where a step fails */
int32_t acm_remap_map(acm_ctx* ctx, const acm_camera* input_cam, const acm_camera* output_cam, double* d_src_xy);

/* ---- rotated remap plans and stereo rectification (beyond the reference) -----
 * R: row-major 3x3 rotation taking input-camera coordinates to output-camera ones, x_out = R * x_in
 * (OpenCV's R1 / R2, the R of initUndistortRectifyMap).  Output pixel (u, v): ray_o = output.unproject((u, v)),
 * ray_i = R^T * ray_o (ray_i[k] = (R[0][k]*x + R[1][k]*y) + R[2][k]*z, each operation rounded), then
 * src = input.project(ray_i); black / NaN where a step fails.  output_cam is required (a Pinhole output camera gives
 * the rectified undistort view).  R must be finite, orthonormal to 1e-9 (max |R R^T - I|) and have det R > 0;
 * otherwise ACM_ERR_INVALID_ARG.  Frames go through acm_remap_rgb8 / acm_remap_rgb8_host and the plan is freed by
 * acm_remap_plan_destroy, as for any plan. */
int32_t acm_remap_plan_create_rotated(acm_ctx* ctx, const acm_camera* input_cam, const acm_camera* output_cam,
                                      const double R[9], int32_t interpolation, acm_remap_plan** out);
/* the rotated remap map: d_src_xy[2*(v*Wo+u)+{0,1}] over the output camera's grid, NaN where a step fails */
int32_t acm_remap_map_rotated(acm_ctx* ctx, const acm_camera* input_cam, const acm_camera* output_cam,
                              const double R[9], double* d_src_xy);

/* Bouguet rectification of a calibrated pair, the rotation part of OpenCV's stereoRectify, on the host (no context,
 * no device): x_cam2 = R * x_cam1 + t.  Outputs R1, R2 (row-major; x_rect1 = R1 x_cam1, x_rect2 = R2 x_cam2) and
 * *baseline = the signed component of R2 * t along the rectified baseline axis; *vertical = 1 when |t'_y| >= |t'_x|
 * (t' = t rotated by half the relative rotation; the pair is stacked vertically and rows become columns, as in
 * OpenCV), else 0.  With one Pinhole camera K shared by both views, P1 = K [I | 0] and P2 = K [I | baseline * e]
 * with e = x (or y when vertical).  Unlike OpenCV, the Rodrigues conversions have no small-angle cut-off.
 * ACM_ERR_INVALID_ARG (message in acm_last_error(NULL)) for a null argument, non-finite input, t = 0, or an R that
 * is not a rotation (the check of acm_remap_plan_create_rotated). */
int32_t acm_stereo_rectify(const double R[9], const double t[3], double R1[9], double R2[9],
                           double* baseline, int32_t* vertical);

/* ---- triangulation of matched pixels of a calibrated pair (beyond the reference) -----
 * x_cam2 = R x_cam1 + t (R row-major; the convention of acm_stereo_rectify).  Per pair, in this order:
 *   1. d1 = first.unproject(uv1), d2 = second.unproject(uv2) in the IEEE form of acm_unproject_ieee (with each model's
 *      pixel-bounds test): UNPROJECT_FIRST / UNPROJECT_SECOND on any CameraModelError.
 *   2. In the first camera's frame: d2' = R^T d2 and c2 = -R^T t, d2'[k] = (R[0][k]*x + R[1][k]*y) + R[2][k]*z with every
 *      operation rounded (the rotated remap's order).
 *   3. Midpoint of the closest approach of s1 d1 and c2 + s2 d2': b = d1.d2', p = d1.c2, q = d2'.c2,
 *      PARALLEL when 1 - b^2 <= ACM_TRI_PARALLEL_EPS (rays within ~1e-6 rad of each other), s1 = (p - b q) / (1 - b^2),
 *      s2 = (b p - q) / (1 - b^2), BEHIND when s1 <= 0 or s2 <= 0, X = ((s1 d1 + c2) + s2 d2') / 2.
 *   4. PROJECT unless X projects into both cameras (project with geometric validity, no image-bounds test, like
 *      acm_project_point_jacobian; the second camera sees R X + t).
 *   5. max_iterations > 0: at most that many damped Gauss-Newton (Levenberg-Marquardt) trials on the 4 pixel residuals
 *      first.project(X) - uv1, second.project(R X + t) - uv2, Jacobian [J1(X); J2(R X + t) R] with the analytic 2x3 point
 *      Jacobians, step from a 3x3 Cholesky of H + lambda diag(H) (H = J^T J); a trial is accepted only when both projections
 *      stay valid and the cost (sum of the squared residuals) decreases.  lambda starts at ACM_TRI_LAMBDA0, is divided by
 *      ACM_TRI_LAMBDA_FACTOR on acceptance and multiplied by it on rejection (a failed factorisation is a rejection); the
 *      loop stops after an accepted step with max|delta| <= ACM_TRI_STEP_TOL * max(1, max|X|).
 * uv1 / uv2: dim-2 f64 buffers of n pixels of the first / second camera; xyz: dim-3 f64 buffer, the point in the FIRST
 * camera's frame, NaN where status != OK.  d_err (optional): two rows of n doubles, |first.project(X) - uv1| and
 * |second.project(R X + t) - uv2| (Euclidean, pixels; NaN where status != OK).  d_status (optional): ACM_TRI_* per pair.
 * ACM_ERR_INVALID_ARG for a null camera or buffer, a dimension or length mismatch, non-f64 buffers, max_iterations < 0,
 * an R that is not a rotation (the check of acm_remap_plan_create_rotated), a non-finite t or t = 0.  n = 0 launches
 * nothing; otherwise one kernel. */
enum {
    ACM_TRI_OK = 0,
    ACM_TRI_UNPROJECT_FIRST = 1,   /* first.unproject(uv1) failed (any CameraModelError) */
    ACM_TRI_UNPROJECT_SECOND = 2,  /* second.unproject(uv2) failed */
    ACM_TRI_PARALLEL = 3,          /* 1 - (d1.d2')^2 <= ACM_TRI_PARALLEL_EPS */
    ACM_TRI_BEHIND = 4,            /* the closest-approach parameter along either ray is <= 0 */
    ACM_TRI_PROJECT = 5            /* the returned point does not project (geometric validity) into both cameras */
};
#define ACM_TRI_PARALLEL_EPS 1e-12
#define ACM_TRI_LAMBDA0 1e-3
#define ACM_TRI_LAMBDA_FACTOR 10.0
#define ACM_TRI_STEP_TOL 1e-12
int32_t acm_triangulate(acm_ctx* ctx, const acm_camera* first, const acm_camera* second, const double R[9], const double t[3],
                        const acm_points* uv1, const acm_points* uv2, int32_t max_iterations, acm_points* xyz,
                        double* d_err, uint8_t* d_status);
/* synchronous host form: AoS f64 in (uvuv...), xyz AoS out (xyzxyz...), err (2n, AoS: e1 e2 per pair) or NULL, status or NULL */
int32_t acm_triangulate_host(acm_ctx* ctx, const acm_camera* first, const acm_camera* second, const double R[9], const double t[3],
                             const double* uv1_aos, const double* uv2_aos, size_t n, int32_t max_iterations,
                             double* xyz_aos, double* err, uint8_t* status);

/* ---- depth images: render a point cloud, back-project a depth image (beyond the reference) -----
 * The camera's resolution W x H is the image (width and height in [1, 2^31 - 1]); images are row-major, pixel (c, r) at r*W + c.
 * Render: x_cam = R x + t (R row-major, x_cam[i] = ((R[i][0] x + R[i][1] y) + R[i][2] z) + t[i], each operation rounded, as
 * acm_triangulate's second camera).  Point i is drawn when, in this order:
 *   1. cam.project(x_cam) is Ok with geometric validity only (no image-bounds test, like acm_project_point_jacobian);
 *   2. rx = round(u), ry = round(v) (half away from zero: the nearest rule of undistort_image) satisfy 0 <= rx < W and
 *      0 <= ry < H (NaN fails);
 *   3. range = sqrt((xc*xc + yc*yc) + zc*zc) is finite and > 0.
 * Depth is the RANGE along the ray, not z: the fisheye models see rays beyond 90 degrees, where z <= 0; z = range * ray_z.
 * Per pixel the key (uint64)bits((float)range) << 32 | i ((float): round to nearest; ranges above FLT_MAX become +inf and
 * are still drawn) is reduced by atomicMin: the nearest point in f32 range wins, ties go to the lowest index, and the image
 * does not depend on scheduling.  d_range (W*H floats) receives the winner's f32 range, d_index (W*H uint32) its index; an
 * empty pixel holds the all-ones key split the same way: range bits 0xFFFFFFFF (a NaN) and index UINT32_MAX.
 * xyz: dim-3 f64 buffer of n < 2^32 - 1 world points.  R must be a rotation (the check of acm_remap_plan_create_rotated) and
 * t finite (zero allowed).  The key image (8 bytes per pixel) lives in the context's scratch arena.  One memset and one
 * resolve kernel per call, plus one render kernel when n > 0.  ACM_ERR_INVALID_ARG for a null camera / buffer, a camera
 * without a resolution, a dimension / dtype mismatch, a bad R or t, or n >= 2^32 - 1 (checked before anything is allocated). */
int32_t acm_render_depth(acm_ctx* ctx, const acm_camera* cam, const double R[9], const double t[3], const acm_points* xyz,
                         float* d_range, uint32_t* d_index);
/* synchronous host form: n AoS points (xyzxyz...) staged in the scratch arena; range / index: W*H host elements; the same
 * kernels, so the same bytes as acm_render_depth */
int32_t acm_render_depth_host(acm_ctx* ctx, const acm_camera* cam, const double R[9], const double t[3], const double* xyz_aos,
                              size_t n, float* range, uint32_t* index);
/* Back-project: pixel (c, r) with range d = d_range[r*W + c]: EMPTY unless d is finite and > 0; ray = cam.unproject((c, r))
 * at the integer pixel centre in the IEEE form of acm_unproject_ieee (with its pixel-bounds test), UNPROJECT when it fails;
 * x_cam = ray * (double)d, then x = R^T (x_cam - t) with x[k] = (R[0][k] q0 + R[1][k] q1) + R[2][k] q2, q = x_cam - t (the
 * rotated remap's order), so that a render followed by a back-projection with the same R, t stays in the world frame.
 * xyz: dim-3 f64 buffer of W*H points in pixel order, NaN where the status is not OK; d_status (optional): ACM_DEPTH_* per
 * pixel.  One kernel. */
enum {
    ACM_DEPTH_OK = 0,
    ACM_DEPTH_EMPTY = 1,      /* range not finite or <= 0 (an empty pixel of acm_render_depth) */
    ACM_DEPTH_UNPROJECT = 2   /* cam.unproject((c, r)) failed (outside the UCM / EUCM / DS domain, KB not converged, ...) */
};
int32_t acm_depth_to_points(acm_ctx* ctx, const acm_camera* cam, const double R[9], const double t[3], const float* d_range,
                            acm_points* xyz, uint8_t* d_status);

/* util::compute_reprojection_error (reference src/util/error_metrics.rs:62-121) */
typedef struct acm_projection_error {
    double rmse, min, max, mean, stddev, median;
    uint64_t count;
} acm_projection_error;
/* With a communicator attached (acm_comm_init_rank) xyz / uv are this rank's shard and the
 * statistics are those of the whole set, identical on every rank: sums added in rank order, the
 * median by a radix select over the all-reduced histogram (an empty shard is allowed). */
int32_t acm_reprojection_error(acm_ctx* ctx, const acm_camera* cam, const acm_points* xyz, const acm_points* uv,
                               acm_projection_error* out);

/* util::sample_points (reference src/util/point_sampling.rs:46-120): grid of cell centres ->
 * unproject -> keep Ok && z > 0, order preserved.  Creates two point buffers of *n_kept points. */
int32_t acm_sample_points(acm_ctx* ctx, const acm_camera* cam, size_t n_requested, acm_points** uv_out,
                          acm_points** xyz_out, size_t* n_kept);
/* The same for one of n_shards contiguous row-major slices of the grid (one per GPU): shard s
 * unprojects cells [s*C/n_shards, (s+1)*C/n_shards) of the C = ncx*ncy grid cells, so the shards'
 * outputs concatenated in order are bit-for-bit acm_sample_points' output.  No collective: the
 * kept counts (*n_kept is this shard's) are all the host has to exchange. */
int32_t acm_sample_points_shard(acm_ctx* ctx, const acm_camera* cam, size_t n_requested, int32_t shard, int32_t n_shards,
                                acm_points** uv_out, acm_points** xyz_out, size_t* n_kept);

/* ---- image-quality diagnostics of the converter (reference src/util/image_quality.rs) ----
 * Images are RGB8, interleaved, row-major (image::RgbImage), resident in HBM. */
/* util::calculate_psnr (image_quality.rs:45-89): pixels black in both images are skipped;
 * +inf for identical (or all-black) images */
int32_t acm_image_psnr(acm_ctx* ctx, const uint8_t* d_img1, const uint8_t* d_img2, uint32_t width, uint32_t height, double* psnr);
/* util::calculate_ssim (image_quality.rs:108-210): 3x3 windows over the interior of the
 * truncated-luma grey images; 1.0 when there is no interior window */
int32_t acm_image_ssim(acm_ctx* ctx, const uint8_t* d_img1, const uint8_t* d_img2, uint32_t width, uint32_t height, double* ssim);
/* The radius-2 disc (dx^2 + dy^2 <= 4, clipped) that create_projection_image (:338-373),
 * create_combined_projection_image[_on_reference] (:389-505) and model_projection_visualization
 * (:553-616) draw at (round(u), round(v)) of every point, in one colour, onto an existing image.
 * d_keep (optional) = one byte per point, 0 skips the point. */
int32_t acm_draw_points_rgb8(acm_ctx* ctx, const acm_points* uv, const uint8_t* d_keep, uint8_t r, uint8_t g, uint8_t b,
                             uint8_t* d_image, uint32_t width, uint32_t height);
typedef struct acm_image_quality {
    double psnr, ssim;
    uint64_t n_points; /* points kept: both projections Ok and the output projection inside the image */
} acm_image_quality;
/* util::compute_image_quality_metrics (image_quality.rs:254-324): project xyz through both models,
 * keep the points both project and whose OUTPUT projection lies in [0,W) x [0,H), rasterise the
 * two projection sets (white discs on black), PSNR + SSIM of the two images.  d_combined (optional,
 * W*H*3 bytes) receives the display image the reference saves: green input discs, then magenta
 * output discs, over d_reference (optional; NULL = black).  ACM_ERR_ZERO_PROJECTION_POINTS when no
 * point is kept.  With a communicator attached xyz is this rank's shard and every rank returns the
 * metrics (and the display image) of the whole set. */
int32_t acm_image_quality_metrics(acm_ctx* ctx, const acm_camera* input_model, const acm_camera* output_model, const acm_points* xyz,
                                  uint32_t width, uint32_t height, const uint8_t* d_reference, uint8_t* d_combined,
                                  acm_image_quality* out);

/* ---- deterministic synthetic inputs (SURVEY.md section 8d), generated in HBM ------------ */
int32_t acm_synth_points3(acm_ctx* ctx, uint64_t seed, size_t first_index, double cos_theta_max, int32_t adversarial, acm_points* xyz);
int32_t acm_synth_pixels(acm_ctx* ctx, uint64_t seed, size_t first_index, double width, double height, acm_points* uv);
int32_t acm_synth_bytes(acm_ctx* ctx, uint64_t seed, size_t first_index, uint8_t* d_out, size_t n);

/* ---- multi-GPU: one process (or context) per GPU, NCCL over NVLink ----------------------- */
/* rank 0 calls acm_comm_get_unique_id and hands the 128 bytes to every rank (any transport) */
int32_t acm_comm_get_unique_id(uint8_t id[128]);
int32_t acm_comm_init_rank(acm_ctx* ctx, int32_t n_ranks, int32_t rank, const uint8_t id[128]);
int32_t acm_comm_destroy(acm_ctx* ctx);
int32_t acm_comm_size(const acm_ctx* ctx); /* 1 when no communicator is attached */

/* Fused exchange over NVLink peer memory (one process per GPU on one NVSwitch box).  Every rank
 * exports a small exchange buffer as a 64-byte CUDA IPC handle, the host gathers the handles of all
 * ranks (any transport) and attaches them.  From then on the reducers of the linearisation kernel store
 * their rank's sums straight into every peer's buffer as tagged cells, wait for the peers' and add them
 * in rank order -- pass, all-reduce (and, for acm_lm_solve, every LM step of the solve) are ONE kernel
 * and every rank holds bit-identical sums.  Replaces the NCCL all-reduce of acm_linearize / acm_lm_solve.
 * Like any collective, the calls that carry an exchange (acm_linearize*, acm_lm_solve, and the
 * all-reduced acm_linear_estimation / acm_reprojection_error) must be made in the same order and the
 * same number of times on every rank: the exchanges are numbered per context.  A rank that waits ~2 s
 * for a peer's cell aborts the exchange on EVERY rank; the calls return ACM_ERR_PEER and the context
 * refuses further exchanges until acm_peer_detach + acm_peer_attach (which zero buffers and counters). */
int32_t acm_peer_export(acm_ctx* ctx, uint8_t handle[64]);
int32_t acm_peer_attach(acm_ctx* ctx, int32_t n_ranks, int32_t rank, const uint8_t* handles /* n_ranks * 64 bytes */);
int32_t acm_peer_detach(acm_ctx* ctx);

/* ---- multi-GPU from ONE host thread (SURVEY.md section 8b: the converter `main`, reference
 *      bin/camera_converter.rs:127-343, is single-threaded and has no launcher) ----------------
 * acm_comm_init_all binds n contexts (one per GPU of this process) into a group: peer access between
 * the devices, the NVLink exchange buffers of acm_peer_* mapped directly (no IPC) and -- when libnccl
 * is present -- one NCCL communicator per context (ncclCommInitAll).  Afterwards every context behaves
 * exactly like a rank of the one-process-per-GPU form, and the *_multi entry points below drive all of
 * them from the calling thread: each context's share runs on a worker thread of the group, the caller
 * blocks until all are done and gets rank 0's result (results are identical on every rank).
 * xyz[i] / uv[i] = the shard resident on ctxs[i]'s GPU. */
int32_t acm_comm_init_all(acm_ctx** ctxs, int32_t n);
int32_t acm_comm_destroy_all(acm_ctx** ctxs, int32_t n);
int32_t acm_linearize_multi(acm_ctx** ctxs, int32_t n, const acm_camera* cam, int32_t residual_kind, acm_points* const* xyz,
                            acm_points* const* uv, acm_normal_equations* out);
int32_t acm_lm_solve_multi(acm_ctx** ctxs, int32_t n, const acm_camera* init, int32_t residual_kind, acm_points* const* xyz,
                           acm_points* const* uv, const double* lower, const double* upper, const acm_lm_config* cfg,
                           double* out_params, acm_lm_result* result);
int32_t acm_linear_estimation_multi(acm_ctx** ctxs, int32_t n, acm_camera* cam, acm_points* const* xyz, acm_points* const* uv);
int32_t acm_reprojection_error_multi(acm_ctx** ctxs, int32_t n, const acm_camera* cam, acm_points* const* xyz, acm_points* const* uv,
                                     acm_projection_error* out);
/* shard i of acm_sample_points_shard on ctxs[i]; n_kept[i] = that shard's count */
int32_t acm_sample_points_multi(acm_ctx** ctxs, int32_t n, const acm_camera* cam, size_t n_requested, acm_points** uv_out,
                                acm_points** xyz_out, size_t* n_kept);

#ifdef __cplusplus
}
#endif
#endif /* ACM_H */
