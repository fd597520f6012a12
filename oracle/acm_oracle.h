/*
 * acm_oracle.h -- CPU ORACLE. TEST INFRASTRUCTURE ONLY.
 *
 * Plain-C restatement of the per-point hot path of amin-abouee/apex-camera-models
 * (reference crate v0.4.1, Rust).  Every function cites the reference file:line it
 * follows.  Nothing under oracle/ may be imported, linked or executed by the product
 * (apex_camera_models_b200/, include/): only tests/, __graft_entry__.smoke() and
 * bench.py's cpu_baseline / --impl reference legs use it, and only as the checker or
 * as the timed CPU baseline.
 *
 * Pinning status (see DESIGN.md "Oracle"):
 *   - project / unproject / validators / sample_points / undistort / reprojection stats
 *     follow in-tree reference code and are pinned by the reference's own known-answer
 *     tests (round-trip tolerances, error classification, YAML sample parameters).
 *   - Jacobians / residual / LM live in the un-vendored crate apex-solver "0.1.5"
 *     (reference Cargo.toml:28, no Cargo.lock): PARITY UNPINNED for those; the oracle
 *     restates the published analytic model derivatives, verified against finite
 *     differences, sympy and scipy.least_squares.
 *
 * Build: gcc -O2 -ffp-contract=off -fno-fast-math  (Rust never contracts a*b+c to FMA).
 */
#ifndef ACM_ORACLE_H
#define ACM_ORACLE_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* model ids (SURVEY.md section 8b) */
enum { ORC_PINHOLE = 0, ORC_RADTAN = 1, ORC_KB = 2, ORC_UCM = 3, ORC_EUCM = 4, ORC_DS = 5, ORC_FOV = 6 };
/* per-point status == CameraModelError variant (reference src/camera/mod.rs:79-113) */
enum { ORC_OK = 0, ORC_POINT_OUTSIDE_IMAGE = 1, ORC_POINT_AT_CENTER = 2, ORC_PROJECTION_OUTSIDE_IMAGE = 3, ORC_NUMERICAL = 4 };
/* residual kinds for the (external, unpinned) factor */
enum { ORC_RES_PIXEL = 0, ORC_RES_ALGEBRAIC = 1 };

typedef struct {
    int32_t model;
    uint32_t width, height;
    int32_t n_params;  /* 4,9,8,5,6,6,5 */
    double p[9];       /* fx,fy,cx,cy,dist... in the reference's struct order */
} orc_model;

int orc_n_params(int model);

/* single point; returns status; outputs are NaN when status != 0 */
int orc_project(const orc_model* m, const double X[3], double uv[2]);
int orc_unproject(const orc_model* m, const double uv[2], double ray[3]);
/* batch over AoS buffers (nalgebra Matrix3xX / Matrix2xX memory order) */
void orc_project_batch(const orc_model* m, const double* xyz, size_t n, double* uv, uint8_t* status, int nthreads);
void orc_unproject_batch(const orc_model* m, const double* uv, size_t n, double* xyz, uint8_t* status, int nthreads);

/* geometric validity used by the factor (no image-bounds test: the factor has no resolution) */
int orc_project_nobounds(const orc_model* m, const double X[3], double uv[2]);
/* 2xP Jacobian of (u,v) w.r.t. params, row-major J[2][P]; returns status (nobounds) */
int orc_project_jacobian(const orc_model* m, const double X[3], double uv[2], double* J);
/* 2x3 Jacobian of (u,v) w.r.t. the 3-D point, row-major Jx[2][3]; returns status (nobounds) */
int orc_project_point_jacobian(const orc_model* m, const double X[3], double uv[2], double Jx[6]);
/* batch forms of the two above over AoS points (J: n x 2 x P, resp. n x 2 x 3 row-major), like orc_project_batch */
void orc_project_jacobian_batch(const orc_model* m, const double* xyz, size_t n, double* uv, double* J, uint8_t* status, int nthreads);
void orc_project_point_jacobian_batch(const orc_model* m, const double* xyz, size_t n, double* uv, double* J, uint8_t* status, int nthreads);
/* residual (2) and its 2xP Jacobian for either residual kind; returns status (nobounds) */
int orc_residual_jacobian(const orc_model* m, int kind, const double X[3], const double uv_obs[2], double r[2], double* J);

/* dense linearisation the way a generic solver does it: materialise r(2N), J(2N x P), then
 * H = J^T J (P x P row-major, full), g = J^T r, cost = 0.5*sum r^2. Invalid points are skipped. */
int orc_linearize(const orc_model* m, int kind, const double* xyz, const double* uv, size_t n,
                  double* H, double* g, double* cost, uint64_t* n_valid, int nthreads);

typedef struct {
    int32_t max_iterations;
    double cost_tolerance, parameter_tolerance, gradient_tolerance;
    double lambda0;
    double invalid_penalty; /* residual assigned to invalid points (0 = skip) */
} orc_lm_config;
typedef struct {
    int32_t status;     /* 0 cost tol, 1 param tol, 2 grad tol, 3 max iter, 4 stalled, <0 failure */
    int32_t iterations; /* LM iterations (solves) */
    int32_t passes;     /* streaming passes over the points */
    double initial_cost, final_cost;
    uint64_t n_valid;
} orc_lm_result;
void orc_lm_default_config(orc_lm_config* c); /* reference bin/camera_converter.rs:410-415 */
int orc_lm_solve(const orc_model* m_init, int kind, const double* xyz, const double* uv, size_t n,
                 const double* lower, const double* upper, const orc_lm_config* cfg, double* out_params,
                 orc_lm_result* res, int nthreads);

/* inherent linear_estimation of each model; updates m->p distortion part. returns 0 or error (<0) */
int orc_linear_estimation(orc_model* m, const double* xyz, const double* uv, size_t n);

/* util::sample_points (reference src/util/point_sampling.rs:46-120); out buffers sized for grid;
 * returns kept count */
size_t orc_sample_grid_size(const orc_model* m, size_t n_requested, int* ncx, int* ncy);
size_t orc_sample_points(const orc_model* m, size_t n_requested, double* uv_out, double* xyz_out);

typedef struct { double rmse, min, max, mean, stddev, median; uint64_t count; } orc_proj_error;
int orc_reprojection_error(const orc_model* m, const double* xyz, const double* uv, size_t n, orc_proj_error* out);

/* util::undistort_image (reference src/util/undistort.rs:14-105); interp 0 nearest, 1 bilinear;
 * target = {fx,fy,cx,cy}; images are RGB8 interleaved row-major */
int orc_undistort_rgb8(const orc_model* m, const double target[4], const uint8_t* in, uint8_t* out, int interp, int nthreads);
/* the remap itself: per output pixel source coords (NaN where projection fails) and floor indices */
void orc_undistort_map(const orc_model* m, const double target[4], double* src_xy /* 2*W*H */);

/* util::image_quality (reference src/util/image_quality.rs; acm_oracle_image.c).  RGB8 interleaved row-major. */
double orc_image_psnr(const uint8_t* a, const uint8_t* b, uint32_t W, uint32_t H);
double orc_image_ssim(const uint8_t* a, const uint8_t* b, uint32_t W, uint32_t H);
void orc_rgb_to_grayscale(const uint8_t* rgb, uint32_t W, uint32_t H, uint8_t* gray);
void orc_draw_points_rgb8(const double* uv, size_t n, uint8_t r, uint8_t g, uint8_t b, uint8_t* img, uint32_t W, uint32_t H);
/* compute_image_quality_metrics; combined / reference may be NULL; returns the kept-point count */
size_t orc_image_quality_metrics(const orc_model* in, const orc_model* out, const double* xyz, size_t n, uint32_t W, uint32_t H,
                                 const uint8_t* reference, uint8_t* combined, double* psnr, double* ssim);
/* util::validate_conversion_accuracy (reference src/util/validation.rs:93-213) */
int orc_validate_conversion(const orc_model* out, const orc_model* in, double errors[5], double* average, double* max_error);

/* deterministic synthetic inputs (SURVEY.md section 8d; transcendental-free so device == host bitwise) */
uint64_t orc_splitmix64(uint64_t x);
void orc_synth_points3(uint64_t seed, size_t i0, size_t n, double cos_max, int adversarial, double* xyz);
void orc_synth_pixels(uint64_t seed, size_t i0, size_t n, double W, double H, double* uv);
void orc_synth_bytes(uint64_t seed, size_t i0, size_t n, uint8_t* out);

#ifdef __cplusplus
}
#endif
#endif
