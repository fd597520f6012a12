//! Raw bindings of `include/acm.h` (ABI version 2).  One `extern "C"` item per symbol of the header,
//! same order.  NOT compiled in this repository's environment (no Rust toolchain in the image); the
//! ctypes table `apex_camera_models_b200/_native.py` is the tested twin of this file and
//! `tests/test_abi_and_host_logic.py` checks that table against the header and the built library.
#![allow(non_camel_case_types)]
use libc::{c_char, c_void, size_t};

pub const ACM_MAX_PARAMS: usize = 9;
pub const ACM_ABI_VERSION: i32 = 2;
pub const ACM_OK: i32 = 0;
pub const ACM_ERR_INVALID_ARG: i32 = -1;
pub const ACM_ERR_CUDA: i32 = -2;
pub const ACM_ERR_NCCL: i32 = -3;
pub const ACM_ERR_INVALID_PARAMS: i32 = -4;
pub const ACM_ERR_NUMERICAL: i32 = -5;
pub const ACM_ERR_NO_DEVICE: i32 = -6;
pub const ACM_ERR_ZERO_PROJECTION_POINTS: i32 = -7;
pub const ACM_ERR_FOCAL_LENGTH: i32 = -8;
pub const ACM_ERR_PRINCIPAL_POINT: i32 = -9;
pub const ACM_ERR_PEER: i32 = -10;
pub const ACM_F64: i32 = 0;
pub const ACM_F32: i32 = 1;
pub const ACM_RESIDUAL_PIXEL: i32 = 0;
pub const ACM_RESIDUAL_ALGEBRAIC: i32 = 1;
pub const ACM_INTERP_NEAREST: i32 = 0;
pub const ACM_INTERP_BILINEAR: i32 = 1;

#[repr(C)]
pub struct acm_ctx { _private: [u8; 0] }
#[repr(C)]
pub struct acm_points { _private: [u8; 0] }
#[repr(C)]
pub struct acm_remap_plan { _private: [u8; 0] }

#[repr(C)]
#[derive(Clone, Copy, Debug)]
pub struct acm_camera {
    pub model: i32,
    pub width: u32,
    pub height: u32,
    pub n_params: i32,
    pub params: [f64; ACM_MAX_PARAMS],
}

#[repr(C)]
#[derive(Clone, Copy)]
pub struct acm_normal_equations {
    pub n_params: i32,
    pub h: [f64; ACM_MAX_PARAMS * ACM_MAX_PARAMS],
    pub g: [f64; ACM_MAX_PARAMS],
    pub cost: f64,
    pub n_valid: u64,
}

#[repr(C)]
#[derive(Clone, Copy, Debug)]
pub struct acm_lm_config {
    pub max_iterations: i32,
    pub cost_tolerance: f64,
    pub parameter_tolerance: f64,
    pub gradient_tolerance: f64,
    pub lambda0: f64,
    pub invalid_penalty: f64,
    pub check_every: i32,
}

#[repr(C)]
#[derive(Clone, Copy, Debug, Default)]
pub struct acm_lm_result {
    pub status: i32,
    pub iterations: i32,
    pub passes: i32,
    pub initial_cost: f64,
    pub final_cost: f64,
    pub n_valid: u64,
    pub elapsed_ms: f64,
    pub device_ms: f64,
}

#[repr(C)]
#[derive(Clone, Copy, Debug, Default)]
pub struct acm_image_quality {
    pub psnr: f64,
    pub ssim: f64,
    pub n_points: u64,
}

#[repr(C)]
#[derive(Clone, Copy, Debug, Default)]
pub struct acm_projection_error {
    pub rmse: f64,
    pub min: f64,
    pub max: f64,
    pub mean: f64,
    pub stddev: f64,
    pub median: f64,
    pub count: u64,
}

extern "C" {
    pub fn acm_ctx_create(device: i32, cuda_stream: *mut c_void, out: *mut *mut acm_ctx) -> i32;
    pub fn acm_ctx_destroy(ctx: *mut acm_ctx) -> i32;
    pub fn acm_ctx_sync(ctx: *mut acm_ctx) -> i32;
    pub fn acm_last_error(ctx: *const acm_ctx) -> *const c_char;
    pub fn acm_abi_version() -> i32;
    pub fn acm_ctx_device_info(ctx: *const acm_ctx, info: *mut i64) -> i32;
    pub fn acm_timer_start(ctx: *mut acm_ctx) -> i32;
    pub fn acm_timer_stop(ctx: *mut acm_ctx, elapsed_ms: *mut f32) -> i32;
    pub fn acm_ctx_kernel_launches(ctx: *const acm_ctx) -> u64;

    pub fn acm_n_params(model: i32) -> i32;
    pub fn acm_camera_new(model: i32, params: *const f64, n: size_t, out: *mut acm_camera, msg: *mut c_char, msg_len: size_t) -> i32;
    pub fn acm_validate_params(cam: *const acm_camera, msg: *mut c_char, msg_len: size_t) -> i32;

    pub fn acm_device_alloc(ctx: *mut acm_ctx, bytes: size_t, out: *mut *mut c_void) -> i32;
    pub fn acm_device_free(ctx: *mut acm_ctx, p: *mut c_void) -> i32;
    pub fn acm_host_alloc_pinned(ctx: *mut acm_ctx, bytes: size_t, out: *mut *mut c_void) -> i32;
    pub fn acm_host_free_pinned(ctx: *mut acm_ctx, p: *mut c_void) -> i32;
    pub fn acm_memcpy_h2d(ctx: *mut acm_ctx, dst: *mut c_void, src: *const c_void, bytes: size_t) -> i32;
    pub fn acm_memcpy_d2h(ctx: *mut acm_ctx, dst: *mut c_void, src: *const c_void, bytes: size_t) -> i32;
    pub fn acm_memcpy_d2d(ctx: *mut acm_ctx, dst: *mut c_void, src: *const c_void, bytes: size_t) -> i32;
    pub fn acm_memset_d(ctx: *mut acm_ctx, dst: *mut c_void, value: i32, bytes: size_t) -> i32;

    pub fn acm_points_create(ctx: *mut acm_ctx, dim: i32, n: size_t, dtype: i32, out: *mut *mut acm_points) -> i32;
    pub fn acm_points_destroy(ctx: *mut acm_ctx, p: *mut acm_points) -> i32;
    pub fn acm_points_len(p: *const acm_points) -> size_t;
    pub fn acm_points_dim(p: *const acm_points) -> i32;
    pub fn acm_points_dtype(p: *const acm_points) -> i32;
    pub fn acm_points_component(p: *const acm_points, c: i32) -> *mut c_void;
    pub fn acm_points_upload_aos_f64(ctx: *mut acm_ctx, p: *mut acm_points, host_aos: *const f64, n: size_t) -> i32;
    pub fn acm_points_download_aos_f64(ctx: *mut acm_ctx, p: *const acm_points, host_aos: *mut f64, n: size_t) -> i32;

    pub fn acm_project(ctx: *mut acm_ctx, cam: *const acm_camera, xyz: *const acm_points, uv: *mut acm_points, d_status: *mut u8) -> i32;
    pub fn acm_unproject(ctx: *mut acm_ctx, cam: *const acm_camera, uv: *const acm_points, xyz: *mut acm_points, d_status: *mut u8) -> i32;
    pub fn acm_unproject_ieee(ctx: *mut acm_ctx, cam: *const acm_camera, uv: *const acm_points, xyz: *mut acm_points, d_status: *mut u8) -> i32;
    pub fn acm_camera_fast_unproject(cam: *const acm_camera) -> i32;
    pub fn acm_project_unproject(ctx: *mut acm_ctx, cam: *const acm_camera, xyz: *const acm_points, uv: *mut acm_points, ray: *mut acm_points, d_status_project: *mut u8, d_status_unproject: *mut u8) -> i32;
    pub fn acm_project_jacobian(ctx: *mut acm_ctx, cam: *const acm_camera, xyz: *const acm_points, uv: *mut acm_points, d_jac: *mut f64, d_status: *mut u8) -> i32;
    pub fn acm_project_point_jacobian(ctx: *mut acm_ctx, cam: *const acm_camera, xyz: *const acm_points, uv: *mut acm_points, d_jac: *mut f64, d_status: *mut u8) -> i32;
    pub fn acm_project_host(ctx: *mut acm_ctx, cam: *const acm_camera, xyz_aos: *const f64, n: size_t, uv_aos: *mut f64, status: *mut u8) -> i32;
    pub fn acm_unproject_host(ctx: *mut acm_ctx, cam: *const acm_camera, uv_aos: *const f64, n: size_t, xyz_aos: *mut f64, status: *mut u8) -> i32;

    pub fn acm_linearize(ctx: *mut acm_ctx, cam: *const acm_camera, residual_kind: i32, xyz: *const acm_points, uv: *const acm_points, out: *mut acm_normal_equations) -> i32;
    pub fn acm_linearize_async(ctx: *mut acm_ctx, cam: *const acm_camera, residual_kind: i32, xyz: *const acm_points, uv: *const acm_points) -> i32;
    pub fn acm_linearize_host(ctx: *mut acm_ctx, cam: *const acm_camera, residual_kind: i32, xyz_aos: *const f64, uv_aos: *const f64, n: size_t, out: *mut acm_normal_equations) -> i32;

    pub fn acm_lm_default_config(cfg: *mut acm_lm_config) -> i32;
    pub fn acm_lm_solve(ctx: *mut acm_ctx, init: *const acm_camera, residual_kind: i32, xyz: *const acm_points, uv: *const acm_points, lower: *const f64, upper: *const f64, cfg: *const acm_lm_config, out_params: *mut f64, result: *mut acm_lm_result) -> i32;

    pub fn acm_linear_estimation(ctx: *mut acm_ctx, cam: *mut acm_camera, xyz: *const acm_points, uv: *const acm_points) -> i32;

    pub fn acm_undistort_rgb8(ctx: *mut acm_ctx, cam: *const acm_camera, target_intrinsics: *const f64, d_frames_in: *const u8, d_frames_out: *mut u8, n_frames: size_t, interpolation: i32) -> i32;
    pub fn acm_undistort_rgb8_host(ctx: *mut acm_ctx, cam: *const acm_camera, target_intrinsics: *const f64, frames_in: *const u8, frames_out: *mut u8, n_frames: size_t, interpolation: i32) -> i32;
    pub fn acm_undistort_map(ctx: *mut acm_ctx, cam: *const acm_camera, target_intrinsics: *const f64, d_src_xy: *mut f64) -> i32;

    pub fn acm_remap_plan_create(ctx: *mut acm_ctx, input_cam: *const acm_camera, output_cam: *const acm_camera, target_intrinsics: *const f64, interpolation: i32, out: *mut *mut acm_remap_plan) -> i32;
    pub fn acm_remap_plan_destroy(ctx: *mut acm_ctx, plan: *mut acm_remap_plan) -> i32;
    pub fn acm_remap_rgb8(ctx: *mut acm_ctx, plan: *const acm_remap_plan, d_frames_in: *const u8, d_frames_out: *mut u8, n_frames: size_t) -> i32;
    pub fn acm_remap_rgb8_host(ctx: *mut acm_ctx, plan: *const acm_remap_plan, frames_in: *const u8, frames_out: *mut u8, n_frames: size_t) -> i32;
    pub fn acm_remap_map(ctx: *mut acm_ctx, input_cam: *const acm_camera, output_cam: *const acm_camera, d_src_xy: *mut f64) -> i32;
    pub fn acm_remap_plan_create_rotated(ctx: *mut acm_ctx, input_cam: *const acm_camera, output_cam: *const acm_camera, r: *const f64, interpolation: i32, out: *mut *mut acm_remap_plan) -> i32;
    pub fn acm_remap_map_rotated(ctx: *mut acm_ctx, input_cam: *const acm_camera, output_cam: *const acm_camera, r: *const f64, d_src_xy: *mut f64) -> i32;
    pub fn acm_stereo_rectify(r: *const f64, t: *const f64, r1: *mut f64, r2: *mut f64, baseline: *mut f64, vertical: *mut i32) -> i32;

    pub fn acm_reprojection_error(ctx: *mut acm_ctx, cam: *const acm_camera, xyz: *const acm_points, uv: *const acm_points, out: *mut acm_projection_error) -> i32;
    pub fn acm_sample_points(ctx: *mut acm_ctx, cam: *const acm_camera, n_requested: size_t, uv_out: *mut *mut acm_points, xyz_out: *mut *mut acm_points, n_kept: *mut size_t) -> i32;
    pub fn acm_sample_points_shard(ctx: *mut acm_ctx, cam: *const acm_camera, n_requested: size_t, shard: i32, n_shards: i32, uv_out: *mut *mut acm_points, xyz_out: *mut *mut acm_points, n_kept: *mut size_t) -> i32;

    pub fn acm_image_psnr(ctx: *mut acm_ctx, d_img1: *const u8, d_img2: *const u8, width: u32, height: u32, psnr: *mut f64) -> i32;
    pub fn acm_image_ssim(ctx: *mut acm_ctx, d_img1: *const u8, d_img2: *const u8, width: u32, height: u32, ssim: *mut f64) -> i32;
    pub fn acm_draw_points_rgb8(ctx: *mut acm_ctx, uv: *const acm_points, d_keep: *const u8, r: u8, g: u8, b: u8, d_image: *mut u8, width: u32, height: u32) -> i32;
    pub fn acm_image_quality_metrics(ctx: *mut acm_ctx, input_model: *const acm_camera, output_model: *const acm_camera, xyz: *const acm_points, width: u32, height: u32, d_reference: *const u8, d_combined: *mut u8, out: *mut acm_image_quality) -> i32;

    pub fn acm_synth_points3(ctx: *mut acm_ctx, seed: u64, first_index: size_t, cos_theta_max: f64, adversarial: i32, xyz: *mut acm_points) -> i32;
    pub fn acm_synth_pixels(ctx: *mut acm_ctx, seed: u64, first_index: size_t, width: f64, height: f64, uv: *mut acm_points) -> i32;
    pub fn acm_synth_bytes(ctx: *mut acm_ctx, seed: u64, first_index: size_t, d_out: *mut u8, n: size_t) -> i32;

    pub fn acm_comm_get_unique_id(id: *mut u8) -> i32;
    pub fn acm_comm_init_rank(ctx: *mut acm_ctx, n_ranks: i32, rank: i32, id: *const u8) -> i32;
    pub fn acm_comm_destroy(ctx: *mut acm_ctx) -> i32;
    pub fn acm_comm_size(ctx: *const acm_ctx) -> i32;
    pub fn acm_peer_export(ctx: *mut acm_ctx, handle: *mut u8) -> i32;
    pub fn acm_peer_attach(ctx: *mut acm_ctx, n_ranks: i32, rank: i32, handles: *const u8) -> i32;
    pub fn acm_peer_detach(ctx: *mut acm_ctx) -> i32;

    // multi-GPU from one host thread (the converter `main` is single-threaded: bin/camera_converter.rs:127-343)
    pub fn acm_comm_init_all(ctxs: *mut *mut acm_ctx, n: i32) -> i32;
    pub fn acm_comm_destroy_all(ctxs: *mut *mut acm_ctx, n: i32) -> i32;
    pub fn acm_linearize_multi(ctxs: *mut *mut acm_ctx, n: i32, cam: *const acm_camera, residual_kind: i32, xyz: *const *mut acm_points, uv: *const *mut acm_points, out: *mut acm_normal_equations) -> i32;
    pub fn acm_lm_solve_multi(ctxs: *mut *mut acm_ctx, n: i32, init: *const acm_camera, residual_kind: i32, xyz: *const *mut acm_points, uv: *const *mut acm_points, lower: *const f64, upper: *const f64, cfg: *const acm_lm_config, out_params: *mut f64, result: *mut acm_lm_result) -> i32;
    pub fn acm_linear_estimation_multi(ctxs: *mut *mut acm_ctx, n: i32, cam: *mut acm_camera, xyz: *const *mut acm_points, uv: *const *mut acm_points) -> i32;
    pub fn acm_reprojection_error_multi(ctxs: *mut *mut acm_ctx, n: i32, cam: *const acm_camera, xyz: *const *mut acm_points, uv: *const *mut acm_points, out: *mut acm_projection_error) -> i32;
    pub fn acm_sample_points_multi(ctxs: *mut *mut acm_ctx, n: i32, cam: *const acm_camera, n_requested: size_t, uv_out: *mut *mut acm_points, xyz_out: *mut *mut acm_points, n_kept: *mut size_t) -> i32;
}
