//! `CameraModel` over the B200 hot path.
//!
//! Source only: the image this repository is built in has no Rust toolchain (`cargo`, `rustc` absent), so this crate has
//! never been compiled -- read it as the binding a maintainer would add, not as tested code.  It is deliberately
//! mechanical: every method is one call into `acm-sys`
//! whose behaviour is covered by the Python twin (`apex_camera_models_b200/camera.py`) in
//! `tests/test_gpu_parity.py`.
//!
//! The wrapper keeps the reference's own struct (YAML loading, `validate_params`, getters stay the
//! reference's code) and routes the per-point work to the GPU:
//!   * `project` / `unproject`            -> `acm_project_host` / `acm_unproject_host` (1-point batch)
//!   * `project_batch` / `unproject_batch`-> the same calls on whole `Matrix3xX` / `Matrix2xX`
//!   * `linear_estimation`                -> `acm_linear_estimation`
//!   * `*OptimizationCost::optimize`      -> `acm_lm_solve` (replaces apex-solver's factor + LM)
//!
//! Drop-in points:
//!   * `impl CameraModel for GpuCamera<M>` -- a `GpuCamera` goes wherever the reference holds a
//!     `Box<dyn CameraModel>` / `&dyn CameraModel` (camera_converter.rs:87-125, undistort.rs:16, validation.rs:95);
//!     `load_from_yaml` / `save_to_yaml` / `validate_params` / the getters are the wrapped model's own.
//!   * `DoubleSphereOptimizationCost` .. `FovOptimizationCost` (README.md:70-81): `new`, `linear_estimation`,
//!     `optimize`, `get_intrinsics`, `get_distortion`.
//!   * `DeviceGroup` -- every GPU of the box from the converter's single thread (`acm_comm_init_all`, `acm_*_multi`).
use acm_sys as sys;
use apex_camera_models::camera::{
    CameraModel, CameraModelError, DoubleSphereModel, EucmModel, FovModel, Intrinsics, KannalaBrandtModel, PinholeModel, RadTanModel,
    Resolution, UcmModel,
};
use nalgebra::{DVector, Matrix2xX, Matrix3xX, Vector2, Vector3};
use std::ffi::CStr;
use std::ptr;
use std::sync::{Arc, Mutex, OnceLock};

pub const PINHOLE: i32 = 0;
pub const RAD_TAN: i32 = 1;
pub const KANNALA_BRANDT: i32 = 2;
pub const UCM: i32 = 3;
pub const EUCM: i32 = 4;
pub const DOUBLE_SPHERE: i32 = 5;
pub const FOV: i32 = 6;

/// One CUDA device + stream (acm_ctx).  The ABI wants the calls on one context issued by one thread at a
/// time: every wrapper below takes `lock` for the duration of its call sequence, which is what makes the
/// `Sync` claim sound (a `GpuCamera` behind `&dyn CameraModel` may be shared like the reference's models).
pub struct Context(*mut sys::acm_ctx, Mutex<()>);
unsafe impl Send for Context {}
unsafe impl Sync for Context {}

static GLOBAL_CONTEXT: OnceLock<Result<Arc<Context>, String>> = OnceLock::new();

impl Context {
    pub fn new(device: i32) -> Result<Self, CameraModelError> {
        if unsafe { sys::acm_abi_version() } != sys::ACM_ABI_VERSION {
            return Err(CameraModelError::NumericalError("libacm.so ABI version differs from the one acm-sys binds".into()));
        }
        let mut h = ptr::null_mut();
        let rc = unsafe { sys::acm_ctx_create(device, ptr::null_mut(), &mut h) };
        if rc != sys::ACM_OK {
            let msg = unsafe { CStr::from_ptr(sys::acm_last_error(ptr::null())) }.to_string_lossy().into_owned();
            return Err(CameraModelError::NumericalError(format!("acm_ctx_create: {msg}")));
        }
        Ok(Context(h, Mutex::new(())))
    }
    /// The process-wide context the trait's context-less constructors (`load_from_yaml`) bind to:
    /// device `$ACM_DEVICE` (default 0), created on first use.  There is no CPU fallback: without a
    /// CUDA device this is an error, not a silent detour through the reference code.
    pub fn global() -> Result<Arc<Context>, CameraModelError> {
        GLOBAL_CONTEXT
            .get_or_init(|| {
                let dev = std::env::var("ACM_DEVICE").ok().and_then(|v| v.parse().ok()).unwrap_or(0);
                Context::new(dev).map(Arc::new).map_err(|e| format!("{e:?}"))
            })
            .clone()
            .map_err(CameraModelError::NumericalError)
    }
    fn lock(&self) -> std::sync::MutexGuard<'_, ()> { self.1.lock().unwrap_or_else(|p| p.into_inner()) }
    fn err(&self, rc: i32) -> CameraModelError {
        let msg = unsafe { CStr::from_ptr(sys::acm_last_error(self.0)) }.to_string_lossy().into_owned();
        match rc {
            sys::ACM_ERR_INVALID_PARAMS => CameraModelError::InvalidParams(msg),
            sys::ACM_ERR_FOCAL_LENGTH => CameraModelError::FocalLengthMustBePositive,
            sys::ACM_ERR_PRINCIPAL_POINT => CameraModelError::PrincipalPointMustBeFinite,
            sys::ACM_ERR_PEER => CameraModelError::NumericalError(format!("multi-GPU exchange failed, re-attach the peers: {msg}")),
            _ => CameraModelError::NumericalError(msg),
        }
    }
}
impl Drop for Context {
    fn drop(&mut self) { unsafe { sys::acm_ctx_destroy(self.0); } }
}

/// status byte -> the `Err(..)` the reference's scalar call returns (mod.rs:79-113)
pub fn status_to_error(status: u8, model: i32) -> Option<CameraModelError> {
    match status {
        0 => None,
        1 => Some(CameraModelError::PointIsOutSideImage),
        2 => Some(CameraModelError::PointAtCameraCenter),
        3 => Some(CameraModelError::ProjectionOutSideImage),
        _ => Some(CameraModelError::NumericalError(
            if model == RAD_TAN { "Jacobian is singular".into() } else { "Unprojection failed to converge".into() })),
    }
}

/// ABI model id of a reference model type (`model_id` of include/acm.h).
pub trait GpuModelId { const MODEL_ID: i32; }
impl GpuModelId for PinholeModel { const MODEL_ID: i32 = PINHOLE; }
impl GpuModelId for RadTanModel { const MODEL_ID: i32 = RAD_TAN; }
impl GpuModelId for KannalaBrandtModel { const MODEL_ID: i32 = KANNALA_BRANDT; }
impl GpuModelId for UcmModel { const MODEL_ID: i32 = UCM; }
impl GpuModelId for EucmModel { const MODEL_ID: i32 = EUCM; }
impl GpuModelId for DoubleSphereModel { const MODEL_ID: i32 = DOUBLE_SPHERE; }
impl GpuModelId for FovModel { const MODEL_ID: i32 = FOV; }

/// A reference model (`M: CameraModel`, e.g. `DoubleSphereModel`) whose per-point work runs on the GPU.
/// Owns a share of its context, so it is `'static` and fits `Box<dyn CameraModel>`.
pub struct GpuCamera<M: CameraModel> {
    pub inner: M,
    pub model_id: i32,
    ctx: Arc<Context>,
}

impl<M: CameraModel + GpuModelId> GpuCamera<M> {
    /// Wrap a reference model; the model id comes from its type.
    pub fn wrap(ctx: Arc<Context>, inner: M) -> Self { GpuCamera { inner, model_id: M::MODEL_ID, ctx } }
}

/// The drop-in: everything that is not per-point work is the wrapped model's own code
/// (reference src/camera/mod.rs:241-340), `project` / `unproject` run on the GPU.
impl<M: CameraModel + GpuModelId> CameraModel for GpuCamera<M> {
    fn project(&self, point_3d: &Vector3<f64>) -> Result<Vector2<f64>, CameraModelError> { self.project_point(point_3d) }
    fn unproject(&self, point_2d: &Vector2<f64>) -> Result<Vector3<f64>, CameraModelError> { self.unproject_point(point_2d) }
    fn load_from_yaml(path: &str) -> Result<Self, CameraModelError>
    where
        Self: Sized,
    {
        let inner = M::load_from_yaml(path)?;
        Ok(GpuCamera::wrap(Context::global()?, inner))
    }
    fn save_to_yaml(&self, path: &str) -> Result<(), CameraModelError> { self.inner.save_to_yaml(path) }
    fn validate_params(&self) -> Result<(), CameraModelError> { self.inner.validate_params() }
    fn get_resolution(&self) -> Resolution { self.inner.get_resolution() }
    fn get_intrinsics(&self) -> Intrinsics { self.inner.get_intrinsics() }
    fn get_distortion(&self) -> Vec<f64> { self.inner.get_distortion() }
    fn get_model_name(&self) -> &'static str { self.inner.get_model_name() }
}

/// `create_input_model` of the converter (camera_converter.rs:87-125) with GPU-backed models: the same
/// `Box<dyn CameraModel>` the rest of `main` consumes.
pub fn create_input_model(model_type: &str, path: &str) -> Result<Box<dyn CameraModel>, CameraModelError> {
    Ok(match model_type.to_lowercase().as_str() {
        "kb" | "kannala_brandt" => Box::new(GpuCamera::<KannalaBrandtModel>::load_from_yaml(path)?),
        "ds" | "double_sphere" => Box::new(GpuCamera::<DoubleSphereModel>::load_from_yaml(path)?),
        "radtan" | "rad_tan" => Box::new(GpuCamera::<RadTanModel>::load_from_yaml(path)?),
        "ucm" | "unified" => Box::new(GpuCamera::<UcmModel>::load_from_yaml(path)?),
        "eucm" | "extended_unified" => Box::new(GpuCamera::<EucmModel>::load_from_yaml(path)?),
        "pinhole" => Box::new(GpuCamera::<PinholeModel>::load_from_yaml(path)?),
        "fov" => Box::new(GpuCamera::<FovModel>::load_from_yaml(path)?),
        other => return Err(CameraModelError::InvalidParams(format!("Unsupported input model type: {other}"))),
    })
}

impl<M: CameraModel> GpuCamera<M> {
    pub fn new(ctx: Arc<Context>, inner: M, model_id: i32) -> Self { GpuCamera { inner, model_id, ctx } }
    pub fn context(&self) -> &Arc<Context> { &self.ctx }
    pub fn camera_block(&self) -> sys::acm_camera { self.block() }

    fn block(&self) -> sys::acm_camera {
        let i = self.inner.get_intrinsics();
        let r = self.inner.get_resolution();
        let d = self.inner.get_distortion();
        let mut params = [0.0f64; sys::ACM_MAX_PARAMS];
        params[..4].copy_from_slice(&[i.fx, i.fy, i.cx, i.cy]);
        params[4..4 + d.len()].copy_from_slice(&d);
        sys::acm_camera { model: self.model_id, width: r.width, height: r.height, n_params: (4 + d.len()) as i32, params }
    }

    /// Batched `project`: returns (uv, status byte per point). Matrix3xX memory is xyzxyz.. as the ABI expects.
    pub fn project_batch(&self, points_3d: &Matrix3xX<f64>) -> Result<(Matrix2xX<f64>, Vec<u8>), CameraModelError> {
        let n = points_3d.ncols();
        let mut uv = Matrix2xX::<f64>::zeros(n);
        let mut st = vec![0u8; n];
        let cam = self.block();
        let _g = self.ctx.lock();
        let rc = unsafe { sys::acm_project_host(self.ctx.0, &cam, points_3d.as_ptr(), n, uv.as_mut_ptr(), st.as_mut_ptr()) };
        if rc != sys::ACM_OK { return Err(self.ctx.err(rc)); }
        Ok((uv, st))
    }

    pub fn unproject_batch(&self, points_2d: &Matrix2xX<f64>) -> Result<(Matrix3xX<f64>, Vec<u8>), CameraModelError> {
        let n = points_2d.ncols();
        let mut xyz = Matrix3xX::<f64>::zeros(n);
        let mut st = vec![0u8; n];
        let cam = self.block();
        let _g = self.ctx.lock();
        let rc = unsafe { sys::acm_unproject_host(self.ctx.0, &cam, points_2d.as_ptr(), n, xyz.as_mut_ptr(), st.as_mut_ptr()) };
        if rc != sys::ACM_OK { return Err(self.ctx.err(rc)); }
        Ok((xyz, st))
    }

    /// `CameraModel::project` (mod.rs:256) for one point: the library's small-batch path (mapped pinned staging,
    /// one kernel, one synchronisation -- no allocation), no matrix temporaries here.
    pub fn project_point(&self, p: &Vector3<f64>) -> Result<Vector2<f64>, CameraModelError> {
        let cam = self.block();
        let (mut uv, mut st) = ([0.0f64; 2], [0u8; 1]);
        let _g = self.ctx.lock();
        let rc = unsafe { sys::acm_project_host(self.ctx.0, &cam, p.as_ptr(), 1, uv.as_mut_ptr(), st.as_mut_ptr()) };
        if rc != sys::ACM_OK { return Err(self.ctx.err(rc)); }
        match status_to_error(st[0], self.model_id) { Some(e) => Err(e), None => Ok(Vector2::new(uv[0], uv[1])) }
    }

    pub fn unproject_point(&self, p: &Vector2<f64>) -> Result<Vector3<f64>, CameraModelError> {
        let cam = self.block();
        let (mut xyz, mut st) = ([0.0f64; 3], [0u8; 1]);
        let _g = self.ctx.lock();
        let rc = unsafe { sys::acm_unproject_host(self.ctx.0, &cam, p.as_ptr(), 1, xyz.as_mut_ptr(), st.as_mut_ptr()) };
        if rc != sys::ACM_OK { return Err(self.ctx.err(rc)); }
        match status_to_error(st[0], self.model_id) { Some(e) => Err(e), None => Ok(Vector3::new(xyz[0], xyz[1], xyz[2])) }
    }

    /// One fused pass: (H = J^T J, g = J^T r, cost, n_valid) -- what `Factor::linearize` + the solver's
    /// J^T J produce in apex-solver, without materialising J.
    pub fn linearize(&self, residual_kind: i32, points_3d: &Matrix3xX<f64>, points_2d: &Matrix2xX<f64>)
        -> Result<sys::acm_normal_equations, CameraModelError> {
        if points_3d.ncols() != points_2d.ncols() {
            return Err(CameraModelError::InvalidParams("Number of 2D and 3D points must match".into()));
        }
        let cam = self.block();
        let mut ne: sys::acm_normal_equations = unsafe { std::mem::zeroed() };
        let _g = self.ctx.lock();
        let rc = unsafe { sys::acm_linearize_host(self.ctx.0, &cam, residual_kind, points_3d.as_ptr(), points_2d.as_ptr(), points_3d.ncols(), &mut ne) };
        if rc != sys::ACM_OK { return Err(self.ctx.err(rc)); }
        Ok(ne)
    }
}

/// Device point buffer owned for the duration of a call.
struct DevicePoints<'c> { ctx: &'c Context, h: *mut sys::acm_points }
impl<'c> DevicePoints<'c> {
    fn upload(ctx: &'c Context, dim: i32, host: *const f64, n: usize) -> Result<Self, CameraModelError> {
        let mut h = ptr::null_mut();
        let mut rc = unsafe { sys::acm_points_create(ctx.0, dim, n, sys::ACM_F64, &mut h) };
        if rc == sys::ACM_OK && n > 0 { rc = unsafe { sys::acm_points_upload_aos_f64(ctx.0, h, host, n) }; }
        if rc != sys::ACM_OK { unsafe { sys::acm_points_destroy(ctx.0, h); } return Err(ctx.err(rc)); }
        Ok(DevicePoints { ctx, h })
    }
    fn adopt(ctx: &'c Context, h: *mut sys::acm_points) -> Self { DevicePoints { ctx, h } }
    fn len(&self) -> usize { unsafe { sys::acm_points_len(self.h) } }
    fn download(&self, out: *mut f64) -> Result<(), CameraModelError> {
        let rc = unsafe { sys::acm_points_download_aos_f64(self.ctx.0, self.h, out, self.len()) };
        if rc != sys::ACM_OK { Err(self.ctx.err(rc)) } else { Ok(()) }
    }
}
impl<'c> Drop for DevicePoints<'c> { fn drop(&mut self) { unsafe { sys::acm_points_destroy(self.ctx.0, self.h); } } }

impl<M: CameraModel> GpuCamera<M> {
    /// `util::sample_points(Some(&model), n) -> (Matrix2xX, Matrix3xX)` (point_sampling.rs:46-120):
    /// grid of cell centres -> unproject -> keep Ok && z > 0, order preserved.
    pub fn sample_points(&self, n: usize) -> Result<(Matrix2xX<f64>, Matrix3xX<f64>), CameraModelError> {
        let cam = self.block();
        let (mut uv, mut xyz, mut kept) = (ptr::null_mut(), ptr::null_mut(), 0usize);
        let _g = self.ctx.lock();
        let rc = unsafe { sys::acm_sample_points(self.ctx.0, &cam, n, &mut uv, &mut xyz, &mut kept) };
        if rc != sys::ACM_OK { return Err(self.ctx.err(rc)); }
        let (uv, xyz) = (DevicePoints::adopt(&self.ctx, uv), DevicePoints::adopt(&self.ctx, xyz));
        let mut p2 = Matrix2xX::<f64>::zeros(kept);
        let mut p3 = Matrix3xX::<f64>::zeros(kept);
        uv.download(p2.as_mut_ptr())?;
        xyz.download(p3.as_mut_ptr())?;
        Ok((p2, p3))
    }

    /// `util::compute_reprojection_error(Some(&model), &points3d, &points2d)` (error_metrics.rs:62-121).
    pub fn compute_reprojection_error(&self, points_3d: &Matrix3xX<f64>, points_2d: &Matrix2xX<f64>)
        -> Result<sys::acm_projection_error, CameraModelError> {
        if points_3d.ncols() != points_2d.ncols() {
            return Err(CameraModelError::InvalidParams("Number of 2D and 3D points must match".into()));
        }
        let n = points_3d.ncols();
        let _g = self.ctx.lock();
        let x = DevicePoints::upload(&self.ctx, 3, points_3d.as_ptr(), n)?;
        let u = DevicePoints::upload(&self.ctx, 2, points_2d.as_ptr(), n)?;
        let cam = self.block();
        let mut out = sys::acm_projection_error::default();
        let rc = unsafe { sys::acm_reprojection_error(self.ctx.0, &cam, x.h, u.h, &mut out) };
        if rc != sys::ACM_OK { return Err(self.ctx.err(rc)); }   // -7 -> UtilError::ZeroProjectionPoints upstream
        Ok(out)
    }

    /// `util::undistort_image(&img, &model, target, method)` (undistort.rs:14-49) over the raw RGB8 buffer
    /// (`RgbImage::as_raw()`); `interpolation` = `sys::ACM_INTERP_NEAREST | ACM_INTERP_BILINEAR`.
    pub fn undistort_image(&self, image: &[u8], width: u32, height: u32, target: Option<Intrinsics>, interpolation: i32)
        -> Result<Vec<u8>, CameraModelError> {
        let r = self.inner.get_resolution();
        if width != r.width || height != r.height || image.len() != width as usize * height as usize * 3 {   // undistort.rs:23-28
            return Err(CameraModelError::InvalidParams(format!("Image {}x{} doesn't match model {}x{}", width, height, r.width, r.height)));
        }
        let cam = self.block();
        let t = target.map(|t| [t.fx, t.fy, t.cx, t.cy]);
        let mut out = vec![0u8; image.len()];
        let _g = self.ctx.lock();
        let rc = unsafe {
            sys::acm_undistort_rgb8_host(self.ctx.0, &cam, t.as_ref().map_or(ptr::null(), |a| a.as_ptr()), image.as_ptr(), out.as_mut_ptr(), 1, interpolation)
        };
        if rc != sys::ACM_OK { Err(self.ctx.err(rc)) } else { Ok(out) }
    }

    /// Remap plan from this camera to `output` (`None`: `undistort_image` with `target`); see [`RemapPlan`].
    pub fn remap_plan<O: CameraModel>(&self, output: Option<&GpuCamera<O>>, target: Option<Intrinsics>, interpolation: i32)
        -> Result<RemapPlan, CameraModelError> {
        let cam = self.block();
        let out_cam = output.map(|o| o.block());
        let (wo, ho) = match output { Some(o) => { let r = o.inner.get_resolution(); (r.width, r.height) } None => { let r = self.inner.get_resolution(); (r.width, r.height) } };
        let r = self.inner.get_resolution();
        let t = target.map(|t| [t.fx, t.fy, t.cx, t.cy]);
        let mut h: *mut sys::acm_remap_plan = ptr::null_mut();
        let _g = self.ctx.lock();
        let rc = unsafe {
            sys::acm_remap_plan_create(self.ctx.0, &cam, out_cam.as_ref().map_or(ptr::null(), |c| c as *const sys::acm_camera),
                                       t.as_ref().map_or(ptr::null(), |a| a.as_ptr()), interpolation, &mut h)
        };
        if rc != sys::ACM_OK { return Err(self.ctx.err(rc)); }
        Ok(RemapPlan { h, ctx: self.ctx.clone(), wi: r.width, hi: r.height, wo, ho })
    }

    /// Rotated remap plan from this camera to `output` (stereo rectification): `r` row-major with x_out = R x_in
    /// (OpenCV's R1 / R2, see [`stereo_rectify`]); the ray between the two models is R^T ray_out.
    pub fn remap_plan_rotated<O: CameraModel>(&self, output: &GpuCamera<O>, r: &[f64; 9], interpolation: i32)
        -> Result<RemapPlan, CameraModelError> {
        let (cam, out_cam) = (self.block(), output.block());
        let (ri, ro) = (self.inner.get_resolution(), output.inner.get_resolution());
        let mut h: *mut sys::acm_remap_plan = ptr::null_mut();
        let _g = self.ctx.lock();
        let rc = unsafe { sys::acm_remap_plan_create_rotated(self.ctx.0, &cam, &out_cam, r.as_ptr(), interpolation, &mut h) };
        if rc != sys::ACM_OK { return Err(self.ctx.err(rc)); }
        Ok(RemapPlan { h, ctx: self.ctx.clone(), wi: ri.width, hi: ri.height, wo: ro.width, ho: ro.height })
    }

    /// README-era `project(&p, compute_jacobian = true)`: uv plus the 2xP Jacobian w.r.t. `[fx, fy, cx, cy, dist..]`
    /// (per-model docs, double_sphere.rs:326-332) and the 2x3 Jacobian w.r.t. the 3-D point (trait doc, mod.rs:246-252).
    pub fn project_with_jacobians(&self, p: &Vector3<f64>)
        -> Result<(Vector2<f64>, nalgebra::DMatrix<f64>, nalgebra::Matrix2x3<f64>), CameraModelError> {
        let cam = self.block();
        let np = cam.n_params as usize;
        let _g = self.ctx.lock();
        let x = DevicePoints::upload(&self.ctx, 3, p.as_ptr(), 1)?;
        let u = DevicePoints::upload(&self.ctx, 2, [0.0f64; 2].as_ptr(), 1)?;
        let (mut dj, mut ds) = (ptr::null_mut(), ptr::null_mut());
        let mut rc = unsafe { sys::acm_device_alloc(self.ctx.0, (2 * np + 6) * 8, &mut dj) };
        if rc == sys::ACM_OK { rc = unsafe { sys::acm_device_alloc(self.ctx.0, 8, &mut ds) }; }
        let mut jp = vec![0.0f64; 2 * np];
        let mut jx = [0.0f64; 6];
        let mut st = [0u8; 1];
        let mut uv = [0.0f64; 2];
        unsafe {
            let djp = dj as *mut f64;
            let djx = djp.add(2 * np);
            if rc == sys::ACM_OK { rc = sys::acm_project_jacobian(self.ctx.0, &cam, x.h, u.h, djp, ds as *mut u8); }
            if rc == sys::ACM_OK { rc = sys::acm_project_point_jacobian(self.ctx.0, &cam, x.h, u.h, djx, ds as *mut u8); }
            if rc == sys::ACM_OK { rc = sys::acm_memcpy_d2h(self.ctx.0, jp.as_mut_ptr() as *mut _, djp as *const _, 2 * np * 8); }
            if rc == sys::ACM_OK { rc = sys::acm_memcpy_d2h(self.ctx.0, jx.as_mut_ptr() as *mut _, djx as *const _, 48); }
            if rc == sys::ACM_OK { rc = sys::acm_memcpy_d2h(self.ctx.0, st.as_mut_ptr() as *mut _, ds as *const _, 1); }
            if rc == sys::ACM_OK { rc = sys::acm_points_download_aos_f64(self.ctx.0, u.h, uv.as_mut_ptr(), 1); }
            if rc == sys::ACM_OK { rc = sys::acm_ctx_sync(self.ctx.0); }
            sys::acm_device_free(self.ctx.0, dj); sys::acm_device_free(self.ctx.0, ds);
        }
        if rc != sys::ACM_OK { return Err(self.ctx.err(rc)); }
        if let Some(e) = status_to_error(st[0], self.model_id) { return Err(e); }
        // one point: the rows of n doubles are the row-major matrices themselves
        Ok((Vector2::new(uv[0], uv[1]), nalgebra::DMatrix::from_row_slice(2, np, &jp), nalgebra::Matrix2x3::from_row_slice(&jx)))
    }
}

/// Resident correspondences + optimiser: the README-era `*OptimizationCost` and the converter's
/// `Problem` + `LevenbergMarquardt::with_config(cfg).optimize(..)` (camera_converter.rs:378-420).
pub struct OptimizationCost {
    ctx: Arc<Context>,
    pub camera: sys::acm_camera,
    xyz: *mut sys::acm_points,
    uv: *mut sys::acm_points,
    pub residual_kind: i32,
}

impl OptimizationCost {
    pub fn new(ctx: Arc<Context>, camera: sys::acm_camera, points_3d: &Matrix3xX<f64>, points_2d: &Matrix2xX<f64>, residual_kind: i32)
        -> Result<Self, CameraModelError> {
        assert_eq!(points_3d.ncols(), points_2d.ncols());
        let n = points_3d.ncols();
        let (mut xyz, mut uv) = (ptr::null_mut(), ptr::null_mut());
        let _g = ctx.lock();
        unsafe {
            let mut rc = sys::acm_points_create(ctx.0, 3, n, sys::ACM_F64, &mut xyz);
            if rc == sys::ACM_OK { rc = sys::acm_points_create(ctx.0, 2, n, sys::ACM_F64, &mut uv); }
            if rc == sys::ACM_OK { rc = sys::acm_points_upload_aos_f64(ctx.0, xyz, points_3d.as_ptr(), n); }
            if rc == sys::ACM_OK { rc = sys::acm_points_upload_aos_f64(ctx.0, uv, points_2d.as_ptr(), n); }
            if rc == sys::ACM_OK { rc = sys::acm_ctx_sync(ctx.0); }
            if rc != sys::ACM_OK { return Err(ctx.err(rc)); }
        }
        drop(_g);
        Ok(OptimizationCost { ctx, camera, xyz, uv, residual_kind })
    }

    pub fn linear_estimation(&mut self) -> Result<(), CameraModelError> {
        let _g = self.ctx.lock();
        let rc = unsafe { sys::acm_linear_estimation(self.ctx.0, &mut self.camera, self.xyz, self.uv) };
        if rc != sys::ACM_OK { Err(self.ctx.err(rc)) } else { Ok(()) }
    }

    /// `bounds`: (lower, upper) per parameter = `problem.set_variable_bounds("params", i, lo, hi)`.
    pub fn optimize(&mut self, bounds: Option<(&[f64], &[f64])>, cfg: Option<sys::acm_lm_config>)
        -> Result<(DVector<f64>, sys::acm_lm_result), CameraModelError> {
        let mut c = unsafe { std::mem::zeroed::<sys::acm_lm_config>() };
        unsafe { sys::acm_lm_default_config(&mut c); }
        let c = cfg.unwrap_or(c);
        let (lo, hi) = match bounds { Some((l, h)) => (l.as_ptr(), h.as_ptr()), None => (ptr::null(), ptr::null()) };
        let mut out = [0.0f64; sys::ACM_MAX_PARAMS];
        let mut res = sys::acm_lm_result::default();
        let _g = self.ctx.lock();
        let rc = unsafe { sys::acm_lm_solve(self.ctx.0, &self.camera, self.residual_kind, self.xyz, self.uv, lo, hi, &c, out.as_mut_ptr(), &mut res) };
        if rc != sys::ACM_OK { return Err(self.ctx.err(rc)); }
        let p = self.camera.n_params as usize;
        self.camera.params[..p].copy_from_slice(&out[..p]);
        Ok((DVector::from_column_slice(&out[..p]), res))
    }

    pub fn get_intrinsics(&self) -> Intrinsics {
        Intrinsics { fx: self.camera.params[0], fy: self.camera.params[1], cx: self.camera.params[2], cy: self.camera.params[3] }
    }
    pub fn get_distortion(&self) -> Vec<f64> { self.camera.params[4..self.camera.n_params as usize].to_vec() }
    pub fn get_resolution(&self) -> Resolution { Resolution { width: self.camera.width, height: self.camera.height } }
}

impl Drop for OptimizationCost {
    fn drop(&mut self) {
        let _g = self.ctx.lock();
        unsafe { sys::acm_points_destroy(self.ctx.0, self.xyz); sys::acm_points_destroy(self.ctx.0, self.uv); }
    }
}

/// Bounds of the converter's `problem.set_variable_bounds` calls and the residual each target minimises
/// (camera_converter.rs:395-400, :536-539, :676-680, :814, :946-947, :1078; SURVEY.md section 8c).
fn converter_bounds(model_id: i32) -> (Vec<f64>, Vec<f64>) {
    let (mut lo, mut hi) = (vec![1.0, 1.0, 0.0, 0.0], vec![2000.0, 2000.0, 2000.0, 2000.0]);
    let d: &[(f64, f64)] = match model_id {
        DOUBLE_SPHERE => &[(1e-6, 1.0), (-5.0, 5.0)],
        KANNALA_BRANDT => &[(-5.0, 5.0); 4],
        RAD_TAN => &[(-5.0, 5.0), (-5.0, 5.0), (-1.0, 1.0), (-1.0, 1.0), (-5.0, 5.0)],
        UCM => &[(1e-6, 10.0)],
        EUCM => &[(1e-6, 1.0), (1e-6, 5.0)],
        FOV => &[(1e-6, 3.0)],
        _ => &[],
    };
    for (l, h) in d { lo.push(*l); hi.push(*h); }
    (lo, hi)
}
fn canonical_residual(model_id: i32) -> i32 {
    match model_id { UCM | EUCM | DOUBLE_SPHERE => sys::ACM_RESIDUAL_ALGEBRAIC, _ => sys::ACM_RESIDUAL_PIXEL }
}

/// The README-era per-model facade (README.md:70-81):
/// `XOptimizationCost::new(initial_model, points_3d, points_2d)`, `.linear_estimation()?`, `.optimize(verbose)?`,
/// `.get_intrinsics()`, `.get_distortion()`.  One newtype per target model, all over `OptimizationCost`.
macro_rules! optimization_cost {
    ($name:ident, $model:ty) => {
        pub struct $name { pub cost: OptimizationCost, pub model: $model }
        impl $name {
            /// Uploads the correspondences once; they stay resident in HBM for `linear_estimation` and `optimize`.
            pub fn new(model: $model, points_3d: Matrix3xX<f64>, points_2d: Matrix2xX<f64>) -> Result<Self, CameraModelError> {
                if points_3d.ncols() != points_2d.ncols() {
                    return Err(CameraModelError::InvalidParams("Number of 2D and 3D points must match".into()));
                }
                let ctx = Context::global()?;
                let id = <$model as GpuModelId>::MODEL_ID;
                let block = GpuCamera::new(ctx.clone(), model.clone(), id).camera_block();
                let cost = OptimizationCost::new(ctx, block, &points_3d, &points_2d, canonical_residual(id))?;
                Ok($name { cost, model })
            }
            fn sync_model(&mut self) -> Result<(), CameraModelError> {
                let p = self.cost.camera.n_params as usize;
                let resolution = self.model.resolution.clone();   // `new` resets it to 0 x 0 (double_sphere.rs:149-152)
                self.model = <$model>::new(&DVector::from_column_slice(&self.cost.camera.params[..p]))?;
                self.model.resolution = resolution;
                Ok(())
            }
            pub fn linear_estimation(&mut self) -> Result<(), CameraModelError> {
                self.cost.linear_estimation()?;
                self.sync_model()
            }
            /// Levenberg-Marquardt with the converter's tolerances and bounds (camera_converter.rs:395-415).
            pub fn optimize(&mut self, verbose: bool) -> Result<(), CameraModelError> {
                let (lo, hi) = converter_bounds(<$model as GpuModelId>::MODEL_ID);
                let (_, res) = self.cost.optimize(Some((&lo, &hi)), None)?;
                if verbose {
                    println!("[LM] status={} iterations={} passes={} cost {:.6e} -> {:.6e} ({:.3} ms on the device)",
                             res.status, res.iterations, res.passes, res.initial_cost, res.final_cost, res.device_ms);
                }
                self.sync_model()
            }
            pub fn get_intrinsics(&self) -> Intrinsics { self.cost.get_intrinsics() }
            pub fn get_distortion(&self) -> Vec<f64> { self.cost.get_distortion() }
        }
    };
}
optimization_cost!(DoubleSphereOptimizationCost, DoubleSphereModel);
optimization_cost!(KannalaBrandtOptimizationCost, KannalaBrandtModel);
optimization_cost!(RadTanOptimizationCost, RadTanModel);
optimization_cost!(UcmOptimizationCost, UcmModel);
optimization_cost!(EucmOptimizationCost, EucmModel);
optimization_cost!(FovOptimizationCost, FovModel);

/// Every GPU of the box from ONE host thread (the converter's `main` has no launcher):
/// `acm_comm_init_all` + the `acm_*_multi` entry points.  Correspondences are sharded by contiguous
/// column ranges `[r*N/G, (r+1)*N/G)`; every call returns the result all ranks agree on.
pub struct DeviceGroup {
    ctxs: Vec<Arc<Context>>,
    raw: Vec<*mut sys::acm_ctx>,
}
pub struct ShardedCorrespondences { xyz: Vec<*mut sys::acm_points>, uv: Vec<*mut sys::acm_points>, owners: Vec<Arc<Context>> }
impl Drop for ShardedCorrespondences {
    fn drop(&mut self) {
        for (i, c) in self.owners.iter().enumerate() { unsafe { sys::acm_points_destroy(c.0, self.xyz[i]); sys::acm_points_destroy(c.0, self.uv[i]); } }
    }
}

impl DeviceGroup {
    pub fn new(devices: &[i32]) -> Result<Self, CameraModelError> {
        let ctxs = devices.iter().map(|d| Context::new(*d).map(Arc::new)).collect::<Result<Vec<_>, _>>()?;
        let mut raw: Vec<_> = ctxs.iter().map(|c| c.0).collect();
        let rc = unsafe { sys::acm_comm_init_all(raw.as_mut_ptr(), raw.len() as i32) };
        if rc != sys::ACM_OK { return Err(ctxs[0].err(rc)); }
        Ok(DeviceGroup { ctxs, raw })
    }
    pub fn len(&self) -> usize { self.ctxs.len() }

    /// Upload contiguous column shards of the correspondences, one per GPU.
    pub fn shard(&self, points_3d: &Matrix3xX<f64>, points_2d: &Matrix2xX<f64>) -> Result<ShardedCorrespondences, CameraModelError> {
        if points_3d.ncols() != points_2d.ncols() {
            return Err(CameraModelError::InvalidParams("Number of 2D and 3D points must match".into()));
        }
        let (n, g) = (points_3d.ncols(), self.len());
        let mut out = ShardedCorrespondences { xyz: vec![], uv: vec![], owners: vec![] };
        for (r, c) in self.ctxs.iter().enumerate() {
            let (lo, hi) = (n * r / g, n * (r + 1) / g);
            let x = DevicePoints::upload(c, 3, unsafe { points_3d.as_ptr().add(3 * lo) }, hi - lo)?;
            let u = DevicePoints::upload(c, 2, unsafe { points_2d.as_ptr().add(2 * lo) }, hi - lo)?;
            out.xyz.push(x.h); out.uv.push(u.h); out.owners.push(c.clone());
            std::mem::forget(x); std::mem::forget(u);   // ownership moves into `out`
        }
        Ok(out)
    }

    pub fn linear_estimation(&mut self, cam: &mut sys::acm_camera, pts: &ShardedCorrespondences) -> Result<(), CameraModelError> {
        let rc = unsafe { sys::acm_linear_estimation_multi(self.raw.as_mut_ptr(), self.raw.len() as i32, cam, pts.xyz.as_ptr(), pts.uv.as_ptr()) };
        if rc != sys::ACM_OK { Err(self.ctxs[0].err(rc)) } else { Ok(()) }
    }

    pub fn linearize(&mut self, cam: &sys::acm_camera, residual_kind: i32, pts: &ShardedCorrespondences) -> Result<sys::acm_normal_equations, CameraModelError> {
        let mut ne: sys::acm_normal_equations = unsafe { std::mem::zeroed() };
        let rc = unsafe { sys::acm_linearize_multi(self.raw.as_mut_ptr(), self.raw.len() as i32, cam, residual_kind, pts.xyz.as_ptr(), pts.uv.as_ptr(), &mut ne) };
        if rc != sys::ACM_OK { Err(self.ctxs[0].err(rc)) } else { Ok(ne) }
    }

    /// The whole LM solve on all GPUs: one persistent kernel per GPU, the normal equations summed over NVLink inside it.
    pub fn optimize(&mut self, cam: &mut sys::acm_camera, residual_kind: i32, pts: &ShardedCorrespondences, bounds: Option<(&[f64], &[f64])>)
        -> Result<sys::acm_lm_result, CameraModelError> {
        let (lo, hi) = match bounds { Some((l, h)) => (l.as_ptr(), h.as_ptr()), None => (ptr::null(), ptr::null()) };
        let mut out = [0.0f64; sys::ACM_MAX_PARAMS];
        let mut res = sys::acm_lm_result::default();
        let rc = unsafe {
            sys::acm_lm_solve_multi(self.raw.as_mut_ptr(), self.raw.len() as i32, cam, residual_kind, pts.xyz.as_ptr(), pts.uv.as_ptr(), lo, hi,
                                    ptr::null(), out.as_mut_ptr(), &mut res)
        };
        if rc != sys::ACM_OK { return Err(self.ctxs[0].err(rc)); }
        let p = cam.n_params as usize;
        cam.params[..p].copy_from_slice(&out[..p]);
        Ok(res)
    }

    pub fn compute_reprojection_error(&mut self, cam: &sys::acm_camera, pts: &ShardedCorrespondences) -> Result<sys::acm_projection_error, CameraModelError> {
        let mut out = sys::acm_projection_error::default();
        let rc = unsafe { sys::acm_reprojection_error_multi(self.raw.as_mut_ptr(), self.raw.len() as i32, cam, pts.xyz.as_ptr(), pts.uv.as_ptr(), &mut out) };
        if rc != sys::ACM_OK { Err(self.ctxs[0].err(rc)) } else { Ok(out) }
    }

    /// `sample_points` with the grid cells split over the GPUs; the shards stay resident, concatenated in rank order
    /// they are bit for bit the single-GPU output.
    pub fn sample_points(&mut self, cam: &sys::acm_camera, n: usize) -> Result<(ShardedCorrespondences, usize), CameraModelError> {
        let g = self.len();
        let (mut uv, mut xyz, mut kept) = (vec![ptr::null_mut(); g], vec![ptr::null_mut(); g], vec![0usize; g]);
        let rc = unsafe { sys::acm_sample_points_multi(self.raw.as_mut_ptr(), g as i32, cam, n, uv.as_mut_ptr(), xyz.as_mut_ptr(), kept.as_mut_ptr()) };
        if rc != sys::ACM_OK { return Err(self.ctxs[0].err(rc)); }
        Ok((ShardedCorrespondences { xyz, uv, owners: self.ctxs.clone() }, kept.iter().sum()))
    }
}
impl Drop for DeviceGroup {
    fn drop(&mut self) { unsafe { sys::acm_comm_destroy_all(self.raw.as_mut_ptr(), self.raw.len() as i32); } }
}

/// RGB8 frames of one camera rendered as another camera sees them (beyond the reference: the output camera's
/// `unproject`, the input camera's `project`, then `interpolate_pixel`, undistort.rs:51-105).  The source coordinates
/// are computed once on the device (32 bytes per output pixel) and reused by every `apply`; dropped with the plan.
pub struct RemapPlan { h: *mut sys::acm_remap_plan, ctx: Arc<Context>, wi: u32, hi: u32, wo: u32, ho: u32 }
unsafe impl Send for RemapPlan {}

impl RemapPlan {
    /// `frames`: whole Wi x Hi RGB8 frames of the input camera; returns the Wo x Ho frames of the output camera.
    pub fn apply(&self, frames: &[u8]) -> Result<Vec<u8>, CameraModelError> {
        let fin = self.wi as usize * self.hi as usize * 3;
        if frames.len() % fin != 0 {   // undistort.rs:23-28
            return Err(CameraModelError::InvalidParams(format!("frames of {} bytes don't match model {}x{}", frames.len(), self.wi, self.hi)));
        }
        let n = frames.len() / fin;
        let mut out = vec![0u8; n * self.wo as usize * self.ho as usize * 3];
        let _g = self.ctx.lock();
        let rc = unsafe { sys::acm_remap_rgb8_host(self.ctx.0, self.h, frames.as_ptr(), out.as_mut_ptr(), n) };
        if rc != sys::ACM_OK { Err(self.ctx.err(rc)) } else { Ok(out) }
    }
    /// Frames resident on the plan's device, enqueued on the context's stream.
    ///
    /// # Safety
    /// `d_in` / `d_out` must be device buffers of `n_frames` input / output frames.
    pub unsafe fn apply_device(&self, d_in: *const u8, d_out: *mut u8, n_frames: usize) -> Result<(), CameraModelError> {
        let _g = self.ctx.lock();
        let rc = sys::acm_remap_rgb8(self.ctx.0, self.h, d_in, d_out, n_frames);
        if rc != sys::ACM_OK { Err(self.ctx.err(rc)) } else { Ok(()) }
    }
    /// Output resolution (width, height).
    pub fn output_size(&self) -> (u32, u32) { (self.wo, self.ho) }
}
impl Drop for RemapPlan {
    fn drop(&mut self) { let _g = self.ctx.lock(); unsafe { sys::acm_remap_plan_destroy(self.ctx.0, self.h); } }
}

/// Bouguet rectification of a calibrated pair, x_cam2 = R x_cam1 + t (the rotation part of OpenCV's `stereoRectify`;
/// host only).  x_rect1 = R1 x_cam1, x_rect2 = R2 x_cam2; `baseline` is the component of R2 t along x (along y when
/// `vertical`).  With one pinhole camera K for both views, P1 = K [I | 0] and P2 = K [I | baseline e].
#[derive(Debug, Clone)]
pub struct StereoRectification { pub r1: [f64; 9], pub r2: [f64; 9], pub baseline: f64, pub vertical: bool }

/// `r` row-major, `t` as in x_cam2 = R x_cam1 + t; see [`StereoRectification`].
pub fn stereo_rectify(r: &[f64; 9], t: &[f64; 3]) -> Result<StereoRectification, CameraModelError> {
    let mut s = StereoRectification { r1: [0.0; 9], r2: [0.0; 9], baseline: 0.0, vertical: false };
    let mut vertical = 0i32;
    let rc = unsafe { sys::acm_stereo_rectify(r.as_ptr(), t.as_ptr(), s.r1.as_mut_ptr(), s.r2.as_mut_ptr(), &mut s.baseline, &mut vertical) };
    if rc != sys::ACM_OK {
        let msg = unsafe { CStr::from_ptr(sys::acm_last_error(ptr::null())) }.to_string_lossy().into_owned();
        return Err(CameraModelError::InvalidParams(msg));
    }
    s.vertical = vertical != 0;
    Ok(s)
}

/// `util::ImageQualityMetrics` (image_quality.rs:20-26).
#[derive(Debug, Clone)]
pub struct ImageQualityMetrics { pub psnr: f64, pub ssim: f64 }

/// RGB8 image staged in HBM for the duration of a call.
struct DeviceImage<'c> { ctx: &'c Context, ptr: *mut std::ffi::c_void, bytes: usize }
impl<'c> DeviceImage<'c> {
    fn new(ctx: &'c Context, bytes: usize, host: Option<&[u8]>) -> Result<Self, CameraModelError> {
        let mut p = ptr::null_mut();
        let mut rc = unsafe { sys::acm_device_alloc(ctx.0, bytes.max(4), &mut p) };
        if rc == sys::ACM_OK && bytes > 0 {
            rc = match host {
                Some(h) => unsafe { sys::acm_memcpy_h2d(ctx.0, p, h.as_ptr() as *const _, bytes) },
                None => unsafe { sys::acm_memset_d(ctx.0, p, 0, bytes) },
            };
        }
        if rc != sys::ACM_OK { return Err(ctx.err(rc)); }
        Ok(DeviceImage { ctx, ptr: p, bytes })
    }
    fn download(&self) -> Result<Vec<u8>, CameraModelError> {
        let mut out = vec![0u8; self.bytes];
        let mut rc = unsafe { sys::acm_memcpy_d2h(self.ctx.0, out.as_mut_ptr() as *mut _, self.ptr, self.bytes) };
        if rc == sys::ACM_OK { rc = unsafe { sys::acm_ctx_sync(self.ctx.0) }; }
        if rc != sys::ACM_OK { Err(self.ctx.err(rc)) } else { Ok(out) }
    }
}
impl<'c> Drop for DeviceImage<'c> { fn drop(&mut self) { unsafe { sys::acm_device_free(self.ctx.0, self.ptr); } } }

/// `util::calculate_psnr(&RgbImage, &RgbImage)` (image_quality.rs:45-89) over raw RGB8 buffers
/// (`RgbImage::as_raw()`), `width` x `height`.
pub fn calculate_psnr(ctx: &Context, img1: &[u8], img2: &[u8], width: u32, height: u32) -> Result<f64, CameraModelError> {
    if img1.len() != img2.len() { return Err(CameraModelError::InvalidParams("Images must have the same dimensions".into())); }
    let (a, b) = (DeviceImage::new(ctx, img1.len(), Some(img1))?, DeviceImage::new(ctx, img2.len(), Some(img2))?);
    let mut out = 0.0f64;
    let rc = unsafe { sys::acm_image_psnr(ctx.0, a.ptr as *const u8, b.ptr as *const u8, width, height, &mut out) };
    if rc != sys::ACM_OK { Err(ctx.err(rc)) } else { Ok(out) }
}

/// `util::calculate_ssim` (image_quality.rs:108-210).
pub fn calculate_ssim(ctx: &Context, img1: &[u8], img2: &[u8], width: u32, height: u32) -> Result<f64, CameraModelError> {
    if img1.len() != img2.len() { return Err(CameraModelError::InvalidParams("Images must have the same dimensions".into())); }
    let (a, b) = (DeviceImage::new(ctx, img1.len(), Some(img1))?, DeviceImage::new(ctx, img2.len(), Some(img2))?);
    let mut out = 0.0f64;
    let rc = unsafe { sys::acm_image_ssim(ctx.0, a.ptr as *const u8, b.ptr as *const u8, width, height, &mut out) };
    if rc != sys::ACM_OK { Err(ctx.err(rc)) } else { Ok(out) }
}

/// `util::compute_image_quality_metrics` (image_quality.rs:254-324) over camera blocks; returns the metrics and,
/// when `want_image`, the combined display image (green input / magenta output projections over `reference`).
pub fn compute_image_quality_metrics(ctx: &Context, input_model: &sys::acm_camera, output_model: &sys::acm_camera,
                                     points_3d: &Matrix3xX<f64>, width: u32, height: u32, reference: Option<&[u8]>, want_image: bool)
    -> Result<(ImageQualityMetrics, Option<Vec<u8>>), CameraModelError> {
    let n = points_3d.ncols();
    let bytes = width as usize * height as usize * 3;
    let mut xyz = ptr::null_mut();
    let mut rc = unsafe { sys::acm_points_create(ctx.0, 3, n, sys::ACM_F64, &mut xyz) };
    if rc == sys::ACM_OK { rc = unsafe { sys::acm_points_upload_aos_f64(ctx.0, xyz, points_3d.as_ptr(), n) }; }
    if rc != sys::ACM_OK { unsafe { sys::acm_points_destroy(ctx.0, xyz); } return Err(ctx.err(rc)); }
    let dref = match reference { Some(r) => Some(DeviceImage::new(ctx, bytes, Some(r))?), None => None };
    let dcomb = if want_image { Some(DeviceImage::new(ctx, bytes, None)?) } else { None };
    let mut out = sys::acm_image_quality::default();
    let rc = unsafe {
        sys::acm_image_quality_metrics(ctx.0, input_model, output_model, xyz, width, height,
                                       dref.as_ref().map_or(ptr::null(), |d| d.ptr as *const u8),
                                       dcomb.as_ref().map_or(ptr::null_mut(), |d| d.ptr as *mut u8), &mut out)
    };
    unsafe { sys::acm_points_destroy(ctx.0, xyz); }
    if rc != sys::ACM_OK { return Err(ctx.err(rc)); }   // ACM_ERR_ZERO_PROJECTION_POINTS -> UtilError::ZeroProjectionPoints upstream
    let img = match dcomb { Some(d) => Some(d.download()?), None => None };
    Ok((ImageQualityMetrics { psnr: out.psnr, ssim: out.ssim }, img))
}
