"""util hot loops of the reference: undistort_image (src/util/undistort.rs:14-105), sample_points
(src/util/point_sampling.rs:46-120), compute_reprojection_error (src/util/error_metrics.rs:62-121); and remap plans
(camera-to-camera image remap, composed of the reference's unproject, project and interpolate_pixel), rotated plans and
stereo rectification."""
from __future__ import annotations

import ctypes as C
import enum
from dataclasses import dataclass

import numpy as np

from . import _native as N
from .camera import CameraModel, Intrinsics, PinholeModel
from .errors import UtilError, raise_call_status
from .runtime import Points

_lib = N.lib


class InterpolationMethod(enum.IntEnum):  # undistort.rs:8-12
    Nearest = 0
    Bilinear = 1


@dataclass
class ProjectionError:  # error_metrics.rs:17-31
    rmse: float
    min: float
    max: float
    mean: float
    stddev: float
    median: float
    count: int = 0


def _target_array(target: Intrinsics | None):
    if target is None:
        return None
    return (C.c_double * 4)(target.fx, target.fy, target.cx, target.cy)


def _matrix3(a, what: str) -> np.ndarray:
    m = np.array(a, dtype=np.float64)
    if m.shape != (3, 3):
        raise UtilError(f"Invalid parameters: {what} must be a 3x3 matrix, got shape {m.shape}")
    return m


def _rotation_array(rotation):
    """Row-major double[9] of a 3x3 rotation (libacm checks that it is one)."""
    return (C.c_double * 9)(*_matrix3(rotation, "rotation").ravel())


def _check_frames(frames: np.ndarray, camera_model: CameraModel) -> np.ndarray:
    """(F, H, W, 3) uint8 frames at the camera's resolution, as undistort.rs:23-28 requires."""
    frames = np.ascontiguousarray(frames, dtype=np.uint8)
    if frames.ndim != 4 or frames.shape[3] != 3:
        raise UtilError("Invalid parameters: expected (F, H, W, 3) uint8 frames")
    res = camera_model.get_resolution()
    _, H, W, _ = frames.shape
    if W != res.width or H != res.height:
        raise UtilError(f"Invalid parameters: Image {W}x{H} doesn't match model {res.width}x{res.height}")
    return frames


def _download_map(ctx, res, call) -> np.ndarray:
    """(H, W, 2) source-coordinate map at resolution `res`: `call(device_ptr)` writes it on the device and returns libacm's
    status; the device buffer is freed whatever happens."""
    d = ctx.device_alloc(max(res.width * res.height, 1) * 16)
    try:
        ctx.check(call(C.c_void_p(d)))
        out = np.empty((res.height, res.width, 2))
        ctx.d2h(out, d)
        ctx.sync()
    finally:
        ctx.device_free(d)
    return out


def undistort_images(frames: np.ndarray, camera_model: CameraModel, target_intrinsics: Intrinsics | None = None,
                     interpolation: InterpolationMethod = InterpolationMethod.Bilinear) -> np.ndarray:
    """Batch form: frames (F, H, W, 3) uint8 -> same shape."""
    frames = _check_frames(frames, camera_model)
    ctx = camera_model.ctx
    cam = camera_model.camera_block()
    out = np.empty_like(frames)
    ctx.check(_lib.acm_undistort_rgb8_host(ctx.handle, C.byref(cam), _target_array(target_intrinsics), frames.ctypes.data_as(C.c_void_p),
                                           out.ctypes.data_as(C.c_void_p), frames.shape[0], int(interpolation)))
    return out


def undistort_image(input_image: np.ndarray, camera_model: CameraModel, target_intrinsics: Intrinsics | None = None,
                    interpolation: InterpolationMethod = InterpolationMethod.Bilinear) -> np.ndarray:
    """`undistort_image(&RgbImage, &dyn CameraModel, Option<Intrinsics>, InterpolationMethod)`;
    image is (H, W, 3) uint8 (image::RgbImage memory order)."""
    img = np.ascontiguousarray(input_image, dtype=np.uint8)
    return undistort_images(img[None], camera_model, target_intrinsics, interpolation)[0]


def undistort_map(camera_model: CameraModel, target_intrinsics: Intrinsics | None = None) -> np.ndarray:
    """(H, W, 2) source coordinates of every output pixel (NaN where the projection fails)."""
    ctx = camera_model.ctx
    cam = camera_model.camera_block()
    target = _target_array(target_intrinsics)
    return _download_map(ctx, camera_model.get_resolution(), lambda d: _lib.acm_undistort_map(ctx.handle, C.byref(cam), target, d))


class RemapPlan:
    """Remap of RGB8 frames from `input_model`'s camera to `output_model`'s, built once on the device and applied to
    any number of frame batches.  Output pixel (u, v) of the output camera's grid samples the input frame at
    input_model.project(output_model.unproject((u, v))) with `interpolation` (undistort.rs:51-105); black where either
    step fails.  With `output_model=None` the plan is `undistort_image(., input_model, target_intrinsics, interpolation)`
    and its output is byte-identical to `undistort_images`.  The plan keeps 32 bytes per output pixel on the device
    until `close()`."""

    def __init__(self, input_model: CameraModel, output_model: CameraModel | None = None, target_intrinsics: Intrinsics | None = None,
                 interpolation: InterpolationMethod = InterpolationMethod.Bilinear, *, rotation=None):
        """`rotation`: a 3x3 rotation R with x_out = R x_in (OpenCV's R1 / R2), applied between the output camera's
        unproject and the input camera's project as ray_in = R^T ray_out.  It needs an output camera."""
        self.ctx = input_model.ctx
        self.input_model = input_model
        self.output_resolution = (output_model or input_model).get_resolution()
        cin = input_model.camera_block()
        cout = output_model.camera_block() if output_model is not None else None
        h = C.c_void_p()
        if rotation is not None:
            if output_model is None or target_intrinsics is not None:
                raise UtilError("Invalid parameters: a rotated remap plan needs an output camera and no target intrinsics")
            self.ctx.check(_lib.acm_remap_plan_create_rotated(self.ctx.handle, C.byref(cin), C.byref(cout), _rotation_array(rotation),
                                                              int(interpolation), C.byref(h)))
        else:
            self.ctx.check(_lib.acm_remap_plan_create(self.ctx.handle, C.byref(cin), C.byref(cout) if cout is not None else None,
                                                      _target_array(target_intrinsics), int(interpolation), C.byref(h)))
        self._h = h

    @property
    def handle(self):
        if not self._h:
            raise UtilError("remap plan is closed")
        return self._h

    def apply(self, frames: np.ndarray) -> np.ndarray:
        """Host frames (F, Hi, Wi, 3) uint8 at the input camera's resolution -> (F, Ho, Wo, 3)."""
        frames = _check_frames(frames, self.input_model)
        r = self.output_resolution
        out = np.empty((frames.shape[0], r.height, r.width, 3), np.uint8)
        self.ctx.check(_lib.acm_remap_rgb8_host(self.ctx.handle, self.handle, frames.ctypes.data_as(C.c_void_p),
                                                out.ctypes.data_as(C.c_void_p), frames.shape[0]))
        return out

    def apply_device(self, in_ptr: int, out_ptr: int, n_frames: int) -> None:
        """Frames resident on the plan's device: n_frames * Wi * Hi * 3 bytes at in_ptr -> n_frames * Wo * Ho * 3 at
        out_ptr, enqueued on the context's stream."""
        self.ctx.check(_lib.acm_remap_rgb8(self.ctx.handle, self.handle, C.c_void_p(in_ptr), C.c_void_p(out_ptr), n_frames))

    def close(self) -> None:
        if self._h:
            h, self._h = self._h, None
            if self.ctx.handle:
                self.ctx.check(_lib.acm_remap_plan_destroy(self.ctx.handle, h))

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def remap_images(frames: np.ndarray, input_model: CameraModel, output_model: CameraModel,
                 interpolation: InterpolationMethod = InterpolationMethod.Bilinear) -> np.ndarray:
    """Frames (F, Hi, Wi, 3) uint8 of `input_model`'s camera -> (F, Ho, Wo, 3) as `output_model`'s camera sees them."""
    frames = _check_frames(frames, input_model)
    with RemapPlan(input_model, output_model, None, interpolation) as plan:
        return plan.apply(frames)


def remap_image(input_image: np.ndarray, input_model: CameraModel, output_model: CameraModel,
                interpolation: InterpolationMethod = InterpolationMethod.Bilinear) -> np.ndarray:
    """One (Hi, Wi, 3) uint8 image -> (Ho, Wo, 3)."""
    img = np.ascontiguousarray(input_image, dtype=np.uint8)
    return remap_images(img[None], input_model, output_model, interpolation)[0]


def remap_map(input_model: CameraModel, output_model: CameraModel, rotation=None) -> np.ndarray:
    """(Ho, Wo, 2) source coordinates on the input frame of every output pixel (NaN where a step fails); `rotation` as in
    `RemapPlan`."""
    ctx = input_model.ctx
    cin, cout = input_model.camera_block(), output_model.camera_block()
    if rotation is not None:
        R = _rotation_array(rotation)
        call = lambda d: _lib.acm_remap_map_rotated(ctx.handle, C.byref(cin), C.byref(cout), R, d)
    else:
        call = lambda d: _lib.acm_remap_map(ctx.handle, C.byref(cin), C.byref(cout), d)
    return _download_map(ctx, output_model.get_resolution(), call)


def stereo_rectify(R, t):
    """Bouguet rectification of a calibrated pair (the rotation part of OpenCV's `stereoRectify`), x_cam2 = R x_cam1 + t.
    Returns (R1, R2, baseline, vertical): x_rect1 = R1 x_cam1, x_rect2 = R2 x_cam2; `baseline` is the signed component
    of R2 t along the rectified baseline axis, which is x, or y when `vertical` (the pair is stacked vertically).  Host
    only; no device needed."""
    Rm = _rotation_array(R)
    tv = np.array(t, dtype=np.float64).ravel()
    if tv.shape != (3,):
        raise UtilError(f"Invalid parameters: translation must have 3 entries, got {tv.size}")
    R1, R2 = (C.c_double * 9)(), (C.c_double * 9)()
    baseline, vertical = C.c_double(), C.c_int32()
    rc = _lib.acm_stereo_rectify(Rm, (C.c_double * 3)(*tv), R1, R2, C.byref(baseline), C.byref(vertical))
    if rc != N.OK:
        raise_call_status(rc, _lib.acm_last_error(None).decode())
    return np.array(R1[:]).reshape(3, 3), np.array(R2[:]).reshape(3, 3), baseline.value, bool(vertical.value)


class StereoRectifier:
    """Rectifies frames of a calibrated pair (x_cam2 = R x_cam1 + t) onto one caller-chosen Pinhole camera shared by both
    views: two rotated remap plans, `left` through R1 and `right` through R2 of `stereo_rectify(R, t)`.  Rectified rows
    correspond (columns when `vertical`); P1 = K [I | 0] and P2 = K [I | baseline e] with e the x (or y) axis.  Any
    camera models work on either side.  The plans stay on the device until `close()`."""

    def __init__(self, left: CameraModel, right: CameraModel, R, t, rectified_pinhole: CameraModel,
                 interpolation: InterpolationMethod = InterpolationMethod.Bilinear):
        if not isinstance(rectified_pinhole, PinholeModel):
            raise UtilError("Invalid parameters: the rectified camera must be a PinholeModel")
        self.R1, self.R2, self.baseline, self.vertical = stereo_rectify(R, t)
        i = rectified_pinhole.get_intrinsics()
        K = np.array([[i.fx, 0.0, i.cx], [0.0, i.fy, i.cy], [0.0, 0.0, 1.0]])
        e = np.zeros((3, 1))
        e[1 if self.vertical else 0, 0] = self.baseline
        self.P1 = K @ np.hstack([np.eye(3), np.zeros((3, 1))])
        self.P2 = K @ np.hstack([np.eye(3), e])
        self.left_plan = RemapPlan(left, rectified_pinhole, None, interpolation, rotation=self.R1)
        try:
            self.right_plan = RemapPlan(right, rectified_pinhole, None, interpolation, rotation=self.R2)
        except Exception:
            self.left_plan.close()
            raise

    def apply(self, left_frames: np.ndarray, right_frames: np.ndarray) -> tuple[np.ndarray, np.ndarray]:
        """(F, H, W, 3) uint8 frames of each camera -> both rectified batches (F, Ho, Wo, 3)."""
        return self.left_plan.apply(left_frames), self.right_plan.apply(right_frames)

    def close(self) -> None:
        self.left_plan.close()
        self.right_plan.close()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()


def sample_points(camera_model: CameraModel, n: int, device: bool = False, shard: tuple[int, int] | None = None):
    """`sample_points(Some(&model), n) -> (Matrix2xX, Matrix3xX)`: (points_2d, points_3d).

    `shard=(rank, world)` returns that rank's contiguous slice of the grid (one slice per GPU; the
    slices concatenated in rank order are the unsharded result)."""
    if camera_model is None:
        raise UtilError("Camera model does not exist")  # the reference panics on None (point_sampling.rs:53)
    ctx = camera_model.ctx
    cam = camera_model.camera_block()
    uv_h, xyz_h, kept = C.c_void_p(), C.c_void_p(), C.c_size_t()
    rank, world = shard if shard is not None else (0, 1)
    ctx.check(_lib.acm_sample_points_shard(ctx.handle, C.byref(cam), n, rank, world, C.byref(uv_h), C.byref(xyz_h), C.byref(kept)))
    uv = Points(ctx, 2, kept.value, _handle=uv_h)
    xyz = Points(ctx, 3, kept.value, _handle=xyz_h)
    if device:
        return uv, xyz
    a, b = uv.numpy(), xyz.numpy()
    uv.free(); xyz.free()
    return a, b


def compute_reprojection_error(camera_model: CameraModel, points3d, points2d) -> ProjectionError:
    if camera_model is None:
        raise UtilError("Camera model does not exist")
    ctx = camera_model.ctx
    own = []
    def dev(a, dim):
        if isinstance(a, Points):
            return a
        p = Points.from_numpy(ctx, np.ascontiguousarray(a, dtype=np.float64).reshape(-1, dim))
        own.append(p)
        return p
    X, UV = dev(points3d, 3), dev(points2d, 2)
    cam = camera_model.camera_block()
    out = N.ProjectionError()
    rc = _lib.acm_reprojection_error(ctx.handle, C.byref(cam), X.handle, UV.handle, C.byref(out))
    for p in own:
        p.free()
    ctx.check(rc)
    return ProjectionError(out.rmse, out.min, out.max, out.mean, out.stddev, out.median, int(out.count))
