"""util hot loops of the reference: undistort_image (src/util/undistort.rs:14-105), sample_points
(src/util/point_sampling.rs:46-120), compute_reprojection_error (src/util/error_metrics.rs:62-121); and remap plans
(camera-to-camera image remap, composed of the reference's unproject, project and interpolate_pixel), rotated plans,
stereo rectification, triangulation of matched pixels of a calibrated pair, and depth images (a point cloud rendered into a
camera's range image, and a range image back-projected into points)."""
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
    status."""
    with ctx.staging() as s:
        d = s.alloc(res.width * res.height * 16)
        ctx.check(call(C.c_void_p(d)))
        out = np.empty((res.height, res.width, 2))
        ctx.d2h(out, d)
        ctx.sync()
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
    with ctx.staging() as s:
        uv, xyz = s.own(Points(ctx, 2, kept.value, _handle=uv_h)), s.own(Points(ctx, 3, kept.value, _handle=xyz_h))
        return s.keep(uv, xyz) if device else (uv.numpy(), xyz.numpy())


def compute_reprojection_error(camera_model: CameraModel, points3d, points2d) -> ProjectionError:
    if camera_model is None:
        raise UtilError("Camera model does not exist")
    ctx = camera_model.ctx
    cam = camera_model.camera_block()
    out = N.ProjectionError()
    with ctx.staging() as s:
        X, UV = s.points(points3d, 3), s.points(points2d, 2)
        ctx.check(_lib.acm_reprojection_error(ctx.handle, C.byref(cam), X.handle, UV.handle, C.byref(out)))
    return ProjectionError(out.rmse, out.min, out.max, out.mean, out.stddev, out.median, int(out.count))


class TriangulationStatus(enum.IntEnum):
    """Per-pair status of `triangulate_points` (include/acm.h ACM_TRI_*), in the order the steps decide it."""
    Ok = N.TRI_OK
    UnprojectFirst = N.TRI_UNPROJECT_FIRST      # the first camera's unproject failed (any CameraModelError)
    UnprojectSecond = N.TRI_UNPROJECT_SECOND    # the second camera's unproject failed
    Parallel = N.TRI_PARALLEL                   # 1 - (d1 . d2')^2 <= 1e-12: the rays are parallel
    Behind = N.TRI_BEHIND                       # the closest approach lies behind either camera
    Project = N.TRI_PROJECT                     # the point does not project into both cameras


def _translation_array(t):
    tv = np.array(t, dtype=np.float64).ravel()
    if tv.shape != (3,):
        raise UtilError(f"Invalid parameters: translation must have 3 entries, got {tv.size}")
    return (C.c_double * 3)(*tv)


def triangulate_points(first: CameraModel, second: CameraModel, R, t, points1, points2, max_iterations: int = 10):
    """3-D points of matched pixels of a calibrated pair, x_cam2 = R x_cam1 + t (the convention of `stereo_rectify`).

    points1 / points2: (N, 2) pixels of `first` / `second` (numpy arrays or device `Points`).  Per pair: both pixels are
    unprojected (IEEE form, with each model's pixel-bounds test), the midpoint of the rays' closest approach is taken in
    the first camera's frame, and with `max_iterations > 0` up to that many damped Gauss-Newton (Levenberg-Marquardt)
    trials minimise the squared pixel errors of the point's projections into both cameras.  Any two camera models work,
    including fields of view beyond 90 degrees.

    Returns (points_3d (N, 3) in the first camera's frame, errors (N, 2) = |first.project(X) - uv1| and
    |second.project(R X + t) - uv2| in pixels, status (N,) uint8 of `TriangulationStatus`); points and errors are NaN
    where the status is not Ok.  Always numpy, whatever the input.

    Rectified pixels of a `StereoRectifier` triangulate with the rectified pinhole on both sides, R = I and
    t = baseline * e (e = x axis, or y when `vertical`); the points are then in the first RECTIFIED frame, and
    `rig.R1.T @ X` takes them back to the first camera's."""
    if first is None or second is None:
        raise UtilError("Camera model does not exist")
    if max_iterations < 0:
        raise UtilError("Invalid parameters: max_iterations must be >= 0")
    ctx = first.ctx
    Rm, tv = _rotation_array(R), _translation_array(t)
    ca, cb = first.camera_block(), second.camera_block()
    if isinstance(points1, Points) or isinstance(points2, Points):
        with ctx.staging() as s:
            a, b = s.points(points1, 2), s.points(points2, 2)
            n = len(a)
            xyz = s.own(Points(ctx, 3, n))
            d = s.alloc(n * 17)  # two rows of errors, then the status bytes
            ctx.check(_lib.acm_triangulate(ctx.handle, C.byref(ca), C.byref(cb), Rm, tv, a.handle, b.handle, int(max_iterations),
                                           xyz.handle, C.c_void_p(d), C.c_void_p(d + 16 * n)))
            err, st = np.empty((2, n)), np.empty(n, np.uint8)
            if n:
                ctx.d2h(err, d); ctx.d2h(st, d + 16 * n)
            ctx.sync()
            pts = xyz.numpy()
        return pts, np.ascontiguousarray(err.T), st
    uv1 = np.ascontiguousarray(points1, dtype=np.float64).reshape(-1, 2)
    uv2 = np.ascontiguousarray(points2, dtype=np.float64).reshape(-1, 2)
    if len(uv1) != len(uv2):
        raise UtilError(f"Invalid parameters: {len(uv1)} pixels of the first camera but {len(uv2)} of the second")
    n = len(uv1)
    xyz, err, st = np.empty((n, 3)), np.empty((n, 2)), np.empty(n, np.uint8)
    ctx.check(_lib.acm_triangulate_host(ctx.handle, C.byref(ca), C.byref(cb), Rm, tv, uv1.ctypes.data_as(C.c_void_p),
                                        uv2.ctypes.data_as(C.c_void_p), n, int(max_iterations), xyz.ctypes.data_as(C.c_void_p),
                                        err.ctypes.data_as(C.c_void_p), st.ctypes.data_as(C.c_void_p)))
    return xyz, err, st


class DepthStatus(enum.IntEnum):
    """Per-pixel status of `depth_to_points` (include/acm.h ACM_DEPTH_*)."""
    Ok = N.DEPTH_OK
    Empty = N.DEPTH_EMPTY            # the range is not finite or <= 0 (an empty pixel of `render_depth`)
    Unproject = N.DEPTH_UNPROJECT    # the model's unproject of the pixel centre failed


def _pose_arrays(R, t):
    """R = None: identity; t = None: zero."""
    return _rotation_array(np.eye(3) if R is None else R), _translation_array(np.zeros(3) if t is None else t)


def render_depth(model: CameraModel, points, R=None, t=None):
    """Z-buffered range image of world points seen by `model`'s camera, x_cam = R x + t (R = None: identity, t = None: zero).

    points: (N, 3) world points (a numpy array or device `Points`), N < 2^32 - 1.  A point is drawn into pixel
    (round(u), round(v)) (half away from zero, the nearest rule of `undistort_image`) when the model projects x_cam (geometric
    validity, any field of view, including rays beyond 90 degrees), the pixel lies inside the image and its range
    |x_cam| is finite and > 0.  Per pixel the nearest point in float32 range wins and ties go to the lower index, so the
    result does not depend on scheduling.  Depth is the RANGE along the ray, not z: z = range * ray_z.

    Returns (range (H, W) float32, NaN where empty; index (H, W) uint32 of the winning point, 0xFFFFFFFF where empty),
    H x W = the model's resolution.  Always numpy."""
    if model is None:
        raise UtilError("Camera model does not exist")
    ctx = model.ctx
    Rm, tv = _pose_arrays(R, t)
    cam = model.camera_block()
    res = model.get_resolution()
    rng, idx = np.empty((res.height, res.width), np.float32), np.empty((res.height, res.width), np.uint32)
    if isinstance(points, Points):
        npix = res.width * res.height
        with ctx.staging() as s:
            d = s.alloc(npix * 8)  # range row, then index row
            ctx.check(_lib.acm_render_depth(ctx.handle, C.byref(cam), Rm, tv, points.handle, C.c_void_p(d), C.c_void_p(d + 4 * npix)))
            ctx.d2h(rng, d); ctx.d2h(idx, d + 4 * npix)
            ctx.sync()
        return rng, idx
    xyz = np.ascontiguousarray(points, dtype=np.float64).reshape(-1, 3)
    ctx.check(_lib.acm_render_depth_host(ctx.handle, C.byref(cam), Rm, tv, xyz.ctypes.data_as(C.c_void_p), len(xyz),
                                         rng.ctypes.data_as(C.c_void_p), idx.ctypes.data_as(C.c_void_p)))
    return rng, idx


def depth_to_points(model: CameraModel, range_image, R=None, t=None):
    """Back-projection of a (H, W) range image of `model`'s camera (H x W = its resolution) into world points, x_cam = R x + t
    as in `render_depth`: pixel (c, r) with a finite range d > 0 gives x = R^T (unproject((c, r)) * d - t), the ray of the
    integer pixel centre (IEEE unproject, with the model's pixel-bounds test).

    Returns (points (H, W, 3) float64, NaN where the status is not Ok; status (H, W) uint8 of `DepthStatus`)."""
    if model is None:
        raise UtilError("Camera model does not exist")
    ctx = model.ctx
    Rm, tv = _pose_arrays(R, t)
    cam = model.camera_block()
    res = model.get_resolution()
    r = np.ascontiguousarray(range_image, dtype=np.float32)
    if r.shape != (res.height, res.width):
        raise UtilError(f"Invalid parameters: range image {r.shape} doesn't match model {res.height}x{res.width} (H, W)")
    npix = res.width * res.height
    with ctx.staging() as s:
        xyz = s.own(Points(ctx, 3, npix))
        d = s.alloc(npix * 5)  # range, then the status bytes
        ctx.h2d(d, r)
        ctx.check(_lib.acm_depth_to_points(ctx.handle, C.byref(cam), Rm, tv, C.c_void_p(d), xyz.handle, C.c_void_p(d + 4 * npix)))
        st = np.empty((res.height, res.width), np.uint8)
        ctx.d2h(st, d + 4 * npix)
        ctx.sync()
        pts = xyz.numpy().reshape(res.height, res.width, 3)
    return pts, st
