"""Image-quality diagnostics of the converter (reference src/util/image_quality.rs) on the GPU:
calculate_psnr (:45-89), calculate_ssim (:108-210), the projection drawings (:338-505, :553-616) and
compute_image_quality_metrics (:254-324).  Images are (H, W, 3) uint8 arrays in image::RgbImage memory
order; they are staged in HBM for the call.  Writing PNG files stays with the caller (out of scope)."""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass

import numpy as np

from . import _native as N
from .camera import CameraModel
from .errors import UtilError
from .runtime import Context, Staging, default_context

_lib = N.lib

GREEN, MAGENTA, WHITE = (0, 255, 0), (255, 0, 255), (255, 255, 255)


@dataclass
class ImageQualityMetrics:  # image_quality.rs:20-26
    psnr: float
    ssim: float


class _DeviceImage:
    """RGB8 image in HBM, owned by the call's `Staging`."""

    def __init__(self, s: Staging, host: np.ndarray | None = None, shape=None):
        self.ctx = ctx = s.ctx
        if host is not None:
            host = np.ascontiguousarray(host, dtype=np.uint8)
            if host.ndim != 3 or host.shape[2] != 3:
                raise UtilError("Invalid parameters: expected an (H, W, 3) uint8 image")
            shape = host.shape
        self.shape = tuple(shape)
        self.nbytes = int(np.prod(self.shape))
        self.ptr = s.alloc(max(self.nbytes, 4))
        if host is not None and self.nbytes:
            ctx.h2d(self.ptr, host)
        elif self.nbytes:
            ctx.check(_lib.acm_memset_d(ctx.handle, C.c_void_p(self.ptr), 0, self.nbytes))

    def numpy(self) -> np.ndarray:
        out = np.empty(self.shape, dtype=np.uint8)
        if self.nbytes:
            self.ctx.d2h(out, self.ptr)
            self.ctx.sync()
        return out


def _compare(fn, img1, img2, ctx: Context | None) -> float:
    """`fn` (acm_image_psnr / acm_image_ssim) of two same-shaped images staged on the device."""
    a, b = np.asarray(img1), np.asarray(img2)
    if a.shape != b.shape:  # image_quality.rs:46-50, :109-113
        raise UtilError("Invalid parameters: Images must have the same dimensions")
    ctx = ctx or default_context()
    out = C.c_double()
    with ctx.staging() as s:
        d1, d2 = _DeviceImage(s, a), _DeviceImage(s, b)
        ctx.check(fn(ctx.handle, C.c_void_p(d1.ptr), C.c_void_p(d2.ptr), d1.shape[1], d1.shape[0], C.byref(out)))
    return float(out.value)


def calculate_psnr(img1: np.ndarray, img2: np.ndarray, ctx: Context | None = None) -> float:
    """PSNR in dB over the pixels that are not black in both images; inf for a perfect match."""
    return _compare(_lib.acm_image_psnr, img1, img2, ctx)


def calculate_ssim(img1: np.ndarray, img2: np.ndarray, ctx: Context | None = None) -> float:
    """Mean 3x3-window SSIM of the truncated-luma grey images (interior windows only)."""
    return _compare(_lib.acm_image_ssim, img1, img2, ctx)


def _draw(ctx: Context | None, layers, host: np.ndarray | None = None, shape=None) -> np.ndarray:
    """Draws each (projections, color) of `layers` in turn on a device copy of `host` (or on black at `shape`) and returns
    the image."""
    ctx = ctx or default_context()
    with ctx.staging() as s:
        d = _DeviceImage(s, host, shape)
        for projections, color in layers:
            pts = s.points(projections, 2)
            ctx.check(_lib.acm_draw_points_rgb8(ctx.handle, pts.handle, None, color[0], color[1], color[2], C.c_void_p(d.ptr),
                                                d.shape[1], d.shape[0]))
        return d.numpy()


def create_projection_image(projections, color, width: int, height: int, ctx: Context | None = None) -> np.ndarray:
    """image_quality.rs:338-373 with one colour for every point: radius-2 discs on black."""
    return _draw(ctx, [(projections, color)], shape=(height, width, 3))


def create_combined_projection_image_on_reference(input_projections, output_projections, reference_image: np.ndarray,
                                                  ctx: Context | None = None) -> np.ndarray:
    """image_quality.rs:389-437: green input discs, then magenta output discs, on a copy of the reference."""
    return _draw(ctx, [(input_projections, GREEN), (output_projections, MAGENTA)], reference_image)


def create_combined_projection_image(input_projections, output_projections, width: int, height: int,
                                     ctx: Context | None = None) -> np.ndarray:
    """image_quality.rs:453-505: the same on a black background."""
    return create_combined_projection_image_on_reference(input_projections, output_projections,
                                                         np.zeros((height, width, 3), np.uint8), ctx)


def model_projection_visualization(points_2d, reference_image: np.ndarray | None, camera_resolution,
                                   ctx: Context | None = None) -> np.ndarray:
    """image_quality.rs:553-616 without the file: green discs on the reference image, or on black at
    `camera_resolution = (width, height)`.  Returns the image the reference would save."""
    if reference_image is not None:
        return _draw(ctx, [(points_2d, GREEN)], reference_image)
    return create_projection_image(points_2d, GREEN, camera_resolution[0], camera_resolution[1], ctx)


def compute_image_quality_metrics(input_model: CameraModel, output_model: CameraModel, optimization_points_3d,
                                  reference_image: np.ndarray | None = None, return_image: bool = False):
    """image_quality.rs:254-324.  Image size = the reference image's, else the input model's resolution.
    Raises ZeroProjectionPoints (through the status code) when no point projects through both models
    into the image.  `return_image=True` also returns the combined display image the reference saves
    (green input / magenta output projections)."""
    ctx = input_model.ctx
    if reference_image is not None:
        ref = np.ascontiguousarray(reference_image, dtype=np.uint8)
        height, width = ref.shape[:2]
    else:
        res = input_model.get_resolution()
        ref, width, height = None, res.width, res.height
    with ctx.staging() as s:
        X = s.points(optimization_points_3d, 3)
        dref = _DeviceImage(s, ref) if ref is not None else None
        dcomb = _DeviceImage(s, shape=(height, width, 3)) if return_image else None
        cin, cout = input_model.camera_block(), output_model.camera_block()
        out = N.ImageQuality()
        ctx.check(_lib.acm_image_quality_metrics(ctx.handle, C.byref(cin), C.byref(cout), X.handle, width, height,
                                                 C.c_void_p(dref.ptr) if dref else None, C.c_void_p(dcomb.ptr) if dcomb else None,
                                                 C.byref(out)))
        m = ImageQualityMetrics(float(out.psnr), float(out.ssim))
        return (m, dcomb.numpy()) if return_image else m
