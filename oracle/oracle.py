"""ctypes loader for the CPU oracle (oracle/build/liboracle.so).

TEST INFRASTRUCTURE ONLY: imported by tests/, __graft_entry__.smoke() and bench.py's
cpu_baseline / --impl reference legs.  The product package never imports this module.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "build", "liboracle.so")

PINHOLE, RADTAN, KB, UCM, EUCM, DS, FOV = range(7)
MODEL_NAMES = ["pinhole", "rad_tan", "kannala_brandt", "ucm", "eucm", "double_sphere", "fov"]
N_PARAMS = [4, 9, 8, 5, 6, 6, 5]
OK, POINT_OUTSIDE_IMAGE, POINT_AT_CENTER, PROJECTION_OUTSIDE_IMAGE, NUMERICAL = range(5)
RES_PIXEL, RES_ALGEBRAIC = 0, 1


class Model(C.Structure):
    _fields_ = [("model", C.c_int32), ("width", C.c_uint32), ("height", C.c_uint32),
                ("n_params", C.c_int32), ("p", C.c_double * 9)]

    def params(self):
        return np.array(self.p[: self.n_params], dtype=np.float64)


class LMConfig(C.Structure):
    _fields_ = [("max_iterations", C.c_int32), ("cost_tolerance", C.c_double),
                ("parameter_tolerance", C.c_double), ("gradient_tolerance", C.c_double),
                ("lambda0", C.c_double), ("invalid_penalty", C.c_double)]


class LMResult(C.Structure):
    _fields_ = [("status", C.c_int32), ("iterations", C.c_int32), ("passes", C.c_int32),
                ("initial_cost", C.c_double), ("final_cost", C.c_double), ("n_valid", C.c_uint64)]


class ProjError(C.Structure):
    _fields_ = [("rmse", C.c_double), ("min", C.c_double), ("max", C.c_double), ("mean", C.c_double),
                ("stddev", C.c_double), ("median", C.c_double), ("count", C.c_uint64)]


def build(force: bool = False) -> str:
    if force or not os.path.exists(_LIB_PATH) or any(
        os.path.getmtime(os.path.join(_HERE, f)) > os.path.getmtime(_LIB_PATH)
        for f in os.listdir(_HERE) if f.endswith((".c", ".h"))
    ):
        subprocess.run(["make", "-C", _HERE, "-s"], check=True)
    return _LIB_PATH


_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(_LIB_PATH):
            build()
        L = C.CDLL(_LIB_PATH)
        dp, u8p, mp = C.POINTER(C.c_double), C.POINTER(C.c_uint8), C.POINTER(Model)
        L.orc_project.argtypes = [mp, dp, dp]; L.orc_project.restype = C.c_int
        L.orc_unproject.argtypes = [mp, dp, dp]; L.orc_unproject.restype = C.c_int
        L.orc_project_nobounds.argtypes = [mp, dp, dp]; L.orc_project_nobounds.restype = C.c_int
        L.orc_project_batch.argtypes = [mp, dp, C.c_size_t, dp, u8p, C.c_int]; L.orc_project_batch.restype = None
        L.orc_unproject_batch.argtypes = [mp, dp, C.c_size_t, dp, u8p, C.c_int]; L.orc_unproject_batch.restype = None
        L.orc_project_jacobian.argtypes = [mp, dp, dp, dp]; L.orc_project_jacobian.restype = C.c_int
        L.orc_project_point_jacobian.argtypes = [mp, dp, dp, dp]; L.orc_project_point_jacobian.restype = C.c_int
        L.orc_project_jacobian_batch.argtypes = [mp, dp, C.c_size_t, dp, dp, u8p, C.c_int]; L.orc_project_jacobian_batch.restype = None
        L.orc_project_point_jacobian_batch.argtypes = [mp, dp, C.c_size_t, dp, dp, u8p, C.c_int]
        L.orc_project_point_jacobian_batch.restype = None
        L.orc_residual_jacobian.argtypes = [mp, C.c_int, dp, dp, dp, dp]; L.orc_residual_jacobian.restype = C.c_int
        L.orc_linearize.argtypes = [mp, C.c_int, dp, dp, C.c_size_t, dp, dp, dp, C.POINTER(C.c_uint64), C.c_int]
        L.orc_linearize.restype = C.c_int
        L.orc_lm_default_config.argtypes = [C.POINTER(LMConfig)]; L.orc_lm_default_config.restype = None
        L.orc_lm_solve.argtypes = [mp, C.c_int, dp, dp, C.c_size_t, dp, dp, C.POINTER(LMConfig), dp, C.POINTER(LMResult), C.c_int]
        L.orc_lm_solve.restype = C.c_int
        L.orc_linear_estimation.argtypes = [mp, dp, dp, C.c_size_t]; L.orc_linear_estimation.restype = C.c_int
        L.orc_sample_grid_size.argtypes = [mp, C.c_size_t, C.POINTER(C.c_int), C.POINTER(C.c_int)]
        L.orc_sample_grid_size.restype = C.c_size_t
        L.orc_sample_points.argtypes = [mp, C.c_size_t, dp, dp]; L.orc_sample_points.restype = C.c_size_t
        L.orc_reprojection_error.argtypes = [mp, dp, dp, C.c_size_t, C.POINTER(ProjError)]
        L.orc_reprojection_error.restype = C.c_int
        L.orc_undistort_rgb8.argtypes = [mp, dp, u8p, u8p, C.c_int, C.c_int]; L.orc_undistort_rgb8.restype = C.c_int
        L.orc_undistort_map.argtypes = [mp, dp, dp]; L.orc_undistort_map.restype = None
        L.orc_image_psnr.argtypes = [u8p, u8p, C.c_uint32, C.c_uint32]; L.orc_image_psnr.restype = C.c_double
        L.orc_image_ssim.argtypes = [u8p, u8p, C.c_uint32, C.c_uint32]; L.orc_image_ssim.restype = C.c_double
        L.orc_rgb_to_grayscale.argtypes = [u8p, C.c_uint32, C.c_uint32, u8p]; L.orc_rgb_to_grayscale.restype = None
        L.orc_draw_points_rgb8.argtypes = [dp, C.c_size_t, C.c_uint8, C.c_uint8, C.c_uint8, u8p, C.c_uint32, C.c_uint32]
        L.orc_draw_points_rgb8.restype = None
        L.orc_image_quality_metrics.argtypes = [mp, mp, dp, C.c_size_t, C.c_uint32, C.c_uint32, u8p, u8p, dp, dp]
        L.orc_image_quality_metrics.restype = C.c_size_t
        L.orc_validate_conversion.argtypes = [mp, mp, dp, dp, dp]; L.orc_validate_conversion.restype = C.c_int
        L.orc_splitmix64.argtypes = [C.c_uint64]; L.orc_splitmix64.restype = C.c_uint64
        L.orc_synth_points3.argtypes = [C.c_uint64, C.c_size_t, C.c_size_t, C.c_double, C.c_int, dp]
        L.orc_synth_points3.restype = None
        L.orc_synth_pixels.argtypes = [C.c_uint64, C.c_size_t, C.c_size_t, C.c_double, C.c_double, dp]
        L.orc_synth_pixels.restype = None
        L.orc_synth_bytes.argtypes = [C.c_uint64, C.c_size_t, C.c_size_t, u8p]; L.orc_synth_bytes.restype = None
        _lib = L
    return _lib


def _dp(a):
    return a.ctypes.data_as(C.POINTER(C.c_double))


def _u8p(a):
    return a.ctypes.data_as(C.POINTER(C.c_uint8))


def make_model(model: int, params, width: int = 0, height: int = 0) -> Model:
    params = [float(x) for x in params]
    assert len(params) == N_PARAMS[model], (model, len(params))
    m = Model()
    m.model, m.width, m.height, m.n_params = model, width, height, len(params)
    for i, v in enumerate(params):
        m.p[i] = v
    return m


def project1(m: Model, X):
    X = np.ascontiguousarray(X, dtype=np.float64); uv = np.empty(2)
    st = lib().orc_project(C.byref(m), _dp(X), _dp(uv))
    return st, uv


def unproject1(m: Model, uv):
    uv = np.ascontiguousarray(uv, dtype=np.float64); ray = np.empty(3)
    st = lib().orc_unproject(C.byref(m), _dp(uv), _dp(ray))
    return st, ray


def project(m: Model, xyz: np.ndarray, nthreads: int = 1):
    """xyz: (N,3) float64 AoS -> (uv (N,2), status (N,) uint8)."""
    xyz = np.ascontiguousarray(xyz, dtype=np.float64); n = xyz.shape[0]
    uv = np.empty((n, 2)); st = np.empty(n, dtype=np.uint8)
    lib().orc_project_batch(C.byref(m), _dp(xyz), n, _dp(uv), _u8p(st), nthreads)
    return uv, st


def unproject(m: Model, uv: np.ndarray, nthreads: int = 1):
    uv = np.ascontiguousarray(uv, dtype=np.float64); n = uv.shape[0]
    xyz = np.empty((n, 3)); st = np.empty(n, dtype=np.uint8)
    lib().orc_unproject_batch(C.byref(m), _dp(uv), n, _dp(xyz), _u8p(st), nthreads)
    return xyz, st


def project_jacobian1(m: Model, X):
    X = np.ascontiguousarray(X, dtype=np.float64); uv = np.empty(2); J = np.zeros((2, m.n_params))
    st = lib().orc_project_jacobian(C.byref(m), _dp(X), _dp(uv), _dp(J))
    return st, uv, J


def project_point_jacobian1(m: Model, X):
    """status, uv, 2x3 Jacobian of (u, v) w.r.t. the 3-D point."""
    X = np.ascontiguousarray(X, dtype=np.float64); uv = np.empty(2); J = np.zeros((2, 3))
    st = lib().orc_project_point_jacobian(C.byref(m), _dp(X), _dp(uv), _dp(J))
    return st, uv, J


def project_jacobian(m: Model, xyz: np.ndarray, nthreads: int = 1):
    """Batch form of project_jacobian1: xyz (N,3) -> (uv (N,2), J (N,2,P), status (N,) uint8)."""
    xyz = np.ascontiguousarray(xyz, dtype=np.float64); n = xyz.shape[0]
    uv = np.empty((n, 2)); J = np.empty((n, 2, m.n_params)); st = np.empty(n, dtype=np.uint8)
    lib().orc_project_jacobian_batch(C.byref(m), _dp(xyz), n, _dp(uv), _dp(J), _u8p(st), nthreads)
    return uv, J, st


def project_point_jacobian(m: Model, xyz: np.ndarray, nthreads: int = 1):
    """Batch form of project_point_jacobian1: xyz (N,3) -> (uv (N,2), J (N,2,3), status (N,) uint8)."""
    xyz = np.ascontiguousarray(xyz, dtype=np.float64); n = xyz.shape[0]
    uv = np.empty((n, 2)); J = np.empty((n, 2, 3)); st = np.empty(n, dtype=np.uint8)
    lib().orc_project_point_jacobian_batch(C.byref(m), _dp(xyz), n, _dp(uv), _dp(J), _u8p(st), nthreads)
    return uv, J, st


def residual_jacobian1(m: Model, kind: int, X, uv_obs):
    X = np.ascontiguousarray(X, dtype=np.float64); uv_obs = np.ascontiguousarray(uv_obs, dtype=np.float64)
    r = np.empty(2); J = np.zeros((2, m.n_params))
    st = lib().orc_residual_jacobian(C.byref(m), kind, _dp(X), _dp(uv_obs), _dp(r), _dp(J))
    return st, r, J


def linearize(m: Model, kind: int, xyz, uv, nthreads: int = 1):
    xyz = np.ascontiguousarray(xyz, dtype=np.float64); uv = np.ascontiguousarray(uv, dtype=np.float64)
    P = m.n_params; H = np.empty((P, P)); g = np.empty(P); cost = C.c_double(); nv = C.c_uint64()
    rc = lib().orc_linearize(C.byref(m), kind, _dp(xyz), _dp(uv), xyz.shape[0], _dp(H), _dp(g), C.byref(cost), C.byref(nv), nthreads)
    if rc != 0:
        raise ValueError("oracle linearize: residual kind not defined for this model")
    return H, g, cost.value, nv.value


def lm_default_config() -> LMConfig:
    c = LMConfig(); lib().orc_lm_default_config(C.byref(c)); return c


def lm_solve(m: Model, kind: int, xyz, uv, lower=None, upper=None, cfg: LMConfig | None = None, nthreads: int = 1):
    xyz = np.ascontiguousarray(xyz, dtype=np.float64); uv = np.ascontiguousarray(uv, dtype=np.float64)
    P = m.n_params
    lo = np.ascontiguousarray(lower if lower is not None else np.full(P, -np.inf), dtype=np.float64)
    hi = np.ascontiguousarray(upper if upper is not None else np.full(P, np.inf), dtype=np.float64)
    cfg = cfg or lm_default_config()
    out = np.empty(P); res = LMResult()
    rc = lib().orc_lm_solve(C.byref(m), kind, _dp(xyz), _dp(uv), xyz.shape[0], _dp(lo), _dp(hi), C.byref(cfg), _dp(out), C.byref(res), nthreads)
    if rc != 0:
        raise ValueError("oracle lm_solve failed")
    return out, res


def linear_estimation(m: Model, xyz, uv) -> int:
    xyz = np.ascontiguousarray(xyz, dtype=np.float64); uv = np.ascontiguousarray(uv, dtype=np.float64)
    return lib().orc_linear_estimation(C.byref(m), _dp(xyz), _dp(uv), xyz.shape[0])


def sample_points(m: Model, n: int):
    total = lib().orc_sample_grid_size(C.byref(m), n, None, None)
    uv = np.empty((total, 2)); xyz = np.empty((total, 3))
    k = lib().orc_sample_points(C.byref(m), n, _dp(uv), _dp(xyz))
    return uv[:k].copy(), xyz[:k].copy()


def reprojection_error(m: Model, xyz, uv) -> ProjError:
    xyz = np.ascontiguousarray(xyz, dtype=np.float64); uv = np.ascontiguousarray(uv, dtype=np.float64)
    out = ProjError()
    rc = lib().orc_reprojection_error(C.byref(m), _dp(xyz), _dp(uv), xyz.shape[0], C.byref(out))
    if rc != 0:
        raise ValueError("ZeroProjectionPoints")
    return out


def undistort_rgb8(m: Model, target, img: np.ndarray, interp: int = 1, nthreads: int = 1) -> np.ndarray:
    img = np.ascontiguousarray(img, dtype=np.uint8); assert img.shape == (m.height, m.width, 3)
    t = np.ascontiguousarray(target, dtype=np.float64); out = np.empty_like(img)
    lib().orc_undistort_rgb8(C.byref(m), _dp(t), _u8p(img), _u8p(out), interp, nthreads)
    return out


def undistort_map(m: Model, target) -> np.ndarray:
    t = np.ascontiguousarray(target, dtype=np.float64); out = np.empty((m.height, m.width, 2))
    lib().orc_undistort_map(C.byref(m), _dp(t), _dp(out))
    return out


def synth_points3(seed: int, i0: int, n: int, cos_max: float, adversarial: bool) -> np.ndarray:
    out = np.empty((n, 3)); lib().orc_synth_points3(seed, i0, n, cos_max, int(adversarial), _dp(out)); return out


def synth_pixels(seed: int, i0: int, n: int, W: float, H: float) -> np.ndarray:
    out = np.empty((n, 2)); lib().orc_synth_pixels(seed, i0, n, W, H, _dp(out)); return out


def synth_bytes(seed: int, i0: int, n: int) -> np.ndarray:
    out = np.empty(n, dtype=np.uint8); lib().orc_synth_bytes(seed, i0, n, _u8p(out)); return out


# ---- util::image_quality (acm_oracle_image.c) ---------------------------------------------------
def _img(a):
    a = np.ascontiguousarray(a, dtype=np.uint8); assert a.ndim == 3 and a.shape[2] == 3
    return a


def image_psnr(a, b) -> float:
    a, b = _img(a), _img(b); assert a.shape == b.shape
    return float(lib().orc_image_psnr(_u8p(a), _u8p(b), a.shape[1], a.shape[0]))


def image_ssim(a, b) -> float:
    a, b = _img(a), _img(b); assert a.shape == b.shape
    return float(lib().orc_image_ssim(_u8p(a), _u8p(b), a.shape[1], a.shape[0]))


def rgb_to_grayscale(a) -> np.ndarray:
    a = _img(a); out = np.empty(a.shape[:2], dtype=np.uint8)
    lib().orc_rgb_to_grayscale(_u8p(a), a.shape[1], a.shape[0], _u8p(out)); return out


def draw_points(img, uv, color) -> np.ndarray:
    """Draws in place (and returns) radius-2 discs of `color` at the rounded points."""
    img = _img(img); uv = np.ascontiguousarray(uv, dtype=np.float64).reshape(-1, 2)
    lib().orc_draw_points_rgb8(_dp(uv), uv.shape[0], color[0], color[1], color[2], _u8p(img), img.shape[1], img.shape[0])
    return img


def image_quality_metrics(m_in: Model, m_out: Model, xyz, W: int, H: int, reference=None, want_image: bool = False):
    xyz = np.ascontiguousarray(xyz, dtype=np.float64).reshape(-1, 3)
    ref = _img(reference) if reference is not None else None
    comb = np.empty((H, W, 3), dtype=np.uint8) if want_image else None
    psnr, ssim = C.c_double(), C.c_double()
    kept = lib().orc_image_quality_metrics(C.byref(m_in), C.byref(m_out), _dp(xyz), xyz.shape[0], W, H,
                                           _u8p(ref) if ref is not None else None, _u8p(comb) if comb is not None else None,
                                           C.cast(C.byref(psnr), C.POINTER(C.c_double)), C.cast(C.byref(ssim), C.POINTER(C.c_double)))
    return kept, psnr.value, ssim.value, comb


def validate_conversion(m_out: Model, m_in: Model):
    err = np.empty(5); avg, mx = C.c_double(), C.c_double()
    valid = lib().orc_validate_conversion(C.byref(m_out), C.byref(m_in), _dp(err), C.cast(C.byref(avg), C.POINTER(C.c_double)),
                                          C.cast(C.byref(mx), C.POINTER(C.c_double)))
    return valid, err, avg.value, mx.value
