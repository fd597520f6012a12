"""ctypes binding of include/acm.h (libacm.so, built in-tree by __graft_entry__.build()).

There is no fallback: if the library is missing, importing this module raises; if no CUDA device
is present, `acm_ctx_create` fails with ACM_ERR_NO_DEVICE and `Context()` raises.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("ACM_LIB_PATH") or os.path.join(_HERE, "lib", "libacm.so")  # the override is a tuning aid (A/B of two builds)

ACM_MAX_PARAMS = 9
ABI_VERSION = 2  # include/acm.h ACM_ABI_VERSION: acm_lm_result gained device_ms, the *_multi entry points
F64, F32 = 0, 1
RESIDUAL_PIXEL, RESIDUAL_ALGEBRAIC = 0, 1
INTERP_NEAREST, INTERP_BILINEAR = 0, 1

OK = 0
ERR_INVALID_ARG, ERR_CUDA, ERR_NCCL, ERR_INVALID_PARAMS, ERR_NUMERICAL = -1, -2, -3, -4, -5
ERR_NO_DEVICE, ERR_ZERO_PROJECTION_POINTS, ERR_FOCAL_LENGTH, ERR_PRINCIPAL_POINT, ERR_PEER = -6, -7, -8, -9, -10


class Camera(C.Structure):
    _fields_ = [("model", C.c_int32), ("width", C.c_uint32), ("height", C.c_uint32),
                ("n_params", C.c_int32), ("params", C.c_double * ACM_MAX_PARAMS)]


class NormalEquations(C.Structure):
    _fields_ = [("n_params", C.c_int32), ("H", C.c_double * (ACM_MAX_PARAMS * ACM_MAX_PARAMS)),
                ("g", C.c_double * ACM_MAX_PARAMS), ("cost", C.c_double), ("n_valid", C.c_uint64)]


class LMConfig(C.Structure):
    _fields_ = [("max_iterations", C.c_int32), ("cost_tolerance", C.c_double), ("parameter_tolerance", C.c_double),
                ("gradient_tolerance", C.c_double), ("lambda0", C.c_double), ("invalid_penalty", C.c_double),
                ("check_every", C.c_int32)]


class LMResult(C.Structure):
    _fields_ = [("status", C.c_int32), ("iterations", C.c_int32), ("passes", C.c_int32),
                ("initial_cost", C.c_double), ("final_cost", C.c_double), ("n_valid", C.c_uint64),
                ("elapsed_ms", C.c_double), ("device_ms", C.c_double)]


class ImageQuality(C.Structure):
    _fields_ = [("psnr", C.c_double), ("ssim", C.c_double), ("n_points", C.c_uint64)]


class ProjectionError(C.Structure):
    _fields_ = [("rmse", C.c_double), ("min", C.c_double), ("max", C.c_double), ("mean", C.c_double),
                ("stddev", C.c_double), ("median", C.c_double), ("count", C.c_uint64)]


_vp, _dp, _u8p = C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_uint8)
_vpp = C.POINTER(C.c_void_p)
_cam = C.POINTER(Camera)

# name -> (restype, argtypes).  Must list every symbol include/acm.h declares
# (tests/test_abi.py parses the header and checks both directions).
SIGNATURES = {
    "acm_ctx_create": (C.c_int32, [C.c_int32, _vp, C.POINTER(_vp)]),
    "acm_ctx_destroy": (C.c_int32, [_vp]),
    "acm_ctx_sync": (C.c_int32, [_vp]),
    "acm_last_error": (C.c_char_p, [_vp]),
    "acm_abi_version": (C.c_int32, []),
    "acm_ctx_device_info": (C.c_int32, [_vp, C.POINTER(C.c_int64)]),
    "acm_timer_start": (C.c_int32, [_vp]),
    "acm_timer_stop": (C.c_int32, [_vp, C.POINTER(C.c_float)]),
    "acm_ctx_kernel_launches": (C.c_uint64, [_vp]),
    "acm_n_params": (C.c_int32, [C.c_int32]),
    "acm_camera_new": (C.c_int32, [C.c_int32, _dp, C.c_size_t, _cam, C.c_char_p, C.c_size_t]),
    "acm_validate_params": (C.c_int32, [_cam, C.c_char_p, C.c_size_t]),
    "acm_device_alloc": (C.c_int32, [_vp, C.c_size_t, C.POINTER(_vp)]),
    "acm_device_free": (C.c_int32, [_vp, _vp]),
    "acm_host_alloc_pinned": (C.c_int32, [_vp, C.c_size_t, C.POINTER(_vp)]),
    "acm_host_free_pinned": (C.c_int32, [_vp, _vp]),
    "acm_memcpy_h2d": (C.c_int32, [_vp, _vp, _vp, C.c_size_t]),
    "acm_memcpy_d2h": (C.c_int32, [_vp, _vp, _vp, C.c_size_t]),
    "acm_memcpy_d2d": (C.c_int32, [_vp, _vp, _vp, C.c_size_t]),
    "acm_memset_d": (C.c_int32, [_vp, _vp, C.c_int, C.c_size_t]),
    "acm_points_create": (C.c_int32, [_vp, C.c_int32, C.c_size_t, C.c_int32, C.POINTER(_vp)]),
    "acm_points_destroy": (C.c_int32, [_vp, _vp]),
    "acm_points_len": (C.c_size_t, [_vp]),
    "acm_points_dim": (C.c_int32, [_vp]),
    "acm_points_dtype": (C.c_int32, [_vp]),
    "acm_points_component": (_vp, [_vp, C.c_int32]),
    "acm_points_upload_aos_f64": (C.c_int32, [_vp, _vp, _vp, C.c_size_t]),
    "acm_points_download_aos_f64": (C.c_int32, [_vp, _vp, _vp, C.c_size_t]),
    "acm_project": (C.c_int32, [_vp, _cam, _vp, _vp, _vp]),
    "acm_unproject": (C.c_int32, [_vp, _cam, _vp, _vp, _vp]),
    "acm_unproject_ieee": (C.c_int32, [_vp, _cam, _vp, _vp, _vp]),
    "acm_camera_fast_unproject": (C.c_int32, [_cam]),
    "acm_project_unproject": (C.c_int32, [_vp, _cam, _vp, _vp, _vp, _vp, _vp]),
    "acm_project_jacobian": (C.c_int32, [_vp, _cam, _vp, _vp, _vp, _vp]),
    "acm_project_point_jacobian": (C.c_int32, [_vp, _cam, _vp, _vp, _vp, _vp]),
    "acm_project_host": (C.c_int32, [_vp, _cam, _vp, C.c_size_t, _vp, _vp]),
    "acm_unproject_host": (C.c_int32, [_vp, _cam, _vp, C.c_size_t, _vp, _vp]),
    "acm_linearize": (C.c_int32, [_vp, _cam, C.c_int32, _vp, _vp, C.POINTER(NormalEquations)]),
    "acm_linearize_async": (C.c_int32, [_vp, _cam, C.c_int32, _vp, _vp]),
    "acm_linearize_host": (C.c_int32, [_vp, _cam, C.c_int32, _vp, _vp, C.c_size_t, C.POINTER(NormalEquations)]),
    "acm_lm_default_config": (C.c_int32, [C.POINTER(LMConfig)]),
    "acm_lm_solve": (C.c_int32, [_vp, _cam, C.c_int32, _vp, _vp, _dp, _dp, C.POINTER(LMConfig), _dp, C.POINTER(LMResult)]),
    "acm_linear_estimation": (C.c_int32, [_vp, _cam, _vp, _vp]),
    "acm_undistort_rgb8": (C.c_int32, [_vp, _cam, _dp, _vp, _vp, C.c_size_t, C.c_int32]),
    "acm_undistort_rgb8_host": (C.c_int32, [_vp, _cam, _dp, _vp, _vp, C.c_size_t, C.c_int32]),
    "acm_undistort_map": (C.c_int32, [_vp, _cam, _dp, _vp]),
    "acm_remap_plan_create": (C.c_int32, [_vp, _cam, _cam, _dp, C.c_int32, C.POINTER(_vp)]),
    "acm_remap_plan_destroy": (C.c_int32, [_vp, _vp]),
    "acm_remap_rgb8": (C.c_int32, [_vp, _vp, _vp, _vp, C.c_size_t]),
    "acm_remap_rgb8_host": (C.c_int32, [_vp, _vp, _vp, _vp, C.c_size_t]),
    "acm_remap_map": (C.c_int32, [_vp, _cam, _cam, _vp]),
    "acm_remap_plan_create_rotated": (C.c_int32, [_vp, _cam, _cam, _dp, C.c_int32, C.POINTER(_vp)]),
    "acm_remap_map_rotated": (C.c_int32, [_vp, _cam, _cam, _dp, _vp]),
    "acm_stereo_rectify": (C.c_int32, [_dp, _dp, _dp, _dp, _dp, C.POINTER(C.c_int32)]),
    "acm_reprojection_error": (C.c_int32, [_vp, _cam, _vp, _vp, C.POINTER(ProjectionError)]),
    "acm_sample_points": (C.c_int32, [_vp, _cam, C.c_size_t, C.POINTER(_vp), C.POINTER(_vp), C.POINTER(C.c_size_t)]),
    "acm_sample_points_shard": (C.c_int32, [_vp, _cam, C.c_size_t, C.c_int32, C.c_int32, C.POINTER(_vp), C.POINTER(_vp), C.POINTER(C.c_size_t)]),
    "acm_image_psnr": (C.c_int32, [_vp, _vp, _vp, C.c_uint32, C.c_uint32, _dp]),
    "acm_image_ssim": (C.c_int32, [_vp, _vp, _vp, C.c_uint32, C.c_uint32, _dp]),
    "acm_draw_points_rgb8": (C.c_int32, [_vp, _vp, _vp, C.c_uint8, C.c_uint8, C.c_uint8, _vp, C.c_uint32, C.c_uint32]),
    "acm_image_quality_metrics": (C.c_int32, [_vp, _cam, _cam, _vp, C.c_uint32, C.c_uint32, _vp, _vp, C.POINTER(ImageQuality)]),
    "acm_synth_points3": (C.c_int32, [_vp, C.c_uint64, C.c_size_t, C.c_double, C.c_int32, _vp]),
    "acm_synth_pixels": (C.c_int32, [_vp, C.c_uint64, C.c_size_t, C.c_double, C.c_double, _vp]),
    "acm_synth_bytes": (C.c_int32, [_vp, C.c_uint64, C.c_size_t, _vp, C.c_size_t]),
    "acm_comm_get_unique_id": (C.c_int32, [_u8p]),
    "acm_comm_init_rank": (C.c_int32, [_vp, C.c_int32, C.c_int32, _u8p]),
    "acm_comm_destroy": (C.c_int32, [_vp]),
    "acm_comm_size": (C.c_int32, [_vp]),
    "acm_peer_export": (C.c_int32, [_vp, _u8p]),
    "acm_peer_attach": (C.c_int32, [_vp, C.c_int32, C.c_int32, _u8p]),
    "acm_peer_detach": (C.c_int32, [_vp]),
    "acm_comm_init_all": (C.c_int32, [_vpp, C.c_int32]),
    "acm_comm_destroy_all": (C.c_int32, [_vpp, C.c_int32]),
    "acm_linearize_multi": (C.c_int32, [_vpp, C.c_int32, _cam, C.c_int32, _vpp, _vpp, C.POINTER(NormalEquations)]),
    "acm_lm_solve_multi": (C.c_int32, [_vpp, C.c_int32, _cam, C.c_int32, _vpp, _vpp, _dp, _dp, C.POINTER(LMConfig), _dp, C.POINTER(LMResult)]),
    "acm_linear_estimation_multi": (C.c_int32, [_vpp, C.c_int32, _cam, _vpp, _vpp]),
    "acm_reprojection_error_multi": (C.c_int32, [_vpp, C.c_int32, _cam, _vpp, _vpp, C.POINTER(ProjectionError)]),
    "acm_sample_points_multi": (C.c_int32, [_vpp, C.c_int32, _cam, C.c_size_t, _vpp, _vpp, C.POINTER(C.c_size_t)]),
}


def load() -> C.CDLL:
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python __graft_entry__.py` (nvcc, sm_100a). "
            "apex_camera_models_b200 has no CPU or PyTorch fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError => the build is stale
        fn.restype, fn.argtypes = res, args
    if lib.acm_abi_version() != ABI_VERSION:
        raise ImportError(f"{LIB_PATH} has ABI version {lib.acm_abi_version()}, this package binds version {ABI_VERSION}: rebuild with `python __graft_entry__.py`")
    return lib


lib = load()
