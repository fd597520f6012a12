"""apex_camera_models_b200 -- B200-native hot path of apex-camera-models.

Python mirror of the reference's `CameraModel` trait surface (reference src/camera/mod.rs:241-340),
the per-model `linear_estimation`, the README-era `*OptimizationCost` facade and the util hot
loops, implemented over the C ABI of include/acm.h (libacm.so, hand-written sm_100a CUDA).

Importing this package loads libacm.so; there is no CPU / PyTorch fallback.  Creating a
`Context` without a CUDA device raises `AcmError`.
"""
from . import _native  # noqa: F401  (raises ImportError if libacm.so has not been built)
from .errors import (AcmError, CameraModelError, FocalLengthMustBePositive, InvalidParams, IOError_, NumericalError,
                     PointAtCameraCenter, PointIsOutSideImage, PrincipalPointMustBeFinite, ProjectionOutSideImage,
                     UtilError, YamlError, ZeroProjectionPoints)
from .runtime import Context, Points, default_context
from .camera import (CameraModel, DoubleSphereModel, EucmModel, FovModel, Intrinsics, KannalaBrandtModel, PinholeModel,
                     RadTanModel, Resolution, UcmModel, MODEL_CLASSES)
from .optimization import (DoubleSphereOptimizationCost, EucmOptimizationCost, FovOptimizationCost,
                           KannalaBrandtOptimizationCost, LevenbergMarquardtConfig, OptimizationCost, RadTanOptimizationCost,
                           UcmOptimizationCost, CONVERTER_BOUNDS, CANONICAL_RESIDUAL)
from .util import (DepthStatus, InterpolationMethod, ProjectionError, RemapPlan, StereoRectifier, TriangulationStatus,
                   compute_reprojection_error, depth_to_points, remap_image, remap_images, remap_map, render_depth, sample_points,
                   stereo_rectify, triangulate_points, undistort_image, undistort_images, undistort_map)
from .image_quality import (ImageQualityMetrics, calculate_psnr, calculate_ssim, compute_image_quality_metrics,
                            create_combined_projection_image, create_combined_projection_image_on_reference,
                            create_projection_image, model_projection_visualization)
from .distributed import ContextGroup, attach_communicator, attach_peers, shard_range

__all__ = [n for n in dir() if not n.startswith("_")]
