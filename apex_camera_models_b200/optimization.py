"""The optimisation facade: README-era `*OptimizationCost::{new, linear_estimation, optimize,
get_intrinsics, get_distortion}` (reference README.md:70-81) and the v0.4.1 converter contract
(`*CameraParamsFactor` + `LevenbergMarquardt::with_config(cfg).optimize`, reference
bin/camera_converter.rs:378-420 and its five clones), over acm_linearize / acm_lm_solve.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass

import numpy as np

from . import _native as N
from .camera import (CameraModel, DoubleSphereModel, EucmModel, FovModel, KannalaBrandtModel, RadTanModel, UcmModel)
from .errors import InvalidParams

_lib = N.lib

# bounds of bin/camera_converter.rs: fx,fy in [1,2000], cx,cy in [0,2000] (:395-398) + per model
_F = [(1.0, 2000.0), (1.0, 2000.0), (0.0, 2000.0), (0.0, 2000.0)]
CONVERTER_BOUNDS = {
    5: _F + [(1e-6, 1.0), (-5.0, 5.0)],                              # DS   :399-400
    2: _F + [(-5.0, 5.0)] * 4,                                       # KB   :536-539
    1: _F + [(-5.0, 5.0), (-5.0, 5.0), (-1.0, 1.0), (-1.0, 1.0), (-5.0, 5.0)],  # RadTan :676-680
    3: _F + [(1e-6, 10.0)],                                          # UCM  :814
    4: _F + [(1e-6, 1.0), (1e-6, 5.0)],                              # EUCM :946-947
    6: _F + [(1e-6, 3.0)],                                           # FOV  :1078
}
# residual minimised per model (SURVEY.md 8c: the README figures are reproduced by the algebraic
# residual for the unified family; the others have no denominator form)
CANONICAL_RESIDUAL = {0: N.RESIDUAL_PIXEL, 1: N.RESIDUAL_PIXEL, 2: N.RESIDUAL_PIXEL, 3: N.RESIDUAL_ALGEBRAIC,
                      4: N.RESIDUAL_ALGEBRAIC, 5: N.RESIDUAL_ALGEBRAIC, 6: N.RESIDUAL_PIXEL}


@dataclass
class LevenbergMarquardtConfig:
    """LevenbergMarquardtConfig::new().with_max_iterations(100).with_cost_tolerance(1e-6)
    .with_parameter_tolerance(1e-8).with_gradient_tolerance(1e-6) (camera_converter.rs:410-415)."""
    max_iterations: int = 100
    cost_tolerance: float = 1e-6
    parameter_tolerance: float = 1e-8
    gradient_tolerance: float = 1e-6
    lambda0: float = 1e-3
    invalid_penalty: float = 0.0
    check_every: int = 4
    verbose: bool = False

    def native(self) -> N.LMConfig:
        c = N.LMConfig()
        c.max_iterations, c.cost_tolerance = self.max_iterations, self.cost_tolerance
        c.parameter_tolerance, c.gradient_tolerance = self.parameter_tolerance, self.gradient_tolerance
        c.lambda0, c.invalid_penalty, c.check_every = self.lambda0, self.invalid_penalty, self.check_every
        return c


@dataclass
class OptimizationResult:
    parameters: np.ndarray
    status: int
    iterations: int
    passes: int
    initial_cost: float
    final_cost: float
    n_valid: int
    elapsed_ms: float
    device_ms: float = 0.0   # first pass to last LM step on the device; device_ms / passes = per-iteration device time

    @property
    def converged(self) -> bool:
        return self.status in (0, 1, 2)


class OptimizationCost:
    """Holds a model and resident 3D-2D correspondences; `linear_estimation()` then `optimize()`."""
    MODEL = CameraModel

    def __init__(self, model: CameraModel, points_3d, points_2d, residual_kind: int | None = None):
        if not isinstance(model, self.MODEL):
            raise InvalidParams(f"{type(self).__name__} needs a {self.MODEL.__name__}")
        self.model = model
        self._staging = s = model.ctx.staging()  # the correspondences staged from host arrays, until free()
        self.points_3d, self.points_2d = s.points(points_3d, 3), s.points(points_2d, 2)
        if len(self.points_3d) != len(self.points_2d):
            s.close()
            raise InvalidParams("Number of 2D and 3D points must match")  # assert_eq! in the factor's new()
        self.residual_kind = CANONICAL_RESIDUAL[model.MODEL_ID] if residual_kind is None else residual_kind
        self.bounds = CONVERTER_BOUNDS.get(model.MODEL_ID)

    def linear_estimation(self):
        self.model.linear_estimation(self.points_3d, self.points_2d)

    def linearize(self):
        """One fused pass: (H = J^T J, g = J^T r, cost, n_valid) at the current parameters."""
        ctx = self.model.ctx
        cam = self.model.camera_block()
        ne = N.NormalEquations()
        ctx.check(_lib.acm_linearize(ctx.handle, C.byref(cam), self.residual_kind, self.points_3d.handle, self.points_2d.handle, C.byref(ne)))
        P = ne.n_params
        return (np.array(ne.H[: P * P]).reshape(P, P), np.array(ne.g[:P]), float(ne.cost), int(ne.n_valid))

    def optimize(self, verbose: bool = False, config: LevenbergMarquardtConfig | None = None, bounds="converter") -> OptimizationResult:
        ctx = self.model.ctx
        cam = self.model.camera_block()
        P = cam.n_params
        cfg = (config or LevenbergMarquardtConfig()).native()
        b = self.bounds if bounds == "converter" else bounds
        lo = hi = None
        if b is not None:
            lo = (C.c_double * P)(*[x[0] for x in b]); hi = (C.c_double * P)(*[x[1] for x in b])
        out = (C.c_double * N.ACM_MAX_PARAMS)()
        res = N.LMResult()
        ctx.check(_lib.acm_lm_solve(ctx.handle, C.byref(cam), self.residual_kind, self.points_3d.handle, self.points_2d.handle,
                                    lo, hi, C.byref(cfg), out, C.byref(res)))
        params = np.array(out[:P])
        self.model.set_params(params)
        r = OptimizationResult(params, res.status, res.iterations, res.passes, res.initial_cost, res.final_cost, int(res.n_valid), res.elapsed_ms, res.device_ms)
        if verbose or (config and config.verbose):
            print(f"[LM] status={r.status} iterations={r.iterations} passes={r.passes} cost {r.initial_cost:.6e} -> {r.final_cost:.6e}")
        return r

    def get_intrinsics(self):
        return self.model.get_intrinsics()

    def get_distortion(self):
        return self.model.get_distortion()

    def free(self):
        self._staging.close()


class DoubleSphereOptimizationCost(OptimizationCost):
    MODEL = DoubleSphereModel


class KannalaBrandtOptimizationCost(OptimizationCost):
    MODEL = KannalaBrandtModel


class RadTanOptimizationCost(OptimizationCost):
    MODEL = RadTanModel


class UcmOptimizationCost(OptimizationCost):
    MODEL = UcmModel


class EucmOptimizationCost(OptimizationCost):
    MODEL = EucmModel


class FovOptimizationCost(OptimizationCost):
    MODEL = FovModel
