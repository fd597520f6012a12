"""The seven camera models behind the reference's `CameraModel` trait surface.

Mirrors reference src/camera/mod.rs:241-340 (project, unproject, load_from_yaml, save_to_yaml,
validate_params, get_resolution, get_intrinsics, get_distortion, get_model_name), each model's
inherent `new(&DVector)` and `linear_estimation`, and the README-era `project(&p,
compute_jacobian)` spelling (reference README.md:119-126).  Every numeric result is produced by
the CUDA library through include/acm.h; batch methods are the intended hot path, the scalar
`project` / `unproject` are one-point batches that raise the reference's error variant.
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass

import numpy as np
import yaml

from . import _native as N
from .errors import (InvalidParams, IOError_, YamlError, raise_call_status, raise_point_status)
from .runtime import Context, Points, default_context

_lib = N.lib


@dataclass
class Intrinsics:  # mod.rs:52-62
    fx: float
    fy: float
    cx: float
    cy: float


@dataclass
class Resolution:  # mod.rs:67-73
    width: int
    height: int


class CameraModel:
    MODEL_ID = -1
    NAME = ""
    DISTORTION_NAMES: tuple = ()
    YAML_DISTORTION_KEY = None       # models whose YAML keeps distortion outside `intrinsics`
    YAML_SAVE_DISTORTION_KEY = None

    def __init__(self, intrinsics: Intrinsics, resolution: Resolution, distortion=(), ctx: Context | None = None):
        distortion = [float(v) for v in distortion]
        if len(distortion) != len(self.DISTORTION_NAMES):
            raise InvalidParams(f"{self.NAME} expects {len(self.DISTORTION_NAMES)} distortion parameters, got {len(distortion)}")
        self.intrinsics = intrinsics
        self.resolution = resolution
        self.distortions = distortion
        self._ctx = ctx

    # ---- plumbing ---------------------------------------------------------------------------
    @property
    def ctx(self) -> Context:
        if self._ctx is None:
            self._ctx = default_context()
        return self._ctx

    def params(self) -> np.ndarray:
        i = self.intrinsics
        return np.array([i.fx, i.fy, i.cx, i.cy] + list(self.distortions), dtype=np.float64)

    def set_params(self, p):
        p = [float(v) for v in p]
        self.intrinsics = Intrinsics(*p[:4])
        self.distortions = p[4:]

    def camera_block(self) -> N.Camera:
        cam = N.Camera()
        cam.model = self.MODEL_ID
        cam.width, cam.height = int(self.resolution.width), int(self.resolution.height)
        p = self.params()
        cam.n_params = len(p)
        for k, v in enumerate(p):
            cam.params[k] = v
        return cam

    def __getattr__(self, name):  # alpha / xi / beta / w / k1.. as attributes, like the Rust structs
        names = type(self).DISTORTION_NAMES
        if name in names:
            return self.distortions[names.index(name)]
        raise AttributeError(name)

    def __repr__(self):
        return f"{type(self).__name__}({self.intrinsics}, {self.resolution}, distortion={self.distortions})"

    # ---- constructors -----------------------------------------------------------------------
    @classmethod
    def new(cls, parameters, ctx: Context | None = None):
        """`<Model>::new(&DVector<f64>)`: length check for every model; Pinhole and RadTan also
        validate (pinhole.rs:101, rad_tan.rs:135).  Resolution is left at 0x0."""
        p = np.ascontiguousarray(parameters, dtype=np.float64).ravel()
        cam = N.Camera()
        msg = C.create_string_buffer(256)
        rc = _lib.acm_camera_new(cls.MODEL_ID, p.ctypes.data_as(C.POINTER(C.c_double)), len(p), C.byref(cam), msg, 256)
        if rc != N.OK:
            raise_call_status(rc, msg.value.decode())
        return cls(Intrinsics(*p[:4]), Resolution(0, 0), p[4:], ctx=ctx)

    @classmethod
    def load_from_yaml(cls, path: str, ctx: Context | None = None):
        """cam0: {intrinsics: [...], resolution: [w, h], (distortion: [...])}; the `camera_model`
        string is not read (mod.rs:412-501)."""
        try:
            with open(path) as f:
                text = f.read()
        except OSError as e:
            raise IOError_(str(e))
        try:
            doc = yaml.safe_load(text)
        except yaml.YAMLError as e:
            raise YamlError(str(e))
        if not doc:
            raise InvalidParams("Empty YAML document")
        cam = doc.get("cam0") if isinstance(doc, dict) else None
        if cam is None:
            raise InvalidParams("Missing 'cam0' node in YAML")
        intr = cam.get("intrinsics")
        if not isinstance(intr, list):
            raise InvalidParams("YAML missing 'intrinsics' array under 'cam0'")
        n_in_intr = 4 if cls.YAML_DISTORTION_KEY else 4 + len(cls.DISTORTION_NAMES)
        if len(intr) < n_in_intr:
            raise InvalidParams(f"Intrinsics array must have at least {n_in_intr} elements, got {len(intr)}")
        res = cam.get("resolution")
        if not isinstance(res, list):
            raise InvalidParams("YAML missing 'resolution' array under 'cam0'")
        if len(res) < 2:
            raise InvalidParams("Resolution array must have at least 2 elements (width, height)")
        for name, v in zip(("fx", "fy", "cx", "cy"), intr[:4]):
            if not isinstance(v, float):
                raise InvalidParams(f"Invalid {name}: not a float")
        if not all(isinstance(v, int) for v in res[:2]):
            raise InvalidParams("Invalid width: not an integer")
        if cls.YAML_DISTORTION_KEY:
            dist = cam.get(cls.YAML_DISTORTION_KEY)
            if not isinstance(dist, list):
                raise InvalidParams("Missing distortion parameters")
            if len(dist) < len(cls.DISTORTION_NAMES):
                raise InvalidParams(f"Expected {len(cls.DISTORTION_NAMES)} distortion parameters, got {len(dist)}")
            dist = dist[: len(cls.DISTORTION_NAMES)]
        else:
            dist = intr[4:]
            if len(dist) != len(cls.DISTORTION_NAMES):
                raise InvalidParams(f"{cls.NAME} model expects exactly {4 + len(cls.DISTORTION_NAMES)} parameters, got {len(intr)}")
        model = cls(Intrinsics(*[float(v) for v in intr[:4]]), Resolution(int(res[0]), int(res[1])), dist, ctx=ctx)
        model.validate_params()
        return model

    def save_to_yaml(self, path: str):
        i = self.intrinsics
        cam = {"camera_model": self.NAME}
        if self.YAML_SAVE_DISTORTION_KEY:
            cam["intrinsics"] = [i.fx, i.fy, i.cx, i.cy]
            cam[self.YAML_SAVE_DISTORTION_KEY] = list(self.distortions)
            cam["rostopic"] = "/cam0/image_raw"
        else:
            cam["intrinsics"] = [i.fx, i.fy, i.cx, i.cy] + list(self.distortions)
        cam["resolution"] = [int(self.resolution.width), int(self.resolution.height)]
        try:
            parent = os.path.dirname(path)
            if parent:
                os.makedirs(parent, exist_ok=True)
            with open(path, "w") as f:
                yaml.safe_dump({"cam0": cam}, f, sort_keys=False)
        except OSError as e:
            raise IOError_(str(e))

    # ---- trait getters ----------------------------------------------------------------------
    def validate_params(self):
        msg = C.create_string_buffer(256)
        cam = self.camera_block()
        rc = _lib.acm_validate_params(C.byref(cam), msg, 256)
        if rc != N.OK:
            raise_call_status(rc, msg.value.decode())

    def get_resolution(self) -> Resolution:
        return Resolution(self.resolution.width, self.resolution.height)

    def get_intrinsics(self) -> Intrinsics:
        i = self.intrinsics
        return Intrinsics(i.fx, i.fy, i.cx, i.cy)

    def get_distortion(self):
        return list(self.distortions)

    def get_model_name(self) -> str:
        return self.NAME

    # ---- hot path: batches ------------------------------------------------------------------
    def project_batch(self, points_3d, dtype: int = N.F64):
        """(N,3) host array or device `Points` -> (uv, status).  Host in -> numpy out ((N,2)
        float64, (N,) uint8); device in -> (`Points`, device status pointer)."""
        ctx = self.ctx
        cam = self.camera_block()
        if isinstance(points_3d, Points):
            with ctx.staging() as s:
                return s.keep(*self._map_points(s, points_3d, len(points_3d), 2, _lib.acm_project))
        a = np.ascontiguousarray(points_3d, dtype=np.float64).reshape(-1, 3)
        n = a.shape[0]
        if dtype == N.F64:
            uv = np.empty((n, 2)); st = np.empty(n, dtype=np.uint8)
            ctx.check(_lib.acm_project_host(ctx.handle, C.byref(cam), a.ctypes.data_as(C.c_void_p), n, uv.ctypes.data_as(C.c_void_p),
                                            st.ctypes.data_as(C.c_void_p)))
            return uv, st
        return self._host_map_via_points(a, 3, 2, _lib.acm_project, dtype)

    def unproject_batch(self, points_2d, dtype: int = N.F64):
        ctx = self.ctx
        cam = self.camera_block()
        if isinstance(points_2d, Points):
            with ctx.staging() as s:
                return s.keep(*self._map_points(s, points_2d, len(points_2d), 3, _lib.acm_unproject))
        a = np.ascontiguousarray(points_2d, dtype=np.float64).reshape(-1, 2)
        n = a.shape[0]
        if dtype == N.F64:
            xyz = np.empty((n, 3)); st = np.empty(n, dtype=np.uint8)
            ctx.check(_lib.acm_unproject_host(ctx.handle, C.byref(cam), a.ctypes.data_as(C.c_void_p), n, xyz.ctypes.data_as(C.c_void_p),
                                              st.ctypes.data_as(C.c_void_p)))
            return xyz, st
        return self._host_map_via_points(a, 2, 3, _lib.acm_unproject, dtype)

    def unproject_batch_ieee(self, points_2d):
        """`unproject` with IEEE arithmetic to the end (acm_unproject_ieee): same status bytes as unproject_batch, values
        bit-identical to the reference's for Pinhole / RadTan / UCM / EUCM / Double Sphere.  (N,2) -> (rays (N,3), status)."""
        a = np.ascontiguousarray(points_2d, dtype=np.float64).reshape(-1, 2)
        return self._host_map_via_points(a, 2, 3, _lib.acm_unproject_ieee, N.F64)

    def _map_points(self, s, src, n, dout, fn):
        """`fn` (acm_project / acm_unproject / acm_unproject_ieee) of the n device points `src`: (dst `Points`, status
        pointer), both owned by `s`."""
        ctx = self.ctx
        dst, st = s.own(Points(ctx, dout, n, src.dtype)), s.alloc(n)
        ctx.check(fn(ctx.handle, C.byref(self.camera_block()), src.handle, dst.handle, C.c_void_p(st)))
        return dst, st

    def _host_map_via_points(self, a, din, dout, fn, dtype):
        ctx = self.ctx
        n = a.shape[0]
        with ctx.staging() as s:
            dst, st_d = self._map_points(s, s.points(a, din, dtype), n, dout, fn)
            out = dst.numpy()
            st = np.empty(n, dtype=np.uint8)
            if n:
                ctx.d2h(st, st_d)
            ctx.sync()
        return out, st

    def round_trip_batch(self, points_3d, dtype: int = N.F64):
        """Fused project -> unproject (BASELINE config 2): (uv, ray, status_project, status_unproject).
        Host (N,3) array in -> numpy out; device `Points` in -> (Points, Points, status ptr, status ptr)."""
        ctx = self.ctx
        cam = self.camera_block()
        with ctx.staging() as s:
            src = s.points(points_3d, 3, dtype)
            n = len(src)
            uv, ray = s.own(Points(ctx, 2, n, src.dtype)), s.own(Points(ctx, 3, n, src.dtype))
            sp, su = s.alloc(n), s.alloc(n)
            ctx.check(_lib.acm_project_unproject(ctx.handle, C.byref(cam), src.handle, uv.handle, ray.handle, C.c_void_p(sp), C.c_void_p(su)))
            if isinstance(points_3d, Points):
                return s.keep(uv, ray, sp, su)
            a, b = uv.numpy(), ray.numpy()
            s1, s2 = np.empty(n, dtype=np.uint8), np.empty(n, dtype=np.uint8)
            if n:
                ctx.d2h(s1, sp); ctx.d2h(s2, su)
            ctx.sync()
        return a, b, s1, s2

    def _jacobian_batch(self, points_3d, fn, rows: int):
        """uv (N,2), J (N,2,rows/2) written by `fn` as `rows` rows of N, status (N,)."""
        ctx = self.ctx
        cam = self.camera_block()
        a = np.ascontiguousarray(points_3d, dtype=np.float64).reshape(-1, 3)
        n = a.shape[0]
        with ctx.staging() as s:
            src, uv = s.points(a, 3), s.own(Points(ctx, 2, n))
            d_j, d_s = s.alloc(n * rows * 8), s.alloc(n)
            ctx.check(fn(ctx.handle, C.byref(cam), src.handle, uv.handle, C.c_void_p(d_j), C.c_void_p(d_s)))
            J = np.empty((rows, n)); st = np.empty(n, dtype=np.uint8)
            if n:
                ctx.d2h(J, d_j); ctx.d2h(st, d_s)
            ctx.sync()
            out = uv.numpy()
        return out, np.ascontiguousarray(J.reshape(2, rows // 2, n).transpose(2, 0, 1)), st

    def project_jacobian_batch(self, points_3d):
        """uv (N,2), J (N,2,P) w.r.t. [fx,fy,cx,cy,dist..], status (N,); geometric validity only."""
        return self._jacobian_batch(points_3d, _lib.acm_project_jacobian, 2 * len(self.params()))

    def project_point_jacobian_batch(self, points_3d):
        """uv (N,2), J (N,2,3) = d(u,v)/d(x,y,z) -- the trait doc's "Jacobian matrix (2x3)" (mod.rs:246-252) --,
        status (N,); geometric validity only, J = 0 where the projection fails."""
        return self._jacobian_batch(points_3d, _lib.acm_project_point_jacobian, 6)

    # ---- trait: scalar project / unproject ---------------------------------------------------
    def project(self, point_3d, compute_jacobian=False):
        """`project(&Vector3) -> Result<Vector2, CameraModelError>` (mod.rs:256); with
        `compute_jacobian=True` (README.md:119-126) returns (uv, 2xP Jacobian w.r.t. the camera parameters, the
        shape the per-model docs give: double_sphere.rs:326-332 "2x6"); `compute_jacobian="point"` returns the
        2x3 Jacobian w.r.t. the 3-D point that the trait doc names (mod.rs:246-252)."""
        p = np.asarray(point_3d, dtype=np.float64).reshape(1, 3)
        uv, st = self.project_batch(p)
        raise_point_status(int(st[0]), self.MODEL_ID)
        if compute_jacobian:
            fn = self.project_point_jacobian_batch if compute_jacobian == "point" else self.project_jacobian_batch
            _, J, stj = fn(p)
            raise_point_status(int(stj[0]), self.MODEL_ID)
            return uv[0], J[0]
        return uv[0]

    def unproject(self, point_2d):
        p = np.asarray(point_2d, dtype=np.float64).reshape(1, 2)
        ray, st = self.unproject_batch(p)
        raise_point_status(int(st[0]), self.MODEL_ID)
        return ray[0]

    # ---- inherent linear_estimation -----------------------------------------------------------
    def linear_estimation(self, points_3d, points_2d):
        """`linear_estimation(&mut self, &Matrix3xX, &Matrix2xX)`; updates the distortion part."""
        ctx = self.ctx
        cam = self.camera_block()
        with ctx.staging() as s:
            X, UV = s.points(points_3d, 3), s.points(points_2d, 2)
            ctx.check(_lib.acm_linear_estimation(ctx.handle, C.byref(cam), X.handle, UV.handle))
        self.set_params(cam.params[: cam.n_params])


class PinholeModel(CameraModel):
    MODEL_ID, NAME, DISTORTION_NAMES = 0, "pinhole", ()

    def linear_estimation(self, points_3d, points_2d):
        raise AttributeError("PinholeModel has no linear_estimation (reference pinhole.rs:387)")


class RadTanModel(CameraModel):
    MODEL_ID, NAME, DISTORTION_NAMES = 1, "rad_tan", ("k1", "k2", "p1", "p2", "k3")
    YAML_DISTORTION_KEY = "distortion"        # rad_tan.rs:574
    YAML_SAVE_DISTORTION_KEY = "distortion"   # rad_tan.rs:695


class KannalaBrandtModel(CameraModel):
    MODEL_ID, NAME, DISTORTION_NAMES = 2, "kannala_brandt", ("k1", "k2", "k3", "k4")
    YAML_DISTORTION_KEY = "distortion"              # kannala_brandt.rs:635
    YAML_SAVE_DISTORTION_KEY = "distortion_coeffs"  # kannala_brandt.rs:737-741 (known asymmetry, kept)


class UcmModel(CameraModel):
    MODEL_ID, NAME, DISTORTION_NAMES = 3, "ucm", ("alpha",)


class EucmModel(CameraModel):
    MODEL_ID, NAME, DISTORTION_NAMES = 4, "eucm", ("alpha", "beta")


class DoubleSphereModel(CameraModel):
    MODEL_ID, NAME, DISTORTION_NAMES = 5, "double_sphere", ("alpha", "xi")


class FovModel(CameraModel):
    MODEL_ID, NAME, DISTORTION_NAMES = 6, "fov", ("w",)


MODEL_CLASSES = {c.MODEL_ID: c for c in (PinholeModel, RadTanModel, KannalaBrandtModel, UcmModel, EucmModel, DoubleSphereModel, FovModel)}
