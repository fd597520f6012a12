"""Device temporaries of the Python wrappers: every wrapper that stages buffers or `Points` on the device frees all of them,
when the call succeeds and when libacm fails after staging.  A ledger wraps libacm's allocators and releasers, so the
check does not depend on when the garbage collector runs."""
from types import SimpleNamespace

import numpy as np
import pytest

from apex_camera_models_b200 import _native as N

pytestmark = pytest.mark.gpu

# name -> positions of the `C.byref(c_void_p)` out-arguments that receive a new device buffer or point handle
ALLOCATORS = {"acm_device_alloc": (2,), "acm_points_create": (4,), "acm_sample_points_shard": (5, 6)}
RELEASERS = ("acm_device_free", "acm_points_destroy")


@pytest.fixture(scope="module")
def acm():
    import apex_camera_models_b200 as m
    return m


@pytest.fixture(scope="module")
def ctx(acm):
    c = acm.Context(0)
    yield c
    c.close()


def _model(acm, ctx, cam):
    cls = acm.MODEL_CLASSES[cam["model_id"]]
    return cls(acm.Intrinsics(*cam["params"][:4]), acm.Resolution(cam["width"], cam["height"]), cam["params"][4:], ctx=ctx)


def _copy(m):
    return type(m)(m.get_intrinsics(), m.get_resolution(), m.get_distortion(), ctx=m.ctx)


def _short(m):
    """`m` with its last distortion coefficient removed: libacm rejects the camera block (ACM_ERR_INVALID_PARAMS)."""
    b = _copy(m)
    b.distortions = b.distortions[:-1]
    return b


def make_env(acm, ctx, cameras):
    kb, ds, pin = (_model(acm, ctx, cameras[n]) for n in ("kannala_brandt", "double_sphere", "pinhole"))
    uv, X = acm.sample_points(kb, 2000)
    rgb = np.random.default_rng(7).integers(0, 256, (3, 512, 512, 3), dtype=np.uint8)
    return SimpleNamespace(
        acm=acm, ctx=ctx, kb=kb, ds=ds, pin=pin, bad_kb=_short(kb), bad_ds=_short(ds), X=X, uv=uv,
        Xd=acm.Points.from_numpy(ctx, X), uvd=acm.Points.from_numpy(ctx, uv),
        uv2=kb.project_batch(X + [-0.1, 0.0, 0.0])[0], t=np.array([-0.1, 0.0, 0.0]),
        rng=acm.render_depth(kb, X)[0], img1=rgb[0], img2=rgb[1], ref=rgb[2],
        behind=np.tile([0.0, 0.0, -1.0], (16, 1)),  # no pinhole projects them
        errors=(acm.AcmError, acm.CameraModelError, acm.UtilError))


def _free(e, *objs):
    """Frees caller-owned results: `Points` and raw status pointers."""
    for o in objs:
        if isinstance(o, e.acm.Points):
            o.free()
        else:
            e.ctx.device_free(o)


def _cost(e, X):
    c = e.acm.OptimizationCost(_copy(e.ds), X, e.uv)
    c.linearize()
    c.free()


# (id, one succeeding call that frees whatever it is handed, one call that fails in libacm after staging or None)
SITES = [
    ("project_batch-device", lambda e: _free(e, *e.kb.project_batch(e.Xd)), lambda e: e.bad_kb.project_batch(e.Xd)),
    ("project_batch-f32", lambda e: e.kb.project_batch(e.X, N.F32), lambda e: e.bad_kb.project_batch(e.X, N.F32)),
    ("unproject_batch-device", lambda e: _free(e, *e.kb.unproject_batch(e.uvd)), lambda e: e.bad_kb.unproject_batch(e.uvd)),
    ("unproject_batch-f32", lambda e: e.kb.unproject_batch(e.uv, N.F32), lambda e: e.bad_kb.unproject_batch(e.uv, N.F32)),
    ("unproject_batch_ieee", lambda e: e.kb.unproject_batch_ieee(e.uv), lambda e: e.bad_kb.unproject_batch_ieee(e.uv)),
    ("round_trip_batch-host", lambda e: e.kb.round_trip_batch(e.X), lambda e: e.bad_kb.round_trip_batch(e.X)),
    ("round_trip_batch-device", lambda e: _free(e, *e.kb.round_trip_batch(e.Xd)), lambda e: e.bad_kb.round_trip_batch(e.Xd)),
    ("project_jacobian_batch", lambda e: e.kb.project_jacobian_batch(e.X), lambda e: e.bad_kb.project_jacobian_batch(e.X)),
    ("project_point_jacobian_batch", lambda e: e.kb.project_point_jacobian_batch(e.X),
     lambda e: e.bad_kb.project_point_jacobian_batch(e.X)),
    ("linear_estimation", lambda e: _copy(e.ds).linear_estimation(e.X, e.uv), lambda e: e.bad_ds.linear_estimation(e.X, e.uv)),
    ("undistort_map", lambda e: e.acm.undistort_map(e.kb), lambda e: e.acm.undistort_map(e.bad_kb)),
    ("remap_map", lambda e: e.acm.remap_map(e.kb, e.ds), lambda e: e.acm.remap_map(e.bad_kb, e.ds)),
    ("remap_map-rotated", lambda e: e.acm.remap_map(e.kb, e.ds, np.eye(3)), lambda e: e.acm.remap_map(e.kb, e.bad_ds, np.eye(3))),
    ("sample_points-host", lambda e: e.acm.sample_points(e.kb, 500), None),
    ("sample_points-device", lambda e: _free(e, *e.acm.sample_points(e.kb, 500, device=True)), None),
    ("compute_reprojection_error", lambda e: e.acm.compute_reprojection_error(e.kb, e.X, e.uv),
     lambda e: e.acm.compute_reprojection_error(e.kb, e.X[:-1], e.uv)),
    ("triangulate_points-device", lambda e: e.acm.triangulate_points(e.kb, e.kb, np.eye(3), e.t, e.uvd, e.uv2),
     lambda e: e.acm.triangulate_points(e.kb, e.kb, np.eye(3), np.zeros(3), e.uvd, e.uv2)),
    ("render_depth-device", lambda e: e.acm.render_depth(e.kb, e.Xd), lambda e: e.acm.render_depth(e.kb, e.Xd, None, [np.nan, 0.0, 0.0])),
    ("depth_to_points", lambda e: e.acm.depth_to_points(e.kb, e.rng), lambda e: e.acm.depth_to_points(e.kb, e.rng, 2.0 * np.eye(3))),
    ("calculate_psnr", lambda e: e.acm.calculate_psnr(e.img1, e.img2, e.ctx), None),
    ("calculate_ssim", lambda e: e.acm.calculate_ssim(e.img1, e.img2, e.ctx), None),
    ("create_projection_image", lambda e: e.acm.create_projection_image(e.uv, (0, 255, 0), 512, 512, e.ctx), None),
    ("create_combined_projection_image_on_reference",
     lambda e: e.acm.create_combined_projection_image_on_reference(e.uv, e.uvd, e.ref, e.ctx), None),
    ("model_projection_visualization-reference", lambda e: e.acm.model_projection_visualization(e.uv, e.ref, None, e.ctx), None),
    ("model_projection_visualization-black", lambda e: e.acm.model_projection_visualization(e.uv, None, (512, 512), e.ctx), None),
    ("compute_image_quality_metrics", lambda e: e.acm.compute_image_quality_metrics(e.kb, e.kb, e.X, e.ref, return_image=True),
     lambda e: e.acm.compute_image_quality_metrics(e.pin, e.pin, e.behind)),
    ("OptimizationCost", lambda e: _cost(e, e.X), lambda e: _cost(e, e.X[:-1])),
]


class Ledger:
    """Device buffers and point handles handed out by libacm while the ledger is installed, keyed by pointer."""

    def __init__(self):
        self.live, self.freed, self.errors = {}, set(), []

    def wrap(self, name, fn):
        if name in ALLOCATORS:
            def call(*args):
                rc = fn(*args)
                if rc == N.OK:
                    for i in ALLOCATORS[name]:
                        p = args[i]._obj.value
                        self.live[p] = name
                        self.freed.discard(p)
                return rc
        else:
            def call(*args):
                p = getattr(args[1], "value", args[1])
                if p in self.live:
                    del self.live[p]
                    self.freed.add(p)
                elif p in self.freed:
                    self.errors.append(f"{name}: second free of {p:#x}")
                # else: allocated before the ledger started (an object of an earlier test being collected)
                return fn(*args)
        return call


@pytest.fixture(scope="module")
def env(acm, ctx, cameras):
    return make_env(acm, ctx, cameras)


@pytest.fixture
def ledger(monkeypatch, env):
    L = Ledger()
    for name in (*ALLOCATORS, *RELEASERS):
        monkeypatch.setattr(N.lib, name, L.wrap(name, getattr(N.lib, name)))
    return L


@pytest.mark.parametrize("site", SITES, ids=[s[0] for s in SITES])
def test_success_frees_temporaries(env, ledger, site):
    site[1](env)
    assert ledger.errors == []
    assert ledger.live == {}, f"{site[0]} left {sorted(ledger.live.values())} allocated"


@pytest.mark.parametrize("site", [s for s in SITES if s[2]], ids=[s[0] for s in SITES if s[2]])
def test_failure_after_staging_frees_temporaries(env, ledger, site):
    with pytest.raises(env.errors) as info:
        site[2](env)
    # `info` keeps the traceback, and the frames' locals with it, alive: only explicit frees count
    assert ledger.errors == []
    assert ledger.live == {}, f"{site[0]} ({info.value!r}) left {sorted(ledger.live.values())} allocated"
