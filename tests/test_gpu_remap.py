"""Remap plans on the GPU (acm_remap_*): maps against the remap oracle (tests/remap_oracle.c) for every model pair,
frame bytes on every path of the dispatch rule, undistort plans against acm_undistort_rgb8, plan reuse, argument
errors and the image_remap CLI."""
import ctypes as C
import os

import numpy as np
import pytest
import yaml

import remap_oracle as R
from conftest import oracle_model

pytestmark = pytest.mark.gpu

EXACT = {"pinhole", "rad_tan", "ucm", "eucm", "double_sphere"}  # unproject<true> + project: +,-,*,/,sqrt only
NAMES = ["pinhole", "rad_tan", "kannala_brandt", "ucm", "eucm", "double_sphere", "fov"]


@pytest.fixture(scope="module")
def acm():
    import apex_camera_models_b200 as m
    return m


@pytest.fixture(scope="module")
def ctx(acm):
    c = acm.Context(0)
    yield c
    c.close()


def sized(cameras, name, W, H, focal_scale=1.0):
    """The sample camera on a W x H grid: focal lengths scaled with the width (times focal_scale), principal point
    near the centre."""
    cam = dict(cameras[name])
    p = list(cam["params"])
    s = W / cam["width"] * focal_scale
    p[0], p[1], p[2], p[3] = p[0] * s, p[1] * s, W / 2.0 + 0.3, H / 2.0 - 0.2
    cam["params"], cam["width"], cam["height"] = p, W, H
    return cam


def gpu_model(acm, ctx, cam):
    cls = acm.MODEL_CLASSES[cam["model_id"]]
    return cls(acm.Intrinsics(*cam["params"][:4]), acm.Resolution(cam["width"], cam["height"]), cam["params"][4:], ctx=ctx)


def launches(ctx):
    from apex_camera_models_b200 import _native as N
    return N.lib.acm_ctx_kernel_launches(ctx.handle)


@pytest.mark.parametrize("mi", NAMES)
@pytest.mark.parametrize("mo", NAMES)
def test_remap_map_all_model_pairs(acm, ctx, O, cameras, mi, mo):
    """Same NaN pattern and floor indices as the oracle; bit-identical values where both models are arithmetic-only."""
    ci, co = sized(cameras, mi, 320, 240), sized(cameras, mo, 288, 224)
    got = acm.remap_map(gpu_model(acm, ctx, ci), gpu_model(acm, ctx, co))
    ref = R.remap_map(oracle_model(O, ci), oracle_model(O, co))
    assert got.shape == (224, 288, 2)
    assert np.array_equal(np.isnan(got), np.isnan(ref))
    ok = ~np.isnan(ref)
    assert ok.sum() > 0
    flips = int(np.sum(np.floor(got[ok]) != np.floor(ref[ok])))
    assert flips == 0, f"{flips} floor indices differ"
    if mi in EXACT and mo in EXACT:
        assert np.array_equal(got[ok], ref[ok])
    else:
        np.testing.assert_allclose(got[ok], ref[ok], rtol=0, atol=1e-9)


FRAME_PAIRS = [("kannala_brandt", "double_sphere"), ("double_sphere", "kannala_brandt"), ("rad_tan", "pinhole"), ("fov", "ucm"),
               ("eucm", "rad_tan"), ("kannala_brandt", "kannala_brandt")]


@pytest.mark.parametrize("mi,mo", FRAME_PAIRS)
def test_remap_frame_bytes(acm, ctx, O, cameras, mi, mo):
    """Device bytes equal interpolate_pixel on the device map; where the map is bit-identical to the oracle's they also
    equal the oracle's remap.  The same camera in and out puts weights of exactly 1 on the exact path."""
    ci, co = sized(cameras, mi, 320, 240), sized(cameras, mo, 320, 240)
    gi, go = gpu_model(acm, ctx, ci), gpu_model(acm, ctx, co)
    oi, oo = oracle_model(O, ci), oracle_model(O, co)
    frames = O.synth_bytes(0xACE50201, 0, 3 * 320 * 240 * 3).reshape(3, 240, 320, 3)
    mp = acm.remap_map(gi, go)
    exact_map = np.array_equal(mp, R.remap_map(oi, oo), equal_nan=True)
    if mi in EXACT and mo in EXACT:
        assert exact_map
    for interp in (acm.InterpolationMethod.Bilinear, acm.InterpolationMethod.Nearest):
        out = acm.remap_images(frames, gi, go, interp)
        assert out.shape == (3, 240, 320, 3)
        for f in range(3):
            ref = R.remap_apply_map(mp, frames[f], int(interp))
            assert np.array_equal(out[f], ref), f"frame {f} interp {interp}: {(out[f] != ref).sum()} bytes differ"
            if exact_map:
                assert np.array_equal(out[f], R.remap_rgb8(oi, oo, frames[f], int(interp)))
        assert np.array_equal(acm.remap_image(frames[1], gi, go, interp), out[1])


@pytest.mark.parametrize("Wi,Hi,Wo,Ho,kernels", [(512, 384, 384, 288, 2),   # TMA + leftover gather
                                                 (756, 480, 640, 480, 1),   # whole-image gather
                                                 (37, 29, 64, 48, 1),       # byte kernel: input width
                                                 (512, 384, 302, 226, 1)])  # byte kernel: output width
@pytest.mark.parametrize("zoom", [1.0, 0.3])
def test_remap_dispatch_paths(acm, ctx, O, cameras, Wi, Hi, Wo, Ho, kernels, zoom):
    """Every path of the plan's dispatch rule with Wi != Wo, 11 frames (the TMA ring wraps around); zoom 0.3 gives
    source boxes larger than the TMA tile, which the leftover gather takes."""
    ci, co = sized(cameras, "kannala_brandt", Wi, Hi), sized(cameras, "double_sphere", Wo, Ho, zoom)
    gi, go = gpu_model(acm, ctx, ci), gpu_model(acm, ctx, co)
    F = 11
    frames = O.synth_bytes(0xACE50202, 0, F * Wi * Hi * 3).reshape(F, Hi, Wi, 3)
    mp = acm.remap_map(gi, go)
    for interp in (acm.InterpolationMethod.Bilinear, acm.InterpolationMethod.Nearest):
        with acm.RemapPlan(gi, go, None, interp) as plan:
            d_in, d_out = ctx.device_alloc(frames.nbytes), ctx.device_alloc(F * Wo * Ho * 3)
            try:
                ctx.h2d(d_in, frames)
                n0 = launches(ctx)
                plan.apply_device(d_in, d_out, F)
                assert launches(ctx) - n0 == kernels
                out = np.empty((F, Ho, Wo, 3), np.uint8); ctx.d2h(out, d_out); ctx.sync()
            finally:
                ctx.device_free(d_in); ctx.device_free(d_out)
        for f in range(F):
            ref = R.remap_apply_map(mp, frames[f], int(interp))
            assert np.array_equal(out[f], ref), f"frame {f} interp {interp}: {(out[f] != ref).sum()} bytes differ"


@pytest.mark.parametrize("in_shift,out_shift", [(1, 1), (1, 0), (0, 1)])
def test_remap_unaligned_device_buffers(acm, ctx, O, cameras, in_shift, out_shift):
    """Frame buffers 1 byte off their allocation: the byte kernel takes them; bytes equal the oracle's on the device map."""
    ci, co = sized(cameras, "kannala_brandt", 512, 384), sized(cameras, "double_sphere", 384, 288)
    gi, go = gpu_model(acm, ctx, ci), gpu_model(acm, ctx, co)
    F = 3
    frames = O.synth_bytes(0xACE50203, 0, F * 512 * 384 * 3).reshape(F, 384, 512, 3)
    mp = acm.remap_map(gi, go)
    d_in, d_out = ctx.device_alloc(frames.nbytes + 16), ctx.device_alloc(F * 384 * 288 * 3 + 16)
    try:
        ctx.h2d(d_in + in_shift, frames)
        for interp in (acm.InterpolationMethod.Bilinear, acm.InterpolationMethod.Nearest):
            with acm.RemapPlan(gi, go, None, interp) as plan:
                plan.apply_device(d_in + in_shift, d_out + out_shift, F)
            out = np.empty((F, 288, 384, 3), np.uint8); ctx.d2h(out, d_out + out_shift); ctx.sync()
            for f in range(F):
                assert np.array_equal(out[f], R.remap_apply_map(mp, frames[f], int(interp)))
    finally:
        ctx.device_free(d_in); ctx.device_free(d_out)


@pytest.mark.parametrize("name,W,H", [("kannala_brandt", 512, 512), ("double_sphere", 752, 480), ("pinhole", 752, 480),
                                      ("rad_tan", 752, 480), ("fov", 320, 200), ("ucm", 1920, 1080), ("kannala_brandt", 37, 29),
                                      ("double_sphere", 756, 480)])
def test_undistort_plan_equals_undistort(acm, ctx, O, cameras, name, W, H):
    """A plan without an output camera is undistort_image: byte-identical to acm_undistort_rgb8 on every path."""
    cam = dict(cameras[name]); cam["width"], cam["height"] = W, H
    if name in ("ucm", "fov"):
        cam["params"] = list(cam["params"]); cam["params"][2] = W / 2.0 + 0.3; cam["params"][3] = H / 2.0 - 0.2
    if (W, H) == (37, 29):
        cam["params"] = [20.0, 20.0, 18.2, 14.1] + cam["params"][4:]
    m = gpu_model(acm, ctx, cam)
    frames = O.synth_bytes(0xACE50204, 0, 3 * W * H * 3).reshape(3, H, W, 3)
    for target in (None, acm.Intrinsics(cam["params"][0] * 0.6, cam["params"][1] * 0.6, W / 2.0, H / 2.0)):
        for interp in (acm.InterpolationMethod.Bilinear, acm.InterpolationMethod.Nearest):
            with acm.RemapPlan(m, None, target, interp) as plan:
                out = plan.apply(frames)
            assert np.array_equal(out, acm.undistort_images(frames, m, target, interp)), f"{name} {W}x{H} {target} {interp}"


@pytest.mark.parametrize("in_shift,out_shift", [(1, 1), (1, 0), (0, 1)])
def test_undistort_plan_unaligned_equals_undistort(acm, ctx, O, cameras, in_shift, out_shift):
    from apex_camera_models_b200 import _native as N
    cam = dict(cameras["kannala_brandt"]); W, H, F = 512, 512, 3
    m = gpu_model(acm, ctx, cam)
    blk = m.camera_block()
    frames = O.synth_bytes(0xACE50205, 0, F * W * H * 3).reshape(F, H, W, 3)
    nb = frames.nbytes
    d_in, d_out, d_ref = ctx.device_alloc(nb + 16), ctx.device_alloc(nb + 16), ctx.device_alloc(nb + 16)
    try:
        ctx.h2d(d_in + in_shift, frames)
        for target in (None, acm.Intrinsics(cam["params"][0] * 0.6, cam["params"][1] * 0.6, W / 2.0, H / 2.0)):
            t = None if target is None else (C.c_double * 4)(target.fx, target.fy, target.cx, target.cy)
            for interp in (acm.InterpolationMethod.Bilinear, acm.InterpolationMethod.Nearest):
                with acm.RemapPlan(m, None, target, interp) as plan:
                    plan.apply_device(d_in + in_shift, d_out + out_shift, F)
                ctx.check(N.lib.acm_undistort_rgb8(ctx.handle, C.byref(blk), t, C.c_void_p(d_in + in_shift), C.c_void_p(d_ref + out_shift),
                                                   F, int(interp)))
                out, ref = np.empty_like(frames), np.empty_like(frames)
                ctx.d2h(out, d_out + out_shift); ctx.d2h(ref, d_ref + out_shift); ctx.sync()
                assert np.array_equal(out, ref), f"target {target} interp {interp}"
    finally:
        ctx.device_free(d_in); ctx.device_free(d_out); ctx.device_free(d_ref)


def test_plan_reuse(acm, ctx, O, cameras):
    """One plan over two batches and frame by frame equals one batched call; two plans from the same inputs agree."""
    ci, co = sized(cameras, "kannala_brandt", 512, 384), sized(cameras, "double_sphere", 384, 288)
    gi, go = gpu_model(acm, ctx, ci), gpu_model(acm, ctx, co)
    frames = O.synth_bytes(0xACE50206, 0, 6 * 512 * 384 * 3).reshape(6, 384, 512, 3)
    with acm.RemapPlan(gi, go) as plan, acm.RemapPlan(gi, go) as twin:
        whole = plan.apply(frames)
        assert np.array_equal(np.concatenate([plan.apply(frames[:2]), plan.apply(frames[2:])]), whole)
        assert np.array_equal(np.stack([plan.apply(frames[f:f + 1])[0] for f in range(6)]), whole)
        assert np.array_equal(twin.apply(frames), whole)
    assert np.array_equal(acm.remap_map(gi, go), acm.remap_map(gi, go), equal_nan=True)


def test_remap_argument_errors(acm, ctx, O, cameras):
    from apex_camera_models_b200 import _native as N
    L = N.lib
    ci, co = sized(cameras, "kannala_brandt", 64, 48), sized(cameras, "double_sphere", 64, 48)
    gi, go = gpu_model(acm, ctx, ci), gpu_model(acm, ctx, co)
    bi, bo = gi.camera_block(), go.camera_block()
    h = C.c_void_p()

    def fails(rc, text):
        assert rc == N.ERR_INVALID_ARG, rc
        assert text in L.acm_last_error(ctx.handle).decode()

    t = (C.c_double * 4)(30.0, 30.0, 32.0, 24.0)
    fails(L.acm_remap_plan_create(ctx.handle, C.byref(bi), C.byref(bo), t, 1, C.byref(h)), "not both")
    for side in ("input", "output"):
        for w, hh, text in ((0, 48, "resolution must be set"), (64, 0, "resolution must be set"), (40000, 20000, "2 GiB")):
            b = N.Camera.from_buffer_copy(bi if side == "input" else bo)
            b.width, b.height = w, hh
            args = (C.byref(b), C.byref(bo)) if side == "input" else (C.byref(bi), C.byref(b))
            fails(L.acm_remap_plan_create(ctx.handle, *args, None, 1, C.byref(h)), f"{side} ")
            fails(L.acm_remap_plan_create(ctx.handle, *args, None, 1, C.byref(h)), text)
            d = ctx.device_alloc(16)
            fails(L.acm_remap_map(ctx.handle, *args, C.c_void_p(d)), text)
            ctx.device_free(d)
    # the undistort host entry checks its camera as plan creation does, before it allocates
    b = N.Camera.from_buffer_copy(bi)
    b.width = 0
    frame = np.zeros((48, 64, 3), np.uint8)
    fails(L.acm_undistort_rgb8_host(ctx.handle, C.byref(b), None, frame.ctypes.data_as(C.c_void_p), frame.ctypes.data_as(C.c_void_p), 1, 1),
          "resolution must be set")
    fails(L.acm_remap_plan_create(ctx.handle, C.byref(bi), C.byref(bo), None, 2, C.byref(h)), "unknown interpolation")
    fails(L.acm_remap_map(ctx.handle, C.byref(bi), C.byref(bo), None), "null output")
    with acm.RemapPlan(gi, go) as plan:
        d_in, d_out = ctx.device_alloc(64 * 48 * 3), ctx.device_alloc(64 * 48 * 3)
        try:
            fails(L.acm_remap_rgb8(ctx.handle, plan.handle, None, C.c_void_p(d_out), 1), "null frame buffer")
            fails(L.acm_remap_rgb8(ctx.handle, plan.handle, C.c_void_p(d_in), None, 1), "null frame buffer")
            fails(L.acm_remap_rgb8(ctx.handle, None, C.c_void_p(d_in), C.c_void_p(d_out), 1), "null plan")
            n0 = launches(ctx)
            assert L.acm_remap_rgb8(ctx.handle, plan.handle, C.c_void_p(d_in), C.c_void_p(d_out), 0) == N.OK
            assert L.acm_remap_rgb8_host(ctx.handle, plan.handle, None, None, 0) == N.OK
            assert launches(ctx) == n0
            other = acm.Context(0)
            try:
                rc = L.acm_remap_rgb8(other.handle, plan.handle, C.c_void_p(d_in), C.c_void_p(d_out), 1)
                assert rc == N.ERR_INVALID_ARG and "another context" in L.acm_last_error(other.handle).decode()
                rc = L.acm_remap_plan_destroy(other.handle, plan.handle)
                assert rc == N.ERR_INVALID_ARG and "another context" in L.acm_last_error(other.handle).decode()
            finally:
                other.close()
        finally:
            ctx.device_free(d_in); ctx.device_free(d_out)
        with pytest.raises(acm.UtilError, match="doesn't match model"):
            plan.apply(np.zeros((1, 49, 64, 3), np.uint8))
    with pytest.raises(acm.UtilError, match="doesn't match model"):
        acm.remap_images(np.zeros((1, 48, 63, 3), np.uint8), gi, go)
    with pytest.raises(acm.UtilError, match="doesn't match model"):
        acm.remap_image(np.zeros((48, 65, 3), np.uint8), gi, go)


def test_image_remap_cli(acm, ctx, O, cameras, tmp_path):
    from PIL import Image

    from apex_camera_models_b200 import image_remap
    ci, co = sized(cameras, "kannala_brandt", 320, 240), sized(cameras, "double_sphere", 256, 192)
    # calibration files in the loaders' format (kannala_brandt.rs:635 reads `distortion`; its saver writes
    # `distortion_coeffs`, so a saved KB file does not load back)
    with open(tmp_path / "in.yaml", "w") as f:
        yaml.safe_dump({"cam0": {"camera_model": "kannala_brandt", "intrinsics": ci["params"][:4], "distortion": ci["params"][4:],
                                 "resolution": [320, 240]}}, f)
    with open(tmp_path / "out.yaml", "w") as f:
        yaml.safe_dump({"cam0": {"camera_model": "double_sphere", "intrinsics": co["params"], "resolution": [256, 192]}}, f)
    img = O.synth_bytes(0xACE50207, 0, 320 * 240 * 3).reshape(240, 320, 3)
    Image.fromarray(img, "RGB").save(tmp_path / "in.png")
    for interp, flag in ((1, []), (0, ["--interpolation", "nearest"])):
        out_png = str(tmp_path / f"out{interp}.png")
        assert image_remap.main(["-i", str(tmp_path / "in.png"), "-c", str(tmp_path / "in.yaml"), "-m", "kb",
                                 "--output-calib", str(tmp_path / "out.yaml"), "--output-model", "ds", "-o", out_png] + flag) == 0
        got = np.asarray(Image.open(out_png).convert("RGB"))
        mi = acm.KannalaBrandtModel.load_from_yaml(str(tmp_path / "in.yaml"), ctx=ctx)
        mo = acm.DoubleSphereModel.load_from_yaml(str(tmp_path / "out.yaml"), ctx=ctx)
        assert got.shape == (192, 256, 3)
        assert np.array_equal(got, R.remap_apply_map(acm.remap_map(mi, mo), img, interp))
    assert os.path.exists(tmp_path / "out1.png")
