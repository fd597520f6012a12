"""Rotated remap plans and stereo rectification on the GPU (acm_remap_plan_create_rotated, acm_remap_map_rotated):
identity rotations against unrotated plans, rotated maps against the rotated oracle (tests/rectify_oracle.c) for every
model pair and against OpenCV's initUndistortRectifyMap frozen in tests/golden/opencv_rectify.json, frame bytes on every
dispatch path, a rectified KB / Double Sphere pair end to end, argument errors, plan reuse and the image_rectify CLI."""
import ctypes as C

import numpy as np
import pytest
import yaml

import rectify_oracle as RO
import remap_oracle as R
from conftest import load_golden, oracle_model
from test_gpu_remap import EXACT, NAMES, gpu_model, launches, sized

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def acm():
    import apex_camera_models_b200 as m
    return m


@pytest.fixture(scope="module")
def ctx(acm):
    c = acm.Context(0)
    yield c
    c.close()


def axis_angle(axis, deg):
    """Rotation matrix of `deg` degrees about `axis` (Rodrigues, numpy)."""
    k = np.asarray(axis, np.float64) / np.linalg.norm(axis)
    K = np.array([[0.0, -k[2], k[1]], [k[2], 0.0, -k[0]], [-k[1], k[0], 0.0]])
    a = np.deg2rad(deg)
    return np.eye(3) + np.sin(a) * K + (1.0 - np.cos(a)) * (K @ K)


ROT10 = axis_angle([0.3, -0.8, 0.5], 10.0)
ROT25 = axis_angle([0.2, 1.0, -0.4], 25.0)


@pytest.mark.parametrize("mi", NAMES)
@pytest.mark.parametrize("mo", NAMES)
def test_identity_rotation_equals_unrotated(acm, ctx, O, cameras, mi, mo):
    """R = I: the rotated map is the unrotated map bit for bit, and a rotated plan's frame bytes equal the plain plan's."""
    ci, co = sized(cameras, mi, 320, 240), sized(cameras, mo, 288, 224)
    gi, go = gpu_model(acm, ctx, ci), gpu_model(acm, ctx, co)
    assert np.array_equal(acm.remap_map(gi, go, rotation=np.eye(3)), acm.remap_map(gi, go), equal_nan=True)
    frames = O.synth_bytes(0xACE5EC01, 0, 2 * 320 * 240 * 3).reshape(2, 240, 320, 3)
    with acm.RemapPlan(gi, go, rotation=np.eye(3)) as rot, acm.RemapPlan(gi, go) as plain:
        assert np.array_equal(rot.apply(frames), plain.apply(frames))


@pytest.mark.parametrize("mi", NAMES)
@pytest.mark.parametrize("mo", NAMES)
def test_rotated_map_all_model_pairs(acm, ctx, O, cameras, mi, mo):
    """10 degrees about a tilted axis: same NaN pattern and floor indices as the rotated oracle; bit-identical values
    where both models are arithmetic-only, within 1e-9 px otherwise."""
    ci, co = sized(cameras, mi, 320, 240), sized(cameras, mo, 288, 224)
    got = acm.remap_map(gpu_model(acm, ctx, ci), gpu_model(acm, ctx, co), rotation=ROT10)
    ref = RO.remap_map_rotated(oracle_model(O, ci), oracle_model(O, co), ROT10)
    assert got.shape == (224, 288, 2)
    assert np.array_equal(np.isnan(got), np.isnan(ref))
    ok = ~np.isnan(ref)
    assert ok.sum() > 0
    assert not np.array_equal(ref, R.remap_map(oracle_model(O, ci), oracle_model(O, co)), equal_nan=True)
    flips = int(np.sum(np.floor(got[ok]) != np.floor(ref[ok])))
    assert flips == 0, f"{flips} floor indices differ"
    if mi in EXACT and mo in EXACT:
        assert np.array_equal(got[ok], ref[ok])
    else:
        np.testing.assert_allclose(got[ok], ref[ok], rtol=0, atol=1e-9)


@pytest.mark.parametrize("idx", range(4))
def test_rotated_map_matches_opencv(acm, ctx, cameras, idx):
    """KB -> Pinhole (cv2.fisheye.initUndistortRectifyMap) and RadTan -> Pinhole (cv2.initUndistortRectifyMap) with R1:
    within 1e-3 px of OpenCV's float32 maps where both are valid and the rotated ray is in front of the input camera
    (OpenCV divides by z; the reference's KB uses atan2)."""
    g = load_golden("opencv_rectify.json")["maps"][idx]
    rc = g["rectified"]
    gi = gpu_model(acm, ctx, dict(cameras[g["camera"]]))
    rect = acm.PinholeModel(acm.Intrinsics(rc["f"], rc["f"], rc["cx"], rc["cy"]), acm.Resolution(rc["width"], rc["height"]), ctx=ctx)
    R1 = np.array(g["R1"])
    mp = acm.remap_map(gi, rect, rotation=R1)
    u, v = np.array(g["u"]), np.array(g["v"])
    got = mp[v, u]
    ref = np.stack([g["map_x"], g["map_y"]], axis=1)
    ray = np.stack([(u - rc["cx"]) / rc["f"], (v - rc["cy"]) / rc["f"], np.ones(len(u))], axis=1) @ R1  # R1^T ray_o
    use = ~np.isnan(got[:, 0]) & np.isfinite(ref).all(axis=1) & (ray[:, 2] > 0)
    assert use.sum() >= 100, use.sum()
    np.testing.assert_allclose(got[use], ref[use], rtol=0, atol=1e-3)


@pytest.mark.parametrize("mi,mo", [("kannala_brandt", "double_sphere"), ("eucm", "pinhole")])
@pytest.mark.parametrize("Wi,Hi,Wo,Ho,kernels", [(512, 384, 384, 288, 2),   # TMA + leftover gather
                                                 (756, 480, 640, 480, 1),   # whole-image gather
                                                 (37, 29, 64, 48, 1),       # byte kernel: input width
                                                 (512, 384, 302, 226, 1)])  # byte kernel: output width
def test_rotated_plan_dispatch_paths(acm, ctx, O, cameras, mi, mo, Wi, Hi, Wo, Ho, kernels):
    """A 25 degree rotation skews the source boxes past the TMA tile (the leftover gather takes them); 11 frames, both
    interpolations.  Bytes equal interpolate_pixel on the device map, and the rotated oracle's where the map is exact."""
    ci, co = sized(cameras, mi, Wi, Hi), sized(cameras, mo, Wo, Ho, 0.6)
    gi, go = gpu_model(acm, ctx, ci), gpu_model(acm, ctx, co)
    oi, oo = oracle_model(O, ci), oracle_model(O, co)
    F = 11
    frames = O.synth_bytes(0xACE5EC02, 0, F * Wi * Hi * 3).reshape(F, Hi, Wi, 3)
    mp = acm.remap_map(gi, go, rotation=ROT25)
    exact = mi in EXACT and mo in EXACT
    if exact:
        assert np.array_equal(mp, RO.remap_map_rotated(oi, oo, ROT25), equal_nan=True)
    for interp in (acm.InterpolationMethod.Bilinear, acm.InterpolationMethod.Nearest):
        with acm.RemapPlan(gi, go, None, interp, rotation=ROT25) as plan:
            d_in, d_out = ctx.device_alloc(frames.nbytes), ctx.device_alloc(F * Wo * Ho * 3)
            try:
                ctx.h2d(d_in, frames)
                n0 = launches(ctx)
                plan.apply_device(d_in, d_out, F)
                assert launches(ctx) - n0 == kernels
                out = np.empty((F, Ho, Wo, 3), np.uint8); ctx.d2h(out, d_out); ctx.sync()
            finally:
                ctx.device_free(d_in); ctx.device_free(d_out)
        assert out.any()
        for f in range(F):
            ref = R.remap_apply_map(mp, frames[f], int(interp))
            assert np.array_equal(out[f], ref), f"frame {f} interp {interp}: {(out[f] != ref).sum()} bytes differ"
            if exact and f in (0, F - 1):
                assert np.array_equal(out[f], RO.remap_rgb8_rotated(oi, oo, ROT25, frames[f], int(interp)))


def _rig(acm, ctx, cameras):
    """A KB left camera and a Double Sphere right camera 12 cm apart, 4 degrees of relative rotation."""
    left = gpu_model(acm, ctx, sized(cameras, "kannala_brandt", 512, 384))
    right = gpu_model(acm, ctx, sized(cameras, "double_sphere", 480, 360))
    Rm = axis_angle([0.1, 1.0, 0.2], 4.0)
    t = np.array([-0.12, 0.004, 0.003])
    rect = acm.PinholeModel(acm.Intrinsics(200.0, 200.0, 199.5, 149.5), acm.Resolution(400, 300), ctx=ctx)
    return left, right, Rm, t, rect


def test_stereo_rectifier_end_to_end(acm, ctx, O, cameras):
    """Known 3-D points placed at integer rectified pixels of both views: each plan's map returns its input camera's
    own projection of the point, and the rectified rows agree."""
    left, right, Rm, t, rect = _rig(acm, ctx, cameras)
    with acm.StereoRectifier(left, right, Rm, t, rect) as rig:
        assert not rig.vertical and rig.baseline < 0
        f, cx, cy = 200.0, 199.5, 149.5
        np.testing.assert_allclose(rig.P1, [[f, 0, cx, 0], [0, f, cy, 0], [0, 0, 1, 0]], rtol=0, atol=0)
        np.testing.assert_allclose(rig.P2, [[f, 0, cx, f * rig.baseline], [0, f, cy, 0], [0, 0, 1, 0]], rtol=0, atol=1e-12)
        map1 = acm.remap_map(left, rect, rotation=rig.R1)
        map2 = acm.remap_map(right, rect, rotation=rig.R2)
        ol, orr = oracle_model(O, sized(cameras, "kannala_brandt", 512, 384)), oracle_model(O, sized(cameras, "double_sphere", 480, 360))
        rng = np.random.default_rng(0xACE5EC03)
        checked = 0
        for _ in range(200):
            u, v, d = int(rng.integers(60, 340)), int(rng.integers(40, 260)), -int(rng.integers(2, 40))
            Z = f * rig.baseline / d                       # disparity u2 - u1 = f * baseline / Z = d pixels
            x_rect = np.array([(u - cx) / f * Z, (v - cy) / f * Z, Z])
            X1 = rig.R1.T @ x_rect
            X2 = Rm @ X1 + t
            if not (0 <= u + d < 400):
                continue
            st1, uv1 = O.project1(ol, X1)
            st2, uv2 = O.project1(orr, X2)
            if st1 != 0 or st2 != 0 or np.isnan(map1[v, u]).any() or np.isnan(map2[v, u + d]).any():
                continue
            np.testing.assert_allclose(map1[v, u], uv1, rtol=0, atol=1e-6)
            np.testing.assert_allclose(map2[v, u + d], uv2, rtol=0, atol=1e-6)
            checked += 1
        assert checked >= 100, checked
        frames_l = O.synth_bytes(0xACE5EC04, 0, 2 * 512 * 384 * 3).reshape(2, 384, 512, 3)
        frames_r = O.synth_bytes(0xACE5EC05, 0, 2 * 480 * 360 * 3).reshape(2, 360, 480, 3)
        out_l, out_r = rig.apply(frames_l, frames_r)
        assert out_l.shape == out_r.shape == (2, 300, 400, 3)
        for fi in range(2):
            assert np.array_equal(out_l[fi], R.remap_apply_map(map1, frames_l[fi]))
            assert np.array_equal(out_r[fi], R.remap_apply_map(map2, frames_r[fi]))


def test_rotated_plan_reuse(acm, ctx, O, cameras):
    """One rotated plan over two batches and frame by frame equals one batched call; a twin plan agrees."""
    left, _, _, _, rect = _rig(acm, ctx, cameras)
    frames = O.synth_bytes(0xACE5EC06, 0, 5 * 512 * 384 * 3).reshape(5, 384, 512, 3)
    with acm.RemapPlan(left, rect, rotation=ROT25) as plan, acm.RemapPlan(left, rect, rotation=ROT25) as twin:
        whole = plan.apply(frames)
        assert np.array_equal(np.concatenate([plan.apply(frames[:2]), plan.apply(frames[2:])]), whole)
        assert np.array_equal(np.stack([plan.apply(frames[f:f + 1])[0] for f in range(5)]), whole)
        assert np.array_equal(twin.apply(frames), whole)


def test_rotated_argument_errors(acm, ctx, cameras):
    from apex_camera_models_b200 import _native as N
    L = N.lib
    gi, go = gpu_model(acm, ctx, sized(cameras, "kannala_brandt", 64, 48)), gpu_model(acm, ctx, sized(cameras, "double_sphere", 64, 48))
    bi, bo = gi.camera_block(), go.camera_block()
    h = C.c_void_p()
    d = ctx.device_alloc(64 * 48 * 16)

    def fails(rc, text):
        assert rc == N.ERR_INVALID_ARG, rc
        assert text in L.acm_last_error(ctx.handle).decode()

    def rot(M):
        return (C.c_double * 9)(*np.ravel(M))

    try:
        for M, text in ((np.where(np.eye(3) == 1, np.nan, 0.0), "non-finite"), (np.diag([1.0, 1.0, np.inf]), "non-finite"),
                        (ROT10 * 1.0001, "not orthonormal"), (ROT10 + 1e-8, "not orthonormal"),
                        (np.diag([1.0, -1.0, 1.0]), "reflection"), (-ROT10, "reflection")):
            fails(L.acm_remap_plan_create_rotated(ctx.handle, C.byref(bi), C.byref(bo), rot(M), 1, C.byref(h)), text)
            assert not h.value
            fails(L.acm_remap_map_rotated(ctx.handle, C.byref(bi), C.byref(bo), rot(M), C.c_void_p(d)), text)
        fails(L.acm_remap_plan_create_rotated(ctx.handle, C.byref(bi), C.byref(bo), None, 1, C.byref(h)), "null rotation")
        fails(L.acm_remap_map_rotated(ctx.handle, C.byref(bi), C.byref(bo), None, C.c_void_p(d)), "null rotation")
        fails(L.acm_remap_plan_create_rotated(ctx.handle, C.byref(bi), None, rot(ROT10), 1, C.byref(h)), "needs an output camera")
        fails(L.acm_remap_map_rotated(ctx.handle, C.byref(bi), None, rot(ROT10), C.c_void_p(d)), "null output camera")
        fails(L.acm_remap_plan_create_rotated(ctx.handle, C.byref(bi), C.byref(bo), rot(ROT10), 2, C.byref(h)), "unknown interpolation")
        fails(L.acm_remap_map_rotated(ctx.handle, C.byref(bi), C.byref(bo), rot(ROT10), None), "null output")
        # 1e-10 off orthonormal is within the 1e-9 tolerance
        assert L.acm_remap_map_rotated(ctx.handle, C.byref(bi), C.byref(bo), rot(ROT10 * (1 + 1e-10)), C.c_void_p(d)) == N.OK
    finally:
        ctx.device_free(d)
    with pytest.raises(acm.AcmError, match="reflection"):
        acm.RemapPlan(gi, go, rotation=-np.eye(3))
    with pytest.raises(acm.UtilError, match="needs an output camera"):
        acm.RemapPlan(gi, None, rotation=np.eye(3))
    with pytest.raises(acm.UtilError, match="3x3"):
        acm.remap_map(gi, go, rotation=np.eye(4))
    with pytest.raises(acm.UtilError, match="PinholeModel"):
        acm.StereoRectifier(gi, go, np.eye(3), [-0.1, 0, 0], go)


def test_image_rectify_cli(acm, ctx, O, cameras, tmp_path):
    """Two small PNG pairs: output shapes and bytes equal the Python StereoRectifier's."""
    from PIL import Image

    from apex_camera_models_b200 import image_rectify as cli
    cl, cr = sized(cameras, "kannala_brandt", 320, 240), sized(cameras, "double_sphere", 256, 192)
    with open(tmp_path / "left.yaml", "w") as f:
        yaml.safe_dump({"cam0": {"camera_model": "kannala_brandt", "intrinsics": cl["params"][:4], "distortion": cl["params"][4:],
                                 "resolution": [320, 240]}}, f)
    with open(tmp_path / "right.yaml", "w") as f:
        yaml.safe_dump({"cam0": {"camera_model": "double_sphere", "intrinsics": cr["params"], "resolution": [256, 192]}}, f)
    for side, (W, H), seed in (("l", (320, 240), 0xACE5EC07), ("r", (256, 192), 0xACE5EC08)):
        (tmp_path / side).mkdir()
        for k in range(2):
            Image.fromarray(O.synth_bytes(seed, k * W * H * 3, W * H * 3).reshape(H, W, 3), "RGB").save(tmp_path / side / f"p{k}.png")
    Rm, t = axis_angle([0.1, 1.0, 0.2], 4.0), [-0.12, 0.004, 0.003]
    for interp, flag in ((acm.InterpolationMethod.Bilinear, []), (acm.InterpolationMethod.Nearest, ["--interpolation", "nearest"])):
        ol, orr = tmp_path / f"outl{int(interp)}", tmp_path / f"outr{int(interp)}"
        assert cli.main(["-l", str(tmp_path / "l"), "-r", str(tmp_path / "r"), "--left-calib", str(tmp_path / "left.yaml"),
                         "--left-model", "kb", "--right-calib", str(tmp_path / "right.yaml"), "--right-model", "ds",
                         "--rotation", *map(repr, Rm.ravel().tolist()), "--translation", *map(repr, t), "--size", "200", "150",
                         "--focal", "110", "--left-output", str(ol), "--right-output", str(orr)] + flag) == 0
        left = acm.KannalaBrandtModel.load_from_yaml(str(tmp_path / "left.yaml"), ctx=ctx)
        right = acm.DoubleSphereModel.load_from_yaml(str(tmp_path / "right.yaml"), ctx=ctx)
        rect = acm.PinholeModel(acm.Intrinsics(110.0, 110.0, 99.5, 74.5), acm.Resolution(200, 150), ctx=ctx)
        frames_l = np.stack([np.asarray(Image.open(tmp_path / "l" / f"p{k}.png").convert("RGB")) for k in range(2)])
        frames_r = np.stack([np.asarray(Image.open(tmp_path / "r" / f"p{k}.png").convert("RGB")) for k in range(2)])
        with acm.StereoRectifier(left, right, Rm, t, rect, interp) as rig:
            ref_l, ref_r = rig.apply(frames_l, frames_r)
        for k in range(2):
            got_l = np.asarray(Image.open(ol / f"p{k}.png").convert("RGB"))
            got_r = np.asarray(Image.open(orr / f"p{k}.png").convert("RGB"))
            assert got_l.shape == got_r.shape == (150, 200, 3)
            assert np.array_equal(got_l, ref_l[k]) and np.array_equal(got_r, ref_r[k])
