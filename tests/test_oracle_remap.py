"""CPU oracle of the camera-to-camera remap (tests/remap_oracle.c): closed-form cases, and its ties to the pinned
undistort oracle."""
import numpy as np
import pytest

import remap_oracle as R
from conftest import oracle_model


def pinhole(O, fx, fy, cx, cy, W, H):
    return O.make_model(O.PINHOLE, [fx, fy, cx, cy], W, H)


def test_same_pinhole_in_and_out_is_identity(O):
    W, H = 64, 48
    m = pinhole(O, 64.0, 64.0, 32.0, 24.0, W, H)
    mp = R.remap_map(m, m)
    u, v = np.meshgrid(np.arange(W, dtype=np.float64), np.arange(H, dtype=np.float64))
    ok = ~np.isnan(mp[..., 0])
    # the round trip through the normalised ray may land a rounding error below 0 in the first row or column
    assert ok[1:, 1:].all() and ok.sum() >= W * H - 8
    np.testing.assert_allclose(mp[..., 0][ok], u[ok], rtol=0, atol=1e-12)
    np.testing.assert_allclose(mp[..., 1][ok], v[ok], rtol=0, atol=1e-12)
    img = O.synth_bytes(0xACE50101, 0, W * H * 3).reshape(H, W, 3)
    near = R.remap_rgb8(m, m, img, 0)
    assert np.array_equal(near[ok], img[ok])
    bil = R.remap_rgb8(m, m, img, 1)
    # x0 + 1 >= W (y0 + 1 >= H) has no bilinear sample: the last column and row stay black
    assert not bil[-1].any() and not bil[:, -1].any()
    assert np.array_equal(bil[1:-1, 1:-1], img[1:-1, 1:-1])


def test_half_focal_length_output_is_affine(O):
    W, H = 80, 60
    fx, fy, cx, cy = 70.0, 66.0, 40.5, 29.25
    mi, mo = pinhole(O, fx, fy, cx, cy, W, H), pinhole(O, fx / 2, fy / 2, cx, cy, W, H)
    mp = R.remap_map(mi, mo)
    u, v = np.meshgrid(np.arange(W, dtype=np.float64), np.arange(H, dtype=np.float64))
    ex, ey = 2.0 * u - cx, 2.0 * v - cy  # src = fx * (u - cx) / (fx / 2) + cx
    inside = (ex >= 0) & (ex < W) & (ey >= 0) & (ey < H)
    edge = (np.abs(ex) < 1e-9) | (np.abs(ex - W) < 1e-9) | (np.abs(ey) < 1e-9) | (np.abs(ey - H) < 1e-9)
    ok = ~np.isnan(mp[..., 0])
    assert np.array_equal(ok[~edge], inside[~edge])
    np.testing.assert_allclose(mp[..., 0][ok], ex[ok], rtol=0, atol=1e-9)
    np.testing.assert_allclose(mp[..., 1][ok], ey[ok], rtol=0, atol=1e-9)


@pytest.mark.parametrize("name", ["kannala_brandt", "double_sphere", "rad_tan", "fov"])
@pytest.mark.parametrize("interp", [0, 1])
def test_apply_map_of_undistort_map_equals_undistort(O, cameras, name, interp):
    """Ties interpolate_pixel of the remap oracle to the one behind the pinned orc_undistort_rgb8."""
    cam = dict(cameras[name]); cam["width"], cam["height"] = 96, 64
    p = list(cam["params"]); p[2], p[3] = 47.3, 31.9; cam["params"] = p
    om = oracle_model(O, cam)
    img = O.synth_bytes(0xACE50102, 0, 96 * 64 * 3).reshape(64, 96, 3)
    for t in (p[:4], [p[0] * 0.6, p[1] * 0.6, 48.0, 32.0]):
        got = R.remap_apply_map(O.undistort_map(om, t), img, interp)
        assert np.array_equal(got, O.undistort_rgb8(om, t, img, interp))


@pytest.mark.parametrize("name", ["kannala_brandt", "double_sphere", "rad_tan", "ucm", "eucm", "fov", "pinhole"])
def test_pinhole_output_agrees_with_undistort_map(O, cameras, name):
    """A pinhole output camera is undistort_image's target: the maps agree to 1e-12 px (not bit for bit: the remap's
    ray is normalised)."""
    cam = cameras[name]
    W, H = 120, 90
    c = dict(cam); c["width"], c["height"] = W, H
    p = list(c["params"]); p[2], p[3] = W / 2 + 0.3, H / 2 - 0.2; c["params"] = p
    om = oracle_model(O, c)
    t = [p[0] * 0.8, p[1] * 0.8, W / 2, H / 2]
    ref = O.undistort_map(om, t)
    got = R.remap_map(om, pinhole(O, *t, W, H))
    both = ~np.isnan(ref[..., 0]) & ~np.isnan(got[..., 0])
    assert both.sum() > 0.5 * W * H
    # the validity differs at most where the projection lands within rounding of the image border
    differ = np.isnan(ref[..., 0]) != np.isnan(got[..., 0])
    assert differ.sum() <= 2, differ.sum()
    np.testing.assert_allclose(got[both], ref[both], rtol=0, atol=1e-12)
