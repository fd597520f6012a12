"""The depth-image oracle (tests/depth_oracle.c) on the CPU: a closed-form pinhole case, an independent numpy z-buffer on
random clouds for all seven models, ties, the pixel-boundary rounding, points that must not be drawn, ranges beyond float32
and every status of the back-projection."""
import numpy as np
import pytest

import depth_oracle as D
from conftest import oracle_model

NAMES = ["pinhole", "rad_tan", "kannala_brandt", "ucm", "eucm", "double_sphere", "fov"]
EMPTY_RANGE_BITS = 0xFFFFFFFF
EMPTY_INDEX = 0xFFFFFFFF


def _axis_angle(axis, deg):
    a = np.asarray(axis, float) / np.linalg.norm(axis)
    K = np.array([[0, -a[2], a[1]], [a[2], 0, -a[0]], [-a[1], a[0], 0]])
    th = np.deg2rad(deg)
    return np.eye(3) + np.sin(th) * K + (1 - np.cos(th)) * K @ K


def _unit_pinhole(O, W=4, H=3):
    """fx = fy = 1, cx = cy = 0: u = x / z exactly, so pixel coordinates can be placed on any double."""
    return O.make_model(0, [1.0, 1.0, 0.0, 0.0], W, H)


def _empty(rng, idx):
    return (rng.view(np.uint32) == EMPTY_RANGE_BITS) & (idx == EMPTY_INDEX)


def _round_half_away(u):
    f, c = np.floor(u), np.ceil(u)
    return np.where(u >= 0, f + (u - f >= 0.5), c - (c - u >= 0.5))


def _numpy_zbuffer(m, xyz, R, t, uv):
    """Independent z-buffer from the oracle's per-point projections: lexsort on (pixel, f32 range, index), first per pixel."""
    x, y, z = xyz[:, 0], xyz[:, 1], xyz[:, 2]
    Q = [((R[i, 0] * x + R[i, 1] * y) + R[i, 2] * z) + t[i] for i in range(3)]
    with np.errstate(invalid="ignore", over="ignore"):
        rng = np.sqrt((Q[0] * Q[0] + Q[1] * Q[1]) + Q[2] * Q[2])
        rx, ry = _round_half_away(uv[:, 0]), _round_half_away(uv[:, 1])
        ok = (rx >= 0) & (rx < m.width) & (ry >= 0) & (ry < m.height) & (rng > 0) & np.isfinite(rng)
        r32 = rng.astype(np.float32)
    i = np.flatnonzero(ok)
    pix = (ry[i] * m.width + rx[i]).astype(np.int64)
    order = np.lexsort((i, r32[i], pix))
    pix, first = pix[order], i[order]
    keep = np.ones(len(pix), bool)
    keep[1:] = pix[1:] != pix[:-1]
    out_r = np.full(m.width * m.height, EMPTY_RANGE_BITS, np.uint32)
    out_i = np.full(m.width * m.height, EMPTY_INDEX, np.uint32)
    out_r[pix[keep]] = r32[first[keep]].view(np.uint32)
    out_i[pix[keep]] = first[keep]
    return out_r.reshape(m.height, m.width), out_i.reshape(m.height, m.width)


def test_closed_form_pinhole(O):
    m = O.make_model(0, [100.0, 100.0, 1.5, 1.5], 4, 3)
    pts = np.array([[0.0, 0.0, 1.0], [0.0, 0.0, 2.0], [0.01, 0.0, 1.0], [0.0, 0.0, -1.0]])
    rng, idx = D.render_depth(m, pts)
    # (0, 0, z) projects to (1.5, 1.5) -> pixel (2, 2), where the nearer point wins; x = 0.01 lands on (2.5, 1.5) -> (3, 2)
    assert idx[2, 2] == 0 and rng[2, 2] == np.float32(1.0)
    assert idx[2, 3] == 2 and rng[2, 3] == np.float32(np.sqrt(0.01 * 0.01 + 1.0))
    filled = np.zeros((3, 4), bool); filled[2, 2] = filled[2, 3] = True
    assert _empty(rng, idx)[~filled].all() and np.isnan(rng[~filled]).all()
    # back-projection of the drawn pixels: the ray through the pixel centre times the range
    xyz, st = D.depth_to_points(m, rng)
    assert (st[filled] == D.OK).all() and (st[~filled] == D.EMPTY).all()
    assert np.isnan(xyz[~filled]).all()
    np.testing.assert_allclose(xyz[2, 2], [0.005, 0.005, 1.0] / np.linalg.norm([0.005, 0.005, 1.0]), rtol=1e-15)
    d = float(rng[2, 3])
    np.testing.assert_allclose(xyz[2, 3], d * np.array([0.015, 0.005, 1.0]) / np.linalg.norm([0.015, 0.005, 1.0]), rtol=1e-15)


@pytest.mark.parametrize("name", NAMES)
@pytest.mark.parametrize("posed", [False, True])
def test_numpy_zbuffer_all_models(O, cameras, name, posed):
    """Random clouds, many points per pixel, duplicated points for ties: the oracle's images equal the numpy z-buffer."""
    cam = dict(cameras[name]); cam["width"], cam["height"] = 96, 64
    p = list(cam["params"]); s = 96 / cameras[name]["width"]
    p[0], p[1], p[2], p[3] = p[0] * s, p[1] * s, 47.7, 31.6
    cam["params"] = p
    m = oracle_model(O, cam)
    rs = np.random.default_rng(0xD3E7 + NAMES.index(name))
    n = 60_000
    d = rs.normal(size=(n, 3)); d /= np.linalg.norm(d, axis=1, keepdims=True)
    xyz = d * rs.uniform(0.5, 8.0, n)[:, None]
    xyz = np.vstack([xyz, xyz[rs.integers(0, n, 5_000)]])  # exact duplicates: equal ranges, the lower index must win
    R, t = (_axis_angle([0.3, -0.8, 0.5], 10.0), np.array([0.1, -0.05, 0.2])) if posed else (np.eye(3), np.zeros(3))
    rng, idx, uv = D.render_depth(m, xyz, R, t, want_uv=True)
    er, ei = _numpy_zbuffer(m, xyz, R, t, uv)
    assert np.array_equal(rng.view(np.uint32), er) and np.array_equal(idx, ei)
    assert (~_empty(rng, idx)).sum() > 500


def test_ties_go_to_the_lower_index(O):
    m = _unit_pinhole(O)
    # the same f32 range from different doubles (1 + 2^-40 rounds to 1.0f), listed high index first
    pts = np.array([[0.0, 0.0, 1.0 + 2.0 ** -40], [0.0, 0.0, 1.0], [0.0, 0.0, 1.0 + 2.0 ** -20], [0.0, 0.0, 1.0]])
    rng, idx = D.render_depth(m, pts)
    assert idx[0, 0] == 0 and rng[0, 0] == np.float32(1.0)
    rng, idx = D.render_depth(m, pts[1:])
    assert idx[0, 0] == 0  # pts[1] and pts[3] are equal; pts[2] is 1 + 2^-20 (a larger float)
    rng, idx = D.render_depth(m, pts[2:3])
    assert rng[0, 0] == np.float32(1.0 + 2.0 ** -20) and rng[0, 0] > np.float32(1.0)


def test_pixel_boundaries(O):
    """round() is half away from zero: u = W - 0.5 rounds to W (dropped), u = -0.5 to -1 (dropped), u = -0.49 to 0 (kept)."""
    m = _unit_pinhole(O, 4, 3)
    cases = [((3.5, 1.0), None), ((-0.5, 1.0), None), ((-0.49, 1.0), (0, 1)), ((3.49, 1.0), (3, 1)), ((2.5, 1.0), (3, 1)),
             ((1.0, 2.5), None), ((1.0, -0.5), None), ((1.0, -0.49), (1, 0)), ((1.0, 2.49), (1, 2))]
    for (u, v), pix in cases:
        rng, idx = D.render_depth(m, np.array([[u, v, 1.0]]))
        if pix is None:
            assert _empty(rng, idx).all(), (u, v)
        else:
            c, r = pix
            assert idx[r, c] == 0 and (~_empty(rng, idx)).sum() == 1, (u, v)


@pytest.mark.parametrize("name", ["pinhole", "kannala_brandt", "double_sphere"])
def test_points_not_drawn(O, cameras, name):
    """NaN coordinates, the camera centre and (for the pinhole) points behind the camera draw nothing."""
    m = oracle_model(O, cameras[name])
    bad = [[np.nan, 0.0, 1.0], [0.0, np.nan, 1.0], [0.0, 0.0, np.nan], [0.0, 0.0, 0.0], [np.inf, 0.0, 1.0]]
    if name == "pinhole":
        bad += [[0.0, 0.0, -1.0], [0.1, 0.2, -5.0], [0.0, 0.0, 1e-9]]
    rng, idx = D.render_depth(m, np.array(bad))
    assert _empty(rng, idx).all()


def test_f32_overflow_is_inf_and_last(O):
    m = _unit_pinhole(O)
    far, near, farther = [0.0, 0.0, 1e39], [0.0, 0.0, 1e30], [0.0, 0.0, 1e100]
    rng, idx = D.render_depth(m, np.array([far]))
    assert np.isposinf(rng[0, 0]) and idx[0, 0] == 0
    rng, idx = D.render_depth(m, np.array([far, farther, near]))
    assert idx[0, 0] == 2 and rng[0, 0] == np.float32(1e30)
    rng, idx = D.render_depth(m, np.array([farther, far]))
    assert idx[0, 0] == 0 and np.isposinf(rng[0, 0])  # both inf in f32: the lower index
    # a range that overflows f64 (x*x = inf) is not finite: not drawn
    rng, idx = D.render_depth(m, np.array([[0.0, 0.0, 1e200]]))
    assert _empty(rng, idx).all()


def test_depth_to_points_statuses(O, cameras):
    m = _unit_pinhole(O, 4, 3)
    r = np.array([[1.0, 0.0, -1.0, np.nan], [np.inf, -np.inf, 2.0, 1e-30], [np.float32(3.4e38), 5e-45, 0.5, -0.0]], np.float32)
    xyz, st = D.depth_to_points(m, r)
    ok = np.array([[1, 0, 0, 0], [0, 0, 1, 1], [1, 1, 1, 0]], bool)
    assert np.array_equal(st == D.OK, ok) and (st[~ok] == D.EMPTY).all()
    assert np.isnan(xyz[~ok]).all() and np.isfinite(xyz[ok]).all()
    # |x| equals the range (unit rays)
    np.testing.assert_allclose(np.linalg.norm(xyz[ok], axis=1), r[ok].astype(np.float64), rtol=1e-15)
    # the UCM sample camera: pixels outside its unproject domain are UNPROJECT
    cam = dict(cameras["ucm"])
    mu = oracle_model(O, cam)
    r = np.full((mu.height, mu.width), 2.0, np.float32)
    _, st = D.depth_to_points(mu, r)
    assert set(np.unique(st).tolist()) <= {D.OK, D.UNPROJECT}
    ref_ok = np.array([O.unproject1(mu, (c, rr))[0] == 0 for rr in (0, mu.height - 1) for c in (0, mu.width - 1)])
    assert np.array_equal(st[[0, 0, -1, -1], [0, -1, 0, -1]] == D.OK, ref_ok)


def test_render_then_back_project_posed(O, cameras):
    """A posed render followed by the back-projection with the same R, t lands every drawn pixel's point on a ray through
    the pixel centre at the f32 range from the camera centre -t R (world frame)."""
    m = oracle_model(O, cameras["double_sphere"])
    R, t = _axis_angle([0.1, 1.0, -0.3], 25.0), np.array([0.3, -0.2, 0.1])
    rs = np.random.default_rng(0xD3E8)
    d = rs.normal(size=(50_000, 3)); d /= np.linalg.norm(d, axis=1, keepdims=True)
    xyz = d * rs.uniform(1.0, 4.0, len(d))[:, None]
    rng, idx = D.render_depth(m, xyz, R, t)
    back, st = D.depth_to_points(m, rng, R, t)
    drawn = ~_empty(rng, idx)
    assert drawn.sum() > 1000 and (st[drawn] == D.OK).all() and (st[~drawn] == D.EMPTY).all()
    cam_pts = back[drawn] @ R.T + t
    np.testing.assert_allclose(np.linalg.norm(cam_pts, axis=1), rng[drawn].astype(np.float64), rtol=1e-12)
