"""The triangulation oracle (tests/triangulate_oracle.c) on the CPU: closed-form pinhole cases, OpenCV's triangulatePoints
frozen in tests/golden/opencv_triangulate.json, the refined points against scipy.optimize.least_squares on the same
residual, and one constructed pair for every status value."""
import numpy as np
import pytest
from scipy.optimize import least_squares

import triangulate_oracle as T
from conftest import load_golden, oracle_model


def axis_angle(axis, deg):
    k = np.asarray(axis, np.float64) / np.linalg.norm(axis)
    K = np.array([[0.0, -k[2], k[1]], [k[2], 0.0, -k[0]], [-k[1], k[0], 0.0]])
    a = np.deg2rad(deg)
    return np.eye(3) + np.sin(a) * K + (1.0 - np.cos(a)) * (K @ K)


def pinhole(O, f=400.0, W=640, H=480):
    return O.make_model(0, [f, f, W / 2.0, H / 2.0], W, H)


@pytest.mark.parametrize("max_iterations", [0, 10])
def test_closed_form_pinhole(O, max_iterations):
    """Rectified pinhole pair, x_cam2 = x_cam1 - b e_x: Z = f b / (u1 - u2), X = (u1 - cx) Z / f, Y = (v - cy) Z / f."""
    m = pinhole(O)
    f, b = 400.0, 0.25
    u1 = np.array([320.0, 100.5, 600.25, 330.0, 12.0])
    v = np.array([240.0, 17.0, 470.5, 250.0, 300.0])
    d = np.array([10.0, 40.0, 3.5, 100.0, 1.0])
    xyz, err, st = T.triangulate(m, m, np.eye(3), [-b, 0.0, 0.0], np.column_stack([u1, v]), np.column_stack([u1 - d, v]), max_iterations)
    assert st.tolist() == [T.OK] * 5
    Z = f * b / d
    ref = np.column_stack([(u1 - 320.0) * Z / f, (v - 240.0) * Z / f, Z])
    # the midpoint divides by 1 - b^2 ~ (disparity / f)^2 = 6e-6 at d = 1 px, which a rounding of b moves by ~1e-10 relative;
    # there the depth moves the pixels by ~1e-10 px only, below what a refinement step can resolve
    np.testing.assert_allclose(xyz, ref, rtol=1e-9, atol=1e-12)
    assert np.all(err <= 1e-9)


@pytest.mark.parametrize("idx", range(3))
def test_matches_opencv(O, cameras, idx):
    """Noise-free pairs of the Pinhole, RadTan and Kannala-Brandt sample cameras: the refined points equal OpenCV's
    triangulatePoints (after undistortPoints / fisheye.undistortPoints) to 1e-6 relative; so does the Pinhole midpoint."""
    g = load_golden("opencv_triangulate.json")
    c = g["cases"][idx]
    m = oracle_model(O, cameras[c["camera"]])
    ref = np.array(c["points_opencv"])
    modes = (0, 10) if c["camera"] == "pinhole" else (10,)
    for it in modes:
        xyz, err, st = T.triangulate(m, m, g["R"], g["t"], c["uv1"], c["uv2"], it)
        assert np.all(st == T.OK)
        np.testing.assert_allclose(xyz, ref, rtol=1e-6, atol=0)
        assert np.all(err < 1e-6)


def _rig_pairs(O, ma, mb, R, t, n, seed, sigma):
    """Ground-truth points 0.5-5 units along rays of random first-camera pixels, their projections into both cameras with
    N(0, sigma) pixel noise; only pairs that both cameras see."""
    rng = np.random.default_rng(seed)
    uv = np.column_stack([rng.uniform(0, ma.width, 2 * n), rng.uniform(0, ma.height, 2 * n)])
    ray, st = O.unproject(ma, uv)
    X = ray * rng.uniform(0.5, 5.0, 2 * n)[:, None]
    uv1, s1 = O.project(ma, X)
    uv2, s2 = O.project(mb, X @ np.asarray(R).T + t)
    ok = (st == 0) & (s1 == 0) & (s2 == 0)
    uv1, uv2, X = uv1[ok][:n], uv2[ok][:n], X[ok][:n]
    assert len(X) == n
    return uv1 + rng.normal(0, sigma, uv1.shape), uv2 + rng.normal(0, sigma, uv2.shape), X


@pytest.mark.parametrize("pair", [("pinhole", "pinhole"), ("kannala_brandt", "double_sphere"), ("rad_tan", "fov")])
def test_refined_matches_scipy(O, cameras, pair):
    """2 000 noisy pairs (sigma = 0.5 px): the oracle's refined points equal scipy's least_squares minimiser of the same
    four residuals from the same start (the midpoint; analytic Jacobian, tolerances 1e-15), and never cost more than the
    midpoint.  Both end where the cost stops changing in f64: the costs agree to 1e-12 relative.  Along the depth of a far
    point the cost is so flat there that the two minimisers may still sit a few 1e-7 apart in space (scipy's xtol stop
    leaves its gradient at up to ~1e-5), so 1e-8 relative holds for 90 % of the points and 1e-6 for all."""
    from test_gpu_remap import sized
    ca, cb = sized(cameras, pair[0], 320, 240), sized(cameras, pair[1], 288, 224)
    ma, mb = oracle_model(O, ca), oracle_model(O, cb)
    R, t = axis_angle([0.3, -0.8, 0.5], 10.0), np.array([-0.1, 0.0, 0.0])
    uv1, uv2, _ = _rig_pairs(O, ma, mb, R, t, 2000, 0x7121A7E1, 0.5)
    xm, em, sm = T.triangulate(ma, mb, R, t, uv1, uv2, 0)
    xr, er, sr = T.triangulate(ma, mb, R, t, uv1, uv2, 10)
    assert np.array_equal(sm, sr)
    ok = np.flatnonzero(sr == T.OK)
    assert len(ok) > 1900
    assert np.all((er[ok] ** 2).sum(1) <= (em[ok] ** 2).sum(1))

    def jac(X, a, b):
        _, _, J1 = O.project_point_jacobian1(ma, X)
        _, _, J2 = O.project_point_jacobian1(mb, R @ X + t)
        return np.vstack([J1, J2 @ R])

    rel = []
    for i in ok:
        a, b = uv1[i], uv2[i]
        fun = lambda X: T.residuals(ma, mb, R, t, a, b, X)
        sol = least_squares(fun, xm[i], jac=lambda X: jac(X, a, b), method="lm", xtol=1e-15, ftol=1e-15, gtol=1e-15)
        c_ours, c_scipy = (fun(xr[i]) ** 2).sum(), (fun(sol.x) ** 2).sum()
        assert abs(c_ours - c_scipy) <= 1e-12 * c_scipy + 1e-14, (i, c_ours, c_scipy)
        rel.append(np.abs(sol.x - xr[i]).max() / np.abs(sol.x).max())
    rel = np.array(rel)
    assert rel.max() <= 1e-6, rel.max()
    assert np.mean(rel <= 1e-8) >= 0.9, np.sort(rel)[-30:]


def test_every_status(O, cameras):
    """One constructed pair per status value, in both modes."""
    m = pinhole(O)
    I3 = np.eye(3)
    cases = [
        (I3, [-0.2, 0.0, 0.0], (340.0, 250.0), (330.0, 250.0), T.OK),
        (I3, [-0.2, 0.0, 0.0], (640.0, 250.0), (330.0, 250.0), T.UNPROJECT_FIRST),     # u = W is outside [0, W)
        (I3, [-0.2, 0.0, 0.0], (340.0, 250.0), (330.0, 480.0), T.UNPROJECT_SECOND),    # v = H
        (I3, [0.0, 0.0, 0.3], (320.0, 240.0), (320.0, 240.0), T.PARALLEL),             # both rays on the common axis
        (I3, [-0.2, 0.0, 0.0], (300.0, 240.0), (340.0, 240.0), T.BEHIND),              # rays diverge: negative disparity
    ]
    for it in (0, 10):
        for R, t, a, b, want in cases:
            xyz, err, st = T.triangulate(m, m, R, t, [a], [b], it)
            assert st[0] == want, (a, b, st[0], want)
            assert np.isnan(xyz[0]).all() == (want != T.OK) and np.isnan(err[0]).all() == (want != T.OK)
    # PROJECT: the 10 degree rig of the other tests; the first of 20 000 seeded random pixel pairs whose midpoint has both ray
    # parameters positive but lies behind one of the cameras (the rays pass each other far apart)
    R, t = axis_angle([0.3, -0.8, 0.5], 10.0), np.array([-0.1, 0.0, 0.0])
    rng = np.random.default_rng(0x7121A7E2)
    uv1 = np.column_stack([rng.uniform(0, 640, 20000), rng.uniform(0, 480, 20000)])
    uv2 = np.column_stack([rng.uniform(0, 640, 20000), rng.uniform(0, 480, 20000)])
    _, _, st = T.triangulate(m, m, R, t, uv1, uv2, 0)
    hits = np.flatnonzero(st == T.PROJECT)
    assert len(hits) > 0
    i = hits[0]
    d1 = np.array([(uv1[i, 0] - 320.0) / 400.0, (uv1[i, 1] - 240.0) / 400.0, 1.0])
    d2 = R.T @ np.array([(uv2[i, 0] - 320.0) / 400.0, (uv2[i, 1] - 240.0) / 400.0, 1.0])
    c2 = -R.T @ t
    s1, s2 = np.linalg.lstsq(np.column_stack([d1, -d2]), c2, rcond=None)[0]
    X = 0.5 * (s1 * d1 + c2 + s2 * d2)
    assert s1 > 0 and s2 > 0 and min(X[2], (R @ X + t)[2]) < 1.5e-8
    for it in (0, 10):
        xyz, err, st1 = T.triangulate(m, m, R, t, uv1[i:i + 1], uv2[i:i + 1], it)
        assert st1[0] == T.PROJECT and np.isnan(xyz).all() and np.isnan(err).all()
