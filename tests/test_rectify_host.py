"""Stereo rectification on the host (acm_stereo_rectify, no device): R1 / R2 against OpenCV's stereoRectify frozen in
tests/golden/opencv_rectify.json, the properties that make rectified rows correspond, argument errors, the C++ wrapper,
and the rotated remap oracle (tests/rectify_oracle.c) that the GPU tests compare against."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import rectify_oracle as RO
import remap_oracle as R
from conftest import load_golden, oracle_model

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = load_golden("opencv_rectify.json")
CASES = {c["name"]: c for c in GOLD["cases"]}


@pytest.fixture(scope="module")
def acm():
    import apex_camera_models_b200 as m
    return m


def rectify(acm, case):
    return acm.stereo_rectify(np.array(case["R"]), np.array(case["t"]))


@pytest.mark.parametrize("name", sorted(CASES))
def test_rectify_matches_opencv(acm, name):
    """Above 1e-4 rad OpenCV's Rodrigues is exact enough to be the reference; below it, OpenCV returns a zero rotation
    vector (sin < 1e-5) and the frozen exact-math restatement is, with OpenCV within twice the angle."""
    c = CASES[name]
    R1, R2, baseline, vertical = rectify(acm, c)
    assert vertical == bool(c["vertical"])
    if c["angle"] > 1e-4 or c["angle"] == 0.0:
        np.testing.assert_allclose(R1, c["cv2_R1"], rtol=0, atol=1e-12)
        np.testing.assert_allclose(R2, c["cv2_R2"], rtol=0, atol=1e-12)
        assert abs(baseline - c["cv2_baseline"]) <= 1e-12 * np.linalg.norm(c["t"])
    else:
        np.testing.assert_allclose(R1, c["exact_R1"], rtol=0, atol=1e-12)
        np.testing.assert_allclose(R2, c["exact_R2"], rtol=0, atol=1e-12)
        assert np.abs(R1 - c["cv2_R1"]).max() <= 2 * c["angle"]
        assert np.abs(R2 - c["cv2_R2"]).max() <= 2 * c["angle"]
    assert abs(baseline - c["exact_baseline"]) <= 1e-12 * np.linalg.norm(c["t"])


@pytest.mark.parametrize("name", sorted(CASES))
def test_rectify_properties(acm, name):
    c = CASES[name]
    Rm, t = np.array(c["R"]), np.array(c["t"])
    R1, R2, baseline, vertical = rectify(acm, c)
    for M in (R1, R2):
        assert np.abs(M @ M.T - np.eye(3)).max() <= 1e-13
        assert abs(np.linalg.det(M) - 1.0) <= 1e-13
    assert np.abs(R1 - R2 @ Rm).max() <= 1e-13
    t2 = R2 @ t
    axis = 1 if vertical else 0
    off = np.delete(t2, axis)
    assert np.abs(off).max() <= 1e-12 * np.linalg.norm(t)
    assert abs(baseline - t2[axis]) <= 1e-15 * np.linalg.norm(t)


@pytest.mark.parametrize("name", sorted(CASES))
def test_rectified_rows_correspond(acm, name):
    """10^4 points in front of both cameras: the shared rectified pinhole puts each point on the same row (column for a
    vertical pair) in both views, and the disparity is -f * baseline / Z_rect."""
    c = CASES[name]
    Rm, t = np.array(c["R"]), np.array(c["t"])
    R1, R2, baseline, vertical = rectify(acm, c)
    f, cx, cy = 400.0, 320.0, 240.0
    rng = np.random.default_rng(0xACE5EC8)
    Xr = np.stack([rng.uniform(-2, 2, 10**4), rng.uniform(-2, 2, 10**4), rng.uniform(1.0, 20.0, 10**4)], axis=1)
    X1 = Xr @ R1   # camera-1 coordinates of points at known rectified positions: X1 = R1^T x_rect
    x1 = X1 @ R1.T
    x2 = (X1 @ Rm.T + t) @ R2.T
    u1, v1 = f * x1[:, 0] / x1[:, 2] + cx, f * x1[:, 1] / x1[:, 2] + cy
    u2, v2 = f * x2[:, 0] / x2[:, 2] + cx, f * x2[:, 1] / x2[:, 2] + cy
    same, disp = (u1 - u2, v1 - v2) if vertical else (v1 - v2, u1 - u2)
    assert np.abs(same).max() <= 1e-9
    np.testing.assert_allclose(disp, -f * baseline / x1[:, 2], rtol=1e-9, atol=0)


def test_rectify_argument_errors(acm):
    from apex_camera_models_b200 import _native as N
    L = N.lib
    good_R, good_t = np.array(CASES["horizontal_negative_baseline"]["R"]), np.array([-0.12, 0.003, 0.002])
    bad = [(np.where(np.eye(3) == 1, np.nan, 0.0), good_t, "non-finite"),
           (good_R, np.array([np.nan, 0.0, 0.0]), "non-finite"),
           (good_R, np.array([np.inf, 0.0, 0.0]), "non-finite"),
           (good_R, np.zeros(3), "translation is zero"),
           (good_R * 1.001, good_t, "not orthonormal"),
           (good_R + 1e-8, good_t, "not orthonormal"),
           (np.diag([1.0, 1.0, -1.0]), good_t, "reflection"),
           (-np.eye(3), good_t, "reflection")]
    for Rm, t, text in bad:
        with pytest.raises(acm.AcmError, match=text):
            acm.stereo_rectify(Rm, t)
    out = [(C.c_double * 9)(), (C.c_double * 9)(), C.c_double(), C.c_int32()]
    Rc, tc = (C.c_double * 9)(*good_R.ravel()), (C.c_double * 3)(*good_t)
    assert L.acm_stereo_rectify(None, tc, out[0], out[1], C.byref(out[2]), C.byref(out[3])) == N.ERR_INVALID_ARG
    assert "null rotation" in L.acm_last_error(None).decode()
    assert L.acm_stereo_rectify(Rc, None, out[0], out[1], C.byref(out[2]), C.byref(out[3])) == N.ERR_INVALID_ARG
    assert L.acm_stereo_rectify(Rc, tc, out[0], None, C.byref(out[2]), C.byref(out[3])) == N.ERR_INVALID_ARG
    assert L.acm_stereo_rectify(Rc, tc, out[0], out[1], C.byref(out[2]), C.byref(out[3])) == N.OK
    with pytest.raises(acm.UtilError, match="3x3"):
        acm.stereo_rectify(np.eye(2), good_t)
    with pytest.raises(acm.UtilError, match="3 entries"):
        acm.stereo_rectify(good_R, [1.0, 0.0])


def test_cpp_stereo_rectify(tmp_path):
    """include/acm.hpp's stereo_rectify compiles, links libacm.so and runs (host only)."""
    exe = str(tmp_path / "rectify_test")
    libdir = os.path.join(ROOT, "apex_camera_models_b200", "lib")
    subprocess.run(["/usr/bin/g++", "-std=c++17", "-O1", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"),
                    os.path.join(ROOT, "tests", "cpp", "rectify_test.cpp"), "-o", exe, "-L", libdir, "-lacm", f"-Wl,-rpath,{libdir}"],
                   check=True)
    for name in ("horizontal_large_rotation", "vertical_positive_baseline"):
        c = CASES[name]
        r = subprocess.run([exe] + [repr(float(v)) for v in np.ravel(c["R"])] + [repr(float(v)) for v in c["t"]], capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
        assert "RECTIFY_TEST_OK" in r.stdout
        vals = [float(v) for v in r.stdout.split()[:19]]
        np.testing.assert_allclose(np.reshape(vals[:9], (3, 3)), c["cv2_R1"], rtol=0, atol=1e-12)
        np.testing.assert_allclose(np.reshape(vals[9:18], (3, 3)), c["cv2_R2"], rtol=0, atol=1e-12)
        assert int(r.stdout.split()[19]) == c["vertical"]


def test_rotated_oracle_identity_and_pinhole_homography(O, cameras):
    """The rotated oracle with R = I is the remap oracle bit for bit; pinhole to pinhole with a rotation is the
    homography K_in R^T K_out^-1."""
    ci, co = dict(cameras["kannala_brandt"]), dict(cameras["double_sphere"])
    mi, mo = oracle_model(O, ci), oracle_model(O, co)
    assert np.array_equal(RO.remap_map_rotated(mi, mo, np.eye(3)), R.remap_map(mi, mo), equal_nan=True)
    Rm = np.array(CASES["horizontal_large_rotation"]["R"])
    pi = {"model_id": 0, "width": 320, "height": 240, "params": [300.0, 310.0, 160.5, 119.5]}
    po = {"model_id": 0, "width": 200, "height": 150, "params": [150.0, 150.0, 100.0, 75.0]}
    got = RO.remap_map_rotated(oracle_model(O, pi), oracle_model(O, po), Rm)
    Ki = np.array([[300.0, 0, 160.5], [0, 310.0, 119.5], [0, 0, 1]])
    Ko = np.array([[150.0, 0, 100.0], [0, 150.0, 75.0], [0, 0, 1]])
    v, u = np.mgrid[0:150, 0:200]
    h = np.stack([u, v, np.ones_like(u)], -1).astype(float) @ (Ki @ Rm.T @ np.linalg.inv(Ko)).T
    front = h[..., 2] > 1e-3
    ok = ~np.isnan(got[..., 0])
    assert ok.sum() > 1000 and np.array_equal(ok & ~front, np.zeros_like(ok))
    np.testing.assert_allclose(got[ok], (h[..., :2] / h[..., 2:])[ok], rtol=0, atol=1e-9)


def test_cli_module_does_not_shadow_stereo_rectify(acm):
    """The CLI lives in its own module name: importing it leaves the package's stereo_rectify function in place."""
    import importlib
    cli = importlib.import_module("apex_camera_models_b200.image_rectify")
    assert callable(cli.main)
    assert callable(acm.stereo_rectify) and acm.stereo_rectify.__module__ == "apex_camera_models_b200.util"
    R1, _, _, _ = acm.stereo_rectify(np.eye(3), [-0.1, 0.0, 0.0])
    assert np.array_equal(R1, np.eye(3))
