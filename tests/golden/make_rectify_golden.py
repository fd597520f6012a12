"""Generate tests/golden/opencv_rectify.json: stereo rectification frozen from OpenCV, for tests that do not import cv2.

  * cases: (R, t) pairs with OpenCV's `stereoRectify` R1 / R2 (and `fisheye.stereoRectify` for horizontal pairs, where
    the two agree) and a float64 numpy restatement of the same algorithm with exact Rodrigues conversions.  OpenCV's
    Rodrigues returns a zero vector below sin(angle) = 1e-5, so below that the restatement is the reference and OpenCV
    is only an anchor within the angle.
  * maps: `fisheye.initUndistortRectifyMap` of the Kannala-Brandt sample camera and `initUndistortRectifyMap` of the
    RadTan sample camera with a case's R1 and a chosen rectified pinhole P, as float32 maps at sampled output pixels.

Run here (no GPU needed):  python tests/golden/make_rectify_golden.py
"""
import json
import os

import cv2
import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
cams = json.load(open(os.path.join(HERE, "cameras.json")))


def rodrigues_matrix(w):
    """Vector -> matrix: cos t I + (1 - cos t)/t^2 w w^T + sin t/t [w]x, 1 - cos t = 2 sin^2(t/2)."""
    w = np.asarray(w, np.float64)
    t = np.sqrt(w @ w)
    a, b, c = 1.0, 0.5, 1.0
    if t > 0:
        h = np.sin(0.5 * t) / t
        a, b, c = np.sin(t) / t, 2.0 * h * h, np.cos(t)
    K = np.array([[0.0, -w[2], w[1]], [w[2], 0.0, -w[0]], [-w[1], w[0], 0.0]])
    return c * np.eye(3) + b * np.outer(w, w) + a * K


def rodrigues_vector(R):
    """Matrix -> vector without a small-angle cut-off; the symmetric part gives the axis beyond 90 degrees."""
    s = 0.5 * np.array([R[2, 1] - R[1, 2], R[0, 2] - R[2, 0], R[1, 0] - R[0, 1]])
    sn = np.sqrt(s @ s)
    c = 0.5 * (np.trace(R) - 1.0)
    t = np.arctan2(sn, c)
    if c >= 0:
        return s * (t / sn if sn > 0 else 1.0)
    i = int(np.argmax(np.diag(R)))
    d = 1.0 - c
    k = np.empty(3)
    k[i] = np.sqrt(max((R[i, i] - c) / d, 0.0))
    for j in range(3):
        if j != i:
            k[j] = 0.5 * (R[i, j] + R[j, i]) / (d * k[i])
    return (-1.0 if k @ s < 0 else 1.0) * t * k


def stereo_rectify(R, t):
    """The rotation part of OpenCV's cvStereoRectify with exact Rodrigues conversions."""
    r_r = rodrigues_matrix(-0.5 * rodrigues_vector(R))
    tp = r_r @ t
    idx = 0 if abs(tp[0]) > abs(tp[1]) else 1
    c, nt = tp[idx], np.sqrt(tp @ tp)
    uu = np.zeros(3)
    uu[idx] = 1.0 if c > 0 else -1.0
    ww = np.cross(tp, uu)
    nw = np.sqrt(ww @ ww)
    if nw > 0:
        ww = ww * (np.arccos(min(abs(c) / nt, 1.0)) / nw)
    wR = rodrigues_matrix(ww)
    R2 = wR @ r_r
    return wR @ r_r.T, R2, float((R2 @ t)[idx]), idx


def axis_angle(axis, deg):
    a = np.asarray(axis, np.float64)
    return rodrigues_matrix(a / np.linalg.norm(a) * np.deg2rad(deg))


CASES = [
    ("horizontal_negative_baseline", axis_angle([0.2, 1.0, 0.1], 2.0), [-0.12, 0.003, 0.002]),
    ("horizontal_positive_baseline", axis_angle([-0.4, 0.3, 1.0], 3.0), [0.11, -0.004, 0.006]),
    ("horizontal_large_rotation", axis_angle([0.3, -1.0, 0.5], 30.0), [-0.3, 0.1, 0.05]),
    ("vertical_negative_baseline", axis_angle([1.0, 0.2, -0.3], 1.5), [0.004, -0.10, 0.003]),
    ("vertical_positive_baseline", axis_angle([0.1, 0.1, 1.0], 4.0), [-0.01, 0.2, 0.01]),
    ("identity_rotation", np.eye(3), [-0.1, 0.0, 0.0]),
    ("rotation_2e-4_rad", axis_angle([0.6, -0.8, 0.1], np.rad2deg(2e-4)), [-0.1, 0.002, -0.001]),
    ("rotation_5e-6_rad", axis_angle([0.6, -0.8, 0.1], np.rad2deg(5e-6)), [-0.1, 0.002, -0.001]),
    ("rotation_1e-9_rad", axis_angle([0.2, 0.5, -0.9], np.rad2deg(1e-9)), [-0.1, 0.001, 0.0]),
    ("rotation_170_deg", axis_angle([0.3, 0.9, 0.2], 170.0), [0.2, -0.05, 0.1]),
    ("rotation_120_deg_vertical", axis_angle([1.0, -0.2, 0.4], 120.0), [0.05, 0.3, -0.02]),
]


def cases():
    K = np.array([[400.0, 0, 320.0], [0, 400.0, 240.0], [0, 0, 1.0]])
    out = []
    for name, R, t in CASES:
        t = np.asarray(t, np.float64)
        R1, R2, P1, P2, _, _, _ = cv2.stereoRectify(K, np.zeros(5), K, np.zeros(5), (640, 480), R, t, alpha=-1)
        eR1, eR2, baseline, idx = stereo_rectify(R, t)
        angle = float(np.arccos(np.clip(0.5 * (np.trace(R) - 1.0), -1.0, 1.0)))
        if angle < 1e-6:
            angle = float(np.linalg.norm(rodrigues_vector(R)))
        row = {"name": name, "R": R.tolist(), "t": t.tolist(), "angle": angle, "vertical": idx,
               "cv2_R1": R1.tolist(), "cv2_R2": R2.tolist(), "cv2_baseline": float(P2[idx, 3] / P2[idx, idx]),
               "exact_R1": eR1.tolist(), "exact_R2": eR2.tolist(), "exact_baseline": baseline}
        if idx == 0:
            fR1, fR2, _, _, _ = cv2.fisheye.stereoRectify(K, np.zeros(4), K, np.zeros(4), (640, 480), R, t, flags=0)
            assert np.abs(fR1 - R1).max() < 1e-12 and np.abs(fR2 - R2).max() < 1e-12, name
        out.append(row)
    return out


def maps(case_rows):
    rng = np.random.default_rng(0xACE5EC7)
    out = []
    for cam_name, W, H, f, case in (("kannala_brandt", 480, 400, 150.0, "horizontal_large_rotation"),
                                    ("kannala_brandt", 480, 400, 150.0, "vertical_negative_baseline"),
                                    ("rad_tan", 640, 400, 380.0, "horizontal_negative_baseline"),
                                    ("rad_tan", 640, 400, 380.0, "horizontal_large_rotation")):
        c = cams[cam_name]
        p = c["params"]
        K = np.array([[p[0], 0, p[2]], [0, p[1], p[3]], [0, 0, 1.0]])
        R1 = np.array(next(r for r in case_rows if r["name"] == case)["exact_R1"])
        P = np.array([[f, 0, W / 2.0, 0], [0, f, H / 2.0, 0], [0, 0, 1.0, 0]])
        if cam_name == "kannala_brandt":
            mx, my = cv2.fisheye.initUndistortRectifyMap(K, np.array(p[4:8]), R1, P, (W, H), cv2.CV_32FC1)
        else:
            mx, my = cv2.initUndistortRectifyMap(K, np.array(p[4:9]), R1, P, (W, H), cv2.CV_32FC1)
        u, v = rng.integers(0, W, 300), rng.integers(0, H, 300)
        out.append({"camera": cam_name, "case": case, "R1": R1.tolist(), "rectified": {"width": W, "height": H, "f": f,
                                                                                       "cx": W / 2.0, "cy": H / 2.0},
                    "u": u.tolist(), "v": v.tolist(), "map_x": mx[v, u].astype(float).tolist(),
                    "map_y": my[v, u].astype(float).tolist()})
    return out


if __name__ == "__main__":
    rows = cases()
    data = {"_comment": "cv2 %s; see make_rectify_golden.py" % cv2.__version__, "cases": rows, "maps": maps(rows)}
    json.dump(data, open(os.path.join(HERE, "opencv_rectify.json"), "w"), indent=1)
    print("wrote opencv_rectify.json")
