"""Depth images on the GPU (acm_render_depth, acm_render_depth_host, acm_depth_to_points; render_depth, depth_to_points):
all seven models against the depth oracle (tests/depth_oracle.c) at 10^6 points with ties, dispatch edges, contention and
determinism, a sphere about the camera, the render / back-project round trip, call forms, launch counts, argument errors
and the C++ wrapper."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import depth_oracle as D
from conftest import oracle_model
from test_gpu_rectify import axis_angle
from test_gpu_remap import EXACT, NAMES, gpu_model, launches, sized

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
POSES = {"identity": (np.eye(3), np.zeros(3)), "posed": (axis_angle([0.3, -0.8, 0.5], 10.0), np.array([0.15, -0.1, 0.3]))}
COS_100 = float(np.cos(np.deg2rad(100.0)))
EMPTY = 0xFFFFFFFF


@pytest.fixture(scope="module")
def acm():
    import apex_camera_models_b200 as m
    return m


@pytest.fixture(scope="module")
def ctx(acm):
    c = acm.Context(0)
    yield c
    c.close()


def _cloud(O, n, seed, n_dup):
    """n points of acm_synth_points3 (100-degree cone, adversarial points every 64th) plus n_dup exact copies of earlier ones
    (equal ranges: the lower index must win)."""
    pts = O.synth_points3(seed, 0, n - n_dup, COS_100, True)
    pick = np.random.default_rng(seed).integers(0, n - n_dup, n_dup)
    return np.vstack([pts, pts[pick]])


def _half_integer_pixels(uv, W):
    """Every pixel a point whose u or v lies within 1e-9 px of a half-integer may round to (both sides of the tie)."""
    near = (np.abs(uv[:, 0] - (np.floor(uv[:, 0]) + 0.5)) <= 1e-9) | (np.abs(uv[:, 1] - (np.floor(uv[:, 1]) + 0.5)) <= 1e-9)
    out = set()
    for u, v in uv[near]:
        for cu in {np.floor(u + 0.5 - 1e-9), np.floor(u + 0.5 + 1e-9)}:
            for cv in {np.floor(v + 0.5 - 1e-9), np.floor(v + 0.5 + 1e-9)}:
                out.add(int(cv) * W + int(cu))
    return out


@pytest.mark.parametrize("pose", list(POSES))
@pytest.mark.parametrize("name", NAMES)
def test_all_models_against_oracle(acm, ctx, O, cameras, name, pose):
    """10^6 seeded points: range and index images byte-identical to the oracle's for the arithmetic-only models; for KB and
    FOV (transcendental project) a differing pixel must be touched by a point within 1e-9 px of a half-integer.
    depth_to_points of the oracle's range image: the oracle's statuses, points bit-identical (arithmetic-only) or within
    1e-12 relative."""
    R, t = POSES[pose]
    cam = sized(cameras, name, 320, 240)
    g, o = gpu_model(acm, ctx, cam), oracle_model(O, cam)
    pts = _cloud(O, 1_000_000, 0xDE9711 + NAMES.index(name), 50_000)
    rng, idx = acm.render_depth(g, pts, R, t)
    ref_rng, ref_idx, uv = D.render_depth(o, pts, R, t, want_uv=True)
    drawn = ref_idx != EMPTY
    assert drawn.sum() > 1000
    if name in EXACT:
        assert rng.tobytes() == ref_rng.tobytes() and idx.tobytes() == ref_idx.tobytes()
    else:
        diff = set(np.flatnonzero((rng.view(np.uint32) != ref_rng.view(np.uint32)) | (idx != ref_idx)).tolist())
        assert diff <= _half_integer_pixels(uv, 320), sorted(diff)[:10]
    back, st = acm.depth_to_points(g, ref_rng, R, t)
    rb, rs = D.depth_to_points(o, ref_rng, R, t)
    assert np.array_equal(st, rs)
    ok = rs == D.OK
    assert ok.sum() > 0.5 * drawn.sum() and np.isnan(back[~ok]).all()
    if name in EXACT:
        assert back[ok].tobytes() == rb[ok].tobytes()
    else:
        scale = ref_rng[ok].astype(np.float64)[:, None] + np.abs(t).max()
        assert np.all(np.abs(back[ok] - rb[ok]) <= 1e-12 * scale)


def _device_render(acm, ctx, g, pts, R, t):
    """acm_render_depth on a device point buffer: (range, index, kernels launched)."""
    from apex_camera_models_b200 import _native as N
    res = g.get_resolution()
    npix = res.width * res.height
    X = acm.Points.from_numpy(ctx, np.asarray(pts, dtype=np.float64).reshape(-1, 3))
    d = ctx.device_alloc(npix * 8)
    cam = g.camera_block()
    try:
        ctx.sync()
        n0 = launches(ctx)
        ctx.check(N.lib.acm_render_depth(ctx.handle, C.byref(cam), (C.c_double * 9)(*np.ravel(R)), (C.c_double * 3)(*np.ravel(t)), X.handle,
                                         C.c_void_p(d), C.c_void_p(d + 4 * npix)))
        k = launches(ctx) - n0
        rng, idx = np.empty((res.height, res.width), np.float32), np.empty((res.height, res.width), np.uint32)
        ctx.d2h(rng, d); ctx.d2h(idx, d + 4 * npix)
        ctx.sync()
    finally:
        ctx.device_free(d)
        X.free()
    return rng, idx, k


def _device_back_launches(acm, ctx, g, rng, R, t):
    """Kernels one acm_depth_to_points call launches."""
    from apex_camera_models_b200 import _native as N
    npix = rng.size
    X = acm.Points(ctx, 3, npix)
    d = ctx.device_alloc(npix * 4)
    cam = g.camera_block()
    try:
        ctx.h2d(d, np.ascontiguousarray(rng))
        ctx.sync()
        n0 = launches(ctx)
        ctx.check(N.lib.acm_depth_to_points(ctx.handle, C.byref(cam), (C.c_double * 9)(*np.ravel(R)), (C.c_double * 3)(*np.ravel(t)),
                                            C.c_void_p(d), X.handle, None))
        k = launches(ctx) - n0
        ctx.sync()
    finally:
        ctx.device_free(d)
        X.free()
    return k


@pytest.mark.parametrize("size", [(1, 1), (7, 5), (320, 240)])
@pytest.mark.parametrize("n", [0, 1, "past_grid"])
def test_dispatch_edges_and_call_forms(acm, ctx, O, cameras, size, n):
    """n = 0 (an all-empty image), n = 1 and n one past a full grid-stride trip (8 blocks per SM of 256 threads) on 1x1,
    odd-sized and ordinary images: the oracle's bytes; the host form equals the device form byte for byte; each form launches
    the render and resolve kernels (only the resolve kernel when n = 0); depth_to_points launches one kernel."""
    if n == "past_grid":
        n = ctx.device_info()["sm_count"] * 8 * 256 + 1
    W, H = size
    cam = sized(cameras, "double_sphere", W, H)
    if W < 100:  # a small image sees the middle of the cloud: focal lengths of a third of the width, centre near (W-1)/2
        cam["params"][:4] = [0.3 * W, 0.3 * W, (W - 1) / 2.0 + 0.1, (H - 1) / 2.0 - 0.1]
    g, o = gpu_model(acm, ctx, cam), oracle_model(O, cam)
    R, t = POSES["posed"]
    pts = _cloud(O, max(n, 64), 0xDE9720, 16)[:n] if n else np.empty((0, 3))
    rng, idx, k = _device_render(acm, ctx, g, pts, R, t)
    assert k == (2 if n else 1)
    n0 = launches(ctx)
    hr, hi = acm.render_depth(g, pts, R, t)
    assert launches(ctx) - n0 == (2 if n else 1)
    assert hr.tobytes() == rng.tobytes() and hi.tobytes() == idx.tobytes()
    pr, pi = acm.render_depth(g, acm.Points.from_numpy(ctx, pts) if n else pts, R, t)
    assert pr.tobytes() == rng.tobytes() and pi.tobytes() == idx.tobytes()
    er, ei = D.render_depth(o, pts, R, t)
    assert rng.tobytes() == er.tobytes() and idx.tobytes() == ei.tobytes()
    if n == 0:
        assert (idx == EMPTY).all() and (rng.view(np.uint32) == EMPTY).all()
    back, st = acm.depth_to_points(g, rng, R, t)
    assert _device_back_launches(acm, ctx, g, rng, R, t) == 1
    rb, rs = D.depth_to_points(o, rng, R, t)
    assert np.array_equal(st, rs) and back.tobytes() == rb.tobytes()


def test_key_image_beyond_l2(acm, ctx, O, cameras):
    """A 4096 x 4096 image (a 134 MB key image, more than the 126 MB L2) with 4 * 10^6 points: the oracle's bytes."""
    cam = sized(cameras, "pinhole", 4096, 4096)
    g, o = gpu_model(acm, ctx, cam), oracle_model(O, cam)
    pts = _cloud(O, 4_000_000, 0xDE9730, 100_000)
    rng, idx = acm.render_depth(g, pts)
    er, ei = D.render_depth(o, pts)
    assert (ei != EMPTY).sum() > 300_000
    assert rng.tobytes() == er.tobytes() and idx.tobytes() == ei.tobytes()


@pytest.mark.parametrize("equal", [False, True])
def test_contention_and_determinism(acm, ctx, cameras, equal):
    """10^6 points on the principal point's pixel: with distinct ranges the nearest wins wherever its index is, with equal
    ranges index 0 wins; three repeated calls (device and host form) are bit-identical."""
    cam = sized(cameras, "pinhole", 320, 240)
    g = gpu_model(acm, ctx, cam)
    n = 1_000_000
    if equal:
        z, winner = np.full(n, 3.0), 0
    else:
        z = 2.0 + np.random.default_rng(0xDE9740).permutation(n) * 1e-5  # distinct in f32 (spacing 2.4e-7 at 2)
        winner = int(np.argmin(z))
    pts = np.column_stack([np.zeros(n), np.zeros(n), z])
    pix = (int(round(cam["params"][3])), int(round(cam["params"][2])))  # (row, col) of (cx, cy)
    first = acm.render_depth(g, pts)
    rng, idx = first
    assert idx[pix] == winner and rng[pix] == np.float32(z[winner])
    assert (idx == EMPTY).sum() == idx.size - 1
    X = acm.Points.from_numpy(ctx, pts)
    try:
        for _ in range(3):
            for again in (acm.render_depth(g, pts), acm.render_depth(g, X)):
                assert again[0].tobytes() == rng.tobytes() and again[1].tobytes() == idx.tobytes()
    finally:
        X.free()


@pytest.mark.parametrize("name", ["kannala_brandt", "double_sphere"])
def test_sphere_about_the_camera(acm, ctx, O, cameras, name):
    """A dense sphere of radius 2.5 about the camera through a wide-angle camera: every drawn pixel holds float(2.5), drawn
    pixels cover most of the image, and through Double Sphere points with z < 0 (rays beyond 90 degrees) are drawn."""
    cam = sized(cameras, name, 512, 512, focal_scale=0.7 if name == "kannala_brandt" else 0.4)
    g = gpu_model(acm, ctx, cam)
    rs = np.random.default_rng(0xDE9750)
    d = rs.normal(size=(4_000_000, 3))
    pts = 2.5 * d / np.linalg.norm(d, axis=1, keepdims=True)
    rng, idx = acm.render_depth(g, pts)
    drawn = idx != EMPTY
    assert drawn.sum() > 0.5 * idx.size
    assert np.all(rng[drawn] == np.float32(2.5))
    if name == "double_sphere":  # the reference's KB project refuses z < 0; Double Sphere draws rays beyond 90 degrees
        assert (pts[idx[drawn], 2] < 0).sum() > 100


# pixel tolerance of project(depth_to_points(...)) against the pixel centre, per model (None: not checked):
# RadTan's unproject stops its Newton loop at |error| < 1e-6 in normalised coordinates; the UCM sample camera has
# alpha = 1.01674 > 1, where the reference's unproject is not the inverse of its project (as MID_TOL in test_gpu_triangulate.py).
PIX_TOL = {"pinhole": 1e-6, "rad_tan": 1e-3, "kannala_brandt": 1e-6, "ucm": None, "eucm": 1e-6, "double_sphere": 1e-6, "fov": 1e-6}


@pytest.mark.parametrize("name", NAMES)
def test_render_back_project_round_trip(acm, ctx, O, cameras, name):
    """Render with a pose, back-project with the same pose: for every drawn pixel |R x_back + t| equals the f32 range to 1e-12
    relative, and x_back projects onto the pixel centre within PIX_TOL."""
    R, t = POSES["posed"]
    cam = sized(cameras, name, 320, 240)
    g, o = gpu_model(acm, ctx, cam), oracle_model(O, cam)
    pts = _cloud(O, 1_000_000, 0xDE9760, 0)
    rng, idx = acm.render_depth(g, pts, R, t)
    back, st = acm.depth_to_points(g, rng, R, t)
    drawn = idx != EMPTY
    ok = drawn & (st == D.OK)
    assert ok.sum() > 0.9 * drawn.sum() and drawn.sum() > 1000
    xc = back[ok] @ R.T + t
    r = rng[ok].astype(np.float64)
    assert np.all(np.abs(np.linalg.norm(xc, axis=1) - r) <= 1e-12 * r)
    if PIX_TOL[name] is not None:
        uv, _, s = O.project_point_jacobian(o, xc)  # geometric validity only: a pixel centre of row / column 0 may land at -1e-13
        rows, cols = np.nonzero(ok)
        # a pixel drawn by a point just inside 90 degrees may have a centre ray just beyond it, which KB's project refuses (z < 0)
        good = s == 0
        assert good.mean() > 0.99 and np.all(xc[~good, 2] < 0)
        err = np.hypot(uv[good, 0] - cols[good], uv[good, 1] - rows[good])
        assert err.max() <= PIX_TOL[name], err.max()


def test_argument_errors(acm, ctx, cameras):
    from apex_camera_models_b200 import _native as N
    L = N.lib
    g = gpu_model(acm, ctx, sized(cameras, "pinhole", 64, 48))
    cam = g.camera_block()
    X, X2, Xf, Xs = acm.Points(ctx, 3, 4), acm.Points(ctx, 2, 4), acm.Points(ctx, 3, 4, N.F32), acm.Points(ctx, 3, 64 * 48)
    Xw = acm.Points(ctx, 3, 64 * 48 - 1)
    d = ctx.device_alloc(64 * 48 * 8)
    R9 = (C.c_double * 9)(*np.eye(3).ravel())
    t3 = (C.c_double * 3)(0.0, 0.0, 0.0)
    vec = lambda v, k: (C.c_double * k)(*np.ravel(v))
    h = lambda p: p.handle if p is not None else None

    def render(c=C.byref(cam), R=R9, t=t3, pts=X, rng=C.c_void_p(d), idx=C.c_void_p(d + 4 * 64 * 48)):
        return L.acm_render_depth(ctx.handle, c, R, t, h(pts), rng, idx)

    def back(c=C.byref(cam), R=R9, t=t3, rng=C.c_void_p(d), out=Xs, st=None):
        return L.acm_depth_to_points(ctx.handle, c, R, t, rng, h(out), st)

    def fails(rc, text):
        assert rc == N.ERR_INVALID_ARG, (rc, text)
        assert text in L.acm_last_error(ctx.handle).decode(), L.acm_last_error(ctx.handle).decode()

    try:
        ctx.check(N.lib.acm_memset_d(ctx.handle, C.c_void_p(d), 0, 64 * 48 * 8))
        assert render() == N.OK and back() == N.OK
        for call in (render, back):
            fails(call(c=None), "null camera")
            fails(call(R=None), "null rotation")
            fails(call(R=vec(np.diag([1.0, 1.0, np.nan]), 9)), "non-finite")
            fails(call(R=vec(np.eye(3) * 1.001, 9)), "not orthonormal")
            fails(call(R=vec(np.diag([1.0, -1.0, 1.0]), 9)), "reflection")
            fails(call(t=None), "null translation")
            fails(call(t=vec([0.0, np.nan, 0.0], 3)), "non-finite")
            nores = g.camera_block(); nores.width = 0
            fails(call(c=C.byref(nores)), "resolution")
        fails(render(pts=None), "null buffer")
        fails(render(rng=None), "null buffer")
        fails(render(idx=None), "null buffer")
        fails(render(pts=X2), "dim-3 f64")
        fails(render(pts=Xf), "dim-3 f64")
        fails(back(rng=None), "null buffer")
        fails(back(out=None), "null buffer")
        fails(back(out=X2), "dim-3 f64")
        fails(back(out=Xw), "width * height")
        bad = g.camera_block(); bad.model = 9
        fails(render(c=C.byref(bad)), "invalid camera model id")
        out_r, out_i = (C.c_float * (64 * 48))(), (C.c_uint32 * (64 * 48))()
        p = (C.c_double * 3)(0.0, 0.0, 1.0)
        assert L.acm_render_depth_host(ctx.handle, C.byref(cam), R9, t3, p, 1, out_r, out_i) == N.OK
        assert L.acm_render_depth_host(ctx.handle, C.byref(cam), R9, t3, None, 0, out_r, out_i) == N.OK
        fails(L.acm_render_depth_host(ctx.handle, C.byref(cam), R9, t3, None, 1, out_r, out_i), "null buffer")
        fails(L.acm_render_depth_host(ctx.handle, C.byref(cam), R9, t3, p, 1, None, out_i), "null buffer")
        # n >= 2^32 - 1 is refused before any allocation or copy (the null source would fail a copy)
        fails(L.acm_render_depth_host(ctx.handle, C.byref(cam), R9, t3, None, 2 ** 32 - 1, out_r, out_i), "2^32 - 1")
        fails(L.acm_render_depth_host(ctx.handle, C.byref(cam), R9, t3, None, 2 ** 40, out_r, out_i), "2^32 - 1")
    finally:
        ctx.device_free(d)
        for q in (X, X2, Xf, Xs, Xw):
            q.free()
    with pytest.raises(acm.UtilError, match="3x3"):
        acm.render_depth(g, np.zeros((1, 3)), np.eye(2))
    with pytest.raises(acm.UtilError, match="3 entries"):
        acm.render_depth(g, np.zeros((1, 3)), None, [1.0, 0.0])
    with pytest.raises(acm.UtilError, match="range image"):
        acm.depth_to_points(g, np.zeros((48, 63), np.float32))
    with pytest.raises(acm.AcmError, match="non-finite"):
        acm.depth_to_points(g, np.zeros((48, 64), np.float32), None, [np.inf, 0.0, 0.0])


def test_cpp_wrapper(acm, ctx, O, cameras, tmp_path):
    """tests/cpp/depth_test.cpp (acm::render_depth, acm::depth_to_points) agrees with render_depth / depth_to_points byte for
    byte."""
    libdir = os.path.join(ROOT, "apex_camera_models_b200", "lib")
    exe = str(tmp_path / "depth_test")
    subprocess.run(["/usr/bin/g++", "-std=c++17", "-O1", "-Wall", "-Werror", "-pthread", "-I", os.path.join(ROOT, "include"),
                    os.path.join(ROOT, "tests", "cpp", "depth_test.cpp"), "-o", exe, "-L", libdir, "-lacm", f"-Wl,-rpath,{libdir}"],
                   check=True)
    g = gpu_model(acm, ctx, dict(cameras["kannala_brandt"]))
    R, t = POSES["posed"]
    pts = _cloud(O, 200_001, 0xDE9770, 1000)
    inp, outp = tmp_path / "in.bin", tmp_path / "out.bin"
    np.concatenate([R.ravel(), t, [float(len(pts))], pts.ravel()]).tofile(inp)
    r = subprocess.run([exe, str(inp), str(outp)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    assert "DEPTH_TEST_OK" in r.stdout
    raw = outp.read_bytes()
    npix = 512 * 512
    rng, idx = acm.render_depth(g, pts, R, t)
    back, st = acm.depth_to_points(g, rng, R, t)
    assert raw[:4 * npix] == rng.tobytes() and raw[4 * npix:8 * npix] == idx.tobytes()
    assert raw[8 * npix:32 * npix] == back.tobytes() and raw[32 * npix:] == st.tobytes()
