"""Triangulation on the GPU (acm_triangulate, acm_triangulate_host, triangulate_points): every model pair against the
triangulation oracle (tests/triangulate_oracle.c) in both modes, recovery of noise-free points, refinement never costing
more than the midpoint, agreement with triangulation of rectified pixels, dispatch edges, call forms and launch counts,
argument errors and the C++ wrapper."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import triangulate_oracle as T
from conftest import oracle_model
from test_gpu_rectify import axis_angle
from test_gpu_remap import EXACT, NAMES, gpu_model, launches, sized

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ROT = axis_angle([0.3, -0.8, 0.5], 10.0)
T_BASE = np.array([-0.1, 0.0, 0.0])
NTHREADS = os.cpu_count() or 1

# Noise-free midpoint tolerance (relative to max |X|) per model, set by how exactly its unproject inverts its project:
#   RadTan: the reference's Newton loop stops at |error| < 1e-6 in normalised coordinates, so a ray is off by up to ~1e-6 rad,
#           which the ~0.02-0.1 rad parallax of the rig magnifies to ~1e-4 relative;
#   UCM:    the sample camera has alpha = 1.01674 > 1, where the reference's unproject is not the inverse of its project (a
#           round trip moves a pixel by up to ~0.6 px, the ray by ~1.6e-3 rad): its midpoints are not checked (refinement,
#           which only uses project, recovers the points);
#   others: closed-form or fully converged inverses, limited by the rounding of 1 - b^2.
MID_TOL = {"pinhole": 1e-9, "rad_tan": 1e-3, "kannala_brandt": 1e-9, "ucm": None, "eucm": 1e-9, "double_sphere": 1e-9, "fov": 1e-9}


@pytest.fixture(scope="module")
def acm():
    import apex_camera_models_b200 as m
    return m


@pytest.fixture(scope="module")
def ctx(acm):
    c = acm.Context(0)
    yield c
    c.close()


def _truth(O, ma, mb, R, t, n, seed):
    """Ground-truth points 0.5-5 units along the rays of random first-camera pixels whose projections fall inside both
    images, and those projections."""
    rng = np.random.default_rng(seed)
    uv = np.column_stack([rng.uniform(0, ma.width, 8 * n), rng.uniform(0, ma.height, 8 * n)])
    ray, st = O.unproject(ma, uv, NTHREADS)
    X = ray * rng.uniform(0.5, 5.0, 8 * n)[:, None]
    uv1, s1 = O.project(ma, X, NTHREADS)
    uv2, s2 = O.project(mb, X @ np.asarray(R).T + t, NTHREADS)
    inside = lambda p, m: (p[:, 0] >= 0) & (p[:, 0] < m.width) & (p[:, 1] >= 0) & (p[:, 1] < m.height)
    ok = np.flatnonzero((st == 0) & (s1 == 0) & (s2 == 0) & inside(uv1, ma) & inside(uv2, mb))[:n]
    return uv1[ok], uv2[ok], X[ok]


def _dataset(O, ma, mb, n, seed):
    """n seeded pairs: 50 % noise-free projections of ground-truth points, 30 % the same with N(0, 0.5 px) noise, 20 % random
    pixel pairs (slightly beyond both images, so that every status occurs).  Returns uv1, uv2, the noise-free mask."""
    rng = np.random.default_rng(seed + 1)
    a1, a2, _ = _truth(O, ma, mb, ROT, T_BASE, n // 2, seed)
    b1, b2, _ = _truth(O, ma, mb, ROT, T_BASE, (3 * n) // 10, seed + 2)
    b1 = b1 + rng.normal(0, 0.5, b1.shape); b2 = b2 + rng.normal(0, 0.5, b2.shape)
    k = n - len(a1) - len(b1)
    c1 = np.column_stack([rng.uniform(-4, ma.width + 4, k), rng.uniform(-4, ma.height + 4, k)])
    c2 = np.column_stack([rng.uniform(-4, mb.width + 4, k), rng.uniform(-4, mb.height + 4, k)])
    clean = np.zeros(n, bool); clean[:len(a1)] = True
    return np.vstack([a1, b1, c1]), np.vstack([a2, b2, c2]), clean


@pytest.mark.parametrize("ma_name", NAMES)
@pytest.mark.parametrize("mb_name", NAMES)
def test_all_model_pairs(acm, ctx, O, cameras, ma_name, mb_name):
    """10^5 seeded pairs, both modes: status bytes equal the oracle's; midpoints bit-identical where both models are
    arithmetic-only, within 1e-9 relative otherwise; refined noise-free points within 1e-9 relative.

    A refined noisy pair ends on a minimum that is flat along the depth, and the LM path to it turns on accept / reject
    decisions that two implementations rounding differently can take differently: a 1e-15 relative change of the input
    moves the oracle's own refined points by up to ~1e-7 relative (rarely 1e-5), and more behind the UCM sample camera,
    whose alpha = 1.01674 lies outside (0, 1].  There 99 % of the points and costs agree to 1e-6 relative.  A random (mismatched) pair may end on different local minima in 10 trials, so only its
    status is compared, and that its refined cost never exceeds its midpoint cost."""
    ca, cb = sized(cameras, ma_name, 320, 240), sized(cameras, mb_name, 288, 224)
    ga, gb = gpu_model(acm, ctx, ca), gpu_model(acm, ctx, cb)
    oa, ob = oracle_model(O, ca), oracle_model(O, cb)
    n = 100_000
    uv1, uv2, clean = _dataset(O, oa, ob, n, 0x7121A7E3)
    idx = np.arange(n)
    noisy = ~clean & (idx < n - n // 5)
    exact = ma_name in EXACT and mb_name in EXACT
    mid_err = None
    for it in (0, 10):
        got, gerr, gst = acm.triangulate_points(ga, gb, ROT, T_BASE, uv1, uv2, it)
        ref, rerr, rst = T.triangulate(oa, ob, ROT, T_BASE, uv1, uv2, it, NTHREADS)
        assert np.array_equal(gst, rst), np.flatnonzero(gst != rst)[:10]
        ok = rst == T.OK
        assert ok.sum() > 10_000 and np.isnan(got[~ok]).all() and np.isnan(gerr[~ok]).all()
        assert np.isfinite(got[ok]).all() and np.isfinite(gerr[ok]).all()
        scale = np.abs(ref).max(axis=1, keepdims=True)
        if it == 0:
            mid_err = gerr
            if exact:
                assert np.array_equal(got[ok], ref[ok]) and np.array_equal(gerr[ok], rerr[ok])
            else:
                assert np.all(np.abs(got[ok] - ref[ok]) <= 1e-9 * scale[ok])
            continue
        tight = ok & clean
        assert np.all(np.abs(got[tight] - ref[tight]) <= 1e-9 * scale[tight])
        m = ok & noisy
        rel = np.abs(got[m] - ref[m]).max(axis=1) / scale[m, 0]
        assert np.quantile(rel, 0.99) <= 1e-6, np.sort(rel)[-20:]
        cg, cr = (gerr[m] ** 2).sum(1), (rerr[m] ** 2).sum(1)
        assert np.quantile(np.abs(cg - cr) / np.maximum(cr, 1e-12), 0.99) <= 1e-6
        assert np.all((gerr[ok] ** 2).sum(1) <= (mid_err[ok] ** 2).sum(1))
    assert {T.OK, T.BEHIND} <= set(np.unique(rst).tolist())


@pytest.mark.parametrize("ma_name", NAMES)
@pytest.mark.parametrize("mb_name", NAMES)
def test_noise_free_recovery(acm, ctx, O, cameras, ma_name, mb_name):
    """Up to 20 000 points seen by both cameras: refined points within 1e-9 relative of the ground truth with errors <= 1e-9
    px; midpoints within MID_TOL."""
    ca, cb = sized(cameras, ma_name, 320, 240), sized(cameras, mb_name, 288, 224)
    ga, gb = gpu_model(acm, ctx, ca), gpu_model(acm, ctx, cb)
    uv1, uv2, X = _truth(O, oracle_model(O, ca), oracle_model(O, cb), ROT, T_BASE, 20_000, 0x7121A7E4)
    assert len(X) >= 2_000
    scale = np.abs(X).max(axis=1, keepdims=True)
    got, err, st = acm.triangulate_points(ga, gb, ROT, T_BASE, uv1, uv2, 10)
    assert np.all(st == T.OK)
    assert np.all(np.abs(got - X) <= 1e-9 * scale)
    assert np.all(err <= 1e-9)
    got, _, st = acm.triangulate_points(ga, gb, ROT, T_BASE, uv1, uv2, 0)
    assert np.all(st == T.OK)
    if MID_TOL[ma_name] is not None and MID_TOL[mb_name] is not None:
        assert np.all(np.abs(got - X) <= max(MID_TOL[ma_name], MID_TOL[mb_name]) * scale)


@pytest.mark.parametrize("pair", [("pinhole", "pinhole"), ("kannala_brandt", "double_sphere"), ("rad_tan", "fov"), ("eucm", "ucm")])
def test_noisy_refinement_never_costs_more(acm, ctx, O, cameras, pair):
    """sigma = 0.5 px: for every Ok pair the refined cost (e1^2 + e2^2) is <= the midpoint's, with the same status."""
    ca, cb = sized(cameras, pair[0], 320, 240), sized(cameras, pair[1], 288, 224)
    ga, gb = gpu_model(acm, ctx, ca), gpu_model(acm, ctx, cb)
    uv1, uv2, _ = _truth(O, oracle_model(O, ca), oracle_model(O, cb), ROT, T_BASE, 50_000, 0x7121A7E5)
    rng = np.random.default_rng(0x7121A7E6)
    uv1 = uv1 + rng.normal(0, 0.5, uv1.shape); uv2 = uv2 + rng.normal(0, 0.5, uv2.shape)
    _, em, sm = acm.triangulate_points(ga, gb, ROT, T_BASE, uv1, uv2, 0)
    _, er, sr = acm.triangulate_points(ga, gb, ROT, T_BASE, uv1, uv2, 10)
    assert np.array_equal(sm, sr)
    ok = sm == T.OK
    assert ok.sum() > 0.9 * len(ok)
    cm, cr = (em[ok] ** 2).sum(1), (er[ok] ** 2).sum(1)
    assert np.all(cr <= cm)
    assert cr.mean() < cm.mean()


@pytest.mark.parametrize("right", ["kannala_brandt", "double_sphere"])
def test_rectification_consistency(acm, ctx, O, cameras, right):
    """Raw KB / Double Sphere matches, and the same points' rectified pinhole pixels with (I, baseline e) of a
    StereoRectifier: after R1^T the two sets of refined points agree to 1e-9 relative."""
    cl, cr = sized(cameras, "kannala_brandt", 512, 384), sized(cameras, right, 480, 360)
    left, rightm = gpu_model(acm, ctx, cl), gpu_model(acm, ctx, cr)
    Rm, t = axis_angle([0.1, 1.0, 0.2], 4.0), np.array([-0.12, 0.004, 0.003])
    rect = acm.PinholeModel(acm.Intrinsics(200.0, 200.0, 199.5, 149.5), acm.Resolution(400, 300), ctx=ctx)
    with acm.StereoRectifier(left, rightm, Rm, t, rect) as rig:
        assert not rig.vertical
        rng = np.random.default_rng(0x7121A7E7)
        # ground truth in the rectified frame: integer-free rectified pixels of the left view, depths 0.5-5
        n = 20_000
        u, v, Z = rng.uniform(10, 390, n), rng.uniform(10, 290, n), rng.uniform(0.5, 5.0, n)
        Xr = np.column_stack([(u - 199.5) / 200.0 * Z, (v - 149.5) / 200.0 * Z, Z])
        X1 = Xr @ rig.R1                  # R1^T x_rect
        X2 = X1 @ Rm.T + t
        ol, orr = oracle_model(O, cl), oracle_model(O, cr)
        uv1, s1 = O.project(ol, X1)
        uv2, s2 = O.project(orr, X2)
        Xr2 = X2 @ rig.R2.T
        ur2 = np.column_stack([200.0 * Xr2[:, 0] / Xr2[:, 2] + 199.5, 200.0 * Xr2[:, 1] / Xr2[:, 2] + 149.5])
        inside = lambda p, W, H: (p[:, 0] >= 0) & (p[:, 0] < W) & (p[:, 1] >= 0) & (p[:, 1] < H)
        keep = (s1 == 0) & (s2 == 0) & inside(ur2, 400, 300) & inside(uv1, 512, 384) & inside(uv2, 480, 360) & (Xr2[:, 2] > 0)
        assert keep.sum() > 5_000
        raw, _, st_raw = acm.triangulate_points(left, rightm, Rm, t, uv1[keep], uv2[keep])
        ur1 = np.column_stack([u, v])[keep]
        rec, _, st_rec = acm.triangulate_points(rect, rect, np.eye(3), [rig.baseline, 0.0, 0.0], ur1, ur2[keep])
        assert np.all(st_raw == T.OK) and np.all(st_rec == T.OK)
        back = rec @ rig.R1               # R1^T X_rect
        scale = np.abs(raw).max(axis=1, keepdims=True)
        assert np.all(np.abs(back - raw) <= 1e-9 * scale)
        assert np.all(np.abs(raw - X1[keep]) <= 1e-9 * scale)


def _device_call(acm, ctx, ga, gb, uv1, uv2, it):
    """acm_triangulate on device buffers: (points, errors (N, 2), status, kernels launched)."""
    from apex_camera_models_b200 import _native as N
    n = len(uv1)
    a, b = acm.Points.from_numpy(ctx, uv1.reshape(-1, 2)), acm.Points.from_numpy(ctx, uv2.reshape(-1, 2))
    xyz = acm.Points(ctx, 3, n)
    d = ctx.device_alloc(max(n, 1) * 17)
    ca, cb = ga.camera_block(), gb.camera_block()
    try:
        ctx.sync()
        n0 = launches(ctx)
        ctx.check(N.lib.acm_triangulate(ctx.handle, C.byref(ca), C.byref(cb), (C.c_double * 9)(*ROT.ravel()), (C.c_double * 3)(*T_BASE),
                                        a.handle, b.handle, it, xyz.handle, C.c_void_p(d), C.c_void_p(d + 16 * n)))
        k = launches(ctx) - n0
        err, st = np.empty((2, n)), np.empty(n, np.uint8)
        if n:
            ctx.d2h(err, d); ctx.d2h(st, d + 16 * n)
        ctx.sync()
        pts = xyz.numpy()
    finally:
        ctx.device_free(d)
        for p in (a, b, xyz):
            p.free()
    return pts, err.T.copy(), st, k


@pytest.mark.parametrize("n", [0, 1, 7, 1001, "past_grid"])
def test_dispatch_edges_and_call_forms(acm, ctx, O, cameras, n):
    """n = 0 launches nothing; n = 1, odd n and an n past the first grid-stride trip (8 blocks per SM of 256 threads) give the
    oracle's status bytes and midpoints; the host form equals the device form byte for byte and each form launches exactly
    one kernel."""
    if n == "past_grid":
        n = ctx.device_info()["sm_count"] * 8 * 256 + 3
    ca, cb = sized(cameras, "kannala_brandt", 320, 240), sized(cameras, "pinhole", 288, 224)
    ga, gb = gpu_model(acm, ctx, ca), gpu_model(acm, ctx, cb)
    oa, ob = oracle_model(O, ca), oracle_model(O, cb)
    if n:
        uv1, uv2, _ = _dataset(O, oa, ob, max(n, 10), 0x7121A7E8)
        uv1, uv2 = uv1[:n].copy(), uv2[:n].copy()
    else:
        uv1, uv2 = np.empty((0, 2)), np.empty((0, 2))
    for it in (0, 10):
        pts, err, st, k = _device_call(acm, ctx, ga, gb, uv1, uv2, it)
        assert k == (1 if n else 0)
        n0 = launches(ctx)
        hp, he, hs = acm.triangulate_points(ga, gb, ROT, T_BASE, uv1, uv2, it)
        assert launches(ctx) - n0 == (1 if n else 0)
        assert hp.tobytes() == pts.tobytes() and he.tobytes() == err.tobytes() and hs.tobytes() == st.tobytes()
        if n:
            dp, de, ds = acm.triangulate_points(ga, gb, ROT, T_BASE, acm.Points.from_numpy(ctx, uv1), uv2, it)
            assert dp.tobytes() == pts.tobytes() and de.tobytes() == err.tobytes() and ds.tobytes() == st.tobytes()
            ref, _, rst = T.triangulate(oa, ob, ROT, T_BASE, uv1, uv2, it, NTHREADS)
            assert np.array_equal(st, rst)
            ok = rst == T.OK
            if it == 0:  # refined points are compared in test_all_model_pairs
                assert np.all(np.abs(pts[ok] - ref[ok]) <= 1e-9 * np.abs(ref[ok]).max(axis=1, keepdims=True))


def test_two_camera_cache_keeps_results(acm, ctx, O, cameras):
    """Alternating calls on a KB / RadTan pair (two cached camera blocks) and on other cameras in between give the same bytes."""
    ca, cb = sized(cameras, "kannala_brandt", 320, 240), sized(cameras, "rad_tan", 288, 224)
    ga, gb = gpu_model(acm, ctx, ca), gpu_model(acm, ctx, cb)
    uv1, uv2, _ = _dataset(O, oracle_model(O, ca), oracle_model(O, cb), 1000, 0x7121A7E9)
    first = acm.triangulate_points(ga, gb, ROT, T_BASE, uv1, uv2)
    gc, gd = gpu_model(acm, ctx, sized(cameras, "rad_tan", 320, 240)), gpu_model(acm, ctx, sized(cameras, "kannala_brandt", 288, 224))
    second = acm.triangulate_points(gc, gd, ROT, T_BASE, uv1, uv2)
    other = gpu_model(acm, ctx, sized(cameras, "fov", 64, 48))
    for _ in range(3):
        again = acm.triangulate_points(ga, gb, ROT, T_BASE, uv1, uv2)
        assert all(x.tobytes() == y.tobytes() for x, y in zip(first, again))
        again = acm.triangulate_points(gc, gd, ROT, T_BASE, uv1, uv2)
        assert all(x.tobytes() == y.tobytes() for x, y in zip(second, again))
        other.project(np.array([0.0, 0.0, 1.0]))


def test_argument_errors(acm, ctx, cameras):
    from apex_camera_models_b200 import _native as N
    L = N.lib
    ga, gb = gpu_model(acm, ctx, sized(cameras, "pinhole", 64, 48)), gpu_model(acm, ctx, sized(cameras, "kannala_brandt", 64, 48))
    ca, cb = ga.camera_block(), gb.camera_block()
    a, b, x = acm.Points(ctx, 2, 4), acm.Points(ctx, 2, 4), acm.Points(ctx, 3, 4)
    a3, b5, x5, af = acm.Points(ctx, 3, 4), acm.Points(ctx, 2, 5), acm.Points(ctx, 3, 5), acm.Points(ctx, 2, 4, N.F32)
    R9 = (C.c_double * 9)(*np.eye(3).ravel())
    t3 = (C.c_double * 3)(-0.1, 0.0, 0.0)

    def vec(v, k):
        return (C.c_double * k)(*np.ravel(v))

    def call(cam_a=C.byref(ca), cam_b=C.byref(cb), R=R9, t=t3, p1=a, p2=b, it=10, out=x):
        h = lambda p: p.handle if p is not None else None
        return L.acm_triangulate(ctx.handle, cam_a, cam_b, R, t, h(p1), h(p2), it, h(out), None, None)

    def fails(rc, text, code=N.ERR_INVALID_ARG):
        assert rc == code, (rc, text)
        assert text in L.acm_last_error(ctx.handle).decode(), L.acm_last_error(ctx.handle).decode()

    try:
        assert call() == N.OK
        fails(call(cam_a=None), "null camera")
        fails(call(cam_b=None), "null camera")
        fails(call(R=None), "null rotation")
        fails(call(R=vec(np.diag([1.0, 1.0, np.nan]), 9)), "non-finite")
        fails(call(R=vec(np.eye(3) * 1.001, 9)), "not orthonormal")
        fails(call(R=vec(np.diag([1.0, -1.0, 1.0]), 9)), "reflection")
        fails(call(t=None), "null translation")
        fails(call(t=vec([np.inf, 0.0, 0.0], 3)), "non-finite")
        fails(call(t=vec([0.0, 0.0, 0.0], 3)), "translation is zero")
        fails(call(it=-1), "max_iterations")
        fails(call(p1=None), "null point buffer")
        fails(call(p2=None), "null point buffer")
        fails(call(out=None), "null point buffer")
        fails(call(p1=a3), "dim 2")
        fails(call(out=b), "dim 3")
        fails(call(p2=b5), "same number")
        fails(call(out=x5), "same number")
        fails(call(p1=af), "f64")
        bad = ga.camera_block(); bad.model = 9
        fails(call(cam_a=C.byref(bad)), "invalid camera model id")
        bad = gb.camera_block(); bad.n_params = 3
        fails(call(cam_b=C.byref(bad)), "expects", N.ERR_INVALID_PARAMS)
        uv = (C.c_double * 2)(1.0, 1.0); out = (C.c_double * 3)()
        assert L.acm_triangulate_host(ctx.handle, C.byref(ca), C.byref(cb), R9, t3, uv, uv, 1, 0, out, None, None) == N.OK
        fails(L.acm_triangulate_host(ctx.handle, C.byref(ca), C.byref(cb), R9, t3, None, uv, 1, 0, out, None, None), "null point buffer")
        fails(L.acm_triangulate_host(ctx.handle, C.byref(ca), C.byref(cb), R9, vec([0.0, 0.0, 0.0], 3), uv, uv, 1, 0, out, None, None),
              "translation is zero")
        fails(L.acm_triangulate_host(ctx.handle, C.byref(ca), C.byref(cb), R9, t3, uv, uv, 1, -2, out, None, None), "max_iterations")
        assert L.acm_triangulate_host(ctx.handle, C.byref(ca), C.byref(cb), R9, t3, None, None, 0, 0, None, None, None) == N.OK
    finally:
        for p in (a, b, x, a3, b5, x5, af):
            p.free()
    with pytest.raises(acm.UtilError, match="3x3"):
        acm.triangulate_points(ga, gb, np.eye(2), [1.0, 0, 0], np.zeros((1, 2)), np.zeros((1, 2)))
    with pytest.raises(acm.UtilError, match="3 entries"):
        acm.triangulate_points(ga, gb, np.eye(3), [1.0, 0], np.zeros((1, 2)), np.zeros((1, 2)))
    with pytest.raises(acm.UtilError, match="max_iterations"):
        acm.triangulate_points(ga, gb, np.eye(3), [1.0, 0, 0], np.zeros((1, 2)), np.zeros((1, 2)), -1)
    with pytest.raises(acm.UtilError, match="pixels of the first camera"):
        acm.triangulate_points(ga, gb, np.eye(3), [1.0, 0, 0], np.zeros((2, 2)), np.zeros((1, 2)))
    with pytest.raises(acm.AcmError, match="translation is zero"):
        acm.triangulate_points(ga, gb, np.eye(3), [0.0, 0, 0], np.zeros((1, 2)), np.zeros((1, 2)))


def test_cpp_wrapper(acm, ctx, O, cameras, tmp_path):
    """tests/cpp/triangulate_test.cpp (acm::triangulate) agrees with triangulate_points byte for byte."""
    libdir = os.path.join(ROOT, "apex_camera_models_b200", "lib")
    exe = str(tmp_path / "triangulate_test")
    subprocess.run(["/usr/bin/g++", "-std=c++17", "-O1", "-Wall", "-Werror", "-pthread", "-I", os.path.join(ROOT, "include"),
                    os.path.join(ROOT, "tests", "cpp", "triangulate_test.cpp"), "-o", exe, "-L", libdir, "-lacm", f"-Wl,-rpath,{libdir}"],
                   check=True)
    ca, cb = dict(cameras["kannala_brandt"]), dict(cameras["double_sphere"])
    ga, gb = gpu_model(acm, ctx, ca), gpu_model(acm, ctx, cb)
    uv1, uv2, _ = _dataset(O, oracle_model(O, ca), oracle_model(O, cb), 3001, 0x7121A7EA)
    n = len(uv1)
    inp, outp = tmp_path / "in.bin", tmp_path / "out.bin"
    np.concatenate([ROT.ravel(), T_BASE, [float(n)], uv1.ravel(), uv2.ravel()]).tofile(inp)
    r = subprocess.run([exe, str(inp), str(outp)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    assert "TRIANGULATE_TEST_OK" in r.stdout
    raw = outp.read_bytes()
    pts, err, st = acm.triangulate_points(ga, gb, ROT, T_BASE, uv1, uv2)
    assert raw[:24 * n] == pts.tobytes() and raw[24 * n:40 * n] == err.tobytes() and raw[40 * n:] == st.tobytes()
