"""GPU parity tests proper: the CUDA path (through the C ABI of include/acm.h) against the CPU
oracle on the same seeded inputs, against the committed golden fixtures, and at BASELINE sizes
through size-independent properties.

Bars (BASELINE.json north_star): status masks, kept sets, remap indices and output bytes are
bit-exact; f64 values within 1e-9 relative; the f32-I/O path within 1e-4 px (or half an f32 ulp
of the coordinate where that is larger, SURVEY.md section 7).
"""
import os
import ctypes as C

import numpy as np
import pytest

from conftest import load_golden, oracle_model

pytestmark = pytest.mark.gpu

MODELS = ["pinhole", "rad_tan", "kannala_brandt", "ucm", "eucm", "double_sphere", "fov"]
EXACT = {"pinhole", "rad_tan", "ucm", "eucm", "double_sphere"}  # project: +,-,*,/,sqrt only => bit-exact values
# unproject: everything a validity test depends on is evaluated exactly (status bytes bit-exact); the
# arithmetic AFTER the last test (normalisation, final quotients / roots) uses <= 2 ulp reciprocals, so
# the values of the arithmetic-only models agree within a few ulp instead of bit for bit (pinhole: still
# bit for bit).  The bar of the contract is 1e-9 relative; these kernels are held to 1e-13.
UNPROJECT_EXACT = {"pinhole"}
ULP_RTOL, ULP_ATOL = 1e-13, 1e-13
# RadTan unproject runs a contracted Newton iteration on cameras that pass the host-side gate: its iterate follows the
# reference's to ~1e-14 (every stopping decision is the reference's, see test_rad_tan_contracted_newton_...)
NEWTON_RTOL = 1e-11
UNIFIED = {"ucm", "eucm", "double_sphere"}
RTOL = 1e-9


@pytest.fixture(scope="module")
def acm():
    import apex_camera_models_b200 as m
    return m


@pytest.fixture(scope="module")
def ctx(acm):
    c = acm.Context(0)
    yield c
    c.close()


def gpu_model(acm, ctx, cam):
    cls = acm.MODEL_CLASSES[cam["model_id"]]
    return cls(acm.Intrinsics(*cam["params"][:4]), acm.Resolution(cam["width"], cam["height"]), cam["params"][4:], ctx=ctx)


def cone(name):
    return np.cos(np.deg2rad(40.0 if name in ("pinhole", "rad_tan") else 100.0))


def assert_close_where_valid(a, b, ok, name, exact_names=EXACT):
    assert np.array_equal(np.isnan(a), np.isnan(b))
    if name in exact_names:
        assert np.array_equal(a[ok], b[ok]), f"{name}: values are not bit-identical"
    elif name in EXACT:  # arithmetic-only model on the unproject side: a few ulp
        rt = NEWTON_RTOL if name == "rad_tan" else ULP_RTOL
        assert np.allclose(a[ok], b[ok], rtol=rt, atol=ULP_ATOL), f"{name}: {np.nanmax(np.abs(a[ok] - b[ok]))}"
    else:
        assert np.allclose(a[ok], b[ok], rtol=RTOL, atol=1e-13)


# ------------------------------------------------------------------ project / unproject ----------
@pytest.mark.parametrize("name", MODELS)
def test_project_matches_oracle(acm, ctx, O, cameras, name):
    cam = cameras[name]
    m, om = gpu_model(acm, ctx, cam), oracle_model(O, cam)
    n = 100_003  # ragged: not a multiple of the 2-point packets
    xyz = O.synth_points3(0xACE50002, 0, n, cone(name), True)
    uv, st = m.project_batch(xyz)
    uvo, sto = O.project(om, xyz)
    assert np.array_equal(st, sto), "status mask must be bit-exact"
    assert len(np.unique(sto)) >= 2
    assert_close_where_valid(uv, uvo, sto == 0, name)


@pytest.mark.parametrize("name", MODELS)
def test_unproject_matches_oracle(acm, ctx, O, cameras, name):
    cam = cameras[name]
    m, om = gpu_model(acm, ctx, cam), oracle_model(O, cam)
    n = 100_003
    px = O.synth_pixels(0xACE50002, 0, n, cam["width"] * 1.05, cam["height"] * 1.05)  # some outside the image
    px[:4] = [[0.0, 0.0], [cam["params"][2], cam["params"][3]], [cam["width"], 1.0], [cam["params"][2] + 0.5e-6 * cam["params"][0], cam["params"][3]]]
    ray, st = m.unproject_batch(px)
    rayo, sto = O.unproject(om, px)
    assert np.array_equal(st, sto)
    assert_close_where_valid(ray, rayo, sto == 0, name, UNPROJECT_EXACT)


@pytest.mark.parametrize("name", MODELS)
def test_fused_round_trip_matches_oracle(acm, ctx, O, cameras, name):
    """BASELINE config 2: project -> unproject in one kernel == oracle project, then oracle unproject."""
    cam = cameras[name]
    m, om = gpu_model(acm, ctx, cam), oracle_model(O, cam)
    n = 65_537
    xyz = O.synth_points3(0xACE50002, 3, n, cone(name), True)
    uv, ray, sp, su = m.round_trip_batch(xyz)
    uvo, spo = O.project(om, xyz)
    assert np.array_equal(sp, spo)
    assert_close_where_valid(uv, uvo, spo == 0, name)
    ok = spo == 0
    rayo, suo = O.unproject(om, uv[ok])  # unproject what the device projected (KB / FOV differ in the last ulps)
    assert np.array_equal(su[ok], suo) and np.array_equal(su[~ok], spo[~ok])
    good = np.zeros(n, bool); good[np.flatnonzero(ok)[suo == 0]] = True
    assert_close_where_valid(ray[ok], rayo, suo == 0, name, UNPROJECT_EXACT)
    assert np.all(np.isnan(ray[~good]))
    # the direction comes back (the sample UCM / EUCM cameras have alpha > 1, for which the reference's
    # unproject is not the exact inverse: ucm.rs:614-616 uses 1e-4 at one point, tests/ use dot > 0.99)
    d = xyz[good] / np.linalg.norm(xyz[good], axis=1, keepdims=True)
    if name in ("ucm", "eucm"):
        assert np.min(np.sum(ray[good] * d, axis=1)) > 0.99
    else:
        assert np.max(np.abs(ray[good] - d)) < 1e-5


@pytest.mark.parametrize("name", sorted(EXACT))
def test_unproject_ieee_is_bit_identical_on_random_cameras(acm, ctx, O, cameras, name):
    """acm_unproject_ieee: the three rewrites in the decision part of unproject -- (u - cx) / fx through the correctly
    rounded reciprocal, RadTan's four divisions through one reciprocal, sqrt(s) < t as s < S -- are bit-IDENTICAL to the
    reference's IEEE operations: with IEEE tails the rays of the arithmetic-only models equal the oracle's bit for bit,
    on the sample camera and on 24 random cameras (200 k pixels each, in and around the image, incl. the principal point)."""
    rng = np.random.default_rng(0xB17 + MODELS.index(name))
    cams = [cameras[name]] + list(_random_cameras(name, rng, 24))
    for k, cam in enumerate(cams):
        m, om = gpu_model(acm, ctx, cam), oracle_model(O, cam)
        Wp, Hp = (cam["width"] or 800), (cam["height"] or 600)
        n = 200_003
        px = O.synth_pixels(0xACE50007, 1000 * k, n, Wp * 1.2, Hp * 1.2) - [0.1 * Wp, 0.1 * Hp]
        px[3::89] = cam["params"][2:4]
        px[5::97, 0] = cam["params"][2]            # u == cx: zero numerators take the division's slow path
        ray, st = m.unproject_batch_ieee(px)
        rayo, sto = O.unproject(om, px, nthreads=8)
        assert np.array_equal(st, sto), (name, cam["params"])
        assert np.array_equal(np.isnan(ray), np.isnan(rayo))
        fin = (sto == 0) & ~np.isnan(rayo).any(axis=1)
        assert fin.sum() > 1000 or k > 0
        assert np.array_equal(ray[fin], rayo[fin]), (name, cam["params"], np.abs(ray[fin] - rayo[fin]).max())
        # and the default (fast-tail) entry point takes the same decisions
        _, st2 = m.unproject_batch(px)
        assert np.array_equal(st2, sto)


def test_kb_contracted_newton_matches_reference_loop(acm, ctx, O, cameras):
    """Kannala-Brandt unproject: cameras that pass the host-side convergence proof run a contracted Newton iteration,
    the others the IEEE loop (acm_camera_fast_unproject tells which).  Both must give the oracle's status bytes bit for bit
    and its rays within 1e-9 -- on the sample camera at two scales, mild random cameras (fast path) and wild ones (IEEE)."""
    import ctypes as C
    from apex_camera_models_b200 import _native as N
    rng = np.random.default_rng(0xCB)
    base = cameras["kannala_brandt"]
    cams = [base, dict(base, params=[8 * v for v in base["params"][:4]] + base["params"][4:], width=4096, height=4096)]
    for _ in range(10):   # mild distortion: must take the contracted path
        cams.append(dict(base, params=base["params"][:4] + list(rng.uniform(-4e-3, 4e-3, 4) * [1, 0.5, 0.5, 0.1]), width=640, height=480))
    for _ in range(6):    # wild distortion (incl. non-monotone theta_d): IEEE loop, NumericalError pixels
        cams.append(dict(base, params=base["params"][:4] + list(rng.uniform(-0.6, 0.6, 4)), width=640, height=480))
    cams.append(dict(cameras["kannala_brandt_inline"]))
    fast = 0
    for k, cam in enumerate(cams):
        m, om = gpu_model(acm, ctx, cam), oracle_model(O, cam)
        blk = m.camera_block()
        flag = N.lib.acm_camera_fast_unproject(C.byref(blk))
        assert flag in (0, 1)
        fast += flag
        if k < 2:
            assert flag == 1, cam["params"]   # the reference's sample camera, at both scales
        W, H = cam["width"], cam["height"]
        n = 300_001
        px = O.synth_pixels(0xACE5000B, 977 * k, n, W * 1.1, H * 1.1) - [0.05 * W, 0.05 * H]
        cx, cy, fx = cam["params"][2], cam["params"][3], cam["params"][0]
        px[1::53] = [cx, cy]                                    # ru == 0
        px[2::59] = [cx + 0.5e-6 * fx, cy]                      # 0 < ru <= 1e-6: NumericalError
        px[3::61] = [cx + 1.000001e-6 * fx, cy]                 # just above the hole
        ray, st = m.unproject_batch(px)
        rayo, sto = O.unproject(om, px, nthreads=8)
        assert np.array_equal(st, sto), (k, cam["params"], np.flatnonzero(st != sto)[:5])
        ok = sto == 0
        assert np.array_equal(np.isnan(ray), np.isnan(rayo))
        fin = ok & ~np.isnan(rayo).any(axis=1)
        assert np.allclose(ray[fin], rayo[fin], rtol=RTOL, atol=1e-12), (k, np.abs(ray[fin] - rayo[fin]).max())
    assert 9 <= fast < len(cams)   # both loops are exercised


def test_rad_tan_contracted_newton_takes_the_reference_decisions(acm, ctx, O, cameras):
    """RadTan unproject (rad_tan.rs:401-524) returns the Newton iterate at which `error.norm() < 1e-6` or
    `delta.norm() < 1e-6` fires -- typically ~1e-9 from the root -- so the GPU must stop at the same iterate as the
    reference: a different decision moves the ray by up to 1e-6.  Cameras that pass the host-side gate run a contracted
    (FMA, one reciprocal) iteration whose decisions carry a guard band and fall back to the IEEE loop inside it; the
    others keep the IEEE loop.  Both: status bytes bit for bit, rays within 1e-11 of the reference's iterate -- on the
    sample camera, on mild random cameras (contracted), on strong distortion that folds over (IEEE, NumericalError
    pixels), and on pixels placed so that a stopping test sits right at its threshold."""
    import ctypes as C
    from apex_camera_models_b200 import _native as N
    rng = np.random.default_rng(0x7A)
    base = cameras["rad_tan"]
    cams = [base, dict(base, params=[4 * v for v in base["params"][:4]] + base["params"][4:], width=4 * base["width"], height=4 * base["height"])]
    for _ in range(10):   # mild distortion: contracted path
        cams.append(dict(base, params=base["params"][:4] + [float(rng.uniform(-0.3, 0.1)), float(rng.uniform(-0.05, 0.1)), float(rng.uniform(-1e-3, 1e-3)),
                                                             float(rng.uniform(-1e-3, 1e-3)), float(rng.uniform(-0.02, 0.02))]))
    for _ in range(6):    # strong distortion on a wide image: the mapping folds over, Newton stalls or meets singular Jacobians
        cams.append(dict(base, params=[0.3 * base["params"][0], 0.3 * base["params"][1]] + base["params"][2:4] +
                                      [float(rng.uniform(-0.6, -0.3)), float(rng.uniform(-0.2, 0.3)), 0.0, 0.0, float(rng.uniform(-0.1, 0.1))]))
    fast = 0
    for k, cam in enumerate(cams):
        m, om = gpu_model(acm, ctx, cam), oracle_model(O, cam)
        blk = m.camera_block()
        flag = N.lib.acm_camera_fast_unproject(C.byref(blk))
        assert flag in (0, 1)
        fast += flag
        if k < 2:
            assert flag == 1, cam["params"]   # the reference's sample camera, at both scales
        W, H = cam["width"], cam["height"]
        n = 300_001
        px = O.synth_pixels(0xACE5000C, 977 * k, n, W * 1.1, H * 1.1) - [0.05 * W, 0.05 * H]
        cx, cy, fx, fy = cam["params"][2], cam["params"][3], cam["params"][0], cam["params"][1]
        px[1::53] = [cx, cy]                                    # the start already satisfies the error test
        # targets at distance ~1e-6 / |k1| ... from the centre: the first error norm sits around its 1e-6 threshold
        t = np.geomspace(1e-3, 3e-2, len(px[2::59]))
        px[2::59] = np.stack([cx + fx * t, cy + fy * 0.5 * t], axis=1)
        ray, st = m.unproject_batch(px)
        rayo, sto = O.unproject(om, px, nthreads=8)
        assert np.array_equal(st, sto), (k, cam["params"], np.flatnonzero(st != sto)[:5])
        ok = sto == 0
        assert np.array_equal(np.isnan(ray), np.isnan(rayo))
        assert np.allclose(ray[ok], rayo[ok], rtol=NEWTON_RTOL, atol=1e-13), (k, flag, np.abs(ray[ok] - rayo[ok]).max())
        # the fused round trip takes the same path
        xyz = O.synth_points3(0xACE50002, 31 * k, 50_001, cone("rad_tan"), True)
        uv, ray2, sp, su = m.round_trip_batch(xyz)
        uvo, spo = O.project(om, xyz)
        assert np.array_equal(sp, spo)
        good = spo == 0
        rayo2, suo = O.unproject(om, uvo[good])
        assert np.array_equal(su[good], suo)
        fin = suo == 0
        assert np.allclose(ray2[good][fin], rayo2[fin], rtol=NEWTON_RTOL, atol=1e-13)
    assert 9 <= fast < len(cams), fast   # both loops are exercised


def _random_cameras(name, rng, count):
    """Random parameter sets that exercise every branch of the validity tests (alpha on both sides
    of 0.5, alpha > 1 for UCM/EUCM, negative xi, w near its bounds, KB without a resolution, ...)."""
    out = []
    for k in range(count):
        W, H = int(rng.integers(64, 2000)), int(rng.integers(64, 1500))
        f = float(rng.uniform(0.2, 1.5) * W)
        intr = [f, f * float(rng.uniform(0.97, 1.03)), W * float(rng.uniform(0.4, 0.6)), H * float(rng.uniform(0.4, 0.6))]
        if name == "pinhole":
            d = []
        elif name == "rad_tan":
            d = [float(rng.uniform(-0.4, 0.2)), float(rng.uniform(-0.1, 0.2)), float(rng.uniform(-2e-3, 2e-3)), float(rng.uniform(-2e-3, 2e-3)), float(rng.uniform(-0.05, 0.05))]
        elif name == "kannala_brandt":
            d = [float(rng.uniform(-0.05, 0.05)), float(rng.uniform(-0.02, 0.02)), float(rng.uniform(-0.01, 0.01)), float(rng.uniform(-0.002, 0.002))]
            if k % 4 == 3:
                W = H = 0  # resolution unset: unproject skips the bounds test (kannala_brandt.rs:447-455)
        elif name == "ucm":
            d = [float(rng.choice([rng.uniform(0.05, 0.5), rng.uniform(0.5, 0.99), rng.uniform(1.0, 1.3), 0.5]))]
        elif name == "eucm":
            d = [float(rng.choice([rng.uniform(0.05, 0.5), rng.uniform(0.5, 0.99), rng.uniform(1.0, 1.2), 0.5])), float(rng.uniform(0.3, 2.5))]
        elif name == "double_sphere":
            d = [float(rng.choice([rng.uniform(0.05, 0.5), rng.uniform(0.5, 1.0), 0.5, 1.0])), float(rng.uniform(-0.6, 0.9))]
        else:  # fov
            d = [float(rng.choice([rng.uniform(0.05, 3.0), 1e-9, 3.0]))]
        out.append({"model_id": MODELS.index(name), "params": intr + d, "width": W, "height": H})
    return out


@pytest.mark.parametrize("name", MODELS)
def test_random_cameras_project_unproject(acm, ctx, O, cameras, name):
    """Same bars as above on 24 random cameras per model: masks bit-exact, values bit-exact for the
    arithmetic-only models and within 1e-9 for KB / FOV, fused round trip consistent."""
    rng = np.random.default_rng(0xACE5 + MODELS.index(name))
    n = 20_003
    for k, cam in enumerate(_random_cameras(name, rng, 24)):
        m, om = gpu_model(acm, ctx, cam), oracle_model(O, cam)
        xyz = O.synth_points3(0xACE50002, 1000 * k, n, float(np.cos(np.deg2rad(rng.uniform(30.0, 120.0)))), True)
        xyz[5::97] *= 1e-3      # points very close to the camera (den < 1e-3 branches)
        xyz[7::101, :2] = 0.0   # on the optical axis (r == 0 branches of KB / FOV)
        uv, st = m.project_batch(xyz)
        uvo, sto = O.project(om, xyz)
        assert np.array_equal(st, sto), (name, cam["params"])
        assert_close_where_valid(uv, uvo, sto == 0, name)
        Wp, Hp = (cam["width"] or 800), (cam["height"] or 600)
        px = O.synth_pixels(0xACE50002, 1000 * k, n, Wp * 1.2, Hp * 1.2) - [0.1 * Wp, 0.1 * Hp]   # in and around the image
        px[3::89] = cam["params"][2:4]                                                            # the principal point itself
        px[4::89] = [cam["params"][2] + 0.5e-6 * cam["params"][0], cam["params"][3]]             # KB's 1e-6 hole
        ray, st = m.unproject_batch(px)
        rayo, sto = O.unproject(om, px)
        assert np.array_equal(st, sto), (name, cam["params"])
        # DS / EUCM can return NaN rays with status Ok (sqrt of a slightly negative radicand): NaN patterns must match too
        assert np.array_equal(np.isnan(ray), np.isnan(rayo))
        fin = (sto == 0) & ~np.isnan(rayo).any(axis=1)
        if name in UNPROJECT_EXACT:
            assert np.array_equal(ray[fin], rayo[fin])
        elif name in EXACT:
            assert np.allclose(ray[fin], rayo[fin], rtol=NEWTON_RTOL if name == "rad_tan" else ULP_RTOL, atol=ULP_ATOL), np.nanmax(np.abs(ray[fin] - rayo[fin]))
        else:
            assert np.allclose(ray[fin], rayo[fin], rtol=RTOL, atol=1e-13)


@pytest.mark.parametrize("name", MODELS)
def test_random_cameras_linearize_and_jacobian(acm, ctx, O, cameras, name):
    """Stress version of test_linearize_matches_oracle: random cameras, points on the axis and 1e-3
    from the camera.  The bar is 2e-8 here instead of 1e-9: the published derivatives contain
    d - z (UCM / EUCM) and d2 - g (DS), which cancel for near-axis points, so a 1-ulp difference in
    sqrt (IEEE in the oracle, MUFU + Newton on the device) is amplified by z / (d - z) in those
    columns -- in both implementations alike.  FOV with w -> 0 is left out for the same reason
    (da/(r w) - a/(r w^2) cancels to 1e-8 at w = 1e-9)."""
    rng = np.random.default_rng(0xBEEF + MODELS.index(name))
    n = 5_001
    STRESS_RTOL = 2e-8
    for k, cam in enumerate(_random_cameras(name, rng, 8)):
        if cam["width"] == 0:
            cam["width"], cam["height"] = 640, 480
        if name == "fov" and cam["params"][4] < 0.05:
            cam["params"][4] = 0.05
        m, om = gpu_model(acm, ctx, cam), oracle_model(O, cam)
        xyz = O.synth_points3(0xACE50003, 500 * k, n, float(np.cos(np.deg2rad(rng.uniform(30.0, 110.0)))), True)
        obs, _ = O.project(om, xyz)
        obs = np.where(np.isnan(obs), 3.0, obs) + rng.normal(0.0, 0.5, (n, 2))
        for kind in ((0, 1) if name in UNIFIED else (0,)):
            cost = acm.OptimizationCost(m, xyz, obs, residual_kind=kind)
            H, g, c, nv = cost.linearize()
            Ho, go, co, nvo = O.linearize(om, kind, xyz, obs, nthreads=4)
            assert nv == nvo, (name, cam["params"])
            dg = np.sqrt(np.abs(np.diag(Ho))) + 1e-300
            assert np.max(np.abs(H - Ho) / np.outer(dg, dg)) < STRESS_RTOL, (name, kind, cam["params"])
            assert np.max(np.abs(g - go) / (dg * np.sqrt(2 * co) + 1e-300)) < STRESS_RTOL
            assert abs(c - co) <= RTOL * co
            cost.free()


def _device_map(acm, ctx, fn, a, dtype):
    """fn (a bound project_batch / unproject_batch) on a device `Points` copy of `a` -> (numpy values, status bytes)."""
    n = a.shape[0]
    src = acm.Points.from_numpy(ctx, a, dtype)
    dst, d_st = fn(src)
    out, st = dst.numpy(), np.empty(n, np.uint8)
    ctx.d2h(st, d_st); ctx.sync()
    ctx.device_free(d_st); src.free(); dst.free()
    return out, st


CHUNK = 4 << 20   # points per staged chunk of the host upload / download (kChunkPoints)


@pytest.mark.parametrize("n", [0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 255, 256, 257, 511, 513, 2047, 2048, 2049, 2 * CHUNK + 3])
def test_edge_sizes(acm, ctx, O, cameras, n):
    """Host f64 input: up to ACM_SMALL_BATCH = 2048 points the small-map kernel, above it the batch kernels behind a
    chunked upload / download (2 * 4 Mi + 3: three chunks, the last of 3 points).  Device `Points` input (n <= 2049) calls
    the batch kernels directly, in f64 (2-point packets) and f32 (4-point packets), so their scalar tails and the
    first-trip prefetch are tested at small n; the f32 leg has the bars of test_f32_io_path."""
    from apex_camera_models_b200 import _native as N
    nt = min(os.cpu_count() or 1, 16)
    for name in ("double_sphere", "kannala_brandt"):
        cam = cameras[name]
        m, om = gpu_model(acm, ctx, cam), oracle_model(O, cam)
        xyz = O.synth_points3(11, 0, n, cone(name), True).reshape(n, 3)
        uv, st = m.project_batch(xyz)
        uvo, sto = O.project(om, xyz, nt)
        assert uv.shape == (n, 2) and np.array_equal(st, sto)
        assert_close_where_valid(uv, uvo, sto == 0, name)
        px = O.synth_pixels(12, 0, n, cam["width"], cam["height"]).reshape(n, 2)
        ray, st = m.unproject_batch(px)
        rayo, sto = O.unproject(om, px, nt)
        assert ray.shape == (n, 3) and np.array_equal(st, sto)
        assert_close_where_valid(ray, rayo, sto == 0, name, UNPROJECT_EXACT)
        if not 0 < n <= 2049:
            continue
        uv, st = _device_map(acm, ctx, m.project_batch, xyz, N.F64)
        uvo, sto = O.project(om, xyz)
        assert np.array_equal(st, sto)
        assert_close_where_valid(uv, uvo, sto == 0, name)
        ray, st = _device_map(acm, ctx, m.unproject_batch, px, N.F64)
        rayo, sto = O.unproject(om, px)
        assert np.array_equal(st, sto)
        assert_close_where_valid(ray, rayo, sto == 0, name, UNPROJECT_EXACT)
        x32 = xyz.astype(np.float32).astype(np.float64)
        uv, st = _device_map(acm, ctx, m.project_batch, x32, N.F32)
        uvo, sto = O.project(om, x32)
        assert np.array_equal(st, sto)
        ok = sto == 0
        tol = np.maximum(1e-4, 0.5 * np.spacing(np.abs(uvo[ok]).astype(np.float32)).astype(np.float64))
        assert np.all(np.abs(uv[ok] - uvo[ok]) <= tol) and np.all(np.isnan(uv[~ok]))
        p32 = px.astype(np.float32).astype(np.float64)
        ray, st = _device_map(acm, ctx, m.unproject_batch, p32, N.F32)
        rayo, sto = O.unproject(om, p32)
        assert np.array_equal(st, sto)
        assert np.all(np.abs(ray[sto == 0] - rayo[sto == 0]) <= 1e-7) and np.all(np.isnan(ray[sto != 0]))


@pytest.mark.parametrize("name", MODELS)
def test_f32_io_path(acm, ctx, O, cameras, name):
    """f32 I/O, f64 math, one final rounding: compare with the f64 oracle evaluated on the same
    f32-rounded inputs.  Tolerance max(1e-4 px, 0.5 ulp_f32(coordinate))."""
    from apex_camera_models_b200 import _native as N
    cam = cameras[name]
    m, om = gpu_model(acm, ctx, cam), oracle_model(O, cam)
    n = 50_001
    xyz = O.synth_points3(0xACE50002, 7, n, cone(name), True).astype(np.float32).astype(np.float64)
    uv, st = m.project_batch(xyz, dtype=N.F32)
    uvo, sto = O.project(om, xyz)
    assert np.array_equal(st, sto)
    ok = sto == 0
    tol = np.maximum(1e-4, 0.5 * np.spacing(np.abs(uvo[ok]).astype(np.float32)).astype(np.float64))
    assert np.all(np.abs(uv[ok] - uvo[ok]) <= tol)
    px = O.synth_pixels(3, 0, n, cam["width"], cam["height"]).astype(np.float32).astype(np.float64)
    ray, st = m.unproject_batch(px, dtype=N.F32)
    rayo, sto = O.unproject(om, px)
    assert np.array_equal(st, sto)
    assert np.all(np.abs(ray[sto == 0] - rayo[sto == 0]) <= 1e-7)


def test_synthetic_generators_are_bit_identical(acm, ctx, O):
    from apex_camera_models_b200 import _native as N
    lib = N.lib
    n = 70_001
    for cosmax, adv, i0 in [(cone("kb"), 1, 0), (cone("pinhole"), 0, 12345), (np.cos(np.deg2rad(85.0)), 0, 10**9)]:
        p = acm.Points(ctx, 3, n)
        ctx.check(lib.acm_synth_points3(ctx.handle, 0xACE50003, i0, cosmax, adv, p.handle))
        assert np.array_equal(p.numpy(), O.synth_points3(0xACE50003, i0, n, cosmax, bool(adv)))
    q = acm.Points(ctx, 2, n)
    ctx.check(lib.acm_synth_pixels(ctx.handle, 5, 17, 752.0, 480.0, q.handle))
    assert np.array_equal(q.numpy(), O.synth_pixels(5, 17, n, 752.0, 480.0))
    nb = 100_003
    d = ctx.device_alloc(nb)
    ctx.check(lib.acm_synth_bytes(ctx.handle, 0xACE50005, 3, C.c_void_p(d), nb))
    out = np.empty(nb, np.uint8); ctx.d2h(out, d); ctx.sync(); ctx.device_free(d)
    assert np.array_equal(out, O.synth_bytes(0xACE50005, 3, nb))


def test_golden_vectors_on_gpu(acm, ctx, cameras):
    """tests/golden/restated_kats.json and the OpenCV cross-check, through the CUDA path."""
    kat = load_golden("restated_kats.json")
    for row in kat["project_unproject"]:
        m = gpu_model(acm, ctx, cameras[row["camera"]])
        uv = m.project(row["point"])
        if row["camera"] in EXACT:
            assert uv.tolist() == row["uv"]
        else:
            assert np.allclose(uv, row["uv"], rtol=1e-13)
        if row.get("ray"):
            assert np.allclose(m.unproject(uv), row["ray"], rtol=1e-12, atol=1e-16)
    cv = load_golden("opencv_cross.json")
    for name in ("kannala_brandt", "kannala_brandt_inline", "rad_tan", "pinhole"):
        cam = dict(cameras[name]); cam["width"] = cam["height"] = 100000  # OpenCV has no bounds test
        m = gpu_model(acm, ctx, cam)
        pts = np.array(cv[name]["points"])
        if name in ("rad_tan", "pinhole"):
            # shift the principal point so that every projection is inside the (huge) image
            cam["params"] = list(cam["params"]); cam["params"][2] += 50000.0; cam["params"][3] += 50000.0
            m = gpu_model(acm, ctx, cam)
            ref = np.array(cv[name]["uv"]) + 50000.0
        else:
            ref = np.array(cv[name]["uv"])
        uv, st = m.project_batch(pts)
        assert np.all(st == 0) and np.max(np.abs(uv - ref)) < 1e-9


def test_pinhole_doc_test_numbers_on_gpu(acm, ctx):
    """pinhole.rs:145-164: the reference's own numeric known answer, through the scalar trait call and the batch kernel."""
    m = acm.PinholeModel.new([500.0, 500.0, 320.0, 240.0], ctx=ctx)
    m.resolution = acm.Resolution(640, 480)
    uv = m.project([0.1, 0.2, 1.0])
    assert abs(uv[0] - 370.0) < 1e-6 and abs(uv[1] - 340.0) < 1e-6
    uvb, st = m.project_batch(np.tile([0.1, 0.2, 1.0], (5000, 1)))
    assert np.all(st == 0) and np.all(uvb == uv)


def test_reference_unit_tests_through_the_trait_surface(acm, ctx, cameras):
    """The reference's error-classification tests (double_sphere.rs:782-801, kannala_brandt.rs:948-974,
    fov.rs:648-666, tests/projection_accuracy.rs) through CameraModel.project / unproject."""
    ds = gpu_model(acm, ctx, cameras["double_sphere"])
    kb = gpu_model(acm, ctx, cameras["kannala_brandt_inline"])
    fov = gpu_model(acm, ctx, cameras["fov"])
    for m in (ds, gpu_model(acm, ctx, cameras["ucm"]), gpu_model(acm, ctx, cameras["eucm"]), kb):
        with pytest.raises(acm.PointIsOutSideImage):
            m.project([0.1, 0.2, -1.0])
    with pytest.raises(acm.PointAtCameraCenter):
        fov.project([0.1, 0.2, -1.0])
    with pytest.raises(acm.PointIsOutSideImage):
        ds.project([0.0, 0.0, 0.0])
    for m in (kb, fov):
        with pytest.raises(acm.PointAtCameraCenter):
            m.project([0.0, 0.0, 0.0])
    with pytest.raises(acm.PointIsOutSideImage):
        kb.unproject([-1.0, 100.0])
    pin = acm.PinholeModel.new([500.0, 500.0, 320.0, 240.0], ctx=ctx)
    pin.resolution = acm.Resolution(640, 480)
    with pytest.raises(acm.PointIsOutSideImage):
        pin.unproject([-100.0, 100.0])
    with pytest.raises(acm.ProjectionOutSideImage):
        pin.project([10.0, 0.0, 1.0])
    for X in [(0.0, 0.0, 1.0), (0.2, 0.1, 1.5), (-0.1, -0.2, 2.0)]:
        ray = pin.unproject(pin.project(X))
        assert abs(float(np.dot(np.array(X) / np.linalg.norm(X), ray)) - 1.0) < 1e-6
    # round trips with the reference's tolerances
    for name, X, tol in [("double_sphere", (0.5, -0.3, 2.0), 1e-6), ("rad_tan", (0.5, -0.3, 2.0), 1e-6),
                         ("kannala_brandt_inline", (0.1, 0.2, 1.0), 1e-5), ("ucm", (0.1, 0.1, 3.0), 1e-4),
                         ("eucm", (0.1, 0.1, 3.0), 1e-4), ("fov", (0.1, 0.1, 3.0), 1e-4)]:
        m = gpu_model(acm, ctx, cameras[name])
        ray = m.unproject(m.project(X))
        assert np.all(np.abs(ray - np.array(X) / np.linalg.norm(X)) < tol)


# ------------------------------------------------------------------ Jacobians / normal equations --
@pytest.mark.parametrize("name", MODELS)
def test_point_jacobian_matches_oracle_mpmath_and_differences(acm, ctx, O, cameras, name):
    """2x3 Jacobian w.r.t. the 3-D point (trait doc mod.rs:246-252): device vs oracle (1e-9), vs the mpmath
    50-digit differences of the model definitions, and vs central differences of the device's own project."""
    cam = cameras[name]
    m, om = gpu_model(acm, ctx, cam), oracle_model(O, cam)
    for n in (2002, 2003):   # even: the 2-point vector kernel; odd: the scalar one
        xyz = O.synth_points3(0xACE50002, 17, n, cone(name), True)
        xyz[::5, :2] *= 1e-9          # near the axis: KB r < EPS / FOV r^2 < sqrt(EPS) branches
        xyz[3::11, :2] = 0.0
        uv, J, st = m.project_point_jacobian_batch(xyz)
        assert J.shape == (n, 2, 3)
        uvo, Jo, sto = O.project_point_jacobian(om, xyz)
        assert_jacobians_match(uv, J, st, uvo, Jo, sto)
    rows = load_golden("mpmath_point_jacobians.json")[name]
    pts = np.array([r["point"] for r in rows])
    _, Jg, stg = m.project_point_jacobian_batch(pts)
    for k, r in enumerate(rows):
        assert stg[k] == 0
        assert np.allclose(Jg[k], np.array(r["J"]), rtol=1e-9, atol=1e-12)
    # central differences of the batch projection itself (smooth region only)
    good = np.flatnonzero((st == 0) & (np.hypot(xyz[:, 0], xyz[:, 1]) > 1e-2) & (xyz[:, 2] > 0.2))[:200]
    h = 1e-6
    for k in range(3):
        d = np.zeros(3); d[k] = h
        up, sp = m.project_batch(xyz[good] + d)
        um, sm = m.project_batch(xyz[good] - d)
        ok = (sp == 0) & (sm == 0)
        fd = (up - um) / (2 * h)
        scale = np.abs(J[good][ok]).max(axis=(1, 2))[:, None]
        assert np.max(np.abs(J[good][ok][:, :, k] - fd[ok]) / scale) < 1e-5
    # the trait-level spelling
    uv1, J1 = m.project(pts[0], compute_jacobian="point")
    assert J1.shape == (2, 3) and np.array_equal(J1, Jg[0])


@pytest.mark.parametrize("name", MODELS)
def test_project_jacobian_matches_oracle_and_mpmath(acm, ctx, O, cameras, name):
    cam = cameras[name]
    m, om = gpu_model(acm, ctx, cam), oracle_model(O, cam)
    for n in (4000, 4001):   # even: the 2-point vector kernel; odd: the scalar one
        xyz = O.synth_points3(0xACE50002, 99, n, cone(name), True)
        uv, J, st = m.project_jacobian_batch(xyz)
        assert J.shape == (n, 2, len(cam["params"]))
        uvo, Jo, sto = O.project_jacobian(om, xyz)
        assert_jacobians_match(uv, J, st, uvo, Jo, sto)
    rows = load_golden("mpmath_jacobians.json")[name]
    pts = np.array([r["point"] for r in rows])
    uv, J, st = m.project_jacobian_batch(pts)
    assert np.all(st == 0)
    for k, r in enumerate(rows):
        assert np.allclose(J[k], np.array(r["J"]), rtol=1e-9, atol=1e-12)
    u1, J1 = m.project(pts[0], compute_jacobian=True)  # README-era spelling
    assert np.array_equal(J1, J[0])


def assert_jacobians_match(uv, J, st, uvo, Jo, sto):
    """Every point against the oracle's batch Jacobian: status bytes bit-exact; where the projection succeeds, uv within
    1e-9 (atol 1e-13) and J within 1e-9 relative plus 1e-12 of the point's largest entry; where it fails, J = 0, uv NaN."""
    assert np.array_equal(st, sto), np.flatnonzero(st != sto)[:8]
    ok = sto == 0
    assert ok.sum() > len(st) // 4
    assert np.allclose(uv[ok], uvo[ok], rtol=RTOL, atol=1e-13)
    scale = np.abs(Jo[ok]).max(axis=(1, 2), keepdims=True)
    bad = (np.abs(J[ok] - Jo[ok]) > RTOL * np.abs(Jo[ok]) + 1e-12 * scale).any(axis=(1, 2))
    assert not bad.any(), np.flatnonzero(ok)[bad][:8]
    assert np.all(J[~ok] == 0.0) and np.all(np.isnan(uv[~ok]))


def _correspondences(O, om, name, n, seed=0xACE50003, noise=0.25):
    xyz = O.synth_points3(seed, 0, n, cone(name), True)
    uv, st = O.project(om, xyz)
    return xyz, np.where(np.isnan(uv), 1.0, uv) + noise


@pytest.mark.parametrize("name", MODELS)
def test_linearize_matches_oracle(acm, ctx, O, cameras, name):
    cam = cameras[name]
    m, om = gpu_model(acm, ctx, cam), oracle_model(O, cam)
    for n in (1, 2, 333, 100_003):
        xyz, obs = _correspondences(O, om, name, n)
        for kind in ((0, 1) if name in UNIFIED else (0,)):
            cost = acm.OptimizationCost(m, xyz, obs, residual_kind=kind)
            H, g, c, nv = cost.linearize()
            Ho, go, co, nvo = O.linearize(om, kind, xyz, obs, nthreads=4)
            assert nv == nvo
            dg = np.sqrt(np.abs(np.diag(Ho))) + 1e-300
            assert np.max(np.abs(H - Ho) / np.outer(dg, dg)) < RTOL       # relative to the natural scale of each entry
            assert np.max(np.abs(g - go) / (dg * np.sqrt(2 * co) + 1e-300)) < RTOL
            assert abs(c - co) <= RTOL * co
            assert np.array_equal(H, H.T)
            H2, g2, c2, _ = cost.linearize()                                # deterministic reduction
            assert np.array_equal(H, H2) and np.array_equal(g, g2) and c == c2
            cost.free()


def test_empty_and_degenerate_inputs(acm, ctx, O, cameras):
    """Empty point sets: zero normal equations, LM returns the (clamped) start, stats raise
    ZeroProjectionPoints like the reference (error_metrics.rs:83-85)."""
    ds = gpu_model(acm, ctx, cameras["double_sphere"])
    empty3, empty2 = np.zeros((0, 3)), np.zeros((0, 2))
    cost = acm.DoubleSphereOptimizationCost(ds, empty3, empty2)
    H, g, c, nv = cost.linearize()
    assert nv == 0 and c == 0.0 and not H.any() and not g.any()
    start = ds.params().copy()
    r = cost.optimize(bounds=None)
    assert np.array_equal(r.parameters, start) and r.n_valid == 0
    with pytest.raises(acm.ZeroProjectionPoints):
        acm.compute_reprojection_error(ds, empty3, empty2)
    uv, st = ds.project_batch(empty3)
    assert uv.shape == (0, 2) and st.shape == (0,)
    # every point invalid
    behind = np.tile([0.0, 0.0, -1.0], (5, 1))
    cost2 = acm.DoubleSphereOptimizationCost(ds, behind, np.zeros((5, 2)), residual_kind=0)
    H, g, c, nv = cost2.linearize()
    assert nv == 0 and c == 0.0 and not H.any()
    # NaN coordinates are invalid points, not poison (oracle: status != Ok -> skipped)
    pts = O.synth_points3(3, 0, 1001, cone("double_sphere"), False)
    om = oracle_model(O, cameras["double_sphere"])
    obs, _ = O.project(om, pts)
    obs += 0.1
    pts[::100] = np.nan
    cost3 = acm.DoubleSphereOptimizationCost(ds, pts, obs, residual_kind=0)
    H, g, c, nv = cost3.linearize()
    Ho, go, co, nvo = O.linearize(om, 0, pts, obs)
    assert nv == nvo == 1001 - 11 and np.all(np.isfinite(H)) and np.allclose(H, Ho, rtol=1e-9) and np.isclose(c, co, rtol=1e-9)


def test_linearize_host_entry_point(acm, ctx, O, cameras):
    """acm_linearize_host (the e2e path of bench.py: nalgebra-layout host buffers in, normal equations
    out) equals the device-buffer path; the cached device staging survives growing and shrinking n."""
    from apex_camera_models_b200 import _native as N
    cam = cameras["double_sphere"]
    m, om = gpu_model(acm, ctx, cam), oracle_model(O, cam)
    block = m.camera_block()
    for n in (1000, 9_000_001, 77, 0):
        xyz, obs = _correspondences(O, om, "double_sphere", n) if n else (np.zeros((0, 3)), np.zeros((0, 2)))
        ne = N.NormalEquations()
        ctx.check(N.lib.acm_linearize_host(ctx.handle, C.byref(block), 0, xyz.ctypes.data_as(C.c_void_p), obs.ctypes.data_as(C.c_void_p), n, C.byref(ne)))
        cost = acm.DoubleSphereOptimizationCost(m, xyz, obs, residual_kind=0)
        H, g, c, nv = cost.linearize()
        assert ne.n_valid == nv and ne.cost == c
        assert np.array_equal(np.array(ne.H[:36]).reshape(6, 6), H) and np.array_equal(np.array(ne.g[:6]), g)
        cost.free()


def test_linearize_argument_errors(acm, ctx, O, cameras):
    kb = gpu_model(acm, ctx, cameras["kannala_brandt"])
    xyz = np.zeros((4, 3)) + [0.1, 0.1, 1.0]
    with pytest.raises(acm.InvalidParams, match="Number of 2D and 3D points must match"):
        acm.KannalaBrandtOptimizationCost(kb, xyz, np.zeros((3, 2)))
    cost = acm.KannalaBrandtOptimizationCost(kb, xyz, np.zeros((4, 2)), residual_kind=1)
    with pytest.raises(acm.AcmError, match="algebraic residual"):
        cost.linearize()
    with pytest.raises(acm.InvalidParams):
        acm.DoubleSphereOptimizationCost(kb, xyz, np.zeros((4, 2)))


# ------------------------------------------------------------------ linear estimation + LM --------
def _kb450(O, cameras, n=500):
    c = cameras["kannala_brandt"]
    uv, xyz = O.sample_points(oracle_model(O, c), n)
    return c["params"][:4], uv, xyz


INITS = {"double_sphere": [0.5, 0.1], "ucm": [0.5], "eucm": [0.5, 1.0], "fov": [1.0], "kannala_brandt": [0.0] * 4, "rad_tan": [0.0] * 5}


@pytest.mark.parametrize("name", ["double_sphere", "ucm", "eucm", "fov", "kannala_brandt"])
def test_linear_estimation_matches_oracle(acm, ctx, O, cameras, name):
    intr, uv, xyz = _kb450(O, cameras)
    cam = {"model_id": cameras[name]["model_id"], "params": intr + INITS[name], "width": 512, "height": 512}
    m, om = gpu_model(acm, ctx, cam), oracle_model(O, cam)
    m.linear_estimation(xyz, uv)
    assert O.linear_estimation(om, xyz, uv) == 0
    got, ref = m.params(), om.params()
    if name == "kannala_brandt":
        assert np.allclose(got[4:], ref[4:], rtol=1e-7, atol=1e-12)  # 2N x 4 system, cond(A) ~ 1e5
    else:
        assert np.allclose(got, ref, rtol=1e-12, atol=0)
    if name in UNIFIED:
        assert abs(got[4] - load_golden("restated_kats.json")["lm_anchors_450"]["linear_alpha"]) < 1e-12


@pytest.mark.parametrize("source", ["kannala_brandt", "fov_exact", "fov_with_nan"])
def test_fov_grid_search_two_stage_matches_oracle(acm, ctx, O, cameras, source):
    """Inputs above 200 k points take the float pre-filter + exact shortlist path of the FOV grid
    search; the chosen w must be the oracle's (fov.rs:175-228 evaluates all 290 candidates)."""
    n = 250_000
    xyz = O.synth_points3(0xACE50009, 0, n, float(np.cos(np.deg2rad(80.0))), False)
    if source == "kannala_brandt":
        src = cameras["kannala_brandt"]
    else:  # data generated by a FOV camera with w on the grid: the minimum is ~0 px, the bound must still hold
        src = {"model_id": cameras["fov"]["model_id"], "params": cameras["kannala_brandt"]["params"][:4] + [0.93], "width": 512, "height": 512}
    uv, st = O.project(oracle_model(O, src), xyz)
    keep = st == 0
    xyz, uv = np.ascontiguousarray(xyz[keep]), np.ascontiguousarray(uv[keep])
    if source == "fov_with_nan":  # a non-finite error in the float stage forces the exact search over every candidate
        uv[1234, 0] = np.nan
    cam = {"model_id": cameras["fov"]["model_id"], "params": cameras["kannala_brandt"]["params"][:4] + [1.0], "width": 512, "height": 512}
    m, om = gpu_model(acm, ctx, cam), oracle_model(O, cam)
    m.linear_estimation(xyz, uv)
    assert O.linear_estimation(om, xyz, uv) == 0
    assert m.params()[4] == om.params()[4]
    if source != "kannala_brandt":
        assert m.params()[4] == 0.93


def test_linear_estimation_rad_tan_and_errors(acm, ctx, O, cameras):
    """tests/parameter_estimation.rs: 50 sampled points -> Ok and non-zero k; n=2 -> Err; mismatch -> Err."""
    c = cameras["rad_tan"]
    src = gpu_model(acm, ctx, c)
    uv, xyz = acm.sample_points(src, 50)
    est = acm.RadTanModel.new(c["params"][:4] + [0.0] * 5, ctx=ctx)
    est.resolution = src.get_resolution()
    est.linear_estimation(xyz, uv)
    assert any(abs(d) > 1e-10 for d in est.distortions)
    om = O.make_model(O.RADTAN, c["params"][:4] + [0.0] * 5, c["width"], c["height"])
    O.linear_estimation(om, xyz, uv)
    assert np.allclose(est.params(), om.params(), rtol=1e-8, atol=1e-12)
    assert est.p1 == 0.0 and est.p2 == 0.0
    uv2, xyz2 = acm.sample_points(src, 2)
    with pytest.raises(acm.InvalidParams):
        acm.RadTanModel.new(c["params"][:4] + [0.0] * 5, ctx=ctx).linear_estimation(xyz2, uv2)
    with pytest.raises(acm.InvalidParams, match="must match"):
        est.linear_estimation(xyz[:5], uv[:10])


CASES = [("double_sphere", 1, 1e-9), ("double_sphere", 0, 5e-8), ("ucm", 1, 1e-9), ("ucm", 0, 1e-9), ("eucm", 1, 1e-9),
         ("eucm", 0, 1e-9), ("fov", 0, 1e-9), ("kannala_brandt", 0, 1e-9), ("rad_tan", 0, None), ("pinhole", 0, 1e-9)]


@pytest.mark.parametrize("name,kind,rtol", CASES)
def test_lm_converges_to_oracle_parameters(acm, ctx, O, cameras, name, kind, rtol):
    """Config 1 (camera_converter --input-model kb --num-points 500 => 450 correspondences): same
    inits, bounds and tolerances as the converter, then re-run with tolerances far below the
    reference's so that both solvers sit at the minimiser.  cond(J^T J) ~ 2e9 for the DS pixel
    residual, hence its looser bound.  Pinhole has neither a linear estimation nor converter bounds: it starts at the
    KB intrinsics and runs unbounded.
    RadTan (rtol None) on this fisheye data is degenerate: points 6e-6 in front of the camera give (x/z)^2 up to 3e10, so
    its linear estimation solves a system of condition 2e28 -- any two implementations return different rounding noise
    there -- and the scaled J^T J at the minimiser has condition 5e16, so the minimiser is not determined in double.
    Both solvers start from the oracle's linear estimate; the converter's configuration (whose stopping tests sit a
    factor 6.8 above and 11 below cost_tolerance at the deciding iterations) must walk the oracle's trajectory, and the
    tight run must converge to the oracle's final cost."""
    intr, uv, xyz = _kb450(O, cameras)
    cam = {"model_id": cameras[name]["model_id"], "params": intr + INITS.get(name, []), "width": 512, "height": 512}
    m, om = gpu_model(acm, ctx, cam), oracle_model(O, cam)
    if name != "pinhole":
        m.linear_estimation(xyz, uv)
        O.linear_estimation(om, xyz, uv)
    if rtol is None:
        m.set_params(om.params())
    b = acm.CONVERTER_BOUNDS.get(m.MODEL_ID)
    lo, hi = (None, None) if b is None else ([x[0] for x in b], [x[1] for x in b])
    start = m.params().copy()
    cost = acm.OptimizationCost(m, xyz, uv, residual_kind=kind)
    # (1) the converter's own configuration: identical trajectory => identical stop
    r = cost.optimize()
    oo, ores = O.lm_solve(om, kind, xyz, uv, lo, hi)
    assert r.status == ores.status and r.iterations == ores.iterations and r.passes == ores.passes
    assert np.allclose(r.parameters, oo, rtol=1e-9)
    # (2) tight
    m.set_params(start)
    tight = acm.LevenbergMarquardtConfig(max_iterations=500, cost_tolerance=0.0, parameter_tolerance=1e-15, gradient_tolerance=0.0)
    r = cost.optimize(config=tight)
    ocfg = O.lm_default_config(); ocfg.max_iterations = 500; ocfg.cost_tolerance = 0.0; ocfg.parameter_tolerance = 1e-15; ocfg.gradient_tolerance = 0.0
    oo, ores = O.lm_solve(om, kind, xyz, uv, lo, hi, ocfg)
    assert r.converged and ores.status in (0, 1, 2)
    if rtol is not None:
        assert np.allclose(r.parameters, oo, rtol=rtol), np.abs(r.parameters - oo) / np.abs(oo)
    assert abs(r.final_cost - ores.final_cost) <= 1e-9 * ores.final_cost + 1e-18  # KB->KB is an exact fit: cost ~ 1e-22
    cost.free()


def test_lm_rank_deficient_normal_equations_take_the_retry_path(acm, ctx, O, cameras):
    """ADVICE round 1: the flag of the Cholesky-retry loop was re-armed while other warps still read it.
    (a) Every point on the optical axis and lambda0 = 0: the columns of fx, fy and the distortion are exactly zero, the
    damped system has exact zero pivots, every attempt fails and doubles a lambda that stays 0 -- the loop runs until
    max_iterations.  Deterministic, so GPU and oracle must agree on every counter, for one block (450 points) and
    many blocks (200 k points).
    (b) Kannala-Brandt data on a single cone angle: the four distortion columns are proportional, H is singular up to
    rounding, the first attempts fail and recover after a few doublings.  The pivots are rounding noise there, so only
    the outcome is compared (both converge to the same cost), not the trajectory."""
    for n in (450, 200_000):
        xyz = np.zeros((n, 3)); xyz[:, 2] = np.linspace(0.5, 3.0, n)
        uv = np.tile([250.0, 260.0], (n, 1))
        for name, kind, init in (("double_sphere", 0, [0.5, 0.1]), ("kannala_brandt", 0, [0.0] * 4), ("ucm", 1, [0.5])):
            cam = {"model_id": cameras[name]["model_id"], "params": [190.0, 190.0, 255.0, 257.0] + init, "width": 512, "height": 512}
            m, om = gpu_model(acm, ctx, cam), oracle_model(O, cam)
            cost = acm.OptimizationCost(m, xyz, uv, residual_kind=kind)
            r = cost.optimize(config=acm.LevenbergMarquardtConfig(max_iterations=60, lambda0=0.0), bounds=None)
            ocfg = O.lm_default_config(); ocfg.max_iterations = 60; ocfg.lambda0 = 0.0
            oo, ores = O.lm_solve(om, kind, xyz, uv, None, None, ocfg)
            assert (r.status, r.iterations, r.passes) == (ores.status, ores.iterations, ores.passes) == (3, 60, 1), (name, n)
            assert np.array_equal(r.parameters, oo) and np.array_equal(r.parameters, cam["params"]), name
            assert r.n_valid == n and np.isclose(r.final_cost, ores.final_cost, rtol=1e-12)
            cost.free()
    rng = np.random.default_rng(11)
    n = 50_000
    phi, rho, th = rng.uniform(0, 2 * np.pi, n), rng.uniform(0.5, 5.0, n), 0.7
    xyz = np.stack([rho * np.sin(th) * np.cos(phi), rho * np.sin(th) * np.sin(phi), rho * np.cos(th)], axis=1)
    truth = dict(cameras["kannala_brandt"])
    uv, st = O.project(oracle_model(O, truth), xyz)
    assert np.all(st == 0)
    cam = {"model_id": truth["model_id"], "params": list(np.array(truth["params"][:4]) * [1.01, 0.99, 1.0, 1.0]) + [0.0] * 4, "width": 512, "height": 512}
    m, om = gpu_model(acm, ctx, cam), oracle_model(O, cam)
    cost = acm.OptimizationCost(m, xyz, uv, residual_kind=0)
    r = cost.optimize(config=acm.LevenbergMarquardtConfig(max_iterations=200, lambda0=1e-30), bounds=None)
    ocfg = O.lm_default_config(); ocfg.max_iterations = 200; ocfg.lambda0 = 1e-30
    oo, ores = O.lm_solve(om, 0, xyz, uv, None, None, ocfg)
    assert r.converged and ores.status in (0, 1, 2)
    assert np.all(np.isfinite(r.parameters)) and r.final_cost <= 1e-6 * r.initial_cost and ores.final_cost <= 1e-6 * ores.initial_cost
    cost.free()


def test_lm_config4_ten_million_correspondences_matches_oracle(acm, ctx, O, cameras):
    """BASELINE config 4 (camera_converter.rs:378-447 at 10 M correspondences): KB -> Double Sphere, converter inits,
    bounds and tolerances, canonical (algebraic) residual.  GPU and oracle must take the same trajectory (status,
    iterations, passes) and end at the same parameters within 1e-9 -- the reductions differ (one thread vs 50 k), so
    this is the test that the kernel's summation error stays far below the solver's decision thresholds."""
    from apex_camera_models_b200 import _native as N
    lib = N.lib
    n = 10_000_000
    kbp = cameras["kannala_brandt"]["params"]
    kb = acm.KannalaBrandtModel(acm.Intrinsics(*kbp[:4]), acm.Resolution(512, 512), kbp[4:], ctx=ctx)
    X = acm.Points(ctx, 3, n)
    ctx.check(lib.acm_synth_points3(ctx.handle, 0xACE50004, 0, float(np.cos(np.deg2rad(85.0))), 0, X.handle))
    UV, st = kb.project_batch(X)
    ctx.device_free(st)
    ds = acm.DoubleSphereModel(acm.Intrinsics(*kbp[:4]), acm.Resolution(512, 512), [0.5, 0.1], ctx=ctx)
    cost = acm.DoubleSphereOptimizationCost(ds, X, UV)
    cost.linear_estimation()
    start = ds.params().copy()
    r = cost.optimize()
    xyz, uv = X.numpy(), UV.numpy()
    om = O.make_model(O.DS, list(kbp[:4]) + [0.5, 0.1], 512, 512)
    assert O.linear_estimation(om, xyz, uv) == 0
    assert np.allclose(start, om.params(), rtol=1e-12)
    b = acm.CONVERTER_BOUNDS[5]
    oo, ores = O.lm_solve(om, O.RES_ALGEBRAIC, xyz, uv, [x[0] for x in b], [x[1] for x in b], nthreads=8)
    assert (r.status, r.iterations, r.passes) == (ores.status, ores.iterations, ores.passes)
    assert r.n_valid == ores.n_valid == n
    assert np.allclose(r.parameters, oo, rtol=1e-9), np.abs(r.parameters - oo) / np.abs(oo)
    assert abs(r.final_cost - ores.final_cost) <= 1e-9 * ores.final_cost
    assert r.device_ms > 0.0 and r.device_ms <= r.elapsed_ms + 1e-3
    X.free(); UV.free()


@pytest.mark.parametrize("name,kind", [("double_sphere", 1), ("ucm", 0), ("eucm", 0)])
def test_lm_grid_sizes_take_the_oracle_trajectory(acm, ctx, O, cameras, name, kind):
    """The solve kernel's grid follows the problem size (never fewer blocks than sums; the reducer blocks split the
    column of block partials over their warps, unevenly when the grid is not a multiple of the warp count): sizes that
    give 29..52 (floor), 79, 131 and the resident maximum of blocks must all walk the oracle's trajectory."""
    kbp = cameras["kannala_brandt"]["params"]
    truth = oracle_model(O, cameras["kannala_brandt"])
    for n in (130, 4_099, 20_011, 33_333, 90_001, 123_457):
        xyz = O.synth_points3(0xACE50010 + n, 0, n, np.cos(np.deg2rad(80.0)), False)
        uv, st = O.project(truth, xyz)
        assert np.all(st == 0)
        cam = {"model_id": cameras[name]["model_id"], "params": list(kbp[:4]) + INITS[name], "width": 512, "height": 512}
        m, om = gpu_model(acm, ctx, cam), oracle_model(O, cam)
        m.linear_estimation(xyz, uv)
        O.linear_estimation(om, xyz, uv)
        b = acm.CONVERTER_BOUNDS[m.MODEL_ID]
        lo, hi = [x[0] for x in b], [x[1] for x in b]
        cost = acm.OptimizationCost(m, xyz, uv, residual_kind=kind)
        r = cost.optimize()
        oo, ores = O.lm_solve(om, kind, xyz, uv, lo, hi)
        assert (r.status, r.iterations, r.passes) == (ores.status, ores.iterations, ores.passes), (name, n)
        assert r.n_valid == ores.n_valid == n
        assert np.allclose(r.parameters, oo, rtol=1e-9), (name, n, np.abs(r.parameters - oo) / np.abs(oo))
        cost.free()


def test_lm_anchors_and_readme_figures(acm, ctx, O, cameras):
    """KB -> DS / UCM on the 450 correspondences ends at the survey's anchors (scipy, 1e-15) and at
    the README's 0.008 px / 0.145 px (README.md:163-164)."""
    A = load_golden("restated_kats.json")["lm_anchors_450"]
    intr, uv, xyz = _kb450(O, cameras)
    tight = acm.LevenbergMarquardtConfig(max_iterations=500, cost_tolerance=0.0, parameter_tolerance=1e-15, gradient_tolerance=0.0)
    ds = acm.DoubleSphereModel(acm.Intrinsics(*intr), acm.Resolution(512, 512), [0.5, 0.1], ctx=ctx)
    assert abs(acm.compute_reprojection_error(ds, xyz, uv).mean - A["ds_initial_mean_px"]) < 1e-4
    cost = acm.DoubleSphereOptimizationCost(ds, xyz, uv)  # canonical residual: algebraic
    cost.linear_estimation()
    assert abs(acm.compute_reprojection_error(ds, xyz, uv).mean - A["linear_only_mean_px"]) < 1e-5
    r = cost.optimize(config=tight)
    assert np.allclose(r.parameters, A["ds_algebraic"]["params"], rtol=5e-9)
    e = acm.compute_reprojection_error(ds, xyz, uv)
    assert abs(e.mean - A["ds_algebraic"]["mean_px"]) < 5e-7 and round(e.mean, 3) == 0.008
    ucm = acm.UcmModel(acm.Intrinsics(*intr), acm.Resolution(512, 512), [0.5], ctx=ctx)
    c2 = acm.UcmOptimizationCost(ucm, xyz, uv)
    c2.linear_estimation(); c2.optimize()
    assert round(acm.compute_reprojection_error(ucm, xyz, uv).mean, 3) == 0.145


def test_lm_recovers_generating_model_and_penalty(acm, ctx, O, cameras):
    c = cameras["double_sphere"]
    truth = oracle_model(O, c)
    xyz = O.synth_points3(0xACE50003, 0, 200_001, np.cos(np.deg2rad(70.0)), False)
    uv, st = O.project(truth, xyz)
    assert np.all(st == 0)
    start = np.array(c["params"]) * np.array([1.02, 0.98, 1.01, 0.99, 0.9, 0.8])
    m = acm.DoubleSphereModel(acm.Intrinsics(*start[:4]), acm.Resolution(752, 480), start[4:], ctx=ctx)
    cost = acm.DoubleSphereOptimizationCost(m, xyz, uv, residual_kind=0)
    tight = acm.LevenbergMarquardtConfig(max_iterations=200, cost_tolerance=0.0, parameter_tolerance=1e-15, gradient_tolerance=0.0)
    r = cost.optimize(config=tight, bounds=None)
    assert np.allclose(r.parameters, c["params"], rtol=1e-9) and r.n_valid == len(xyz)
    # invalid_penalty: residual (pen, pen) for invalid points, as the former in-tree factor did
    xyz2 = xyz[:1000].copy(); xyz2[::10, 2] = -5.0
    m2 = acm.DoubleSphereModel(acm.Intrinsics(*c["params"][:4]), acm.Resolution(752, 480), c["params"][4:], ctx=ctx)
    c2 = acm.DoubleSphereOptimizationCost(m2, xyz2, uv[:1000], residual_kind=0)
    r0 = c2.optimize(config=acm.LevenbergMarquardtConfig(max_iterations=0), bounds=None)  # evaluation only
    r1 = c2.optimize(config=acm.LevenbergMarquardtConfig(max_iterations=0, invalid_penalty=1e3), bounds=None)
    assert r0.status == 3 and r0.passes == 1 and r0.n_valid == r1.n_valid
    n_bad = 1000 - r0.n_valid
    assert n_bad > 0 and abs((r1.initial_cost - r0.initial_cost) - n_bad * 1e6) <= 1e-6 * n_bad * 1e6


# ------------------------------------------------------------------ util hot loops ----------------
@pytest.mark.parametrize("name,n", [("kannala_brandt", 500), ("kannala_brandt", 10_000), ("double_sphere", 100), ("rad_tan", 50),
                                    ("ucm", 777), ("eucm", 1000), ("fov", 300), ("pinhole", 64), ("kannala_brandt", 1_000_000)])
def test_sample_points_matches_oracle(acm, ctx, O, cameras, name, n):
    cam = cameras[name]
    m, om = gpu_model(acm, ctx, cam), oracle_model(O, cam)
    uv, xyz = acm.sample_points(m, n)
    uvo, xyzo = O.sample_points(om, n)
    assert uv.shape == uvo.shape, "kept set differs"
    assert np.array_equal(uv, uvo)  # same pixels in the same order
    if name in EXACT:
        assert np.array_equal(xyz, xyzo)
    else:
        assert np.allclose(xyz, xyzo, rtol=RTOL, atol=1e-15)
    if (name, n) == ("kannala_brandt", 500):
        assert len(uv) == 450
    if (name, n) == ("kannala_brandt", 10_000):
        assert len(uv) == 9294


@pytest.mark.parametrize("name", ["double_sphere", "kannala_brandt", "pinhole", "fov"])
def test_reprojection_error_matches_oracle(acm, ctx, O, cameras, name):
    cam = cameras[name]
    m, om = gpu_model(acm, ctx, cam), oracle_model(O, cam)
    for n in (1, 2, 451, 100_004):
        xyz, obs = _correspondences(O, om, name, n, noise=0.0)
        rng = np.random.default_rng(n)
        obs = obs + rng.normal(0, 0.3, obs.shape)
        try:
            eo = O.reprojection_error(om, xyz, obs)
        except ValueError:
            with pytest.raises(acm.ZeroProjectionPoints):
                acm.compute_reprojection_error(m, xyz, obs)
            continue
        e = acm.compute_reprojection_error(m, xyz, obs)
        assert e.count == eo.count
        for f in ("rmse", "min", "max", "mean", "stddev", "median"):
            assert np.isclose(getattr(e, f), getattr(eo, f), rtol=1e-9, atol=1e-13), f
    with pytest.raises(acm.ZeroProjectionPoints):
        acm.compute_reprojection_error(m, np.tile([0.0, 0.0, -1.0], (8, 1)), np.zeros((8, 2)))


@pytest.mark.parametrize("name,W,H", [("kannala_brandt", 512, 512), ("double_sphere", 752, 480), ("pinhole", 752, 480),
                                      ("rad_tan", 752, 480), ("fov", 320, 200), ("ucm", 1920, 1080), ("kannala_brandt", 37, 29)])
def test_undistort_bytes_and_remap_indices(acm, ctx, O, cameras, name, W, H):
    """undistort.rs:14-105: output bytes and remap indices are bit-exact (KB / FOV depend on the
    device atan2: count index flips, expected 0)."""
    cam = dict(cameras[name]); cam["width"], cam["height"] = W, H
    if name in ("ucm", "fov"):  # keep the principal point inside the test image
        cam["params"] = list(cam["params"]); cam["params"][2] = W / 2.0 + 0.3; cam["params"][3] = H / 2.0 - 0.2
    if (W, H) == (37, 29):
        cam["params"] = [20.0, 20.0, 18.2, 14.1] + cam["params"][4:]
    m, om = gpu_model(acm, ctx, cam), oracle_model(O, cam)
    frames = O.synth_bytes(0xACE50005, 0, 3 * W * H * 3).reshape(3, H, W, 3)
    for target in (None, acm.Intrinsics(cam["params"][0] * 0.6, cam["params"][1] * 0.6, W / 2.0, H / 2.0)):
        t = cam["params"][:4] if target is None else [target.fx, target.fy, target.cx, target.cy]
        mp = acm.undistort_map(m, target)
        mpo = O.undistort_map(om, t)
        assert np.array_equal(np.isnan(mp), np.isnan(mpo))
        ok = ~np.isnan(mpo)
        flips = int(np.sum(np.floor(mp[ok]) != np.floor(mpo[ok])))
        assert flips == 0, f"{flips} remap indices differ"
        if name in EXACT:
            assert np.array_equal(mp[ok], mpo[ok])
        for interp in (acm.InterpolationMethod.Bilinear, acm.InterpolationMethod.Nearest):
            out = acm.undistort_images(frames, m, target, interp)
            for f in range(3):
                ref = O.undistort_rgb8(om, t, frames[f], int(interp), nthreads=4)
                assert np.array_equal(out[f], ref), f"{name} frame {f} interp {interp}: {(out[f] != ref).sum()} bytes differ"
    one = acm.undistort_image(frames[0], m)
    assert np.array_equal(one, acm.undistort_images(frames[:1], m)[0])
    with pytest.raises(acm.UtilError, match="doesn't match model"):
        acm.undistort_image(np.zeros((H + 1, W, 3), np.uint8), m)


def test_undistort_many_frames_ring_wraparound(acm, ctx, O, cameras):
    """The TMA path keeps 4 frames in flight per warp: 11 frames take every stage through three
    phases of its mbarrier; the bytes of every frame must still equal the oracle's."""
    cam = dict(cameras["kannala_brandt"]); W, H = 512, 512
    m, om = gpu_model(acm, ctx, cam), oracle_model(O, cam)
    F = 11
    frames = O.synth_bytes(0xACE50006, 0, F * W * H * 3).reshape(F, H, W, 3)
    out = acm.undistort_images(frames, m)
    for f in range(F):
        ref = O.undistort_rgb8(om, cam["params"][:4], frames[f], 1, nthreads=4)
        assert np.array_equal(out[f], ref), f"frame {f}: {(out[f] != ref).sum()} bytes differ"


# ------------------------------------------------------------------ BASELINE sizes: properties -----
def test_full_size_round_trip_and_linearity(acm, ctx, O, cameras):
    """100 M synthetic points (BASELINE configs 2 and 3): project -> unproject returns the input
    direction; the normal equations of the whole equal the sum over shards; repeat runs are
    bit-identical."""
    from apex_camera_models_b200 import _native as N
    lib = N.lib
    n = 100_000_000
    cam = cameras["double_sphere"]
    m = gpu_model(acm, ctx, dict(cam, width=100000, height=100000, params=cam["params"][:2] + [50000.0, 50000.0] + cam["params"][4:]))
    X = acm.Points(ctx, 3, n)
    ctx.check(lib.acm_synth_points3(ctx.handle, 0xACE50002, 0, np.cos(np.deg2rad(100.0)), 1, X.handle))
    UV, st = m.project_batch(X)
    R, st2 = m.unproject_batch(UV)
    # sample-check the round trip on strided slices brought back to the host
    k = 1_000_003
    xs = np.empty((3, k)); rs = np.empty((3, k)); s1 = np.empty(k, np.uint8); s2 = np.empty(k, np.uint8)
    off = 37_000_000
    for c in range(3):
        ctx.d2h(xs[c], X.component_ptr(c) + 8 * off); ctx.d2h(rs[c], R.component_ptr(c) + 8 * off)
    ctx.d2h(s1, st + off); ctx.d2h(s2, st2 + off); ctx.sync()
    ok = (s1 == 0) & (s2 == 0)
    assert ok.mean() > 0.9
    d = xs[:, ok] / np.linalg.norm(xs[:, ok], axis=0)
    assert np.max(np.abs(np.sum(d * rs[:, ok], axis=0) - 1.0)) < 1e-9
    xo = O.synth_points3(0xACE50002, off, 4096, np.cos(np.deg2rad(100.0)), True)
    assert np.array_equal(xs[:, :4096].T, xo)
    _, sto = O.project(oracle_model(O, dict(cam, width=100000, height=100000, params=cam["params"][:2] + [50000.0, 50000.0] + cam["params"][4:])), xo)
    assert np.array_equal(s1[:4096], sto)
    # status census must match the generator's design: every 64th point is adversarial
    ctx.device_free(st2); R.free()
    # linearity of the normal equations over shards
    cost = acm.DoubleSphereOptimizationCost(m, X, UV, residual_kind=0)
    # perturb the model so residuals are non-zero
    m.set_params(m.params() * np.array([1.001, 0.999, 1.0, 1.0, 1.01, 0.98]))
    H, g, c, nv = cost.linearize()
    H2, g2, c2, nv2 = cost.linearize()
    assert np.array_equal(H, H2) and np.array_equal(g, g2) and c == c2 and nv == nv2
    # shards: views into the same buffers (4 contiguous quarters, 256-byte aligned offsets)
    Hs = np.zeros_like(H); gs = np.zeros_like(g); cs = 0.0; nvs = 0
    q = n // 4
    for r in range(4):
        Xs = acm.Points(ctx, 3, q); UVs = acm.Points(ctx, 2, q)
        for cc in range(3):
            ctx.d2d(Xs.component_ptr(cc), X.component_ptr(cc) + 8 * q * r, 8 * q)
        for cc in range(2):
            ctx.d2d(UVs.component_ptr(cc), UV.component_ptr(cc) + 8 * q * r, 8 * q)
        ctx.sync()
        sc = acm.DoubleSphereOptimizationCost(m, Xs, UVs, residual_kind=0)
        h_, g_, c_, n_ = sc.linearize()
        Hs += h_; gs += g_; cs += c_; nvs += n_
        Xs.free(); UVs.free()
    assert nvs == nv
    assert np.allclose(Hs, H, rtol=1e-12) and np.allclose(gs, g, rtol=1e-9, atol=1e-9 * np.abs(g).max()) and np.isclose(cs, c, rtol=1e-12)
    ctx.device_free(st); X.free(); UV.free()


@pytest.mark.gpu
def test_multi_gpu_converter_pipeline_matches_single_gpu():
    """sample_points(shard) -> linear_estimation -> LM -> reprojection statistics on 2 GPUs (NCCL and
    fused NVLink exchange) against the same pipeline on one GPU; needs two visible GPUs."""
    import subprocess
    import sys
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, ACM_CHECK_POINTS="200000")
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
                        "--master-port", "29533", os.path.join(root, "scripts", "multi_gpu_check.py")], capture_output=True, text=True,
                       timeout=600, env=env, cwd=root)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]


KB_YAML = """cam0:
  camera_model: kannala_brandt
  intrinsics: [{fx}, {fy}, {cx}, {cy}]
  distortion: [{k1}, {k2}, {k3}, {k4}]
  resolution: [512, 512]
"""


@pytest.mark.gpu
def test_camera_converter_cli_config1(acm, cameras, tmp_path, capsys):
    """BASELINE config 1: `camera_converter --input-model kb --input-path samples/kannala_brandt.yaml
    --num-points 500` through the GPU path; 450 correspondences, README figures (README.md:161-166)."""
    from apex_camera_models_b200 import camera_converter as cc
    p = cameras["kannala_brandt"]["params"]
    y = tmp_path / "kb.yaml"
    y.write_text(KB_YAML.format(fx=p[0], fy=p[1], cx=p[2], cy=p[3], k1=p[4], k2=p[5], k3=p[6], k4=p[7]))
    out_dir = tmp_path / "out"
    assert cc.main(["-i", "kb", "-p", str(y), "-n", "500", "-o", str(out_dir)]) == 0
    text = capsys.readouterr().out
    assert "Valid 3D-2D correspondences: 450 / 500" in text
    kb = cc.load_input_model("kb", str(y))
    kept, metrics, pts = cc.convert_all(kb, 500)
    assert kept == 450
    by = {m.model_name: m for m in metrics}
    assert [m.model_name for m in metrics] == ["Double Sphere", "Radial-Tangential", "Unified Camera Model",
                                               "Extended Unified Camera Model", "Field-of-View"]  # KB is the input
    assert abs(by["Double Sphere"].final_reprojection_error.mean - 0.0077324) < 2e-6      # README "0.008 px"
    assert abs(by["Unified Camera Model"].final_reprojection_error.mean - 0.1452208) < 2e-6  # README "0.145 px"
    assert abs(by["Double Sphere"].initial_reprojection_error.mean - 10.0321) < 1e-3      # README "+10.02 px"
    assert by["Double Sphere"].validation_results.status in ("EXCELLENT", "GOOD")
    assert by["Radial-Tangential"].final_reprojection_error.mean > 50.0                   # README: "EXPECTED" failure on fisheye input
    ds = acm.DoubleSphereModel.load_from_yaml(str(out_dir / "double_sphere.yaml"))
    assert np.allclose(ds.params(), by["Double Sphere"].model.params(), rtol=0, atol=1e-12)
    # the files the reference writes next to the models: report, correspondences, projection images
    report = (out_dir / "camera_conversion_results_kb.txt").read_text(encoding="utf-8")
    assert "INPUT MODEL TYPE: KB" in report and "DOUBLE SPHERE MODEL:" in report and "Image Quality Assessment:" in report
    assert "Final Parameters: DoubleSphere(DoubleSphere [fx: " in report
    csv = (out_dir / "point_correspondences_apex.csv").read_text().split("\n")
    assert csv[2] == "# Total points: 450" and len([l for l in csv if l and not l.startswith("#")]) == 450
    assert (out_dir / "point_correspondences_apex_rust.txt").exists()
    from PIL import Image
    for name in ("kb_projection.png", "double_sphere_apex_projection.png", "radial_tangential_apex_projection.png", "fov_apex_projection.png"):
        assert Image.open(out_dir / name).size == (512, 512), name
    assert by["Double Sphere"].image_quality is not None and by["Double Sphere"].image_quality.ssim > 0.99


@pytest.mark.gpu
def test_image_undistort_cli(acm, ctx, O, cameras, tmp_path):
    """bin/image_undistort.rs flags through the GPU path: PNG in, PNG out, bytes equal to the oracle's."""
    from PIL import Image
    from apex_camera_models_b200 import image_undistort as iu
    p = cameras["kannala_brandt"]["params"]
    y = tmp_path / "kb.yaml"
    y.write_text(KB_YAML.format(fx=p[0], fy=p[1], cx=p[2], cy=p[3], k1=p[4], k2=p[5], k3=p[6], k4=p[7]))
    img = O.synth_bytes(0xACE50007, 0, 512 * 512 * 3).reshape(512, 512, 3)
    Image.fromarray(img, "RGB").save(tmp_path / "in.png")
    assert iu.main(["-i", str(tmp_path / "in.png"), "-c", str(y), "-o", str(tmp_path / "out.png"), "-m", "kb", "--target-fx", "150.0"]) == 0
    got = np.asarray(Image.open(tmp_path / "out.png").convert("RGB"))
    cam = dict(cameras["kannala_brandt"])
    ref = O.undistort_rgb8(oracle_model(O, cam), [150.0, p[1], p[2], p[3]], img, 1, nthreads=4)
    assert np.array_equal(got, ref)
