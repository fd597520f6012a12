"""The streaming kernels past their first grid-stride trip, against the CPU oracle.

At the sizes of test_gpu_parity.py most threads handle one packet, or a few, which is no more than their ring or
prefetch holds.  The code that runs at real sizes -- the cp.async ring of the normal-equation kernels and its stage
wrap, the four-points-per-trip loop and its odd-packet tail, the register prefetch of the next packet in the batch
maps, the 2-point vector form of the Jacobian kernels, the block shapes chosen by size -- is reached only when every
thread streams several packets.  Every size here is derived from the device (never a fixed SM count):

    S = sm_count,  T = S * 2048  (the most threads sm_100 keeps resident, whatever the occupancy)

and each docstring names the path its size reaches.  The bars are those of test_gpu_parity.py, imported from there:
status bytes bit-exact, values bit-exact or within the per-model bars, normal equations within 1e-9 of their natural
scale, n_valid exact.
"""
import ctypes as C
import os

import numpy as np
import pytest

from conftest import oracle_model
from test_gpu_parity import (EXACT, INITS, MODELS, RTOL, UNIFIED, UNPROJECT_EXACT, assert_close_where_valid, assert_jacobians_match,
                             cone, gpu_model)

pytestmark = pytest.mark.gpu

NT = min(os.cpu_count() or 1, 16)   # oracle threads (per-point results do not depend on it)
PAIRS = [(name, 0) for name in MODELS] + [(name, 1) for name in MODELS if name in UNIFIED]
PAIR_IDS = [f"{n}-{'algebraic' if k else 'pixel'}" for n, k in PAIRS]


@pytest.fixture(scope="module")
def acm():
    import apex_camera_models_b200 as m
    return m


@pytest.fixture(scope="module")
def ctx(acm):
    c = acm.Context(0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def sizes(ctx):
    S = int(ctx.device_info()["sm_count"])
    T = S * 2048
    z = {
        "S": S, "T": T,
        # batch maps: S*8 blocks of 256 threads; one trip = S*8*256 packets of 2 (f64) or 4 (f32) points
        "map_f64": 3 * (S * 8 * 256 * 2) + 1001,
        "map_f32": [3 * (S * 8 * 256 * 4) + 4003, 3 * (S * 8 * 256 * 4) + 4002],
        # Jacobian kernels, vector form: S*4 blocks of 256 threads, 2 points per thread and trip
        "jac": [3 * (S * 4 * 256 * 2), 3 * (S * 4 * 256 * 2) + 1],
        # normal equations and LM solve: at least 6 packets per thread at any occupancy
        "lin": 12 * T + 75,
    }
    print(f"\n[steady-state sizes] device_info={ctx.device_info()} " + ", ".join(f"{k}={v}" for k, v in z.items()))
    return z


def fetch_status(ctx, ptr, n):
    out = np.empty(n, np.uint8)
    if n:
        ctx.d2h(out, ptr)
    ctx.sync()
    ctx.device_free(ptr)
    return out


def fast_unproject(cam_block):
    from apex_camera_models_b200 import _native as N
    return N.lib.acm_camera_fast_unproject(C.byref(cam_block))


def pixels_in_and_around(O, cam, n, seed):
    """Pixels 5 % beyond the image on every side, with the principal point and KB's 1e-6 hole at non-periodic places."""
    W, H = cam["width"], cam["height"]
    px = O.synth_pixels(seed, 0, n, W * 1.1, H * 1.1) - [0.05 * W, 0.05 * H]
    rng = np.random.default_rng(seed)
    cx, cy, fx = cam["params"][2], cam["params"][3], cam["params"][0]
    px[rng.choice(n, 2000, replace=False)] = [cx, cy]
    px[rng.choice(n, 2000, replace=False)] = [cx + 0.5e-6 * fx, cy]
    px[-1] = [cx, cy]   # the ragged tail point
    return px


# ------------------------------------------------------------------ A. batch maps --------------------------------
@pytest.mark.parametrize("name", MODELS)
def test_batch_maps_f64_at_steady_state(acm, ctx, O, cameras, sizes, name):
    """acm_project / acm_unproject / acm_unproject_ieee / acm_project_unproject on device f64 `Points`.

    grid_for(n / 2 + 2, 256, 8) is capped at S*8 blocks: one grid-stride trip covers S*8*256 packets of 2 points.
    n = 3 * (S*8*256*2) + 1001 makes every thread take at least three packets, so the prefetch branch `pn < npk` of
    the pipelined kernels (project: RadTan, KB, DS; unproject: all but RadTan; round trip: Pinhole, DS) loads packets
    that are evaluated one trip later, the fourth trip is ragged (500 packets) and one point goes through the scalar
    tail.  The KB and RadTan sample cameras take the contracted-Newton unproject loop (asserted)."""
    from apex_camera_models_b200 import _native as N
    cam = cameras[name]
    m, om = gpu_model(acm, ctx, cam), oracle_model(O, cam)
    if name in ("kannala_brandt", "rad_tan"):
        assert fast_unproject(m.camera_block()) == 1
    n = sizes["map_f64"]
    xyz = O.synth_points3(0xACE50012, 0, n, cone(name), True)
    X = acm.Points.from_numpy(ctx, xyz)
    UV, sp = m.project_batch(X)
    uv, st = UV.numpy(), fetch_status(ctx, sp, n)
    uvo, sto = O.project(om, xyz, NT)
    assert np.array_equal(st, sto), np.flatnonzero(st != sto)[:8]
    assert len(np.unique(sto)) >= 2
    assert_close_where_valid(uv, uvo, sto == 0, name)
    UV.free()

    px = pixels_in_and_around(O, cam, n, 0xACE50013)
    PX = acm.Points.from_numpy(ctx, px)
    R, su = m.unproject_batch(PX)
    ray, st = R.numpy(), fetch_status(ctx, su, n)
    rayo, sto = O.unproject(om, px, NT)
    assert np.array_equal(st, sto), np.flatnonzero(st != sto)[:8]
    assert_close_where_valid(ray, rayo, sto == 0, name, UNPROJECT_EXACT)
    # IEEE tails: same status bytes; the arithmetic-only models bit for bit
    cb = m.camera_block()
    R2 = acm.Points(ctx, 3, n)
    s2 = ctx.device_alloc(n)
    ctx.check(N.lib.acm_unproject_ieee(ctx.handle, C.byref(cb), PX.handle, R2.handle, C.c_void_p(s2)))
    ray2, st2 = R2.numpy(), fetch_status(ctx, s2, n)
    assert np.array_equal(st2, sto)
    assert np.array_equal(np.isnan(ray2), np.isnan(rayo))
    fin = (sto == 0) & ~np.isnan(rayo).any(axis=1)
    if name in EXACT:
        assert np.array_equal(ray2[fin], rayo[fin]), np.abs(ray2[fin] - rayo[fin]).max()
    else:
        assert np.allclose(ray2[fin], rayo[fin], rtol=RTOL, atol=1e-13)
    R.free(); R2.free(); PX.free()

    UV, RAY, sp, su = m.round_trip_batch(X)
    uv, ray = UV.numpy(), RAY.numpy()
    sp, su = fetch_status(ctx, sp, n), fetch_status(ctx, su, n)
    uvo, spo = O.project(om, xyz, NT)
    assert np.array_equal(sp, spo)
    assert_close_where_valid(uv, uvo, spo == 0, name)
    ok = spo == 0
    rayo, suo = O.unproject(om, uv[ok], NT)   # unproject what the device projected (KB / FOV differ in the last ulps)
    assert np.array_equal(su[ok], suo) and np.array_equal(su[~ok], spo[~ok])
    assert_close_where_valid(ray[ok], rayo, suo == 0, name, UNPROJECT_EXACT)
    good = np.zeros(n, bool); good[np.flatnonzero(ok)[suo == 0]] = True
    assert np.all(np.isnan(ray[~good]))
    UV.free(); RAY.free(); X.free()


@pytest.mark.parametrize("tail", [3, 2])
@pytest.mark.parametrize("name", MODELS)
def test_batch_maps_f32_at_steady_state(acm, ctx, O, cameras, sizes, name, tail):
    """The f32 forms of the same kernels: packets of 4 points, one trip = S*8*256*4 points.  n = 3 * (S*8*256*4) +
    4000 + tail: three full trips for every thread (prefetch branch taken), a ragged fourth trip, and a scalar tail of 3
    or 2 points (n % 4).  Bars of test_f32_io_path: the oracle runs on the same f32-rounded inputs, values within
    max(1e-4 px, half an f32 ulp), rays within 1e-7, status bytes bit-exact."""
    from apex_camera_models_b200 import _native as N
    cam = cameras[name]
    m, om = gpu_model(acm, ctx, cam), oracle_model(O, cam)
    n = sizes["map_f32"][0 if tail == 3 else 1]
    assert n % 4 == tail
    xyz = O.synth_points3(0xACE50014, 0, n, cone(name), True).astype(np.float32).astype(np.float64)
    X = acm.Points.from_numpy(ctx, xyz, N.F32)
    UV, sp = m.project_batch(X)
    uv, st = UV.numpy(), fetch_status(ctx, sp, n)
    uvo, stp = O.project(om, xyz, NT)
    assert np.array_equal(st, stp), np.flatnonzero(st != stp)[:8]
    ok = stp == 0
    tol = np.maximum(1e-4, 0.5 * np.spacing(np.abs(uvo[ok]).astype(np.float32)).astype(np.float64))
    assert np.all(np.abs(uv[ok] - uvo[ok]) <= tol)
    assert np.all(np.isnan(uv[~ok]))
    UV.free()

    px = pixels_in_and_around(O, cam, n, 0xACE50015).astype(np.float32).astype(np.float64)
    PX = acm.Points.from_numpy(ctx, px, N.F32)
    R, su = m.unproject_batch(PX)
    ray, st = R.numpy(), fetch_status(ctx, su, n)
    rayo, sto = O.unproject(om, px, NT)
    assert np.array_equal(st, sto), np.flatnonzero(st != sto)[:8]
    assert np.all(np.abs(ray[sto == 0] - rayo[sto == 0]) <= 1e-7)
    assert np.all(np.isnan(ray[sto != 0]))
    R.free(); PX.free()

    UV, RAY, sp, su = m.round_trip_batch(X)
    uv, ray = UV.numpy(), RAY.numpy()
    sp, su = fetch_status(ctx, sp, n), fetch_status(ctx, su, n)
    assert np.array_equal(sp, stp)
    assert np.all(np.abs(uv[ok] - uvo[ok]) <= tol)
    rayo, suo = O.unproject(om, uv[ok], NT)   # the kernel unprojects the f32-rounded projection it stores
    assert np.array_equal(su[ok], suo) and np.array_equal(su[~ok], sp[~ok])
    fin = suo == 0
    assert np.all(np.abs(ray[ok][fin] - rayo[fin]) <= 1e-7)
    UV.free(); RAY.free(); X.free()


# ------------------------------------------------------------------ C. Jacobian kernels ---------------------------
def jacobian_inputs(O, name, n):
    xyz = O.synth_points3(0xACE50016, 0, n, cone(name), True)
    rng = np.random.default_rng(n)
    xyz[rng.choice(n, n // 50, replace=False), :2] *= 1e-9   # near the axis: KB r < EPS / FOV r^2 < sqrt(EPS) branches
    xyz[rng.choice(n, n // 100, replace=False), :2] = 0.0
    return xyz


@pytest.mark.parametrize("odd", [0, 1])
@pytest.mark.parametrize("name", MODELS)
def test_jacobians_at_steady_state(acm, ctx, O, cameras, sizes, name, odd):
    """acm_project_jacobian and acm_project_point_jacobian past one grid-stride trip, every point against the oracle.

    Even n takes the vector form NV = 2 (grid_for(n / 2, 256, 4): S*4 blocks, one trip = S*4*256*2 points), so
    n = 3 * (S*4*256*2) gives every thread three trips of 16-byte loads and paired stores; n + 1 takes the scalar form
    (grid_for(n, 256, 4), one trip = S*4*256 points): six full trips and one more point.  Failed points: J = 0, uv NaN."""
    cam = cameras[name]
    m, om = gpu_model(acm, ctx, cam), oracle_model(O, cam)
    n = sizes["jac"][odd]
    xyz = jacobian_inputs(O, name, n)
    uv, J, st = m.project_jacobian_batch(xyz)
    uvo, Jo, sto = O.project_jacobian(om, xyz, NT)
    assert_jacobians_match(uv, J, st, uvo, Jo, sto)
    uv, J, st = m.project_point_jacobian_batch(xyz)
    uvo, Jo, sto = O.project_point_jacobian(om, xyz, NT)
    assert_jacobians_match(uv, J, st, uvo, Jo, sto)


# ------------------------------------------------------------------ D. one-pass normal equations -------------------
def invalid_mix(O, om, name, n, seed):
    """Correspondences of the sample camera (0.5 px noise) in which an RNG-chosen 2 % of the points lie behind the
    camera, where every model rejects them.  Non-periodic, unlike the generator's adversarial points (every 64th)."""
    xyz = O.synth_points3(seed, 0, n, cone(name), False)
    obs, _ = O.project(om, xyz, NT)
    rng = np.random.default_rng(seed)
    obs = np.where(np.isnan(obs), 1.0, obs) + rng.normal(0.0, 0.5, (n, 2))
    bad = rng.choice(n, n // 50, replace=False)
    xyz[bad, :2] *= 0.1
    xyz[bad, 2] = -1.0 - np.abs(xyz[bad, 2])
    return xyz, obs


def assert_normal_equations_match(H, g, c, nv, Ho, go, co, nvo):
    """Bars of test_linearize_matches_oracle."""
    assert nv == nvo
    dg = np.sqrt(np.abs(np.diag(Ho))) + 1e-300
    assert np.max(np.abs(H - Ho) / np.outer(dg, dg)) < RTOL
    assert np.max(np.abs(g - go) / (dg * np.sqrt(2 * co) + 1e-300)) < RTOL
    assert abs(c - co) <= RTOL * co
    assert np.array_equal(H, H.T)


def linearize_once(ctx, cost):
    before = ctx.kernel_launches()
    out = cost.linearize()
    assert ctx.kernel_launches() - before == 1
    return out


@pytest.mark.parametrize("name,kind", PAIRS, ids=PAIR_IDS)
def test_linearize_at_steady_state(acm, ctx, O, cameras, sizes, name, kind):
    """lin_kernel<M, KIND, BS, false> (one pass, one launch) at n = 12*T + 75.

    The grid is min(ceil(pairs / BS), S * blocks_per_sm) <= T / BS blocks, so every thread streams at least
    (n / 2) / T >= 6 packets: more than the deepest ring (4), so every stage of every ring is reused; the four-point
    loop of KB / FOV runs at least two trips, and as the packet count per thread is 6 or 7 at full occupancy the
    odd-packet tail runs too.  n is odd: block 0 / thread 0 adds the last point.  The block shape is the model's
    (128 threads for KB, 256 for the others); a repeat call is bit-identical."""
    cam = cameras[name]
    m, om = gpu_model(acm, ctx, cam), oracle_model(O, cam)
    n = sizes["lin"]
    xyz, obs = invalid_mix(O, om, name, n, 0xACE50017 + 16 * MODELS.index(name) + kind)
    Ho, go, co, nvo = O.linearize(om, kind, xyz, obs, nthreads=NT)
    assert n - nvo >= n // 100, (n, nvo)   # the rejected points are there
    X, UV = acm.Points.from_numpy(ctx, xyz), acm.Points.from_numpy(ctx, obs)
    cost = acm.OptimizationCost(m, X, UV, residual_kind=kind)
    H, g, c, nv = linearize_once(ctx, cost)
    assert_normal_equations_match(H, g, c, nv, Ho, go, co, nvo)
    H2, g2, c2, nv2 = linearize_once(ctx, cost)
    assert np.array_equal(H, H2) and np.array_equal(g, g2) and c == c2 and nv == nv2
    X.free(); UV.free()


def valid_points(O, om, name, n, seed, cos_max=None):
    """The first n points of a seeded stream that project inside the image: (xyz, oracle uv)."""
    cos_max = cone(name) if cos_max is None else cos_max
    xyz = O.synth_points3(seed, 0, n + n // 2, cos_max, False)
    uv, st = O.project(om, xyz, NT)
    keep = np.flatnonzero(st == 0)
    assert len(keep) >= n
    keep = keep[:n]
    return np.ascontiguousarray(xyz[keep]), np.ascontiguousarray(uv[keep])


@pytest.mark.parametrize("name", MODELS)
def test_linearize_census_at_steady_state(acm, ctx, O, cameras, sizes, name):
    """Pixel residual at n = 12*T + 75 (the size of test_linearize_at_steady_state): every point is valid and observed
    at the oracle's projection, except K markers observed 1 px to the right, at indices 0..63, n-64..n-1 (the odd last
    point is block 0 / thread 0's) and 4096 random ones.  The markers carry the whole cost and gradient, so cost / c0
    (c0: the oracle's cost of one marker) and |g[cx]| must round to exactly K: a dropped or doubled packet, or one read
    from a stale ring slot, moves them by a whole unit whatever the tolerance."""
    cam = cameras[name]
    m, om = gpu_model(acm, ctx, cam), oracle_model(O, cam)
    n = sizes["lin"]
    xyz, obs = valid_points(O, om, name, n, 0xACE50018)
    rng = np.random.default_rng(0xACE50018)
    marks = np.concatenate([np.arange(64), np.arange(n - 64, n), 64 + rng.choice(n - 128, 4096, replace=False)])
    K = len(np.unique(marks))
    assert K == 64 + 64 + 4096
    obs[marks, 0] += 1.0
    _, _, c0, nv0 = O.linearize(om, 0, xyz[marks[:1]], obs[marks[:1]])
    assert nv0 == 1 and 0.49 < c0 < 0.51
    X, UV = acm.Points.from_numpy(ctx, xyz), acm.Points.from_numpy(ctx, obs)
    cost = acm.OptimizationCost(m, X, UV, residual_kind=0)
    H, g, c, nv = linearize_once(ctx, cost)
    assert nv == n, nv - n
    assert round(c / c0) == K, c / c0 - K
    assert round(abs(g[2])) == K, abs(g[2]) - K
    X.free(); UV.free()


# ------------------------------------------------------------------ E. LM solve --------------------------------------
def solve_problem(acm, ctx, O, cameras, name, n, seed):
    """(model at its start, oracle model at the same start, X, UV, host xyz, host uv, lower, upper) for one pair.
    KB-generated correspondences (80-degree cone, 512 x 512) for KB / UCM / EUCM / DS / FOV, started from the device's
    linear estimation like the converter; the sample RadTan camera's for RadTan (started from its linear estimation)
    and Pinhole (started from the RadTan intrinsics).  Seeded Gaussian noise of 0.3 px on every observation keeps the
    final cost far above rounding level, so the stopping decisions are not rounding noise."""
    if name in ("rad_tan", "pinhole"):
        src = cameras["rad_tan"]
        xyz, uv = valid_points(O, oracle_model(O, src), "rad_tan", n, seed)
        W, H = src["width"], src["height"]
        intr = src["params"][:4]
    else:
        src = cameras["kannala_brandt"]
        xyz, uv = valid_points(O, oracle_model(O, src), name, n, seed, float(np.cos(np.deg2rad(80.0))))
        W, H = 512, 512
        intr = src["params"][:4]
    uv += np.random.default_rng(seed).normal(0.0, 0.3, uv.shape)
    cam = {"model_id": MODELS.index(name), "params": list(intr) + ([0.0] * 5 if name == "rad_tan" else INITS.get(name, [])),
           "width": W, "height": H}
    m = gpu_model(acm, ctx, cam)
    X, UV = acm.Points.from_numpy(ctx, xyz), acm.Points.from_numpy(ctx, uv)
    if name != "pinhole":
        m.linear_estimation(X, UV)
    om = oracle_model(O, dict(cam, params=list(m.params())))
    b = acm.CONVERTER_BOUNDS.get(m.MODEL_ID)
    lo, hi = (None, None) if b is None else ([x[0] for x in b], [x[1] for x in b])
    return m, om, X, UV, xyz, uv, lo, hi


def solve_once(ctx, cost, **kw):
    before = ctx.kernel_launches()
    r = cost.optimize(**kw)
    assert ctx.kernel_launches() - before == 1
    return r


def assert_same_solve(r, oo, ores, what):
    msg = (what, (r.status, r.iterations, r.passes, r.final_cost), (ores.status, ores.iterations, ores.passes, ores.final_cost))
    assert (r.status, r.iterations, r.passes) == (ores.status, ores.iterations, ores.passes), msg
    assert r.n_valid == ores.n_valid, msg
    assert np.allclose(r.parameters, oo, rtol=1e-9, atol=0), (msg, np.abs(r.parameters - oo) / np.abs(oo))
    assert abs(r.final_cost - ores.final_cost) <= 1e-9 * ores.final_cost, msg


@pytest.mark.parametrize("name,kind", PAIRS, ids=PAIR_IDS)
def test_lm_solve_at_steady_state(acm, ctx, O, cameras, sizes, name, kind):
    """lin_kernel<M, KIND, BS, true> (the whole solve in one cooperative launch) at n = 12*T + 75, with the converter's
    configuration and bounds (Pinhole: none).  Below WIDE_BLOCK_FROM the solve runs 128-thread blocks, at most T / 128
    of them, so every thread streams at least 6 packets per pass and the solve ring (2-4 deep) wraps within each pass.
    It must walk the oracle's trajectory: status, iterations and passes equal, n_valid exact, parameters and final cost
    within 1e-9."""
    n = sizes["lin"]
    m, om, X, UV, xyz, uv, lo, hi = solve_problem(acm, ctx, O, cameras, name, n, 0xACE50019 + MODELS.index(name))
    oo, ores = O.lm_solve(om, kind, xyz, uv, lo, hi, nthreads=NT)
    cost = acm.OptimizationCost(m, X, UV, residual_kind=kind)
    r = solve_once(ctx, cost, bounds="converter" if lo is not None else None)
    assert_same_solve(r, oo, ores, (name, kind))
    X.free(); UV.free()


@pytest.mark.parametrize("n_offset", [-1, 1])
@pytest.mark.parametrize("kind", [0, 1])
def test_lm_solve_double_sphere_around_wide_block_threshold(acm, ctx, O, cameras, sizes, kind, n_offset):
    """Double Sphere switches its solve from 128-thread blocks (capped at 2 per SM) to one uncapped 256-thread block
    per SM at WIDE_BLOCK_FROM = 4,000,000 correspondences: n = 3,999,999 and 4,000,001 run either form, with at
    least (n / 2) / T packets per thread and pass, on both residuals."""
    n = 4_000_000 + n_offset
    m, om, X, UV, xyz, uv, lo, hi = solve_problem(acm, ctx, O, cameras, "double_sphere", n, 0xACE5001A)
    oo, ores = O.lm_solve(om, kind, xyz, uv, lo, hi, nthreads=NT)
    cost = acm.OptimizationCost(m, X, UV, residual_kind=kind)
    r = solve_once(ctx, cost)
    assert_same_solve(r, oo, ores, ("double_sphere", kind, n))
    X.free(); UV.free()


@pytest.mark.parametrize("name,kind", PAIRS, ids=PAIR_IDS)
def test_lm_invalid_penalty_at_steady_state(acm, ctx, O, cameras, sizes, name, kind):
    """invalid_penalty inside the solve kernel (cost += 2 pen^2 / 2 per rejected point, counted per thread from its
    packet count) at n = 12*T + 75 with 2 % rejected points: the initial cost of an evaluation-only solve
    (max_iterations = 0) for penalty 1 and 10, then a full solve with penalty 1 along the oracle's trajectory."""
    cam = cameras[name]
    n = sizes["lin"]
    truth = oracle_model(O, cam)
    xyz, obs = invalid_mix(O, truth, name, n, 0xACE5001B + 16 * MODELS.index(name) + kind)
    start = dict(cam, params=list(np.array(cam["params"][:4]) * [1.01, 0.99, 1.005, 0.995]) + cam["params"][4:])
    m, om = gpu_model(acm, ctx, start), oracle_model(O, start)
    b = acm.CONVERTER_BOUNDS.get(m.MODEL_ID)
    lo, hi = (None, None) if b is None else ([x[0] for x in b], [x[1] for x in b])
    X, UV = acm.Points.from_numpy(ctx, xyz), acm.Points.from_numpy(ctx, obs)
    cost = acm.OptimizationCost(m, X, UV, residual_kind=kind)
    bounds = "converter" if lo is not None else None
    for pen in (1.0, 10.0):
        ocfg = O.lm_default_config(); ocfg.max_iterations = 0; ocfg.invalid_penalty = pen
        oo, ores = O.lm_solve(om, kind, xyz, obs, lo, hi, ocfg, nthreads=NT)
        assert n - ores.n_valid >= n // 100
        m.set_params(start["params"])
        r = solve_once(ctx, cost, config=acm.LevenbergMarquardtConfig(max_iterations=0, invalid_penalty=pen), bounds=bounds)
        assert (r.status, r.iterations, r.passes, r.n_valid) == (ores.status, ores.iterations, ores.passes, ores.n_valid)
        assert abs(r.initial_cost - ores.initial_cost) <= RTOL * ores.initial_cost, (pen, r.initial_cost, ores.initial_cost)
    ocfg = O.lm_default_config(); ocfg.invalid_penalty = 1.0
    oo, ores = O.lm_solve(om, kind, xyz, obs, lo, hi, ocfg, nthreads=NT)
    m.set_params(start["params"])
    r = solve_once(ctx, cost, config=acm.LevenbergMarquardtConfig(invalid_penalty=1.0), bounds=bounds)
    assert abs(r.initial_cost - ores.initial_cost) <= RTOL * ores.initial_cost
    assert_same_solve(r, oo, ores, (name, kind, "penalty 1"))
    X.free(); UV.free()
