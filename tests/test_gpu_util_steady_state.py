"""The kernels around the LM solve in the converter (acm_util.cu, acm_image.cu) at converter scale, at their branch edges
and against exact references.

test_gpu_parity.py compares reprojection statistics, sample_points and linear estimation with the oracle at sizes where
most threads handle one point or none.  Here every size is derived from the device (S = sm_count):

    N = 3 * S * 2048 + 77

which gives >= 3 grid-stride trips of the radix-select histogram (S*8 blocks of 256), >= 6 of reprojection pass 1
(S*4 blocks), 12 of the linest_* kernels (S*2 blocks) and >= 55 points per thread of the FOV pre-filter (64 blocks):
its float sums are flushed to double every 16 points, so every thread flushes several times.

Bars: the arithmetic-only models (EXACT of test_gpu_parity.py) project bit for bit like the oracle, so their error
counts, minima, maxima and medians are held bit-exact, and the sums within 1e-12 of math.fsum; KB and FOV keep the 1e-9
of test_gpu_parity.py.  Linear estimation is held to the exact least-squares solutions of tests/util_reference.py.
"""
import ctypes as C
import math
import os

import numpy as np
import pytest

from conftest import oracle_model
from test_gpu_parity import EXACT, MODELS, RTOL, UNIFIED, cone, gpu_model
import util_reference as R

pytestmark = pytest.mark.gpu

NT = min(os.cpu_count() or 1, 16)   # oracle threads where the oracle takes them
KB_CONE = float(np.cos(np.deg2rad(80.0)))


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
    z = {
        "S": S,
        "N": 3 * S * 2048 + 77,
        "pass1_trip": S * 4 * 256,
        "select_trip": S * 8 * 256,
        "linest_trip": S * 2 * 256,
        "prefilter_threads": 64 * 256,
    }
    print(f"\n[util steady-state sizes] device_info={ctx.device_info()} " + ", ".join(f"{k}={v}" for k, v in z.items()))
    return z


def oracle_error_class(acm, rc):
    return {-2: acm.InvalidParams, -4: acm.NumericalError}[rc]


# ------------------------------------------------------------------ reprojection statistics ----------------------
FIELDS = ("rmse", "min", "max", "mean", "stddev", "median")


def reproj_data(O, om, name, n, seed):
    """Correspondences with every 13th point moved behind the camera (Double Sphere still accepts about half of them)
    and, for Pinhole and RadTan, a 60-degree cone, so that many points project outside the image.  Observations: the oracle's projection plus 0.3 px of noise."""
    cos_max = float(np.cos(np.deg2rad(60.0))) if name in ("pinhole", "rad_tan") else cone(name)
    xyz = O.synth_points3(seed, 0, n, cos_max, False)
    xyz[::13, 2] = -1.0 - np.abs(xyz[::13, 2])
    uv, st = O.project(om, xyz, NT)
    uv = np.where(np.isnan(uv), 0.0, uv) + np.random.default_rng(seed).normal(0.0, 0.3, (n, 2))
    return xyz, uv, st


def error_vector(O, om, xyz, uv):
    """The errors of the points the oracle's projection accepts (with its image-bounds test), in point order."""
    p, st = O.project(om, xyz, NT)
    ok = st == 0
    dx, dy = p[ok, 0] - uv[ok, 0], p[ok, 1] - uv[ok, 1]
    with np.errstate(over="ignore"):
        return np.sqrt(dx * dx + dy * dy)


def exact_stats(e, mean_for_stddev=None):
    """count / min / max / median as the reference defines them, the sums through math.fsum.  The standard deviation
    is taken about `mean_for_stddev` when given: about a mean of 0.1 px and a spread of 1e-14, one ulp of the mean moves
    it by 1e-8 relative, so the second pass is checked on the mean it was given."""
    m = len(e)
    s = np.sort(e)
    median = (s[m // 2 - 1] + s[m // 2]) / 2.0 if m % 2 == 0 else s[m // 2]
    with np.errstate(invalid="ignore", over="ignore"):
        mean = math.fsum(e) / m
        rmse = math.sqrt(math.fsum(e * e) / m)
        mu = mean if mean_for_stddev is None else mean_for_stddev
        d = e - mu
        var = math.fsum(d * d) / m if math.isfinite(mu) else math.nan
    return {"count": m, "min": s[0], "max": s[-1], "median": median, "mean": mean, "rmse": rmse,
            "stddev": math.sqrt(var) if var == var else math.nan}


def same(a, b):
    return (a == b) or (a != a and b != b)


def close(a, b, rtol, atol=0.0):
    if not (math.isfinite(a) and math.isfinite(b)):
        return same(a, b)
    return abs(a - b) <= rtol * abs(b) + atol


def assert_stats(acm, m, om, O, name, xyz, uv):
    e = acm.compute_reprojection_error(m, xyz, uv)
    eo = O.reprojection_error(om, xyz, uv)
    assert e.count == eo.count
    for f in FIELDS:   # the NaN / inf pattern is the oracle's
        a, b = getattr(e, f), getattr(eo, f)
        assert math.isfinite(a) == math.isfinite(b) and math.isnan(a) == math.isnan(b), (f, a, b)
    if name in EXACT:
        ref = exact_stats(error_vector(O, om, xyz, uv), e.mean)
        assert e.count == ref["count"]
        for f in ("min", "max", "median"):
            assert same(getattr(e, f), ref[f]) and same(getattr(eo, f), ref[f]), (f, getattr(e, f), getattr(eo, f), ref[f])
        for f in ("mean", "rmse", "stddev"):
            assert close(getattr(e, f), ref[f], 1e-12), (f, getattr(e, f), ref[f])
    else:
        for f in FIELDS:
            assert close(getattr(e, f), getattr(eo, f), 1e-9, 1e-13), (f, getattr(e, f), getattr(eo, f))
    return e


@pytest.mark.parametrize("name", MODELS)
def test_reprojection_error_at_converter_scale(acm, ctx, O, cameras, sizes, name):
    """All 7 models at N points (>= 6 trips of pass 1, >= 3 of the select histogram, an odd count) and at 2 and 3
    points (point 0 is behind the camera), with rejected points interleaved."""
    cam = cameras[name]
    m, om = gpu_model(acm, ctx, cam), oracle_model(O, cam)
    for n in (sizes["N"], 2, 3):
        xyz, uv, st = reproj_data(O, om, name, n, 0xACE5B000 + MODELS.index(name))
        if n > 3:
            assert n - np.count_nonzero(st == 0) >= n // 30
            if name in ("pinhole", "rad_tan"):
                assert np.any((st != 0) & (xyz[:, 2] > 0))   # outside the image
        if not np.any(st == 0):
            with pytest.raises(acm.ZeroProjectionPoints):
                acm.compute_reprojection_error(m, xyz, uv)
            continue
        e = assert_stats(acm, m, om, O, name, xyz, uv)
        assert e.count == np.count_nonzero(st == 0)


def median_case(O, om, case, n, odd, seed):
    """Observations for one edge case of the radix select: (xyz, uv).  Every 13th point is behind the camera, and one
    more when that is needed for an odd (even) number of valid points."""
    xyz = O.synth_points3(seed, 0, n, cone("double_sphere"), False)
    xyz[::13, 2] = -1.0 - np.abs(xyz[::13, 2])
    _, st = O.project(om, xyz, NT)
    if (np.count_nonzero(st == 0) % 2 == 1) != odd:
        j = np.flatnonzero(st == 0)[0]
        xyz[j, 2] = -1.0 - abs(xyz[j, 2])
    p, st = O.project(om, xyz, NT)
    ok = np.flatnonzero(st == 0)
    assert (len(ok) % 2 == 1) == odd
    uv = np.where(np.isnan(p), 0.0, p)
    rng = np.random.default_rng(seed)
    if case == "ties":
        uv[:, 0] += 0.1
    elif case == "half_zero":    # floor(m / 2) errors exactly 0, the others >= 0.5: the middle ranks straddle the top digit
        pos = rng.permutation(ok)[: len(ok) - len(ok) // 2]
        uv[pos, 0] += rng.uniform(0.5, 2.0, len(pos))
    elif case == "inf":          # 1 % of the errors overflow to +inf: mean and rmse inf, stddev NaN, median finite
        big = rng.choice(ok, len(ok) // 100, replace=False)
        uv[big, 0] += 1e300
    return xyz, uv


@pytest.mark.parametrize("case", ["zero", "ties", "half_zero", "inf"])
@pytest.mark.parametrize("parity", ["odd", "even"])
def test_reprojection_median_edge_cases(acm, ctx, O, cameras, sizes, case, parity):
    """Double Sphere (bit-exact projections) at about N points, with an odd and an even number of valid errors:
    every error exactly 0; heavy ties (observation = projection + 0.1 px); half the errors 0 and half positive, so that
    for an even count the two middle ranks fall in different buckets of the first digit; some errors +inf."""
    cam = cameras["double_sphere"]
    m, om = gpu_model(acm, ctx, cam), oracle_model(O, cam)
    xyz, uv = median_case(O, om, case, sizes["N"], parity == "odd", 0xACE5B100)
    e = assert_stats(acm, m, om, O, "double_sphere", xyz, uv)
    assert (e.count % 2 == 1) == (parity == "odd")
    if case == "zero":
        assert e.max == 0.0 and e.median == 0.0 and e.mean == 0.0
    elif case == "ties":
        assert len(np.unique(error_vector(O, om, xyz, uv))) < e.count // 100
    elif case == "half_zero":   # odd: the smallest positive error; even: half of it
        assert e.min == 0.0 and (0.49 if parity == "odd" else 0.24) <= e.median < 2.0
    else:
        assert e.max == math.inf and e.mean == math.inf and math.isnan(e.stddev) and math.isfinite(e.median)


@pytest.mark.parametrize("parity", ["odd", "even"])
def test_reprojection_tiny_errors(acm, ctx, O, sizes, parity):
    """Errors between 1e-160 and 1e-155, whose squares (and the squared deviations) are subnormal, mixed with exact
    zeros: a Pinhole camera with its principal point at (0, 0), points just off the axis on the +x side and every
    observation at (0, 0).  (An error sqrt(dx^2 + dy^2) is never itself subnormal: such a dx^2 underflows to 0.)"""
    n = sizes["N"] + (0 if parity == "odd" else 1)
    cam = {"model_id": MODELS.index("pinhole"), "params": [500.0, 500.0, 0.0, 0.0], "width": 640, "height": 480}
    m, om = gpu_model(acm, ctx, cam), oracle_model(O, cam)
    rng = np.random.default_rng(0xACE5B200)
    xyz = np.zeros((n, 3))
    xyz[:, 0] = np.exp(rng.uniform(np.log(2e-163), np.log(2e-158), n))
    xyz[::7, 0] = 0.0
    xyz[:, 2] = 1.0
    uv = np.zeros((n, 2))
    e = assert_stats(acm, m, om, O, "pinhole", xyz, uv)
    assert e.count == n and e.min == 0.0 and 0.0 < e.median < 1e-154 and 0.0 < e.stddev < 1e-154


def test_reprojection_error_of_sampled_device_points(acm, ctx, O, cameras, sizes):
    """The converter's path: compute_reprojection_error on the device Points that sample_points(device=True) returns
    (KB: some cells are dropped, so their capacity exceeds their length) equals the same call on host copies."""
    cam = cameras["kannala_brandt"]
    m = gpu_model(acm, ctx, cam)
    n = sizes["N"]
    UV, X = acm.sample_points(m, n, device=True)
    ncx, ncy = (math.floor(math.sqrt(n * r) + 0.5) for r in (cam["width"] / cam["height"], cam["height"] / cam["width"]))
    assert len(X) < ncx * ncy
    uv, xyz = UV.numpy(), X.numpy()
    obs = uv + np.random.default_rng(3).normal(0.0, 0.3, uv.shape)
    OBS = acm.Points.from_numpy(ctx, obs)
    for pts, ref in ((UV, uv), (OBS, obs)):
        e_dev = acm.compute_reprojection_error(m, X, pts)
        e_host = acm.compute_reprojection_error(m, xyz, ref)
        for f in FIELDS + ("count",):
            assert same(getattr(e_dev, f), getattr(e_host, f)), f
        assert e_dev.count == len(xyz)
    eo = O.reprojection_error(oracle_model(O, cam), xyz, obs)
    assert e_dev.count == eo.count and close(e_dev.median, eo.median, 1e-9, 1e-13)
    UV.free(); X.free(); OBS.free()


# ------------------------------------------------------------------ sample_points -----------------------------------
def square(cam, side=512):
    return dict(cam, width=side, height=side)


@pytest.mark.parametrize("k", [512, 513, 887])
@pytest.mark.parametrize("name", MODELS)
def test_sample_points_block_scan_tiles(acm, ctx, O, cameras, name, k):
    """A square camera and n = k^2 give k^2 cells: k = 512 is exactly 1024 blocks (one scan tile), 513 one block past
    the first tile, 887 three tiles and 2 blocks.  Pixels bit-exact and in order; rays bit-exact for EXACT."""
    cam = square(cameras[name])
    m, om = gpu_model(acm, ctx, cam), oracle_model(O, cam)
    nblk = (k * k + 255) // 256
    assert (k, nblk) in ((512, 1024), (513, 1029), (887, 3074))
    uv, xyz = acm.sample_points(m, k * k)
    uvo, xyzo = O.sample_points(om, k * k)
    assert uv.shape == uvo.shape, "kept set differs"
    assert np.array_equal(uv, uvo)
    if name in EXACT:
        assert np.array_equal(xyz, xyzo)
    else:
        assert np.allclose(xyz, xyzo, rtol=RTOL, atol=1e-15)


@pytest.mark.parametrize("n_shards", [2, 3, 7, 8])
@pytest.mark.parametrize("name", ["kannala_brandt", "rad_tan"])
def test_sample_points_shards_concatenate_to_the_whole(acm, ctx, cameras, name, n_shards):
    """acm_sample_points_shard (the multi-GPU converter's split, a pure function of (shard, n_shards)) on one GPU: the
    shards in order are bit-identical to the unsharded output.  887^2 cells put every shard boundary mid-row and
    mid-block."""
    m = gpu_model(acm, ctx, square(cameras[name]))
    k = 887
    cells = k * k
    bounds = [cells * s // n_shards for s in range(1, n_shards)]
    assert all(b % k and b % 256 for b in bounds), bounds
    uv, xyz = acm.sample_points(m, cells)
    parts = [acm.sample_points(m, cells, shard=(s, n_shards)) for s in range(n_shards)]
    assert all(len(p[0]) > 0 for p in parts)
    assert np.array_equal(np.concatenate([p[0] for p in parts]), uv)
    assert np.array_equal(np.concatenate([p[1] for p in parts]), xyz)


def test_sample_points_more_shards_than_cells(acm, ctx, O, cameras):
    """n_requested = 2 on a square camera is one cell: with 8 shards, shards 0-6 are empty and return no point and no
    error, shard 7 returns the cell."""
    cam = square(cameras["double_sphere"])
    m, om = gpu_model(acm, ctx, cam), oracle_model(O, cam)
    uvo, xyzo = O.sample_points(om, 2)
    assert len(uvo) == 1
    parts = [acm.sample_points(m, 2, shard=(s, 8)) for s in range(8)]
    assert [len(p[0]) for p in parts] == [0] * 7 + [1]
    assert np.array_equal(parts[7][0], uvo) and np.array_equal(parts[7][1], xyzo)


# ------------------------------------------------------------------ linear estimation --------------------------------
INITS = {"double_sphere": [0.5, 0.1], "ucm": [0.5], "eucm": [0.5, 1.0], "fov": [1.0], "kannala_brandt": [0.0] * 4, "rad_tan": [0.0] * 5}


def kb_source(O, cameras, n, seed, cos_max=KB_CONE, noise=0.2):
    """Correspondences of the KB sample camera on a 512 x 512 image: (intrinsics, xyz, noisy uv)."""
    c = cameras["kannala_brandt"]
    xyz = O.synth_points3(seed, 0, n, cos_max, False)
    uv, st = O.project(oracle_model(O, dict(c, width=512, height=512)), xyz, NT)
    uv = np.where(np.isnan(uv), 0.0, uv) + np.random.default_rng(seed).normal(0.0, noise, (n, 2))
    return c["params"][:4], xyz, uv


def estimate(acm, ctx, O, model_id, params, xyz, uv):
    """(device params, oracle params) after linear estimation from the same start."""
    cam = {"model_id": model_id, "params": list(params), "width": 512, "height": 512}
    m, om = gpu_model(acm, ctx, cam), oracle_model(O, cam)
    X, UV = acm.Points.from_numpy(ctx, xyz), acm.Points.from_numpy(ctx, uv)
    m.linear_estimation(X, UV)
    X.free(); UV.free()
    assert O.linear_estimation(om, xyz, uv) == 0
    return m.params(), om.params()


def normwise(x, ref):
    return np.linalg.norm(np.asarray(x) - ref) / np.linalg.norm(ref)


@pytest.mark.parametrize("name", sorted(UNIFIED))
def test_linear_estimation_unified_at_converter_scale(acm, ctx, O, cameras, sizes, name):
    """linest_unified_kernel at N (12 trips): the device's rows are IEEE arithmetic like the numpy rows, its sums
    double-double, so alpha is within 2 ulp of the exact least-squares solution; the oracle sums sequentially (within
    1e-12)."""
    intr, xyz, uv = kb_source(O, cameras, sizes["N"], 0xACE5C000)
    A, b = R.unified_rows(xyz, uv, intr)
    ref = R.ls_reference(A, b, 1e-10)[0]
    assert 0.0 < ref <= 1.0                       # no clamp applies
    got, orc = estimate(acm, ctx, O, cameras[name]["model_id"], intr + INITS[name], xyz, uv)
    assert abs(got[4] - ref) <= 2 * np.spacing(ref), ((got[4] - ref) / np.spacing(ref))
    assert abs(got[4] - orc[4]) <= 1e-12 * abs(orc[4])
    assert np.array_equal(got[:4], intr)


def kb_with_branches(O, cameras, n, seed):
    """KB correspondences with points on the axis (rw < EPS; half of them observed at the principal point) and points
    at or behind the camera (z <= EPS), at RNG-chosen places."""
    intr, xyz, uv = kb_source(O, cameras, n, seed)
    rng = np.random.default_rng(seed)
    idx = rng.permutation(n)
    axis, behind = idx[:2000], idx[2000:3000]
    xyz[axis, :2] = 0.0
    uv[axis[:1000]] = intr[2:4]
    xyz[behind[:500], 2] = 0.0
    xyz[behind[500:], 2] = -np.abs(xyz[behind[500:], 2])
    return intr, xyz, uv


def test_linear_estimation_kannala_brandt_at_converter_scale(acm, ctx, O, cameras, sizes):
    """linest_kb_kernel and its GridReduce<1, 0, 14> at N.  theta comes from acm_atan2_q1, a few ulp from the numpy
    rows', so the bar against the exact solution is 1e-10 normwise; against the oracle 1e-12."""
    intr, xyz, uv = kb_with_branches(O, cameras, sizes["N"], 0xACE5C100)
    A, b, numerical = R.kb_rows(xyz, uv, intr)
    assert not numerical
    ref = R.ls_reference(A, b, R.EPS)
    got, orc = estimate(acm, ctx, O, cameras["kannala_brandt"]["model_id"], intr + INITS["kannala_brandt"], xyz, uv)
    assert normwise(got[4:8], ref) <= 1e-10, (got[4:8], ref)
    assert normwise(got[4:8], orc[4:8]) <= 1e-12, (got[4:8], orc[4:8])


def test_linear_estimation_kannala_brandt_450_sample_against_exact(acm, ctx, O, cameras):
    """The 450-point sample (test_gpu_parity.py holds it to the oracle within 1e-7).  cond(A) is ~670 (cond of the
    normal matrix ~4.5e5); moving every theta of the numpy rows by a random 2 ulp moves the exact solution by at most
    1.2e-13 normwise, so 1e-11 leaves two orders of magnitude for the device's theta."""
    c = cameras["kannala_brandt"]
    uv, xyz = O.sample_points(oracle_model(O, c), 500)
    assert len(uv) == 450
    intr = c["params"][:4]
    A, b, _ = R.kb_rows(xyz, uv, intr)
    ref = R.ls_reference(A, b, R.EPS)
    got, _ = estimate(acm, ctx, O, c["model_id"], intr + INITS["kannala_brandt"], xyz, uv)
    assert normwise(got[4:8], ref) <= 1e-11, normwise(got[4:8], ref)


def test_linear_estimation_rad_tan_at_converter_scale(acm, ctx, O, cameras, sizes):
    """linest_radtan_kernel and its GridReduce<0, 0, 9> at N correspondences of the sample RadTan camera (40-degree
    cone, 0.1 px noise): 1e-12 normwise against the exact solution and the oracle; p1 = p2 = 0."""
    c = cameras["rad_tan"]
    n = sizes["N"]
    xyz = O.synth_points3(0xACE5C200, 0, n + n // 2, float(np.cos(np.deg2rad(40.0))), False)
    uv, st = O.project(oracle_model(O, c), xyz, NT)
    keep = np.flatnonzero(st == 0)[:n]
    assert len(keep) == n
    xyz, uv = np.ascontiguousarray(xyz[keep]), np.ascontiguousarray(uv[keep]) + np.random.default_rng(5).normal(0.0, 0.1, (n, 2))
    intr = c["params"][:4]
    A, b = R.radtan_rows(xyz, uv, intr)
    ref = R.ls_reference(A, b, 1e-10)
    cam = dict(c, params=intr + INITS["rad_tan"])
    m, om = gpu_model(acm, ctx, cam), oracle_model(O, cam)
    m.linear_estimation(xyz, uv)
    assert O.linear_estimation(om, xyz, uv) == 0
    got, orc = m.params(), om.params()
    assert normwise(got[[4, 5, 8]], ref) <= 1e-12, (got[[4, 5, 8]], ref)
    assert normwise(got[[4, 5, 8]], orc[[4, 5, 8]]) <= 1e-12
    assert got[6] == 0.0 and got[7] == 0.0


# ------------------------------------------------------------------ FOV grid search ----------------------------------
def fov_cone(O, cameras, n, behind_only=False, seed=0xACE5D000):
    """A FOV camera with w = 0.93 on a 100-degree cone (about 15 % of the points behind the camera; with
    `behind_only`, only such points), 0.3 px noise."""
    intr = cameras["kannala_brandt"]["params"][:4]
    fx, fy, cx, cy = intr
    cos100 = float(np.cos(np.deg2rad(100.0)))
    if behind_only:
        xyz = O.synth_points3(seed, 0, 8 * n, cos100, False)
        xyz = np.ascontiguousarray(xyz[xyz[:, 2] < 0][:n])
        assert len(xyz) == n
    else:
        xyz = O.synth_points3(seed, 0, n, cos100, False)
    x, y, z = xyz[:, 0], xyz[:, 1], xyz[:, 2]
    r = np.sqrt(x * x + y * y)
    rd = np.arctan2(2.0 * math.tan(0.93 / 2.0) * r, z) / (r * 0.93)
    uv = np.column_stack([fx * x * rd + cx, fy * y * rd + cy]) + np.random.default_rng(seed).normal(0.0, 0.3, (n, 2))
    assert np.count_nonzero(z < 0) > n // 10
    return intr, xyz, uv


def fov_flat(n, seed=0xACE5D100):
    """Every observation at (40, 30), fx = 190, principal point (256, 256), and points within 1e-7 of the axis along
    the direction from the principal point towards the observation: the near-axis projection moves towards the
    observation by fx * r * 2 tan(w / 2) / w, so the mean error falls with w by ~3e-8 relative per unit of that factor.
    All 290 candidates lie within 2.4e-7 of the minimum, the arg-min is the last one (w = 2.99), and it is 1.6e-8 below
    the runner-up."""
    rng = np.random.default_rng(seed)
    c, o = np.array([256.0, 256.0]), np.array([40.0, 30.0])
    d = (c - o) / np.linalg.norm(c - o)
    mag, perp = rng.uniform(0.0, 1e-7, n), rng.normal(0.0, 1e-8, n)
    xyz = np.column_stack([-mag * d[0] - perp * d[1], -mag * d[1] + perp * d[0], np.ones(n)])
    return [190.0, 190.0, 256.0, 256.0], xyz, np.tile(o, (n, 1))


def fov_check(acm, ctx, O, cameras, intr, xyz, uv):
    means = R.fov_mean_errors(xyz, uv, intr)
    best, gap = R.fov_runner_up_gap(means)
    assert gap >= 1e-9, gap                                  # no tie for the device's summation order to break
    got, orc = estimate(acm, ctx, O, cameras["fov"]["model_id"], intr + INITS["fov"], xyz, uv)
    assert orc[4] == R.FOV_W[R.fov_argmin(means)]
    assert got[4] == orc[4], (got[4], orc[4])
    return means, got[4]


@pytest.mark.parametrize("n", ["N", "N_behind", 199_999, 200_000])
def test_fov_grid_search_behind_the_camera(acm, ctx, O, cameras, sizes, n):
    """The z < 0 branches of both FOV kernels (atan2 in the exact search, pi - a in the float pre-filter) on a
    100-degree cone, at N (pre-filter with >= 55 points per thread, its flushes, then the exact shortlist) and on
    either side of the 200,000-point switch to the two-stage search.  In the cone 85 % of the points lie in front
    and decide the arg-min on their own, so the N_behind set (N points, all behind the camera) is the one that needs
    the pre-filter's z < 0 branch to shortlist w = 0.93."""
    intr, xyz, uv = fov_cone(O, cameras, sizes["N"], behind_only=n == "N_behind")
    n = sizes["N"] if n in ("N", "N_behind") else n
    means, w = fov_check(acm, ctx, O, cameras, intr, xyz[:n], uv[:n])
    assert w == 0.93


def test_fov_grid_search_shortlist_overflow(acm, ctx, O, cameras, sizes):
    """A flat error curve at N: the pre-filter's shortlist (every candidate within its float rounding bound, ~1e-5
    relative, of the best) holds more than 32 candidates, so the search falls back to the exact evaluation of all
    290.  Any candidate within 1e-6 of the minimum is certainly on the shortlist, and more than 32 of them precede the
    arg-min: a shortlist cut to its first 32 entries would miss it."""
    intr, xyz, uv = fov_flat(sizes["N"])
    means = R.fov_mean_errors(xyz, uv, intr)
    i = R.fov_argmin(means)
    best, _ = R.fov_runner_up_gap(means)
    near = (means - best) / best <= 1e-6
    assert np.count_nonzero(near) > 32
    assert np.count_nonzero(near[:i]) > 32
    _, w = fov_check(acm, ctx, O, cameras, intr, xyz, uv)
    assert w == R.FOV_W[i] == 2.99


# ------------------------------------------------------------------ minimum counts and errors ------------------------
@pytest.mark.parametrize("name,minimum", [("kannala_brandt", 4), ("fov", 2), ("eucm", 1), ("rad_tan", 3)])
def test_linear_estimation_minimum_counts(acm, ctx, O, cameras, name, minimum):
    """One point below the model's minimum: InvalidParams where the oracle returns -2.  At the minimum: the oracle's
    result (KB against the exact solution: cond(A) ~2e4 for these 4 points)."""
    c = cameras["kannala_brandt"]
    uv, xyz = O.sample_points(oracle_model(O, c), 500)
    if name == "rad_tan":
        rc_cam = cameras["rad_tan"]
        uv, xyz = O.sample_points(oracle_model(O, rc_cam), 500)
        intr, W, H = rc_cam["params"][:4], rc_cam["width"], rc_cam["height"]
    else:
        intr, W, H = c["params"][:4], 512, 512
    pick = np.linspace(0, len(uv) - 1, minimum).astype(int)
    cam = {"model_id": cameras[name]["model_id"], "params": intr + INITS[name], "width": W, "height": H}
    for k in (minimum - 1, minimum):
        sub = pick[:k] if k < minimum else pick
        x3, x2 = np.ascontiguousarray(xyz[sub]).reshape(-1, 3), np.ascontiguousarray(uv[sub]).reshape(-1, 2)
        m, om = gpu_model(acm, ctx, cam), oracle_model(O, cam)
        rc = O.linear_estimation(om, x3, x2)
        if k < minimum:
            assert rc == -2
            with pytest.raises(oracle_error_class(acm, rc)):
                m.linear_estimation(x3, x2)
            continue
        assert rc == 0
        m.linear_estimation(x3, x2)
        got, orc = m.params(), om.params()
        if name == "kannala_brandt":
            A, b, _ = R.kb_rows(x3, x2, intr)
            assert normwise(got[4:8], R.ls_reference(A, b, R.EPS)) <= 1e-8
        elif name == "fov":
            assert got[4] == orc[4]
        else:
            assert np.allclose(got, orc, rtol=1e-9, atol=1e-12), (got, orc)


def test_linear_estimation_kannala_brandt_zero_focal_product(acm, ctx, O, cameras):
    """fx = 1e-20 makes |fx * x_r| < EPS for off-axis points: NumericalError, where the oracle returns -4."""
    c = cameras["kannala_brandt"]
    uv, xyz = O.sample_points(oracle_model(O, c), 500)
    cam = {"model_id": c["model_id"], "params": [1e-20] + c["params"][1:4] + INITS["kannala_brandt"], "width": 512, "height": 512}
    m, om = gpu_model(acm, ctx, cam), oracle_model(O, cam)
    rc = O.linear_estimation(om, xyz, uv)
    assert rc == -4
    with pytest.raises(oracle_error_class(acm, rc)):
        m.linear_estimation(xyz, uv)


# ------------------------------------------------------------------ PSNR / SSIM byte path ------------------------------
def test_image_metrics_on_unaligned_device_buffers(acm, ctx, O):
    """acm_image_psnr / acm_image_ssim on images 1, 2 or 3 bytes into their allocations (either or both): psnr_kernel
    then reads bytes instead of 4-pixel words.  640 x 480 and 1023 x 517 (a tail after the last 4-pixel group); a black
    block shared by both images exercises the skip, and the last pixels differ.  PSNR equals the oracle's exactly,
    SSIM within 1e-12."""
    from apex_camera_models_b200 import _native as N
    for W, H in ((640, 480), (1023, 517)):
        a = O.synth_bytes(0xACE5E000 + W, 0, W * H * 3).reshape(H, W, 3)
        b = np.clip(a.astype(int) + np.random.default_rng(W).integers(-20, 21, a.shape), 0, 255).astype(np.uint8)
        a[100:150, 200:300] = 0
        b[100:150, 200:300] = 0
        a[-1, -1], b[-1, -1] = (250, 0, 0), (0, 0, 250)
        psnr_o, ssim_o = O.image_psnr(a, b), O.image_ssim(a, b)
        nbytes = W * H * 3
        pa, pb = ctx.device_alloc(nbytes + 4), ctx.device_alloc(nbytes + 4)
        try:
            for off in (1, 2, 3):
                for oa, ob in ((off, 0), (0, off), (off, off)):
                    ctx.h2d(pa + oa, a)
                    ctx.h2d(pb + ob, b)
                    out = C.c_double()
                    ctx.check(N.lib.acm_image_psnr(ctx.handle, C.c_void_p(pa + oa), C.c_void_p(pb + ob), W, H, C.byref(out)))
                    assert out.value == psnr_o, (W, oa, ob, out.value, psnr_o)
                    ctx.check(N.lib.acm_image_ssim(ctx.handle, C.c_void_p(pa + oa), C.c_void_p(pb + ob), W, H, C.byref(out)))
                    assert abs(out.value - ssim_o) <= 1e-12, (W, oa, ob, out.value, ssim_o)
        finally:
            ctx.device_free(pa); ctx.device_free(pb)
