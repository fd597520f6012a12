"""The exact references of tests/util_reference.py checked against exact rational arithmetic and against the oracle,
before the GPU tests (test_gpu_util_steady_state.py) hold the device's linear estimation to them.  CPU only."""
import math
import random
from fractions import Fraction

import numpy as np
import pytest

from conftest import oracle_model
import util_reference as R

RAD_TAN_TRUTH_CONE = float(np.cos(np.deg2rad(40.0)))
KB_CONE = float(np.cos(np.deg2rad(80.0)))


def assert_exact_dot(a, b):
    exact = sum((Fraction(x) * Fraction(y) for x, y in zip(a, b)), Fraction(0))
    hi, lo = R.exact_dot(np.array(a), np.array(b))
    assert hi == float(exact), (hi, float(exact))              # Fraction -> float rounds to nearest
    assert lo == float(exact - Fraction(hi)), (lo, float(exact - Fraction(hi)))


def test_exact_dot_is_exact_on_adversarial_inputs():
    """Cancelling sums, products whose low word carries the result, and wide exponent ranges."""
    e = 2.0 ** -30
    assert_exact_dot([1e16, 1.0, -1e16], [1.0, 1.0, 1.0])                        # the 1 survives the cancellation
    assert_exact_dot([1.0 + e, -1.0], [1.0 - e, 1.0])                             # = -2^-60: only the low word
    assert_exact_dot([1.0 + 2.0 ** -52, 1.0 + 2.0 ** -52, -1.0], [1.0 - 2.0 ** -52, 1.0 + 2.0 ** -52, 2.0])
    assert_exact_dot([3.0 ** 20, -(3.0 ** 20)], [3.0 ** 20 + 1.0, 3.0 ** 20])     # products beyond 2^53
    hi, lo = R.exact_dot(np.array([1e16, 1.0, -1e16]), np.ones(3))
    assert (hi, lo) == (1.0, 0.0)
    hi, lo = R.exact_dot(np.array([1.0 + e, -1.0]), np.array([1.0 - e, 1.0]))
    assert hi == -(2.0 ** -60) and lo == 0.0
    rng = random.Random(5)
    for _ in range(200):
        n = rng.randint(1, 40)
        a = [rng.uniform(-1, 1) * 2.0 ** rng.randint(-40, 40) for _ in range(n)]
        b = [rng.uniform(-1, 1) * 2.0 ** rng.randint(-40, 40) for _ in range(n)]
        if rng.random() < 0.5:             # append the negated sum of the products: massive cancellation
            k = float(sum(Fraction(x) * Fraction(y) for x, y in zip(a, b)))
            a.append(-k); b.append(1.0)
        assert_exact_dot(a, b)


def test_ls_reference_solves_exactly_representable_systems():
    """A system with an exact solution is solved to the last bit, and sigma <= eps components are dropped."""
    rng = np.random.default_rng(3)
    A = rng.integers(-50, 50, (40, 3)).astype(np.float64)
    x = np.array([0.5, -0.25, 3.0])
    assert np.array_equal(R.ls_reference(A, A @ x, 1e-10), x)
    B = np.column_stack([A[:, 0], A[:, 0]])          # rank 1: the minimum-norm solution
    assert np.allclose(R.ls_reference(B, A[:, 0], 1e-10), [0.5, 0.5], rtol=1e-15, atol=0)


def normwise(x, ref):
    return np.linalg.norm(np.asarray(x) - ref) / np.linalg.norm(ref)


def kb_sample_450(O, cameras):
    c = cameras["kannala_brandt"]
    uv, xyz = O.sample_points(oracle_model(O, c), 500)
    assert len(uv) == 450
    return c["params"][:4], xyz, uv


def kb_correspondences(O, cameras, n, seed):
    c = cameras["kannala_brandt"]
    xyz = O.synth_points3(seed, 0, n, KB_CONE, False)
    uv, st = O.project(oracle_model(O, dict(c, width=512, height=512)), xyz, 8)
    assert np.all(st == 0)
    return c["params"][:4], xyz, uv + np.random.default_rng(seed).normal(0.0, 0.2, uv.shape)


def rad_tan_correspondences(O, cameras, n, seed):
    c = cameras["rad_tan"]
    xyz = O.synth_points3(seed, 0, n + n // 2, RAD_TAN_TRUTH_CONE, False)
    uv, st = O.project(oracle_model(O, c), xyz, 8)
    keep = np.flatnonzero(st == 0)[:n]
    assert len(keep) == n
    xyz, uv = np.ascontiguousarray(xyz[keep]), np.ascontiguousarray(uv[keep])
    return c["params"][:4], xyz, uv + np.random.default_rng(seed).normal(0.0, 0.1, uv.shape)


def oracle_estimate(O, model_id, params, xyz, uv):
    om = O.make_model(model_id, params, 512, 512)
    assert O.linear_estimation(om, xyz, uv) == 0
    return om.params()


@pytest.mark.parametrize("name", ["ucm", "eucm", "double_sphere"])
def test_ls_reference_unified_alpha_matches_oracle(O, cameras, name):
    """alpha of the 2N x 1 unified system on the 450-point KB sample and on 200,000 KB correspondences: 1e-13."""
    for intr, xyz, uv in (kb_sample_450(O, cameras), kb_correspondences(O, cameras, 200_000, 0xACE5A1)):
        A, b = R.unified_rows(xyz, uv, intr)
        ref = R.ls_reference(A, b, 1e-10)[0]
        init = {"ucm": [0.5], "eucm": [0.5, 1.0], "double_sphere": [0.5, 0.1]}[name]
        alpha = oracle_estimate(O, cameras[name]["model_id"], intr + init, xyz, uv)[4]
        assert 0.0 < ref <= 1.0                      # no clamp of the model applies
        assert abs(alpha - ref) <= 1e-13 * abs(ref), (alpha, ref)


def test_ls_reference_kannala_brandt_matches_oracle(O, cameras):
    """k1..k4 on the 450-point sample (cond(A) ~ 1e5) and on 300,000 noisy correspondences in an 80-degree cone."""
    for intr, xyz, uv in (kb_sample_450(O, cameras), kb_correspondences(O, cameras, 300_000, 0xACE5A2)):
        A, b, numerical = R.kb_rows(xyz, uv, intr)
        assert not numerical
        ref = R.ls_reference(A, b, R.EPS)
        got = oracle_estimate(O, cameras["kannala_brandt"]["model_id"], intr + [0.0] * 4, xyz, uv)[4:8]
        assert normwise(got, ref) <= 1e-12, (got, ref, normwise(got, ref))


def test_ls_reference_rad_tan_matches_oracle(O, cameras):
    """k1, k2, k3 of the 2N x 3 RadTan system on 300,000 noisy correspondences of the sample camera."""
    intr, xyz, uv = rad_tan_correspondences(O, cameras, 300_000, 0xACE5A3)
    A, b = R.radtan_rows(xyz, uv, intr)
    ref = R.ls_reference(A, b, 1e-10)
    p = oracle_estimate(O, cameras["rad_tan"]["model_id"], intr + [0.0] * 5, xyz, uv)
    got = p[[4, 5, 8]]
    assert normwise(got, ref) <= 1e-12, (got, ref)
    assert p[6] == 0.0 and p[7] == 0.0


def test_kb_rows_take_the_oracle_branches(O, cameras):
    """Points on the axis (rw < EPS, with u == cx or not), behind or at the camera (z <= EPS) and fx * x_r == 0."""
    intr, xyz, uv = kb_correspondences(O, cameras, 1000, 0xACE5A4)
    xyz[:10, :2] = 0.0                       # on the axis
    uv[:5] = intr[2:4]                       # ... observed at the principal point: b = -theta
    xyz[10:20, 2] = -xyz[10:20, 2]           # behind: zero rows
    xyz[20:25, 2] = 0.0
    A, b, numerical = R.kb_rows(xyz, uv, intr)
    assert not numerical
    assert not A[20:50].any() and not b[20:50].any()
    assert np.all(b[:10] == 0.0) and np.all(A[:20] == 0.0)      # theta == 0 on the axis
    ref = R.ls_reference(A, b, R.EPS)
    got = oracle_estimate(O, cameras["kannala_brandt"]["model_id"], intr + [0.0] * 4, xyz, uv)[4:8]
    assert normwise(got, ref) <= 1e-11, (got, ref)
    _, _, numerical = R.kb_rows(xyz, uv, [1e-20, intr[1], intr[2], intr[3]])
    assert numerical
    assert O.linear_estimation(O.make_model(cameras["kannala_brandt"]["model_id"], [1e-20] + intr[1:] + [0.0] * 4, 512, 512), xyz, uv) == -4


def test_fov_evaluator_arg_min_matches_oracle(O, cameras):
    """The numpy evaluator of the 290 FOV candidates picks the oracle's w, on KB-generated correspondences."""
    intr, xyz, uv = kb_correspondences(O, cameras, 20_000, 0xACE5A5)
    means = R.fov_mean_errors(xyz, uv, intr)
    w = oracle_estimate(O, cameras["fov"]["model_id"], intr + [1.0], xyz, uv)[4]
    assert R.FOV_W[R.fov_argmin(means)] == w
    best, gap = R.fov_runner_up_gap(means)
    assert gap > 1e-9 and math.isfinite(best)
