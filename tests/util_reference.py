"""Exact references for the linear estimation of the camera models (CPU only, no GPU).

The device reduces the normal equations of the linear initialisers with exact products and double-double sums
(acm_util.cu), so the oracle's plain-double Jacobi SVD is not precise enough to hold it to its own accuracy.  These
helpers are:

- `exact_dot`: the dot product of two float64 vectors as a double-double (hi, lo) with hi + lo within one rounding of
  the exact sum: exact products (Veltkamp / Dekker splitting), then `math.fsum`, which is exactly rounded;
- `ls_reference`: the least-squares solution with nalgebra's `SVD::solve(b, eps)` semantics, from the Gram matrix of
  exact dot products, solved in mpmath at 50 digits;
- row builders that restate `orc_linear_estimation` (oracle/acm_oracle_solver.c) in numpy, row for row;
- `fov_mean_errors`: the mean error of each of the 290 FOV grid candidates in the oracle's arithmetic, used to build
  test data and to assert that a test's arg-min is not a tie.
"""
import math

import numpy as np

EPS = 2.220446049250313e-16            # f64::EPSILON
SQRT_EPS = 1.4901161193847656e-08      # its square root, the FOV near-axis threshold
FOV_W = np.arange(10, 300) / 100.0     # the FOV grid w = i / 100, i in [10, 300)
_SPLIT = 134217729.0                   # 2^27 + 1


def two_prod(a, b):
    """Elementwise (p, e) with p = fl(a * b) and p + e == a * b exactly (no FMA: numpy rounds every operation).
    Exact while no product or partial product leaves the normal range."""
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    p = a * b
    c = _SPLIT * a
    ah = c - (c - a)
    al = a - ah
    c = _SPLIT * b
    bh = c - (c - b)
    bl = b - bh
    e = ((ah * bh - p) + ah * bl + al * bh) + al * bl
    return p, e


def exact_dot(a, b):
    """sum(a[i] * b[i]) as a double-double: hi is the exactly rounded sum, lo the exactly rounded remainder."""
    p, e = two_prod(np.ravel(a), np.ravel(b))
    terms = np.concatenate([p, e]).tolist()
    hi = math.fsum(terms)
    terms.append(-hi)
    return hi, math.fsum(terms)


def ls_reference(A, b, eps, dps=50):
    """x = argmin |A x - b| as nalgebra's SVD::solve(b, eps): with the Gram matrix G = A^T A = Q diag(lambda) Q^T, the
    components whose singular value sqrt(lambda) is <= eps are dropped.  G and A^T b are exact_dot's double-doubles
    (relative error ~1e-32), the eigen-decomposition runs in mpmath at `dps` digits."""
    import mpmath as mp
    A = np.asarray(A, np.float64)
    A = A.reshape(len(A), -1)
    k = A.shape[1]
    cols = [np.ascontiguousarray(A[:, j]) for j in range(k)]
    with mp.workdps(dps):
        def dd(a, c):
            hi, lo = exact_dot(a, c)
            return mp.mpf(hi) + mp.mpf(lo)
        G, c = mp.matrix(k, k), mp.matrix(k, 1)
        for i in range(k):
            for j in range(i, k):
                G[i, j] = G[j, i] = dd(cols[i], cols[j])
            c[i] = dd(cols[i], b)
        lam, Q = mp.eigsy(G)
        x = [mp.mpf(0)] * k
        for i in range(k):
            if not (lam[i] > 0 and mp.sqrt(lam[i]) > eps):
                continue
            coef = mp.fsum(Q[r, i] * c[r] for r in range(k)) / lam[i]
            for r in range(k):
                x[r] += Q[r, i] * coef
        return np.array([float(v) for v in x])


def _interleave(r0, r1):
    """Rows 2i and 2i+1 from the per-point rows r0[i] and r1[i]."""
    r0, r1 = np.asarray(r0), np.asarray(r1)
    out = np.empty((2 * len(r0),) + r0.shape[1:])
    out[0::2], out[1::2] = r0, r1
    return out


def unified_rows(xyz, uv, intr):
    """UCM / EUCM / Double Sphere: 2N x 1 system a = (u - cx)(d - z), b = fx x - (u - cx) z."""
    fx, fy, cx, cy = intr
    x, y, z = xyz[:, 0], xyz[:, 1], xyz[:, 2]
    u, v = uv[:, 0], uv[:, 1]
    d = np.sqrt(x * x + y * y + z * z)
    u_cx, v_cy = u - cx, v - cy
    A = _interleave(u_cx * (d - z), v_cy * (d - z))[:, None]
    b = _interleave((fx * x) - (u_cx * z), (fy * y) - (v_cy * z))
    return A, b


def kb_rows(xyz, uv, intr):
    """Kannala-Brandt: rows [t^3, t^5, t^7, t^9] twice per point (zero rows where z <= EPS) and the right-hand side,
    including the on-axis (rw < EPS) branches.  Also returns whether the oracle stops with -4 ("fx * x_r is zero")."""
    fx, fy, cx, cy = intr
    xw, yw, zw = xyz[:, 0], xyz[:, 1], xyz[:, 2]
    u, v = uv[:, 0], uv[:, 1]
    front = zw > EPS
    with np.errstate(divide="ignore", invalid="ignore"):
        rw = np.sqrt(xw * xw + yw * yw)
        th = np.arctan2(rw, zw)
        t2 = th * th
        t3 = t2 * th
        t5 = t3 * t2
        t7 = t5 * t2
        t9 = t7 * t2
        axis = rw < EPS
        x_r = np.where(axis, 0.0, xw / rw)
        y_r = np.where(axis, 0.0, yw / rw)
        numerical = front & (((np.abs(fx * x_r) < EPS) & (np.abs(x_r) > EPS)) | ((np.abs(fy * y_r) < EPS) & (np.abs(y_r) > EPS)))
        bx = np.where(np.abs(x_r) > EPS, (u - cx) / (fx * x_r) - th, np.where(np.abs(u - cx) < EPS, -th, 0.0))
        by = np.where(np.abs(y_r) > EPS, (v - cy) / (fy * y_r) - th, np.where(np.abs(v - cy) < EPS, -th, 0.0))
    T = np.where(front[:, None], np.stack([t3, t5, t7, t9], 1), 0.0)
    A = _interleave(T, T)
    b = _interleave(np.where(front, bx, 0.0), np.where(front, by, 0.0))
    return A, b, bool(numerical.any())


def radtan_rows(xyz, uv, intr):
    """RadTan: rows fx xn [r^2, r^4, r^6] and fy yn [...], b = u - (fx xn + cx)."""
    fx, fy, cx, cy = intr
    x, y, z = xyz[:, 0], xyz[:, 1], xyz[:, 2]
    xn, yn = x / z, y / z
    r2 = xn * xn + yn * yn
    r4 = r2 * r2
    r6 = r4 * r2
    A = _interleave(np.stack([fx * xn * r2, fx * xn * r4, fx * xn * r6], 1), np.stack([fy * yn * r2, fy * yn * r4, fy * yn * r6], 1))
    b = _interleave(uv[:, 0] - (fx * xn + cx), uv[:, 1] - (fy * yn + cy))
    return A, b


def fov_mean_errors(xyz, uv, intr):
    """Mean reprojection error of every FOV grid candidate (fov.rs:175-228 as the oracle evaluates it, NaN where no
    error is finite).  Sums are numpy's pairwise sums, not the oracle's sequential ones: the means agree to ~1e-15."""
    fx, fy, cx, cy = intr
    x, y, z = xyz[:, 0], xyz[:, 1], xyz[:, 2]
    r2 = x * x + y * y
    r = np.sqrt(r2)
    small = r2 < SQRT_EPS
    out = np.full(len(FOV_W), np.nan)
    with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
        for i, w in enumerate(FOV_W):
            t = math.tan(w / 2.0)
            a = np.arctan2(2.0 * t * r, z)
            rd = np.where(small, 2.0 * t / w, a / (r * w))
            du = (fx * (x * rd) + cx) - uv[:, 0]
            dv = (fy * (y * rd) + cy) - uv[:, 1]
            e = np.sqrt(du * du + dv * dv)
            fin = np.isfinite(e)
            if fin.any():
                out[i] = e[fin].sum() / fin.sum()
    return out


def fov_argmin(means):
    """Index of the candidate the grid search picks: the first strict minimum in ascending w (NaN never wins)."""
    best, best_i = np.inf, None
    for i, m in enumerate(means):
        if m < best:
            best, best_i = m, i
    return best_i


def fov_runner_up_gap(means):
    """(best, relative gap between the best and the second-best candidate)."""
    s = np.sort(means[np.isfinite(means)])
    return s[0], (s[1] - s[0]) / s[0]
