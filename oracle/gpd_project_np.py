"""Plain normal estimator for the GPD image projection (PointNetGPD/model/dataset.py:78-86, `get_normal`).

TEST INFRASTRUCTURE ONLY (see oracle/__init__.py).

The reference estimates normals with Open3D (`estimate_normals` with KDTreeSearchParamHybrid(radius=0.1, max_nn=30)),
which is not available here.  This is a plain restatement written independently of the product code
(pointnetgpd_b200/projection.py, csrc/project.cuh):

  * neighbours by brute force: every point at squared distance <= 0.1^2 (the point itself included), the 30 smallest
    by (squared distance, index);
  * one-pass covariance of the neighbours (sums of x, y, z and their products in neighbour order, divided by the count);
  * the eigenvector of the smallest eigenvalue from the closed-form symmetric 3x3 solver of D. Eberly, "A Robust
    Eigensolver for 3 x 3 Symmetric Matrices" (Geometric Tools), one matrix at a time in Python floats;
  * fewer than 3 neighbours, or a solver result of zero length (zero covariance), give (0, 0, 1).

make_golden_gpd_project.py hands `get_normal` to the reference's own collect_pc / project_pc / cal_projection as the
method of a stub `self`.
"""
import math

import numpy as np

RADIUS = 0.1
MAX_NN = 30


def _cross(a, b):
    return [a[1] * b[2] - a[2] * b[1], a[2] * b[0] - a[0] * b[2], a[0] * b[1] - a[1] * b[0]]


def _dot(a, b):
    return a[0] * b[0] + a[1] * b[1] + a[2] * b[2]


def _mat_vec(m, u):
    return [m[0][0] * u[0] + m[0][1] * u[1] + m[0][2] * u[2],
            m[1][0] * u[0] + m[1][1] * u[1] + m[1][2] * u[2],
            m[2][0] * u[0] + m[2][1] * u[1] + m[2][2] * u[2]]


def _simple_eigenvector(m, value):
    """Unit eigenvector of the simple eigenvalue `value`: the longest cross product of two rows of m - value*I."""
    rows = [[m[r][c] - (value if r == c else 0.0) for c in range(3)] for r in range(3)]
    best, best_len2 = None, None
    for i, j in ((0, 1), (0, 2), (1, 2)):
        c = _cross(rows[i], rows[j])
        l2 = _dot(c, c)
        if best is None or l2 > best_len2:
            best, best_len2 = c, l2
    s = math.sqrt(best_len2)
    return [best[0] / s, best[1] / s, best[2] / s]


def _second_eigenvector(m, w, value):
    """Eigenvector of `value` in the plane orthogonal to the unit eigenvector w."""
    if abs(w[0]) > abs(w[1]):
        inv = 1.0 / math.sqrt(w[0] * w[0] + w[2] * w[2])
        u = [-w[2] * inv, 0.0, w[0] * inv]
    else:
        inv = 1.0 / math.sqrt(w[1] * w[1] + w[2] * w[2])
        u = [0.0, w[2] * inv, -w[1] * inv]
    v = _cross(w, u)
    mu, mv = _mat_vec(m, u), _mat_vec(m, v)
    a, b, c = _dot(u, mu) - value, _dot(u, mv), _dot(v, mv) - value      # the 2x2 matrix (a b; b c) in the (u, v) basis
    if abs(a) >= abs(c):
        diag, off = a, b
    else:
        diag, off = c, b
    if max(abs(diag), abs(off)) <= 0.0:
        return u
    if abs(diag) >= abs(off):
        t = off / diag
        diag_n = 1.0 / math.sqrt(1.0 + t * t)
        off_n = t * diag_n
    else:
        t = diag / off
        off_n = 1.0 / math.sqrt(1.0 + t * t)
        diag_n = t * off_n
    if abs(a) >= abs(c):                   # row (a, b): null vector (b, -a)
        cu, cv = off_n, diag_n
    else:                                  # row (b, c): null vector (c, -b)
        cu, cv = diag_n, off_n
    return [cu * u[k] - cv * v[k] for k in range(3)]


def smallest_eigenvector(cov):
    """cov: 3x3 nested lists (symmetric).  Unit eigenvector of the smallest eigenvalue, or [0,0,0] when max entry == 0."""
    mx = max(max(row) for row in cov)
    if mx == 0.0:
        return [0.0, 0.0, 0.0]
    m = [[cov[r][c] / mx for c in range(3)] for r in range(3)]
    off = m[0][1] * m[0][1] + m[0][2] * m[0][2] + m[1][2] * m[1][2]
    if off > 0.0:
        q = (m[0][0] + m[1][1] + m[2][2]) / 3.0
        b00, b11, b22 = m[0][0] - q, m[1][1] - q, m[2][2] - q
        p = math.sqrt((b00 * b00 + b11 * b11 + b22 * b22 + off * 2.0) / 6.0)
        c00 = b11 * b22 - m[1][2] * m[1][2]
        c01 = m[0][1] * b22 - m[1][2] * m[0][2]
        c02 = m[0][1] * m[1][2] - b11 * m[0][2]
        half_det = min(max((b00 * c00 - m[0][1] * c01 + m[0][2] * c02) / (p * p * p) * 0.5, -1.0), 1.0)
        angle = math.acos(half_det) / 3.0
        beta2 = math.cos(angle) * 2.0
        beta0 = math.cos(angle + 2.09439510239319549) * 2.0
        beta1 = -(beta0 + beta2)
        ev = [q + p * beta0, q + p * beta1, q + p * beta2]
        first = 2 if half_det >= 0.0 else 0          # the eigenvalue that is simple by construction
        other = 2 - first
        w_first = _simple_eigenvector(m, ev[first])
        if ev[first] < ev[other] and ev[first] < ev[1]:
            return w_first
        w1 = _second_eigenvector(m, w_first, ev[1])
        if ev[1] < ev[0] and ev[1] < ev[2]:
            return w1
        return _cross(w1, w_first) if first == 2 else _cross(w_first, w1)
    d = [cov[0][0], cov[1][1], cov[2][2]]
    if d[0] < d[1] and d[0] < d[2]:
        return [1.0, 0.0, 0.0]
    if d[1] < d[0] and d[1] < d[2]:
        return [0.0, 1.0, 0.0]
    return [0.0, 0.0, 1.0]


def neighbours(points, i):
    """Indices of the neighbours of point i, ascending (squared distance, index)."""
    e = points - points[i]
    d2 = e[:, 0] * e[:, 0] + e[:, 1] * e[:, 1] + e[:, 2] * e[:, 2]
    cand = np.flatnonzero(d2 <= RADIUS * RADIUS)
    cand = cand[np.lexsort((cand, d2[cand]))]
    return cand[:MAX_NN]


def normal_of(points, nb):
    if len(nb) < 3:
        return [0.0, 0.0, 1.0]
    s = [0.0] * 9
    for j in nb:
        x, y, z = (float(v) for v in points[j])
        for k, v in enumerate((x, y, z, x * x, x * y, x * z, y * y, y * z, z * z)):
            s[k] += v
    s = [v / len(nb) for v in s]
    cxy, cxz, cyz = s[4] - s[0] * s[1], s[5] - s[0] * s[2], s[7] - s[1] * s[2]
    cov = [[s[3] - s[0] * s[0], cxy, cxz], [cxy, s[6] - s[1] * s[1], cyz], [cxz, cyz, s[8] - s[2] * s[2]]]
    n = smallest_eigenvector(cov)
    return [0.0, 0.0, 1.0] if n == [0.0, 0.0, 0.0] else n


def get_normal(points, radius=RADIUS, max_nn=MAX_NN, only=None):
    """Normals [P,3] float64 of every point of `points` ([P,3], the frame the covariance is taken in).  `only`: compute
    just these rows (the others are left NaN)."""
    assert radius == RADIUS and max_nn == MAX_NN
    points = np.asarray(points, dtype=np.float64)
    out = np.full((len(points), 3), np.nan)
    for i in (range(len(points)) if only is None else only):
        out[i] = normal_of(points, neighbours(points, i))
    return out
