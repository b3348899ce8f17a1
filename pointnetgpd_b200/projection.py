"""GPD image projection on the CPU: vectorised numpy plus `scipy.spatial.cKDTree`.

Semantics of BaseGraspDataset.project_pc / cal_projection (PointNetGPD/model/dataset.py:78-198), the same numbers as the
CUDA path (`pgpd_gpd_project`, csrc/project.cuh; `prep.project`).  This is the path DataLoader workers run: they are
forked after the training script has initialised CUDA, so they cannot use the GPU.

  normals  up to 30 nearest cloud points within distance 0.1 (the point itself included), searched in the cloud frame and
           ordered by (squared distance, index); one-pass covariance of their grasp-frame coordinates in fp64; the
           eigenvector of its smallest eigenvalue from the closed-form symmetric 3x3 solver (Eberly, "A Robust
           Eigensolver for 3 x 3 Symmetric Matrices").  Fewer than 3 neighbours or a zero covariance give (0, 0, 1).
  voxels   per axis order: index floor(coord / (width / 59) + 30); the first 50 points of a voxel in input order; the
           voxel normal is the fp32 sum of their normals over the count; per pixel the voxel with the largest z index
           wins; occupancy is its count over the image maximum.
"""
import numpy as np
from scipy.spatial import cKDTree

IMG = 60
MAX_NN = 30
RADIUS = 0.1
VOXEL_CAP = 50
MIN_POINTS = 50
ORDERS = ((0, 1, 2), (1, 2, 0), (0, 2, 1))
_TWO_THIRDS_PI = 2.09439510239319549


def _cross(a, b):
    return np.stack([a[:, 1] * b[:, 2] - a[:, 2] * b[:, 1], a[:, 2] * b[:, 0] - a[:, 0] * b[:, 2],
                     a[:, 0] * b[:, 1] - a[:, 1] * b[:, 0]], axis=1)


def _dot(a, b):
    return a[:, 0] * b[:, 0] + a[:, 1] * b[:, 1] + a[:, 2] * b[:, 2]


def _matvec(a, u):
    """a: [n,6] = (a00, a01, a02, a11, a12, a22)"""
    return np.stack([a[:, 0] * u[:, 0] + a[:, 1] * u[:, 1] + a[:, 2] * u[:, 2],
                     a[:, 1] * u[:, 0] + a[:, 3] * u[:, 1] + a[:, 4] * u[:, 2],
                     a[:, 2] * u[:, 0] + a[:, 4] * u[:, 1] + a[:, 5] * u[:, 2]], axis=1)


def _evec_of_simple(a, e):
    r0 = np.stack([a[:, 0] - e, a[:, 1], a[:, 2]], axis=1)
    r1 = np.stack([a[:, 1], a[:, 3] - e, a[:, 4]], axis=1)
    r2 = np.stack([a[:, 2], a[:, 4], a[:, 5] - e], axis=1)
    c = np.stack([_cross(r0, r1), _cross(r0, r2), _cross(r1, r2)], axis=1)         # [n,3 candidates,3]
    d = np.stack([_dot(c[:, 0], c[:, 0]), _dot(c[:, 1], c[:, 1]), _dot(c[:, 2], c[:, 2])], axis=1)
    imax = np.where(d[:, 1] > d[:, 0], 1, 0)                                        # ties go to the earlier candidate
    imax = np.where(d[:, 2] > d[np.arange(len(d)), imax], 2, imax)
    rows = np.arange(len(d))
    return c[rows, imax] / np.sqrt(d[rows, imax])[:, None]


def _evec_orthogonal(a, w, e):
    big_x = np.abs(w[:, 0]) > np.abs(w[:, 1])
    inv_x = 1.0 / np.sqrt(w[:, 0] * w[:, 0] + w[:, 2] * w[:, 2])
    inv_y = 1.0 / np.sqrt(w[:, 1] * w[:, 1] + w[:, 2] * w[:, 2])
    zero = np.zeros(len(w))
    u = np.where(big_x[:, None], np.stack([-w[:, 2] * inv_x, zero, w[:, 0] * inv_x], axis=1),
                 np.stack([zero, w[:, 2] * inv_y, -w[:, 1] * inv_y], axis=1))
    v = _cross(w, u)
    au, av = _matvec(a, u), _matvec(a, v)
    m00, m01, m11 = _dot(u, au) - e, _dot(u, av), _dot(v, av) - e
    f00, f01, f11 = np.abs(m00), np.abs(m01), np.abs(m11)
    # |m00| >= |m11|: normalise the row (m00, m01); otherwise the row (m01, m11)
    r0 = f00 >= f11
    p, q = np.where(r0, m00, m11), m01                 # the row's diagonal entry and off-diagonal entry
    fp, fq = np.abs(p), f01
    ratio_p = q / p                                    # |p| >= |q|
    cp = 1.0 / np.sqrt(1.0 + ratio_p * ratio_p)
    ratio_q = p / q                                    # |q| > |p|
    cq = 1.0 / np.sqrt(1.0 + ratio_q * ratio_q)
    by_p = fp >= fq
    # r0:  (m00, m01) -> return m01*u - m00*v;   else (m11, m01) -> return m11*u - m01*v
    p_n = np.where(by_p, cp, ratio_q * cq)             # normalised diagonal entry
    q_n = np.where(by_p, ratio_p * cp, cq)             # normalised off-diagonal entry
    cu = np.where(r0, q_n, p_n)
    cv = np.where(r0, p_n, q_n)
    out = cu[:, None] * u - cv[:, None] * v
    flat = np.maximum(fp, fq) <= 0.0
    return np.where(flat[:, None], u, out)


def smallest_eigenvectors(cov):
    """cov: [n,6] symmetric 3x3 matrices (c00, c01, c02, c11, c12, c22) -> [n,3] unit eigenvectors of the smallest
    eigenvalue; the zero vector where the largest entry is 0."""
    cov = np.asarray(cov, dtype=np.float64)
    n = len(cov)
    out = np.zeros((n, 3))
    mx = cov.max(axis=1)
    with np.errstate(all="ignore"):
        a = cov / mx[:, None]
        off = a[:, 1] * a[:, 1] + a[:, 2] * a[:, 2] + a[:, 4] * a[:, 4]
        q = (a[:, 0] + a[:, 3] + a[:, 5]) / 3.0
        b00, b11, b22 = a[:, 0] - q, a[:, 3] - q, a[:, 5] - q
        p = np.sqrt((b00 * b00 + b11 * b11 + b22 * b22 + off * 2.0) / 6.0)
        c00 = b11 * b22 - a[:, 4] * a[:, 4]
        c01 = a[:, 1] * b22 - a[:, 4] * a[:, 2]
        c02 = a[:, 1] * a[:, 4] - b11 * a[:, 2]
        det = (b00 * c00 - a[:, 1] * c01 + a[:, 2] * c02) / (p * p * p)
        hd = np.minimum(np.maximum(det * 0.5, -1.0), 1.0)
        ang = np.arccos(hd) / 3.0
        beta2 = np.cos(ang) * 2.0
        beta0 = np.cos(ang + _TWO_THIRDS_PI) * 2.0
        beta1 = -(beta0 + beta2)
        e0, e1, e2 = q + p * beta0, q + p * beta1, q + p * beta2
        pos = hd >= 0.0
        first_e = np.where(pos, e2, e0)                # the eigenvalue that is simple by construction
        w_first = _evec_of_simple(a, first_e)
        w1 = _evec_orthogonal(a, w_first, e1)
        third = np.where(pos[:, None], _cross(w1, w_first), _cross(w_first, w1))
        first_smallest = np.where(pos, (e2 < e0) & (e2 < e1), (e0 < e1) & (e0 < e2))
        mid_smallest = (e1 < e0) & (e1 < e2)
        gen = np.where(first_smallest[:, None], w_first, np.where(mid_smallest[:, None], w1, third))
    diag = np.where(((cov[:, 0] < cov[:, 3]) & (cov[:, 0] < cov[:, 5]))[:, None], [1.0, 0.0, 0.0],
                    np.where(((cov[:, 3] < cov[:, 0]) & (cov[:, 3] < cov[:, 5]))[:, None], [0.0, 1.0, 0.0], [0.0, 0.0, 1.0]))
    sel = mx != 0.0
    out[sel] = np.where((off > 0.0)[sel, None], gen[sel], diag[sel])
    return out


def estimate_normals(pc, pc_t, query, tree=None):
    """Normals of the points `query` (indices into the cloud): neighbours searched in the cloud frame `pc` [P,3],
    covariance from the grasp-frame coordinates `pc_t` [P,3] (fp64).  Returns [len(query),3] float64."""
    pc = np.asarray(pc, dtype=np.float64)
    query = np.asarray(query, dtype=np.int64)
    P = len(pc)
    out = np.tile([0.0, 0.0, 1.0], (len(query), 1))
    if len(query) == 0:
        return out
    tree = cKDTree(pc) if tree is None else tree
    k = min(MAX_NN, P)
    _, jj = tree.query(pc[query], k=k, distance_upper_bound=RADIUS * (1 + 1e-9))
    jj = jj.reshape(len(query), k)
    ok = jj < P
    js = np.where(ok, jj, 0)
    e = pc[js] - pc[query][:, None, :]
    d2 = e[..., 0] * e[..., 0] + e[..., 1] * e[..., 1] + e[..., 2] * e[..., 2]
    ok &= d2 <= RADIUS * RADIUS
    d2 = np.where(ok, d2, np.inf)
    order = np.lexsort((np.where(ok, js, P), d2), axis=-1)             # (squared distance, index)
    js = np.take_along_axis(js, order, axis=1)
    ok = np.take_along_axis(ok, order, axis=1)
    cnt = ok.sum(axis=1)
    t = np.asarray(pc_t, dtype=np.float64)[js]                          # [Q,k,3]
    s = np.zeros((len(query), 9))
    for n in range(k):                                                  # one neighbour at a time: a fixed summation order
        x, y, z = (np.where(ok[:, n], t[:, n, d], 0.0) for d in range(3))
        s += np.stack([x, y, z, x * x, x * y, x * z, y * y, y * z, z * z], axis=1)
    many = cnt >= 3
    s = s[many] / cnt[many, None]
    cov = np.stack([s[:, 3] - s[:, 0] * s[:, 0], s[:, 4] - s[:, 0] * s[:, 1], s[:, 5] - s[:, 0] * s[:, 2],
                    s[:, 6] - s[:, 1] * s[:, 1], s[:, 7] - s[:, 1] * s[:, 2], s[:, 8] - s[:, 2] * s[:, 2]], axis=1)
    v = smallest_eigenvectors(cov)
    zero = (v == 0.0).all(axis=1)
    v[zero] = [0.0, 0.0, 1.0]
    out[many] = v
    return out


def _image(pts, nrm32, width, order):
    """(occupancy [60,60], normals [60,60,3]) indexed [x][y], float64 (cal_projection)."""
    occ = np.zeros((IMG, IMG))
    nimg = np.zeros((IMG, IMG, 3))
    c = pts[:, list(order)]
    if len(c) == 0 or max(c[:, 0].max() - c[:, 0].min(), c[:, 1].max() - c[:, 1].min()) == 0:
        return occ, nimg
    res = width / (IMG - 1)
    v = np.clip(np.floor(c / res + IMG / 2), 0, IMG - 1).astype(np.int64)
    key = (v[:, 0] * IMG + v[:, 1]) * 64 + v[:, 2]
    srt = np.argsort(key, kind="stable")                                 # (voxel, input position)
    ks = key[srt]
    start = np.r_[True, ks[1:] != ks[:-1]]
    vid = np.cumsum(start) - 1
    first = np.flatnonzero(start)
    rank = np.arange(len(ks)) - first[vid]
    keep = rank < VOXEL_CAP
    ukey = ks[first]
    count = np.bincount(vid[keep], minlength=len(ukey))
    sums = np.zeros((len(ukey), 3), np.float32)
    np.add.at(sums, vid[keep], nrm32[srt][keep])                        # in order: a sequential fp32 sum per voxel
    mean = sums / count[:, None]
    pix = ukey >> 6
    win = np.r_[pix[1:] != pix[:-1], True]                               # the largest z of each pixel
    px, py = pix[win] // IMG, pix[win] % IMG
    occ[px, py] = count[win]
    nimg[px, py] = mean[win]
    return occ / occ.max(), nimg


def project_points(pts, nrm, width, chann):
    """pts: [n,3] grasp-frame points of a box (fp64, ascending cloud index); nrm: their normals.  Rows whose normal has
    a NaN are dropped first.  Returns the image [chann,60,60] float64 in the model's layout (out[c][y][x])."""
    pts = np.asarray(pts, dtype=np.float64)
    nrm = np.asarray(nrm, dtype=np.float64)
    good = ~np.isnan(nrm).any(axis=1)
    pts, nrm32 = pts[good], nrm[good].astype(np.float32)
    planes = []
    for o, order in enumerate(ORDERS[:1] if chann == 3 else ORDERS):
        occ, nimg = _image(pts, nrm32, width, order)
        if chann == 12:
            planes.append(occ[..., None])
        planes.append(nimg)
    return np.concatenate(planes, axis=2).transpose(2, 1, 0)


def project_grasp(pc, center, rows, width, chann, tree=None):
    """Crop + normals + images for one grasp (frame: center [3], rows [3,3]) of the cloud pc [P,3].
    Returns (in_ind, image [chann,60,60] float64 or None when fewer than 50 points are in the box)."""
    pc = np.asarray(pc)
    pc_t = (pc - center) @ np.asarray(rows).T
    half = np.array([width / 4, width / 2, width / 4])
    in_ind = np.nonzero(np.all((pc_t > -half) & (pc_t < half), axis=1))[0]
    if len(in_ind) < MIN_POINTS:
        return in_ind, None
    nrm = estimate_normals(pc, pc_t, in_ind, tree)
    return in_ind, project_points(pc_t[in_ind], nrm, width, chann)
