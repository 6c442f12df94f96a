"""NumPy restatement of rsc_estimate_normals (include/rsc.h, DESIGN.md section 8): the neighbour lists bit for bit,
the normals to eigen-solver accuracy.

  - N(i): the k_eff = min(k, finite points) finite points j smallest in (d2(i, j), j) order,
    d2 = ((xj - xi)^2 + (yj - yi)^2) + (zj - zi)^2 in float64 of the float32 values (NumPy rounds every operation
    and never fuses), i itself included.  Brute force in chunks for small clouds; for large ones a cKDTree query
    for k + delta candidates, re-ranked by the exact rule, with delta widened until the last candidate is provably
    farther than the k-th.
  - covariance in float64, mean and sums in list order, divided by k_eff; numpy.linalg.eigh; the normal is the
    eigenvector of the smallest eigenvalue, (0,0,0) when k_eff < 3 or the middle eigenvalue <= TAU * the largest.
  - sign: towards the viewpoint (n . (v - p_i) >= 0), else the component of largest magnitude positive (first axis
    on ties); float32 rounding of the normalised float64 vector last.
"""
from __future__ import annotations

import numpy as np

TAU = 2.0 ** -40


def _d2(q, P):
    """d2 of the query rows q (m, 3) to the points P (..., 3), float64, in the defined grouping"""
    dx = P[..., 0] - q[:, 0:1]
    dy = P[..., 1] - q[:, 1:2]
    dz = P[..., 2] - q[:, 2:3]
    return (dx * dx + dy * dy) + dz * dz


def _rank(d2, cand, keff):
    """the first keff of each row of candidates `cand` (cloud indices) by (d2, index)"""
    order = np.lexsort((cand, d2), axis=-1)[:, :keff]
    return np.take_along_axis(cand, order, 1), np.take_along_axis(d2, order, 1)


def knn_bruteforce(xyz, k, chunk=512):
    """(n, k) int64 neighbour lists, -1 beyond k_eff and for non-finite points"""
    xyz = np.asarray(xyz, np.float32)
    n = len(xyz)
    out = np.full((n, k), -1, np.int64)
    fidx = np.nonzero(np.isfinite(xyz).all(1))[0]
    keff = min(k, len(fidx))
    if keff == 0:
        return out
    X = xyz[fidx].astype(np.float64)
    for s in range(0, len(fidx), chunk):
        q = X[s:s + chunk]
        d2 = _d2(q, X[None, :, :])
        # the keff smallest distances, then the exact order among them; rows with a tie across the cut take a full
        # stable sort (columns are in index order, so a stable sort by d2 is the (d2, index) order)
        part = np.argpartition(d2, keff - 1, axis=1)[:, :keff]
        dk = np.take_along_axis(d2, part, 1)
        cut = dk.max(1)
        tied = (d2 == cut[:, None]).sum(1) != (dk == cut[:, None]).sum(1)
        lists, _ = _rank(dk, fidx[part], keff)
        if tied.any():
            lists[tied] = fidx[np.argsort(d2[tied], axis=1, kind="stable")[:, :keff]]
        out[fidx[s:s + chunk], :keff] = lists
    return out


def knn_kdtree(xyz, k, delta=8, chunk=1 << 20):
    """knn_bruteforce's lists through a cKDTree: k + delta candidates per query, re-ranked exactly; rows whose
    (k + delta)-th candidate is not provably farther than the k-th are queried again with a doubled delta"""
    from scipy.spatial import cKDTree

    xyz = np.asarray(xyz, np.float32)
    n = len(xyz)
    out = np.full((n, k), -1, np.int64)
    fidx = np.nonzero(np.isfinite(xyz).all(1))[0]
    nf = len(fidx)
    keff = min(k, nf)
    if keff == 0:
        return out
    X = xyz[fidx].astype(np.float64)
    tree = cKDTree(X)
    todo = np.arange(nf)
    d = delta
    while len(todo):
        kq = min(keff + d, nf)
        redo = []
        for s in range(0, len(todo), chunk):
            rows = todo[s:s + chunk]
            dist, loc = tree.query(X[rows], kq)
            dist, loc = dist.reshape(len(rows), kq), loc.reshape(len(rows), kq)
            cand = fidx[loc]
            d2 = _d2(X[rows], X[loc])
            lists, dk = _rank(d2, cand, keff)
            out[fidx[rows], :keff] = lists
            if kq < nf:
                # every point the tree did not return has kd-distance >= dist[:, -1]; its exact d2 is within a relative
                # 1e-12 of that squared, so it is strictly beyond the k-th when this holds
                ok = dist[:, -1] * dist[:, -1] * (1.0 - 1e-12) > dk[:, -1]
                redo.append(rows[~ok])
        todo = np.concatenate(redo) if redo else np.arange(0)
        d *= 2
    return out


def knn(xyz, k, brute_max=20_000):
    return knn_bruteforce(xyz, k) if len(xyz) <= brute_max else knn_kdtree(xyz, k)


def pca_normals(xyz, nbr, viewpoint=None):
    """(normals float32 (n, 3), normals float64 before rounding, eigenvalues (n, 3) ascending) from the lists"""
    xyz = np.asarray(xyz, np.float32)
    n, k = nbr.shape
    n64 = np.zeros((n, 3))
    ev = np.zeros((n, 3))
    rows = np.nonzero(np.isfinite(xyz).all(1))[0]
    keff = min(k, len(rows))
    if keff < 3 or len(rows) == 0:
        return n64.astype(np.float32), n64, ev
    P = xyz.astype(np.float64)[nbr[rows, :keff]]  # (m, keff, 3), in list order
    m = np.zeros((len(rows), 3))
    for t in range(keff):
        m = m + P[:, t]
    m = m / keff
    D = P - m[:, None, :]
    C = np.zeros((len(rows), 3, 3))
    for a, b in ((0, 0), (0, 1), (0, 2), (1, 1), (1, 2), (2, 2)):
        s = np.zeros(len(rows))
        for t in range(keff):
            s = s + D[:, t, a] * D[:, t, b]
        C[:, a, b] = C[:, b, a] = s / keff
    w, V = np.linalg.eigh(C)
    v = V[:, :, 0]
    v = v / np.sqrt((v[:, 0] * v[:, 0] + v[:, 1] * v[:, 1]) + v[:, 2] * v[:, 2])[:, None]
    p = xyz[rows].astype(np.float64)
    if viewpoint is not None:
        vp = np.asarray(viewpoint, np.float64)
        s = (v[:, 0] * (vp[0] - p[:, 0]) + v[:, 1] * (vp[1] - p[:, 1])) + v[:, 2] * (vp[2] - p[:, 2])
        flip = s < 0
    else:
        big = np.argmax(np.abs(v), axis=1)  # the first axis on ties
        flip = v[np.arange(len(v)), big] < 0
    v[flip] = -v[flip]
    v[~(w[:, 1] > TAU * w[:, 2])] = 0.0
    n64[rows] = v
    ev[rows] = w
    return n64.astype(np.float32), n64, ev


def estimate_normals(xyz, k=16, viewpoint=None):
    """-> (normals float32 (n, 3), neighbour lists (n, k) int64, float64 normals, eigenvalues)"""
    nbr = knn(xyz, k)
    nrm, n64, ev = pca_normals(xyz, nbr, viewpoint)
    return nrm, nbr, n64, ev
