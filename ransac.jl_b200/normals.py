"""Oriented PCA normals of the k nearest neighbours, computed on the device (rsc_estimate_normals).

Raw scans (LiDAR, photogrammetry, depth cameras) come as coordinates only, but every cloud of this library needs
an oriented unit normal per point.  For a single scan, pass the sensor position as `viewpoint`:

    RANSACCloud(V, estimate_normals(V, viewpoint=s), 2)

Without one sensor position (CAD or mesh samples, merged scans, photogrammetry, normals of arbitrary sign),
`orient_normals` makes the signs consistent by propagation over the k-NN graph (rsc_orient_normals):

    RANSACCloud(V, orient_normals(V), 2)

The definition (neighbours, covariance, degenerate cases, sign rules) is in include/rsc.h and DESIGN.md section 8;
oracle/normals_oracle.py and oracle/orient_oracle.py restate them in NumPy.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional

import numpy as np

from ._lib import Context, lib


def estimate_normals(vertices, k: int = 16, viewpoint=None, device: int = 0, ctx: Optional[Context] = None,
                     return_neighbours: bool = False):
    """Unit normals (N, 3) float32 of the points `vertices` (N, 3), from the k (3..32) nearest neighbours of each.

    float64 input is rounded to float32 first, as `rsc_cloud_create_f64` does, so the result is the one of the
    float32 cloud the device stores.  `viewpoint` (3 values) orients every normal towards it; without one the
    component of largest magnitude is made positive, a coin flip from point to point on a curved surface: for a cloud
    without one viewpoint, use `orient_normals`.  Points with a non-finite coordinate, and points whose
    neighbourhood is collinear or a single point, get (0, 0, 0).  With `return_neighbours=True` the result is
    `(normals, neighbours)`, neighbours (N, k) int64: row i lists the neighbours of point i by (distance, index),
    itself included, -1 beyond the number of finite points.
    """
    v = np.ascontiguousarray(np.asarray(vertices), dtype=np.float32)
    if v.ndim != 2 or v.shape[1] != 3:
        raise ValueError("estimate_normals: vertices must have shape (N, 3)")
    n = int(v.shape[0])
    ctx = ctx if ctx is not None else Context.get(device)
    vp = None
    if viewpoint is not None:
        vp = np.ascontiguousarray(np.asarray(viewpoint, dtype=np.float64).reshape(3))
    nrm = np.empty((n, 3), np.float32)
    nbr = np.empty((n, k), np.int64) if return_neighbours and n > 0 and 3 <= k <= 32 else None
    ctx.check(lib.rsc_estimate_normals(ctx.h, v.ctypes.data, n, int(k), None if vp is None else vp.ctypes.data,
                                       nrm.ctypes.data, None if nbr is None else nbr.ctypes.data, None))
    return (nrm, nbr) if return_neighbours else nrm


def orient_normals(vertices, normals=None, k: int = 16, device: int = 0, ctx: Optional[Context] = None,
                   return_tree: bool = False):
    """Normals (N, 3) float32 with consistent signs, for clouds without one viewpoint (rsc_orient_normals).

    `normals` (N, 3) are oriented as given; with `normals=None` they are first estimated as
    `estimate_normals(vertices, k)` does, from the same neighbour search.  The signs follow the minimum spanning forest
    of the k-nearest-neighbour graph weighted by 1 - |n_i . n_j|: each tree's root (its point of largest z) gets a
    positive z component, and a child keeps its parent's sign when their normals make an angle of at most 90 degrees.
    Each output row is its input row, negated or not.  Points with a non-finite coordinate or a zero or non-finite
    normal are returned unchanged and join no tree.  float64 input is rounded to float32 first.  With
    `return_tree=True` the result is `(normals, edges, stats)`: edges (E, 2) int64, the forest's (lo, hi) pairs in
    ascending order, and stats {"vertices", "edges", "trees", "rounds"}.
    """
    v = np.ascontiguousarray(np.asarray(vertices), dtype=np.float32)
    if v.ndim != 2 or v.shape[1] != 3:
        raise ValueError("orient_normals: vertices must have shape (N, 3)")
    n = int(v.shape[0])
    nin = None
    if normals is not None:
        nin = np.ascontiguousarray(np.asarray(normals), dtype=np.float32)
        if nin.shape != v.shape:
            raise ValueError("orient_normals: normals must have the shape of vertices")
    ctx = ctx if ctx is not None else Context.get(device)
    out = np.empty((n, 3), np.float32)
    edges = np.empty((max(n, 1), 2), np.int64) if return_tree else None
    stats = np.zeros(4, np.int64)
    ctx.check(lib.rsc_orient_normals(ctx.h, v.ctypes.data, n, int(k), None if nin is None else nin.ctypes.data,
                                     out.ctypes.data, None if edges is None else edges.ctypes.data, stats.ctypes.data))
    if not return_tree:
        return out
    names = ("vertices", "edges", "trees", "rounds")
    return out, edges[:stats[1]].copy(), {a: int(b) for a, b in zip(names, stats)}
