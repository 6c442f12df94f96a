"""NumPy restatement of rsc_orient_normals (include/rsc.h, DESIGN.md section 8), bit for bit: the k-NN graph of the
normals, its minimum spanning forest by (w, lo, hi) through SciPy's Kruskal on the edge ranks, and a breadth-first walk
of each tree from its max-z root, built independently of the device's Borůvka rounds.  The neighbour lists are those
of oracle/normals_oracle.py."""
from __future__ import annotations

import numpy as np


def unit_vertices(xyz, nrm):
    """(vertex mask, float64 unit normals): finite coordinates and a finite normal with (x^2 + y^2) + z^2 > 0"""
    xyz = np.asarray(xyz, np.float32)
    n64 = np.asarray(nrm, np.float32).astype(np.float64)
    with np.errstate(invalid="ignore", over="ignore"):
        len2 = (n64[:, 0] * n64[:, 0] + n64[:, 1] * n64[:, 1]) + n64[:, 2] * n64[:, 2]
        vert = np.isfinite(xyz).all(1) & np.isfinite(n64).all(1) & (len2 > 0)
    u = np.zeros_like(n64)
    u[vert] = n64[vert] / np.sqrt(len2[vert])[:, None]
    return vert, u


def dot(u, a, b):
    return (u[a, 0] * u[b, 0] + u[a, 1] * u[b, 1]) + u[a, 2] * u[b, 2]


def knn_graph(xyz, nrm, nbr):
    """the undirected edges of the orientation graph: (lo, hi) int64 in ascending order, w = 1 - |d| and d, float64"""
    vert, u = unit_vertices(xyz, nrm)
    n, k = nbr.shape
    i = np.repeat(np.arange(n), k)
    j = np.asarray(nbr, np.int64).reshape(-1)
    ok = (j >= 0) & (j != i)
    i, j = i[ok], j[ok]
    ok = vert[i] & vert[j]
    i, j = i[ok], j[ok]
    key = np.unique(np.minimum(i, j) * n + np.maximum(i, j))  # duplicates merged, ascending (lo, hi)
    lo, hi = key // n, key % n
    d = dot(u, lo, hi)
    return lo, hi, 1.0 - np.abs(d), d


def boruvka_rounds(n, lo, hi, rank):
    """the number of Borůvka rounds (every component with a crossing edge takes its minimum one, by rank) until no
    edge crosses components"""
    from scipy.sparse import coo_matrix
    from scipy.sparse.csgraph import connected_components

    comp = np.arange(n)
    rounds = 0
    while True:
        cu, cv = comp[lo], comp[hi]
        cross = cu != cv
        if not cross.any():
            return rounds
        rounds += 1
        best = np.full(n, np.inf)
        np.minimum.at(best, cu[cross], rank[cross])
        np.minimum.at(best, cv[cross], rank[cross])
        chosen = np.isin(rank, best[np.isfinite(best)]) & cross
        g = coo_matrix((np.ones(chosen.sum()), (cu[chosen], cv[chosen])), shape=(n, n))
        _, lab = connected_components(g, directed=False)
        comp = lab[comp]


def orient_mst(xyz, nrm, nbr):
    """rsc_orient_normals' definition (include/rsc.h), independently of the device algorithm: Kruskal
    (scipy.sparse.csgraph.minimum_spanning_tree) on the ranks of the edges in (w, lo, hi) order, then a breadth-first
    walk of each tree from its max-z root.  -> (normals float32 (n, 3), F's edges (E, 2) int64 ascending,
    stats int64 [vertices, edges of F, trees, Borůvka rounds])"""
    from scipy.sparse import coo_matrix
    from scipy.sparse.csgraph import breadth_first_order, connected_components, minimum_spanning_tree

    xyz = np.asarray(xyz, np.float32)
    nrm = np.asarray(nrm, np.float32)
    n = len(xyz)
    vert, u = unit_vertices(xyz, nrm)
    lo, hi, w, _ = knn_graph(xyz, nrm, nbr)
    m = len(lo)
    rank = np.empty(m)
    rank[np.lexsort((hi, lo, w))] = np.arange(1, m + 1)  # distinct and exact: the forest is the unique one
    T = minimum_spanning_tree(coo_matrix((rank, (lo, hi)), shape=(n, n)).tocsr()).tocoo()
    tl, th = np.minimum(T.row, T.col).astype(np.int64), np.maximum(T.row, T.col).astype(np.int64)
    order = np.lexsort((th, tl))
    tl, th = tl[order], th[order]
    _, lab = connected_components(T, directed=False)
    # roots: the largest z of each tree, the lowest index on ties; a virtual node n joins them for one walk
    vidx = np.nonzero(vert)[0]
    by = vidx[np.lexsort((vidx, -xyz[vidx, 2].astype(np.float64)))]
    _, first = np.unique(lab[by], return_index=True)
    roots = by[first]
    G = coo_matrix((np.ones(len(tl) + len(roots)), (np.concatenate([tl, np.full(len(roots), n)]), np.concatenate([th, roots]))),
                   shape=(n + 1, n + 1)).tocsr()
    _, pred = breadth_first_order(G, n, directed=False, return_predecessors=True)
    # flip bit of each tree edge (parent, child): d < 0; parity to the root by pointer doubling up the walk
    par = np.zeros(n + 1, np.int64)
    anc = np.arange(n + 1)
    child = vidx[~np.isin(vidx, roots)]
    anc[child] = pred[child]
    par[child] = (dot(u, pred[child], child) < 0).astype(np.int64)
    anc[roots] = roots
    while (anc[anc] != anc).any():
        par = par ^ par[anc]
        anc = anc[anc]
    uz = u[roots, 2]
    big = u[roots, np.argmax(np.abs(u[roots]), axis=1)]
    neg = np.where(uz != 0, uz < 0, big < 0).astype(np.int64)
    rs = np.zeros(n + 1, np.int64)
    rs[roots] = neg
    flip = np.zeros(n, bool)
    flip[vidx] = (rs[anc[vidx]] ^ par[vidx]).astype(bool)
    out = nrm.copy()
    out[flip] = -out[flip]
    stats = np.array([len(vidx), len(tl), len(vidx) - len(tl), boruvka_rounds(n, lo, hi, rank)], np.int64)
    return out, np.stack([tl, th], 1), stats
