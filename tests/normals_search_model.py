"""Host restatement of the level choices of the device k-NN search (rsc_normals.cu): the start level of every query
(the deepest whose cell holds >= k_eff points), the 27-cell blocks it scans, the r_safe acceptance test in the same
float64 operations, and so the exact number of (query, candidate) distances the device reports as `pairs`.  The
neighbour lists do not depend on these choices (they are compared with oracle/normals_oracle.py); this model shows
which queries escalate and which scan the whole box."""
import numpy as np


def search_model(xyz, k):
    """-> (pairs, start level and accepting level of every finite point, in index order)"""
    xyz = np.asarray(xyz, np.float32)
    fin = np.isfinite(xyz).all(1)
    fidx = np.nonzero(fin)[0]
    X = xyz[fidx].astype(np.float64)
    nf = len(fidx)
    keff = min(k, nf)
    D = 21
    lo = X.min(0) if nf else np.zeros(3)
    w = (X.max(0) - lo) if nf else np.ones(3)
    w = np.where(w > 0, w, 1.0)
    c = np.clip(np.floor((X - lo) / w * 2.0 ** D), 0, 2 ** D - 1).astype(np.int64)
    cells = []  # per level: sorted keys, order, counts lookup
    for l in range(1, D + 2):
        cc = c >> (D - (l - 1))
        key = (cc[:, 0] << 42) | (cc[:, 1] << 21) | cc[:, 2]
        order = np.argsort(key, kind="stable")
        cells.append((key[order], order, cc))
    pairs = 0
    start_lv, acc_lv = np.zeros(nf, int), np.zeros(nf, int)
    for q in range(nf):
        lv = 1
        for l in range(D + 1, 0, -1):
            sk, _, cc = cells[l - 1]
            kq = (cc[q, 0] << 42) | (cc[q, 1] << 21) | cc[q, 2]
            if np.searchsorted(sk, kq, "right") - np.searchsorted(sk, kq, "left") >= keff:
                lv = l
                break
        start_lv[q] = lv
        while True:
            sk, order, cc = cells[lv - 1]
            ncell = 1 << (lv - 1)
            members = []
            for dx in (-1, 0, 1):
                for dy in (-1, 0, 1):
                    for dz in (-1, 0, 1):
                        v = cc[q] + (dx, dy, dz)
                        if (v < 0).any() or (v >= ncell).any():
                            continue
                        kq = (v[0] << 42) | (v[1] << 21) | v[2]
                        members.append(order[np.searchsorted(sk, kq, "left"):np.searchsorted(sk, kq, "right")])
            m = np.concatenate(members)
            pairs += len(m)
            dd = X[m] - X[q]
            d2 = (dd[:, 0] * dd[:, 0] + dd[:, 1] * dd[:, 1]) + dd[:, 2] * dd[:, 2]
            kd = np.sort(d2)[keff - 1]
            r = np.inf
            for a in range(3):
                qa = int(cc[q, a])
                h = w[a] / ncell
                e = 2.0 ** -48 * (abs(lo[a]) + w[a] + abs(X[q, a]))
                if qa >= 2:
                    r = min(r, (X[q, a] - (lo[a] + float(qa - 1) * h)) - e)
                if qa + 2 < ncell:
                    r = min(r, ((lo[a] + float(qa + 2) * h) - X[q, a]) - e)
            if r == np.inf or (r > 0 and kd < (r * r) * (1.0 - 2.0 ** -40)):
                break
            lv -= 1
        acc_lv[q] = lv
    return pairs, start_lv, acc_lv
