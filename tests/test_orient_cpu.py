"""Normal orientation without a GPU: the NumPy oracle of rsc_orient_normals (oracle/orient_oracle.py orient_mst)
against a plain-Python Kruskal, on the scenes it is meant for (random signs, estimated normals without a viewpoint)
through the C oracle's ransac(), and the build of rsc_orient.cu."""
import os
import shutil
import subprocess

import numpy as np
import pytest

from oracle import normals_oracle as NO
from oracle import orient_oracle as OO
from tests.test_normals_cpu import E2E_MIN_FOUND, ROOT, lattice

K = 16


def mixed_scene():
    """curved primitives, little noise, no outliers: where signs decide what ransac() recovers"""
    from ransac_jl_b200 import scenes

    return scenes.scene_mixed(21, 40_000, noise_frac=0.002, jitter_deg=0.0, outlier_frac=0.0, counts=(3, 3, 3, 2))


def random_signs(nrm, seed=3):
    s = np.random.default_rng(seed).choice(np.float32([-1, 1]), len(nrm))
    return (nrm * s[:, None]).astype(np.float32)


def consistency(scene, nrm):
    """per primitive, the share of its points whose normal agrees with the primitive's majority sign relative to the
    ground truth"""
    agree = np.einsum("ij,ij->i", nrm.astype(np.float64), scene.normals.astype(np.float64)) > 0
    out = []
    for p in range(len(scene.primitives)):
        a = agree[scene.labels == p]
        out.append(max(a.mean(), 1 - a.mean()))
    return np.array(out)


def kruskal(n, lo, hi, w):
    """the minimum spanning forest by (w, lo, hi), with a plain union-find"""
    parent = list(range(n))

    def find(x):
        while parent[x] != x:
            parent[x] = parent[parent[x]]
            x = parent[x]
        return x

    out = []
    for e in sorted(range(len(lo)), key=lambda e: (w[e], lo[e], hi[e])):
        a, b = find(int(lo[e])), find(int(hi[e]))
        if a != b:
            parent[max(a, b)] = min(a, b)
            out.append((int(lo[e]), int(hi[e])))
    return sorted(out)


def small_graphs():
    rng = np.random.default_rng(11)
    out = {}
    for t in range(4):
        xyz = rng.normal(size=(300, 3)).astype(np.float32)
        out[f"random{t}"] = (xyz, rng.normal(size=(300, 3)).astype(np.float32))
    # two far-apart blobs: two components
    xyz = np.concatenate([rng.normal(size=(150, 3)), rng.normal(size=(150, 3)) + 1e4]).astype(np.float32)
    out["two_blobs"] = (xyz, rng.normal(size=(300, 3)).astype(np.float32))
    # identical normals on a lattice: every weight ties, only (lo, hi) decides
    lat = lattice(6)
    out["ties"] = (lat, np.tile(np.float32([0.0, 0.6, 0.8]), (len(lat), 1)))
    # opposite signs on the same lattice: |d| still ties everywhere
    out["ties_signed"] = (lat, random_signs(out["ties"][1], 4))
    return out


@pytest.mark.parametrize("name", ["random0", "random1", "random2", "random3", "two_blobs", "ties", "ties_signed"])
@pytest.mark.parametrize("k", [4, K])
def test_forest_equals_kruskal(name, k):
    xyz, nrm = small_graphs()[name]
    nbr = NO.knn_bruteforce(xyz, k)
    lo, hi, w, _ = OO.knn_graph(xyz, nrm, nbr)
    _, edges, stats = OO.orient_mst(xyz, nrm, nbr)
    assert [tuple(e) for e in edges.tolist()] == kruskal(len(xyz), lo, hi, w)
    assert stats[1] == len(edges) and stats[0] - stats[1] == stats[2]
    assert 1 <= stats[3] <= int(np.ceil(np.log2(stats[0])))


@pytest.mark.parametrize("name", ["random0", "two_blobs", "ties"])
def test_forest_spans_each_component(name):
    from scipy.sparse import coo_matrix
    from scipy.sparse.csgraph import connected_components

    xyz, nrm = small_graphs()[name]
    nbr = NO.knn_bruteforce(xyz, 8)
    lo, hi, _, _ = OO.knn_graph(xyz, nrm, nbr)
    _, edges, stats = OO.orient_mst(xyz, nrm, nbr)
    n = len(xyz)
    nc_graph, lab_graph = connected_components(coo_matrix((np.ones(len(lo)), (lo, hi)), shape=(n, n)), directed=False)
    nc_tree, lab_tree = connected_components(coo_matrix((np.ones(len(edges)), (edges[:, 0], edges[:, 1])), shape=(n, n)),
                                             directed=False)
    assert nc_graph == nc_tree == stats[2]
    # the same partition
    assert len(set(zip(lab_graph, lab_tree))) == nc_graph
    if name == "two_blobs":
        assert stats[2] == 2


def test_unusable_points_are_copied_and_signs_follow_the_tree():
    xyz, nrm = small_graphs()["random0"]
    nrm = nrm.copy()
    xyz = xyz.copy()
    nrm[3] = 0
    nrm[5] = np.nan
    nrm[7, 1] = np.inf
    xyz[9, 2] = np.nan
    nbr = NO.knn_bruteforce(xyz, 8)
    out, edges, stats = OO.orient_mst(xyz, nrm, nbr)
    assert out[[3, 5, 7, 9]].tobytes() == nrm[[3, 5, 7, 9]].tobytes()
    assert stats[0] == len(xyz) - 4 and not np.isin([3, 5, 7, 9], edges).any()
    # each output row is its input row, with the sign bit flipped or not
    assert ((out.view(np.uint32) ^ nrm.view(np.uint32)) & 0x7FFFFFFF == 0).all()
    # along every tree edge the oriented normals agree (d >= 0)
    _, u = OO.unit_vertices(xyz, out)
    assert (OO.dot(u, edges[:, 0], edges[:, 1]) >= 0).all()
    # the root of the (single) tree has a positive z component
    v = np.nonzero(np.isfinite(xyz).all(1) & (np.abs(nrm).sum(1) > 0) & np.isfinite(nrm).all(1))[0]
    assert stats[2] == 1
    r = v[np.argmax(xyz[v, 2])]
    assert out[r, 2] > 0


def test_random_signs_become_consistent():
    sc = mixed_scene()
    nbr = NO.knn(sc.vertices, K)
    flipped = random_signs(sc.normals)
    assert consistency(sc, flipped).min() < 0.55
    out, _, stats = OO.orient_mst(sc.vertices, flipped, nbr)
    assert (consistency(sc, out) == 1.0).all()
    assert stats[3] <= int(np.ceil(np.log2(stats[0])))


def _c_ransac(sc, nrm, scan):
    import ransac_jl_b200 as R
    from oracle import c_oracle
    from ransac_jl_b200 import scenes
    from tests.helpers import oracle_params

    if not c_oracle.available():
        pytest.skip("oracle/liboracle.so not built")
    op = oracle_params(R.ransacparameters(iteration=scan.iteration))
    subs = R.makesubsets(len(sc.vertices), scan.subsets, np.random.default_rng(1234))
    got, _, _ = c_oracle.ransac(sc.vertices, nrm, subs[0], op, scan.seed)
    return scenes.recovered(sc, [(g[0], g[3]) for g in got])


# primitives the C oracle's loop recovers on mixed_scene() with the ground-truth normals (scan_scenario()'s settings);
# random signs then MST orientation recover as many, and the device loop must too
MIXED_FOUND = 7


def test_oriented_random_signs_recover_like_the_ground_truth():
    from ransac_jl_b200 import scenes

    scan = scenes.scan_scenario()
    sc = mixed_scene()
    flipped = random_signs(sc.normals)
    out, _, _ = OO.orient_mst(sc.vertices, flipped, NO.knn(sc.vertices, K))
    truth = _c_ransac(sc, sc.normals, scan)
    assert len(truth) == MIXED_FOUND
    assert len(_c_ransac(sc, out, scan)) >= len(truth)


def test_estimated_and_oriented_normals_recover_the_scan_without_a_viewpoint():
    from ransac_jl_b200 import scenes

    scan = scenes.scan_scenario()
    sc = scan.scene
    est, nbr, _, _ = NO.estimate_normals(sc.vertices, K)
    out, _, _ = OO.orient_mst(sc.vertices, est, nbr)
    assert consistency(sc, out).min() > 0.99
    assert len(_c_ransac(sc, out, scan)) >= E2E_MIN_FOUND


def test_null_context_is_refused_without_a_device():
    import ransac_jl_b200 as R

    xyz = np.zeros((4, 3), np.float32)
    nrm = np.zeros((4, 3), np.float32)
    assert R._lib.lib.rsc_orient_normals(None, xyz.ctypes.data, 4, 8, None, nrm.ctypes.data, None, None) == R._lib.RSC_E_ARG
    assert "rsc_orient_normals" in R._lib.SIGNATURES
    assert R.orient_normals is R.normals.orient_normals


@pytest.mark.skipif(shutil.which("nvcc") is None and not os.path.exists("/usr/local/cuda/bin/nvcc"), reason="nvcc not found")
def test_kernels_compile_for_sm100a_without_spills(tmp_path):
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    csrc = os.path.join(ROOT, "ransac.jl_b200", "csrc")
    r = subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-fmad=false",
                        "-I" + os.path.join(ROOT, "include"), "-I" + csrc, "-Xptxas", "-v", "-c",
                        os.path.join(csrc, "rsc_orient.cu"), "-o", str(tmp_path / "o.o")], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    log = r.stderr
    for kernel in ("hook_kernel", "min_w_kernel", "min_key_kernel", "jump_kernel", "cross_scatter_kernel", "sign_kernel"):
        assert kernel in log
    spills = [line for line in log.splitlines() if "spill" in line]
    assert spills and all(" 0 bytes spill stores, 0 bytes spill loads" in line for line in spills), "\n".join(spills)
