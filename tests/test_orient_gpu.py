"""rsc_orient_normals on the device against the NumPy oracle (oracle/orient_oracle.py orient_mst), bit for bit on
the output normals, the forest's edges and the stats, and oriented normals feeding the device RANSAC loop."""
import ctypes as C

import numpy as np
import pytest

from oracle import normals_oracle as NO
from oracle import orient_oracle as OO
from ransac_jl_b200 import scenes
from tests.test_normals_cpu import E2E_MIN_FOUND, lattice
from tests.test_orient_cpu import MIXED_FOUND, consistency, mixed_scene, random_signs, small_graphs

pytestmark = pytest.mark.gpu


def _dev(xyz, nrm, k):
    import ransac_jl_b200 as R

    return R.orient_normals(xyz, nrm, k=k, return_tree=True)


def _check(xyz, nrm, k, nbr=None):
    """device == oracle: normals bit for bit, F's edges, stats; returns the device result"""
    out, edges, stats = _dev(xyz, nrm, k)
    if nbr is None:
        nbr = NO.knn(xyz, k)
    if nrm is None:
        import ransac_jl_b200 as R

        nrm = R.estimate_normals(xyz, k=k)
    want, wedges, wstats = OO.orient_mst(xyz, nrm, nbr)
    assert out.tobytes() == want.tobytes()
    np.testing.assert_array_equal(edges, wedges)
    assert [stats[s] for s in ("vertices", "edges", "trees", "rounds")] == wstats.tolist()
    if stats["vertices"] > 1:
        assert stats["rounds"] <= int(np.ceil(np.log2(stats["vertices"])))
    return out, edges, stats


def _special():
    rng = np.random.default_rng(21)
    out = {name: g for name, g in small_graphs().items()}
    # several components: two blobs far apart (a lone point far from both joins the nearer through its own list)
    xyz = np.concatenate([rng.normal(size=(400, 3)), rng.normal(size=(300, 3)) + 1e3, [[5e3, 5e3, 5e3]]]).astype(np.float32)
    out["components"] = (xyz, rng.normal(size=(701, 3)).astype(np.float32))
    # coincident points: 7 copies of each of 200 positions, so i is not always first in its own list
    dup = np.repeat(rng.uniform(-1, 1, size=(200, 3)).astype(np.float32), 7, axis=0)
    perm = rng.permutation(len(dup))
    out["coincident"] = (dup[perm], rng.normal(size=(len(dup), 3)).astype(np.float32))
    # zero, NaN and Inf normals, NaN and Inf coordinates, a -0 z coordinate and a normal with z == 0
    xyz = rng.normal(size=(2000, 3)).astype(np.float32)
    nrm = rng.normal(size=(2000, 3)).astype(np.float32)
    nrm[rng.choice(2000, 40, replace=False)] = 0
    nrm[rng.choice(2000, 30, replace=False), rng.integers(0, 3, 30)] = np.nan
    nrm[rng.choice(2000, 20, replace=False), rng.integers(0, 3, 20)] = -np.inf
    xyz[rng.choice(2000, 30, replace=False), rng.integers(0, 3, 30)] = np.nan
    xyz[rng.choice(2000, 20, replace=False)] = np.inf
    out["non_finite"] = (xyz, nrm)
    # the top of the cloud at z == +-0 with z == 0 normals: the root's sign comes from the largest-magnitude rule
    xyz = rng.uniform(-1, 1, size=(500, 3)).astype(np.float32)
    xyz[:, 2] = -np.abs(xyz[:, 2])
    xyz[[10, 20, 30], 2] = np.float32([0.0, -0.0, 0.0])
    nrm = rng.normal(size=(500, 3)).astype(np.float32)
    nrm[[10, 20, 30], 2] = 0.0
    nrm[[10, 20, 30], 0] = np.float32([-2.0, 1.0, 0.5])
    out["flat_root"] = (xyz, nrm)
    return out


@pytest.mark.parametrize("name", ["random0", "two_blobs", "ties", "ties_signed", "components", "coincident", "non_finite",
                                  "flat_root"])
@pytest.mark.parametrize("k", [3, 16, 32])
def test_equals_the_oracle(name, k):
    xyz, nrm = _special()[name]
    _, _, stats = _check(xyz, nrm, k, NO.knn_bruteforce(xyz, k))
    if name == "components":
        assert stats["trees"] >= 2


@pytest.mark.parametrize("k", [3, 16, 32])
def test_tiny_clouds(k):
    rng = np.random.default_rng(k)
    for n in sorted({1, 2, 3, k - 1, k, k + 1}):
        xyz = rng.normal(size=(n, 3)).astype(np.float32)
        nrm = rng.normal(size=(n, 3)).astype(np.float32)
        _check(xyz, nrm, k, NO.knn_bruteforce(xyz, k))
        _check(xyz, None, k, NO.knn_bruteforce(xyz, k))


def test_estimating_mode_equals_orienting_the_estimate():
    import ransac_jl_b200 as R

    sc = scenes.scan_scenario().scene
    a, ea, sa = _check(sc.vertices, None, 16)
    b, eb, sb = _dev(sc.vertices, R.estimate_normals(sc.vertices, k=16), 16)
    assert a.tobytes() == b.tobytes() and sa == sb
    np.testing.assert_array_equal(ea, eb)


def test_in_place():
    from ransac_jl_b200._lib import Context, lib

    xyz, nrm = _special()["non_finite"]
    want = _dev(xyz, nrm, 12)[0]
    ctx = Context.get(0)
    buf = nrm.copy()
    ctx.check(lib.rsc_orient_normals(ctx.h, xyz.ctypes.data, len(xyz), 12, buf.ctypes.data, buf.ctypes.data, None, None))
    assert buf.tobytes() == want.tobytes()


def test_one_million_point_scene_mixed():
    sc = scenes.scene_mixed(41, 1_000_000)
    _, _, stats = _check(sc.vertices, random_signs(sc.normals), 16)
    assert stats["vertices"] == 1_000_000


def test_random_signs_orient_like_the_ground_truth_in_the_device_loop():
    import ransac_jl_b200 as R

    scan = scenes.scan_scenario()
    sc = mixed_scene()
    out = R.orient_normals(sc.vertices, random_signs(sc.normals))
    assert (consistency(sc, out) == 1.0).all()
    pc = R.RANSACCloud(sc.vertices, out, scan.subsets)
    ext, _ = R.ransac(pc, R.ransacparameters(iteration=scan.iteration), True, seed=scan.seed)
    assert len(scenes.recovered(sc, [(e.shape.kind, np.asarray(e.inpoints)) for e in ext])) >= MIXED_FOUND


def test_oriented_estimates_drive_the_device_loop_without_a_viewpoint():
    import ransac_jl_b200 as R

    scan = scenes.scan_scenario()
    sc = scan.scene
    nrm = R.orient_normals(sc.vertices)
    assert consistency(sc, nrm).min() > 0.99
    pc = R.RANSACCloud(sc.vertices, nrm, scan.subsets)
    ext, _ = R.ransac(pc, R.ransacparameters(iteration=scan.iteration), True, seed=scan.seed)
    assert len(scenes.recovered(sc, [(e.shape.kind, np.asarray(e.inpoints)) for e in ext])) >= E2E_MIN_FOUND


def test_refusals():
    import ransac_jl_b200 as R
    from ransac_jl_b200._lib import RSC_E_ARG, Context, RscError, lib

    xyz = lattice(3)
    for k in (2, 33, -1):
        with pytest.raises(RscError, match="k must be"):
            R.orient_normals(xyz, k=k)
    with pytest.raises(RscError, match="n must be"):
        R.orient_normals(np.zeros((0, 3), np.float32))
    ctx = Context.get(0)
    out = np.zeros((27, 3), np.float32)
    assert lib.rsc_orient_normals(ctx.h, None, 27, 8, None, out.ctypes.data, None, None) == RSC_E_ARG
    assert b"must not be NULL" in lib.rsc_last_error(ctx.h)
    assert lib.rsc_orient_normals(ctx.h, xyz.ctypes.data, 27, 8, None, None, None, None) == RSC_E_ARG
    assert lib.rsc_orient_normals(ctx.h, xyz.ctypes.data, 1 << 31, 8, None, out.ctypes.data, None, None) == RSC_E_ARG
    stats = (C.c_int64 * 4)()
    assert lib.rsc_orient_normals(ctx.h, xyz.ctypes.data, 27, 8, None, out.ctypes.data, None, stats) == 0
    assert stats[0] == stats[1] + stats[2] and stats[3] >= 0
