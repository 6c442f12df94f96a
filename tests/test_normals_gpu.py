"""rsc_estimate_normals on the device against the NumPy oracle (oracle/normals_oracle.py): neighbour lists bit for bit
on clouds built to stress the exact search (ties, cell boundaries, level escalation, a search of the whole box,
non-finite rows, tiny clouds), normals to eigen-solver accuracy, and device normals feeding the device RANSAC loop.
The distances the device evaluates equal those of a host model of its level choices (tests/normals_search_model.py),
which shows that the escalation and whole-box paths run."""
import ctypes as C

import numpy as np
import pytest

from oracle import normals_oracle as NO
from ransac_jl_b200 import scenes
from tests.normals_search_model import search_model
from tests.test_normals_cpu import E2E_MIN_FOUND, clouds, lattice

VIEW = scenes.SCAN_VIEWPOINT

pytestmark = pytest.mark.gpu


def _dev(xyz, k, viewpoint=None):
    import ransac_jl_b200 as R

    return R.estimate_normals(xyz, k=k, viewpoint=viewpoint, return_neighbours=True)


def _special():
    rng = np.random.default_rng(9)
    out = dict(clouds())
    # integer coordinates in [0, 256]: with this bounding box every one lies on a cell boundary of many levels
    b = rng.integers(0, 257, size=(6000, 3)).astype(np.float32)
    b[0], b[1] = 0, 256
    out["cell_boundaries"] = b
    # a dense cluster inside a sparse cloud, density ratio 10^6 : 1 (some queries escalate one level)
    out["density_contrast"] = np.concatenate([rng.uniform(-50, 50, (5000, 3)), rng.uniform(-0.5, 0.5, (5000, 3))]).astype(np.float32)
    # a lone far outlier: its own cell holds too few points at every level below the whole box, so it starts there
    o = rng.uniform(0, 1, (3000, 3)).astype(np.float32)
    o[1234] = 1e6
    out["far_outlier"] = o
    nf = rng.normal(size=(4000, 3)).astype(np.float32)
    nf[rng.choice(4000, 300, replace=False), rng.integers(0, 3, 300)] = np.nan
    nf[rng.choice(4000, 50, replace=False)] = np.inf
    nf[17, 2] = -np.inf
    out["non_finite"] = nf
    return out


def escalating(k):
    """a query whose start cell (level 3, side 1/4 of the box) holds it and k - 1 points in the opposite corner, farther
    than the 3x3x3 block reaches: its search must escalate to level 2, which covers the whole box"""
    rng = np.random.default_rng(k)
    corner = rng.uniform(0, 1e-3, (k - 1, 3))
    far = rng.uniform(0.6, 1.0, (50, 3))
    return np.concatenate([corner, [[0.249, 0.249, 0.249], [1.0, 1.0, 1.0]], far]).astype(np.float32)


def _pairs(xyz, k):
    from ransac_jl_b200._lib import Context, lib

    ctx = Context.get(0)
    xyz = np.ascontiguousarray(xyz, np.float32)
    out = np.empty_like(xyz)
    pairs = C.c_int64(-1)
    ctx.check(lib.rsc_estimate_normals(ctx.h, xyz.ctypes.data, len(xyz), k, None, out.ctypes.data, None, C.byref(pairs)))
    return pairs.value


@pytest.mark.parametrize("name", ["lattice", "duplicates", "cell_boundaries", "density_contrast", "far_outlier", "non_finite",
                                  "escalating"])
@pytest.mark.parametrize("k", [3, 16])
def test_search_levels_and_distance_counts(name, k):
    xyz = escalating(k) if name == "escalating" else _special()[name]
    pairs, start, accept = search_model(xyz, k)
    assert _pairs(xyz, k) == pairs
    if name == "escalating":
        q = k - 1  # the query in the corner
        assert start[q] == 3 and accept[q] == 2
        np.testing.assert_array_equal(_dev(xyz, k)[1], NO.knn_bruteforce(xyz, k))
    if name == "far_outlier":
        assert start[1234] == 1 and accept[1234] == 1 and (start[np.arange(len(xyz)) != 1234] > 1).all()
    if name == "density_contrast" and k == 3:
        assert (accept < start).any()


@pytest.mark.parametrize("name", ["random", "lattice", "duplicates", "cell_boundaries", "density_contrast", "far_outlier",
                                  "non_finite"])
@pytest.mark.parametrize("k", [3, 16, 32])
def test_lists_equal_the_oracle(name, k):
    xyz = _special()[name]
    nrm, nbr = _dev(xyz, k)
    want = NO.knn_bruteforce(xyz, k)
    np.testing.assert_array_equal(nbr, want)
    wn, _, _ = NO.pca_normals(xyz, want)
    np.testing.assert_array_equal((nrm == 0).all(1), (wn == 0).all(1))


@pytest.mark.parametrize("k", [3, 16, 32])
def test_tiny_clouds(k):
    rng = np.random.default_rng(k)
    for n in sorted({1, 2, 3, k - 1, k, k + 1}):
        xyz = rng.normal(size=(n, 3)).astype(np.float32)
        nrm, nbr = _dev(xyz, k)
        want = NO.knn_bruteforce(xyz, k)
        np.testing.assert_array_equal(nbr, want)
        wn, _, _ = NO.pca_normals(xyz, want)
        if n < 3:
            assert (nrm == 0).all()
        np.testing.assert_array_equal((nrm == 0).all(1), (wn == 0).all(1))


def _compare_normals(xyz, nrm, viewpoint, k):
    want, nbr, n64, ev = NO.estimate_normals(xyz, k, viewpoint)
    zero = (want == 0).all(1)
    np.testing.assert_array_equal((nrm == 0).all(1), zero)
    healthy = ~zero & ((ev[:, 1] - ev[:, 0]) > 1e-6 * ev[:, 2])
    got = nrm[healthy].astype(np.float64)
    cos = np.abs(np.einsum("ij,ij->i", got / np.linalg.norm(got, axis=1)[:, None], n64[healthy]))
    ang = np.arccos(np.minimum(cos, 1.0))
    assert ang.max() < 1e-6, ang.max()
    same = np.einsum("ij,ij->i", got, n64[healthy]) > 0
    if viewpoint is not None:
        d = np.asarray(viewpoint) - xyz[healthy].astype(np.float64)
        s = np.einsum("ij,ij->i", n64[healthy], d)
        rounding = np.abs(s) < 1e-9 * np.linalg.norm(d, axis=1)
        assert (same | rounding).all()
    else:
        assert same.all()
    return nbr


@pytest.mark.parametrize("viewpoint", [None, VIEW])
def test_normals_match_the_oracle_on_a_scan(viewpoint):
    sc = scenes.scene_view(3, 30_000, viewpoint=VIEW, noise_frac=0.002)
    nrm, nbr = _dev(sc.vertices, 16, viewpoint)
    want = _compare_normals(sc.vertices, nrm, viewpoint, 16)
    np.testing.assert_array_equal(nbr, want)


def test_one_million_point_scene_mixed():
    sc = scenes.scene_mixed(41, 1_000_000)
    nrm, nbr = _dev(sc.vertices, 16, VIEW)
    want = NO.knn_kdtree(sc.vertices, 16)
    np.testing.assert_array_equal(nbr, want)
    rows = np.random.default_rng(0).choice(len(sc.vertices), 20_000, replace=False)
    wn, n64, ev = NO.pca_normals(sc.vertices, want, VIEW)
    healthy = (ev[rows, 1] - ev[rows, 0]) > 1e-6 * ev[rows, 2]
    g = nrm[rows][healthy].astype(np.float64)
    assert np.abs(g - n64[rows][healthy]).max() < 1e-6


def test_permutation_permutes_every_output_bit():
    rng = np.random.default_rng(4)
    xyz = rng.normal(size=(50_000, 3)).astype(np.float32)
    perm = rng.permutation(len(xyz))
    inv = np.empty_like(perm)
    inv[perm] = np.arange(len(perm))
    a_n, a_b = _dev(xyz, 16, VIEW)
    b_n, b_b = _dev(xyz[perm], 16, VIEW)
    assert b_n.tobytes() == a_n[perm].tobytes()
    np.testing.assert_array_equal(b_b, inv[a_b[perm]])


def test_float64_input_is_its_float32_rounding():
    import ransac_jl_b200 as R

    rng = np.random.default_rng(6)
    x64 = rng.normal(size=(20_000, 3)) * 10.0
    a = R.estimate_normals(x64, k=12, viewpoint=VIEW)
    b = R.estimate_normals(x64.astype(np.float32), k=12, viewpoint=VIEW)
    assert a.dtype == np.float32 and a.shape == (20_000, 3)
    assert a.tobytes() == b.tobytes()


def test_device_normals_drive_the_device_loop():
    import ransac_jl_b200 as R

    scan = scenes.scan_scenario()
    sc = scan.scene
    nrm = R.estimate_normals(sc.vertices, viewpoint=scan.viewpoint)
    pc = R.RANSACCloud(sc.vertices, nrm, scan.subsets)
    ext, _ = R.ransac(pc, R.ransacparameters(iteration=scan.iteration), True, seed=scan.seed)
    found = scenes.recovered(sc, [(e.shape.kind, np.asarray(e.inpoints)) for e in ext])
    assert len(found) >= E2E_MIN_FOUND


def test_refusals():
    import ransac_jl_b200 as R
    from ransac_jl_b200._lib import RSC_E_ARG, Context, RscError, lib

    xyz = lattice(3)
    for k in (2, 33, -1):
        with pytest.raises(RscError, match="k must be"):
            R.estimate_normals(xyz, k=k)
    with pytest.raises(RscError, match="n must be"):
        R.estimate_normals(np.zeros((0, 3), np.float32))
    ctx = Context.get(0)
    out = np.zeros((27, 3), np.float32)
    assert lib.rsc_estimate_normals(ctx.h, None, 27, 8, None, out.ctypes.data, None, None) == RSC_E_ARG
    assert b"must not be NULL" in lib.rsc_last_error(ctx.h)
    assert lib.rsc_estimate_normals(ctx.h, xyz.ctypes.data, 27, 8, None, None, None, None) == RSC_E_ARG
    assert lib.rsc_estimate_normals(ctx.h, xyz.ctypes.data, 1 << 31, 8, None, out.ctypes.data, None, None) == RSC_E_ARG
    pairs = C.c_int64(-1)
    assert lib.rsc_estimate_normals(ctx.h, xyz.ctypes.data, 27, 8, None, out.ctypes.data, None, C.byref(pairs)) == 0
    assert pairs.value >= 27 * 8
