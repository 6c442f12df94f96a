"""Normal estimation without a GPU: the NumPy oracle (oracle/normals_oracle.py) against itself and against analytic
answers, the scene it is calibrated on, and the C ABI / kernel build side of rsc_estimate_normals."""
import os
import shutil
import subprocess

import numpy as np
import pytest

from oracle import normals_oracle as NO

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def lattice(m=6, spacing=1.0):
    g = np.arange(m, dtype=np.float32) * np.float32(spacing)
    return np.stack(np.meshgrid(g, g, g, indexing="ij"), -1).reshape(-1, 3).astype(np.float32)


def clouds():
    rng = np.random.default_rng(5)
    rand = rng.normal(size=(3000, 3)).astype(np.float32)
    dup = np.repeat(rng.uniform(-1, 1, size=(300, 3)).astype(np.float32), 7, axis=0)
    return {"random": rand, "lattice": lattice(), "duplicates": dup[rng.permutation(len(dup))]}


@pytest.mark.parametrize("name", ["random", "lattice", "duplicates"])
@pytest.mark.parametrize("k", [3, 16, 32])
def test_bruteforce_and_kdtree_lists_agree(name, k):
    xyz = clouds()[name]
    np.testing.assert_array_equal(NO.knn_bruteforce(xyz, k), NO.knn_kdtree(xyz, k, delta=1))


def test_plane_normals_are_analytic():
    rng = np.random.default_rng(1)
    nrm = np.array([1.0, -2.0, 0.5])
    nrm /= np.linalg.norm(nrm)
    b = np.cross(nrm, [0, 0, 1.0])
    b /= np.linalg.norm(b)
    c = np.cross(nrm, b)
    uv = rng.uniform(-10, 10, size=(2000, 2))
    # float32 points exactly on a plane: axis-aligned normal, since a tilted plane cannot hold float32 points exactly
    xyz = np.zeros((2000, 3), np.float32)
    xyz[:, :2] = uv.astype(np.float32)
    xyz[:, 2] = np.float32(3.0)
    n32, _, n64, _ = NO.estimate_normals(xyz, 16, viewpoint=(0, 0, -5.0))
    np.testing.assert_allclose(n64, np.tile([0, 0, -1.0], (2000, 1)), atol=1e-12)
    # a tilted plane: within the rounding of the float32 coordinates
    xyz = (uv[:, :1] * b + uv[:, 1:] * c + 5.0).astype(np.float32)
    _, _, n64, _ = NO.estimate_normals(xyz, 16)
    ref = nrm * np.sign(nrm[np.argmax(np.abs(nrm))])
    assert np.abs(n64 - ref).max() < 1e-4


def test_lattice_ties_resolve_by_index():
    xyz = lattice()
    nbr = NO.knn_bruteforce(xyz, 7)
    # an interior point: itself, then its 6 face neighbours in ascending index order
    i = (2 * 6 + 3) * 6 + 2
    assert nbr[i, 0] == i
    assert list(nbr[i, 1:]) == sorted([i - 36, i - 6, i - 1, i + 1, i + 6, i + 36])
    # a corner with k = 5: itself, 3 face neighbours, then the lowest-index of the 3 edge-diagonal ones
    assert list(NO.knn_bruteforce(xyz, 5)[0]) == [0, 1, 6, 36, 7]


def test_sign_rules():
    rng = np.random.default_rng(2)
    xyz = np.zeros((500, 3), np.float32)
    xyz[:, 0] = rng.uniform(-1, 1, 500)
    xyz[:, 2] = rng.uniform(-1, 1, 500)  # the plane y = 0
    up, _, _, _ = NO.estimate_normals(xyz, 8, viewpoint=(0, 10.0, 0))
    down, _, _, _ = NO.estimate_normals(xyz, 8, viewpoint=(0, -10.0, 0))
    canon, _, _, _ = NO.estimate_normals(xyz, 8)
    np.testing.assert_allclose(up, np.tile(np.float32([0, 1, 0]), (500, 1)), atol=1e-6)
    np.testing.assert_allclose(down, -up, atol=1e-6)
    np.testing.assert_allclose(canon, up, atol=1e-6)  # largest component positive
    # a tilted cloud: the component of largest magnitude is positive
    xyz = (rng.normal(size=(400, 3)) * [5.0, 5.0, 0.1] @ np.linalg.qr(rng.normal(size=(3, 3)))[0]).astype(np.float32)
    _, _, n64, _ = NO.estimate_normals(xyz, 12)
    assert (n64[np.arange(400), np.argmax(np.abs(n64), axis=1)] > 0).all()


def test_nan_rows_and_small_clouds():
    xyz = lattice(3)
    xyz[4] = np.nan
    xyz[10, 1] = np.inf
    nrm, nbr, _, _ = NO.estimate_normals(xyz, 8)
    assert (nrm[[4, 10]] == 0).all() and (nbr[[4, 10]] == -1).all()
    assert not np.isin([4, 10], nbr).any()
    assert (np.abs(np.linalg.norm(nrm[np.isfinite(xyz).all(1)], axis=1) - 1) < 1e-6).all()
    for n in (1, 2):  # k_eff < 3: zero normals, lists of the finite points
        nrm, nbr, _, _ = NO.estimate_normals(xyz[:n] * 0 + np.float32([[0, 0, 0], [1, 0, 0]])[:n], 16)
        assert (nrm == 0).all() and (nbr[:, n:] == -1).all() and (nbr[:, :n] >= 0).all()
    tri = np.float32([[0, 0, 0], [1, 0, 0], [0, 1, 0], [5, 5, 0]])
    nrm, nbr, _, _ = NO.estimate_normals(tri, 16)  # n < k: every finite point
    assert (nbr[:, 4:] == -1).all()
    np.testing.assert_allclose(nrm, np.tile(np.float32([0, 0, 1]), (4, 1)), atol=1e-6)
    line = np.float32([[t, 2 * t, 0] for t in range(10)])
    assert (NO.estimate_normals(line, 4)[0] == 0).all()  # collinear neighbourhoods


def test_scene_view_faces_the_viewpoint():
    from ransac_jl_b200 import scenes

    view = scenes.SCAN_VIEWPOINT
    sc = scenes.scene_view(11, 20_000, viewpoint=view, noise_frac=0.0)
    assert sc.vertices.shape == (20_000, 3) and (sc.labels >= 0).all()
    facing = np.einsum("ij,ij->i", sc.normals.astype(np.float64), np.asarray(view) - sc.vertices)
    assert (facing > -1e-3).all()
    # a viewpoint at the centre of a sphere sees none of its outside: refused instead of drawing forever
    probe = scenes.scene_view(11, 100, noise_frac=0.0, counts=(0, 1, 0, 0))
    with pytest.raises(ValueError, match="faces the viewpoint"):
        scenes.scene_view(11, 100, viewpoint=probe.primitives[0].shape.center, noise_frac=0.0, counts=(0, 1, 0, 0))


# the device run on the scan scenario must recover at least this many primitives: the C oracle's loop finds all 8 with
# the analytic normals and 6 with the oracle's estimated normals (test below)
E2E_MIN_FOUND = 6


def test_oracle_normals_recover_the_primitives_in_the_c_loop():
    import ransac_jl_b200 as R
    from oracle import c_oracle
    from ransac_jl_b200 import scenes

    if not c_oracle.available():
        pytest.skip("oracle/liboracle.so not built")
    from tests.helpers import oracle_params

    scan = scenes.scan_scenario()
    sc = scan.scene
    op = oracle_params(R.ransacparameters(iteration=scan.iteration))
    subs = R.makesubsets(len(sc.vertices), scan.subsets, np.random.default_rng(1234))
    est, _, _, _ = NO.estimate_normals(sc.vertices, 16, viewpoint=scan.viewpoint)
    cos = np.einsum("ij,ij->i", est, sc.normals)
    assert np.median(cos) > 0.99 and (cos > 0).mean() > 0.99  # the viewpoint orients them like the ground truth
    found = {}
    for name, nrm in (("analytic", sc.normals), ("estimated", est)):
        got, _, _ = c_oracle.ransac(sc.vertices, nrm, subs[0], op, scan.seed)
        found[name] = scenes.recovered(sc, [(g[0], g[3]) for g in got])
    assert len(found["analytic"]) == len(sc.primitives) == 8
    assert len(found["estimated"]) >= E2E_MIN_FOUND


def test_null_context_is_refused_without_a_device():
    import ctypes as C

    import ransac_jl_b200 as R

    xyz = np.zeros((4, 3), np.float32)
    nrm = np.zeros((4, 3), np.float32)
    assert R._lib.lib.rsc_estimate_normals(None, xyz.ctypes.data, 4, 8, None, nrm.ctypes.data, None, None) == R._lib.RSC_E_ARG
    assert "rsc_estimate_normals" in R._lib.SIGNATURES
    assert R._lib.SIGNATURES["rsc_estimate_normals"][1][-1] == C.POINTER(C.c_int64)


@pytest.mark.skipif(shutil.which("nvcc") is None and not os.path.exists("/usr/local/cuda/bin/nvcc"), reason="nvcc not found")
def test_kernel_compiles_for_sm100a_without_spills(tmp_path):
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    csrc = os.path.join(ROOT, "ransac.jl_b200", "csrc")
    r = subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-fmad=false",
                        "-I" + os.path.join(ROOT, "include"), "-I" + csrc, "-Xptxas", "-v", "-c",
                        os.path.join(csrc, "rsc_normals.cu"), "-o", str(tmp_path / "n.o")], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    log = r.stderr
    assert "knn_normals_kernel" in log
    spills = [line for line in log.splitlines() if "spill" in line]
    assert spills and all(" 0 bytes spill stores, 0 bytes spill loads" in line for line in spills), "\n".join(spills)
