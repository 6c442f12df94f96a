"""Flattened octree + level-weighted cell sampler (extension, SURVEY 8(f)-1) against its restatement in
oracle/ransac_oracle.py (MortonOctree, sample_minimal_set_octree): Morton order, leaf depths, drawn
sets and levels, and the whole loop with level-weight updates must be identical."""
import numpy as np
import pytest

from oracle import ransac_oracle as O
from tests.helpers import oracle_params

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def R():
    import ransac_jl_b200 as R

    return R


def _scene(n, seed=91):
    from ransac_jl_b200 import scenes

    return scenes.scene_mixed(seed, n, noise_frac=0.003, jitter_deg=1.5, outlier_frac=0.15, counts=(3, 2, 1, 1))


@pytest.mark.parametrize("nlevels", [1, 4, 8, 11])
def test_cells_match_oracle(R, nlevels):
    sc = _scene(50_000)
    pc = R.RANSACCloud(sc.vertices, sc.normals, 2).build_cells(nlevels)
    codes, perm, ld = pc.get_cells()
    oc = O.MortonOctree(sc.vertices, nlevels)
    np.testing.assert_array_equal(codes.astype(np.int64), oc.codes)
    np.testing.assert_array_equal(perm.astype(np.int64), oc.perm)  # stable order: ties keep the point order
    np.testing.assert_array_equal(ld.astype(np.int32), oc.leafdepth)


def test_duplicate_points_and_flat_axis(R):
    """coincident points (the reference's tree would recurse forever, Q20) and a degenerate axis"""
    rng = np.random.default_rng(2)
    V = rng.uniform(-5, 5, (3000, 3)).astype(np.float32)
    V[:, 2] = 1.25  # flat in z
    V[100:140] = V[7]  # 41 coincident points: their cell never drops to <= 8 points
    N = np.tile(np.array([[0, 0, 1.0]], np.float32), (3000, 1))
    pc = R.RANSACCloud(V, N, 1).build_cells(9)
    codes, perm, ld = pc.get_cells()
    oc = O.MortonOctree(V, 9)
    np.testing.assert_array_equal(perm.astype(np.int64), oc.perm)
    np.testing.assert_array_equal(ld.astype(np.int32), oc.leafdepth)
    assert ld[7] == 9


def test_cell_sampler_matches_oracle(R):
    sc = _scene(40_000)
    pc = R.RANSACCloud(sc.vertices, sc.normals, 2).build_cells(8)
    en = np.random.default_rng(3).random(pc.size) > 0.35
    pc.isenabled = en
    params = R.ransacparameters()
    lw = np.array([0.05, 0.1, 0.3, 0.2, 0.15, 0.1, 0.06, 0.04])
    S = 3000
    shapes, sets, idx, level = R.sample_fit_cells(pc, params, seed=77, set0=5000, S=S, levelweight=lw)
    oc = O.MortonOctree(sc.vertices, 8)
    opc = O.Cloud(sc.vertices, sc.normals, [s.copy() for s in pc.subsets], en.copy())
    cum = O.level_cumsum(lw)
    en_sorted = en[oc.perm]
    nfail = 0
    for s in range(S):
        ok, lvl, sd = O.sample_minimal_set_octree(opc, oc, 3, O.SetStream(77, 5000 + s), cum, en_sorted)
        assert level[s] == lvl, s
        if ok:
            np.testing.assert_array_equal(idx[s], sd)
        else:
            nfail += 1
            assert (idx[s] == -1).all()
    assert 0 < nfail < S  # both outcomes occur (small cells run out of enabled points)
    assert len(np.unique(level)) >= 5
    # the candidates are the fits of exactly those sets
    op = oracle_params(params)
    want = []
    for s in range(S):
        if idx[s, 0] >= 0:
            want += [(s, sh.kind) for sh in O.forcefit(opc.vertices[idx[s]], opc.normals[idx[s]], op)]
    assert [(int(a), sh.to_cand().type) for a, sh in zip(sets, shapes)] == want


@pytest.mark.parametrize("loop_cull", ["0", "2"], ids=["dense", "culled-scorer-in-K2-and-K5"])
def test_loop_with_cell_sampler_matches_oracle(R, monkeypatch, loop_cull):
    """both ways of scoring inside the loop: the dense kernels, and the culled scorer on the subset's Morton view for
    every batch of new candidates (K2) and for the re-scoring of the store after an extraction (K5)"""
    monkeypatch.setenv("RSC_LOOP_CULL", loop_cull)
    sc = _scene(60_000, seed=92)
    pc = R.RANSACCloud(sc.vertices, sc.normals, 4).build_cells(8)
    params = R.ransacparameters(iteration={"tau": 500, "minsubsetN": 128, "itermax": 50})
    extracted, _ = R.ransac(pc, params, True, seed=11, sampler="octree")
    oc = O.MortonOctree(sc.vertices, 8)
    opc = O.Cloud(sc.vertices, sc.normals, [s.copy() for s in pc.subsets])
    tr = O.RansacTrace()
    want = O.ransac(opc, oracle_params(params), True, seed=11, trace=tr, octree=oc)
    assert len(extracted) == len(want) and len(want) >= 3
    for got, w in zip(extracted, want):
        assert got.shape.to_cand().type == w.shape.kind
        np.testing.assert_array_equal(got.inpoints, w.inpoints)
    np.testing.assert_array_equal(pc.isenabled, opc.isenabled)
    np.testing.assert_allclose(pc.levelweight, tr.levelweight, rtol=1e-12)
    # and the root-cell run is untouched by the presence of the cells
    a, _ = R.ransac(pc, params, True, seed=11)
    pc2 = R.RANSACCloud(sc.vertices, sc.normals, pc.subsets)
    b, _ = R.ransac(pc2, params, True, seed=11)
    assert [len(x.inpoints) for x in a] == [len(x.inpoints) for x in b]


def test_cell_sampler_batched_with_a_refresh_period_matches_oracle_and_batch1(R, monkeypatch):
    """lw_period = 8: the level weights are refreshed every 8 iterations, so the loop can run up to 8 iterations
    per speculative batch; the results equal the oracle's loop with the same period AND the run forced to one
    iteration per batch (RSC_BATCH=1) -- the period defines the result, the batching does not"""
    sc = _scene(60_000, seed=93)
    params = R.ransacparameters(iteration={"tau": 500, "minsubsetN": 128, "itermax": 48})
    pc = R.RANSACCloud(sc.vertices, sc.normals, 4).build_cells(8)
    batched, _ = R.ransac(pc, params, True, seed=13, sampler="octree", lw_period=8)
    lw_b = pc.levelweight.copy()
    monkeypatch.setenv("RSC_BATCH", "1")
    single, _ = R.ransac(pc, params, True, seed=13, sampler="octree", lw_period=8)
    monkeypatch.delenv("RSC_BATCH")
    assert len(batched) == len(single)
    for a, b in zip(batched, single):
        assert list(a.shape.to_cand().p) == list(b.shape.to_cand().p)
        np.testing.assert_array_equal(a.inpoints, b.inpoints)
    np.testing.assert_array_equal(lw_b, pc.levelweight)
    oc = O.MortonOctree(sc.vertices, 8)
    opc = O.Cloud(sc.vertices, sc.normals, [s.copy() for s in pc.subsets])
    tr = O.RansacTrace()
    want = O.ransac(opc, oracle_params(params), True, seed=13, trace=tr, octree=oc, lw_period=8)
    assert len(batched) == len(want) and len(want) >= 3
    for got, w in zip(batched, want):
        assert got.shape.to_cand().type == w.shape.kind
        np.testing.assert_array_equal(got.inpoints, w.inpoints)
    np.testing.assert_allclose(lw_b, tr.levelweight, rtol=1e-12)
    # a different period is a different (equally valid) schedule
    other, _ = R.ransac(pc, params, True, seed=13, sampler="octree", lw_period=1)
    assert len(other) >= 3


def test_reference_grid_leaf_depth(R):
    # test/octree.jl:116-139 on the device structure: 6^3 grid, every leaf at depth 3
    ps = (np.array([[i, j, k] for i in range(6) for j in range(6) for k in range(6)], float) / 3).astype(np.float32)
    for nlevels in (3, 6):
        pc = R.RANSACCloud(ps, ps, 1).build_cells(nlevels)
        _, perm, ld = pc.get_cells()
        assert (ld == 3).all()
        np.testing.assert_array_equal(perm.astype(np.int64), O.MortonOctree(ps, nlevels).perm)


def test_cell_sampler_with_empty_batches_matches_oracle(R):
    """one plane type, one set per iteration: most iterations fit no candidate, so most batches are empty -- their
    level statistics must add nothing to the level scores"""
    sc = _scene(20_000, seed=94)
    subsets = R.makesubsets(len(sc.vertices), 2, np.random.default_rng(1234))
    params = R.ransacparameters([R.FittedPlane], iteration={"tau": 200, "minsubsetN": 1, "itermax": 300})
    pc = R.RANSACCloud(sc.vertices, sc.normals, subsets).build_cells(8)
    extracted, _ = R.ransac(pc, params, True, seed=17, sampler="octree")
    oc = O.MortonOctree(sc.vertices, 8)
    opc = O.Cloud(sc.vertices, sc.normals, [s.copy() for s in subsets])
    tr = O.RansacTrace()
    want = O.ransac(opc, oracle_params(params), True, seed=17, trace=tr, octree=oc)
    assert tr.candidates_scored < tr.iterations  # (at most one candidate per iteration: some iterations had none)
    assert len(extracted) == len(want)
    np.testing.assert_array_equal(pc.isenabled, opc.isenabled)
    np.testing.assert_allclose(pc.levelweight, tr.levelweight, rtol=1e-12)
