"""K5, the device loop's re-scoring of its candidate store after an extraction, on its own (rsc_debug_k5_hits drives
k5_hits and k5_compact as the loop calls them).  For every stored candidate the hit count must be, exactly, the
float64 oracle's number of compatible points among the newly disabled subset points (all of them counted as
enabled), and the store must keep, in order, the candidates the reference's removeinvalidshapes! keeps: not the
extracted one, none with a hit.  Covered: the gathered form (scratch set sized by the extracted candidate's score,
including a bound that is too small, so the masked fallback runs) and the masked form; the subset itself and its
Morton view as the source; the culled, small-batch and dense scorers; float32 and exact float64 clouds."""
import ctypes as C

import numpy as np
import pytest

from oracle import c_oracle as CO
from tests.helpers import oracle_params

pytestmark = pytest.mark.gpu

GATHERED, MASKED, VIEW = 0, 1, 2


@pytest.fixture(scope="module")
def R():
    import ransac_jl_b200 as R

    return R


def _words(mask):
    n = len(mask)
    packed = np.zeros(((n + 63) // 64) * 8, np.uint8)
    pb = np.packbits(np.asarray(mask, bool), bitorder="little")
    packed[: len(pb)] = pb
    return packed


def _k5(R, pc, cands, old_en, new_en, bound, form, best, params=None):
    """-> hits, flags (queue overflow, scratch overflow of the first attempt), survivors"""
    from ransac_jl_b200._lib import lib

    params = params or R.ransacparameters()
    pc.upload_subset(0)
    pc.isenabled = old_en
    arr = R.pack_cands(cands)
    nst = len(cands)
    hit = np.full(nst, -7, np.int32)
    flags = np.full(2, -7, np.int32)
    surv = np.full(nst, -7, np.int32)
    ns = C.c_int32()
    w = _words(new_en)
    cp = R.to_c(params)
    pc.ctx.check(lib.rsc_debug_k5_hits(pc.handle, C.byref(cp), arr, nst, w.ctypes.data, bound, form, best, hit.ctypes.data,
                                       flags.ctypes.data, surv.ctypes.data, C.byref(ns)))
    np.testing.assert_array_equal(pc.isenabled, new_en)  # the cloud keeps the mask of after the extraction
    return hit, flags, surv[: ns.value]


def _want(R, pc, cands, P, N, old_en, new_en, best, params=None):
    op = oracle_params(params or R.ransacparameters())
    sub = pc.subsets[0]
    newly = sub[old_en[sub] & ~new_en[sub]]
    hit = CO.score_counts(cands, P[newly], N[newly], op)[0] if len(newly) else np.zeros(len(cands), np.int32)
    surv = np.array([i for i in range(len(cands)) if i != best and hit[i] == 0], np.int32)
    return hit, surv, len(newly)


def _check(R, pc, cands, P, N, old_en, new_en, bound, form, best, params=None):
    hit, flags, surv = _k5(R, pc, cands, old_en, new_en, bound, form, best, params)
    want, wsurv, k = _want(R, pc, cands, P, N, old_en, new_en, best, params)
    np.testing.assert_array_equal(hit, want, err_msg=f"hits, form={form} newly={k} bound={bound}")
    np.testing.assert_array_equal(surv, wsurv, err_msg="survivors")
    return hit, flags, k


def _scene(R, n, seed, r=2):
    from ransac_jl_b200 import scenes

    sc = scenes.scene_mixed(seed, n, noise_frac=0.004, jitter_deg=1.5, outlier_frac=0.1, counts=(2, 1, 1, 1))
    V = np.ascontiguousarray(sc.vertices, np.float32)
    N = np.ascontiguousarray(sc.normals, np.float32)
    pc = R.RANSACCloud(V, N, r)
    return sc, pc, V.astype(np.float64), N.astype(np.float64)


def _masks(pc, k, seed, p_off=0.2):
    """old mask (some points disabled already) and new = old minus k enabled subset-0 points minus some points outside
    subset 0 (which must not count)"""
    rng = np.random.default_rng(seed)
    n = pc.size
    old = rng.random(n) >= p_off
    sub = pc.subsets[0]
    cand = sub[old[sub]]
    assert len(cand) >= k
    new = old.copy()
    new[rng.choice(cand, k, replace=False)] = False
    other = np.setdiff1d(np.arange(n), sub)
    new[rng.choice(other, min(len(other), 300), replace=False)] = False
    return old, new


@pytest.fixture(scope="module")
def mid(R):
    sc, pc, P, N = _scene(R, 20_000, 5)
    from ransac_jl_b200 import scenes

    cands = scenes.perturbed_candidates(sc, 75, seed=5)
    yield sc, pc, P, N, cands
    pc.close()


@pytest.mark.parametrize("view", [False, True], ids=["subset", "view"])
@pytest.mark.parametrize("form", [GATHERED, MASKED], ids=["gathered", "masked"])
@pytest.mark.parametrize("k", [0, 1, 511, 512, 513])
def test_newly_disabled_counts(R, mid, k, form, view):
    sc, pc, P, N, cands = mid
    old, new = _masks(pc, k, 100 + k)
    hit, flags, _ = _check(R, pc, cands, P, N, old, new, max(k, 1), form | (VIEW if view else 0), best=7)
    assert flags[1] == 0
    if k >= 511:
        assert (hit > 0).sum() > 5 and (hit == 0).sum() > 5


@pytest.mark.parametrize("view", [False, True], ids=["subset", "view"])
def test_scratch_bound_edges_and_fallback(R, mid, view):
    """newly disabled = the scratch size fits; one more overflows it, and the masked repeat gives the same answer"""
    sc, pc, P, N, cands = mid
    v = VIEW if view else 0
    for k, bound, over in ((512, 512, 0), (513, 512, 1), (1024, 1024, 0), (1025, 1024, 1), (513, 513, 0), (600, 1, 1)):
        old, new = _masks(pc, k, 7 * k + bound)
        _, flags, _ = _check(R, pc, cands, P, N, old, new, bound, GATHERED | v, best=0)
        assert flags[1] == over, (k, bound)


@pytest.mark.parametrize("nst", [1, 4095, 4096, 4097, 9000])
def test_store_sizes_and_scorers(R, mid, monkeypatch, nst):
    """every scorer K5 can take: culled (view, large store or RSC_LOOP_CULL=2), small-batch (nst <= 4096), dense
    (RSC_NO_SMALL, or beyond the small scorer's limits)"""
    from ransac_jl_b200 import scenes

    sc, pc, P, N, _ = mid
    cands = scenes.perturbed_candidates(sc, (nst + 3) // 4, seed=nst)[:nst]
    old, new = _masks(pc, 700, nst)
    best = nst // 2
    for cull in ("0", "1", "2"):
        monkeypatch.setenv("RSC_LOOP_CULL", cull)
        for nosmall in (False, True):
            if nosmall:
                monkeypatch.setenv("RSC_NO_SMALL", "1")
            else:
                monkeypatch.delenv("RSC_NO_SMALL", raising=False)
            for form in (GATHERED, MASKED, GATHERED | VIEW, MASKED | VIEW):
                _check(R, pc, cands, P, N, old, new, 700, form, best)


def test_beyond_the_small_scorers_evaluations(R, monkeypatch):
    """4096 candidates x a 40 k-point subset in the masked form is past the small scorer's 1.2e8 evaluations: the
    dense scorer takes it (the culled one on the view with the default RSC_LOOP_CULL, nst >= 4096)"""
    from ransac_jl_b200 import scenes

    sc, pc, P, N = _scene(R, 80_000, 9)
    cands = scenes.perturbed_candidates(sc, 1024, seed=9)
    old, new = _masks(pc, 900, 9)
    for cull in ("0", "1"):
        monkeypatch.setenv("RSC_LOOP_CULL", cull)
        for form in (GATHERED, MASKED, MASKED | VIEW):
            _check(R, pc, cands, P, N, old, new, 900, form, best=4095)
    pc.close()


@pytest.mark.parametrize("view", [False, True], ids=["subset-map", "view-cidx"])
def test_exact_cloud_reads_the_sources_float64_map(R, monkeypatch, view):
    """an exact float64 cloud whose points sit within ~1e-8 relative of the thresholds: the gathered scratch set's
    float64 map must follow its source (the subset's map, or the view's cidx), or the in-band decisions read other
    points"""
    from tests.test_exact_f64_gpu import threshold_scene
    from ransac_jl_b200 import scenes

    shapes, V, N = threshold_scene(R, seed=6, per_shape=1500)
    sub = np.random.default_rng(6).permutation(len(V))[: len(V) // 2].astype(np.int64)
    pc = R.RANSACCloud(V, N, [sub], exact=True)
    cands = list(shapes) + scenes.perturbed_candidates(scenes.scene_c1(), 5, seed=6)
    v = VIEW if view else 0
    for cull in ("0", "2"):
        monkeypatch.setenv("RSC_LOOP_CULL", cull)
        for k in (1, 513, 3000):
            old, new = _masks(pc, k, k)
            hit, _, _ = _check(R, pc, cands, V, N, old, new, k, GATHERED | v, best=1)
            assert k < 3000 or (hit[: len(shapes)] > 0).sum() >= len(shapes) // 2
            _check(R, pc, cands, V, N, old, new, k, MASKED | v, best=1)
    pc.close()
