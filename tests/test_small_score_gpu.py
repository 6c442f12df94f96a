"""The device loop's small-batch scorer (rsc_small.cu) on its own, through rsc_debug_score_small: a thread per
point, 128-candidate chunks in shared memory spread over gridDim.y, a candidate count read from the device and
clamped to the launch's capacity, whole padding words skipped per warp, and in-band pairs decided inline in FP64.
Its two counts (compatible real points cv, compatible enabled points ce) must be the float64 oracle's, bit for
bit, and agree with rsc_score's policy counts (ce, but cv for spheres under quirk Q4) on the same inputs."""
import ctypes as C
import math

import numpy as np
import pytest

from oracle import c_oracle as CO
from tests.helpers import adversarial_case, oracle_params

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def R():
    import ransac_jl_b200 as R

    return R


def _pack(cands):
    from ransac_jl_b200 import _lib

    if isinstance(cands, C.Array):
        return cands
    arr = (_lib.rsc_cand * len(cands))()
    for i, s in enumerate(cands):
        arr[i] = s.to_cand() if hasattr(s, "to_cand") else s
    return arr


def _small(R, pc, cands, params, subset=-1, count=-1, cap=None):
    """(cv, ce) of the small-batch scorer; count >= 0: the synchronisation-free form with capacity `cap`"""
    from ransac_jl_b200._lib import lib

    arr = _pack(cands)
    cap = len(arr) if cap is None else cap
    assert cap <= len(arr)
    if subset >= 0:
        pc.upload_subset(subset)
    cv = np.full(cap, -7, np.int32)  # (overwritten everywhere: the scorer zeroes its outputs)
    ce = np.full(cap, -7, np.int32)
    cp = R.to_c(params)
    pc.ctx.check(lib.rsc_debug_score_small(pc.handle, C.byref(cp), subset, arr, cap, count, cv.ctypes.data, ce.ctypes.data))
    return cv, ce


def _oracle(cands, P, N, op, en):
    """float64 oracle: cv over every point, ce over the enabled points only, and the Q4 policy counts"""
    P = np.asarray(P, np.float64)
    N = np.asarray(N, np.float64)
    cv = CO.score_counts(cands, P, N, op)[0]
    ce = CO.score_counts(cands, P[en], N[en], op)[0] if en.any() else np.zeros(len(cands), np.int32)
    pol = CO.score_counts(cands, P, N, op, enabled=en)[0]
    return cv, ce, pol


def _check(R, pc, cands, P, N, en, params=None, subset=-1, idx=None):
    """the small-batch scorer against the oracle and rsc_score, in both launch forms; returns (cv, ce)"""
    params = params or R.ransacparameters()
    op = oracle_params(params)
    if idx is not None:
        P, N, en = P[idx], N[idx], en[idx]
    cv_w, ce_w, pol_w = _oracle(cands, P, N, op, en)
    cv, ce = _small(R, pc, cands, params, subset)
    np.testing.assert_array_equal(cv, cv_w, err_msg="cv (compatible real points)")
    np.testing.assert_array_equal(ce, ce_w, err_msg="ce (compatible enabled points)")
    sphere = np.array([s.to_cand().type == 1 for s in cands])
    np.testing.assert_array_equal(np.where(sphere, cv, ce), pol_w, err_msg="Q4 policy counts")
    dense, _ = R.score_counts(pc, cands, subset, params)
    np.testing.assert_array_equal(dense, pol_w, err_msg="rsc_score")
    # the synchronisation-free form: the count on the device, equal to the capacity
    cv2, ce2 = _small(R, pc, cands, params, subset, count=len(cands))
    np.testing.assert_array_equal(cv2, cv)
    np.testing.assert_array_equal(ce2, ce)
    return cv, ce


def _cloud(R, n, seed, disable=0.3, **kw):
    from ransac_jl_b200 import scenes

    sc = scenes.scene_mixed(seed, max(n, 64), noise_frac=0.004, jitter_deg=1.5, outlier_frac=0.1, counts=(1, 1, 1, 1))
    V = np.ascontiguousarray(sc.vertices[:n], np.float32)
    N = np.ascontiguousarray(sc.normals[:n], np.float32)
    pc = R.RANSACCloud(V, N, kw.get("subsets", 1))
    en = np.random.default_rng(seed).random(n) >= disable
    pc.isenabled = en
    return sc, pc, V.astype(np.float64), N.astype(np.float64), en


@pytest.mark.parametrize("ncand", [1, 127, 128, 129, 255, 257, 4096, 4097, 5000])
def test_candidate_chunks_and_rows_of_chunks(R, ncand):
    """many candidates against 512 points: the 128-candidate chunks, a partial last chunk, and gridDim.y > 1
    (a 512-point set has 2 point tiles, so the chunks are spread over up to ceil(C / 128) rows)"""
    from ransac_jl_b200 import scenes

    sc, pc, P, N, en = _cloud(R, 512, 40 + ncand % 97)
    cands = scenes.perturbed_candidates(sc, (ncand + 3) // 4, seed=ncand)[:ncand]
    cv, ce = _check(R, pc, cands, P, N, en)
    assert cv.sum() > 0 and (cv >= ce).all()
    if ncand >= 128:
        assert (cv[-64:] > 0).any(), "the last chunk's candidates see points"
        sphere = np.array([c.to_cand().type == 1 for c in cands])
        assert (cv[sphere] > ce[sphere]).any(), "spheres count the disabled points in cv"
    pc.close()


@pytest.mark.parametrize("npts", [1, 31, 32, 33, 511, 512, 513, 2049])
def test_point_counts_and_padding_words(R, npts):
    """ragged point counts: partial last words, whole padding words in the last 256-point tile, one and several
    tiles; on the whole cloud and on a subset copy (whose padding starts earlier)"""
    from ransac_jl_b200 import scenes

    sc, pc, P, N, en = _cloud(R, npts, 7 + npts, subsets=2)
    cands = scenes.perturbed_candidates(sc, 75, seed=npts)
    _check(R, pc, cands, P, N, en)
    sub = pc.subsets[0]
    if len(sub):
        _check(R, pc, cands, P, N, en, subset=0, idx=sub)
    pc.close()


def test_all_points_disabled_and_all_enabled(R):
    from ransac_jl_b200 import scenes

    sc, pc, P, N, en = _cloud(R, 700, 3)
    cands = scenes.perturbed_candidates(sc, 30, seed=3)
    pc.isenabled = np.zeros(700, bool)
    cv, ce = _check(R, pc, cands, P, N, np.zeros(700, bool))
    assert (ce == 0).all() and cv.sum() > 0
    pc.enable_all()
    cv, ce = _check(R, pc, cands, P, N, np.ones(700, bool))
    np.testing.assert_array_equal(cv, ce)
    pc.close()


def test_adversarial_candidates_and_points(R):
    """NaN / Inf / zero-axis candidates, points on axes and at centres, zero and non-unit normals, huge and tiny
    radii, wide and flat cones (tests.helpers.adversarial_case), with disabled points"""
    from ransac_jl_b200 import _lib
    from ransac_jl_b200.shapes import from_cand

    oshapes, P, N = adversarial_case()
    cands = []
    for sh in oshapes:
        c = _lib.rsc_cand(type=int(sh.kind), outwards=int(bool(sh.outwards)))
        for i, v in enumerate(sh.params7()):
            c.p[i] = float(v)
        cands.append(from_cand(c))
    pc = R.RANSACCloud(P.astype(np.float32), N.astype(np.float32), 2)
    en = np.random.default_rng(9).random(len(P)) >= 0.25
    pc.isenabled = en
    cv, ce = _check(R, pc, cands, P, N, en)
    assert cv.sum() > 0
    _check(R, pc, cands, P, N, en, subset=1, idx=pc.subsets[1])
    pc.close()


def test_out_of_range_type_ids_count_nothing(R):
    """type ids outside 0..3 compile to no column (-1): zero counts, and their neighbours in the chunk are unaffected"""
    from ransac_jl_b200 import scenes

    sc, pc, P, N, en = _cloud(R, 1000, 5)
    cands = scenes.perturbed_candidates(sc, 70, seed=5)  # 280: three chunks
    params = R.ransacparameters()
    cv0, ce0 = _check(R, pc, cands, P, N, en)
    arr = _pack(cands)
    bad = [0, 1, 127, 128, 200, 279]
    for j, t in zip(bad, (-1, 4, 7, 16, -100, 2**31 - 1)):
        arr[j].type = t
    for count in (-1, len(cands)):
        cv, ce = _small(R, pc, arr, params, count=count)
        assert (cv[bad] == 0).all() and (ce[bad] == 0).all()
        keep = np.setdiff1d(np.arange(len(cands)), bad)
        np.testing.assert_array_equal(cv[keep], cv0[keep])
        np.testing.assert_array_equal(ce[keep], ce0[keep])
    assert (cv0[bad] > 0).any()  # (so zero is not what those candidates scored anyway)
    pc.close()


def test_wide_flat_cones_and_non_unit_vectors(R):
    """cones of 120 to 330 degrees opening (wide-cone column, flat and reflex angles), non-unit plane normals,
    cylinder and cone axes, and non-unit point normals"""
    from ransac_jl_b200 import FittedCone, FittedCylinder, FittedPlane, scenes

    sc, pc0, P, N, en = _cloud(R, 3000, 21)
    pc0.close()
    rng = np.random.default_rng(21)
    N = N * rng.uniform(0.3, 3.0, (len(N), 1))
    N = N.astype(np.float32).astype(np.float64)
    pc = R.RANSACCloud(P.astype(np.float32), N.astype(np.float32), 1)
    pc.isenabled = en
    cands = []
    for i, s in enumerate(scenes.perturbed_candidates(sc, 60, seed=21)):
        k = float(rng.choice([0.25, 0.7, 1.0, 1.9, 4.0]))
        if isinstance(s, FittedPlane):
            s = FittedPlane(s.point, np.asarray(s.normal) * k)
        elif isinstance(s, FittedCylinder):
            s = FittedCylinder(np.asarray(s.axis) * k, s.center, s.radius, s.outwards)
        elif isinstance(s, FittedCone):
            deg = [120.0, 150.0, 179.0, 180.0, 181.0, 240.0, 300.0, 330.0][i % 8]
            s = FittedCone(s.apex, np.asarray(s.axis) * k, math.radians(deg), s.outwards)
        cands.append(s)
    cv, ce = _check(R, pc, cands, P, N, en)
    cones = np.array([isinstance(s, FittedCone) for s in cands])
    assert cv[cones].sum() > 0
    pc.close()


def test_cloud_far_from_origin(R):
    """a scene shifted by 2000 units: the FP32 band widens and more pairs go to the inline FP64 decision"""
    from ransac_jl_b200 import FittedCone, FittedCylinder, FittedPlane, FittedSphere, scenes

    sc = scenes.scene_mixed(33, 4000, noise_frac=0.004, jitter_deg=1.5, outlier_frac=0.1, counts=(1, 1, 1, 1))
    shift = np.array([2000.0, -2000.0, 2000.0])
    V = (sc.vertices.astype(np.float64) + shift).astype(np.float32)
    N = np.asarray(sc.normals, np.float32)
    pc = R.RANSACCloud(V, N, 2)
    en = np.random.default_rng(33).random(len(V)) >= 0.3
    pc.isenabled = en
    cands = []
    for s in scenes.perturbed_candidates(sc, 40, seed=33):
        if isinstance(s, FittedPlane):
            s = FittedPlane(np.asarray(s.point) + shift, s.normal)
        elif isinstance(s, FittedSphere):
            s = FittedSphere(np.asarray(s.center) + shift, s.radius, s.outwards)
        elif isinstance(s, FittedCylinder):
            a = np.asarray(s.axis)
            c = np.asarray(s.center) + shift
            s = FittedCylinder(a, c - a * float(a @ c), s.radius, s.outwards)
        else:
            s = FittedCone(np.asarray(s.apex) + shift, s.axis, s.opang, s.outwards)
        cands.append(s)
    cv, ce = _check(R, pc, cands, V.astype(np.float64), N.astype(np.float64), en)
    assert cv.sum() > 1000
    _check(R, pc, cands, V.astype(np.float64), N.astype(np.float64), en, subset=0, idx=pc.subsets[0])
    pc.close()


def test_exact_cloud_decides_on_the_unrounded_points(R):
    """an exact float64 cloud whose points sit within ~1e-8 relative of the thresholds: the inline FP64 decision
    reads the caller's float64 coordinates (through the subset's map on a subset), so the counts are the oracle's
    on the unrounded points, which a float32 cloud of the same points does not reproduce"""
    from tests.test_exact_f64_gpu import threshold_scene

    shapes, V, N = threshold_scene(R, seed=4, per_shape=600)
    sub = np.random.default_rng(4).permutation(len(V))[: len(V) // 3].astype(np.int64)
    ex = R.RANSACCloud(V, N, [sub], exact=True)
    en = np.random.default_rng(5).random(len(V)) >= 0.2
    ex.isenabled = en
    params = R.ransacparameters()
    cv, ce = _check(R, ex, shapes, V, N, en, params)
    _check(R, ex, shapes, V, N, en, params, subset=0, idx=sub)
    rd = R.RANSACCloud(V, N, [sub])  # rounds to float32 on upload
    rd.isenabled = en
    cv_rd, _ = _small(R, rd, shapes, params)
    assert (cv_rd != cv).any(), "the scene has teeth: the rounded points decide differently"
    ex.close()
    rd.close()


@pytest.mark.parametrize("ncand", [129, 4097])
def test_count_on_the_device(R, ncand):
    """the synchronisation-free form: a count below the capacity scores the first `count` candidates and leaves
    zeros behind them; a count above the capacity scores the capacity"""
    from ransac_jl_b200 import scenes

    sc, pc, P, N, en = _cloud(R, 800, 61)
    cands = scenes.perturbed_candidates(sc, (ncand + 3) // 4, seed=61)[:ncand]
    params = R.ransacparameters()
    cv, ce = _check(R, pc, cands, P, N, en, params)
    for count in (0, 1, 127, 128, ncand - 1):
        cv2, ce2 = _small(R, pc, cands, params, count=count)
        np.testing.assert_array_equal(cv2[:count], cv[:count], err_msg=f"count={count}")
        np.testing.assert_array_equal(ce2[:count], ce[:count], err_msg=f"count={count}")
        assert (cv2[count:] == 0).all() and (ce2[count:] == 0).all(), f"count={count}"
    for count in (ncand + 1, 10 * ncand, 2**40):
        cv2, ce2 = _small(R, pc, cands, params, count=count)
        np.testing.assert_array_equal(cv2, cv, err_msg=f"count={count}")
        np.testing.assert_array_equal(ce2, ce, err_msg=f"count={count}")
    # a capacity smaller than the array: only the first `cap` candidates exist for the scorer
    cv3, ce3 = _small(R, pc, cands, params, count=ncand, cap=ncand - 5)
    np.testing.assert_array_equal(cv3, cv[: ncand - 5])
    np.testing.assert_array_equal(ce3, ce[: ncand - 5])
    pc.close()
