"""User-defined shapes on the device (rsc_user.cu): counts, masks and inlier lists of NVRTC-compiled
rsc_user_compatible programs equal their NumPy twins bit for bit (tests/user_shapes.py), the extraction
behaves like a built-in one, the host loop gives the same result with a device slab as with a NumPy slab,
and built-in scoring is unaffected."""
import ctypes as C
import math
import os
import sys
from dataclasses import dataclass

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import user_shapes as U  # noqa: E402

pytestmark = pytest.mark.gpu

K = U.constants(0.3, math.radians(5))
KT = U.constants(0.05, math.radians(10))


@pytest.fixture(scope="module")
def R():
    import ransac_jl_b200 as R

    return R


def _compile(R, ctx, src):
    b = src.encode()
    tid = C.c_int32()
    ctx.check(R._lib.lib.rsc_user_shape_compile(ctx.h, b, len(b), C.byref(tid)))
    return tid.value


def _recs(R, tid, recs):
    arr = (R._lib.rsc_cand * max(len(recs), 1))()
    for i, p in enumerate(recs):
        arr[i].type = tid
        arr[i].outwards = 0
        arr[i].p[:] = [float(v) for v in p] + [0.0] * (7 - len(p))
    return arr


def _user_score(R, pc, tid, recs, k, subset, want_masks=True):
    M = pc.size if subset < 0 else len(pc.subsets[subset])
    counts = np.zeros(len(recs), np.int32)
    masks = np.zeros((len(recs), (M + 31) // 32), np.uint32) if want_masks else None
    kk = np.ascontiguousarray(k, dtype=np.float64)
    rc = R._lib.lib.rsc_user_score(pc.handle, kk.ctypes.data, len(kk), _recs(R, tid, recs), len(recs), subset, counts.ctypes.data,
                                   masks.ctypes.data if want_masks else None)
    return rc, counts, masks


def _twin_check(R, pc, V, N, tid, twin, recs, k, subset, want_masks=True):
    """device counts / masks == twin on subset `subset` (-1: whole cloud) under the cloud's enabled mask"""
    if subset >= 0:
        pc.upload_subset(subset)
    idx = np.arange(pc.size) if subset < 0 else pc.subsets[subset]
    rc, counts, masks = _user_score(R, pc, tid, recs, k, subset, want_masks)
    pc.ctx.check(rc)
    en = pc.isenabled[idx]
    P, Nn = V[idx].astype(np.float64), N[idx].astype(np.float64)
    for i, p in enumerate(recs):
        want = twin(np.asarray(p, np.float64), k, P, Nn) & en
        assert int(counts[i]) == int(want.sum()), (i, subset)
        if want_masks:
            assert np.array_equal(R.unpack_mask(masks[i], len(idx)), want), (i, subset)
    return counts


def _scene(rng, n_torus=20_000, n_slab=15_000, n_out=10_000):
    tp, tn = U.torus_points(rng, [3.0, -2.0, 1.0], [0.3, 0.2, 1.0], 6.0, 1.5, n_torus, noise=0.01)
    sp = np.c_[rng.uniform(-20, 20, (n_slab, 2)), np.full(n_slab, 7.0) + rng.normal(0, 0.02, n_slab)]
    sn = np.tile([0.0, 0.0, 1.0], (n_slab, 1)) + rng.normal(0, 0.02, (n_slab, 3))
    op = rng.uniform(-20, 20, (n_out, 3))
    on = rng.normal(size=(n_out, 3))
    V = np.r_[tp, sp, op].astype(np.float32)
    N = np.r_[tn, sn, on]
    N = (N / np.linalg.norm(N, axis=1, keepdims=True)).astype(np.float32)
    perm = rng.permutation(len(V))
    return V[perm], N[perm]


def _torus_cands(rng, C):
    out = [U.torus_record([3.0, -2.0, 1.0], [0.3, 0.2, 1.0], 6.0, 1.5)]
    while len(out) < C:
        out.append(U.torus_record([3.0, -2.0, 1.0] + rng.normal(0, 0.05, 3), np.array([0.3, 0.2, 1.0]) + rng.normal(0, 0.05, 3),
                                  6.0 + rng.normal(0, 0.05), 1.5 + rng.normal(0, 0.02)))
    return out[:C]


def _slab_cands(rng, C):
    return [[7.0]] + [[7.0 + rng.normal(0, 0.2)] for _ in range(C - 1)]


@pytest.fixture(scope="module")
def scene(R):
    rng = np.random.default_rng(5)
    V, N = _scene(rng)
    pc = R.RANSACCloud(V, N, 3)
    en = rng.random(pc.size) > 0.3
    pc.isenabled = en
    return pc, V, N


def test_score_parity_mixed_scene_whole_cloud_and_subsets(R, scene):
    pc, V, N = scene
    rng = np.random.default_rng(1)
    tt, ts = _compile(R, pc.ctx, U.TORUS_SRC), _compile(R, pc.ctx, U.SLAB_SRC)
    assert tt >= R._lib.RSC_USER_TYPE0 and ts >= R._lib.RSC_USER_TYPE0 and tt != ts
    assert _compile(R, pc.ctx, U.TORUS_SRC) == tt  # cached by source
    tor, slab = _torus_cands(rng, 40), _slab_cands(rng, 40)
    for subset in (-1, 0, 1):
        c = _twin_check(R, pc, V, N, tt, U.torus_twin, tor, KT, subset)
        assert c[0] > 0.5 * 20_000 * 0.7 / (1 if subset < 0 else 3)  # the true torus is found
        _twin_check(R, pc, V, N, ts, U.slab_twin, slab, K, subset)


@pytest.mark.parametrize("n", [1, 31, 32, 33, 511, 513, 1025, 1 << 20])
def test_score_parity_ragged_sizes(R, n):
    rng = np.random.default_rng(n)
    V, N = _scene(rng, n_torus=(n + 1) // 2, n_slab=n // 4, n_out=n - (n + 1) // 2 - n // 4)
    pc = R.RANSACCloud(V, N, 1)
    pc.isenabled = rng.random(n) > 0.3
    tt, ts = _compile(R, pc.ctx, U.TORUS_SRC), _compile(R, pc.ctx, U.SLAB_SRC)
    C_ = 7 if n >= (1 << 20) else 33
    for subset in (-1, 0):
        _twin_check(R, pc, V, N, tt, U.torus_twin, _torus_cands(rng, C_), KT, subset)
        _twin_check(R, pc, V, N, ts, U.slab_twin, _slab_cands(rng, C_), K, subset)


@pytest.mark.parametrize("C_", [1, 7, 300, 5000])
def test_score_parity_candidate_counts(R, C_):
    rng = np.random.default_rng(C_)
    V, N = _scene(rng, 3000, 2000, 1500)
    pc = R.RANSACCloud(V, N, 2)
    pc.isenabled = rng.random(pc.size) > 0.3
    tt = _compile(R, pc.ctx, U.TORUS_SRC)
    tor = _torus_cands(rng, C_)
    _twin_check(R, pc, V, N, tt, U.torus_twin, tor, KT, 0)
    _twin_check(R, pc, V, N, tt, U.torus_twin, tor, KT, -1, want_masks=C_ <= 300)


def test_score_parity_nan_parameters(R, scene):
    pc, V, N = scene
    tt, ts = _compile(R, pc.ctx, U.TORUS_SRC), _compile(R, pc.ctx, U.SLAB_SRC)
    good = U.torus_record([3.0, -2.0, 1.0], [0.3, 0.2, 1.0], 6.0, 1.5)
    tor = [list(good)]
    for j in range(7):
        p = list(good)
        p[j] = float("nan")
        tor.append(p)
    tor.append([0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 6.0])  # zero axis: r = 0, a = nan
    c = _twin_check(R, pc, V, N, tt, U.torus_twin, tor, KT, 0)
    assert c[0] > 0 and (c[1:] == 0).all()
    _twin_check(R, pc, V, N, ts, U.slab_twin, [[float("nan")], [7.0]], K, 0)
    _twin_check(R, pc, V, N, ts, U.slab_twin, [[7.0]], [float("nan"), K[1]], 0)


def _extract(R, pc, tid, rec, k, disable):
    kk = np.ascontiguousarray(k, dtype=np.float64)
    cand = _recs(R, tid, [rec])[0]
    out = np.zeros(pc.size, np.int64)
    n = C.c_int64()
    pc.ctx.check(R._lib.lib.rsc_user_refit_extract(pc.handle, kk.ctypes.data, len(kk), C.byref(cand), out.ctypes.data, C.byref(n),
                                                   int(disable)))
    return out[: n.value].copy()


def test_extraction_lists_and_disabled_bits(R):
    rng = np.random.default_rng(11)
    V, N = _scene(rng)
    pc = R.RANSACCloud(V, N, 2)
    pc.upload_subset(1)
    en0 = rng.random(pc.size) > 0.3
    pc.isenabled = en0
    tt, ts = _compile(R, pc.ctx, U.TORUS_SRC), _compile(R, pc.ctx, U.SLAB_SRC)
    P, Nn = V.astype(np.float64), N.astype(np.float64)
    trec = U.torus_record([3.0, -2.0, 1.0], [0.3, 0.2, 1.0], 6.0, 1.5)
    want_t = np.flatnonzero(U.torus_twin(np.asarray(trec), KT, P, Nn) & en0)
    got = _extract(R, pc, tt, trec, KT, disable=False)
    assert np.array_equal(got, want_t) and len(got) > 10_000
    assert np.array_equal(pc.isenabled, en0)  # disable=0 leaves the mask as it was
    got = _extract(R, pc, tt, trec, KT, disable=True)
    assert np.array_equal(got, want_t)
    en1 = en0.copy()
    en1[want_t] = False
    assert np.array_equal(pc.isenabled, en1)  # exactly those bits cleared
    # the subset copies follow the cleared bits: the user torus finds nothing left on subsets 1 and 2
    for subset in (0, 1):
        _twin_check(R, pc, V, N, tt, U.torus_twin, [trec], KT, subset)
        assert _user_score(R, pc, tt, [trec], KT, subset)[1][0] == 0
    # extract the slab; a built-in plane through it (same eps / alpha) then counts only what is left enabled
    from tests.helpers import oracle_mask, oracle_params

    plane = R.FittedPlane([0.0, 0.0, 7.0], [0.0, 0.0, 1.0])
    params = R.ransacparameters([R.FittedPlane])
    before = [int(R.score_counts(pc, [plane], j, params)[0][0]) for j in (0, 1)]
    want_s = np.flatnonzero(U.slab_twin(np.array([7.0]), K, P, Nn) & en1)
    assert np.array_equal(_extract(R, pc, ts, [7.0], K, disable=True), want_s) and len(want_s) > 5000
    en1[want_s] = False
    assert np.array_equal(pc.isenabled, en1)
    assert pc.count_enabled() == int(en1.sum())
    for j, subset in enumerate((0, 1)):
        sub = pc.subsets[subset]
        counts, masks = R.score_counts(pc, [plane], subset, params, want_masks=True)
        want = oracle_mask(plane, V[sub], N[sub], oracle_params(params), enabled=en1[sub])
        assert np.array_equal(R.unpack_mask(masks[0], len(sub)), want) and int(counts[0]) == int(want.sum())
        assert int(counts[0]) < before[j] // 10
        _twin_check(R, pc, V, N, ts, U.slab_twin, [[7.0]], K, subset)
        _twin_check(R, pc, V, N, tt, U.torus_twin, _torus_cands(np.random.default_rng(3), 5), KT, subset)


def test_host_loop_numpy_slab_equals_device_slab(R):
    from ransac_jl_b200.shapes import on_device

    NumpySlab, DeviceSlab = U.slab_classes(R)
    assert on_device(DeviceSlab) and not on_device(NumpySlab) and not on_device(R.FittedSphere)
    rng = np.random.default_rng(9)
    n_slab, n_sph, n_out = 6000, 5000, 2000
    slab = np.c_[rng.uniform(-20, 20, (n_slab, 2)), np.full(n_slab, 7.0) + rng.normal(0, 0.02, n_slab)]
    slab_n = np.tile([0.0, 0.0, 1.0], (n_slab, 1))
    d = rng.normal(size=(n_sph, 3))
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    sph, sph_n = np.array([30.0, 0, -10]) + 6.0 * d, d
    out = rng.uniform(-40, 40, (n_out, 3))
    out_n = rng.normal(size=(n_out, 3))
    out_n /= np.linalg.norm(out_n, axis=1, keepdims=True)
    V = np.r_[slab, sph, out].astype(np.float32)
    N = np.r_[slab_n, sph_n, out_n].astype(np.float32)
    perm = rng.permutation(len(V))
    V, N = V[perm], N[perm]
    pc = R.RANSACCloud(V, N, 2)
    res = {}
    for cls in (NumpySlab, DeviceSlab):
        params = R.ransacparameters([R.FittedSphere, cls], iteration={"tau": 500, "minsubsetN": 64, "itermax": 60})
        ex, _ = R.ransac(pc, params, True, seed=3)
        res[cls] = (ex, pc.isenabled.copy())
    (a, ea), (b, eb) = res[NumpySlab], res[DeviceSlab]
    kinds = [type(e.shape).__name__ for e in b]
    assert "DeviceSlab" in kinds and "FittedSphere" in kinds, kinds
    assert len(a) == len(b)
    for x, y in zip(a, b):
        assert isinstance(x.shape, R.FittedSphere) == isinstance(y.shape, R.FittedSphere)
        if isinstance(x.shape, R.FittedSphere):
            assert list(x.shape.to_cand().p) == list(y.shape.to_cand().p)
        else:
            assert x.shape.z0 == y.shape.z0
        assert np.array_equal(x.inpoints, y.inpoints)
    assert np.array_equal(ea, eb)


def test_builtin_scores_unchanged_by_user_shapes(R):
    from ransac_jl_b200 import scenes

    sc = scenes.scene_c1()
    pc = R.RANSACCloud(sc.vertices, sc.normals, 2)
    params = R.ransacparameters()
    cands = [p.shape for p in sc.primitives] + scenes.perturbed_candidates(sc, 4, seed=1)
    before = R.score_counts(pc, cands, 0, params, want_masks=True)
    tt, ts = _compile(R, pc.ctx, U.TORUS_SRC), _compile(R, pc.ctx, U.SLAB_SRC)
    rng = np.random.default_rng(2)
    V, N = sc.vertices.astype(np.float32), sc.normals.astype(np.float32)
    _twin_check(R, pc, V, N, tt, U.torus_twin, _torus_cands(rng, 9), KT, 0)
    _twin_check(R, pc, V, N, ts, U.slab_twin, _slab_cands(rng, 9), K, -1)
    after = R.score_counts(pc, cands, 0, params, want_masks=True)
    assert np.array_equal(before[0], after[0]) and np.array_equal(before[1], after[1])


def test_errors(R, scene):
    pc, V, N = scene
    L, ctx = R._lib.lib, pc.ctx
    E_ARG, E_STATE = R._lib.RSC_E_ARG, R._lib.RSC_E_STATE
    tid = C.c_int32(-7)
    b = U.BROKEN_SRC.encode()
    assert L.rsc_user_shape_compile(ctx.h, b, len(b), C.byref(tid)) == E_ARG
    msg = L.rsc_last_error(ctx.h).decode()
    assert "rsc_user_shape.cu(4): error" in msg, msg
    b = b"__device__ bool compatible(double x) { return x > 0.0; }\n"
    assert L.rsc_user_shape_compile(ctx.h, b, len(b), C.byref(tid)) == E_ARG
    # after a failed compile the context still scores built-ins
    sph = R.FittedSphere([3.0, -2.0, 1.0], 6.0, True)
    R.score_counts(pc, [sph], 0, R.ransacparameters())
    tt, ts = _compile(R, ctx, U.TORUS_SRC), _compile(R, ctx, U.SLAB_SRC)
    trec = U.torus_record([3.0, -2.0, 1.0], [0.3, 0.2, 1.0], 6.0, 1.5)
    mixed = _recs(R, tt, [trec, [7.0]])
    mixed[1].type = ts
    counts = np.zeros(2, np.int32)
    kk = np.ascontiguousarray(KT)
    assert L.rsc_user_score(pc.handle, kk.ctypes.data, 2, mixed, 2, 0, counts.ctypes.data, None) == E_ARG
    for bad in (0, 3, 99, R._lib.RSC_USER_TYPE0 + 1000):  # built-in and unknown types
        assert _user_score(R, pc, bad, [trec], KT, 0)[0] == E_ARG
    assert _user_score(R, pc, tt, [trec], [0.0] * 9, 0)[0] == E_ARG  # nk = 9
    assert _user_score(R, pc, tt, [trec], KT, 2)[0] == E_STATE  # subset 3 not uploaded
    cand = _recs(R, 99, [trec])[0]
    n = C.c_int64()
    assert L.rsc_user_refit_extract(pc.handle, kk.ctypes.data, 2, C.byref(cand), None, C.byref(n), 0) == E_ARG
    # sharded storage is refused
    sh = R.RANSACCloud(V[:4096], N[:4096], [np.zeros(0, np.int64)], shard=(0, 8192))
    assert sh.is_shard
    assert _user_score(R, sh, tt, [trec], KT, -1)[0] == E_STATE
    cand = _recs(R, tt, [trec])[0]
    assert L.rsc_user_refit_extract(sh.handle, kk.ctypes.data, 2, C.byref(cand), None, C.byref(n), 0) == E_STATE
    sh.close()
    # and the context still works
    _twin_check(R, pc, V, N, tt, U.torus_twin, [trec], KT, 0)
