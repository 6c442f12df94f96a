"""User-defined shapes inside the sampler and the device loop: rsc_sample_fit_user draws rsc_sample_fit's sets and
returns its built-in candidates plus the user fits (equal to their Python twins bit for bit) in (set, position)
order; rsc_ransac_run_user gives what an independent host plug-in loop gives; with built-ins only it is
rsc_ransac_run."""
import ctypes as C
import math
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import user_fit_shapes as U  # noqa: E402
from ransac_jl_b200.shapes import SHAPE_KIND  # noqa: E402

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def R():
    import ransac_jl_b200 as R

    return R


@pytest.fixture(scope="module")
def classes(R):
    return U.shape_classes(R)


def _params(R, types, plane=None, **it):
    p = R.ransacparameters(list(types), iteration=dict({"tau": 400, "minsubsetN": 128, "itermax": 400}, **it))
    if plane:
        p["plane"] = dict(p.get("plane", {}), **plane)
    p.setdefault("slab", {"eps": 0.3, "alpha": math.radians(5), "tol": 0.1})
    p.setdefault("zcyl", {"eps": 0.05, "alpha": math.radians(10)})
    return p


def _raw_sample(R, pc, params, types, seed, set0, S):
    from ransac_jl_b200.fitting import _builtin_params, fit_order
    from ransac_jl_b200.params import to_c

    cp = to_c(_builtin_params(params))
    slots, _ = fit_order(pc, types, params)
    cap = max(S * len(types), 1)
    out = (R._lib.rsc_cand * cap)()
    out_set = np.zeros(cap, np.int32)
    idx = np.zeros((S, cp.drawN), np.int64)
    n = C.c_int32()
    pc.ctx.check(R._lib.lib.rsc_sample_fit_user(pc.handle, C.byref(cp), slots, len(types), seed, set0, S, out, out_set.ctypes.data,
                                                idx.ctypes.data, C.byref(n)))
    return [out[i] for i in range(n.value)], out_set[: n.value].copy(), idx


@pytest.fixture(scope="module")
def scene(R):
    rng = np.random.default_rng(21)
    V, N = U.mixed_scene(rng, 60_000)
    pc = R.RANSACCloud(V, N, 3)
    pc.isenabled = rng.random(pc.size) > 0.3
    return pc, V, N


@pytest.mark.parametrize("drawN", [3, 5])
@pytest.mark.parametrize("order", ["mixed", "user", "empty"])
def test_sample_fit_user_parity(R, classes, scene, drawN, order):
    pc, V, N = scene
    (_, _), (_, _), (DS, DZ) = classes
    types = {"mixed": [R.FittedPlane, DS, R.FittedSphere, DZ], "user": [DZ, DS], "empty": []}[order]
    params = _params(R, [R.FittedPlane, R.FittedSphere, DS, DZ], drawN=drawN)
    S, seed, set0 = 4096, 77, 1000
    got, sets, idx = _raw_sample(R, pc, params, types, seed, set0, S)
    bt = [t for t in types if t in SHAPE_KIND] or [R.FittedPlane]
    bparams = dict(params, iteration=dict(params["iteration"], shape_types=bt))
    from ransac_jl_b200.params import to_c

    cp = to_c(bparams)
    ref = (R._lib.rsc_cand * (S * len(bt)))()
    ref_set = np.zeros(S * len(bt), np.int32)
    ref_idx = np.zeros((S, drawN), np.int64)
    n = C.c_int32()
    pc.ctx.check(R._lib.lib.rsc_sample_fit(pc.handle, C.byref(cp), seed, set0, S, ref, ref_set.ctypes.data, ref_idx.ctypes.data, C.byref(n)))
    assert np.array_equal(idx, ref_idx)  # the same Philox sets whatever the order
    if not types:
        assert got == [] and (idx[:, 0] >= 0).sum() > S // 2
        return
    pos = {}
    for i, t in enumerate(types):
        pos[t if t in SHAPE_KIND else pc.ctx.user_type(t)] = i
    kind = {R._lib.RSC_PLANE: R.FittedPlane, R._lib.RSC_SPHERE: R.FittedSphere}
    keys = [(int(s), pos[kind.get(c.type, c.type)]) for c, s in zip(got, sets)]
    assert keys == sorted(keys) and len(set(keys)) == len(keys)  # (set, position in the order)
    b_got = [bytes(c) for c in got if c.type < R._lib.RSC_NTYPES]
    if any(t in SHAPE_KIND for t in types):
        assert b_got == [bytes(ref[i]) for i in range(n.value)]  # built-ins bit for bit
    Vd, Nd = V.astype(np.float64), N.astype(np.float64)
    for t, twin in ((DS, U.slab_fit_twin), (DZ, U.zcyl_fit_twin)):
        if t not in types:
            continue
        tid = pc.ctx.user_type(t)
        k = t.device_constants(params)
        mine = {int(s): c for c, s in zip(got, sets) if c.type == tid}
        want = {}
        for s_ in range(S):
            if idx[s_, 0] < 0:
                continue
            r = twin(Vd[idx[s_]], Nd[idx[s_]], k)
            if r is not None:
                want[s_] = r
        assert sorted(mine) == sorted(want), (t.__name__, len(mine), len(want))
        if drawN == 3:  # (five points on one small cylinder are rare draws)
            assert len(want) > 0, t.__name__
        for s_, r in want.items():
            c = mine[s_]
            assert c.outwards == 0 and list(c.p) == list(r) + [0.0] * (7 - len(r)), (t.__name__, s_)


def _rec(R, shape):
    if type(shape) in SHAPE_KIND:
        return (type(shape).__name__, list(shape.to_cand().p), shape.to_cand().outwards)
    p, o = shape.device_record()
    return (type(shape).__name__.replace("Numpy", "").replace("Scored", "").replace("Device", ""), [float(v) for v in p], int(o))


def _compare_loops(R, pc, dev_types, host_types, seed=3, **it):
    from ransac_jl_b200.iterations import _ransac_device, _ransac_host

    pd = _params(R, dev_types, **it)
    pc.enable_all()
    a, _ = _ransac_device(pc, pd, seed, order=dev_types)
    ea = pc.isenabled.copy()
    ph = _params(R, host_types, **it)
    pc.enable_all()
    b, _ = _ransac_host(pc, ph, seed)
    eb = pc.isenabled.copy()
    assert [_rec(R, x.shape) for x in a] == [_rec(R, y.shape) for y in b]
    for x, y in zip(a, b):
        assert np.array_equal(x.inpoints, y.inpoints)
    assert np.array_equal(ea, eb)
    return a


def test_device_loop_equals_host_plugin_loop_mixed(R, classes):
    (NS, NZ), _, (DS, DZ) = classes
    rng = np.random.default_rng(5)
    V, N = U.mixed_scene(rng, 200_000)
    pc = R.RANSACCloud(V, N, 3)
    a = _compare_loops(R, pc, [R.FittedPlane, DS, R.FittedSphere, DZ], [R.FittedPlane, NS, R.FittedSphere, NZ])
    kinds = {type(x.shape).__name__ for x in a}
    assert {"DeviceZCyl", "FittedPlane", "FittedSphere"} <= kinds, kinds  # (planes come first and take the slabs)


def test_device_loop_equals_host_plugin_loop_user_only(R, classes):
    (NS, NZ), _, (DS, DZ) = classes
    rng = np.random.default_rng(6)
    V, N = U.mixed_scene(rng, 120_000)
    pc = R.RANSACCloud(V, N, 2)
    a = _compare_loops(R, pc, [DZ, DS], [NZ, NS])
    assert len(a) >= 3


def test_device_loop_equals_host_plugin_loop_slab_and_plane_on_the_same_sets(R, classes):
    (NS, _), _, (DS, _) = classes
    rng = np.random.default_rng(8)
    parts = [U.slab_points(rng, 7.0, 20.0, 30_000, noise=0.002), U.slab_points(rng, -3.0, 15.0, 20_000, noise=0.002)]
    out = rng.uniform(-20, 20, (10_000, 3))
    on = rng.normal(size=(10_000, 3))
    V = np.concatenate([p for p, _ in parts] + [out]).astype(np.float32)
    N = np.concatenate([q for _, q in parts] + [on / np.linalg.norm(on, axis=1, keepdims=True)]).astype(np.float32)
    pc = R.RANSACCloud(V, N, 2)
    for dev, host in (([R.FittedPlane, DS], [R.FittedPlane, NS]), ([DS, R.FittedPlane], [NS, R.FittedPlane])):
        _compare_loops(R, pc, dev, host, plane={"eps": 0.3, "alpha": math.radians(5)})


def test_device_loop_equals_host_loop_one_million_points(R, classes):
    _, (SS, SZ), (DS, DZ) = classes
    rng = np.random.default_rng(9)
    V, N = U.mixed_scene(rng, 1_000_000)
    pc = R.RANSACCloud(V, N, 3)
    a = _compare_loops(R, pc, [R.FittedPlane, DS, R.FittedSphere, DZ], [R.FittedPlane, SS, R.FittedSphere, SZ], tau=2000)
    assert len(a) >= 4


@pytest.fixture(scope="module")
def inv_scene(R):
    rng = np.random.default_rng(12)
    V, N = U.mixed_scene(rng, 150_000)
    return R.RANSACCloud(V, N, 3)


def _run(R, pc, types, seed=4):
    from ransac_jl_b200.iterations import _ransac_device

    pc.enable_all()
    ex, _ = _ransac_device(pc, _params(R, types), seed, order=types)
    return [(_rec(R, e.shape), e.inpoints.copy()) for e in ex], pc.isenabled.copy(), pc.last_run_iterations


@pytest.mark.parametrize("env", [{"RSC_BATCH": "1"}, {"RSC_NO_SMALL": "1"}, {"RSC_SMALL_CAP": "1"}])
def test_results_do_not_depend_on_the_batching_or_scorer(R, classes, inv_scene, env, monkeypatch):
    _, _, (DS, DZ) = classes
    types = [R.FittedPlane, DS, R.FittedSphere, R.FittedCylinder, DZ]
    base = _run(R, inv_scene, types)
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    other = _run(R, inv_scene, types)
    assert [s for s, _ in base[0]] == [s for s, _ in other[0]]
    assert all(np.array_equal(x, y) for (_, x), (_, y) in zip(base[0], other[0]))
    assert np.array_equal(base[1], other[1]) and base[2] == other[2] and len(base[0]) >= 4


@pytest.mark.parametrize("which", ["c1", "noisy"])
def test_builtin_only_order_equals_ransac_run(R, which):
    from ransac_jl_b200 import scenes
    from ransac_jl_b200.iterations import _ransac_device

    types = [R.FittedPlane, R.FittedCone, R.FittedCylinder, R.FittedSphere]
    if which == "c1":
        sc, params = scenes.scene_c1(), R.ransacparameters(types)
    else:  # minsubsetN 96: segment bounds from seg_bounds_kernel
        sc = scenes.scene_mixed(81, 20_000, noise_frac=0.002, jitter_deg=1.0, outlier_frac=0.1, counts=(3, 1, 1, 1))
        params = R.ransacparameters(types, iteration={"tau": 200, "minsubsetN": 96, "itermax": 40})
    pc = R.RANSACCloud(sc.vertices, sc.normals, 3)
    res = []
    for order in (None, types):
        pc.enable_all()
        ex, _ = _ransac_device(pc, params, 11, order=order)
        res.append(([(bytes(e.shape.to_cand()), e.inpoints.copy()) for e in ex], pc.isenabled.copy(), pc.last_run_iterations,
                    pc.last_run_batches))
    (a, ea, ia, ba), (b, eb, ib, bb) = res
    assert [x for x, _ in a] == [y for y, _ in b] and len(a) >= 2
    assert all(np.array_equal(x, y) for (_, x), (_, y) in zip(a, b))
    assert np.array_equal(ea, eb) and ia == ib and ba == bb


def test_errors(R, classes, scene):
    pc, V, N = scene
    (NS, _), (SS, _), (DS, DZ) = classes
    L = R._lib.lib
    E_ARG, E_STATE = R._lib.RSC_E_ARG, R._lib.RSC_E_STATE
    from ransac_jl_b200.params import to_c

    params = _params(R, [R.FittedPlane, DS])
    cp = to_c(dict(params, iteration=dict(params["iteration"], shape_types=[R.FittedPlane])))
    ts = pc.ctx.user_type(DS)
    t_nofit = pc.ctx.user_type(SS)  # compatibility source only

    def order(types):
        arr = (R._lib.rsc_shape_slot * max(len(types), 1))()
        for i, t in enumerate(types):
            arr[i].type = t
            arr[i].nk = 3 if t >= R._lib.RSC_USER_TYPE0 else 0
            arr[i].k[:3] = U.slab_constants()
        return arr

    def sample(types, cloud=pc):
        out = (R._lib.rsc_cand * 1024)()
        n = C.c_int32()
        return L.rsc_sample_fit_user(cloud.handle, C.byref(cp), order(types), len(types), 1, 0, 64, out, None, None, C.byref(n))

    def run(types, cloud=pc, flags=0):
        c2 = to_c(dict(params, iteration=dict(params["iteration"], shape_types=[R.FittedPlane])))
        c2.compat_flags |= flags
        h = C.c_void_p()
        rc = L.rsc_ransac_run_user(cloud.handle, C.byref(c2), order(types), len(types), 1, C.byref(h))
        if rc == 0:
            L.rsc_run_destroy(h)
        return rc

    assert sample([0, ts]) == 0
    for bad in ([0, t_nofit], [ts, 99], [ts, R._lib.RSC_USER_TYPE0 + 500], [0, 0], [ts, 1, ts], list(range(4)) + [ts] * 5):
        assert sample(bad) == E_ARG, bad
        assert run(bad) == E_ARG, bad
    assert sample([0, t_nofit]) == E_ARG and "no rsc_user_fit" in L.rsc_last_error(pc.ctx.h).decode()
    for flag in (R._lib.RSC_SAMPLER_OCTREE, R._lib.RSC_SCORE_PROGRESSIVE, R._lib.RSC_REFIT_LSQ, R._lib.RSC_EXTRACT_BITMAP):
        assert run([0, ts], flags=flag) == E_STATE
    os.environ["RSC_LOOP_HOSTWALK"] = "1"
    try:
        assert run([0, ts]) == E_STATE
    finally:
        del os.environ["RSC_LOOP_HOSTWALK"]
    sh = R.RANSACCloud(V[:4096], N[:4096], [np.zeros(0, np.int64)], shard=(0, 8192))
    tsh = sh.ctx.user_type(DS)
    assert run([0, tsh], cloud=sh) == E_STATE and sample([0, tsh], cloud=sh) == E_STATE
    sh.close()
    rg = R.RANSACCloud(V[:8192], N[:8192], 1)
    assert L.rsc_cloud_set_range(rg.handle, 0, 4096) == 0
    assert run([0, rg.ctx.user_type(DS)], cloud=rg) == E_STATE
    # the public routing: an extension switch keeps the host loop, which still fits DeviceSlab on the device
    pc.enable_all()
    ex, _ = R.ransac(pc, _params(R, [R.FittedPlane, DS], itermax=50), True, seed=2, lsq=True)
    assert all(type(e.shape) in (R.FittedPlane, DS) for e in ex)
    pc.enable_all()
    assert run([0, ts]) == 0
