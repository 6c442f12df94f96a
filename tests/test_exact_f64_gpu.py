"""Exact float64 clouds (rsc_cloud_create_f64_exact) on the device: every decision and every fit is the float64
one of the caller's UNROUNDED coordinates, bit for bit against the oracles on the same float64 arrays.  The
threshold scene puts points within ~1e-8 relative of eps and cos(alpha), where the rounding cloud
(rsc_cloud_create_f64) must and does decide differently -- so the comparisons can fail."""
import ctypes as C
import math
import os
import sys

import numpy as np
import pytest

from oracle import c_oracle as CO
from oracle import ransac_oracle as O
from tests import fp32_model as M
from tests.helpers import oracle_mask, oracle_params

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import user_fit_shapes as U  # noqa: E402

pytestmark = pytest.mark.gpu
KAPPA_IN = {0: 1.0, 1: 3.0, 2: 3.0, 3: 4.0}


@pytest.fixture(scope="module")
def R():
    import ransac_jl_b200 as R

    return R


def _unit(rng, n=None):
    v = rng.normal(size=(3,) if n is None else (n, 3))
    return v / np.linalg.norm(v, axis=-1, keepdims=True)


def _perp(a, rng, n):
    """n unit vectors perpendicular to the unit vector a"""
    v = rng.normal(size=(n, 3))
    v -= np.outer(v @ a, a)
    return v / np.linalg.norm(v, axis=1, keepdims=True)


def threshold_scene(R, seed=3, per_shape=3000, shift=0.0):
    """Shapes of every type (narrow and wide cones) and points whose float64 distance to the surface is
    eps (1 +- 1e-8) or whose normal makes an angle alpha (1 +- 1e-7) with the surface normal; plus
    clearly-inside and clearly-outside points and uniform clutter.  Nothing is float32-representable."""
    rng = np.random.default_rng(seed)
    eps, alpha = 0.3, math.radians(5)
    shapes, P, N = [], [], []
    for i in range(10):
        kind = i % 5
        outw = bool(rng.integers(2))
        c = rng.uniform(-20, 20, 3) + shift
        if kind == 0:
            nrm = _unit(rng)
            sh = R.FittedPlane(c, nrm)
            u = _perp(nrm, rng, per_shape)
            base = c + u * rng.uniform(0, 15, (per_shape, 1))
            sn = np.tile(nrm, (per_shape, 1))
        elif kind == 1:
            Rr = rng.uniform(2, 10)
            sh = R.FittedSphere(c, Rr, outw)
            d = _unit(rng, per_shape)
            base = c + Rr * d
            sn = d if outw else -d
        elif kind == 2:
            a = _unit(rng)
            Rr = rng.uniform(2, 10)
            sh = R.FittedCylinder(a, c - a * float(a @ c), Rr, outw)
            d = _perp(a, rng, per_shape)
            base = c + Rr * d + np.outer(rng.uniform(-10, 10, per_shape), a)
            sn = d if outw else -d
        else:
            a = _unit(rng)
            opang = math.radians(40.0 if kind == 3 else 150.0)  # kind 4: a wide cone (column type kConeWide)
            sh = R.FittedCone(c, a, opang, outw)
            th = opang / 2
            d = _perp(a, rng, per_shape)
            h = rng.uniform(1, 10, (per_shape, 1))
            base = c + h * a + h * math.tan(th) * d
            nv = math.cos(th) * d - math.sin(th) * a  # outward surface normal
            sn = nv if outw else -nv
        m = per_shape
        kindsel = rng.integers(4, size=m)  # 0/1: distance near eps, 2/3: angle near alpha
        tsign = np.where(rng.random(m) < 0.5, -1.0, 1.0)
        t = np.where(kindsel < 2, tsign * eps * (1 + rng.uniform(-1e-8, 1e-8, m)), rng.uniform(-0.5, 0.5, m) * eps)
        p = base + t[:, None] * sn
        ang = np.where(kindsel >= 2, alpha * (1 + rng.uniform(-1e-7, 1e-7, m)), rng.uniform(0, 0.8, m) * alpha)
        q = _perp_rows(sn, rng)
        n = np.cos(ang)[:, None] * sn + np.sin(ang)[:, None] * q
        shapes.append(sh)
        P.append(p)
        N.append(n)
    clutter = rng.uniform(-30, 30, (20_000, 3)) + shift
    P.append(clutter)
    N.append(_unit(rng, 20_000))
    V = np.concatenate(P)
    Nn = np.concatenate(N)
    perm = rng.permutation(len(V))
    return shapes, np.ascontiguousarray(V[perm]), np.ascontiguousarray(Nn[perm])


def _perp_rows(sn, rng):
    v = rng.normal(size=sn.shape)
    v -= (v * sn).sum(1, keepdims=True) * sn
    return v / np.linalg.norm(v, axis=1, keepdims=True)


def _masks_vs_oracle(R, pc, shapes, V, N, subset=-1, idx=None):
    params = R.ransacparameters()
    op = oracle_params(params)
    counts, masks = R.score_counts(pc, shapes, subset, params, want_masks=True)
    Vs, Ns = (V, N) if idx is None else (V[idx], N[idx])
    differ = 0
    for i, sh in enumerate(shapes):
        want = oracle_mask(sh, Vs, Ns, op)
        got = R.unpack_mask(masks[i], len(Vs))
        differ += int((got != want).sum())
        if pc.exact:
            np.testing.assert_array_equal(got, want, err_msg=f"candidate {i}")
            assert counts[i] == want.sum()
    return differ


@pytest.fixture(scope="module")
def tscene(R):
    shapes, V, N = threshold_scene(R)
    return shapes, V, N


def test_threshold_scene_exact_cloud_equals_oracle_and_rounding_cloud_does_not(R, tscene):
    shapes, V, N = tscene
    cands = shapes
    sub = np.random.default_rng(1).permutation(len(V))[: len(V) // 3].astype(np.int64)
    ex = R.RANSACCloud(V, N, [sub], exact=True)
    rd = R.RANSACCloud(V, N, [sub])
    assert ex.exact and not rd.exact
    assert _masks_vs_oracle(R, ex, cands, V, N) == 0
    assert _masks_vs_oracle(R, ex, cands, V, N, subset=0, idx=sub) == 0
    differ = _masks_vs_oracle(R, rd, cands, V, N)
    print(f"rounding cloud: {differ} (candidate, point) decisions differ from the oracle on the unrounded points")
    assert differ > 1000  # the scene has teeth
    op = oracle_params(R.ransacparameters())
    want = np.array([oracle_mask(s, V, N, op).sum() for s in cands])
    # device-resident candidates and masks
    import torch

    arr = R.pack_cands(cands)
    raw = np.frombuffer(bytes(arr), np.uint8)
    d_c = torch.from_numpy(raw.copy()).cuda()
    d_counts = torch.zeros(len(cands), dtype=torch.int32, device="cuda")
    words = (len(V) + 31) // 32
    d_masks = torch.zeros((len(cands), words), dtype=torch.int32, device="cuda")
    cp = R.to_c(R.ransacparameters())
    ex.ctx.check(R._lib.lib.rsc_score_dev_masks(ex.handle, C.byref(cp), C.c_void_p(d_c.data_ptr()), len(cands), -1,
                                                C.c_void_p(d_counts.data_ptr()), C.c_void_p(d_masks.data_ptr()), None))
    torch.cuda.synchronize()
    np.testing.assert_array_equal(d_counts.cpu().numpy(), want)
    mk = d_masks.cpu().numpy().view(np.uint32)
    for i, s in enumerate(cands):
        bits = np.unpackbits(mk[i].view(np.uint8), bitorder="little")[: len(V)].astype(bool)
        np.testing.assert_array_equal(bits, oracle_mask(s, V, N, op))
    # culled scorer: whole cloud (Morton copy) and subset (Morton view)
    ex.build_cells(8)
    got, _ = R.score_counts_culled(ex, cands, R.ransacparameters())
    np.testing.assert_array_equal(got, want)
    got, _ = R.score_counts_culled(ex, cands, R.ransacparameters(), 0)
    np.testing.assert_array_equal(got, [oracle_mask(s, V[sub], N[sub], op).sum() for s in cands])
    # K4: refit inlier lists (each on a fresh enabled mask)
    for s in cands:
        ex.enable_all()
        np.testing.assert_array_equal(R.refit(s, ex, R.ransacparameters()).inpoints, np.flatnonzero(oracle_mask(s, V, N, op)))
    ex.close()
    rd.close()


def test_float64_rounding_scene_on_exact_cloud_has_no_difference(R):
    """the scene of test_float64_cloud_decides_on_the_float32_roundings: differ == 0 on the exact cloud"""
    from ransac_jl_b200 import scenes

    sc = scenes.scene_mixed(61, 60_000, noise_frac=0.004, jitter_deg=2.0, outlier_frac=0.2)
    rng = np.random.default_rng(5)
    V64 = sc.vertices.astype(np.float64) + rng.uniform(-1e-6, 1e-6, sc.vertices.shape)
    N64 = sc.normals.astype(np.float64) + rng.uniform(-1e-8, 1e-8, sc.normals.shape)
    pc = R.RANSACCloud(V64, N64, [np.arange(len(V64), dtype=np.int64)], exact=True)
    cands = [p.shape for p in sc.primitives] + scenes.perturbed_candidates(sc, 6, seed=2)
    assert _masks_vs_oracle(R, pc, cands, V64, N64, subset=0, idx=np.arange(len(V64))) == 0
    pc.close()


def test_fits_on_exact_cloud_are_the_float64_fits_of_the_unrounded_points(R):
    """rsc_sample_fit and rsc_fit_batch on an exact cloud give, bit for bit, what rsc_fit_points gives for the
    unrounded coordinates of the drawn sets (and the C oracle's fits within the tolerance test_fit_gpu.py uses);
    on the rounded coordinates rsc_fit_points gives other bits, so the comparison can fail"""
    from ransac_jl_b200 import scenes
    from tests.test_fit_gpu import _compare, _sets

    sc = scenes.scene_mixed(71, 30_000)
    rng = np.random.default_rng(8)
    V = sc.vertices.astype(np.float64) + rng.uniform(-1e-6, 1e-6, sc.vertices.shape)
    N = sc.normals.astype(np.float64) + rng.uniform(-1e-7, 1e-7, sc.normals.shape)
    pc = R.RANSACCloud(V, N, 2, exact=True)
    params = R.ransacparameters()
    shapes, sets, idx = R.sample_fit(pc, params, 4242, 17, 3000)
    good = np.flatnonzero(idx[:, 0] >= 0)
    assert len(good) == 3000 and len(shapes) > 5

    def same(x, y):
        assert len(x) == len(y)
        for a, b in zip(x, y):
            ca, cb = a.to_cand(), b.to_cand()
            assert ca.type == cb.type and ca.outwards == cb.outwards and list(ca.p) == list(cb.p)

    sh2, sets2 = R.fit_points(pc, V[idx[good]], N[idx[good]], params)
    np.testing.assert_array_equal(sets, good[sets2])
    same(shapes, sh2)
    bidx = _sets(sc, 6000, 3)  # half the sets inside one primitive: fits succeed
    sh3, sets3 = R.fit_batch(pc, bidx, params)
    sh4, sets4 = R.fit_points(pc, V[bidx], N[bidx], params)
    np.testing.assert_array_equal(sets3, sets4)
    same(sh3, sh4)
    want, want_set = CO.fit_points(V[bidx], N[bidx], oracle_params(params))
    assert min(_compare(R, sh3, sets3, want, want_set)) > 30
    Vr, Nr = V.astype(np.float32).astype(np.float64), N.astype(np.float32).astype(np.float64)
    shr, _ = R.fit_points(pc, Vr[bidx], Nr[bidx], params)
    assert len(shr) != len(sh3) or sum(list(a.to_cand().p) != list(b.to_cand().p) for a, b in zip(shr, sh3)) > 100
    pc.close()


def _loop_scene(n, seed):
    from ransac_jl_b200 import scenes

    sc = scenes.scene_c1() if n is None else scenes.scene_mixed(seed, n, noise_frac=0.002, jitter_deg=1.0, outlier_frac=0.1,
                                                                  counts=(3, 1, 1, 1))
    rng = np.random.default_rng(seed)
    V = sc.vertices.astype(np.float64) + rng.uniform(-1e-6, 1e-6, sc.vertices.shape)
    N = sc.normals.astype(np.float64) + rng.uniform(-1e-6, 1e-6, sc.normals.shape)
    return V, N


@pytest.mark.parametrize("scene,loop", [("c1", "default"), ("c1", "cull_always"), ("c1", "cull_never"), ("c1", "hostwalk"),
                                        ("c1", "hostwalk_cull_always"), ("1Mi", "default"), ("1Mi", "cull_always")])
def test_ransac_on_exact_cloud_equals_c_oracle_on_unrounded_input(R, monkeypatch, scene, loop):
    from tests.test_ransac_gpu import _compare_runs

    if scene == "c1":
        V, N = _loop_scene(None, 31)
        nsub, params, seed = 2, R.ransacparameters(), 4321
    else:
        V, N = _loop_scene(1 << 20, 32)
        nsub, params, seed = 8, R.ransacparameters(iteration={"tau": 3000, "minsubsetN": 256, "itermax": 40}), 99
    cull_always, hostwalk = ("RSC_LOOP_CULL", "2"), ("RSC_LOOP_HOSTWALK", "1")
    env = {"cull_always": [cull_always], "cull_never": [("RSC_LOOP_CULL", "0")], "hostwalk": [hostwalk],
           "hostwalk_cull_always": [hostwalk, cull_always]}
    for kv in env.get(loop, []):
        monkeypatch.setenv(*kv)
    pc = R.RANSACCloud(V, N, nsub, exact=True)
    extracted, _ = R.ransac(pc, params, True, seed=seed)
    want, en, _ = CO.ransac(V, N, pc.subsets[0], oracle_params(params), seed)
    assert len(extracted) == len(want) >= 3
    for got, w in zip(extracted, want):
        c = got.shape.to_cand()
        assert c.type == w[0] and (c.type == 0 or bool(c.outwards) == w[1])
        # (device and oracle fits agree to rounding, as in test_ransac_gpu.py; the inlier lists exactly)
        np.testing.assert_allclose(np.array(c.p[:]), w[2], rtol=1e-5, atol=1e-5 * max(1.0, np.abs(w[2]).max()))
        np.testing.assert_array_equal(got.inpoints, w[3])
    np.testing.assert_array_equal(pc.isenabled, en)
    pc.close()


def test_representable_data_gives_the_float32_cloud_results(R):
    from ransac_jl_b200 import scenes

    sc = scenes.scene_c1()
    V32, N32 = sc.vertices.astype(np.float32), sc.normals.astype(np.float32)
    a = R.RANSACCloud(V32, N32, 2)
    b = R.RANSACCloud(V32.astype(np.float64), N32.astype(np.float64), [s.copy() for s in a.subsets], exact=True)
    cands = [p.shape for p in sc.primitives] + scenes.perturbed_candidates(sc, 8, seed=3)
    params = R.ransacparameters()
    for sub in (-1, 0):
        ca, ma = R.score_counts(a, cands, sub, params, want_masks=True)
        cb, mb = R.score_counts(b, cands, sub, params, want_masks=True)
        np.testing.assert_array_equal(ca, cb)
        np.testing.assert_array_equal(ma, mb)
    ea, _ = R.ransac(a, params, True, seed=7)
    eb, _ = R.ransac(b, params, True, seed=7)
    assert len(ea) == len(eb) >= 3
    for x, y in zip(ea, eb):
        assert list(x.shape.to_cand().p) == list(y.shape.to_cand().p)
        np.testing.assert_array_equal(x.inpoints, y.inpoints)
    a.close()
    b.close()


def test_refusals(R, tscene):
    _, V, N = tscene
    lib = R._lib.lib
    pc = R.RANSACCloud(V, N, 2, exact=True)
    V32, N32 = V.astype(np.float32), N.astype(np.float32)
    cases = {
        "cloud_update": lambda: lib.rsc_cloud_update(pc.handle, V32.ctypes.data, N32.ctypes.data, len(V)),
        "set_range": lambda: lib.rsc_cloud_set_range(pc.handle, 0, 2048),
    }
    for name, call in cases.items():
        assert call() == -5, name
        assert b"exact" in lib.rsc_last_error(pc.ctx.h), name
    params = R.ransacparameters()
    with pytest.raises(R._lib.RscError, match="exact"):
        R.lsq_refit(R.FittedPlane([0, 0, 0], [0, 0, 1]), pc, params)
    with pytest.raises(R._lib.RscError, match="exact"):
        R.bitmap_filter(R.FittedPlane([0, 0, 0], [0, 0, 1]), pc, np.arange(10, dtype=np.int64), 0.1)
    pc.build_cells(6)
    for kw in ({"progressive": True}, {"lsq": True}, {"sampler": "octree"}, {"bitmap": (0.1, False)}):
        with pytest.raises(R._lib.RscError, match="exact"):
            R.ransac(pc, params, True, seed=1, **kw)
    with pytest.raises(R._lib.RscError, match="exact"):
        R.sample_fit_cells(pc, params, 1, 0, 16, np.ones(6) / 6)
    with pytest.raises(ValueError, match="shard"):
        R.RANSACCloud(V, N, 1, exact=True, shard=(0, 2 * len(V)))
    pc.close()


@pytest.mark.parametrize("offset", [0.0, 2000.0], ids=["around_origin", "far_from_origin"])
def test_on_device_band_audit_against_unrounded_margins(R, offset):
    """rsc_debug_margins on an exact cloud returns the widened bands; the FP32 margins of the rounded points stay
    within half of them of the float64 margins of the unrounded points, over >= 1e8 pairs"""
    from ransac_jl_b200 import scenes
    from tests.test_guard_band_gpu import _cands

    rng = np.random.default_rng(13)
    npts = 1 << 20
    sc = scenes.scene_mixed(22, npts, noise_frac=0.01, jitter_deg=3.0, outlier_frac=0.3)
    V = sc.vertices.astype(np.float64) + rng.uniform(-1e-5, 1e-5, sc.vertices.shape)
    Nn = sc.normals.astype(np.float64) + rng.uniform(-1e-7, 1e-7, sc.normals.shape)
    cands = _cands(rng, sc, 20)
    if offset:
        V = V + offset
        moved = []
        for s in cands:
            c = s.to_cand()
            p = list(c.p)
            if c.type in (0, 1, 3):
                p[0:3] = [x + offset for x in p[0:3]]
            else:
                ctr = np.array(p[3:6]) + offset
                a = np.array(p[0:3])
                p[3:6] = list(ctr - a * float(a @ ctr))
            moved.append(R.from_cand(R._lib.rsc_cand(c.type, c.outwards, (C.c_double * 7)(*p))))
        cands = moved
    pc = R.RANSACCloud(V, Nn, [np.zeros(0, np.int64)], exact=True)
    Cn = len(cands)
    assert Cn * npts >= 1e8
    arr = R.pack_cands(cands)
    cp = R.to_c(R.ransacparameters())
    margins = np.zeros((Cn, npts), np.float32)
    bands = np.zeros(Cn, np.float32)
    cols = np.zeros(Cn, np.int32)
    diffs = C.c_int64()
    pc.ctx.check(R._lib.lib.rsc_debug_margins(pc.handle, C.byref(cp), arr, Cn, 0, npts, margins.ctypes.data, bands.ctypes.data,
                                              cols.ctypes.data, C.byref(diffs)))
    assert diffs.value == 0
    p32, n32 = V.astype(np.float32).astype(np.float64), Nn.astype(np.float32).astype(np.float64)
    pmax = float(np.float32(np.sqrt(np.float32((p32 ** 2).sum(1).max()))) * np.float32(1.000001))
    nmax = float(np.float32(np.sqrt(np.float32((n32 ** 2).sum(1).max()))) * np.float32(1.000001))
    eps, cosa = 0.3, math.cos(math.radians(5))
    worst = {}
    for i, s in enumerate(cands):
        c = s.to_cand()
        _, band, scale = M.record(c.type, bool(c.outwards), list(c.p), pmax, nmax, eps, cosa)
        wide = band * (M.KAPPA[c.type] + KAPPA_IN[c.type]) / M.KAPPA[c.type]
        assert bands[i] == pytest.approx(wide, rel=1e-5), "the device's band is not (kappa + kappa_in) * 2^-24 * L"
        m64 = M.margin64(c.type, bool(c.outwards), list(c.p), V, Nn, eps, cosa) * scale
        m32 = margins[i].astype(np.float64)
        ok = np.isfinite(m64) & np.isfinite(m32)
        ratio = float(np.abs(m32[ok] - m64[ok]).max() / bands[i])
        worst[int(cols[i])] = max(worst.get(int(cols[i]), 0.0), ratio)
        assert ratio < 0.5, (i, c.type, ratio)
    print(f"exact cloud, offset {offset}: {Cn * npts:.3g} pairs; worst |m32 - m64(unrounded)| / band: "
          + ", ".join(f"{k}: {v:.3f}" for k, v in sorted(worst.items())))
    pc.close()


def test_user_shapes_on_exact_cloud_match_numpy_twins_on_unrounded_input(R):
    (NS, NZ), _, (DS, DZ) = U.shape_classes(R)
    rng = np.random.default_rng(17)
    V, N = U.mixed_scene(rng, 120_000)
    V = V.astype(np.float64) + rng.uniform(-1e-6, 1e-6, V.shape)
    N = N.astype(np.float64) + rng.uniform(-1e-7, 1e-7, N.shape)
    pc = R.RANSACCloud(V, N, 3, exact=True)
    params = R.ransacparameters([R.FittedPlane, DS, DZ], iteration={"tau": 400, "minsubsetN": 128, "itermax": 400})
    params["slab"] = {"eps": 0.3, "alpha": math.radians(5), "tol": 0.1}
    params["zcyl"] = {"eps": 0.05, "alpha": math.radians(10)}
    ks, kz = U.slab_constants(), U.zcyl_constants()
    slabs = [DS.from_device_record([z], 0) for z in rng.uniform(-5, 5, 24)]
    zcyls = [DZ.from_device_record([x, y, r], 0) for x, y, r in zip(rng.uniform(-5, 5, 24), rng.uniform(-5, 5, 24), rng.uniform(1, 6, 24))]
    for cands, twin, k in ((slabs, U.slab_twin, ks), (zcyls, U.zcyl_twin, kz)):
        counts, masks = R.user_score_counts(pc, cands, -1, params, want_masks=True)
        for i, s in enumerate(cands):
            want = twin(s.device_record()[0], k, V, N)
            np.testing.assert_array_equal(R.unpack_mask(masks[i], len(V)), want)
            assert counts[i] == want.sum()
        for s in cands[:6]:
            pc.enable_all()
            np.testing.assert_array_equal(R.refit(s, pc, params).inpoints, np.flatnonzero(twin(s.device_record()[0], k, V, N)))
    from tests.test_user_fit_gpu import _compare_loops

    def unrounded_fit(base):  # the NumPy twins of user_fit_shapes.py fit on float32 roundings; these on the points as given
        class T(base):
            @classmethod
            def fit(cls, p, n, pc, params):
                r = cls.FIT_TWIN(np.asarray(p, np.float64), np.asarray(n, np.float64), cls.device_constants(params))
                return None if r is None else cls.from_device_record(r, False)

        T.__name__ = T.__qualname__ = base.__name__
        return T

    a = _compare_loops(R, pc, [R.FittedPlane, DS, DZ], [R.FittedPlane, unrounded_fit(NS), unrounded_fit(NZ)])
    assert len(a) >= 3
    pc.close()
