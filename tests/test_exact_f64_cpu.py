"""CPU checks of exact float64 clouds (rsc_cloud_create_f64_exact): the device evaluates the float32
ROUNDINGS of the caller's float64 points in FP32 and decides in FP64 on the unrounded ones, so

  * the float32 model of the kernel arithmetic on fl32(p), fl32(n) must stay within half the WIDENED guard
    band (kappa + kappa_in, rsc_eval.cuh) of the float64 margin of the unrounded p, n;
  * the culling criterion, evaluated on tile spheres of the rounded points, must never skip a tile that holds
    a compatible unrounded point;
  * the new entry points are declared where every binding looks for them."""
import math
import os
import re

import numpy as np
import pytest

from oracle import ransac_oracle as O
from tests import fp32_model as M
from tests.test_cull_model import TILES, check_no_false_culls

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KAPPA_IN = {0: 1.0, 1: 3.0, 2: 3.0, 3: 4.0}  # must match rsc::kappa_in()


def unrounded_case(seed=12345, n=4000, shift=0.0):
    """adversarial_case-like inputs WITHOUT the final float32 rounding: every shape type, wide / flat cones,
    non-unit axes and normals, huge and tiny radii; coordinates carry bits below float32 resolution."""
    rng = np.random.default_rng(seed)
    P = rng.normal(size=(n, 3)) * rng.choice([0.1, 1.0, 30.0], size=(n, 1)) + shift
    N = rng.normal(size=(n, 3))
    N /= np.linalg.norm(N, axis=1, keepdims=True)
    N[:50] *= rng.uniform(0.2, 3.0, (50, 1))
    shapes = []
    for i in range(160):
        kind = i % 4
        a = rng.normal(size=3)
        if i % 5:
            a /= np.linalg.norm(a)
        q = P[rng.integers(n)] + rng.normal(size=3) * rng.choice([0.0, 0.05, 1.0])
        outw = bool(rng.integers(2))
        if kind == 0:
            p7 = [*q, *a, 0.0]
        elif kind == 1:
            p7 = [*q, float(rng.choice([1e-3, 0.5, 3.0, 200.0])), 0, 0, 0]
        elif kind == 2:
            p7 = [*a, *q, float(rng.choice([1e-3, 0.5, 3.0, 200.0]))]
        else:
            p7 = [*q, *a, math.radians(float(rng.choice([1.0, 20.0, 90.0, 121.0, 150.0, 179.0, 200.0, 300.0])))]
        shapes.append((kind, outw, [float(x) for x in p7]))
    assert (P.astype(np.float32).astype(np.float64) != P).mean() > 0.99  # really not float32-representable
    return shapes, P, N


def _bounds(P, N):
    """pmax / nmax as the device computes them: from the float32 values, times 1.000001"""
    p32, n32 = P.astype(np.float32).astype(np.float64), N.astype(np.float32).astype(np.float64)
    return float(np.sqrt((p32 ** 2).sum(1)).max()) * 1.000001, float(np.sqrt((n32 ** 2).sum(1)).max()) * 1.000001


@pytest.mark.parametrize("shift", [0.0, 2000.0])
def test_fp32_model_of_rounded_points_within_widened_band_of_unrounded_margin(shift):
    shapes, P, N = unrounded_case(shift=shift)
    pmax, nmax = _bounds(P, N)
    eps, cosa = 0.3, math.cos(math.radians(5))
    P32, N32 = P.astype(np.float32), N.astype(np.float32)
    worst, worst_plain = {}, {}
    for kind, outw, p in shapes:
        if kind == 3 and math.cos(p[6] / 2) < 0.5 and not math.sin(p[6] / 2) >= 1 / 16:
            continue  # needle cone: infinite band, every pair is decided in FP64
        r, band, scale = M.record(kind, outw, p, pmax, nmax, eps, cosa)
        wide = band * (M.KAPPA[kind] + KAPPA_IN[kind]) / M.KAPPA[kind]
        with np.errstate(all="ignore"):
            m32 = M.margin32(kind, r, P32, N32, eps, cosa).astype(np.float64)
            m64 = M.margin64(kind, outw, p, P, N, eps, cosa) * scale
        ok = np.isfinite(m32) & np.isfinite(m64)
        col = kind if not (kind == 3 and len(r) == 11) else 4
        worst[col] = max(worst.get(col, 0.0), float((np.abs(m32 - m64)[ok] / wide).max()))
        worst_plain[col] = max(worst_plain.get(col, 0.0), float((np.abs(m32 - m64)[ok] / band).max()))
    print("max |m32(rounded) - m64(unrounded)| / widened band per column type:", worst)
    print("... / band of a rounding cloud:", worst_plain)
    assert set(worst) == {0, 1, 2, 3, 4}  # every column type, wide cones included
    for col, ratio in worst.items():
        assert ratio < 0.5, (col, ratio)


@pytest.mark.parametrize("shift", [0.0, 2000.0])
def test_culling_never_skips_a_tile_with_a_compatible_unrounded_point(shift):
    """tile spheres come from the float32 roundings (what the device stores), compatibility from the oracle on
    the unrounded points; the model uses the narrower band of a rounding cloud, the stricter case"""
    shapes, V, N = unrounded_case(seed=7, n=3000, shift=shift)
    oshapes = [O.shape_from_params7(k, o, p) for k, o, p in shapes]
    for tile in TILES:
        culled, total = check_no_false_culls(oshapes, V, N, O.default_parameters(), 6, tile)
        assert culled > 0 or tile == 4096


def test_exact_entry_points_are_declared_everywhere():
    hdr = open(os.path.join(ROOT, "include", "rsc.h")).read()
    assert re.search(r"int32_t rsc_cloud_create_f64_exact\(rsc_ctx\* ctx, const double\* xyz, const double\* nrm, int64_t n, rsc_cloud\*\* out\);", hdr)
    assert "int32_t rsc_cloud_is_exact(const rsc_cloud* cloud);" in hdr
    from ransac_jl_b200 import _lib

    for name in ("rsc_cloud_create_f64_exact", "rsc_cloud_is_exact"):
        assert name in _lib.SIGNATURES
    jl = open(os.path.join(ROOT, "julia", "RANSACB200", "src", "RANSACB200.jl")).read()
    assert "fn(:rsc_cloud_create_f64_exact)" in jl and "exact::Bool=false" in jl


def test_exact_symbols_are_exported_by_the_library():
    so = os.path.join(ROOT, "ransac.jl_b200", "libransac_b200.so")
    if not os.path.exists(so):
        pytest.skip("library not built")
    import ctypes

    lib = ctypes.CDLL(so)
    for name in ("rsc_cloud_create_f64_exact", "rsc_cloud_is_exact"):
        assert hasattr(lib, name)
    lib.rsc_cloud_is_exact.restype = ctypes.c_int32
    assert lib.rsc_cloud_is_exact(None) == 0


def test_exact_with_shard_is_refused_before_any_device_work():
    import ransac_jl_b200 as R

    V = np.zeros((4, 3))
    with pytest.raises(ValueError, match="shard"):
        R.RANSACCloud(V, V, 1, exact=True, shard=(0, 8))
