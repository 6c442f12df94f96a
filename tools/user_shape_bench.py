"""Throughput of user-defined shapes on the device (rsc_user.cu); prints one JSON line.

  torus    rsc_user_score: 4096 torus candidates (tests/user_shapes.py, float64, NVRTC-compiled) x 16 Mi points, whole-
           cloud counts; kernel time from the library's CUDA events (rsc_stats.score_ms) over --steps calls after
           --warmup; for context the built-in dense K2 on 4096 cylinders over the same cloud (FP32 with a float64
           guard band), and the NumPy twin of the torus test on a slice (a CPU rate, this host)
  loop     ransac() on the plug-in scene of tests/test_plugin_gpu.py (z-slab + built-in sphere) with the slab in
           NumPy and with the slab on the device; seconds of each, results asserted identical

python -m tools.user_shape_bench [--points 16777216] [--cands 4096] [--steps 10] [--warmup 2] [--out FILE]
"""
from __future__ import annotations

import argparse
import json
import math
import subprocess
import sys
import time

import numpy as np


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                       text=True, check=True).stdout.strip().splitlines()[0]
    name, power, clock = [s.strip() for s in q.split(",")]
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def torus_scene(rng, n):
    from tests import user_shapes as U

    per = n // 8
    V, N = [], []
    for i in range(6):
        c = rng.uniform(-40, 40, 3)
        a = rng.normal(size=3)
        p, q = U.torus_points(rng, c, a, rng.uniform(4, 10), rng.uniform(0.5, 2.0), per, noise=0.01)
        V.append(p)
        N.append(q)
    m = n - 6 * per
    V.append(rng.uniform(-50, 50, (m, 3)))
    q = rng.normal(size=(m, 3))
    N.append(q / np.linalg.norm(q, axis=1, keepdims=True))
    return np.concatenate(V).astype(np.float32), np.concatenate(N).astype(np.float32)


def timed(fn, ctx, steps, warmup):
    for _ in range(warmup):
        fn()
    ms, t0 = [], time.perf_counter()
    for _ in range(steps):
        fn()
        ms.append(ctx.stats().score_ms)
    return ms, time.perf_counter() - t0


def bench_torus(R, args):
    import ctypes as C

    from tests import user_shapes as U

    rng = np.random.default_rng(7)
    V, N = torus_scene(rng, args.points)
    pc = R.RANSACCloud(V, N, 1)
    ctx = pc.ctx
    src = U.TORUS_SRC.encode()
    tid = C.c_int32()
    t0 = time.perf_counter()
    ctx.check(R._lib.lib.rsc_user_shape_compile(ctx.h, src, len(src), C.byref(tid)))
    compile_s = time.perf_counter() - t0
    recs = [U.torus_record(rng.uniform(-40, 40, 3), rng.normal(size=3), rng.uniform(4, 10), rng.uniform(0.5, 2.0))
            for _ in range(args.cands)]
    arr = (R._lib.rsc_cand * args.cands)()
    for i, p in enumerate(recs):
        arr[i].type = tid.value
        arr[i].p[:] = p
    k = np.array(U.constants(0.05, math.radians(10)))
    counts = np.zeros(args.cands, np.int32)

    def user():
        ctx.check(R._lib.lib.rsc_user_score(pc.handle, k.ctypes.data, 2, arr, args.cands, -1, counts.ctypes.data, None))

    ms_u, wall_u = timed(user, ctx, args.steps, args.warmup)
    pairs = args.cands * args.points
    # context: the built-in dense K2 on cylinders over the same cloud
    cyl = [R.FittedCylinder(rng.normal(size=3), rng.uniform(-40, 40, 3), rng.uniform(1, 10), True) for _ in range(args.cands)]
    for c in cyl:
        c.axis /= np.linalg.norm(c.axis)
    params = R.ransacparameters()
    ms_c, wall_c = timed(lambda: R.score_counts(pc, cyl, -1, params), ctx, args.steps, args.warmup)
    # the NumPy twin on a slice (CPU)
    sl = min(args.points, 1 << 20)
    P, Nn = V[:sl].astype(np.float64), N[:sl].astype(np.float64)
    ncpu = 8
    t0 = time.perf_counter()
    twin = np.array([int((U.torus_twin(np.asarray(p), k, P, Nn)).sum()) for p in recs[:ncpu]])
    cpu_s = time.perf_counter() - t0
    # spot check: the device counts of the slice agree with the twin
    pcs = R.RANSACCloud(V[:sl], N[:sl], 1, ctx=ctx)
    cs = np.zeros(ncpu, np.int32)
    ctx.check(R._lib.lib.rsc_user_score(pcs.handle, k.ctypes.data, 2, arr, ncpu, -1, cs.ctypes.data, None))
    assert np.array_equal(cs, twin), (cs, twin)
    med_u, med_c = float(np.median(ms_u)), float(np.median(ms_c))
    return {
        "points": args.points, "cands": args.cands, "steps": args.steps, "warmup": args.warmup,
        "nvrtc_compile_s": round(compile_s, 3),
        "user_torus_fp64": {"kernel_ms_median": round(med_u, 3), "kernel_ms_min": round(min(ms_u), 3),
                            "G_pairs_per_s": round(pairs / (med_u * 1e-3) / 1e9, 1),
                            "call_s_mean": round(wall_u / args.steps, 4), "inliers_total": int(counts.sum())},
        "builtin_cylinder_dense_k2": {"kernel_ms_median": round(med_c, 3), "G_pairs_per_s": round(pairs / (med_c * 1e-3) / 1e9, 1),
                                      "call_s_mean": round(wall_c / args.steps, 4)},
        "numpy_twin_cpu": {"cands": ncpu, "points": sl, "seconds": round(cpu_s, 3),
                           "G_pairs_per_s_cpu": round(ncpu * sl / cpu_s / 1e9, 4), "matches_device": True},
    }


def bench_loop(R):
    from tests import user_shapes as U

    NumpySlab, DeviceSlab = U.slab_classes(R)
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
    pc = R.RANSACCloud(V[perm], N[perm], 2)
    res, secs = {}, {}
    for rep in range(3):  # best of 3 (host-side times)
        for cls in (NumpySlab, DeviceSlab):
            params = R.ransacparameters([R.FittedSphere, cls], iteration={"tau": 500, "minsubsetN": 64, "itermax": 60})
            t0 = time.perf_counter()
            ex, _ = R.ransac(pc, params, True, seed=3)
            dt = time.perf_counter() - t0
            secs[cls] = min(secs.get(cls, dt), dt)
            res[cls] = ([(type(e.shape).__name__.replace("Numpy", "").replace("Device", ""), e.inpoints.tolist()) for e in ex],
                        pc.isenabled.copy())
    (a, ea), (b, eb) = res[NumpySlab], res[DeviceSlab]
    assert a == b and np.array_equal(ea, eb), "device slab and NumPy slab differ"
    return {"points": len(V), "shapes": len(a), "numpy_slab_s": round(secs[NumpySlab], 4), "device_slab_s": round(secs[DeviceSlab], 4),
            "identical": True}


def main(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--points", type=int, default=1 << 24)
    ap.add_argument("--cands", type=int, default=4096)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=None)
    args = ap.parse_args(argv)
    import ransac_jl_b200 as R

    line = {"gpu": gpu_info(), "torus": bench_torus(R, args), "loop": bench_loop(R)}
    s = json.dumps(line)
    print(s)
    if args.out:
        with open(args.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    sys.exit(main())
