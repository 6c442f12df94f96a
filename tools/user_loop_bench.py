"""User-defined shapes in the device loop (rsc_ransac_run_user) against the host plug-in loop; prints one JSON line.

  host_vs_device  a seeded scene of built-in primitives, slabs and vertical cylinders (tests/user_fit_shapes.py,
                  mixed_scene) at --points points, order [Plane, Sphere, Cylinder, Cone, Slab, ZCyl]:
                  (a) the host plug-in loop: host fits, device scoring (the shapes' compatibility source only);
                  (b) the device loop with the shapes' rsc_user_fit.  ransac() wall time from host arrays and the
                  device-loop time (rsc_run_seconds) of (b); the results are asserted identical
  device_10m      the same scene and order at --big points, device loop only; beside it the built-in part of the
                  order alone on the same cloud, and each run's mean device-loop time per speculative batch (the two
                  runs extract different shapes, so the difference bounds rather than isolates what the user fit and
                  score launches add per batch)
  c4_regression   built-in-only rsc_ransac_run on c4 (scene_cad, 10 M points, tau = n / 1000, minsubsetN 8192,
                  itermax 400, 32 subsets), device-loop seconds (rsc_run_seconds) of this tree against the tree given
                  by --parent (a built checkout of the parent commit), alternated process by process; the extracted
                  shapes and lists are asserted identical
Each leg runs --warmup untimed and --steps timed calls; (a) and (b) alternate.  The card's name and power limit
are read in the same run.

python -m tools.user_loop_bench [--points 1000000] [--big 10000000] [--steps 3] [--warmup 1] [--parent DIR] [--rounds 2]
                                [--out FILE]
"""
from __future__ import annotations

import argparse
import hashlib
import json
import math
import os
import statistics
import subprocess
import sys
import time

import numpy as np

from tools.user_shape_bench import gpu_info


def _params(R, types):
    p = R.ransacparameters(list(types), iteration={"tau": 2000, "minsubsetN": 128, "itermax": 2000})
    p.setdefault("slab", {"eps": 0.3, "alpha": math.radians(5), "tol": 0.1})
    p.setdefault("zcyl", {"eps": 0.05, "alpha": math.radians(10)})
    return p


def _key(R, ex):
    out = []
    for e in ex:
        s = e.shape
        rec = list(s.to_cand().p) if type(s) in (R.FittedPlane, R.FittedSphere, R.FittedCylinder, R.FittedCone) else list(s.device_record()[0])
        out.append((type(s).__name__.replace("Scored", "").replace("Device", ""), rec, e.inpoints.tobytes()))
    return out


def c4_worker(steps: int, warmup: int):
    """one process in one tree: c4 device-loop seconds of rsc_ransac_run + a digest of the result (JSON on stdout)"""
    import ransac_jl_b200 as R
    from ransac_jl_b200 import scenes

    sc = scenes.scene_cad(10_000_000)
    pc = R.RANSACCloud(sc.vertices, sc.normals, 32)
    params = R.ransacparameters(iteration={"tau": 10_000, "minsubsetN": 8192, "itermax": 400})
    secs, digest = [], None
    for step in range(warmup + steps):
        ex, _ = R.ransac(pc, params, True, seed=2024)
        if step >= warmup:
            secs.append(pc.last_run_seconds)
        h = hashlib.sha256()
        for e in ex:
            h.update(bytes(e.shape.to_cand()))
            h.update(e.inpoints.tobytes())
        digest = h.hexdigest()
    print(json.dumps({"device_loop_seconds": secs, "shapes": len(ex), "batches": pc.last_run_batches, "digest": digest}))


def c4_regression(parent: str, rounds: int, steps: int, warmup: int):
    here = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = {"parent": [], "this": []}
    for _ in range(rounds):
        for name, tree in (("parent", os.path.abspath(parent)), ("this", here)):
            env = dict(os.environ, PYTHONPATH=tree)
            r = subprocess.run([sys.executable, os.path.abspath(__file__), "--c4-worker", "--steps", str(steps), "--warmup", str(warmup)],
                               cwd=tree, env=env, capture_output=True, text=True, check=True)
            out[name].append(json.loads(r.stdout.strip().splitlines()[-1]))
    digests = {d["digest"] for v in out.values() for d in v}
    assert len(digests) == 1, "the parent and this tree extract different shapes on c4"
    res = {"identical": True, "shapes": out["this"][0]["shapes"], "batches": out["this"][0]["batches"]}
    for name, v in out.items():
        allsecs = [x for d in v for x in d["device_loop_seconds"]]
        res[name + "_device_loop_s_median"] = statistics.median(allsecs)
        res[name + "_device_loop_s"] = allsecs
    res["ratio_this_over_parent"] = res["this_device_loop_s_median"] / res["parent_device_loop_s_median"]
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--points", type=int, default=1_000_000)
    ap.add_argument("--big", type=int, default=10_000_000)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--out", default=None)
    ap.add_argument("--parent", default=None, help="a built checkout of the parent commit: adds the c4_regression leg")
    ap.add_argument("--rounds", type=int, default=2, help="c4_regression: alternations of parent / this tree")
    ap.add_argument("--c4-worker", action="store_true", help=argparse.SUPPRESS)
    a = ap.parse_args()
    if a.c4_worker:
        return c4_worker(a.steps, a.warmup)
    import ransac_jl_b200 as R
    from tests import user_fit_shapes as U

    _, (SS, SZ), (DS, DZ) = U.shape_classes(R)
    base = [R.FittedPlane, R.FittedSphere, R.FittedCylinder, R.FittedCone]
    res = {"gpu": gpu_info(), "order": ["Plane", "Sphere", "Cylinder", "Cone", "Slab", "ZCyl"]}

    V, N = U.mixed_scene(np.random.default_rng(31), a.points)
    pc = R.RANSACCloud(V, N, 3)
    variants = {"host_loop": base + [SS, SZ], "device_loop": base + [DS, DZ]}
    times = {k: [] for k in variants}
    loop_s, keys = [], {}
    for step in range(a.warmup + a.steps):
        for name, types in variants.items():
            t0 = time.perf_counter()
            ex, _ = R.ransac(pc, _params(R, types), True, seed=5)
            dt = time.perf_counter() - t0
            keys[name] = _key(R, ex)
            if step >= a.warmup:
                times[name].append(dt)
                if name == "device_loop":
                    loop_s.append(pc.last_run_seconds)
    assert keys["host_loop"] == keys["device_loop"], "host and device loop differ"
    res["host_vs_device"] = {
        "points": a.points, "shapes": len(keys["device_loop"]), "identical": True,
        "host_loop_s_median": statistics.median(times["host_loop"]),
        "device_loop_ransac_s_median": statistics.median(times["device_loop"]),
        "device_loop_run_seconds_median": statistics.median(loop_s),
        "host_loop_s": times["host_loop"], "device_loop_ransac_s": times["device_loop"],
    }
    res["host_vs_device"]["speedup_ransac"] = res["host_vs_device"]["host_loop_s_median"] / res["host_vs_device"]["device_loop_ransac_s_median"]
    pc.close()

    if a.big > 0:
        V, N = U.mixed_scene(np.random.default_rng(31), a.big)
        pc = R.RANSACCloud(V, N, 3)
        legs = {}
        for name, types in (("mixed", variants["device_loop"]), ("builtin_only", base)):
            t, ls = [], []
            for step in range(a.warmup + a.steps):
                t0 = time.perf_counter()
                ex, _ = R.ransac(pc, _params(R, types), True, seed=5)
                if step >= a.warmup:
                    t.append(time.perf_counter() - t0)
                    ls.append(pc.last_run_seconds)
            med = statistics.median(ls)
            legs[name] = {"shapes": len(ex), "ransac_s_median": statistics.median(t), "run_seconds_median": med, "run_seconds": ls,
                          "batches": pc.last_run_batches, "host_syncs": pc.last_run_syncs,
                          "ms_per_batch": 1e3 * med / max(pc.last_run_batches, 1)}
        res["device_10m"] = dict(legs["mixed"], points=a.big, builtin_only=legs["builtin_only"])
        pc.close()
    if a.parent:
        res["c4_regression"] = c4_regression(a.parent, a.rounds, a.steps, a.warmup)
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
