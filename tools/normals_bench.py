"""Cost of device normal estimation (rsc_estimate_normals) on one GPU, next to ransac() on the same scene:

  * c4 (10 M-point CAD-like scene) and c5 (LiDAR-like, --c5-points, 10^8 by default) with k = 8 / 16 / 32: the
    median wall time of the synchronising call (host in / host out) after a warm-up call, points/s, and the
    (query, candidate) distances evaluated per query;
  * ransac() on the same scene with its generated normals, for scale (median of --reps runs after a warm-up);
  * on the single-scan scene_view, the primitives ransac() recovers with analytic and with estimated normals.

The GPU's name and power limit are read in the same run.  Prints one JSON line (and writes it to --out).
    python tools/normals_bench.py --out profiles/r5_normals_bench.json"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import ransac_jl_b200 as R
from ransac_jl_b200 import scenes
from ransac_jl_b200._lib import Context, lib

ap = argparse.ArgumentParser()
ap.add_argument("--ks", default="8,16,32")
ap.add_argument("--calls", type=int, default=5, help="timed calls per (scene, k)")
ap.add_argument("--reps", type=int, default=3, help="timed ransac() runs per scene")
ap.add_argument("--c5-points", type=int, default=100_000_000)
ap.add_argument("--out", default="")
args = ap.parse_args()
if not torch.cuda.is_available():
    sys.exit("normals_bench: needs a GPU")

gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                     text=True).stdout.strip().splitlines()
out = {"gpu": gpu[0] if gpu else "unknown", "ks": args.ks, "calls": args.calls}
ctx = Context.get(0)


def timed_normals(V, k):
    nrm = np.empty_like(V)
    pairs = C.c_int64()
    ts = []
    for rep in range(args.calls + 1):  # the first call is a warm-up
        t0 = time.perf_counter()
        ctx.check(lib.rsc_estimate_normals(ctx.h, V.ctypes.data, len(V), k, None, nrm.ctypes.data, None, C.byref(pairs)))
        if rep:
            ts.append(time.perf_counter() - t0)
    return float(np.median(ts)), pairs.value / len(V)


def timed_ransac(V, N, r, it):
    pc = R.RANSACCloud(V, N, r)
    params = R.ransacparameters(iteration=it)
    ts = []
    for rep in range(args.reps + 1):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        R.ransac(pc, params, True, seed=99)
        torch.cuda.synchronize()
        if rep:
            ts.append(time.perf_counter() - t0)
    pc.close()
    return float(np.median(ts))


def bench(tag, V, N, r, it):
    for k in [int(x) for x in args.ks.split(",")]:
        s, ppq = timed_normals(V, k)
        out[f"{tag}_k{k}_s"] = round(s, 4)
        out[f"{tag}_k{k}_points_per_s"] = round(len(V) / s, 1)
        out[f"{tag}_k{k}_pairs_per_query"] = round(ppq, 2)
    out[f"{tag}_points"] = len(V)
    out[f"{tag}_ransac_s"] = round(timed_ransac(V, N, r, it), 4)


sc = scenes.scene_cad()
bench("c4", sc.vertices, sc.normals, 32, {"tau": len(sc.vertices) // 1000, "minsubsetN": 8192, "itermax": 400})
del sc
if args.c5_points:
    sc = scenes.scene_lidar(args.c5_points)
    bench("c5", sc.vertices, sc.normals, 64, {"tau": len(sc.vertices) // 500, "minsubsetN": 8192, "itermax": 200})
    del sc

# shapes ransac() recovers on one scan with analytic and with estimated normals
scan = scenes.scan_scenario()
sc = scan.scene
for name, nrm in (("analytic", sc.normals), ("estimated", R.estimate_normals(sc.vertices, viewpoint=scan.viewpoint))):
    pc = R.RANSACCloud(sc.vertices, nrm, scan.subsets)
    ext, _ = R.ransac(pc, R.ransacparameters(iteration=scan.iteration), True, seed=scan.seed)
    out[f"view_shapes_{name}"] = len(ext)
    out[f"view_recovered_{name}"] = len(scenes.recovered(sc, [(e.shape.kind, np.asarray(e.inpoints)) for e in ext]))
    pc.close()
out["view_primitives"] = len(sc.primitives)

line = json.dumps(out)
print(line)
if args.out:
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(line + "\n")
