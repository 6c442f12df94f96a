"""Cost of normal orientation without a viewpoint (rsc_orient_normals) on one GPU, next to the k-NN search it builds on:

  * c4 (10 M-point CAD-like scene) and c5 (LiDAR-like, --c5-points, 10^8 by default), k = 16: the median wall time of
    the synchronising host-in / host-out call after a warm-up call, with given normals (the scene's, with random
    signs) and with nrm_in = NULL (estimate, then orient), next to rsc_estimate_normals at the same k;
  * the Borůvka rounds, the vertices and trees of the forest, and on c4 the graph's edges (the symmetric union of the
    device's k-NN lists, counted on the host; too large to sort on the host at 10^8 points);
  * on c4, the per-primitive consistency of the oriented random-sign normals against the ground truth.

The GPU's name and power limit are read in the same run.  Prints one JSON line (and writes it to --out).
    python tools/orient_bench.py --out profiles/r6_orient_bench.json"""
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
from ransac_jl_b200 import scenes
from ransac_jl_b200._lib import Context, lib

ap = argparse.ArgumentParser()
ap.add_argument("--k", type=int, default=16)
ap.add_argument("--calls", type=int, default=3, help="timed calls per (scene, mode)")
ap.add_argument("--c5-points", type=int, default=100_000_000)
ap.add_argument("--out", default="")
args = ap.parse_args()
if not torch.cuda.is_available():
    sys.exit("orient_bench: needs a GPU")

gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                     text=True).stdout.strip().splitlines()
out = {"gpu": gpu[0] if gpu else "unknown", "k": args.k, "calls": args.calls}
ctx = Context.get(0)


def timed(call):
    ts = []
    for rep in range(args.calls + 1):  # the first call is a warm-up
        t0 = time.perf_counter()
        call()
        if rep:
            ts.append(time.perf_counter() - t0)
    return float(np.median(ts))


def bench(tag, sc, small):
    V, k = sc.vertices, args.k
    flipped = (sc.normals * np.random.default_rng(3).choice(np.float32([-1, 1]), len(V))[:, None]).astype(np.float32)
    res = np.empty_like(V)
    stats = (C.c_int64 * 4)()
    out[f"{tag}_points"] = len(V)
    out[f"{tag}_estimate_s"] = round(timed(lambda: ctx.check(lib.rsc_estimate_normals(
        ctx.h, V.ctypes.data, len(V), k, None, res.ctypes.data, None, None))), 4)
    out[f"{tag}_orient_given_s"] = round(timed(lambda: ctx.check(lib.rsc_orient_normals(
        ctx.h, V.ctypes.data, len(V), k, flipped.ctypes.data, res.ctypes.data, None, stats))), 4)
    for i, name in enumerate(("vertices", "forest_edges", "trees", "rounds")):
        out[f"{tag}_given_{name}"] = int(stats[i])
    if small:
        agree = np.einsum("ij,ij->i", res.astype(np.float64), sc.normals.astype(np.float64)) > 0
        per = [float(max(a.mean(), 1 - a.mean())) for a in (agree[sc.labels == p] for p in range(len(sc.primitives))) if len(a)]
        out[f"{tag}_consistency_min"] = round(min(per), 5)
        out[f"{tag}_consistency_median"] = round(float(np.median(per)), 5)
        out[f"{tag}_primitives"] = len(per)
    out[f"{tag}_orient_estimate_s"] = round(timed(lambda: ctx.check(lib.rsc_orient_normals(
        ctx.h, V.ctypes.data, len(V), k, None, res.ctypes.data, None, stats))), 4)
    for i, name in enumerate(("vertices", "forest_edges", "trees", "rounds")):
        out[f"{tag}_estimated_{name}"] = int(stats[i])
    if not small:
        return
    # the graph's edges: the symmetric union of the lists, counted on the device's own lists
    nbr = np.empty((len(V), k), np.int64)
    ctx.check(lib.rsc_estimate_normals(ctx.h, V.ctypes.data, len(V), k, None, res.ctypes.data, nbr.ctypes.data, None))
    i = np.repeat(np.arange(len(V), dtype=np.int64), k)
    j = nbr.reshape(-1)
    del nbr
    keep = (j >= 0) & (j != i)
    key = np.minimum(i[keep], j[keep]) * len(V) + np.maximum(i[keep], j[keep])
    del i, j, keep
    key.sort()
    out[f"{tag}_graph_edges_all_points"] = int(1 + np.count_nonzero(key[1:] != key[:-1])) if len(key) else 0


sc = scenes.scene_cad()
bench("c4", sc, True)
del sc
if args.c5_points:
    sc = scenes.scene_lidar(args.c5_points)
    bench("c5", sc, False)
    del sc

line = json.dumps(out)
print(line)
if args.out:
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(line + "\n")
