"""Cost of exact float64 clouds (rsc_cloud_create_f64_exact) against rounding ones (rsc_cloud_create_f64) built
from the same unrounded float64 arrays, on one GPU:

  * dense whole-cloud scoring, c3 workload (4096 candidates x 16 Mi points): ms per step, G evals/s and the
    (candidate, point) pairs decided in FP64 per step (rsc_ctx_stats().exact_pairs);
  * culled whole-cloud scoring of the same candidates (rsc_score_culled);
  * ransac() on the 10 M-point c4 scene: wall time and the device loop's own time;
  * upload time and HBM footprint.

The two kinds of cloud alternate within every measurement.  Prints one JSON line (and writes it to --out).
    python tools/exact_f64_bench.py --out /tmp/exact_f64_bench.json"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import ransac_jl_b200 as R
from ransac_jl_b200 import scenes

ap = argparse.ArgumentParser()
ap.add_argument("--points", type=int, default=16 << 20)
ap.add_argument("--cands", type=int, default=4096)
ap.add_argument("--steps", type=int, default=10)
ap.add_argument("--reps", type=int, default=3, help="ransac() runs per kind of cloud")
ap.add_argument("--no-c4", action="store_true")
ap.add_argument("--out", default="")
args = ap.parse_args()
if not torch.cuda.is_available():
    sys.exit("exact_f64_bench: needs a GPU")


def unrounded(sc, seed):
    rng = np.random.default_rng(seed)
    V = sc.vertices.astype(np.float64) + rng.uniform(-1e-6, 1e-6, sc.vertices.shape)
    N = sc.normals.astype(np.float64) + rng.uniform(-1e-7, 1e-7, sc.normals.shape)
    return V, N


def mem_used():
    torch.cuda.synchronize()
    free, total = torch.cuda.mem_get_info()
    return total - free


def make_clouds(V, N, subsets, reps=3):
    """one cloud of each kind; creation timed `reps` times, the kinds alternating (median).  The HBM figure is the
    device memory the last creation took, when the context's upload scratch is already allocated."""
    clouds, times, mem = {}, {"rounding": [], "exact": []}, {}
    for _ in range(reps):
        for kind in ("rounding", "exact"):
            if kind in clouds:
                clouds.pop(kind).close()
            m0 = mem_used()
            t0 = time.perf_counter()
            pc = R.RANSACCloud(V, N, subsets, exact=kind == "exact")
            pc.count_enabled()  # waits for the chunked upload
            times[kind].append(time.perf_counter() - t0)
            mem[kind] = mem_used() - m0
            clouds[kind] = pc
    return clouds, {k: round(float(np.median(v)), 4) for k, v in times.items()}, mem


gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
out = {"gpu": gpu, "points": args.points, "candidates": args.cands}
params = R.ransacparameters()

# ---- c3: dense and culled whole-cloud scoring ----
sc = scenes.scene_c3(args.points)
cands = scenes.perturbed_candidates(sc, args.cands // 4, seed=7)
V, N = unrounded(sc, 3)
del sc
clouds, t, mem = make_clouds(V, N, [np.zeros(0, np.int64)])
for kind in clouds:
    out[f"upload_s_{kind}"] = t[kind]
    out[f"hbm_bytes_{kind}"] = int(mem[kind])
for kind, pc in clouds.items():  # warm-up
    R.score_counts(pc, cands, -1, params)
res = {k: {"ms": [], "exact_pairs": []} for k in clouds}
for _ in range(args.steps):
    for kind, pc in clouds.items():
        s0 = pc.ctx.stats().exact_pairs
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        counts, _ = R.score_counts(pc, cands, -1, params)
        torch.cuda.synchronize()
        res[kind]["ms"].append((time.perf_counter() - t0) * 1e3)
        res[kind]["exact_pairs"].append(int(pc.ctx.stats().exact_pairs - s0))
        res[kind]["counts"] = counts
evals = len(cands) * args.points
for kind, r in res.items():
    ms = float(np.median(r["ms"]))
    out[f"dense_ms_{kind}"] = round(ms, 3)
    out[f"dense_G_evals_s_{kind}"] = round(evals / (ms * 1e-3) / 1e9, 1)
    out[f"dense_fp64_pairs_per_step_{kind}"] = int(np.median(r["exact_pairs"]))
out["dense_ms_ratio_exact_over_rounding"] = round(out["dense_ms_exact"] / out["dense_ms_rounding"], 4)
out["dense_counts_differ"] = int((res["exact"]["counts"] != res["rounding"]["counts"]).sum())
# culled
cres = {k: [] for k in clouds}
for kind, pc in clouds.items():
    pc.build_cells(11)
    R.score_counts_culled(pc, cands, params)  # builds the Morton copy
for _ in range(args.steps):
    for kind, pc in clouds.items():
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        R.score_counts_culled(pc, cands, params)
        torch.cuda.synchronize()
        cres[kind].append((time.perf_counter() - t0) * 1e3)
for kind in clouds:
    out[f"culled_ms_{kind}"] = round(float(np.median(cres[kind])), 3)
for pc in clouds.values():
    pc.close()
del clouds, V, N

# ---- c4: ransac() on the 10 M-point CAD-like scene ----
if not args.no_c4:
    sc = scenes.scene_cad()
    it = {"tau": sc.vertices.shape[0] // 1000, "minsubsetN": 8192, "itermax": 400}
    p4 = R.ransacparameters(iteration=it)
    V, N = unrounded(sc, 4)
    del sc
    subsets = R.makesubsets(len(V), 32, np.random.default_rng(1234))
    clouds, t, mem = make_clouds(V, N, subsets)
    for kind in clouds:
        out[f"c4_upload_s_{kind}"] = t[kind]
        out[f"c4_hbm_bytes_{kind}"] = int(mem[kind])
    wall = {k: [] for k in clouds}
    loop = {k: [] for k in clouds}
    shapes = {}
    for rep in range(args.reps + 1):  # the first run of each is a warm-up
        for kind, pc in clouds.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            ex, _ = R.ransac(pc, p4, True, seed=99)
            torch.cuda.synchronize()
            if rep:
                wall[kind].append(time.perf_counter() - t0)
                loop[kind].append(pc.last_run_seconds)  # (ransac() returns it truncated to 10 ms)
            shapes[kind] = [len(e.inpoints) for e in ex]
    for kind in clouds:
        out[f"c4_ransac_wall_s_{kind}"] = round(float(np.median(wall[kind])), 4)
        out[f"c4_device_loop_s_{kind}"] = round(float(np.median(loop[kind])), 4)
        out[f"c4_shapes_{kind}"] = len(shapes[kind])
    out["c4_wall_ratio_exact_over_rounding"] = round(out["c4_ransac_wall_s_exact"] / out["c4_ransac_wall_s_rounding"], 4)
    out["c4_inlier_totals_differ"] = shapes["exact"] != shapes["rounding"]
    for pc in clouds.values():
        pc.close()

line = json.dumps(out)
print(line)
if args.out:
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(line + "\n")
