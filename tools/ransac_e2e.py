"""End-to-end ransac() on the BASELINE.json scenes (c2 / c4 / c5) at 1..8 GPUs, one process per GPU.

Used by bench.py (the `ransac` key of its JSON line, every N) and runnable on its own:
  python -m torch.distributed.run --nnodes=1 --nproc-per-node 8 --master-addr 127.0.0.1 --master-port 29517 \
      tools/ransac_e2e.py --scene c5

Layout at N > 1: SHARDED STORAGE -- every rank holds and uploads only its point range, the library sums
counts / hits / mask words with its own NCCL communicator (rsc_ctx_comm_init); torch.distributed only
carries the NCCL id, the barriers and the max-over-ranks of the timings.

What is timed ("seconds"): from host arrays (float32, pageable, as a caller has them) to the result on
the host -- cloud creation (host->device copy of the rank's points, SoA transposition, subset-1 copy),
the device loop, and fetching the rank's inlier index lists.  Scene generation, the subset permutation
and the NCCL set-up are outside.  The max over ranks is reported.

Checks (outside the timed region):
  * N = 1, c2 / c4: the C oracle's loop (oracle/oracle.c::orc_ransac) on the same scene -- shapes, inlier
    lists and final isenabled must be identical; its run time is the CPU ransac() baseline
  * every N: `digest` = per-shape (count, sum of mixed indices) summed over the ranks -- equal digests
    at different N mean equal results without gathering 10^7..10^8 indices
  * every N (c5 always, c4 at N > 1): replay -- every rank re-derives each extracted shape's inlier list
    on ITS points with the C oracle's compatibles* under the enabled mask of that moment
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

SCENES = {
    # name: (points, subsets r, iteration parameters as a function of n)
    "c2": (1 << 20, 32, lambda n: {"tau": n // 100, "minsubsetN": 4096, "itermax": 200}),
    "c4": (10_000_000, 32, lambda n: {"tau": n // 1000, "minsubsetN": 8192, "itermax": 400}),
    "c5": (100_000_000, 64, lambda n: {"tau": n // 500, "minsubsetN": 8192, "itermax": 200}),
}
_K1, _K2 = np.uint64(0x9E3779B97F4A7C15), np.uint64(0xC2B2AE3D27D4EB4F)


def _gen_chunk(args):
    from ransac_jl_b200 import scenes

    tag, i, n = args
    part = scenes.scene_lidar_chunk(i, n)
    np.save(f"{tag}_v{i}.npy", part.vertices)
    np.save(f"{tag}_n{i}.npy", part.normals)
    return i


def load_scene_range(which: str, n: int, lo: int, hi: int, rank: int, world: int, barrier):
    """float32 vertices / normals of the point range [lo, hi) of the scene (and the whole scene's arrays
    when they exist in this process, else None)."""
    from ransac_jl_b200 import scenes

    if which == "c2":
        sc = scenes.scene_c2(n)
        return sc.vertices[lo:hi], sc.normals[lo:hi], sc
    if which == "c4":
        sc = scenes.scene_cad(n)
        return sc.vertices[lo:hi], sc.normals[lo:hi], sc
    # c5: independent 12.5 M-point chunks, generated side by side (ranks x worker processes) into /dev/shm
    ch = scenes.LIDAR_CHUNK
    nch = (n + ch - 1) // ch
    tag = f"/dev/shm/rsc_c5_{n}_{os.environ.get('MASTER_PORT', '0')}"
    mine = [(tag, i, min(ch, n - i * ch)) for i in range(rank, nch, world)]
    workers = max(1, min(len(mine), (os.cpu_count() or 2) // (2 * world)))
    if workers > 1:
        import multiprocessing as mp

        with mp.get_context("spawn").Pool(workers) as pool:
            pool.map(_gen_chunk, mine)
    else:
        for a in mine:
            _gen_chunk(a)
    barrier()
    V = np.empty((hi - lo, 3), np.float32)
    Nn = np.empty((hi - lo, 3), np.float32)
    for i in range(nch):
        a, b = max(lo, i * ch), min(hi, min(n, (i + 1) * ch))
        if a < b:
            V[a - lo : b - lo] = np.load(f"{tag}_v{i}.npy", mmap_mode="r")[a - i * ch : b - i * ch]
            Nn[a - lo : b - lo] = np.load(f"{tag}_n{i}.npy", mmap_mode="r")[a - i * ch : b - i * ch]
    barrier()
    if rank == 0:
        for i in range(nch):
            os.remove(f"{tag}_v{i}.npy"), os.remove(f"{tag}_n{i}.npy")
    return V, Nn, None


def digest(extracted, allreduce_sum):
    """per shape: [type, total inliers, sum over inliers of mix(index)] -- additive over ranks"""
    rows = np.zeros((len(extracted), 2), np.int64)
    for i, e in enumerate(extracted):
        u = e.inpoints.astype(np.uint64)
        mix = (u * _K1) ^ ((u * _K2) >> np.uint64(29))
        rows[i, 0] = len(u)
        rows[i, 1] = int(mix.sum(dtype=np.uint64).astype(np.int64)) if len(u) else 0
    rows = allreduce_sum(rows)
    return [[int(e.shape.to_cand().type), int(a), f"{int(b) & 0xFFFFFFFFFFFFFFFF:016x}"] for e, (a, b) in zip(extracted, rows)]


def replay_local(extracted, V, N, params, nthreads):
    """every extracted shape's list on this rank's points == the C oracle's refit (compatibles* among the
    points still enabled at that moment, ascending), shape after shape.  Returns mismatching shapes."""
    from oracle import c_oracle
    from tests.helpers import oracle_params

    op = oracle_params(params)
    P64, N64 = V.astype(np.float64), N.astype(np.float64)
    en = np.ones(len(V), bool)
    bad = 0
    for e in extracted:
        _, _, m = c_oracle.score_counts([e.shape], P64, N64, op, enabled=en, want_masks=True, nthreads=nthreads)
        m = m[0] & en  # refit works on the enabled points for every type (e.g. sphere.jl:181-185)
        bad += int(not np.array_equal(np.flatnonzero(m), e.local_idx))
        en[m] = False
    return bad


def run(which: str, rank: int, world: int, local: int, dist=None, n_override: int = 0, check: bool = True, cpu_loop: bool = True,
        reps: int = 5, return_extracted: bool = False):
    """The JSON record of `which`; with return_extracted, (record, what ransac() returned in the last timed run)."""
    import torch

    import ransac_jl_b200 as R
    from ransac_jl_b200 import shard

    n0, r, itf = SCENES[which]
    n = n_override or n0
    it = itf(n)
    params = R.ransacparameters(iteration=it)
    dev = torch.device("cuda", local)

    def barrier():
        if world > 1:
            dist.barrier()

    def allmax(x):
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def allsum_i64(a):
        t = torch.from_numpy(np.ascontiguousarray(a)).to(dev)
        if world > 1:
            dist.all_reduce(t)
        return t.cpu().numpy()

    lo, hi = shard.partition(n, world)[rank] if world > 1 else (0, n)
    t_gen = time.perf_counter()
    V, Nn, sc = load_scene_range(which, n, lo, hi, rank, world, barrier)
    V, Nn = np.ascontiguousarray(V), np.ascontiguousarray(Nn)
    subsets = R.makesubsets(n, r, np.random.default_rng(1234))
    sub0 = [subsets[0]]  # the reference scores subset 1 only (iterations.jl:95)
    del subsets
    t_gen = time.perf_counter() - t_gen
    ctx = R.Context.get(local)
    if world > 1:
        shard.init_comm(ctx)

    def make_cloud(v=None, nn=None):
        v, nn = (V, Nn) if v is None else (v, nn)
        if world > 1:
            return R.RANSACCloud(v, nn, sub0, device=local, shard=(lo, n))
        return R.RANSACCloud(v, nn, sub0, device=local)

    # warm-up: allocations, NCCL channels, kernel loading, GPU clocks (the scene generation left the GPU idle)
    pc = make_cloud()
    R.ransac(pc, R.ransacparameters(iteration=dict(it, itermax=min(it["itermax"], 100))), True, seed=1)
    pc.close()
    best, all_secs = None, []
    for rep in range(reps):
        torch.cuda.synchronize()
        barrier()
        t0 = time.perf_counter()
        pc = make_cloud()
        pc.count_enabled()  # waits for the upload (the copy itself is asynchronous)
        t1 = time.perf_counter()
        ex, _ = R.ransac(pc, params, True, seed=2024)
        t2 = time.perf_counter()
        res = {"seconds": allmax(t2 - t0), "upload_seconds": allmax(t1 - t0), "ransac_call_seconds": allmax(t2 - t1),
               "device_loop_seconds": allmax(pc.last_run_seconds), "host_syncs": pc.last_run_syncs, "batches": pc.last_run_batches,
               "iterations": pc.last_run_iterations}
        all_secs.append(res["seconds"])
        if best is None or res["seconds"] < best[0]["seconds"]:
            best = (res, ex, pc.isenabled)
        pc.close()
    ex_last = ex
    res, ex, enabled_local = best
    res = dict(res, seconds_all_runs=all_secs, timing=f"best of {reps} runs (all listed), each from pageable host arrays to the result on the host")
    # the same call with the caller's arrays in PAGE-LOCKED memory (include/rsc.h: read by DMA, no staging copy on the host)
    try:
        tv, tn = torch.from_numpy(V).pin_memory(), torch.from_numpy(Nn).pin_memory()
        pin = []
        for rep in range(2):
            torch.cuda.synchronize()
            barrier()
            t0 = time.perf_counter()
            pc = make_cloud(tv.numpy(), tn.numpy())
            pc.count_enabled()
            t1 = time.perf_counter()
            ex_p, _ = R.ransac(pc, params, True, seed=2024)
            t2 = time.perf_counter()
            pin.append((allmax(t2 - t0), allmax(t1 - t0)))
            assert [len(e.inpoints) for e in ex_p] == [len(e.inpoints) for e in ex]
            pc.close()
        res["page_locked_host_arrays"] = {"seconds": min(p[0] for p in pin), "upload_seconds": min(p[1] for p in pin),
                                          "seconds_all_runs": [p[0] for p in pin]}
        del tv, tn
    except Exception as e:  # informational
        res["page_locked_host_arrays"] = {"error": repr(e)}
    for e in ex:
        e.local_idx = e.inpoints - lo
    out = {"scene": which, "points": n, "n_gpus": world, "subsets": r, "iteration": it,
           "layout": "sharded storage, library NCCL" if world > 1 else "single GPU", **res,
           "n_shapes": len(ex), "points_extracted": int(sum(e.total for e in ex)),
           "h2d_bytes_per_rank": int((hi - lo) * 24), "scene_generation_seconds": t_gen,
           "digest": digest(ex, allsum_i64)}
    threads_per_rank = max(1, (os.cpu_count() or 1) // world)
    if check and (which == "c5" or world > 1):
        bad = replay_local(ex, V, Nn, params, threads_per_rank)
        still = int(np.count_nonzero(enabled_local)) + int(sum(len(e.inpoints) for e in ex))
        bad_total = int(allsum_i64(np.array([bad, int(still != hi - lo)], np.int64)).sum())
        out["replay"] = {"shapes": len(ex), "mismatching_lists": bad_total,
                         "checker": "oracle/oracle.c::orc_score refit replay on every rank's points"}
    if rank == 0 and world == 1 and cpu_loop and which in ("c2", "c4") and sc is not None:
        from oracle import c_oracle
        from tests.helpers import oracle_params

        t0 = time.perf_counter()
        want, en, info = c_oracle.ransac(sc.vertices, sc.normals, sub0[0], oracle_params(params), 2024)
        dt = time.perf_counter() - t0
        same = len(want) == len(ex) and all(
            e.shape.to_cand().type == w[0] and np.allclose(np.array(e.shape.to_cand().p[:]), w[2], rtol=1e-5, atol=1e-3)
            and np.array_equal(e.inpoints, w[3]) for e, w in zip(ex, want)) and bool(np.array_equal(en, enabled_local))
        out["cpu_ransac"] = {"seconds": dt, "cores": info["threads"], "kind": "port",
                             "what": "oracle/oracle.c::orc_ransac, the C restatement of RANSAC.jl's loop (iterations.jl:35-162) on the "
                                     "same scene, parameters and Philox minimal sets (Julia is not installed)",
                             "phase_seconds": {"sample_fit": info["seconds"][0], "score": info["seconds"][1], "refit_bookkeeping": info["seconds"][2]},
                             "n_shapes": len(want)}
        out["matches_cpu_oracle"] = bool(same)
    if sc is not None and getattr(sc, "labels", None) is not None and world == 1:
        out["recall"] = recall(sc, ex)
    if which == "c4" and world == 1 and sc is not None:
        # extension: the same scene with the level-weighted octree-cell sampler (the strategy the reference documents;
        # ~16 k candidates per iteration instead of ~60: the loop scores them with the culled scorer, DESIGN.md section 8)
        try:
            cs_all = []
            for rep in range(3):  # the first run also sizes the loop's scratch buffers
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                pc = make_cloud()
                pc.build_cells(8)
                ex_o, _ = R.ransac(pc, params, True, seed=2024, sampler="octree", lw_period=16)
                cs_all.append(time.perf_counter() - t0)
                loop_s = pc.last_run_seconds
                pc.close()
            out["cell_sampler"] = {"seconds": min(cs_all[1:]), "seconds_all_runs": cs_all, "device_loop_seconds": loop_s,
                                   "octree_levels": 8, "lw_period": 16, "n_shapes": len(ex_o),
                                   "points_extracted": int(sum(len(e.inpoints) for e in ex_o)),
                                   "recall": recall(sc, ex_o) if getattr(sc, "labels", None) is not None else None,
                                   "timing": "host arrays -> octree cells -> ransac() -> result on the host"}
        except Exception as e:  # informational
            out["cell_sampler"] = {"error": repr(e)}
    return (out, ex_last) if return_extracted else out


def recall(sc, ex, thresh=0.5):
    """ground truth of the generator: a primitive counts as found when one extracted shape holds at least
    `thresh` of its points (and those points are at least half of that shape's list)"""
    labels = np.asarray(sc.labels)
    nprim = len(sc.primitives)
    size = np.bincount(labels[labels >= 0], minlength=nprim)
    found = np.zeros(nprim, bool)
    for e in ex:
        lab = labels[e.inpoints]
        lab = lab[lab >= 0]
        if len(lab) == 0:
            continue
        cnt = np.bincount(lab, minlength=nprim)
        j = int(cnt.argmax())
        if cnt[j] >= thresh * size[j] and cnt[j] >= 0.5 * len(e.inpoints):
            found[j] = True
    big = size >= max(1, int(0.005 * len(labels)))
    return {"primitives": int(nprim), "found": int(found.sum()), "primitives_over_0.5pct_of_cloud": int(big.sum()),
            "found_among_those": int((found & big).sum()),
            "points_on_primitives": int((labels >= 0).sum()), "points_of_found_primitives": int(size[found].sum())}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scene", default="c4", choices=list(SCENES))
    ap.add_argument("--points", type=int, default=0)
    ap.add_argument("--no-check", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    args = ap.parse_args()
    import torch
    import torch.distributed as dist

    rank, world, local = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1)), int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    out = run(args.scene, rank, world, local, dist if world > 1 else None, args.points, not args.no_check, not args.no_cpu)
    if rank == 0:
        print(json.dumps(out))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
