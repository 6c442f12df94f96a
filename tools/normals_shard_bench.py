"""Cost of the sharded normals (rsc_estimate_normals_shard, rsc_orient_normals_shard) over N GPUs of one box, one
process per GPU, the library's NCCL communicator:

    python -m torch.distributed.run --nproc_per_node N tools/normals_shard_bench.py --out profiles/x.json

  * c4 (scene_cad, 10 M points) and c5 (scene_lidar, --c5-points, 10^8 by default) at k = 16, the settings of
    tools/normals_bench.py and tools/orient_bench.py; each rank holds its rows of shard.partition(n, N);
  * the median of --calls synchronising calls after two warm-up calls, the maximum over the ranks, for estimation and
    for orientation with nrm_in = NULL;
  * one more call of each with RSC_NORMALS_TRACE=1 (synchronising between phases): the per-phase split (gather,
    prepare, search, exchange, forest; maximum over the ranks) and the per-rank search time, min and max;
  * the all-reduce calls and bytes of one call (rsc_ctx_comm_stats);
  * per-rank SHA-256 digests of the output rows.  With N = 1 the digests of the output cut by shard.partition(n, M)
    for M in --digest-worlds are written too; --reference (the N = 1 JSON) then checks a run at N > 1 against it.

--shared-gpu: every rank runs on cuda:0 and the all-reduces are host-staged over gloo (the library's host callback),
so that the protocol at N > 1 can be measured on a single GPU.  The callback passes a token from rank to rank between
the gather and the row exchange, so the ranks' prepare steps and searches run one at a time and each rank's search
time is that of its slice alone on one B200, which is what it costs on a GPU of its own.  Only the traced call is
reported then (search per rank, prepare, forest, the all-reduce calls and bytes counted in the callback, digests);
call times, the gather and the exchange include the token waits and the host staging and are not reported, and the
forest, which every rank builds at the same time on the one GPU, is an upper bound of its cost on separate GPUs.

The GPU's name and power limit are read in the same run.  Rank 0 prints one JSON line (and writes it to --out)."""
import argparse
import ctypes as C
import hashlib
import json
import os
import re
import statistics
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from ransac_jl_b200 import scenes, shard
from ransac_jl_b200._lib import Context, lib

ap = argparse.ArgumentParser()
ap.add_argument("--k", type=int, default=16)
ap.add_argument("--calls", type=int, default=3, help="timed calls per (scene, call)")
ap.add_argument("--c5-points", type=int, default=100_000_000)
ap.add_argument("--digest-worlds", default="2,4,8")
ap.add_argument("--reference", default="", help="the N = 1 result, to check the digests of a run at N > 1")
ap.add_argument("--shared-gpu", action="store_true", help="all ranks on cuda:0, host-staged gloo all-reduces")
ap.add_argument("--out", default="")
args = ap.parse_args()
if not torch.cuda.is_available():
    sys.exit("normals_shard_bench: needs a GPU")

dist.init_process_group("gloo")
rank, world = dist.get_rank(), dist.get_world_size()
dev = 0 if args.shared_gpu else int(os.environ.get("LOCAL_RANK", rank))
torch.cuda.set_device(dev)
ctx = Context.get(dev)
AR = {"i": 0, "calls": 0, "bytes": 0}  # the all-reduces of the current call (--shared-gpu)


def install_turns():
    """the host-staged callback of shard.attach_comm(..., comm="host"), plus the token that serialises the searches:
    the 3rd all-reduce of a call is the gather, the 4th the row exchange"""
    from ransac_jl_b200 import _lib
    from ransac_jl_b200.shard import _DevInt32

    ext = torch.cuda.ExternalStream(ctx.stream, device=torch.device("cuda", dev))
    token = torch.zeros(1)

    def _allreduce(user, ptr, count, stream):
        try:
            i = AR["i"]
            AR["i"] += 1
            AR["calls"] += 1
            AR["bytes"] += 4 * count
            t = torch.as_tensor(_DevInt32(ptr, count), device=torch.device("cuda", dev))
            with torch.cuda.stream(ext):
                if i == 3:
                    ext.synchronize()  # this rank's search is done: the next rank may start
                    if rank + 1 < world:
                        dist.send(token, rank + 1)
                h = t.cpu()
                dist.all_reduce(h)
                t.copy_(h)
                if i == 2 and rank > 0:
                    ext.synchronize()
                    dist.recv(token, rank - 1)
            return 0
        except Exception as e:
            print(f"[normals_shard_bench] all-reduce callback failed: {e!r}")
            return 1

    ctx._allreduce_cb = _lib.ALLREDUCE_FN(_allreduce)
    ctx.check(lib.rsc_ctx_set_allreduce(ctx.h, C.cast(ctx._allreduce_cb, C.c_void_p), None))


if args.shared_gpu:
    install_turns()
else:
    shard.attach_comm(ctx, comm="nccl")
gpu = subprocess.run(["nvidia-smi", "-i", str(dev), "--query-gpu=name,power.limit", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip().splitlines()
out = {"gpu": gpu[0] if gpu else "unknown", "gpus": world, "k": args.k, "calls": args.calls,
       "shared_gpu": args.shared_gpu}
TRACE = re.compile(r"gather ([\d.]+) prepare ([\d.]+) search ([\d.]+) exchange ([\d.]+) forest ([\d.]+) ms")
PHASES = ("gather", "prepare", "search", "exchange", "forest")


def gathered(x):
    parts = [None] * world
    dist.all_gather_object(parts, x)
    return parts


def traced(call):
    """one call with RSC_NORMALS_TRACE=1; -> its phase times in ms (the library prints them to stderr)"""
    os.environ["RSC_NORMALS_TRACE"] = "1"
    sys.stderr.flush()
    saved = os.dup(2)
    with tempfile.TemporaryFile(mode="w+") as f:
        os.dup2(f.fileno(), 2)
        try:
            call()
        finally:
            os.dup2(saved, 2)
            os.close(saved)
            del os.environ["RSC_NORMALS_TRACE"]
        f.seek(0)
        m = TRACE.search(f.read())
    return [float(x) for x in m.groups()]


def comm_stats():
    if args.shared_gpu:
        return AR["calls"], AR["bytes"]
    calls, nbytes = C.c_int64(), C.c_int64()
    ctx.check(lib.rsc_ctx_comm_stats(ctx.h, C.byref(calls), C.byref(nbytes)))
    return calls.value, nbytes.value


def digest(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()[:16]


def measure(tag, name, call, res, n):
    def run():
        AR["i"] = 0
        call()

    ts = []
    warmups = 1 if args.shared_gpu else 2
    for rep in range(warmups + (0 if args.shared_gpu else args.calls)):
        dist.barrier()
        t0 = time.perf_counter()
        run()
        if rep >= warmups:
            ts.append(time.perf_counter() - t0)
    c0 = comm_stats()
    dist.barrier()
    ph = traced(run)
    c1 = comm_stats()
    parts = gathered((statistics.median(ts) if ts else None, ph, digest(res)))
    shown = ("prepare", "search", "forest") if args.shared_gpu else PHASES
    if not args.shared_gpu:
        out[f"{tag}_{name}_s"] = round(max(p[0] for p in parts), 4)
    for i, p in enumerate(PHASES):
        if p in shown:
            out[f"{tag}_{name}_{p}_ms"] = round(max(q[1][i] for q in parts), 2)
    out[f"{tag}_{name}_search_ms_min"] = round(min(q[1][2] for q in parts), 2)
    out[f"{tag}_{name}_search_ms_ranks"] = [round(q[1][2], 2) for q in parts]
    out[f"{tag}_{name}_allreduce_calls"] = c1[0] - c0[0]
    out[f"{tag}_{name}_allreduce_bytes"] = c1[1] - c0[1]
    out[f"{tag}_{name}_digests"] = [q[2] for q in parts]
    if world == 1:
        for m in [int(x) for x in args.digest_worlds.split(",") if x]:
            out[f"{tag}_{name}_digests_{m}"] = [digest(res[a:b]) for a, b in shard.partition(n, m)]


def bench(tag, sc):
    V, k, n = sc.vertices, args.k, len(sc.vertices)
    lo, hi = shard.partition(n, world)[rank]
    Vl = np.ascontiguousarray(V[lo:hi], dtype=np.float32)
    res = np.empty((hi - lo, 3), np.float32)
    stats = (C.c_int64 * 4)()
    out[f"{tag}_points"] = n
    measure(tag, "estimate", lambda: ctx.check(lib.rsc_estimate_normals_shard(
        ctx.h, Vl.ctypes.data, hi - lo, lo, n, k, None, res.ctypes.data, None, None)), res, n)
    measure(tag, "orient", lambda: ctx.check(lib.rsc_orient_normals_shard(
        ctx.h, Vl.ctypes.data, hi - lo, lo, n, k, None, res.ctypes.data, None, stats)), res, n)
    for i, name in enumerate(("vertices", "forest_edges", "trees", "rounds")):
        out[f"{tag}_orient_{name}"] = int(stats[i])
    if world == 1:  # one rank: the single call's result, bit for bit
        ctx.check(lib.rsc_estimate_normals(ctx.h, Vl.ctypes.data, n, k, None, res.ctypes.data, None, None))
        out[f"{tag}_estimate_equals_single_call"] = digest(res) == out[f"{tag}_estimate_digests"][0]
        ctx.check(lib.rsc_orient_normals(ctx.h, Vl.ctypes.data, n, k, None, res.ctypes.data, None, None))
        out[f"{tag}_orient_equals_single_call"] = digest(res) == out[f"{tag}_orient_digests"][0]


sc = scenes.scene_cad()
bench("c4", sc)
del sc
if args.c5_points:
    sc = scenes.scene_lidar(args.c5_points)
    bench("c5", sc)
    del sc

if args.reference and world > 1:
    with open(args.reference) as f:
        ref = json.loads(f.readline())
    out["digests_match_reference"] = all(out[key] == ref.get(f"{key}_{world}")
                                         for key in out if key.endswith("_digests"))
if args.shared_gpu:
    lib.rsc_ctx_set_allreduce(ctx.h, None, None)
else:
    shard.detach_comm(ctx)
if rank == 0:
    line = json.dumps(out)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")
dist.barrier()
dist.destroy_process_group()
