"""rsc_estimate_normals_shard / rsc_orient_normals_shard: every rank passes its rows of a cloud and gets its rows of
the single call's result back, bit for bit.  Two or three processes share cuda:0 and sum their buffers through a
host-staged gloo all-reduce (shard.attach_comm(..., comm="host")); NCCL refuses two ranks on one device, so the
library's NCCL path is checked here with one rank (the all-reduce accounting).

One process group per world size runs every case of that size, and rank 0 compares each against the single call in
the same process; the tests read the verdicts."""
import ctypes as C
import os
import sys

import numpy as np
import pytest
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pytestmark = pytest.mark.gpu

K = 16
VIEWPOINT = (10.0, -20.0, 150.0)


def _mixed(with_bad_rows: bool):
    """~40 k points of scene_mixed; with_bad_rows: NaN / Inf rows and a block of 200 coincident points"""
    from ransac_jl_b200 import scenes

    sc = scenes.scene_mixed(81, 40_000, noise_frac=0.002, jitter_deg=1.0, outlier_frac=0.1, counts=(3, 1, 1, 1))
    v, nrm = sc.vertices.astype(np.float32).copy(), sc.normals.astype(np.float32).copy()
    if with_bad_rows:
        v[100] = np.nan
        v[2000, 1] = np.inf
        v[30000, 2] = -np.inf
        v[5000:5200] = v[5000]
    return v, nrm


def _random_signs(nrm, seed=3):
    s = np.where(np.random.default_rng(seed).random(len(nrm)) < 0.5, -1.0, 1.0).astype(np.float32)
    return nrm * s[:, None]


def _tiny(n):
    return np.random.default_rng(100 + n).normal(size=(n, 3)).astype(np.float32)


def _ranges_two(n):
    h = n // 2
    return [(0, h), (h, n)]


def _ranges_three_empty_middle(n):
    a = 12_345
    return [(0, a), (a, a), (a, n)]


def _estimate_cases(world):
    from ransac_jl_b200 import shard

    v, _ = _mixed(True)
    n = len(v)
    if world == 2:
        yield "estimate_aligned_vp", v, shard.partition(n, 2), VIEWPOINT
        yield "estimate_aligned_novp", v, shard.partition(n, 2), None
        for m in (1, 2, K - 1, K, K + 1):
            yield f"estimate_tiny_{m}", _tiny(m), _ranges_two(m), None
    else:
        yield "estimate_unaligned_empty_vp", v, _ranges_three_empty_middle(n), VIEWPOINT
        yield "estimate_unaligned_empty_novp", v, _ranges_three_empty_middle(n), None


def _orient_cases(world):
    from ransac_jl_b200 import shard

    v, nrm = _mixed(True)
    n = len(v)
    given = _random_signs(nrm)
    given[7] = 0.0  # a zero normal and a NaN normal join no tree
    given[8, 0] = np.nan
    if world == 2:
        yield "orient_aligned_given", v, given, shard.partition(n, 2)
        yield "orient_aligned_null", v, None, shard.partition(n, 2)
        for m in (1, 2, K - 1, K, K + 1):
            yield f"orient_tiny_{m}", _tiny(m), None, _ranges_two(m)
    else:
        yield "orient_unaligned_empty_given", v, given, _ranges_three_empty_middle(n)
        yield "orient_unaligned_empty_null", v, None, _ranges_three_empty_middle(n)


def _refusal_cases(n):
    """name -> per-rank (global_offset, rows, n_global, k, null_output) on two ranks"""
    h = n // 2
    return {
        "refuse_k": [(0, h, n, K, False), (h, n - h, n, 8, False)],
        "refuse_n_global": [(0, h, n, K, False), (h, n - h, n + 1, K, False)],
        "refuse_overlap": [(0, h + 10, n, K, False), (h, n - h, n, K, False)],
        "refuse_gap": [(0, h - 10, n, K, False), (h, n - h, n, K, False)],
        "refuse_shifted": [(0, h, n, K, False), (h - 10, n - h, n, K, False)],  # the sum of n is right: coverage
        "refuse_null_output": [(0, h, n, K, False), (h, n - h, n, K, True)],
    }


def _worker(rank, world, port, q):
    try:
        _cases_on_rank(rank, world, port, q)
    except BaseException:
        import traceback

        q.put({"rank": rank, "error": traceback.format_exc()})
        raise


def _cases_on_rank(rank, world, port, q):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    sys.path.insert(0, ROOT)
    import torch.distributed as dist

    dist.init_process_group("gloo", rank=rank, world_size=world)
    import ransac_jl_b200 as R
    from ransac_jl_b200 import shard
    from ransac_jl_b200._lib import RSC_E_ARG, Context, lib

    ctx = Context.get(0)
    shard.attach_comm(ctx, comm="host")
    ref = Context(0)  # the single calls, on a context without a communicator
    verdicts = {}

    def gather(x):
        parts = [None] * world
        dist.all_gather_object(parts, x)
        return parts

    def verdict(name, problems):
        if rank == 0:
            verdicts[name] = "; ".join(problems) or None

    for name, v, ranges, vp in _estimate_cases(world):
        lo, hi = ranges[rank]
        nrm, nbr = R.estimate_normals(v[lo:hi], k=K, viewpoint=vp, ctx=ctx, return_neighbours=True,
                                      shard=(lo, len(v)))
        pairs = C.c_int64()
        xl, scratch = np.ascontiguousarray(v[lo:hi]), np.empty((hi - lo, 3), np.float32)
        ctx.check(lib.rsc_estimate_normals_shard(ctx.h, xl.ctypes.data, hi - lo, lo, len(v), K, None, scratch.ctypes.data,
                                                 None, C.byref(pairs)))
        parts = gather((nrm, nbr, pairs.value))
        if rank == 0:
            problems = []
            want, wnbr = R.estimate_normals(v, k=K, viewpoint=vp, ctx=ref, return_neighbours=True)
            wpairs, wscratch = C.c_int64(), np.empty_like(v)
            ref.check(lib.rsc_estimate_normals(ref.h, v.ctypes.data, len(v), K, None, wscratch.ctypes.data, None,
                                               C.byref(wpairs)))
            got = np.concatenate([p[0] for p in parts])
            if got.view(np.uint32).tobytes() != want.view(np.uint32).tobytes():
                problems.append(f"normals differ in {int((got.view(np.uint32) != want.view(np.uint32)).any(1).sum())} rows")
            if not np.array_equal(np.concatenate([p[1] for p in parts]), wnbr):
                problems.append("neighbour lists differ")
            if sum(p[2] for p in parts) != wpairs.value:
                problems.append(f"pairs {sum(p[2] for p in parts)} != {wpairs.value}")
            verdict(name, problems)

    for name, v, given, ranges in _orient_cases(world):
        lo, hi = ranges[rank]
        out, edges, stats = R.orient_normals(v[lo:hi], None if given is None else given[lo:hi], k=K, ctx=ctx,
                                             return_tree=True, shard=(lo, len(v)))
        parts = gather((out, edges, stats))
        if rank == 0:
            problems = []
            want, wedges, wstats = R.orient_normals(v, given, k=K, ctx=ref, return_tree=True)
            got = np.concatenate([p[0] for p in parts])
            if got.view(np.uint32).tobytes() != want.view(np.uint32).tobytes():
                problems.append("normals differ")
            for r, p in enumerate(parts):
                if not np.array_equal(p[1], wedges) or p[2] != wstats:
                    problems.append(f"rank {r}: forest {p[2]} != {wstats}")
            verdict(name, problems)

    v, _ = _mixed(False)
    for name, per_rank in (_refusal_cases(len(v)) if world == 2 else {}).items():
        off, rows, n_global, k, null_out = per_rank[rank]
        xyz = np.ascontiguousarray(v[off:off + rows])
        out = np.empty((rows, 3), np.float32)
        rc = lib.rsc_estimate_normals_shard(ctx.h, xyz.ctypes.data, rows, off, n_global, k, None,
                                            None if null_out else out.ctypes.data, None, None)
        msg = lib.rsc_last_error(ctx.h).decode()
        rc_o = lib.rsc_orient_normals_shard(ctx.h, xyz.ctypes.data, rows, off, n_global, k, None,
                                            None if null_out else out.ctypes.data, None, None)
        parts = gather((rc, rc_o, msg, null_out))
        if rank == 0:
            problems = [f"rank {r}: rc {p[0]} / {p[1]}" for r, p in enumerate(parts) if (p[0], p[1]) != (RSC_E_ARG, RSC_E_ARG)]
            problems += [f"rank {r}: {p[2]!r} does not name its NULL output" for r, p in enumerate(parts)
                         if p[3] and "NULL" not in p[2]]
            verdict(name, problems)

    # a refused call leaves the communicator usable: the next call on the same ranks succeeds
    lo, hi = shard.partition(len(v), world)[rank] if world == 2 else _ranges_three_empty_middle(len(v))[rank]
    R.estimate_normals(v[lo:hi], k=K, ctx=ctx, shard=(lo, len(v)))

    if world == 2:  # orient_normals(shard=...) -> ShardedCloud -> ransac() -> gather_extracted
        n = len(v)
        params = R.ransacparameters(iteration={"tau": 400, "minsubsetN": 128, "itermax": 120})
        subsets = R.makesubsets(n, 4, np.random.default_rng(1234))
        lo, hi = shard.partition(n, world)[rank]
        nl = R.orient_normals(v[lo:hi], k=K, ctx=ctx, shard=(lo, n))
        pc = shard.ShardedCloud(v[lo:hi], nl, subsets, (lo, hi), n, comm="host")
        ex = shard.gather_extracted(R.ransac(pc, params, True, seed=99)[0])
        if rank == 0:
            pc1 = R.RANSACCloud(v, R.orient_normals(v, k=K, ctx=ref), subsets, ctx=ref)
            want = R.ransac(pc1, params, True, seed=99)[0]
            problems = [] if len(want) == len(ex) >= 3 else [f"{len(ex)} shapes, single call {len(want)}"]
            for a, b in zip(ex, want):
                if list(a.shape.to_cand().p) != list(b.shape.to_cand().p) or not np.array_equal(a.inpoints, b.inpoints):
                    problems.append("a shape or its inliers differ")
            verdict("end_to_end", problems)
            pc1.close()
        pc.close()

    if rank == 0:
        q.put(verdicts)
    shard.detach_comm(ctx)
    dist.barrier()
    dist.destroy_process_group()


_RESULTS = {}


def _run(world):
    """every case of `world` ranks sharing cuda:0, once per session; -> {case: None or the problems}"""
    if world in _RESULTS:
        return _RESULTS[world]
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 31600 + (os.getpid() + world) % 2000
    procs = [ctx.Process(target=_worker, args=(rk, world, port, q)) for rk in range(world)]
    for p in procs:
        p.start()
    import queue as _queue

    res = None
    for _ in range(120):  # a crashed or stuck worker must not leave the test waiting for the queue
        try:
            res = q.get(timeout=5)
            break
        except _queue.Empty:
            if any(p.exitcode not in (None, 0) for p in procs):
                break
    for p in procs:
        p.join(120)
    stuck = [p for p in procs if p.exitcode is None]
    for p in stuck:
        p.kill()
        p.join()
    assert not stuck, f"a rank did not finish: {res}"
    assert res is not None and "error" not in res, res
    assert all(p.exitcode == 0 for p in procs), [p.exitcode for p in procs]
    _RESULTS[world] = res
    return res


@pytest.mark.parametrize("case", ["estimate_aligned_vp", "estimate_aligned_novp"] +
                         [f"estimate_tiny_{m}" for m in (1, 2, K - 1, K, K + 1)])
def test_estimate_two_ranks_equals_single_call(case):
    assert _run(2)[case] is None


@pytest.mark.parametrize("case", ["estimate_unaligned_empty_vp", "estimate_unaligned_empty_novp"])
def test_estimate_three_ranks_unaligned_with_empty_rank(case):
    assert _run(3)[case] is None


@pytest.mark.parametrize("case", ["orient_aligned_given", "orient_aligned_null"] +
                         [f"orient_tiny_{m}" for m in (1, 2, K - 1, K, K + 1)])
def test_orient_two_ranks_equals_single_call(case):
    assert _run(2)[case] is None


@pytest.mark.parametrize("case", ["orient_unaligned_empty_given", "orient_unaligned_empty_null"])
def test_orient_three_ranks_unaligned_with_empty_rank(case):
    assert _run(3)[case] is None


@pytest.mark.parametrize("case", ["refuse_k", "refuse_n_global", "refuse_overlap", "refuse_gap", "refuse_shifted",
                                  "refuse_null_output"])
def test_disagreeing_ranks_are_all_refused(case):
    assert _run(2)[case] is None


def test_end_to_end_sharded_orientation_feeds_sharded_ransac():
    assert _run(2)["end_to_end"] is None


def test_without_communicator_is_a_state_error():
    import ransac_jl_b200 as R
    from ransac_jl_b200._lib import RSC_E_STATE, Context, RscError

    ctx = Context(0)
    v = _tiny(40)
    with pytest.raises(RscError) as e:
        R.estimate_normals(v, ctx=ctx, shard=(0, 40))
    assert e.value.code == RSC_E_STATE
    with pytest.raises(RscError) as e:
        R.orient_normals(v, ctx=ctx, shard=(0, 40))
    assert e.value.code == RSC_E_STATE


def test_library_nccl_single_rank_all_reduce_accounting():
    """one rank on the library's NCCL: 4 all-reduces per call, of the bytes include/rsc.h states, and the single
    call's result"""
    import ransac_jl_b200 as R
    from ransac_jl_b200._lib import Context, lib

    v, nrm = _mixed(True)
    n = len(v)
    ctx = Context(0)
    ident = (C.c_uint8 * 128)()
    ctx.check(lib.rsc_comm_unique_id(ident))
    ctx.check(lib.rsc_ctx_comm_init(ctx.h, ident, 0, 1))

    def stats():
        calls, nbytes = C.c_int64(), C.c_int64()
        ctx.check(lib.rsc_ctx_comm_stats(ctx.h, C.byref(calls), C.byref(nbytes)))
        return calls.value, nbytes.value

    try:
        s0 = stats()
        got, nbr = R.estimate_normals(v, k=K, ctx=ctx, return_neighbours=True, shard=(0, n))
        s1 = stats()
        got2 = R.estimate_normals(v, k=K, ctx=ctx, viewpoint=VIEWPOINT, shard=(0, n))
        s2 = stats()
        ori = R.orient_normals(v, k=K, ctx=ctx, shard=(0, n))
        s3 = stats()
        ori2 = R.orient_normals(v, _random_signs(nrm), k=K, ctx=ctx, shard=(0, n))
        s4 = stats()
    finally:
        ctx.check(lib.rsc_ctx_comm_destroy(ctx.h))
    check = 104 + 4
    assert (s1[0] - s0[0], s1[1] - s0[1]) == (4, check + (16 + 12 + 8 * K) * n)
    assert (s2[0] - s1[0], s2[1] - s1[1]) == (4, check + (16 + 12) * n)
    assert (s3[0] - s2[0], s3[1] - s2[1]) == (4, check + (28 + 4 * K) * n)
    assert (s4[0] - s3[0], s4[1] - s3[1]) == (4, check + (28 + 4 * K) * n)
    ref = Context(0)
    want, wnbr = R.estimate_normals(v, k=K, ctx=ref, return_neighbours=True)
    assert got.tobytes() == want.tobytes() and np.array_equal(nbr, wnbr)
    assert got2.tobytes() == R.estimate_normals(v, k=K, ctx=ref, viewpoint=VIEWPOINT).tobytes()
    assert ori.tobytes() == R.orient_normals(v, k=K, ctx=ref).tobytes()
    assert ori2.tobytes() == R.orient_normals(v, _random_signs(nrm), k=K, ctx=ref).tobytes()
