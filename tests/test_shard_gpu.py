"""Multi-rank runs of the device loop on ONE GPU: two processes share cuda:0 and sum their buffers
through a host-staged gloo all-reduce (rsc_ctx_set_allreduce) -- NCCL refuses two ranks on one device,
the library's own NCCL path is exercised by bench.py / tools/ransac_multi.py on multi-GPU boxes.

  * sharded storage (rsc_cloud_create_shard): every rank holds half of the cloud, minimal sets come from
    the replicated enabled mask, coordinates are gathered from their owners, inlier lists stay
    distributed -- the joined result equals the C oracle's loop (and so the single-GPU loop);
  * replicated storage with a cloud smaller than 2048 x ranks: one rank's range is empty and it still
    joins every all-reduce (ADVICE round 1);
  * replicated storage with each extension switch of the loop (progressive scoring, the cell sampler, the
    least-squares refit, the bitmap filter, the host-walked decision, RSC_LOOP_CULL=2, K5's masked form): every
    rank scores its slice of the newly disabled points after an extraction and the hits are all-reduced, and the
    result equals the single-process run of the same configuration."""
import os
import sys

import numpy as np
import pytest
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pytestmark = pytest.mark.gpu


def _scene(which):
    from ransac_jl_b200 import scenes

    if which == "c1":
        return scenes.scene_c1(), 2, {}, 4321
    if which == "tiny":
        sc = scenes.scene_c1()
        keep = np.random.default_rng(5).permutation(len(sc.vertices))[:1500]
        return scenes.Scene(sc.vertices[keep], sc.normals[keep], None, sc.primitives), 2, {"tau": 50, "itermax": 60}, 11
    return (scenes.scene_mixed(81, 40_000, noise_frac=0.002, jitter_deg=1.0, outlier_frac=0.1, counts=(3, 1, 1, 1)), 4,
            {"tau": 400, "minsubsetN": 128, "itermax": 120}, 99)


# replicated runs with an extension switch: (environment, ransac() keywords)
SWITCHES = {
    "progressive": ({}, {"progressive": True}),
    "octree_lw1": ({}, {"sampler": "octree", "lw_period": 1}),
    "octree_lw16": ({}, {"sampler": "octree", "lw_period": 16}),
    "lsq": ({}, {"lsq": True}),
    "bitmap": ({}, {"bitmap": (1.5, False)}),
    "hostwalk": ({"RSC_LOOP_HOSTWALK": "1"}, {}),
    # (a ranged run never takes the culled scorer, which needs the whole subset's Morton view: this case compares the
    # dense ranged run with the culled single-process run)
    "loop_cull2": ({"RSC_LOOP_CULL": "2"}, {}),
    "k5_masked": ({"RSC_K5_MASKED": "1"}, {}),
}


def _run_switch(R, pc, params, seed, switch):
    """ransac() under one entry of SWITCHES (its environment is set by the caller); -> (extracted, info)"""
    _, kw = SWITCHES[switch] if switch else ({}, {})
    if kw.get("sampler") == "octree":
        pc.build_cells(8)
    ex, _ = R.ransac(pc, params, True, seed=seed, **kw)
    lw = getattr(pc, "levelweight", None)
    info = {"iterations": pc.last_run_iterations, "refined": pc.last_refined,
            "levelweight": None if lw is None or not kw.get("sampler") else np.asarray(lw).copy()}
    return ex, info


def _worker(rank, world, port, which, layout, q, switch=None):
    for k, v in (SWITCHES[switch][0] if switch else {}).items():
        os.environ[k] = v
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    sys.path.insert(0, ROOT)
    import torch.distributed as dist

    dist.init_process_group("gloo", rank=rank, world_size=world)
    import ransac_jl_b200 as R
    from ransac_jl_b200 import shard

    sc, r, itp, seed = _scene(which)
    n = len(sc.vertices)
    params = R.ransacparameters(iteration=itp)
    subsets = R.makesubsets(n, r, np.random.default_rng(1234))
    if layout == "shard":
        lo, hi = shard.partition(n, world)[rank]
        pc = shard.ShardedCloud(sc.vertices[lo:hi], sc.normals[lo:hi], subsets, (lo, hi), n, comm="host")
        ex, _ = R.ransac(pc, params, True, seed=seed)
        assert all(len(e.inpoints) == 0 or (e.inpoints.min() >= lo and e.inpoints.max() < hi) for e in ex)
        local_en = pc.isenabled
        totals = [e.total for e in ex]
        ex = shard.gather_extracted(ex)
        info = None
        parts = [None] * world
        dist.all_gather_object(parts, local_en)
        enabled = np.concatenate(parts)
    else:
        pc = R.RANSACCloud(sc.vertices, sc.normals, subsets)
        sh = shard.ShardedContext(pc, comm="host")
        ex, info = _run_switch(R, pc, params, seed, switch)
        enabled = pc.isenabled
        totals = [e.total for e in ex]
        sh.close()
    if rank == 0:
        q.put(([(e.shape.to_cand().type, bool(e.shape.to_cand().outwards), list(e.shape.to_cand().p), e.inpoints) for e in ex],
               enabled, totals, pc.last_run_syncs, pc.last_run_batches, info))
    dist.barrier()
    dist.destroy_process_group()


def _two_ranks(which, layout, switch=None):
    """runs _worker on two ranks sharing cuda:0; -> rank 0's result"""
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29600 + os.getpid() % 2000
    procs = [ctx.Process(target=_worker, args=(rk, 2, port, which, layout, q, switch)) for rk in range(2)]
    for p in procs:
        p.start()
    import queue as _queue

    res = None
    for _ in range(120):  # a crashed worker must not leave the test waiting for the queue
        try:
            res = q.get(timeout=5)
            break
        except _queue.Empty:
            if any(p.exitcode not in (None, 0) for p in procs):
                break
    for p in procs:
        p.join(120)
        assert p.exitcode == 0
    assert res is not None
    return res


def _equal_c_oracle(which, got, enabled, totals):
    from oracle import c_oracle
    import ransac_jl_b200 as R
    from tests.helpers import oracle_params

    sc, r, itp, seed = _scene(which)
    subsets = R.makesubsets(len(sc.vertices), r, np.random.default_rng(1234))
    want, en, info = c_oracle.ransac(sc.vertices, sc.normals, subsets[0], oracle_params(R.ransacparameters(iteration=itp)), seed)
    assert len(got) == len(want) and len(want) >= 2
    for g, w, tot in zip(got, want, totals):
        assert g[0] == w[0] and (g[0] == 0 or g[1] == w[1])
        np.testing.assert_allclose(g[2], w[2], rtol=1e-5, atol=1e-5 * max(1.0, np.abs(w[2]).max()))
        np.testing.assert_array_equal(g[3], w[3])
        assert tot == len(w[3])
    np.testing.assert_array_equal(enabled, en)
    return want


@pytest.mark.parametrize("which,layout", [("c1", "shard"), ("noisy", "shard"), ("tiny", "replicated"), ("noisy", "replicated")])
def test_two_ranks_one_gpu_match_c_oracle(which, layout):
    res = _two_ranks(which, layout)
    got, enabled, totals, syncs, batches, _ = res
    want = _equal_c_oracle(which, got, enabled, totals)
    # 2 synchronisations per batch + 1 per extraction (+ set-up)
    assert syncs <= 2 * batches + len(want) + 8


@pytest.mark.parametrize("which,switch", [("noisy", s) for s in SWITCHES] +
                         [("tiny", "progressive"), ("tiny", "octree_lw16"), ("tiny", "hostwalk"), ("tiny", "k5_masked")])
def test_two_ranks_replicated_with_extension_switches(which, switch, monkeypatch):
    """replicated storage, two ranks with a point range each: every rank scores its slice of the newly disabled
    subset points after an extraction and the hits are all-reduced.  Shapes (bit for bit), inlier lists, final
    enabled mask, iterations, progressive refinements and level weights equal the single-process run of the same
    configuration; the switches that leave the reference's loop as it is also equal the C oracle's loop.  On the
    tiny scene (1500 points, ranges aligned to 2048) rank 1 owns no point, so its slice of subset 1 is empty."""
    import ransac_jl_b200 as R

    got, enabled, totals, _, _, info = _two_ranks(which, "replicated", switch)
    for k, v in SWITCHES[switch][0].items():
        monkeypatch.setenv(k, v)
    sc, r, itp, seed = _scene(which)
    subsets = R.makesubsets(len(sc.vertices), r, np.random.default_rng(1234))
    pc = R.RANSACCloud(sc.vertices, sc.normals, subsets)
    want, winfo = _run_switch(R, pc, R.ransacparameters(iteration=itp), seed, switch)
    assert len(got) == len(want) and len(want) >= 2
    for g, w, tot in zip(got, want, totals):
        c = w.shape.to_cand()
        assert (g[0], g[1]) == (c.type, bool(c.outwards))
        assert g[2] == list(c.p)  # bit for bit
        np.testing.assert_array_equal(g[3], w.inpoints)
        assert tot == len(w.inpoints)
    np.testing.assert_array_equal(enabled, pc.isenabled)
    assert info["iterations"] == winfo["iterations"] and info["refined"] == winfo["refined"]
    if switch == "progressive":
        assert winfo["refined"] > 0
    if winfo["levelweight"] is not None:
        np.testing.assert_array_equal(info["levelweight"], winfo["levelweight"])
    else:
        assert info["levelweight"] is None
    pc.close()
    # environment-only switches run the reference's loop: the C oracle's too.  The keyword switches (progressive
    # scoring, the cell sampler, the least-squares refit, the bitmap filter) change the loop itself; the single-process
    # run they are compared with here is pinned to the NumPy oracle's loop of the same switch by test_progressive.py,
    # test_octree_gpu.py, test_lsq.py and test_bitmap_gpu.py.
    if not SWITCHES[switch][1]:
        _equal_c_oracle(which, got, enabled, totals)


def test_library_nccl_communicator_single_rank():
    """the library's own NCCL path on one GPU: rsc_comm_unique_id + rsc_ctx_comm_init with one rank (libnccl.so.2
    is dlopen-ed here), then the device loop with a point range -- every count / hit / mask exchange goes through
    ncclAllReduce on the context stream and the result equals the plain run"""
    import ctypes as C

    import ransac_jl_b200 as R
    from ransac_jl_b200 import scenes
    from ransac_jl_b200._lib import lib

    sc, r, itp, seed = _scene("noisy")
    params = R.ransacparameters(iteration=itp)
    ctx = R.Context(0)  # a context of its own: the communicator stays with it
    pc = R.RANSACCloud(sc.vertices, sc.normals, r, ctx=ctx)
    plain, _ = R.ransac(pc, params, True, seed=seed)
    ident = (C.c_uint8 * 128)()
    ctx.check(lib.rsc_comm_unique_id(ident))
    ctx.check(lib.rsc_ctx_comm_init(ctx.h, ident, 0, 1))
    try:
        ctx.check(lib.rsc_cloud_set_range(pc.handle, 0, pc.size))
        viacomm, _ = R.ransac(pc, params, True, seed=seed)
        calls, nbytes = C.c_int64(), C.c_int64()
        ctx.check(lib.rsc_ctx_comm_stats(ctx.h, C.byref(calls), C.byref(nbytes)))
    finally:
        ctx.check(lib.rsc_ctx_comm_destroy(ctx.h))
    assert calls.value >= 2 * len(plain) and nbytes.value > 0
    assert len(plain) == len(viacomm) >= 3
    for a, b in zip(plain, viacomm):
        assert list(a.shape.to_cand().p) == list(b.shape.to_cand().p)
        np.testing.assert_array_equal(a.inpoints, b.inpoints)
    pc.close()
