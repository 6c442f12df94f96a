"""Point-range sharding over the GPUs of one box: one process per GPU (include/rsc.h, "point-range
sharding").

`ShardedCloud` is the sharded-storage layout: every rank uploads only its own point range
(`partition`), the library keeps the whole cloud's enabled mask replicated, draws identical Philox
minimal sets on every rank and gathers their coordinates from the owning ranks; per-candidate counts,
K5 hits and the cleared enabled words are summed with NCCL **inside the library**
(`rsc_ctx_comm_init`; torch.distributed only carries the 128-byte NCCL id from rank 0 to the others).
`ShardedContext` is the older replicated-storage layout (whole cloud on every rank + a range per rank),
which also supports the extension switches; it can use the library's NCCL too or a host callback.
`attach_comm` puts either communicator on a bare `Context`, for the sharded normals:

    orient_normals(V[lo:hi], shard=(lo, n), ctx=ctx) -> ShardedCloud(V[lo:hi], N_lo_hi, subsets, (lo, hi), n) -> ransac()
"""
from __future__ import annotations

import ctypes as C
from typing import List, Tuple

import numpy as np

from . import _lib
from ._lib import lib

ALIGN = 2048  # refit CTAs cover 2048 points; score tiles 512


def partition(n: int, world: int, align: int = ALIGN) -> List[Tuple[int, int]]:
    """Contiguous point ranges [lo, hi) per rank: aligned to `align`, covering [0, n) exactly once.
    Trailing ranks may be empty when n is small."""
    blocks = (n + align - 1) // align
    out = []
    for r in range(world):
        lo = (blocks * r // world) * align
        hi = (blocks * (r + 1) // world) * align
        out.append((min(lo, n), min(hi, n)))
    return out


def exchange_comm_id(group=None) -> bytes:
    """The 128-byte NCCL unique id of the library's communicator on every rank: rank 0 of the group draws it
    (rsc_comm_unique_id; needs libnccl.so.2 but no GPU), torch.distributed -- any backend -- broadcasts it."""
    import torch.distributed as dist

    ident = [None]
    if dist.get_rank(group) == 0:
        buf = (C.c_uint8 * 128)()
        rc = lib.rsc_comm_unique_id(buf)
        if rc != 0:
            raise _lib.RscError(rc, "rsc_comm_unique_id failed (libnccl.so.2 not loadable?)")
        ident = [bytes(buf)]
    dist.broadcast_object_list(ident, src=dist.get_global_rank(group, 0) if group is not None else 0, group=group)
    return ident[0]


def init_comm(ctx, group=None) -> None:
    """NCCL communicator of the library on `ctx` (one per process): rank 0 draws the NCCL unique id,
    torch.distributed broadcasts its 128 bytes, every rank calls rsc_ctx_comm_init (collective)."""
    import torch.distributed as dist

    if getattr(ctx, "_comm", False):
        return
    rank, world = dist.get_rank(group), dist.get_world_size(group)
    buf = (C.c_uint8 * 128).from_buffer_copy(exchange_comm_id(group))
    ctx.check(lib.rsc_ctx_comm_init(ctx.h, buf, rank, world))
    ctx._comm = True


def close_comm(ctx) -> None:
    if getattr(ctx, "_comm", False):
        lib.rsc_ctx_comm_destroy(ctx.h)
        ctx._comm = False


class _DevInt32:
    """__cuda_array_interface__ view of a raw device pointer (int32[n])."""

    def __init__(self, ptr: int, n: int):
        self.__cuda_array_interface__ = {"shape": (n,), "typestr": "<i4", "data": (ptr, False), "version": 3}


def ShardedCloud(vertices_local, normals_local, subsets, rank_range: Tuple[int, int], n_global: int, device: int = 0,
                 group=None, comm: str = "nccl"):
    """Sharded storage: a RANSACCloud over this rank's range [lo, hi) of a cloud of n_global points.
    `subsets` = the whole cloud's subsets (global indices, the same on every rank); `comm` = "nccl" (the
    library's own communicator) or "callback" (torch.distributed through rsc_ctx_set_allreduce)."""
    from .cloud import RANSACCloud

    lo, hi = rank_range
    assert len(vertices_local) == hi - lo
    pc = RANSACCloud(vertices_local, normals_local, subsets, device=device, shard=(lo, n_global))
    if comm == "nccl":
        init_comm(pc.ctx, group)
    else:
        pc._sharded = ShardedContext(pc, group, set_range=False, comm=comm)
    return pc


def attach_comm(ctx, group=None, comm: str = "nccl") -> None:
    """Puts a communicator on a bare `Context`, as the collective calls on it need (`estimate_normals(...,
    shard=...)`, `orient_normals(..., shard=...)`, sharded clouds).  comm="nccl": the library's own NCCL
    (`init_comm`); "callback": a host callback into torch.distributed on device tensors (rsc_ctx_set_allreduce);
    "host": the same callback staged through host memory (any torch.distributed backend, e.g. gloo: ranks may then
    share a GPU)."""
    if comm == "nccl":
        init_comm(ctx, group)
        return
    import torch
    import torch.distributed as dist

    ext = torch.cuda.ExternalStream(ctx.stream, device=torch.device("cuda", ctx.device))
    host_staged = comm == "host"

    def _allreduce(user, ptr, count, stream):
        try:
            t = torch.as_tensor(_DevInt32(ptr, count), device=torch.device("cuda", ctx.device))
            with torch.cuda.stream(ext):
                if host_staged:
                    h = t.cpu()
                    dist.all_reduce(h, group=group)
                    t.copy_(h)
                else:
                    dist.all_reduce(t, group=group)
            return 0
        except Exception as e:  # never let an exception cross the C boundary
            print(f"[rsc] all-reduce callback failed: {e!r}")
            return 1

    ctx._allreduce_cb = _lib.ALLREDUCE_FN(_allreduce)  # keep alive while installed
    ctx.check(lib.rsc_ctx_set_allreduce(ctx.h, C.cast(ctx._allreduce_cb, C.c_void_p), None))


def detach_comm(ctx) -> None:
    """Removes what `attach_comm` put on `ctx`."""
    if getattr(ctx, "_comm", False):
        close_comm(ctx)
    else:
        lib.rsc_ctx_set_allreduce(ctx.h, None, None)
        ctx._allreduce_cb = None


class ShardedContext:
    """Replicated storage: installs an all-reduce (host callback into torch.distributed, or the library's
    NCCL with comm="nccl") on a context and the rank's point range on a cloud.  comm="host" stages the
    callback through host memory (any torch.distributed backend, e.g. gloo: ranks may then share a GPU)."""

    def __init__(self, pc, group=None, set_range: bool = True, comm: str = "callback"):
        import torch.distributed as dist

        self.pc = pc
        self.rank = dist.get_rank(group)
        self.world = dist.get_world_size(group)
        self.range = partition(pc.size, self.world)[self.rank]
        self.comm = comm
        attach_comm(pc.ctx, group, comm)
        if set_range:
            lo, hi = self.range  # an empty range (lo == hi) is a rank that only joins the all-reduces
            pc.ctx.check(lib.rsc_cloud_set_range(pc.handle, lo, hi))
            pc.ranged = True  # (ransac() keeps such a cloud out of rsc_ransac_run_user)

    def close(self):
        detach_comm(self.pc.ctx)


def gather_extracted(extracted, group=None):
    """Sharded storage leaves every shape's inlier list distributed (each rank holds the ascending
    indices of its range): concatenate the parts in rank order on every rank (torch.distributed)."""
    import torch.distributed as dist

    from .shapes import ExtractedShape

    parts = [None] * dist.get_world_size(group)
    dist.all_gather_object(parts, [e.inpoints for e in extracted], group=group)
    return [ExtractedShape(e.shape, np.concatenate([p[i] for p in parts])) for i, e in enumerate(extracted)]
