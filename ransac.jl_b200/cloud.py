"""RANSACCloud: host-side mirror of the reference's point-cloud container (src/octree.jl:37-138).

The cloud lives in HBM as SoA float32 behind an `rsc_cloud` handle; `subsets` is the random
partition the reference builds with `randperm` (octree.jl:129-135) and subset 1 -- the only one the
reference ever scores (iterations.jl:95) -- is uploaded eagerly as a gathered contiguous copy.
`isenabled` is read from / written to the device bitmask (BitArray.chunks layout).

The octree of the reference is not built: its level weights are degenerate (octree.jl:82-84 swaps
levelweight/levelscore), so every minimal set is drawn from the root cell = all enabled points.
"""
from __future__ import annotations

import ctypes as C
from typing import List, Optional, Sequence, Union

import numpy as np

from . import _lib
from ._lib import Context, lib


def makesubsets(n: int, numofsubsets: int, rng: np.random.Generator) -> List[np.ndarray]:
    """octree.jl:129-135: randperm split into numofsubsets pieces, the last takes the remainder."""
    assert numofsubsets > 0, "At least 1 subset please!"
    ssl = n // numofsubsets
    alls = rng.permutation(n).astype(np.int64)
    subs = [alls[i * ssl : (i + 1) * ssl] for i in range(numofsubsets - 1)]
    subs.append(alls[(numofsubsets - 1) * ssl :])
    return subs


class RANSACCloud:
    """RANSACCloud(vertices, normals, numofsubsets | subsets; force_eltype=None, exact=False).

    vertices/normals: (N,3) arrays (float32 or float64; the device copy is float32).
    exact=True with float64 input keeps the float64 coordinates on the device too
    (rsc_cloud_create_f64_exact, +48 B/point): every decision and fit is then the float64 one of
    the caller's unrounded points.  float32 input is exact already.  Not with `shard=`.
    """

    def __init__(
        self,
        vertices,
        normals,
        subsets: Union[int, Sequence[np.ndarray]] = 1,
        force_eltype=None,
        device: int = 0,
        seed: int = 1234,
        shard: Optional[tuple] = None,
        ctx: Optional[Context] = None,
        exact: bool = False,
    ):
        if exact and shard is not None:
            raise ValueError("RANSACCloud: exact=True does not support sharded storage (shard=)")
        v = np.asarray(vertices)
        n = np.asarray(normals)
        assert v.shape == n.shape, "Every point must have a normal."
        assert v.ndim == 2 and v.shape[1] == 3
        if force_eltype is not None:
            v = v.astype(force_eltype)
            n = n.astype(force_eltype)
        if v.dtype not in (np.float32, np.float64):
            v = v.astype(np.float64)
            n = n.astype(np.float64)
        self.vertices = np.ascontiguousarray(v)
        self.normals = np.ascontiguousarray(n.astype(v.dtype, copy=False))
        self.size = int(v.shape[0])
        if isinstance(subsets, (int, np.integer)):
            # a shard draws the subsets of the WHOLE cloud (global indices, the same on every rank)
            self.subsets = makesubsets(self.size if shard is None else int(shard[1]), int(subsets), np.random.default_rng(seed))
        else:
            self.subsets = [np.ascontiguousarray(s, dtype=np.int64) for s in subsets]
        self.ctx = ctx if ctx is not None else Context.get(device)
        self._h = C.c_void_p()
        self.is_shard = False
        self.global_offset, self.n_global = 0, self.size
        if shard is not None:
            self.global_offset, self.n_global = int(shard[0]), int(shard[1])
            if self.vertices.dtype != np.float32:
                self.vertices = self.vertices.astype(np.float32)
                self.normals = self.normals.astype(np.float32)
            rc = lib.rsc_cloud_create_shard(
                self.ctx.h, self.vertices.ctypes.data, self.normals.ctypes.data, self.size,
                self.global_offset, self.n_global, C.byref(self._h))
            self.is_shard = self.n_global > self.size
        elif self.vertices.dtype == np.float32:
            rc = lib.rsc_cloud_create(self.ctx.h, self.vertices.ctypes.data, self.normals.ctypes.data, self.size, C.byref(self._h))
        elif exact:
            rc = lib.rsc_cloud_create_f64_exact(self.ctx.h, self.vertices.ctypes.data, self.normals.ctypes.data, self.size, C.byref(self._h))
        else:
            rc = lib.rsc_cloud_create_f64(self.ctx.h, self.vertices.ctypes.data, self.normals.ctypes.data, self.size, C.byref(self._h))
        self.ctx.check(rc)
        self._uploaded = set()
        if len(self.subsets) and len(self.subsets[0]):
            self.upload_subset(0)

    # -- device handle ------------------------------------------------------------------
    @property
    def handle(self):
        return self._h

    @property
    def exact(self) -> bool:
        """True when every device decision and fit is the float64 one of the points as given
        (float32 input, or float64 input with exact=True)."""
        return self.vertices.dtype == np.float32 or bool(lib.rsc_cloud_is_exact(self._h))

    def upload_subset(self, subset_id: int):
        if subset_id in self._uploaded:
            return
        s = self.subsets[subset_id]
        self.ctx.check(lib.rsc_cloud_set_subset(self._h, subset_id, s.ctypes.data, len(s)))
        self._uploaded.add(subset_id)

    # -- flattened octree (extension, SURVEY 8(f)-1) --------------------------------------
    def build_cells(self, nlevels: int = 8):
        """Morton-ordered octree cells for the level-weighted sampler (replaces RegionTrees,
        octree.jl:158-244): level 1 = bounding box, every level halves each axis."""
        self.ctx.check(lib.rsc_cloud_build_cells(self._h, int(nlevels)))
        self.nlevels = int(nlevels)
        return self

    def get_cells(self):
        """(sorted Morton codes, sorted position -> point index, leafdepth per point)"""
        codes = np.zeros(self.size, np.uint32)
        perm = np.zeros(self.size, np.uint32)
        ld = np.zeros(self.size, np.uint8)
        self.ctx.check(lib.rsc_cloud_get_cells(self._h, codes.ctypes.data, perm.ctypes.data, ld.ctypes.data))
        return codes, perm, ld

    # -- pc.isenabled -------------------------------------------------------------------
    @property
    def isenabled(self) -> np.ndarray:
        words = np.zeros((self.size + 63) // 64, dtype=np.uint64)
        self.ctx.check(lib.rsc_cloud_get_enabled(self._h, words.ctypes.data))
        return np.unpackbits(words.view(np.uint8), bitorder="little")[: self.size].astype(bool)

    @isenabled.setter
    def isenabled(self, mask):
        mask = np.asarray(mask, dtype=bool)
        assert mask.shape == (self.size,)
        nbytes = ((self.size + 63) // 64) * 8
        packed = np.zeros(nbytes, dtype=np.uint8)
        pb = np.packbits(mask, bitorder="little")
        packed[: len(pb)] = pb
        self.ctx.check(lib.rsc_cloud_set_enabled(self._h, packed.ctypes.data))

    def enable_all(self):
        self.ctx.check(lib.rsc_cloud_enable_all(self._h))

    def count_enabled(self) -> int:
        n = lib.rsc_cloud_count_enabled(self._h)
        if n < 0:
            raise _lib.RscError(-2, "rsc_cloud_count_enabled failed")
        return int(n)

    def close(self):
        if self._h:
            lib.rsc_cloud_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __repr__(self):
        return f"RANSACCloud of size {self.size} & {len(self.subsets)} subsets"
