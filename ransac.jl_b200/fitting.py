"""Host-side mirror of the reference's per-shape operator API and candidate bookkeeping:
`fit`, `scorecandidate(s)`, `refit`, `forcefitshapes`, `IterationCandidates`, `findhighestscore`
(src/fitting.jl:15-221 and src/shapes/*.jl).  Every built-in shape routes to the CUDA library
through the C ABI; there is no Python/NumPy implementation of the math here.  User-defined shapes
with `cuda_source` score and refit on the device too (rsc_user_score, rsc_user_refit_extract).
"""
from __future__ import annotations

import ctypes as C
from typing import List, Optional, Sequence, Tuple

import numpy as np

from . import _lib
from ._lib import lib
from .cloud import RANSACCloud
from .confidence import ConfidenceInterval, estimatescore, estimatescore_f64, isoverlap
from .params import to_c
from .shapes import SHAPE_KIND, ExtractedShape, FittedShape, device_fit, from_cand, on_device, pack_cands, user_cand


# ---- fit (fitting.jl:30; plane.jl:33, sphere.jl:87, cylinder.jl:135, cone.jl:123) ------------
def fit_points(pc: RANSACCloud, p, n, params) -> Tuple[List[FittedShape], np.ndarray]:
    """Batched forcefitshapes!: p, n are (S, k, 3); returns candidates in (set, shape_types) order
    and the source set of each."""
    p = np.ascontiguousarray(p, dtype=np.float64)
    n = np.ascontiguousarray(n, dtype=np.float64)
    assert p.shape == n.shape and p.ndim == 3 and p.shape[2] == 3, "Size must be the same."
    S, k = p.shape[0], p.shape[1]
    assert k > 2, "At least 3 point is needed."
    cp = to_c(params)
    cap = max(S * cp.n_shape_types, 1)
    out = (_lib.rsc_cand * cap)()
    out_set = np.zeros(cap, dtype=np.int32)
    out_n = C.c_int32()
    pc.ctx.check(lib.rsc_fit_points(pc.ctx.h, C.byref(cp), p.ctypes.data, n.ctypes.data, S, k, out, out_set.ctypes.data, C.byref(out_n)))
    return [from_cand(out[i]) for i in range(out_n.value)], out_set[: out_n.value].copy()


def fit(shape_type, p, n, pc: RANSACCloud, params) -> Optional[FittedShape]:
    """fit(::Type{S}, p, n, pc, params): one shape type, one minimal set -> shape or None."""
    one = dict(params)
    one["iteration"] = dict(params["iteration"], shape_types=[shape_type])
    shapes, _ = fit_points(pc, np.asarray(p, dtype=np.float64)[None], np.asarray(n, dtype=np.float64)[None], one)
    return shapes[0] if shapes else None


def fit_batch(pc: RANSACCloud, idx, params) -> Tuple[List[FittedShape], np.ndarray]:
    """forcefitshapes! for S minimal sets given as (S, drawN) point indices into the cloud."""
    idx = np.ascontiguousarray(idx, dtype=np.int64)
    S = idx.shape[0]
    cp = to_c(params)
    assert idx.shape[1] == cp.drawN
    cap = max(S * cp.n_shape_types, 1)
    out = (_lib.rsc_cand * cap)()
    out_set = np.zeros(cap, dtype=np.int32)
    out_n = C.c_int32()
    pc.ctx.check(lib.rsc_fit_batch(pc.handle, C.byref(cp), idx.ctypes.data, S, out, out_set.ctypes.data, C.byref(out_n)))
    return [from_cand(out[i]) for i in range(out_n.value)], out_set[: out_n.value].copy()


def sample_fit(pc: RANSACCloud, params, seed: int, set0: int, S: int):
    """samplepointcloud4! + forcefitshapes! for S minimal sets (fitting.jl:383-430, :165-173)."""
    cp = to_c(params)
    cap = max(S * cp.n_shape_types, 1)
    out = (_lib.rsc_cand * cap)()
    out_set = np.zeros(cap, dtype=np.int32)
    out_idx = np.zeros((S, cp.drawN), dtype=np.int64)
    out_n = C.c_int32()
    pc.ctx.check(lib.rsc_sample_fit(pc.handle, C.byref(cp), seed, set0, S, out, out_set.ctypes.data, out_idx.ctypes.data, C.byref(out_n)))
    return [from_cand(out[i]) for i in range(out_n.value)], out_set[: out_n.value].copy(), out_idx


def fit_order(pc: RANSACCloud, types, params):
    """rsc_shape_slot[] of a fit order: built-in kinds, and user classes that fit on the device (`device_fit`) under
    their compiled type ids with their `device_constants`.  Returns (slots, {type id: class})."""
    if len(types) > _lib.RSC_MAX_ORDER:
        raise ValueError(f"at most {_lib.RSC_MAX_ORDER} shape types in one fit order")
    slots = (_lib.rsc_shape_slot * max(len(types), 1))()
    classes = {}
    for i, t in enumerate(types):
        if t in SHAPE_KIND:
            slots[i].type = SHAPE_KIND[t]
            continue
        if not device_fit(t):
            raise TypeError(f"{t.__name__} does not fit on the device (cuda_source with rsc_user_fit, from_device_record)")
        k = _user_constants(t, params)
        slots[i].type = pc.ctx.user_type(t)
        slots[i].nk = len(k)
        slots[i].k[: len(k)] = list(k)
        classes[slots[i].type] = t
    return slots, classes


def shape_from_record(c: _lib.rsc_cand, classes) -> FittedShape:
    """A built-in rsc_cand, or a user record under a type id of `classes` (fit_order) via `from_device_record`."""
    if c.type in classes:
        return classes[c.type].from_device_record(list(c.p), bool(c.outwards))
    return from_cand(c)


def sample_fit_user(pc: RANSACCloud, params, types, seed: int, set0: int, S: int):
    """sample_fit with a mixed fit order (rsc_sample_fit_user): built-ins and device-fitting user classes in the
    order `types`; the candidates come back in (set, position) order.  `types = []` only draws the sets."""
    cp = to_c(_builtin_params(params))
    slots, classes = fit_order(pc, types, params)
    cap = max(S * len(types), 1)
    out = (_lib.rsc_cand * cap)()
    out_set = np.zeros(cap, dtype=np.int32)
    out_idx = np.zeros((S, cp.drawN), dtype=np.int64)
    out_n = C.c_int32()
    pc.ctx.check(lib.rsc_sample_fit_user(pc.handle, C.byref(cp), slots, len(types), seed, set0, S, out, out_set.ctypes.data,
                                         out_idx.ctypes.data, C.byref(out_n)))
    return [shape_from_record(out[i], classes) for i in range(out_n.value)], out_set[: out_n.value].copy(), out_idx


def sample_fit_cells(pc: RANSACCloud, params, seed: int, set0: int, S: int, levelweight):
    """samplepointcloud4! with the level-weighted octree-cell sampler (pc.build_cells first) +
    forcefitshapes!.  Returns (shapes, set of each shape, indices (S, drawN), level of each set)."""
    cp = to_c(params)
    lw = np.ascontiguousarray(levelweight, dtype=np.float64)
    cap = max(S * cp.n_shape_types, 1)
    out = (_lib.rsc_cand * cap)()
    out_set = np.zeros(cap, dtype=np.int32)
    out_idx = np.zeros((S, cp.drawN), dtype=np.int64)
    out_level = np.zeros(S, dtype=np.int32)
    out_n = C.c_int32()
    pc.ctx.check(lib.rsc_sample_fit_cells(pc.handle, C.byref(cp), seed, set0, S, lw.ctypes.data, len(lw), out, out_set.ctypes.data,
                                          out_idx.ctypes.data, out_level.ctypes.data, C.byref(out_n)))
    return [from_cand(out[i]) for i in range(out_n.value)], out_set[: out_n.value].copy(), out_idx, out_level


# ---- scoring (fitting.jl:45,181-190; shapes/*.jl scorecandidate) -------------------------------
def score_counts(pc: RANSACCloud, candidates: Sequence[FittedShape], subsetID: int, params, want_masks=False,
                 compat_flags=None):
    """Raw device scoring: inlier counts (and packed masks) of candidates against subset `subsetID`
    (0-based; -1 = whole cloud)."""
    Cn = len(candidates)
    counts = np.zeros(Cn, dtype=np.int32)
    if Cn == 0:
        return counts, None
    if subsetID >= 0:
        pc.upload_subset(subsetID)
        M = len(pc.subsets[subsetID])
    else:
        M = pc.size
    arr = pack_cands(candidates)
    cp = to_c(params, compat_flags)
    masks = np.zeros((Cn, (M + 31) // 32), dtype=np.uint32) if want_masks else None
    pc.ctx.check(lib.rsc_score(pc.handle, C.byref(cp), arr, Cn, subsetID, counts.ctypes.data, masks.ctypes.data if want_masks else None))
    return counts, masks


def score_counts_culled(pc: RANSACCloud, candidates: Sequence[FittedShape], params, subsetID: int = -1):
    """Extension: the counts of `score_counts(pc, candidates, subsetID, params)` without evaluating the
    (candidate, 128-point Morton tile) pairs that provably hold no compatible point.  subsetID = -1: the whole
    cloud (`rsc_score_culled`; needs `pc.build_cells()`); subsetID >= 0 (0-based, like score_counts): that subset
    (`rsc_score_culled_subset`; sorts a copy of the subset on first use).  Returns (counts, info) with info =
    pairs_total, pairs_survived, kernel_ms."""
    Cn = len(candidates)
    counts = np.zeros(Cn, dtype=np.int32)
    if Cn == 0:
        return counts, {"pairs_total": 0, "pairs_survived": 0, "kernel_ms": 0.0}
    arr = pack_cands(candidates)
    cp = to_c(params)
    tot, sur, ms = C.c_int64(), C.c_int64(), C.c_double()
    if subsetID >= 0:
        pc.ctx.check(lib.rsc_score_culled_subset(pc.handle, C.byref(cp), arr, Cn, subsetID, counts.ctypes.data, C.byref(tot),
                                                 C.byref(sur), C.byref(ms)))
    else:
        pc.ctx.check(lib.rsc_score_culled(pc.handle, C.byref(cp), arr, Cn, counts.ctypes.data, C.byref(tot), C.byref(sur), C.byref(ms)))
    return counts, {"pairs_total": tot.value, "pairs_survived": sur.value, "kernel_ms": ms.value}


def unpack_mask(row: np.ndarray, M: int) -> np.ndarray:
    return np.unpackbits(row.view(np.uint8), bitorder="little")[:M].astype(bool)


def _user_constants(shape_class, params):
    k = np.ascontiguousarray([float(v) for v in shape_class.device_constants(params)], dtype=np.float64)
    if len(k) > 8:
        raise ValueError(f"{shape_class.__name__}.device_constants: at most 8 constants, got {len(k)}")
    return k


def user_score_counts(pc: RANSACCloud, candidates: Sequence[FittedShape], subsetID: int, params, want_masks=False):
    """Raw device scoring of user-defined shapes of ONE class with `cuda_source` (rsc_user_score, the analogue of
    `score_counts`): inlier counts (and packed masks) against subset `subsetID` (0-based; -1 = whole cloud)."""
    Cn = len(candidates)
    counts = np.zeros(Cn, dtype=np.int32)
    if Cn == 0:
        return counts, None
    cls = type(candidates[0])
    if not on_device(cls) or any(type(c) is not cls for c in candidates):
        raise TypeError("user_score_counts: candidates of one user-defined shape class with cuda_source")
    if subsetID >= 0:
        pc.upload_subset(subsetID)
        M = len(pc.subsets[subsetID])
    else:
        M = pc.size
    tid = pc.ctx.user_type(cls)
    arr = (_lib.rsc_cand * Cn)()
    for i, c in enumerate(candidates):
        arr[i] = user_cand(c, tid)
    k = _user_constants(cls, params)
    masks = np.zeros((Cn, (M + 31) // 32), dtype=np.uint32) if want_masks else None
    pc.ctx.check(lib.rsc_user_score(pc.handle, k.ctypes.data, len(k), arr, Cn, subsetID, counts.ctypes.data,
                                    masks.ctypes.data if want_masks else None))
    return counts, masks


def _builtin_params(params):
    it = params["iteration"]
    return dict(params, iteration=dict(it, shape_types=[t for t in it["shape_types"] if t in SHAPE_KIND]))


def scorecandidates(pc: RANSACCloud, candidates: Sequence[FittedShape], subsetID: int, params):
    """scorecandidates!: [(ConfidenceInterval, inpoints)] in input order.  Built-in shapes are scored in ONE
    launch (rsc_score), each user-defined class with `cuda_source` in one launch of its own (rsc_user_score);
    any other user-defined shape calls its own `scorecandidate` (docs/src/newprimitive.md:16)."""
    sub = pc.subsets[subsetID]
    out = [None] * len(candidates)
    groups: dict = {}
    for i, c in enumerate(candidates):
        t = type(c)
        if t in SHAPE_KIND:
            groups.setdefault(None, []).append(i)
        elif on_device(t):
            groups.setdefault(t, []).append(i)
        else:
            out[i] = c.scorecandidate(pc, subsetID, params)
    for cls, idx in groups.items():
        cs = [candidates[i] for i in idx]
        if cls is None:
            counts, masks = score_counts(pc, cs, subsetID, _builtin_params(params), want_masks=True)
        else:
            counts, masks = user_score_counts(pc, cs, subsetID, params, want_masks=True)
        for j, i in enumerate(idx):
            m = unpack_mask(masks[j], len(sub))
            out[i] = (estimatescore(len(sub), pc.size, int(counts[j])), sub[m])
    return out


def scorecandidate(pc: RANSACCloud, candidate: FittedShape, subsetID: int, params):
    """scorecandidate(pc, candidate, subsetID, params) -> (score, inpoints)."""
    return scorecandidates(pc, [candidate], subsetID, params)[0]


def bitmap_filter(s: FittedShape, pc: RANSACCloud, idx, beta: float, eight: bool = False):
    """Extension (the paper's third compatibility criterion, docs/src/ransac.md:106-112; dead code in the
    reference, src/parameterspacebitmap.jl): of the points `idx`, those whose cell of the shape's parameter-space
    bitmap (cell size ~ beta) lies in the largest connected component.  Returns (kept indices, info dict)."""
    idx = np.ascontiguousarray(idx, dtype=np.int64)
    out = np.zeros(max(1, len(idx)), dtype=np.int64)
    n = C.c_int64()
    info = (C.c_int32 * 4)()
    cand = s.to_cand()
    pc.ctx.check(lib.rsc_bitmap_filter(pc.handle, C.byref(cand), float(beta), int(eight), idx.ctypes.data, len(idx), out.ctypes.data,
                                       C.byref(n), info))
    return out[: n.value].copy(), {"nu": info[0], "nv": info[1], "components": info[2], "largest_cells": info[3]}


# ---- refit (fitting.jl:57; shapes/*.jl refit) + invalidate_indexes! (fitting.jl:197) -----------
def refit(s: FittedShape, pc: RANSACCloud, params, disable: bool = False) -> ExtractedShape:
    """Compatible enabled points of the whole cloud (ascending), optionally disabled: rsc_refit_extract for built-in
    shapes, rsc_user_refit_extract for user-defined shapes with `cuda_source`."""
    out = np.zeros(pc.size, dtype=np.int64)
    n = C.c_int64()
    if on_device(type(s)):
        cand = user_cand(s, pc.ctx.user_type(type(s)))
        k = _user_constants(type(s), params)
        pc.ctx.check(lib.rsc_user_refit_extract(pc.handle, k.ctypes.data, len(k), C.byref(cand), out.ctypes.data, C.byref(n),
                                                int(disable)))
        return ExtractedShape(s, out[: n.value].copy())
    cand = s.to_cand()
    cp = to_c(_builtin_params(params))
    pc.ctx.check(lib.rsc_refit_extract(pc.handle, C.byref(cp), C.byref(cand), out.ctypes.data, C.byref(n), int(disable)))
    return ExtractedShape(s, out[: n.value].copy())


def lsq_refit(s: FittedShape, pc: RANSACCloud, params, band: float = 3.0):
    """Extension (SURVEY 8(f)-4): least-squares refit of `s` to the enabled points compatible with it
    inside band * eps -- the refit of the paper, which the reference leaves out
    (docs/src/ransac.md:163-169).  Returns (refined shape, points used, rms distance)."""
    cand, out = s.to_cand(), _lib.rsc_cand()
    cp = to_c(params)
    n, rms = C.c_int64(), C.c_double()
    pc.ctx.check(lib.rsc_refit_lsq(pc.handle, C.byref(cp), C.byref(cand), float(band), C.byref(out), C.byref(n), C.byref(rms)))
    return from_cand(out), n.value, rms.value


def invalidate_indexes(pc: RANSACCloud, indexlist):
    en = pc.isenabled
    en[np.asarray(indexlist, dtype=np.int64) - pc.global_offset] = False
    pc.isenabled = en


# ---- candidate store (fitting.jl:94-158) --------------------------------------------------------
class IterationCandidates:
    """SoA store of (shape, score, inpoints) -- fitting.jl:94-131."""

    def __init__(self):
        self.shapes: List[FittedShape] = []
        self.scores: List[ConfidenceInterval] = []
        self.inpoints: List[np.ndarray] = []
        # progressive scoring (extension): [subsets evaluated, compatible points among them, their size]
        self.evaluated: List[list] = []

    def __len__(self):
        return len(self.shapes)

    def recordscore(self, shape, score, inpoints, subset_size: int = -1):
        self.shapes.append(shape)
        self.scores.append(score)
        self.inpoints.append(inpoints)
        self.evaluated.append([1, len(inpoints), subset_size])
        return self

    def deleteat(self, arg):
        idx = sorted([arg] if np.isscalar(arg) else list(arg), reverse=True)
        for i in idx:
            del self.shapes[i], self.scores[i], self.inpoints[i], self.evaluated[i]
        return self


def refine_progressive(pc: RANSACCloud, A: IterationCandidates, params) -> int:
    """Progressive subset scoring -- what iterations.jl:110 leaves as "TODO: refine if best.overlap"
    (docs/src/ransac.md:137-141; Schnabel et al. 2007, sec. 4.5.1).  While the interval of the best
    candidate overlaps another one (`isoverlap`), the least-evaluated candidates among the best and its
    overlappers are scored on their next subset -- one `rsc_score` launch per round, counts only -- and
    re-estimated from the union of the subsets seen so far.  Returns the number
    of (candidate, subset) evaluations made."""
    r, done = len(pc.subsets), 0
    while len(A) > 1:
        best, overlap = findhighestscore(A)
        if not overlap:
            break
        group = [i for i in range(len(A)) if i == best or isoverlap(A.scores[i], A.scores[best])]
        lmin = min(A.evaluated[i][0] for i in group)
        if lmin >= r:
            break
        todo = [i for i in group if A.evaluated[i][0] == lmin]
        dev = [i for i in todo if type(A.shapes[i]) in SHAPE_KIND]
        counts = dict(zip(dev, score_counts(pc, [A.shapes[i] for i in dev], lmin, _builtin_params(params))[0])) if dev else {}
        for cls in {type(A.shapes[i]) for i in todo if on_device(type(A.shapes[i]))}:  # one launch per user class
            ui = [i for i in todo if type(A.shapes[i]) is cls]
            counts.update(zip(ui, user_score_counts(pc, [A.shapes[i] for i in ui], lmin, params)[0]))
        for i in todo:  # other user-defined shapes score themselves (docs/src/newprimitive.md:16)
            c = counts[i] if i in counts else len(A.shapes[i].scorecandidate(pc, lmin, params)[1])
            ev = A.evaluated[i]
            ev[0], ev[1], ev[2] = ev[0] + 1, ev[1] + int(c), ev[2] + len(pc.subsets[lmin])
            A.scores[i] = estimatescore_f64(ev[2], pc.size, ev[1])
        done += len(todo)
    return done


def findhighestscore(A: IterationCandidates):
    """fitting.jl:140-158 -> (index, overlap); index -1 when empty (0-based)."""
    if len(A) == 0:
        return -1, False
    ind, highest = 0, A.scores[0].E
    for i, sc in enumerate(A.scores):
        if sc.E > highest:
            highest, ind = sc.E, i
    for i, sc in enumerate(A.scores):
        if i != ind and isoverlap(sc, A.scores[ind]):
            return ind, True
    return ind, False
