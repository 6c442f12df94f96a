"""ransac(pc, params, setenabled; reset_rand): mirror of src/iterations.jl:14-162.

For the four built-in shape types the whole loop runs inside the CUDA library behind one C-ABI call
(`rsc_ransac_run`).  User-defined shapes whose `cuda_source` also fits (`shapes.device_fit`) join that loop
(`rsc_ransac_run_user`) unless an extension switch is asked for.  Otherwise, if `shape_types` contains a
user-defined FittedShape subclass, the loop runs here and calls that class's own
`fit`/`scorecandidate`/`refit` methods -- the reference's plug-in contract (docs/src/newprimitive.md:12-18)
-- while built-in types still score on the device.  A user shape with `cuda_source` scores and refits on the
device (rsc_user_score, rsc_user_refit_extract), and fits there too when it can (rsc_sample_fit_user).
"""
from __future__ import annotations

import ctypes as C
import time
from typing import List, Tuple

import numpy as np

from . import _lib
from ._lib import lib
from .cloud import RANSACCloud
from .confidence import estimatescore_f64, prob
from .fitting import (IterationCandidates, findhighestscore, fit_order, lsq_refit, refine_progressive, refit, sample_fit,
                      sample_fit_user, scorecandidates, shape_from_record)
from .params import to_c
from .shapes import SHAPE_KIND, ExtractedShape, device_fit, on_device


def _all_builtin(params) -> bool:
    return all(t in SHAPE_KIND for t in params["iteration"]["shape_types"])


def ransac(pc: RANSACCloud, params, setenabled: bool = True, reset_rand: bool = False, seed: int = 1234,
           sampler: str = "root", progressive: bool = False, lsq: bool = False, bitmap=None,
           lw_period: int = 1) -> Tuple[List[ExtractedShape], float]:
    """Run efficient RANSAC on `pc`; returns (extracted shapes, seconds).

    `reset_rand=True` pins the sampler seed to 1234 like `Random.seed!(1234)` (iterations.jl:36);
    the Philox stream is of course not Julia's (SURVEY Q19).  `sampler="octree"` (extension, needs
    `pc.build_cells()`) draws the minimal sets from level-weighted octree cells -- what the reference
    is written for -- instead of from the root cell, which is what its shipped code does (Q1); the
    final level weights are left in `pc.levelweight`; `lw_period=P` refreshes the level weights every P iterations
    instead of after each one, which lets the device loop batch its iterations (same results at any batch size).  `progressive=True` (extension) refines
    overlapping scores on further subsets before each extraction test (`fitting.refine_progressive`,
    the reference's "TODO: refine if best.overlap", iterations.jl:110; `RSC_SCORE_PROGRESSIVE` in the
    device loop) and leaves the number of extra (candidate, subset) evaluations in `pc.last_refined`.
    `lsq=True` (extension) refits the best candidate by least squares to the compatible points within
    3 eps before it is extracted (`fitting.lsq_refit`; the paper's refit, docs/src/ransac.md:163-169).
    `bitmap=(beta, eight)` (extension) extracts, of every shape's compatible points, only those in the largest
    connected component of its parameter-space bitmap (`fitting.bitmap_filter`, `RSC_EXTRACT_BITMAP`; the paper's
    third compatibility criterion, which the reference documents and leaves out, docs/src/ransac.md:106-112)."""
    if setenabled:
        pc.enable_all()
    if reset_rand:
        seed = 1234
    if _all_builtin(params):
        return _ransac_device(pc, params, seed, sampler, lsq, progressive, bitmap, lw_period)
    if _device_order(pc, params["iteration"]["shape_types"]) and sampler == "root" and not progressive and not lsq and bitmap is None:
        return _ransac_device(pc, params, seed, order=params["iteration"]["shape_types"])
    if bitmap is not None:
        raise ValueError("the bitmap filter is only available in the device loop (built-in shape types)")
    if sampler != "root":
        raise ValueError("the octree sampler is only available in the device loop (built-in shape types)")
    return _ransac_host(pc, params, seed, progressive, lsq)


def _device_order(pc, types) -> bool:
    """True when rsc_ransac_run_user takes `types`: built-ins and device-fitting user classes only, at most
    RSC_MAX_ORDER of them, none twice, on a whole (not sharded, not ranged) cloud."""
    return (all(t in SHAPE_KIND or device_fit(t) for t in types) and len(types) <= _lib.RSC_MAX_ORDER
            and len(set(types)) == len(types) and not pc.is_shard and not getattr(pc, "ranged", False))


def _ransac_device(pc, params, seed, sampler="root", lsq=False, progressive=False, bitmap=None, lw_period=1, order=None):
    """The device loop: rsc_ransac_run, or rsc_ransac_run_user for a fit order `order` of built-in and device-fitting
    user classes (no extension switches then)."""
    classes = {}
    if order is not None:
        slots, classes = fit_order(pc, order, params)
        params = dict(params, iteration=dict(params["iteration"], shape_types=[t for t in order if t in SHAPE_KIND]))
    cp = to_c(params)
    cp.lw_period = max(1, int(lw_period))  # octree sampler: refresh period of the level weights (1 = every iteration)
    if bitmap is not None:
        pc.ctx.check(lib.rsc_ctx_set_bitmap(pc.ctx.h, float(bitmap[0]), int(bool(bitmap[1]))))
        cp.compat_flags |= _lib.RSC_EXTRACT_BITMAP
    if progressive:
        for j in range(len(pc.subsets)):  # the refinement scores on the subsets 2..r too
            pc.upload_subset(j)
        cp.compat_flags |= _lib.RSC_SCORE_PROGRESSIVE
    if lsq:
        cp.compat_flags |= _lib.RSC_REFIT_LSQ
    if sampler == "octree":
        cp.compat_flags |= _lib.RSC_SAMPLER_OCTREE
    elif sampler != "root":
        raise ValueError("sampler must be 'root' or 'octree'")
    run = C.c_void_p()
    if order is not None:
        pc.ctx.check(lib.rsc_ransac_run_user(pc.handle, C.byref(cp), slots, len(order), seed, C.byref(run)))
    else:
        pc.ctx.check(lib.rsc_ransac_run(pc.handle, C.byref(cp), seed, C.byref(run)))
    try:
        out = []
        for i in range(lib.rsc_run_nshapes(run)):
            cand = _lib.rsc_cand()
            n = C.c_int64()
            pc.ctx.check(lib.rsc_run_shape(run, i, C.byref(cand), C.byref(n)))
            idx = np.empty(n.value, dtype=np.int64)  # filled by rsc_run_inpoints (device -> host)
            if n.value:
                pc.ctx.check(lib.rsc_run_inpoints(run, i, idx.ctypes.data))
            ex = ExtractedShape(shape_from_record(cand, classes), idx)
            # sharded storage: `inpoints` is this rank's part of the list (shard.gather_extracted joins them)
            ex.total = int(lib.rsc_run_shape_total(run, i))
            out.append(ex)
        secs = lib.rsc_run_seconds(run)
        nbatch = C.c_int32()
        pc.last_run_syncs = int(lib.rsc_run_syncs(run, C.byref(nbatch)))
        pc.last_run_batches = int(nbatch.value)
        pc.last_run_iterations = int(lib.rsc_run_iterations(run))
        pc.last_refined = int(lib.rsc_run_refined(run))
        lw, ls = np.zeros(11), np.zeros(11)
        nl = lib.rsc_run_levelweight(run, lw.ctypes.data, ls.ctypes.data)
        if nl:
            pc.levelweight, pc.levelscore = lw[:nl].copy(), ls[:nl].copy()
    finally:
        lib.rsc_run_destroy(run)
    pc.last_run_seconds = secs  # unrounded device-loop time (the return value is truncated like the reference's)
    return out, int(secs * 100) / 100.0


def _ransac_host(pc, params, seed, progressive=False, lsq=False):
    """iterations.jl:35-162 on the host, for parameter sets with user-defined shapes and for
    progressive scoring."""
    it = params["iteration"]
    drawN, minsubsetN, prob_det, tau = it["drawN"], it["minsubsetN"], it["prob_det"], it["tau"]
    sidx = {"lengthC": 0, "allcand": 1, "nofminset": 2}
    builtin = [t for t in it["shape_types"] if t in SHAPE_KIND]
    # built-ins and user shapes that fit on the device: one rsc_sample_fit_user call per iteration; the other user
    # shapes fit here, on the same drawn sets
    devfit = [t for t in it["shape_types"] if t in SHAPE_KIND or device_fit(t)]
    custom = [t for t in it["shape_types"] if t not in devfit]
    bparams = dict(params, iteration=dict(it, shape_types=builtin))
    t0 = time.time()
    scored = IterationCandidates()
    extracted: List[ExtractedShape] = []
    cc = [0, 0, 0]
    M1 = len(pc.subsets[0])
    pc.last_refined = 0
    for k in range(1, it["itermax"] + 1):
        if pc.count_enabled() < tau:
            break
        if devfit == builtin and builtin:
            cands, csets, idx = sample_fit(pc, bparams, seed, (k - 1) * minsubsetN, minsubsetN)
        else:  # device-fitting user types: merged candidates; no device-fitting type at all: the same sets, drawn only
            cands, csets, idx = sample_fit_user(pc, params, devfit, seed, (k - 1) * minsubsetN, minsubsetN)
        if custom:
            # forcefitshapes! (fitting.jl:165-173) appends per minimal set in shape_types order: merge the device's
            # built-in candidates with the user's by (set, position in shape_types) -- findhighestscore is
            # "first maximum wins", so the order decides ties
            pos = {t: i for i, t in enumerate(it["shape_types"])}
            keyed = [((int(s), pos[type(c)]), c) for c, s in zip(cands, csets)]
            for si, row in enumerate(idx):
                if row[0] < 0:
                    continue
                for t in custom:
                    f = t.fit(pc.vertices[row], pc.normals[row], pc, params)
                    if f is not None:
                        keyed.extend(((si, pos[t]), c) for c in (f if isinstance(f, (list, tuple)) else [f]))
            keyed.sort(key=lambda kc: kc[0])  # stable
            cands = [c for _, c in keyed]
        cc[1] += len(cands)
        # built-in and device-capable user shapes: one batched call (one launch per class); other user shapes
        # score themselves
        b = [c for c in cands if type(c) in SHAPE_KIND or on_device(type(c))]
        res = dict(zip(map(id, b), scorecandidates(pc, b, 0, params))) if b else {}
        for c in cands:
            sc, ip = res[id(c)] if id(c) in res else c.scorecandidate(pc, 0, params)
            if progressive:
                sc = estimatescore_f64(M1, pc.size, len(ip))
            scored.recordscore(c, sc, ip, M1)
        cc[2] = k * minsubsetN
        cc[0] = len(scored)
        if len(scored) >= 1:
            if progressive:
                pc.last_refined += refine_progressive(pc, scored, bparams)
            best, _ = findhighestscore(scored)
            scr = scored.scores[best].E
            if prob(scr, cc[sidx[it["extract_s"]]], pc.size, drawN) > prob_det:
                shp = scored.shapes[best]
                if lsq and type(shp) in SHAPE_KIND:
                    shp = lsq_refit(shp, pc, bparams)[0]
                dev = type(shp) in SHAPE_KIND or on_device(type(shp))
                ex = refit(shp, pc, params, disable=True) if dev else shp.refit(pc, params)
                if ex is not None:  # a user's refit may return nothing: the reference then skips the extraction (iterations.jl:130)
                    if not dev:
                        from .fitting import invalidate_indexes
                        invalidate_indexes(pc, ex.inpoints)
                    extracted.append(ex)
                    scored.deleteat(best)
                    en = pc.isenabled
                    dead = [j for j in range(len(scored)) if not en[scored.inpoints[j]].all()]
                    scored.deleteat(dead)
                    if progressive:  # refined scores may count points of the subsets 2..r that were just extracted
                        for j in range(len(scored)):
                            if scored.evaluated[j][0] > 1:
                                scored.evaluated[j] = [1, len(scored.inpoints[j]), M1]
                                scored.scores[j] = estimatescore_f64(M1, pc.size, len(scored.inpoints[j]))
        if prob(tau, cc[sidx[it["terminate_s"]]], pc.size, drawN) > prob_det:
            break
    return extracted, int((time.time() - t0) * 100) / 100.0
