"""Digests of ransac() runs over the loop's configurations: one JSON line per configuration with hashes of the
extracted candidates' bytes, of their inlier lists and of the final enabled mask, plus the iterations, the
progressive refinements, the level weights / scores of the cell sampler, the host synchronisations, the batches
and the device-loop seconds.  Two builds of the library (RSC_LIB_PATH) compute the same results when every field
but `seconds`, `syncs` and `batches` is equal: those three describe how a run got there, and may differ between
builds whose batching or synchronisation differs (results do not depend on the batch sizes).

  python tools/loop_digest.py [--only NAME,...] [--skip-c4]
"""
import argparse
import hashlib
import json
import math
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def _h(*arrays) -> str:
    d = hashlib.sha256()
    for a in arrays:
        d.update(a if isinstance(a, bytes) else np.ascontiguousarray(a).tobytes())
    return d.hexdigest()[:16]


def _shape_bytes(s) -> bytes:
    return bytes(s.to_cand()) if hasattr(s, "to_cand") else repr(s.device_record()).encode()


def digest(R, name, pc, params, seed, env=(), **kw):
    for k, v in env:
        os.environ[k] = v
    try:
        ex, _ = R.ransac(pc, params, True, seed=seed, **kw)
    finally:
        for k, _ in env:
            del os.environ[k]
    out = {"config": name, "shapes": len(ex), "cands": _h(*[_shape_bytes(e.shape) for e in ex]),
           "inliers": _h(*[np.asarray(e.inpoints, np.int64) for e in ex]), "enabled": _h(np.asarray(pc.isenabled, np.uint8)),
           "iterations": pc.last_run_iterations, "refined": pc.last_refined, "syncs": pc.last_run_syncs,
           "batches": pc.last_run_batches, "seconds": pc.last_run_seconds}
    if kw.get("sampler") == "octree":
        out["levelweight"] = [float(x).hex() for x in pc.levelweight]
        out["levelscore"] = [float(x).hex() for x in pc.levelscore]
    print(json.dumps(out), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--only", default="", help="comma-separated configuration name prefixes")
    ap.add_argument("--skip-c4", action="store_true")
    args = ap.parse_args()
    only = [s for s in args.only.split(",") if s]

    import ransac_jl_b200 as R
    from ransac_jl_b200 import scenes

    def want(name):
        return not only or any(name.startswith(o) for o in only)

    variants = [("default", ()), ("cull0", (("RSC_LOOP_CULL", "0"),)), ("cull2", (("RSC_LOOP_CULL", "2"),)),
                ("batch1", (("RSC_BATCH", "1"),)), ("nosmall", (("RSC_NO_SMALL", "1"),)), ("k5masked", (("RSC_K5_MASKED", "1"),)),
                ("hostwalk", (("RSC_LOOP_HOSTWALK", "1"),))]
    scenes_ = [("c2", lambda: scenes.scene_c2(1 << 20), 32, lambda n: {"tau": n // 100, "minsubsetN": 4096, "itermax": 200})]
    if not args.skip_c4:
        scenes_.append(("c4", lambda: scenes.scene_cad(10_000_000), 32, lambda n: {"tau": n // 1000, "minsubsetN": 8192, "itermax": 400}))
    for tag, make, r, itf in scenes_:
        if only and not any(o.startswith(tag) for o in only):
            continue
        sc = make()
        n = len(sc.vertices)
        params = R.ransacparameters(iteration=itf(n))
        pc = R.RANSACCloud(sc.vertices, sc.normals, R.makesubsets(n, r, np.random.default_rng(1234)))
        for v, env in variants:
            if want(f"{tag}_{v}"):
                digest(R, f"{tag}_{v}", pc, params, 2024, env)
        if want(f"{tag}_lsq"):
            digest(R, f"{tag}_lsq", pc, params, 2024, lsq=True)
        if want(f"{tag}_bitmap"):
            digest(R, f"{tag}_bitmap", pc, params, 2024, bitmap=(1.5, False))
        if want(f"{tag}_progressive"):
            digest(R, f"{tag}_progressive", pc, params, 2024, progressive=True)
        if want(f"{tag}_octree"):
            pc.build_cells(8)
            for lw in (1, 16):
                if want(f"{tag}_octree_lw{lw}"):
                    digest(R, f"{tag}_octree_lw{lw}", pc, params, 2024, sampler="octree", lw_period=lw)
        pc.close()

    # an exact float64 cloud (c1, jittered below float32 resolution)
    if want("exact"):
        sc = scenes.scene_c1()
        rng = np.random.default_rng(31)
        V = sc.vertices.astype(np.float64) + rng.uniform(-1e-6, 1e-6, sc.vertices.shape)
        N = sc.normals.astype(np.float64) + rng.uniform(-1e-6, 1e-6, sc.normals.shape)
        pc = R.RANSACCloud(V, N, 2, exact=True)
        params = R.ransacparameters()
        for v, env in (("default", ()), ("cull2", (("RSC_LOOP_CULL", "2"),)), ("hostwalk", (("RSC_LOOP_HOSTWALK", "1"),)),
                       ("hostwalk_cull2", (("RSC_LOOP_HOSTWALK", "1"), ("RSC_LOOP_CULL", "2")))):
            if want(f"exact_c1_{v}"):
                digest(R, f"exact_c1_{v}", pc, params, 4321, env)
        pc.close()

    # a user fit order: the slab of tests/user_fit_shapes.py with a plane
    if want("user"):
        import user_fit_shapes as U

        _, _, (DS, _) = U.shape_classes(R)
        V, N = U.mixed_scene(np.random.default_rng(5), 200_000)
        pc = R.RANSACCloud(V, N, 3)
        params = R.ransacparameters([R.FittedPlane, DS], iteration={"tau": 400, "minsubsetN": 128, "itermax": 400})
        params["slab"] = {"eps": 0.3, "alpha": math.radians(5), "tol": 0.1}
        digest(R, "user_slab_plane", pc, params, 2)
        pc.close()


if __name__ == "__main__":
    main()
