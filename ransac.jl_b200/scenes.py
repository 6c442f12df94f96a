"""Seeded synthetic scenes for the BASELINE.json configs (SURVEY.md section 8d).

The reference ships no example cloud (`examplepc3` is undefined in the repo, NEWS.md:43), so the
generator is ours.  Coordinates are generated in float64 with numpy PCG64 and rounded to float32, so
the float32 device data and the float64 oracle see identical inputs.  Scene units: bounding box
~100, which makes the default eps = 0.3 / alpha = 5 deg meaningful.
"""
from __future__ import annotations

import math
from dataclasses import dataclass, field
from typing import List, Tuple

import numpy as np

from .shapes import FittedCone, FittedCylinder, FittedPlane, FittedSphere


def _unit(v):
    return v / np.linalg.norm(v, axis=-1, keepdims=True)


def _rand_unit(rng, n=None):
    v = rng.normal(size=(3,) if n is None else (n, 3))
    return _unit(v)


def _frame(a):
    """two unit vectors orthogonal to unit vector a"""
    t = np.array([1.0, 0, 0]) if abs(a[0]) < 0.9 else np.array([0, 1.0, 0])
    b = _unit(np.cross(a, t))
    return b, np.cross(a, b)


@dataclass
class Primitive:
    kind: str
    shape: object  # the generating Fitted* shape (ground truth)
    size: float  # characteristic size (for noise scaling)
    area: float
    extra: dict = field(default_factory=dict)


def sample_primitive(rng, prim: Primitive, n: int) -> Tuple[np.ndarray, np.ndarray]:
    s = prim.shape
    if prim.kind == "plane":
        b, c = _frame(s.normal)
        u = rng.uniform(-0.5, 0.5, n) * prim.extra["sx"]
        v = rng.uniform(-0.5, 0.5, n) * prim.extra["sy"]
        p = s.point + u[:, None] * b + v[:, None] * c
        nn = np.broadcast_to(s.normal, p.shape).copy()
    elif prim.kind == "sphere":
        d = _rand_unit(rng, n)
        p = s.center + s.radius * d
        nn = d if s.outwards else -d
    elif prim.kind == "cylinder":
        b, c = _frame(s.axis)
        phi = rng.uniform(0, 2 * math.pi, n)
        h = rng.uniform(-0.5, 0.5, n) * prim.extra["L"]
        rad = np.cos(phi)[:, None] * b + np.sin(phi)[:, None] * c
        p = s.center + prim.extra["h0"] * s.axis + h[:, None] * s.axis + s.radius * rad
        nn = rad if s.outwards else -rad
    elif prim.kind == "cone":
        b, c = _frame(s.axis)
        th = s.opang / 2
        phi = rng.uniform(0, 2 * math.pi, n)
        h0, h1 = prim.extra["h0"], prim.extra["h1"]
        h = np.sqrt(rng.uniform(h0 * h0, h1 * h1, n))  # area-uniform along the slant
        rad = np.cos(phi)[:, None] * b + np.sin(phi)[:, None] * c
        p = s.apex + h[:, None] * s.axis + (h * math.tan(th))[:, None] * rad
        nn = math.cos(th) * rad - math.sin(th) * s.axis
        if not s.outwards:
            nn = -nn
    else:
        raise ValueError(prim.kind)
    return p, nn


def _jitter_normals(rng, nn, deg):
    if deg <= 0:
        return nn
    t = math.tan(math.radians(deg))
    return _unit(nn + rng.normal(size=nn.shape) * (t / math.sqrt(2)))


@dataclass
class Scene:
    vertices: np.ndarray  # (N,3) float32
    normals: np.ndarray  # (N,3) float32
    labels: np.ndarray  # (N,) int32, -1 = outlier
    primitives: List[Primitive]


def build_scene(rng, prims: List[Primitive], n_total: int, noise_frac: float, jitter_deg: float,
                outlier_frac: float, shuffle: bool = True, weights=None) -> Scene:
    n_out = int(round(n_total * outlier_frac))
    n_in = n_total - n_out
    w = np.array([p.area for p in prims]) if weights is None else np.asarray(weights, float)
    cnt = np.floor(w / w.sum() * n_in).astype(int)
    cnt[0] += n_in - cnt.sum()
    P, Nn, Lb = [], [], []
    for i, (pr, c) in enumerate(zip(prims, cnt)):
        p, nn = sample_primitive(rng, pr, int(c))
        if noise_frac > 0:
            p = p + nn * rng.normal(scale=noise_frac * pr.size, size=(len(p), 1))
        nn = _jitter_normals(rng, nn, jitter_deg)
        P.append(p), Nn.append(nn), Lb.append(np.full(len(p), i, np.int32))
    P = np.concatenate(P)
    lo, hi = P.min(0), P.max(0)
    if n_out:
        P = np.concatenate([P, rng.uniform(lo, hi, size=(n_out, 3))])
        Nn.append(_rand_unit(rng, n_out))
        Lb.append(np.full(n_out, -1, np.int32))
    Nn = np.concatenate(Nn)
    Lb = np.concatenate(Lb)
    if shuffle:
        perm = rng.permutation(len(P))
        P, Nn, Lb = P[perm], Nn[perm], Lb[perm]
    v32 = np.ascontiguousarray(P, dtype=np.float32)
    n32 = np.ascontiguousarray(Nn, dtype=np.float32)
    return Scene(v32, n32, Lb, prims)


# ---- primitive factories ---------------------------------------------------------------------
def make_plane(rng, box=100.0, smin=20.0, smax=60.0):
    n = _rand_unit(rng)
    c = rng.uniform(-box / 2, box / 2, 3)
    sx, sy = rng.uniform(smin, smax, 2)
    return Primitive("plane", FittedPlane(c, n), float(max(sx, sy)), float(sx * sy), {"sx": sx, "sy": sy})


def make_sphere(rng, box=100.0, rmin=5.0, rmax=15.0):
    c = rng.uniform(-box / 2, box / 2, 3)
    R = rng.uniform(rmin, rmax)
    return Primitive("sphere", FittedSphere(c, R, bool(rng.integers(2))), float(2 * R), float(4 * math.pi * R * R))


def make_cylinder(rng, box=100.0, rmin=3.0, rmax=10.0, lmin=20.0, lmax=60.0):
    a = _rand_unit(rng)
    q = rng.uniform(-box / 2, box / 2, 3)
    h0 = float(np.dot(a, q))
    c = q - a * h0  # the reference stores the axis point on the plane through the origin (cylinder.jl:114)
    R = rng.uniform(rmin, rmax)
    L = rng.uniform(lmin, lmax)
    return Primitive("cylinder", FittedCylinder(a, c, R, bool(rng.integers(2))), float(max(L, 2 * R)),
                     float(2 * math.pi * R * L), {"L": L, "h0": h0})


def make_cone(rng, box=100.0, hmin=25.0, hmax=45.0):
    a = _rand_unit(rng)
    apex = rng.uniform(-box / 2, box / 2, 3)
    half = math.radians(rng.uniform(10, 35))
    h1 = rng.uniform(hmin, hmax)
    h0 = h1 * rng.uniform(0.15, 0.3)
    area = math.pi * math.tan(half) / math.cos(half) * (h1 * h1 - h0 * h0)
    return Primitive("cone", FittedCone(apex, a, 2 * half, bool(rng.integers(2))), float(h1), float(area),
                     {"h0": h0, "h1": h1})


# ---- the named configs -----------------------------------------------------------------------
def scene_c1(seed: int = 1234) -> Scene:
    """c1: 10 000 points, plane 4000 (10x10 patch) + sphere 3000 (R=3) + cylinder 3000 (R=2, L=10),
    no noise.  Runs end-to-end on the CPU oracle."""
    rng = np.random.default_rng(seed)
    prims = [
        Primitive("plane", FittedPlane([0, 0, 0], [0, 0, 1.0]), 10.0, 100.0, {"sx": 10.0, "sy": 10.0}),
        Primitive("sphere", FittedSphere([12.0, 0, 4.0], 3.0, True), 6.0, 113.0),
        Primitive("cylinder", FittedCylinder([0, 1.0, 0], [-10.0, 0, 5.0], 2.0, True), 10.0, 125.0, {"L": 10.0, "h0": 0.0}),
    ]
    return build_scene(rng, prims, 10_000, 0.0, 0.0, 0.0, shuffle=True, weights=[4, 3, 3])


def scene_mixed(seed: int, n: int, noise_frac=0.01, jitter_deg=2.0, outlier_frac=0.2,
                counts=(6, 3, 2, 2)) -> Scene:
    """c2/c3 generator: 6 planes, 3 spheres, 2 cylinders, 2 cones; area-weighted share of the inlier
    points, Gaussian offset along the normal (sigma = noise_frac * primitive size), normal jitter,
    uniform outliers with random normals."""
    rng = np.random.default_rng(seed)
    prims = [make_plane(rng) for _ in range(counts[0])]
    prims += [make_sphere(rng) for _ in range(counts[1])]
    prims += [make_cylinder(rng) for _ in range(counts[2])]
    prims += [make_cone(rng) for _ in range(counts[3])]
    return build_scene(rng, prims, n, noise_frac, jitter_deg, outlier_frac)


_VIEW_DRAWS = 64  # batches of 2x the wanted points drawn per primitive before scene_view gives up


def scene_view(seed: int, n: int, viewpoint=(0.0, 0.0, 150.0), noise_frac: float = 0.002, counts=(3, 2, 2, 1)) -> Scene:
    """One scan from `viewpoint` with ground-truth oriented normals: primitives from the factories above (spheres,
    cylinders and cones with outward normals), of which only the points whose analytic normal faces the viewpoint
    are kept (back-face culling, no occlusion; planes are two-sided), with the normals flipped towards the viewpoint.
    Area-weighted share of the n points, Gaussian offset along the normal (sigma = noise_frac * primitive size), no
    outliers, no normal jitter.  ValueError when a primitive barely faces the viewpoint (e.g. one inside a sphere)."""
    rng = np.random.default_rng(seed)
    prims = [make_plane(rng) for _ in range(counts[0])]
    prims += [make_sphere(rng) for _ in range(counts[1])]
    prims += [make_cylinder(rng) for _ in range(counts[2])]
    prims += [make_cone(rng) for _ in range(counts[3])]
    for p in prims:
        if p.kind != "plane":
            p.shape.outwards = True
    vp = np.asarray(viewpoint, np.float64)
    w = np.array([p.area for p in prims])
    cnt = np.floor(w / w.sum() * n).astype(int)
    cnt[0] += n - cnt.sum()
    P, Nn, Lb = [], [], []
    for i, (pr, c) in enumerate(zip(prims, cnt)):
        got_p, got_n, have = [], [], 0
        for _ in range(_VIEW_DRAWS):
            if have >= c:
                break
            p, nn = sample_primitive(rng, pr, max(2 * int(c), 64))
            facing = np.einsum("ij,ij->i", nn, vp - p)
            if pr.kind == "plane":
                nn = np.where(facing[:, None] < 0, -nn, nn)
            else:
                p, nn = p[facing > 0], nn[facing > 0]
            got_p.append(p), got_n.append(nn)
            have += len(p)
        if have < c:
            raise ValueError(f"scene_view: too little of primitive {i} ({pr.kind}) faces the viewpoint {tuple(vp)}")
        p, nn = np.concatenate(got_p)[:c], np.concatenate(got_n)[:c]
        if noise_frac > 0:
            p = p + nn * rng.normal(scale=noise_frac * pr.size, size=(len(p), 1))
        P.append(p), Nn.append(nn), Lb.append(np.full(len(p), i, np.int32))
    perm = rng.permutation(n)
    P, Nn, Lb = np.concatenate(P)[perm], np.concatenate(Nn)[perm], np.concatenate(Lb)[perm]
    return Scene(np.ascontiguousarray(P, dtype=np.float32), np.ascontiguousarray(Nn, dtype=np.float32), Lb, prims)


def recovered(scene: Scene, shapes, frac: float = 0.5) -> set:
    """indices of the ground-truth primitives of `scene` found among `shapes` [(kind, inlier indices)]: a shape of the
    same kind whose inliers are mostly the primitive's points and cover at least `frac` of them"""
    kinds = {"plane": 0, "sphere": 1, "cylinder": 2, "cone": 3}
    sizes = np.bincount(scene.labels[scene.labels >= 0], minlength=len(scene.primitives))
    found = set()
    for kind, idx in shapes:
        if len(idx) == 0:
            continue
        lab = np.bincount(scene.labels[idx] + 1, minlength=len(scene.primitives) + 1)[1:]
        i = int(np.argmax(lab))
        if kinds[scene.primitives[i].kind] == kind and lab[i] >= 0.5 * len(idx) and lab[i] >= frac * sizes[i]:
            found.add(i)
    return found


SCAN_VIEWPOINT = (30.0, -20.0, 160.0)


@dataclass
class ScanScenario:
    scene: Scene
    viewpoint: tuple
    subsets: int
    seed: int
    iteration: dict


def scan_scenario() -> ScanScenario:
    """Normals for a raw scan, end to end: a noisy 40 000-point scene_view from SCAN_VIEWPOINT with 8 primitives, and the
    ransac() settings run on it.  With the analytic normals the C oracle's loop recovers all 8 primitives (`recovered`),
    with normals estimated from the coordinates (k = 16, towards the viewpoint) 6 of them."""
    return ScanScenario(scene_view(21, 40_000, viewpoint=SCAN_VIEWPOINT, noise_frac=0.002), SCAN_VIEWPOINT, 2, 4321,
                        {"tau": 100, "minsubsetN": 50, "itermax": 200})


def scene_c2(n: int = 1 << 20, seed: int = 2) -> Scene:
    return scene_mixed(seed, n)


def scene_c3(n: int = 16 << 20, seed: int = 3) -> Scene:
    return scene_mixed(seed, n)


def scene_cad(n: int = 10_000_000, seed: int = 4, nprims: int = 200) -> Scene:
    """c4: CAD-like, 200 primitives of mixed type: 180 small ones (sizes log-uniform 1-10 % of the
    box) on 20 larger base shapes (10-40 %), area-weighted point share, 0.5 % noise, 5 % outliers.
    (With the reference's root-cell sampler, Q1, only the larger shapes reach the detection
    probability; the small ones are what the octree-level sampler of SURVEY 8(f) is for.)"""
    rng = np.random.default_rng(seed)
    prims = []
    for i in range(nprims):
        s = 100.0 * (10 ** rng.uniform(-1, -0.4) if i < 20 else 10 ** rng.uniform(-2, -1))
        k = i % 4
        if k == 0:
            prims.append(make_plane(rng, smin=s, smax=2 * s))
        elif k == 1:
            prims.append(make_sphere(rng, rmin=s / 2, rmax=s))
        elif k == 2:
            prims.append(make_cylinder(rng, rmin=s / 4, rmax=s / 2, lmin=s, lmax=2 * s))
        else:
            prims.append(make_cone(rng, hmin=s, hmax=2 * s))
    return build_scene(rng, prims, n, 0.005, 1.0, 0.05)


LIDAR_CHUNK = 12_500_000


def lidar_primitives(seed: int = 5):
    rng = np.random.default_rng(seed)
    prims = [make_plane(rng, box=100.0, smin=80.0, smax=100.0) for _ in range(8)]
    prims += [make_cylinder(rng, rmin=0.3, rmax=1.0, lmin=5.0, lmax=15.0) for _ in range(30)]
    w = [0.6 / 8] * 8 + [0.1 / 30] * 30
    return prims, w


def scene_lidar_chunk(i: int, n_chunk: int, seed: int = 5) -> Scene:
    """points [i*LIDAR_CHUNK, i*LIDAR_CHUNK + n_chunk) of the c5 scene: every chunk is an independent
    shuffled draw from the same primitives (so ranks can generate chunks side by side)"""
    prims, w = lidar_primitives(seed)
    return build_scene(np.random.default_rng([seed, 1000 + i]), prims, n_chunk, 0.002, 2.0, 0.3, weights=w)


def scene_lidar(n: int = 100_000_000, seed: int = 5) -> Scene:
    """c5: LiDAR-like, 8 large planes (60 %), 30 cylinders (10 %), 30 % outliers; generated in
    chunks of 12.5 M points."""
    parts = []
    for i, lo in enumerate(range(0, n, LIDAR_CHUNK)):
        parts.append(scene_lidar_chunk(i, min(LIDAR_CHUNK, n - lo), seed))
    return Scene(np.concatenate([p.vertices for p in parts]), np.concatenate([p.normals for p in parts]),
                 np.concatenate([p.labels for p in parts]), parts[0].primitives)


def perturbed_candidates(scene: Scene, per_type: int, seed: int = 7, pos=0.3, ang_deg=1.5, rel=0.01):
    """Candidates near the scene's true primitives (realistic inlier rates): `per_type` of each of
    plane, sphere, cylinder, cone (types without a primitive in the scene get random shapes)."""
    rng = np.random.default_rng(seed)
    by = {"plane": [], "sphere": [], "cylinder": [], "cone": []}
    for p in scene.primitives:
        by[p.kind].append(p.shape)

    def tilt(a):
        return _unit(a + rng.normal(size=3) * math.tan(math.radians(ang_deg)))

    out = []
    for kind in ("plane", "sphere", "cylinder", "cone"):
        for _ in range(per_type):
            src = by[kind][rng.integers(len(by[kind]))] if by[kind] else None
            dp = rng.normal(size=3) * pos
            if kind == "plane":
                s = src or make_plane(rng).shape
                sign = 1.0 if rng.integers(2) else -1.0
                out.append(FittedPlane(s.point + dp, sign * tilt(s.normal)))
            elif kind == "sphere":
                s = src or make_sphere(rng).shape
                out.append(FittedSphere(s.center + dp, s.radius * (1 + rng.normal() * rel), s.outwards))
            elif kind == "cylinder":
                s = src or make_cylinder(rng).shape
                a = tilt(s.axis)
                c = s.center + dp
                c = c - a * float(np.dot(a, c))
                out.append(FittedCylinder(a, c, s.radius * (1 + rng.normal() * rel), s.outwards))
            else:
                s = src or make_cone(rng).shape
                out.append(FittedCone(s.apex + dp, tilt(s.axis), s.opang * (1 + rng.normal() * rel), s.outwards))
    return out
