"""Fitted-shape types: mirror of FittedPlane/FittedSphere/FittedCylinder/FittedCone
(src/shapes/plane.jl:8-11, sphere.jl:9-13, cylinder.jl:11-16, cone.jl:11-19) and ExtractedShape
(src/fitting.jl:81-84), with the conversion to/from the 64-byte C-ABI candidate record."""
from __future__ import annotations

from dataclasses import dataclass
from typing import Sequence

import numpy as np

from . import _lib


class FittedShape:
    """Abstract base (fitting.jl:8): user shapes subclass this and plug into the host loop.

    A user shape may also run its scoring and refit on the device.  It then defines three members:
    `cuda_source` (class attribute: CUDA C defining `rsc_user_compatible`, include/rsc.h), `device_record(self)`
    -> (p, outwards) with at most 7 floats, and the staticmethod `device_constants(params)` -> at most 8 floats
    (thresholds such as eps and cos(alpha), computed on the host).  Its `fit` stays on the host unless its
    `cuda_source` also defines `rsc_user_fit` and the class provides the classmethod `from_device_record(p, outwards)`
    (the inverse of `device_record`): then it fits on the device too, and a parameter set of such shapes and built-ins
    runs in the device loop (`device_fit`)."""

    kind = -1
    cuda_source = None

    def to_cand(self) -> _lib.rsc_cand:  # pragma: no cover - abstract
        raise NotImplementedError


def on_device(shape_class) -> bool:
    """True for a user-defined shape class that brings device source (`cuda_source`)."""
    return shape_class not in SHAPE_KIND and getattr(shape_class, "cuda_source", None) is not None


def device_fit(shape_class) -> bool:
    """True for a user-defined shape class that fits on the device: its `cuda_source` defines `rsc_user_fit` and it
    turns device records back into instances with `from_device_record(p, outwards)`."""
    return (on_device(shape_class) and "rsc_user_fit" in shape_class.cuda_source
            and callable(getattr(shape_class, "from_device_record", None)))


def user_cand(s: FittedShape, type_id: int) -> _lib.rsc_cand:
    """The rsc_cand of a device-capable user shape: its `device_record` under the compiled type id."""
    p, outwards = s.device_record()
    p = [float(v) for v in p]
    if len(p) > 7:
        raise ValueError(f"{type(s).__name__}.device_record: at most 7 parameters, got {len(p)}")
    c = _lib.rsc_cand(type=int(type_id), outwards=int(bool(outwards)))
    c.p[:] = p + [0.0] * (7 - len(p))
    return c


def _v3(x):
    a = np.asarray(x, dtype=np.float64).reshape(3)
    return a


@dataclass
class FittedPlane(FittedShape):
    point: np.ndarray
    normal: np.ndarray
    kind = _lib.RSC_PLANE

    def __post_init__(self):
        self.point, self.normal = _v3(self.point), _v3(self.normal)

    def to_cand(self):
        c = _lib.rsc_cand(type=self.kind, outwards=1)
        c.p[:] = [*self.point, *self.normal, 0.0]
        return c


@dataclass
class FittedSphere(FittedShape):
    center: np.ndarray
    radius: float
    outwards: bool
    kind = _lib.RSC_SPHERE

    def __post_init__(self):
        self.center = _v3(self.center)

    def to_cand(self):
        c = _lib.rsc_cand(type=self.kind, outwards=int(bool(self.outwards)))
        c.p[:] = [*self.center, float(self.radius), 0.0, 0.0, 0.0]
        return c


@dataclass
class FittedCylinder(FittedShape):
    axis: np.ndarray
    center: np.ndarray
    radius: float
    outwards: bool
    kind = _lib.RSC_CYLINDER

    def __post_init__(self):
        self.axis, self.center = _v3(self.axis), _v3(self.center)

    def to_cand(self):
        c = _lib.rsc_cand(type=self.kind, outwards=int(bool(self.outwards)))
        c.p[:] = [*self.axis, *self.center, float(self.radius)]
        return c


@dataclass
class FittedCone(FittedShape):
    apex: np.ndarray
    axis: np.ndarray
    opang: float
    outwards: bool
    kind = _lib.RSC_CONE

    def __post_init__(self):
        self.apex, self.axis = _v3(self.apex), _v3(self.axis)

    def to_cand(self):
        c = _lib.rsc_cand(type=self.kind, outwards=int(bool(self.outwards)))
        c.p[:] = [*self.apex, *self.axis, float(self.opang)]
        return c


SHAPE_KIND = {FittedPlane: 0, FittedSphere: 1, FittedCylinder: 2, FittedCone: 3}
KIND_SHAPE = {v: k for k, v in SHAPE_KIND.items()}


def strt(s: FittedShape) -> str:
    """strt (plane.jl:19, sphere.jl:22, cylinder.jl:24, cone.jl:27)."""
    return {0: "plane", 1: "sphere", 2: "cylinder", 3: "cone"}[s.kind]


def from_cand(c: _lib.rsc_cand) -> FittedShape:
    p = list(c.p)
    if c.type == _lib.RSC_PLANE:
        return FittedPlane(p[0:3], p[3:6])
    if c.type == _lib.RSC_SPHERE:
        return FittedSphere(p[0:3], p[3], bool(c.outwards))
    if c.type == _lib.RSC_CYLINDER:
        return FittedCylinder(p[0:3], p[3:6], p[6], bool(c.outwards))
    if c.type == _lib.RSC_CONE:
        return FittedCone(p[0:3], p[3:6], p[6], bool(c.outwards))
    raise ValueError(f"unknown shape type {c.type}")


def pack_cands(shapes: Sequence[FittedShape]):
    """ctypes array of rsc_cand for a list of shapes."""
    arr = (_lib.rsc_cand * max(len(shapes), 1))()
    for i, s in enumerate(shapes):
        arr[i] = s.to_cand()
    return arr


def cands_to_numpy(arr, n: int) -> np.ndarray:
    """View n rsc_cand records as a (n, 8) float64 array (column 0 packs type/outwards)."""
    return np.frombuffer(arr, dtype=np.float64, count=8 * n).reshape(n, 8)


@dataclass
class ExtractedShape:
    """fitting.jl:81-84 -- `inpoints` are ascending 0-based global indices here."""

    shape: FittedShape
    inpoints: np.ndarray
