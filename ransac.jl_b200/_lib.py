"""ctypes binding of libransac_b200.so (include/rsc.h).

There is no CPU fallback: if the shared library is missing this module raises ImportError, and
without an sm_100 device `rsc_ctx_create` fails (RSC_E_NODEVICE) -- loudly, by design.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("RSC_LIB_PATH") or os.path.join(_HERE, "libransac_b200.so")  # (the override is for kernel-variant experiments)

RSC_PLANE, RSC_SPHERE, RSC_CYLINDER, RSC_CONE = 0, 1, 2, 3
RSC_NTYPES = 4
RSC_S_LENGTHC, RSC_S_ALLCAND, RSC_S_NOFMINSET = 0, 1, 2
RSC_COMPAT_SPHERE_IGNORES_ENABLED = 1
RSC_E_NODEVICE = -3
RSC_E_ARG, RSC_E_STATE = -1, -5
RSC_USER_TYPE0 = 16  # type ids of user-defined shapes compiled on a context (rsc_user_shape_compile)

ERRORS = {-1: "RSC_E_ARG", -2: "RSC_E_CUDA", -3: "RSC_E_NODEVICE", -4: "RSC_E_NOMEM", -5: "RSC_E_STATE", -6: "RSC_E_NCCL"}


class rsc_cand(C.Structure):
    _fields_ = [("type", C.c_int32), ("outwards", C.c_int32), ("p", C.c_double * 7)]


class rsc_shape_slot(C.Structure):
    """one position of a fit order (rsc_sample_fit_user, rsc_ransac_run_user): a built-in kind or a user type id"""

    _fields_ = [("type", C.c_int32), ("nk", C.c_int32), ("k", C.c_double * 8)]


RSC_MAX_ORDER = 8


class rsc_params(C.Structure):
    _fields_ = [
        ("drawN", C.c_int32),
        ("minsubsetN", C.c_int32),
        ("prob_det", C.c_double),
        ("tau", C.c_int64),
        ("itermax", C.c_int32),
        ("extract_s", C.c_int32),
        ("terminate_s", C.c_int32),
        ("n_shape_types", C.c_int32),
        ("shape_types", C.c_int32 * 4),
        ("collin_threshold", C.c_double),
        ("parallelthrdeg", C.c_double),
        ("eps", C.c_double * 4),
        ("alpha", C.c_double * 4),
        ("sphere_par", C.c_double),
        ("minconeopang", C.c_double),
        ("compat_flags", C.c_uint32),
        ("lw_period", C.c_uint32),
    ]


class rsc_stats(C.Structure):
    _fields_ = [
        ("evals", C.c_int64),
        ("exact_pairs", C.c_int64),
        ("sets_drawn", C.c_int64),
        ("cands_scored", C.c_int64),
        ("score_launches", C.c_int64),
        ("score_ms", C.c_double),
        ("last_kernel_ms", C.c_double),
        ("refit_mask_ms", C.c_double),
    ]


#: every symbol include/rsc.h declares: (restype, argtypes)
_P = C.c_void_p
SIGNATURES = {
    "rsc_version": (C.c_int32, []),
    "rsc_params_default": (None, [C.POINTER(rsc_params)]),
    "rsc_ctx_create": (C.c_int32, [C.c_int32, C.POINTER(_P)]),
    "rsc_ctx_destroy": (None, [_P]),
    "rsc_last_error": (C.c_char_p, [_P]),
    "rsc_ctx_stats": (C.c_int32, [_P, C.POINTER(rsc_stats)]),
    "rsc_ctx_stream": (_P, [_P]),
    "rsc_ctx_last_kernel": (C.c_int32, [_P, C.POINTER(C.c_double), C.POINTER(C.c_int64)]),
    "rsc_cloud_create": (C.c_int32, [_P, _P, _P, C.c_int64, C.POINTER(_P)]),
    "rsc_cloud_create_f64": (C.c_int32, [_P, _P, _P, C.c_int64, C.POINTER(_P)]),
    "rsc_cloud_create_f64_exact": (C.c_int32, [_P, _P, _P, C.c_int64, C.POINTER(_P)]),
    "rsc_cloud_is_exact": (C.c_int32, [_P]),
    "rsc_cloud_create_shard": (C.c_int32, [_P, _P, _P, C.c_int64, C.c_int64, C.c_int64, C.POINTER(_P)]),
    "rsc_cloud_update": (C.c_int32, [_P, _P, _P, C.c_int64]),
    "rsc_cloud_destroy": (None, [_P]),
    "rsc_cloud_size": (C.c_int64, [_P]),
    "rsc_cloud_set_subset": (C.c_int32, [_P, C.c_int32, _P, C.c_int64]),
    "rsc_cloud_subset_size": (C.c_int64, [_P, C.c_int32]),
    "rsc_cloud_get_enabled": (C.c_int32, [_P, _P]),
    "rsc_cloud_set_enabled": (C.c_int32, [_P, _P]),
    "rsc_cloud_enable_all": (C.c_int32, [_P]),
    "rsc_cloud_count_enabled": (C.c_int64, [_P]),
    "rsc_score": (C.c_int32, [_P, C.POINTER(rsc_params), _P, C.c_int32, C.c_int32, _P, _P]),
    "rsc_score_dev": (C.c_int32, [_P, C.POINTER(rsc_params), _P, C.c_int32, C.c_int32, _P, _P]),
    "rsc_score_dev_masks": (C.c_int32, [_P, C.POINTER(rsc_params), _P, C.c_int32, C.c_int32, _P, _P, _P]),
    "rsc_debug_margins": (C.c_int32, [_P, C.POINTER(rsc_params), _P, C.c_int32, C.c_int64, C.c_int64, _P, _P, _P, C.POINTER(C.c_int64)]),
    "rsc_debug_score_small": (C.c_int32, [_P, C.POINTER(rsc_params), C.c_int32, _P, C.c_int32, C.c_int64, _P, _P]),
    "rsc_debug_k5_hits": (C.c_int32, [_P, C.POINTER(rsc_params), _P, C.c_int32, _P, C.c_int32, C.c_int32, C.c_int32, _P, _P, _P,
                                       C.POINTER(C.c_int32)]),
    "rsc_debug_refit_mask_ms": (C.c_int32, [_P, C.POINTER(rsc_params), C.POINTER(rsc_cand), C.c_int32, C.POINTER(C.c_double), C.POINTER(C.c_int64)]),
    "rsc_estimate_score": (None, [C.c_int64, C.c_int64, C.c_int64, C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_double)]),
    "rsc_fit_batch": (C.c_int32, [_P, C.POINTER(rsc_params), _P, C.c_int32, _P, _P, C.POINTER(C.c_int32)]),
    "rsc_fit_points": (C.c_int32, [_P, C.POINTER(rsc_params), _P, _P, C.c_int32, C.c_int32, _P, _P, C.POINTER(C.c_int32)]),
    "rsc_sample_fit": (C.c_int32, [_P, C.POINTER(rsc_params), C.c_uint64, C.c_uint64, C.c_int32, _P, _P, _P, C.POINTER(C.c_int32)]),
    "rsc_cloud_build_cells": (C.c_int32, [_P, C.c_int32]),
    "rsc_cloud_cells_levels": (C.c_int32, [_P]),
    "rsc_cloud_get_cells": (C.c_int32, [_P, _P, _P, _P]),
    "rsc_sample_fit_cells": (C.c_int32, [_P, C.POINTER(rsc_params), C.c_uint64, C.c_uint64, C.c_int32, _P, C.c_int32, _P, _P, _P, _P,
                                         C.POINTER(C.c_int32)]),
    "rsc_level_cumsum": (None, [_P, C.c_int32, _P]),
    "rsc_update_levelweight": (None, [_P, _P, C.c_int32]),
    "rsc_refit_extract": (C.c_int32, [_P, C.POINTER(rsc_params), C.POINTER(rsc_cand), _P, C.POINTER(C.c_int64), C.c_int32]),
    "rsc_score_culled_subset": (C.c_int32, [_P, C.POINTER(rsc_params), _P, C.c_int32, C.c_int32, _P, C.POINTER(C.c_int64),
                                            C.POINTER(C.c_int64), C.POINTER(C.c_double)]),
    "rsc_score_culled": (C.c_int32, [_P, C.POINTER(rsc_params), _P, C.c_int32, _P, C.POINTER(C.c_int64), C.POINTER(C.c_int64),
                                     C.POINTER(C.c_double)]),
    "rsc_refit_lsq": (C.c_int32, [_P, C.POINTER(rsc_params), C.POINTER(rsc_cand), C.c_double, C.POINTER(rsc_cand),
                                  C.POINTER(C.c_int64), C.POINTER(C.c_double)]),
    "rsc_ctx_set_bitmap": (C.c_int32, [_P, C.c_double, C.c_int32]),
    "rsc_bitmap_filter": (C.c_int32, [_P, C.POINTER(rsc_cand), C.c_double, C.c_int32, _P, C.c_int64, _P, C.POINTER(C.c_int64), _P]),
    "rsc_ctx_set_allreduce": (C.c_int32, [_P, _P, _P]),
    "rsc_comm_unique_id": (C.c_int32, [_P]),
    "rsc_ctx_comm_init": (C.c_int32, [_P, _P, C.c_int32, C.c_int32]),
    "rsc_ctx_comm_destroy": (C.c_int32, [_P]),
    "rsc_ctx_comm_stats": (C.c_int32, [_P, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "rsc_ctx_allreduce": (C.c_int32, [_P, _P, C.c_int64, _P]),
    "rsc_run_shape_total": (C.c_int64, [_P, C.c_int32]),
    "rsc_run_syncs": (C.c_int32, [_P, C.POINTER(C.c_int32)]),
    "rsc_cloud_set_range": (C.c_int32, [_P, C.c_int64, C.c_int64]),
    "rsc_ransac_run": (C.c_int32, [_P, C.POINTER(rsc_params), C.c_uint64, C.POINTER(_P)]),
    "rsc_run_nshapes": (C.c_int32, [_P]),
    "rsc_run_iterations": (C.c_int32, [_P]),
    "rsc_run_refined": (C.c_int64, [_P]),
    "rsc_run_seconds": (C.c_double, [_P]),
    "rsc_run_levelweight": (C.c_int32, [_P, _P, _P]),
    "rsc_run_shape": (C.c_int32, [_P, C.c_int32, C.POINTER(rsc_cand), C.POINTER(C.c_int64)]),
    "rsc_run_inpoints": (C.c_int32, [_P, C.c_int32, _P]),
    "rsc_run_destroy": (None, [_P]),
    "rsc_user_shape_check": (C.c_int32, [_P, C.c_int64, _P, C.c_int64]),
    "rsc_user_shape_compile": (C.c_int32, [_P, _P, C.c_int64, C.POINTER(C.c_int32)]),
    "rsc_user_score": (C.c_int32, [_P, _P, C.c_int32, _P, C.c_int32, C.c_int32, _P, _P]),
    "rsc_user_refit_extract": (C.c_int32, [_P, _P, C.c_int32, C.POINTER(rsc_cand), _P, C.POINTER(C.c_int64), C.c_int32]),
    "rsc_sample_fit_user": (C.c_int32, [_P, C.POINTER(rsc_params), _P, C.c_int32, C.c_uint64, C.c_uint64, C.c_int32, _P, _P, _P,
                                        C.POINTER(C.c_int32)]),
    "rsc_ransac_run_user": (C.c_int32, [_P, C.POINTER(rsc_params), _P, C.c_int32, C.c_uint64, C.POINTER(_P)]),
    "rsc_estimate_normals": (C.c_int32, [_P, _P, C.c_int64, C.c_int32, _P, _P, _P, C.POINTER(C.c_int64)]),
    "rsc_orient_normals": (C.c_int32, [_P, _P, C.c_int64, C.c_int32, _P, _P, _P, _P]),
    "rsc_estimate_normals_shard": (C.c_int32, [_P, _P, C.c_int64, C.c_int64, C.c_int64, C.c_int32, _P, _P, _P,
                                               C.POINTER(C.c_int64)]),
    "rsc_orient_normals_shard": (C.c_int32, [_P, _P, C.c_int64, C.c_int64, C.c_int64, C.c_int32, _P, _P, _P, _P]),
}

if not os.path.exists(LIB_PATH):
    raise ImportError(
        f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
        "(make -C ransac.jl_b200/csrc). There is no CPU fallback."
    )



class _LazyLib:
    """libransac_b200.so, dlopen-ed on first use.  Importing the package (host-side types, parameters,
    scene generators) must not map the CUDA library: bench.py's `--impl reference` arm and the CPU
    oracle tools import those without touching the product.  A missing library is still an import-time
    error (above), and the first call fails loudly if it cannot be loaded."""

    _cdll = None

    def _load(self):
        if _LazyLib._cdll is None:
            cdll = C.CDLL(LIB_PATH)
            for name, (res, args) in SIGNATURES.items():
                f = getattr(cdll, name)  # AttributeError here = header/library mismatch
                f.restype = res
                f.argtypes = args
            _LazyLib._cdll = cdll
        return _LazyLib._cdll

    def __getattr__(self, name):
        return getattr(self._load(), name)


lib = _LazyLib()


def loaded() -> bool:
    """True once libransac_b200.so has been mapped into this process."""
    return _LazyLib._cdll is not None


RSC_SCORE_PROGRESSIVE = 16  # compat_flags: progressive subset scoring in rsc_ransac_run (extension)
RSC_EXTRACT_BITMAP = 32  # compat_flags: keep the largest connected component of the parameter-space bitmap (extension)
RSC_REFIT_LSQ = 8  # compat_flags: least-squares refit before each extraction (extension, include/rsc.h)
RSC_SAMPLER_OCTREE = 2  # compat_flags: level-weighted octree-cell sampler (extension, include/rsc.h)

ALLREDUCE_FN = C.CFUNCTYPE(C.c_int32, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p)


class RscError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"{ERRORS.get(code, code)}: {msg}")
        self.code = code


class Context:
    """One CUDA device + stream (rsc_ctx). Created lazily per device."""

    _by_device: dict = {}

    def __init__(self, device: int = 0):
        h = _P()
        rc = lib.rsc_ctx_create(device, C.byref(h))
        if rc != 0:
            raise RscError(rc, "rsc_ctx_create failed (an sm_100 / B200 device is required; no CPU fallback)")
        self.h = h
        self.device = device
        self._user_types: dict = {}  # user shape class -> type id of its compiled cuda_source

    @classmethod
    def get(cls, device: int = 0) -> "Context":
        if device not in cls._by_device:
            cls._by_device[device] = Context(device)
        return cls._by_device[device]

    def check(self, rc: int):
        if rc != 0:
            raise RscError(rc, lib.rsc_last_error(self.h).decode())

    def stats(self) -> rsc_stats:
        s = rsc_stats()
        self.check(lib.rsc_ctx_stats(self.h, C.byref(s)))
        return s

    def user_type(self, shape_class) -> int:
        """Type id of a user-defined shape class with `cuda_source` on this context: compiled with NVRTC on first
        use (rsc_user_shape_compile; the library caches by source, so equal sources share one id)."""
        tid = self._user_types.get(shape_class)
        if tid is None:
            src = shape_class.cuda_source.encode()
            out = C.c_int32()
            self.check(lib.rsc_user_shape_compile(self.h, src, len(src), C.byref(out)))
            tid = self._user_types[shape_class] = out.value
        return tid

    @property
    def stream(self) -> int:
        return lib.rsc_ctx_stream(self.h) or 0
