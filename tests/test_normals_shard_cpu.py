"""The sharded forms of estimate_normals / orient_normals without a device: shape and shard-tuple errors raise
ValueError before any device work, the C entry points refuse a null context, and the bindings declare them."""
import ctypes as C

import numpy as np
import pytest


def _api():
    import ransac_jl_b200 as R

    return R


@pytest.mark.parametrize("shard", [(0,), (0, 1, 2), "ab", (0.5, 10), (None, 10), 7])
def test_shard_must_be_a_pair_of_integers(shard):
    R = _api()
    v = np.zeros((4, 3), np.float32)
    with pytest.raises(ValueError, match="pair"):
        R.estimate_normals(v, shard=shard)
    with pytest.raises(ValueError, match="pair"):
        R.orient_normals(v, shard=shard)


@pytest.mark.parametrize("shard", [(-1, 10), (8, 10), (0, 3), (0, 0), (0, 2**31), (7, 10)])
def test_rows_must_fit_inside_the_global_range(shard):
    R = _api()
    v = np.zeros((4, 3), np.float32)
    with pytest.raises(ValueError, match="n_global"):
        R.estimate_normals(v, shard=shard)
    with pytest.raises(ValueError, match="n_global"):
        R.orient_normals(v, shard=shard)


def test_shapes_are_checked_before_the_shard():
    R = _api()
    with pytest.raises(ValueError, match=r"\(N, 3\)"):
        R.estimate_normals(np.zeros((4, 2), np.float32), shard=(0, 4))
    with pytest.raises(ValueError, match=r"\(N, 3\)"):
        R.orient_normals(np.zeros(12, np.float32), shard=(0, 4))
    with pytest.raises(ValueError, match="shape of vertices"):
        R.orient_normals(np.zeros((4, 3), np.float32), np.zeros((3, 3), np.float32), shard=(0, 4))
    with pytest.raises(ValueError, match="viewpoint"):
        R.estimate_normals(np.zeros((4, 3), np.float32), viewpoint=(1.0, 2.0), shard=(0, 4))


def test_an_empty_rank_is_a_valid_range():
    from ransac_jl_b200.normals import _shard_range

    assert _shard_range("f", (5, 5), 0) == (5, 5)
    assert _shard_range("f", (np.int64(2), 10), 8) == (2, 10)


def test_null_context_is_refused_and_the_bindings_declare_the_entry_points():
    R = _api()
    lib = R._lib.lib
    xyz = np.zeros((4, 3), np.float32)
    nrm = np.zeros((4, 3), np.float32)
    assert lib.rsc_estimate_normals_shard(None, xyz.ctypes.data, 4, 0, 4, 8, None, nrm.ctypes.data, None, None) == R._lib.RSC_E_ARG
    assert lib.rsc_orient_normals_shard(None, xyz.ctypes.data, 4, 0, 4, 8, None, nrm.ctypes.data, None, None) == R._lib.RSC_E_ARG
    sig = R._lib.SIGNATURES
    assert sig["rsc_estimate_normals_shard"][1][2:5] == [C.c_int64] * 3
    assert sig["rsc_estimate_normals_shard"][1][-1] == C.POINTER(C.c_int64)
    assert sig["rsc_orient_normals_shard"][1][2:6] == [C.c_int64, C.c_int64, C.c_int64, C.c_int32]


def test_attach_comm_is_exported_next_to_the_sharded_cloud():
    from ransac_jl_b200 import shard

    assert callable(shard.attach_comm) and callable(shard.detach_comm)
