"""Device fits of user-defined shapes compile without a GPU: NVRTC builds rsc_user_fit_kernel for sm_100a next to the
scoring and mask kernels when the source defines rsc_user_fit, without spills; a broken fit is refused with NVRTC's
line number, and a source without a fit compiles as before."""
import ctypes as C
import os
import re
import sys

import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import user_fit_shapes as U  # noqa: E402


def _check(src):
    import ransac_jl_b200 as R

    b = src.encode()
    log = C.create_string_buffer(1 << 16)
    rc = R._lib.lib.rsc_user_shape_check(b, len(b), log, len(log))
    return rc, log.value.decode()


def _entries(log):
    return re.findall(r"Compiling entry function '(\w+)'", log)


@pytest.mark.parametrize("name", ["SLAB_SRC", "ZCYL_SRC"])
def test_fit_kernel_compiles_for_sm100a_without_spills(name):
    rc, log = _check(getattr(U, name))
    assert rc == 0, log
    assert sorted(_entries(log)) == ["rsc_user_fit_kernel", "rsc_user_mask_kernel", "rsc_user_score_kernel"], log
    assert "sm_100a" in log, log
    spills = re.findall(r"(\d+) bytes spill stores, (\d+) bytes spill loads", log)
    assert len(spills) == 3 and all(s == ("0", "0") for s in spills), log


def test_broken_fit_is_refused_with_its_line_number():
    import ransac_jl_b200 as R

    rc, log = _check(U.BROKEN_FIT_SRC)
    assert rc == R._lib.RSC_E_ARG
    assert f"rsc_user_shape.cu({U.BROKEN_FIT_LINE}): error" in log, log


def test_source_without_fit_has_no_fit_kernel():
    rc, log = _check(U.SLAB_COMPAT)
    assert rc == 0, log
    assert sorted(_entries(log)) == ["rsc_user_mask_kernel", "rsc_user_score_kernel"], log


def test_shape_slot_layout():
    import ransac_jl_b200 as R

    s = R._lib.rsc_shape_slot
    assert C.sizeof(s) == 72
    assert (s.type.offset, s.nk.offset, s.k.offset) == (0, 4, 8)
    assert R._lib.RSC_MAX_ORDER == 8


def test_device_fit_helper_and_twins():
    import ransac_jl_b200 as R
    from ransac_jl_b200.shapes import device_fit, on_device

    (NS, NZ), (SS, SZ), (DS, DZ) = U.shape_classes(R)
    assert not any(device_fit(c) for c in (NS, NZ, SS, SZ, R.FittedPlane))
    assert device_fit(DS) and device_fit(DZ) and on_device(SS) and not on_device(NS)
    # the z-cylinder twin: a set on x^2 + y^2 = 4 around (1, 2) fits, parallel normals do not
    import numpy as np

    th = np.array([0.1, 1.7, 3.9, 5.0])
    P = np.c_[1 + 2 * np.cos(th), 2 + 2 * np.sin(th), th]
    N = np.c_[np.cos(th), np.sin(th), 0 * th]
    r = U.zcyl_fit_twin(P, N, U.zcyl_constants())
    assert r is not None and abs(r[0] - 1) < 1e-9 and abs(r[1] - 2) < 1e-9 and abs(r[2] - 2) < 1e-9
    assert U.zcyl_fit_twin(P[[0, 0, 1]], N[[0, 0, 1]], U.zcyl_constants()) is None
    assert U.slab_fit_twin(np.c_[P[:, :2], np.full(4, 3.0)], np.tile([0, 0, 1.0], (4, 1)), U.slab_constants()) == [3.0]
