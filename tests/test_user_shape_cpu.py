"""rsc_user_shape_check needs no GPU: NVRTC compiles the user-shape kernel template together with a user's
rsc_user_compatible for sm_100a on any host.  The two test shapes compile without spills, a broken source is
refused with NVRTC's diagnostic, and a source without the entry function is refused before compiling."""
import ctypes as C
import os
import re
import sys

import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import user_shapes as U  # noqa: E402


def _check(src: str):
    import ransac_jl_b200 as R

    b = src.encode()
    log = C.create_string_buffer(1 << 16)
    rc = R._lib.lib.rsc_user_shape_check(b, len(b), log, len(log))
    return rc, log.value.decode()


@pytest.mark.parametrize("name", ["SLAB_SRC", "TORUS_SRC"])
def test_user_shape_compiles_for_sm100a_without_spills(name):
    rc, log = _check(getattr(U, name))
    assert rc == 0, log
    for kernel in ("rsc_user_score_kernel", "rsc_user_mask_kernel"):
        assert f"Compiling entry function '{kernel}' for 'sm_100a'" in log, log
    spills = re.findall(r"(\d+) bytes spill stores, (\d+) bytes spill loads", log)
    assert len(spills) == 2 and all(s == ("0", "0") for s in spills), log
    regs = [int(r) for r in re.findall(r"Used (\d+) registers", log)]
    assert len(regs) == 2 and max(regs) <= 255


def test_broken_source_is_refused_with_the_diagnostic():
    import ransac_jl_b200 as R

    rc, log = _check(U.BROKEN_SRC)
    assert rc == R._lib.RSC_E_ARG
    assert "rsc_user_shape.cu(4): error" in log, log  # the user's own line number


def test_source_without_entry_function_is_refused():
    import ransac_jl_b200 as R

    rc, log = _check("__device__ bool compatible(double x) { return x > 0.0; }\n")
    assert rc == R._lib.RSC_E_ARG and "rsc_user_compatible" in log
    rc, log = _check("// mentions rsc_user_compatible but does not define it\n__device__ int f() { return 1; }\n")
    assert rc == R._lib.RSC_E_ARG and log


def test_log_is_truncated_to_the_callers_buffer():
    import ransac_jl_b200 as R

    b = U.TORUS_SRC.encode()
    log = C.create_string_buffer(b"\xff" * 17)
    assert R._lib.lib.rsc_user_shape_check(b, len(b), log, 16) == 0
    assert len(log.value) == 15 and log.raw[15:16] == b"\0" and log.raw[16:17] == b"\xff"
    assert R._lib.lib.rsc_user_shape_check(None, 0, None, 0) == R._lib.RSC_E_ARG
