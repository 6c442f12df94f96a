"""The Julia binding's side of the device fit of user shapes: its RscShapeSlot mirror has the layout of
include/rsc.h's rsc_shape_slot (checked against the ctypes mirror field by field), and it binds the two calls that
take a fit order (their argument types are checked against the header by test_julia_binding_lint.py)."""
import ctypes as C

from tests.test_julia_binding_lint import BINDING, _ccalls, _ctype_of, _julia_struct


def test_shape_slot_mirror_matches_the_ctypes_struct():
    import ransac_jl_b200 as R

    cs = R._lib.rsc_shape_slot
    jf = _julia_struct("RscShapeSlot")
    assert [f for f, _ in jf] == [f for f, _ in cs._fields_]

    class J(C.Structure):
        _fields_ = [(f, _ctype_of(t)) for f, t in jf]

    assert C.sizeof(J) == C.sizeof(cs) == 72
    for f, _ in jf:
        assert getattr(J, f).offset == getattr(cs, f).offset and getattr(J, f).size == getattr(cs, f).size, f


def test_fit_order_calls_are_bound():
    bound = {c[0] for c in _ccalls(open(BINDING).read())}
    assert {"rsc_sample_fit_user", "rsc_ransac_run_user", "rsc_user_shape_compile"} <= bound
