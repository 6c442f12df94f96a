"""The Julia binding exposes device normal estimation: it binds rsc_estimate_normals (its argument types are checked
against the header by test_julia_binding_lint.py, which also checks the INTEGRATION.md snippet)."""
from tests.test_julia_binding_lint import BINDING, _ccalls


def test_estimate_normals_is_bound():
    calls = [c for c in _ccalls(open(BINDING).read()) if c[0] == "rsc_estimate_normals"]
    assert len(calls) == 1 and len(calls[0][2]) == 8
    assert "function estimate_normals(vertices::Vector{SVector{3,Float32}}; k::Integer=16, viewpoint=nothing)" in open(BINDING).read()
