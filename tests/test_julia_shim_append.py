"""The Julia shim binds ElasticGPE's append! for a B200-resident GPE and a GPBatch through gprb_batch_append, by
extending Base.append! (no new export can clash with GaussianProcesses).  The ccall's argument list is checked against
the header by test_julia_shim_signatures.py; here it is checked once more for this entry point alone."""
import os
import re

from test_julia_shim_signatures import JL2C, header_prototypes

SHIM = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "gpr.jl_b200", "julia", "GPRB200.jl")


def _src():
    with open(SHIM, encoding="utf-8") as f:
        return re.sub(r"#.*", "", f.read())


def test_append_surface_is_bound():
    src = _src()
    assert re.search(r"function Base\.append!\(batch::GPBatch, xs::AbstractVector\{<:AbstractMatrix\}, ys::AbstractMatrix\)", src)
    assert re.search(r"function Base\.append!\(gp::B200GPE, x::AbstractMatrix, y::AbstractVector\)", src)
    assert src.count("ccall((:gprb_batch_append, LIB)") == 1
    for field in ("gp.x = ", "gp.y = ", "gp.nobs += k"):
        assert field in src


def test_append_ccall_matches_header():
    src = _src()
    m = re.search(r"ccall\(\(:gprb_batch_append, LIB\), (\w+), \(([^)]*)\)", src)
    assert m
    ret, params = header_prototypes()["gprb_batch_append"]
    assert m.group(1) == "Cint" and ret == "int"
    jl = [t.strip() for t in m.group(2).split(",") if t.strip()]
    assert len(jl) == len(params)
    for j, c in zip(jl, params):
        assert c in JL2C[j], (j, c)


def test_append_adds_no_export():
    src = _src()
    exports = re.findall(r"^\s*export\s+(.*)$", src, flags=re.M)
    assert not any("append" in e for e in exports)
    assert "@eval export append" not in src
