"""The Julia shim binds predict_grad for a B200-resident GPE and a GPBatch through gprb_predict_grad, and requires the
prior mean's Jacobian from the caller for a mean other than MeanZero.  The ccall's argument list is checked against the
header by test_julia_shim_signatures.py."""
import os
import re

SHIM = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "gpr.jl_b200", "julia", "GPRB200.jl")


def _src():
    with open(SHIM, encoding="utf-8") as f:
        return re.sub(r"#.*", "", f.read())


def test_predict_grad_surface_is_bound():
    src = _src()
    assert re.search(r"function predict_grad\(gp::B200GPE, x::AbstractMatrix;\s*var::Bool\s*=\s*true,\s*mean_jacobian\s*=\s*nothing\)", src)
    assert re.search(r"function predict_grad\(batch::GPBatch, Xstar::AbstractMatrix;\s*var::Bool\s*=\s*true,\s*mean_jacobian\s*=\s*nothing\)", src)
    assert "ccall((:gprb_predict_grad, LIB)" in src
    assert src.count('throw(ArgumentError("predict_grad: the prior mean') == 2


def test_predict_grad_is_exported_only_where_gaussianprocesses_lacks_it():
    src = _src()
    assert re.search(r"for name in \(:predict_grad,\)\s*if isdefined\(GaussianProcesses, name\)\s*@eval import GaussianProcesses: \$name\s*"
                     r"else\s*@eval function \$name end\s*@eval export \$name\s*end", src)
