"""The Julia shim serves predict_LOO, logp_CVLOO and dlogpdθ_CVLOO of a B200-resident GPE itself: without these methods
GaussianProcesses' generic cross-validation code would read the placeholder gp.cK and the lazily filled gp.alpha.  The
ccall's argument list is checked against the header by test_julia_shim_signatures.py."""
import os
import re

SHIM = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "gpr.jl_b200", "julia", "GPRB200.jl")


def _src():
    with open(SHIM, encoding="utf-8") as f:
        return re.sub(r"#.*", "", f.read())


def test_cross_validation_surface_is_bound():
    src = _src()
    assert re.search(r"function predict_LOO\(gp::B200GPE\)", src)
    assert re.search(r"function logp_CVLOO\(gp::B200GPE\)", src)
    assert re.search(r"function dlogpdθ_CVLOO\(gp::B200GPE;\s*noise::Bool\s*=\s*true,\s*domean::Bool\s*=\s*true,\s*kern::Bool\s*=\s*true\)", src)
    for name in ("predict_LOO", "logp_CVLOO", "dlogpdθ_CVLOO"):
        assert re.search(name + r"\(batch::GPBatch", src), name
    assert "ccall((:gprb_eval_loo, LIB)" in src


def test_gaussianprocesses_is_extended_only_where_it_defines_the_name():
    src = _src()
    assert re.search(r"for name in \(:predict_LOO, :logp_CVLOO, :dlogpdθ_CVLOO\)", src)
    assert re.search(r"if isdefined\(GaussianProcesses, name\)\s*@eval import GaussianProcesses: \$name\s*else\s*"
                     r"@eval function \$name end\s*@eval export \$name\s*end", src)
