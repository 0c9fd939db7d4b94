"""The Julia shim serves predict_f, full_cov and rand! of a B200-resident GPE itself: without these methods
GaussianProcesses' generic predictMVN / rand! would read the placeholder gp.cK and the lazily filled gp.alpha."""
import os
import re

SHIM = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "gpr.jl_b200", "julia", "GPRB200.jl")


def test_prediction_surface_is_bound():
    src = re.sub(r"#.*", "", open(SHIM).read())
    assert re.search(r"GaussianProcesses\.predict_f\(gp::B200GPE,[^)]*;\s*full_cov::Bool\s*=\s*false\)", src)
    assert re.search(r"GaussianProcesses\.predict_y\(gp::B200GPE,[^)]*;\s*full_cov::Bool\s*=\s*false\)", src)
    assert re.search(r"Random\.rand!\(gp::B200GPE,\s*x::AbstractMatrix,\s*A::DenseMatrix\)", src)
    assert "ccall((:gprb_predict_cov, LIB)" in src and "ccall((:gprb_sample_posterior, LIB)" in src
    assert "PosDefException" in src
