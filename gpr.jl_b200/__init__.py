"""gpr.jl_b200 - B200-native GP-regression hot path of GPR.jl behind the reference's GP surface.

Layout (only what the path needs):
  csrc/      hand-written sm_100a CUDA kernels + the C ABI (include/gprb200.h) -> libgprb200.so
  lib.py     ctypes binding of the C ABI (the executable stand-in for a Julia ``ccall``)
  gp.py      host-side mirror of the calls the reference makes: SEArd, MeanZero, GP/GPE, optimize!, predict_y
             (+ predict_f, full_cov and rand of the same GaussianProcesses.jl surface, and its leave-one-out
             cross-validation: predict_LOO, logp_CVLOO, dlogpdtheta_CVLOO; predict_grad for the Jacobians of the
             posterior mean and variance with respect to the test inputs; append for ElasticGPE's append!)
  data.py    synthetic CState-shaped datasets (src/CState.jl:20 layout) and theta_0 fixtures
  shard.py   trial -> rank partition and the final gather (torch.distributed)
  julia/     GPRB200.jl ccall shim (written, not runnable in this image)

There is no CPU fallback: importing works anywhere, but every compute entry raises when
libgprb200.so or a B200 is missing.
"""
from .lib import GprbError, Library, load_library, library_path  # noqa: F401
from .gp import (  # noqa: F401
    SEArd, Mat12Ard, Mat32Ard, Mat52Ard, MeanZero, MeanFunction, MeanDynamics, MDCache,
    GPE, GP, GPBatch, LBFGS, BackTracking, Options, optimize, optimize_b, predict_y, predict_f, rand,
    predict_LOO, logp_CVLOO, dlogpdtheta_CVLOO, predict_grad, append,
)

__version__ = "0.1.0"
