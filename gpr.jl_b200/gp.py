"""Host-side mirror of the GP surface the reference calls (GaussianProcesses.jl names and argument meaning),
driving libgprb200.so through the C ABI.  Reference call sites this mirrors (relative to /root/reference):

    kernel = SEArd(log.(params[2:end]), log(params[1]))                 examples/maximal_coordinates/CPnoise.jl:38
    mean   = MeanZero() | MeanDynamics(mechanism, getmu, id, cache)     CPnoise.jl:39, src/mDynamics.jl:13-55
    gp     = GP(xtrain_old, yi, mean, kernel)                           CPnoise.jl:40
    GaussianProcesses.optimize!(gp, LBFGS(linesearch=BackTracking(order=2)), Optim.Options(time_limit=10.))   :41
    mu, s2 = predict_y(gp, obs)                                         examples/utils/predictdynamics.jl:13

Arrays follow Julia's orientation: ``X`` is d x n (one CState sample per column, src/CState.jl:20), ``Xstar`` d x m.
What is new relative to the reference is *batching*: ``GPBatch`` evaluates / optimises / predicts many independent
GPs (the G outputs of a trial, times the trials resident on this GPU) in one library call.  A single ``GP(...)``
is a batch of one, so the reference's per-GP call sequence works unchanged.

The prior mean is evaluated on the host (zero-parameter Mean plug-in protocol of src/mDynamics.jl:29-55) exactly
once per training set - it does not depend on theta - and only ``y - m(X)`` goes to the device.
"""
from __future__ import annotations

import ctypes as C
import math
import os
from dataclasses import dataclass, field

import numpy as np

from .lib import GprbError, LbfgsOpts, OptResult, as_f64, load_library, _d

# ------------------------------------------------------------------------------------------------
# kernels (GaussianProcesses kernels/se_ard.jl, mat*_ard.jl): params [ll_1..ll_d, lsigma]
# ------------------------------------------------------------------------------------------------


class _ArdKernel:
    kind = 0

    def __init__(self, ll, lsigma):
        self.ll = np.array(ll, dtype=np.float64).reshape(-1)
        self.lsigma = float(lsigma)

    @property
    def dim(self):
        return self.ll.size

    def get_params(self):
        return np.concatenate([self.ll, [self.lsigma]])

    def set_params(self, hyp):
        hyp = np.asarray(hyp, dtype=np.float64)
        if hyp.size != self.dim + 1:
            raise ValueError(f"{type(self).__name__} has {self.dim + 1} parameters, got {hyp.size}")
        self.ll = hyp[:-1].copy()
        self.lsigma = float(hyp[-1])

    def num_params(self):
        return self.dim + 1


class SEArd(_ArdKernel):
    """ARD squared exponential, k = s2 exp(-1/2 sum_d (x_d - x'_d)^2 / l_d^2); SEArd(ll, lsigma) takes logs."""
    kind = 0


class Mat12Ard(_ArdKernel):
    kind = 1


class Mat32Ard(_ArdKernel):
    kind = 2


class Mat52Ard(_ArdKernel):
    kind = 3


# ------------------------------------------------------------------------------------------------
# means: the zero-parameter Mean plug-in protocol (src/mDynamics.jl:29-36)
# ------------------------------------------------------------------------------------------------


class MeanFunction:
    def num_params(self):
        return 0

    def get_params(self):
        return np.zeros(0)

    def get_param_names(self):
        return []

    def grad_mean(self, x):
        return np.zeros(0)

    def set_params(self, hyp):
        if len(hyp) != 0:
            raise ValueError("Mean function has no parameters")  # src/mDynamics.jl:34-36

    def mean(self, x):  # x: one sample (d,)
        raise NotImplementedError

    def mean_matrix(self, X):  # X: d x n  ->  [mean(m, X[:, i]) for i]
        return np.array([self.mean(X[:, i]) for i in range(X.shape[1])], dtype=np.float64)

    def jacobian(self, x):  # x: one sample (d,)  ->  d m(x) / dx, (d,); needed by predict_grad
        raise NotImplementedError(f"{type(self).__name__} has no jacobian(x)")


class MeanZero(MeanFunction):
    def mean(self, x):
        return 0.0

    def mean_matrix(self, X):
        return np.zeros(X.shape[1])


class MDCache:
    """Single-entry cache shared by the G GPs of a trial (src/mDynamics.jl:6-11)."""

    def __init__(self):
        self.key = np.zeros(0)
        self.data = np.zeros(0)


class MeanDynamics(MeanFunction):
    """Prior mean = component ``muID`` of the nominal one-step dynamics (src/mDynamics.jl:13-55).

    ``mechanism`` is any host callable ``state(13N,) -> next state(13N,)`` standing in for
    ``setstates!`` + ``ConstrainedDynamics.newton!`` (ConstrainedDynamics.jl stays on the host and is not part of
    this path); ``getmu(next_state) -> vector`` selects the output coordinates (``getμ(ids)``, mDynamics.jl:57-60).
    """

    def __init__(self, mechanism, getmu, muID, cache=None, xtransform=None):
        self.mechanism = mechanism
        self.getmu = getmu
        self.muID = int(muID)  # 1-based like the reference
        self.cache = cache if cache is not None else MDCache()
        self.xtransform = xtransform or (lambda x, _m: x)

    def mean(self, x):
        x = np.asarray(x, dtype=np.float64)
        c = self.cache
        if c.key.shape != x.shape or not np.array_equal(c.key, x):  # cache invalid (mDynamics.jl:42)
            c.key = x.copy()
            c.data = np.asarray(self.getmu(self.mechanism(self.xtransform(x, self.mechanism))), dtype=np.float64)
        return float(c.data[self.muID - 1])


def getmu(ids):
    """``getμ(ids)`` (src/mDynamics.jl:57-60): 1-based CState indices of the predicted coordinates."""
    idx = np.asarray(ids, dtype=np.int64) - 1
    return lambda state: np.asarray(state)[idx]


# ------------------------------------------------------------------------------------------------
# optimiser configuration objects (Optim.jl / LineSearches.jl names)
# ------------------------------------------------------------------------------------------------


@dataclass
class BackTracking:
    order: int = 2
    c_1: float = 1e-4
    rho_hi: float = 0.5
    rho_lo: float = 0.1
    iterations: int = 1000


@dataclass
class LBFGS:
    m: int = 10
    linesearch: BackTracking = field(default_factory=BackTracking)


@dataclass
class Options:
    """Optim.Options subset.  The reference gives every GP its own ``time_limit=10.`` seconds of CPU wall clock
    (CPnoise.jl:41).  With ``cost_value`` / ``cost_grad`` (seconds one value-only / value+gradient evaluation takes on the
    machine being emulated, e.g. the reference CPU) the limit runs on a deterministic PER-GP virtual clock - what
    "10 s per GP" means there, reproducibly; without them ``time_limit`` is the wall clock of the whole lock-step
    batch.  ``max_evals`` (per-GP cap on evaluations) and ``iterations`` are the other deterministic stopping rules."""
    time_limit: float = float("nan")
    iterations: int = 1000
    g_abstol: float = 1e-8
    max_evals: int = 0
    cost_value: float = 0.0
    cost_grad: float = 0.0


# ------------------------------------------------------------------------------------------------
# context
# ------------------------------------------------------------------------------------------------


class _Context:
    _inst = None

    def __init__(self):
        self.lib = load_library()
        dev = int(os.environ.get("GPRB200_DEVICE", os.environ.get("LOCAL_RANK", "0")))
        h = C.c_void_p()
        self.lib.check(self.lib.dll.gprb_init(C.byref(h), dev))
        self.handle = h
        self.device = dev

    @classmethod
    def get(cls):
        if cls._inst is None:
            cls._inst = _Context()
        return cls._inst

    def launch_count(self):
        return int(self.lib.dll.gprb_launch_count(self.handle))

    def device_info(self):
        out = (C.c_int64 * 4)()
        self.lib.check(self.lib.dll.gprb_device_info(self.handle, out))
        return {"sm_count": out[0], "clock_khz": out[1], "l2_bytes": out[2], "free_bytes": out[3]}

    # -- multi-GPU: the library's own NCCL communicator (one rank per process) and the final gather ----------
    def comm_init(self, rank=None, world=None):
        """Join this process's context into the library's NCCL clique.  Rank 0 draws the unique id
        (gprb_comm_unique_id) and it travels through torch.distributed's broadcast - any host-side channel would do
        (Distributed.jl / MPI / a file on the Julia side); the data path itself never touches torch."""
        import torch
        import torch.distributed as dist
        rank = dist.get_rank() if rank is None else rank
        world = dist.get_world_size() if world is None else world
        if world == 1 or getattr(self, "_comm", False):
            return
        buf = (C.c_ubyte * 128)()
        if rank == 0:
            self.lib.check(self.lib.dll.gprb_comm_unique_id(buf))
        t = torch.tensor(list(bytes(buf)), dtype=torch.uint8)
        if dist.get_backend() == "nccl":
            t = t.cuda(self.device)
        dist.broadcast(t, 0)
        idb = (C.c_ubyte * 128)(*t.cpu().tolist())
        self.lib.check(self.lib.dll.gprb_comm_init_rank(self.handle, world, rank, idb))
        self._comm = True

    def gather(self, local: dict, n_rows: int, width: int):
        """gprb_gather: {global row id -> (width,) float64} of this rank -> (n_rows, width) on every rank (NaN rows
        where nobody contributed).  One ncclAllGather over NVLink inside libgprb200.so."""
        ids = np.ascontiguousarray(sorted(local), dtype=np.int32)
        rows = np.ascontiguousarray(np.stack([np.asarray(local[int(i)], dtype=np.float64) for i in ids])
                                    if len(ids) else np.zeros((0, width)))
        out = np.empty((n_rows, width))
        self.lib.check(self.lib.dll.gprb_gather(self.handle, n_rows, width, len(ids),
                                                ids.ctypes.data_as(C.POINTER(C.c_int32)), _d(rows), _d(out)))
        return out


def context():
    return _Context.get()


# ------------------------------------------------------------------------------------------------
# GPE / GPBatch
# ------------------------------------------------------------------------------------------------


class GPE:
    """Exact GP with Gaussian likelihood (GaussianProcesses.GPE): fields read by the reference's callers."""

    def __init__(self, X, y, mean, kernel, logNoise=-2.0):
        X = np.asarray(X, dtype=np.float64)
        y = np.asarray(y, dtype=np.float64).reshape(-1)
        if X.ndim != 2 or X.shape[1] != y.size:
            raise ValueError(f"X must be d x n with n = length(y); got X {X.shape}, y {y.shape}")
        if kernel.dim != X.shape[0]:
            raise ValueError(f"kernel has {kernel.dim} length-scales but X has {X.shape[0]} rows")
        self.x = X
        self.y = y
        self.mean = mean
        self.kernel = kernel
        self.logNoise = float(logNoise)
        self.dim, self.nobs = X.shape
        self._batch = None
        self._slot = -1
        self._res = (float("nan"), None, 0)  # (mll, dmll, info) while the GP is not resident in a batch

    # Results of the last evaluation.  While the GP is resident in a GPBatch they are views into the batch's result
    # arrays (one vectorised store per evaluation instead of a Python loop over the GPs of the batch).
    @property
    def mll(self):
        b = self._batch
        return float(b._mll[self._slot]) if b is not None else self._res[0]

    @property
    def dmll(self):
        b = self._batch
        if b is None:
            return self._res[1]
        return b._grad[self._slot].copy() if b._has_grad[self._slot] else None

    @property
    def info(self):
        b = self._batch
        return int(b._info[self._slot]) if b is not None else self._res[2]

    # GaussianProcesses.get_params order: [logNoise; mean params (none); kernel params]
    def get_params(self):
        return np.concatenate([[self.logNoise], self.mean.get_params(), self.kernel.get_params()])

    def set_params(self, hyp):
        hyp = np.asarray(hyp, dtype=np.float64)
        self.logNoise = float(hyp[0])
        self.kernel.set_params(hyp[1:])

    @property
    def target(self):
        return self.mll

    @property
    def alpha(self):
        return self._batch.alpha(self._slot)


def GP(X, y, mean, kernel, logNoise=-2.0):
    """``GP(X, y, mean, kernel)``: construct and run the initial ``update_mll!`` (a batch of one)."""
    gp = GPE(X, y, mean, kernel, logNoise)
    GPBatch([gp]).update_mll()
    return gp


class GPBatch:
    """B independent GPs resident on one GPU.  GPs that share the same ``X`` array object share one device
    dataset (the G outputs of a trial, CPnoise.jl:37-43)."""

    def __init__(self, gps):
        gps = list(gps)
        if not gps:
            raise ValueError("empty batch")
        self.gps = gps
        self.ctx = context()
        self.lib = self.ctx.lib
        d, n = gps[0].dim, gps[0].nobs
        kind = gps[0].kernel.kind
        for g in gps:
            if (g.dim, g.nobs) != (d, n) or g.kernel.kind != kind:
                raise ValueError("all GPs of a batch must share d, n and the kernel family")
        self.d, self.n, self.P, self.B = d, n, d + 2, len(gps)
        self._ds = {}
        ds_handles = (C.c_void_p * self.B)()
        ymm = np.empty((self.B, n))
        # per-GP results of the last evaluation (GPE.mll / .dmll / .info read them); seeded with what the GPs carry
        prev = [(g.mll, g.dmll, g.info) for g in gps]
        self._mll = np.array([r[0] for r in prev], dtype=np.float64)
        self._info = np.array([r[2] for r in prev], dtype=np.int32)
        self._grad = np.full((self.B, self.P), np.nan)
        self._has_grad = np.zeros(self.B, dtype=bool)
        for b, r in enumerate(prev):
            if r[1] is not None:
                self._grad[b], self._has_grad[b] = r[1], True
        # all distinct training sets of the batch live in ONE device allocation and go up in one copy + one transpose
        # launch (gprb_datasets_create); the host block is (T, n, d) C-order == T column-major d x n matrices back to back
        uniq = {}
        for g in gps:
            uniq.setdefault(id(g.x), g.x)
        self._keep = list(uniq.values())
        block = np.empty((len(uniq), n, d))
        for t, Xu in enumerate(self._keep):
            block[t] = Xu.T
        hs = (C.c_void_p * len(uniq))()
        ptrs = (C.POINTER(C.c_double) * len(uniq))(*[_d(block[t]) for t in range(len(uniq))])
        self.lib.check(self.lib.dll.gprb_datasets_create(self.ctx.handle, len(uniq), n, d, ptrs, d, hs))
        for key, h in zip(uniq, hs):
            self._ds[key] = C.c_void_p(h)
        for b, g in enumerate(gps):
            ds_handles[b] = self._ds[id(g.x)]
            g._batch, g._slot = self, b
        # m(X) is theta-independent (zero-parameter means, src/mDynamics.jl:29-31): evaluated once per training set,
        # column-major across the GPs of a trial so a shared MDCache hits for the other G-1 outputs.
        mX = self._means([g.x for g in gps])
        for b, g in enumerate(gps):
            ymm[b] = g.y - mX[b]
        self.ymm = ymm
        h = C.c_void_p()
        self.lib.check(self.lib.dll.gprb_batch_create(self.ctx.handle, self.B, ds_handles, _d(ymm), kind, C.byref(h)))
        self.handle = h

    def close(self):
        """Free the device memory of the batch and its datasets now (GPE <-> GPBatch reference cycles otherwise keep it
        alive until the garbage collector runs - tens of GB at the benchmark sizes)."""
        if getattr(self, "handle", None):
            self.lib.dll.gprb_batch_destroy(self.handle)
            self.handle = None
        for h in getattr(self, "_ds", {}).values():
            self.lib.dll.gprb_dataset_destroy(h)
        self._ds = {}
        for g in getattr(self, "gps", []):
            if g._batch is self:
                g._res = (g.mll, g.dmll, g.info)  # the GP keeps its last results
                g._batch, g._slot = None, -1

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _means(self, blocks):
        """m(block_b[:, s]) for every GP b and column s -> list of (m_b,) arrays; GPs sharing the same block object
        are evaluated column by column together (MDCache semantics of src/mDynamics.jl:41-55)."""
        out = [None] * self.B
        groups = {}
        for b, (g, blk) in enumerate(zip(self.gps, blocks)):
            if isinstance(g.mean, MeanZero):
                out[b] = np.zeros(blk.shape[1])
            else:
                groups.setdefault(id(blk), []).append(b)
        for members in groups.values():
            blk = blocks[members[0]]
            vals = np.empty((len(members), blk.shape[1]))
            for s in range(blk.shape[1]):
                x = np.ascontiguousarray(blk[:, s])
                for k, b in enumerate(members):
                    vals[k, s] = self.gps[b].mean.mean(x)
            for k, b in enumerate(members):
                out[b] = vals[k]
        return out

    # -- parameters ---------------------------------------------------------------------------
    def get_params(self):
        return np.stack([g.get_params() for g in self.gps])  # (B, P)

    def set_params(self, theta):
        for g, t in zip(self.gps, np.asarray(theta)):
            g.set_params(t)

    # -- evaluation ---------------------------------------------------------------------------
    def eval(self, theta=None, grad=True, active=None):
        """One objective evaluation per active GP -> (mll (B,), grad (B,P) or None, info (B,))."""
        theta = as_f64(self.get_params() if theta is None else theta).reshape(self.B, self.P)
        mll = np.full(self.B, np.nan)
        g = np.full((self.B, self.P), np.nan) if grad else None
        info = np.zeros(self.B, dtype=np.int32)
        act = None
        if active is not None:
            act = np.ascontiguousarray(active, dtype=np.uint8)
        self.lib.check(self.lib.dll.gprb_eval(
            self.handle, _d(theta), act.ctypes.data_as(C.POINTER(C.c_uint8)) if act is not None else None,
            _d(mll), _d(g), info.ctypes.data_as(C.POINTER(C.c_int32))))
        sel = slice(None) if act is None else act.astype(bool)
        self._mll[sel], self._info[sel], self._has_grad[sel] = mll[sel], info[sel], bool(grad)
        if grad:
            self._grad[sel] = g[sel]
        return mll, g, info

    def eval_mixed(self, theta, mode):
        """gprb_eval_mixed: mode[b] = 0 skip / 1 value only / 2 value + gradient, one pipeline pass for all of them.
        -> (mll (B,), grad (B,P) with NaN rows where no gradient was asked, info (B,))."""
        theta = as_f64(theta).reshape(self.B, self.P)
        mode = np.ascontiguousarray(mode, dtype=np.uint8)
        mll = np.full(self.B, np.nan)
        g = np.full((self.B, self.P), np.nan)
        info = np.zeros(self.B, dtype=np.int32)
        self.lib.check(self.lib.dll.gprb_eval_mixed(self.handle, _d(theta), mode.ctypes.data_as(C.POINTER(C.c_uint8)),
                                                    _d(mll), _d(g), info.ctypes.data_as(C.POINTER(C.c_int32))))
        sel, wg = mode != 0, mode == 2
        self._mll[sel], self._info[sel], self._has_grad[sel] = mll[sel], info[sel], wg[sel]
        self._grad[wg] = g[wg]
        return mll, g, info

    def eval_loo(self, theta=None, grad=True, active=None, mu_var=False):
        """Leave-one-out cross-validation (gprb_eval_loo): evaluates like ``eval(theta, grad=True)`` - the batch's mll,
        dmll and info are updated - then logp_CVLOO and, with ``grad``, its gradient for every active GP.
        -> (logp (B,), grad (B,P) | None, info (B,)); with ``mu_var`` also (mu (B,n), var (B,n)) of y - m(X).
        A GP with info < 0 gets logp = -Inf and NaN rows; rows of inactive GPs are NaN."""
        theta = as_f64(self.get_params() if theta is None else theta).reshape(self.B, self.P)
        mll = np.full(self.B, np.nan)
        g = np.full((self.B, self.P), np.nan)
        logp = np.full(self.B, np.nan)
        gl = np.full((self.B, self.P), np.nan) if grad else None
        mu = np.full((self.B, self.n), np.nan) if mu_var else None
        var = np.full((self.B, self.n), np.nan) if mu_var else None
        info = np.zeros(self.B, dtype=np.int32)
        act = None if active is None else np.ascontiguousarray(active, dtype=np.uint8)
        self.lib.check(self.lib.dll.gprb_eval_loo(
            self.handle, _d(theta), act.ctypes.data_as(C.POINTER(C.c_uint8)) if act is not None else None,
            _d(mll), _d(g), _d(logp), _d(gl), _d(mu), _d(var), info.ctypes.data_as(C.POINTER(C.c_int32))))
        sel = slice(None) if act is None else act.astype(bool)
        self._mll[sel], self._info[sel], self._has_grad[sel] = mll[sel], info[sel], True
        self._grad[sel] = g[sel]
        if mu_var:
            return logp, gl, info, (mu, var)
        return logp, gl, info

    def predict_LOO(self, active=None):
        """``predict_LOO``: leave-one-out predictive mean (m(X) included) and variance of every training point
        -> (mu (B,n), var (B,n)), NaN rows for a GP whose evaluation failed."""
        _, _, _, (mu, var) = self.eval_loo(grad=False, active=active, mu_var=True)
        return mu + np.stack(self._means([g.x for g in self.gps])), var

    def eval_device(self, theta_ptr, mll_ptr, grad_ptr=None, info_ptr=None, stream=0):
        """gprb_eval_device: theta (B,P) / mll (B,) / grad (B,P) / info (B,) are raw device pointers (ints, e.g.
        ``torch.Tensor.data_ptr()``); no payload crosses PCIe.  Ordered after ``stream`` (a cudaStream_t handle)."""
        self.lib.check(self.lib.dll.gprb_eval_device(self.handle, C.c_void_p(theta_ptr), C.c_void_p(mll_ptr),
                                                     C.c_void_p(grad_ptr) if grad_ptr else None,
                                                     C.c_void_p(info_ptr) if info_ptr else None, C.c_void_p(stream)))

    def update_data(self, trials_X=None, ymm=None):
        """Re-upload inputs into the resident allocations: ``trials_X`` = list of new d x n arrays, one per distinct
        dataset in creation order; ``ymm`` (B, n) new targets (y - m(X))."""
        if trials_X is not None:
            hs = list(self._ds.values())
            if len(trials_X) != len(hs):
                raise ValueError(f"expected {len(hs)} input matrices, got {len(trials_X)}")
            keep = [as_f64(np.asarray(Xn).T) for Xn in trials_X]  # views when Xn is already d x n column-major
            harr = (C.c_void_p * len(hs))(*[h.value for h in hs])
            parr = (C.POINTER(C.c_double) * len(hs))(*[_d(k) for k in keep])
            self.lib.check(self.lib.dll.gprb_datasets_update(self.ctx.handle, len(hs), harr, parr, self.d))
        if ymm is not None:
            ymm = as_f64(ymm).reshape(self.B, self.n)
            self.lib.check(self.lib.dll.gprb_batch_set_targets(self.handle, _d(ymm)))
            self.ymm = ymm

    def append(self, trials_X_new, Y_new):
        """``append!`` for every GP of the batch (gprb_batch_append): ``trials_X_new`` holds one d x k array per distinct
        dataset in creation order (as for ``update_data``), ``Y_new`` (B, k) the raw targets of the new samples.  The batch
        subtracts m(X_new) itself.  Every GP with a resident state is conditioned on its enlarged data at the theta of
        that state, bit-identical to a fresh value-only evaluation there -> (mll (B,), info (B,)); GPs without a state
        get NaN / 0 and stay without one."""
        keys = list(self._ds)
        if len(trials_X_new) != len(keys):
            raise ValueError(f"expected {len(keys)} input blocks, got {len(trials_X_new)}")
        blocks = [np.asarray(x, dtype=np.float64) for x in trials_X_new]
        k = blocks[0].shape[1] if blocks[0].ndim == 2 else 0
        for x in blocks:
            if x.ndim != 2 or x.shape != (self.d, k):
                raise ValueError(f"every input block must be d x k = {self.d} x {k}, got {x.shape}")
        if k < 1:
            raise ValueError("append needs at least one new sample")
        Y_new = np.asarray(Y_new, dtype=np.float64).reshape(self.B, k)
        trial = {key: t for t, key in enumerate(keys)}
        gp_blocks = [blocks[trial[id(g.x)]] for g in self.gps]
        ymm_new = as_f64(Y_new - np.stack(self._means(gp_blocks)))
        keep = [as_f64(x.T) for x in blocks]  # k x d C-order = d x k column-major
        parr = (C.POINTER(C.c_double) * len(keep))(*[_d(x) for x in keep])
        mll = np.full(self.B, np.nan)
        info = np.zeros(self.B, dtype=np.int32)
        self.lib.check(self.lib.dll.gprb_batch_append(self.handle, k, parr, self.d, _d(ymm_new), _d(mll),
                                                      info.ctypes.data_as(C.POINTER(C.c_int32))))
        # one new x per trial, still shared by the trial's GPs (the dataset key is the array's identity)
        grown = {key: np.concatenate([self._keep[t], blocks[t]], axis=1) for t, key in enumerate(keys)}
        for b, g in enumerate(self.gps):
            g.x = grown[id(g.x)]
            g.y = np.concatenate([g.y, Y_new[b]])
            g.nobs += k
        self._ds = {id(grown[key]): self._ds[key] for key in keys}
        self._keep = [grown[key] for key in keys]
        self.n += k
        self.ymm = np.concatenate([self.ymm, ymm_new], axis=1)
        sel = ~np.isnan(mll)
        self._mll[sel], self._info[sel], self._has_grad[sel] = mll[sel], info[sel], False
        return mll, info

    def set_diag_offset(self, offset=None):
        """gprb_batch_set_diag_offset: fixed per-GP nugget added to the diagonal of K (None resets it)."""
        off = None if offset is None else as_f64(np.broadcast_to(np.asarray(offset, dtype=np.float64), (self.B,)).copy())
        self.lib.check(self.lib.dll.gprb_batch_set_diag_offset(self.handle, _d(off)))

    def update_mll(self):
        return self.eval(grad=False)

    def update_mll_and_dmll(self):
        return self.eval(grad=True)

    # -- optimisation -------------------------------------------------------------------------
    def optimize(self, method: LBFGS | None = None, options: Options | None = None):
        method = method or LBFGS()
        options = options or Options()
        if method.linesearch.order != 2:
            raise ValueError("only BackTracking(order=2) - the reference's choice - is implemented")
        o = LbfgsOpts()
        self.lib.dll.gprb_lbfgs_default_opts(C.byref(o))
        o.m = method.m
        o.iterations = options.iterations
        o.max_evals = options.max_evals
        o.ls_iterations = method.linesearch.iterations
        o.g_abstol = options.g_abstol
        o.time_limit = options.time_limit if math.isfinite(options.time_limit) else 0.0
        o.cost_value, o.cost_grad = options.cost_value, options.cost_grad
        o.c_1, o.rho_hi, o.rho_lo = method.linesearch.c_1, method.linesearch.rho_hi, method.linesearch.rho_lo
        theta = as_f64(self.get_params()).copy()
        res = (OptResult * self.B)()
        self.lib.check(self.lib.dll.gprb_optimize(self.handle, _d(theta), C.byref(o), res))
        self.set_params(theta)
        out = []
        for b, gp in enumerate(self.gps):
            r = res[b]
            self._mll[b], self._info[b], self._has_grad[b] = r.mll, r.info, False
            out.append({"minimizer": theta[b].copy(), "minimum": -r.mll, "g_norm": r.g_norm, "iterations": r.iterations,
                        "f_calls": r.f_calls, "g_calls": r.fg_calls, "converged": bool(r.converged),
                        "ls_failed": bool(r.ls_failed), "info": r.info})
        return out

    # -- prediction ---------------------------------------------------------------------------
    def _test_block(self, Xstar, per_gp):
        """Staged test inputs for gprb_predict / gprb_predict_cov / gprb_sample_posterior -> (Xs, stride, m, mstar|None)."""
        if per_gp:
            blocks = [as_f64(np.asarray(x, dtype=np.float64).T) for x in Xstar]
            m = blocks[0].shape[0]
            Xs = np.ascontiguousarray(np.stack(blocks))  # (B, m, d)
            stride = m * self.d
            xs_cols = [np.asarray(x, dtype=np.float64) for x in Xstar]
        else:
            Xstar = np.asarray(Xstar, dtype=np.float64)
            if Xstar.ndim == 1:
                Xstar = Xstar.reshape(-1, 1)
            m = Xstar.shape[1]
            Xs = as_f64(Xstar.T)
            stride = 0
            xs_cols = None
        mstar = None
        if not all(isinstance(g.mean, MeanZero) for g in self.gps):
            mstar = np.ascontiguousarray(np.stack(self._means(xs_cols if per_gp else [Xstar] * self.B)))
        return Xs, stride, m, mstar

    def predict_y(self, Xstar, var=True, per_gp=False, full_cov=False):
        """Xstar d x m shared by all GPs, or (per_gp=True) a sequence of B d x m blocks.  -> mu (B,m), var (B,m)|None;
        full_cov=True: mu (B,m), Sigma_y (B,m,m) (``predict_y(gp, X*; full_cov=true)``)."""
        if full_cov:
            return self._predict_cov(Xstar, per_gp, add_noise=True)
        Xs, stride, m, mstar = self._test_block(Xstar, per_gp)
        mu = np.empty((self.B, m))
        v = np.empty((self.B, m)) if var else None
        self.lib.check(self.lib.dll.gprb_predict(self.handle, m, _d(Xs), stride, _d(mstar), _d(mu), _d(v)))
        return mu, v

    def predict_f(self, Xstar, full_cov=False, per_gp=False):
        """Latent posterior (``predict_f``): mu (B,m) and var_f (B,m) = max(predict_y's variance - exp(2 logNoise), 0),
        or with full_cov=True Sigma_f (B,m,m) = K** - K*' K^-1 K* (symmetric, not clamped)."""
        if full_cov:
            return self._predict_cov(Xstar, per_gp, add_noise=False)
        mu, v = self.predict_y(Xstar, var=True, per_gp=per_gp)
        noise = np.exp(2.0 * np.array([g.logNoise for g in self.gps]))
        return mu, np.maximum(v - noise[:, None], 0.0)

    def _predict_cov(self, Xstar, per_gp, add_noise):
        Xs, stride, m, mstar = self._test_block(Xstar, per_gp)
        mu = np.empty((self.B, m))
        cov = np.empty((self.B, m, m))
        self.lib.check(self.lib.dll.gprb_predict_cov(self.handle, m, _d(Xs), stride, _d(mstar), 1 if add_noise else 0,
                                                     _d(mu), _d(cov)))
        return mu, cov.transpose(0, 2, 1)  # column-major m x m per GP; Sigma is symmetric, the transpose is a free view

    def rand(self, Xstar, nsamples=1, Z=None, rng=None, per_gp=False):
        """Posterior draws of the latent function at Xstar (``rand(gp, X*, n)``): draws[b] = mu_b 1' + L_b Z[b] with
        L_b the lower factor of make_posdef!(Sigma_f).  Z (B, m, nsamples) standard normals; by default drawn from
        ``rng`` (a numpy Generator) GP by GP in Julia's ``randn(m, n)`` order.  -> (draws (B, m, ns), info (B,)):
        info 0..10 = jitter rung, -1 = indefinite after 10 jitters, -2 = non-finite Sigma_f or no state (NaN draws)."""
        Xs, stride, m, mstar = self._test_block(Xstar, per_gp)
        if Z is None:
            rng = np.random.default_rng() if rng is None else rng
            Zc = rng.standard_normal((self.B, nsamples, m))  # per GP: column-major m x ns, filled column by column
        else:
            Z = np.asarray(Z, dtype=np.float64)
            if Z.shape != (self.B, m, nsamples):
                raise ValueError(f"Z must have shape {(self.B, m, nsamples)}, got {Z.shape}")
            Zc = Z.transpose(0, 2, 1)
        Zc = np.ascontiguousarray(Zc, dtype=np.float64)
        out = np.empty((self.B, nsamples, m))
        info = np.zeros(self.B, dtype=np.int32)
        self.lib.check(self.lib.dll.gprb_sample_posterior(self.handle, m, _d(Xs), stride, _d(mstar), nsamples, _d(Zc), _d(out),
                                                          info.ctypes.data_as(C.POINTER(C.c_int32))))
        return out.transpose(0, 2, 1), info

    def predict_grad(self, Xstar, var=True, per_gp=False):
        """Posterior mean and variance with their Jacobians with respect to the test inputs (gprb_predict_grad)
        -> (mu (B,m), var (B,m) | None, dmu (B,m,d), dvar (B,m,d) | None); dmu[b, j, p] = d mu_bj / d x*_jp.
        ``var=False`` computes the mean and its Jacobian only (no triangular substitution).  dvar is the gradient of the
        unclamped variance K** - k*' K^-1 k* (the same for predict_f and predict_y; the floor at 0 is not differentiated).
        A prior mean other than MeanZero must implement ``jacobian(x)``."""
        for g in self.gps:
            if not isinstance(g.mean, MeanZero) and type(g.mean).jacobian is MeanFunction.jacobian:
                raise NotImplementedError(f"predict_grad: the prior mean {type(g.mean).__name__} has no jacobian(x)")
        Xs, stride, m, mstar = self._test_block(Xstar, per_gp)
        dmstar = None
        if mstar is not None:
            blocks = [np.asarray(x, dtype=np.float64) for x in Xstar] if per_gp else [Xs.T] * self.B
            dmstar = np.zeros((self.B, m, self.d))
            for b, g in enumerate(self.gps):
                if not isinstance(g.mean, MeanZero):
                    for s in range(m):
                        dmstar[b, s] = g.mean.jacobian(np.ascontiguousarray(blocks[b][:, s]))
        mu = np.empty((self.B, m))
        v = np.empty((self.B, m)) if var else None
        dmu = np.empty((self.B, m, self.d))
        dv = np.empty((self.B, m, self.d)) if var else None
        self.lib.check(self.lib.dll.gprb_predict_grad(self.handle, m, _d(Xs), stride, _d(mstar), _d(dmstar), _d(mu), _d(v),
                                                      _d(dmu), _d(dv)))
        return mu, v, dmu, dv

    def predict_async(self, slot, gp0, gp1, blocks, var=False, gps_per_block=1):
        """gprb_predict_async: enqueue the prediction of GPs gp0..gp1-1 on pipeline ``slot`` (0 or 1) and return at
        once.  ``blocks``: one d x m array shared by the range, or a sequence of d x m blocks, one per ``gps_per_block``
        consecutive GPs (the G outputs of a trial read the trial's own states).  Prior means m(x*) are evaluated here
        on the host (src/mDynamics.jl:41-55) before the call, like predict_y."""
        cnt = gp1 - gp0
        if isinstance(blocks, np.ndarray) and blocks.ndim == 2:
            Xs, stride, m = as_f64(blocks.T), 0, blocks.shape[1]
            cols = [blocks] * cnt
        else:
            blks = [np.asarray(x, dtype=np.float64) for x in blocks]
            if len(blks) != (cnt + gps_per_block - 1) // gps_per_block:
                raise ValueError("one test block per gps_per_block GPs expected")
            m = blks[0].shape[1]
            Xs = np.ascontiguousarray(np.stack([c.T for c in blks]))  # (blocks, m, d)
            stride = m * self.d
            cols = [blks[k // gps_per_block] for k in range(cnt)]
        mstar = None
        if not all(isinstance(g.mean, MeanZero) for g in self.gps[gp0:gp1]):
            mstar = np.ascontiguousarray(np.stack(self._means_range(gp0, gp1, cols)))
        self.lib.check(self.lib.dll.gprb_predict_async(self.handle, slot, gp0, gp1, m, _d(Xs), stride, gps_per_block,
                                                       _d(mstar), 1 if var else 0))
        self._pending = getattr(self, "_pending", {})
        self._pending[slot] = (cnt, m, var)

    def predict_wait(self, slot):
        """gprb_predict_wait -> (mu (cnt, m), var (cnt, m) | None) of the prediction enqueued on ``slot``."""
        cnt, m, var = self._pending.pop(slot)
        mu = np.empty((cnt, m))
        v = np.empty((cnt, m)) if var else None
        self.lib.check(self.lib.dll.gprb_predict_wait(self.handle, slot, _d(mu), _d(v)))
        return mu, v

    def last_predict_ms(self, slot=0):
        out = np.zeros(1)
        self.lib.check(self.lib.dll.gprb_last_predict_ms(self.handle, slot, _d(out)))
        return float(out[0])

    def _means_range(self, gp0, gp1, cols):
        """m(x*) for the GPs gp0..gp1-1 (cols[k] = d x m block of GP gp0+k), MDCache order preserved."""
        sub = GPBatch.__new__(GPBatch)
        sub.gps, sub.B = self.gps[gp0:gp1], gp1 - gp0
        return GPBatch._means(sub, cols)

    # -- parity taps --------------------------------------------------------------------------
    def _tap(self, fn, b, shape):
        out = np.empty(shape, order="F")
        self.lib.check(getattr(self.lib.dll, fn)(self.handle, b, _d(out)))
        return out

    def K(self, b):
        return self._tap("gprb_get_K", b, (self.n, self.n))

    def chol_U(self, b):
        return self._tap("gprb_get_chol", b, (self.n, self.n))

    def alpha(self, b):
        return self._tap("gprb_get_alpha", b, (self.n,))

    def Kinv(self, b):
        return self._tap("gprb_get_Kinv", b, (self.n, self.n))

    # -- timing hooks -------------------------------------------------------------------------
    def set_profiling(self, on: bool):
        self.lib.check(self.lib.dll.gprb_set_profiling(self.handle, 1 if on else 0))

    def last_stage_ms(self):
        out = np.zeros(8)
        self.lib.check(self.lib.dll.gprb_last_stage_ms(self.handle, _d(out)))
        return dict(zip(["assembly", "cholesky", "solve", "inverse", "gradient", "total", "gemm", "gemm_launches"], out.tolist()))

    def last_gemm_launch_ms(self):
        """Per tile-GEMM launch device time (ms) of the last profiled evaluation, labelled by mode and step."""
        out = np.zeros(4 * (self.n // 128 + 2))
        k = self.lib.dll.gprb_last_gemm_launch_ms(self.handle, _d(out), out.size)
        J = (self.n + 127) // 128
        labels = []
        for j in range(J):
            if j > 0:  # block column 0 has no update terms: its diagonal block is factorised straight from K
                labels.append(("chol_diag", j))
            if j + 1 < J:
                labels.append(("chol_col", j))
        labels += [("trtri_row", i) for i in range(1, J)] + [("lauum", 0)]
        return [(m, st, float(t)) for (m, st), t in zip(labels[:k], out[:k])]


def optimize(gp, method: LBFGS | None = None, options: Options | None = None):
    """``GaussianProcesses.optimize!(gp, method, options)``.  ``gp`` may be one GPE (reference call pattern) or a
    sequence of GPEs / a GPBatch (batched lock-step optimisation, one library call)."""
    if isinstance(gp, GPBatch):
        return gp.optimize(method, options)
    if isinstance(gp, GPE):
        if gp._batch is None or gp._batch.B != 1:
            GPBatch([gp])
        return gp._batch.optimize(method, options)[0]
    gps = list(gp)
    b = gps[0]._batch
    if b is None or b.gps != gps:
        b = GPBatch(gps)
    return b.optimize(method, options)


optimize_b = optimize  # ``optimize!`` (the bang is not a Python identifier character)


def append(gp, x, y):
    """``append!(gp, x, y)`` (ElasticGPE): add the samples x (d x k) with targets y (k,) to one GPE and condition it on
    them at its current parameters.  A GP that shares its batch moves to a batch of its own first (like ``optimize``).
    For a GPBatch, x is the list of per-dataset blocks and y (B, k), see ``GPBatch.append``.  Returns ``gp``."""
    if isinstance(gp, GPBatch):
        gp.append(x, y)
        return gp
    if gp._batch is None or gp._batch.B != 1:
        GPBatch([gp]).update_mll()
    x = np.asarray(x, dtype=np.float64)
    gp._batch.append([x.reshape(gp.dim, -1)], np.asarray(y, dtype=np.float64).reshape(1, -1))
    return gp


def predict_y(gp, Xstar, var=True):
    """``predict_y(gp, Xstar) -> (mu, sigma2)`` for one GPE (d x m test block), or batched for a GPBatch."""
    if isinstance(gp, GPBatch):
        return gp.predict_y(Xstar, var=var)
    if gp._batch is None:
        GPBatch([gp]).update_mll()
    b = gp._batch
    if b.B == 1:
        mu, v = b.predict_y(Xstar, var=var)
        return mu[0], (v[0] if var else None)
    mu, v = b.predict_y(Xstar, var=var)
    return mu[gp._slot], (v[gp._slot] if var else None)


def _resident(gp):
    if gp._batch is None:
        GPBatch([gp]).update_mll()
    return gp._batch


def predict_f(gp, Xstar, full_cov=False):
    """``predict_f(gp, Xstar; full_cov) -> (mu, sigma2 | Sigma_f)`` for one GPE, or batched for a GPBatch."""
    if isinstance(gp, GPBatch):
        return gp.predict_f(Xstar, full_cov=full_cov)
    mu, v = _resident(gp).predict_f(Xstar, full_cov=full_cov)
    return mu[gp._slot], v[gp._slot]


def _only(gp):
    """(batch, active mask) for a call that evaluates one GPE alone in its batch's pass."""
    b = _resident(gp)
    act = np.zeros(b.B, dtype=np.uint8)
    act[gp._slot] = 1
    return b, act


def predict_grad(gp, Xstar, var=True):
    """``predict_grad(gp, Xstar) -> (mu (m,), var (m,) | None, dmu (m,d), dvar (m,d) | None)`` for one GPE (d x m test
    block): the posterior mean and variance with their Jacobians with respect to the test inputs; batched
    ((B,m), (B,m), (B,m,d), (B,m,d)) for a GPBatch.  See ``GPBatch.predict_grad``."""
    if isinstance(gp, GPBatch):
        return gp.predict_grad(Xstar, var=var)
    mu, v, dmu, dv = _resident(gp).predict_grad(Xstar, var=var)
    k = gp._slot
    return mu[k], (v[k] if var else None), dmu[k], (dv[k] if var else None)


def predict_LOO(gp):
    """``predict_LOO(gp) -> (mu, sigma2)``: leave-one-out predictive mean and variance at the n training inputs of one
    GPE ((n,), (n,)), or batched ((B,n), (B,n)) for a GPBatch."""
    if isinstance(gp, GPBatch):
        return gp.predict_LOO()
    b, act = _only(gp)
    mu, var = b.predict_LOO(active=act)
    return mu[gp._slot], var[gp._slot]


def logp_CVLOO(gp):
    """``logp_CVLOO(gp)``: leave-one-out log predictive probability of one GPE (float), or (B,) for a GPBatch
    (-Inf where the factorisation failed)."""
    if isinstance(gp, GPBatch):
        return gp.eval_loo(grad=False)[0]
    b, act = _only(gp)
    return float(b.eval_loo(grad=False, active=act)[0][gp._slot])


def dlogpdtheta_CVLOO(gp):
    """``dlogpdθ_CVLOO(gp)``: gradient of logp_CVLOO with respect to [logNoise; kernel params] (P,), or (B,P) for a
    GPBatch (NaN rows where the factorisation failed)."""
    if isinstance(gp, GPBatch):
        return gp.eval_loo(grad=True)[1]
    b, act = _only(gp)
    return b.eval_loo(grad=True, active=act)[1][gp._slot]


def rand(gp, Xstar, nsamples=1, Z=None, rng=None):
    """``rand(gp, Xstar, n)``: posterior draws (m, n) of one GPE (Z: (m, n) standard normals, or drawn from ``rng``);
    raises LinAlgError where make_posdef! gives up.  For a GPBatch: ``GPBatch.rand`` -> (draws (B, m, n), info)."""
    if isinstance(gp, GPBatch):
        return gp.rand(Xstar, nsamples, Z=Z, rng=rng)
    b = _resident(gp)
    m = np.asarray(Xstar).reshape(np.asarray(Xstar).shape[0], -1).shape[1]
    if Z is None:
        rng = np.random.default_rng() if rng is None else rng
        Z = rng.standard_normal((nsamples, m)).T
    Zb = np.zeros((b.B, m, nsamples))
    Zb[gp._slot] = Z
    draws, info = b.rand(Xstar, nsamples, Z=Zb)
    if info[gp._slot] < 0:
        raise np.linalg.LinAlgError(f"posterior covariance is not positive definite (info {int(info[gp._slot])})")
    return draws[gp._slot]
