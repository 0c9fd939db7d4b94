"""GPU tests of the round-2 C-ABI surface: per-GP failure masking at predict time, the asynchronous prediction
pipelines and the overlapped rollout, one-allocation dataset uploads, several contexts per process, the in-library
NCCL gather, and the per-GP virtual time limit of the batched optimiser."""
import ctypes as C
import os

import numpy as np
import pytest

from oracle import gp_oracle as go

pytestmark = pytest.mark.gpu


def rel(a, b):
    a, b = np.asarray(a, float), np.asarray(b, float)
    return float(np.max(np.abs(a - b)) / max(np.max(np.abs(b)), 1e-300))


def _cp_batch(gprb, ntrials, n, seed=0, n_test=0):
    from gpr_jl_b200 import data
    trials = [data.make_trial("CP", n, seed=seed + t, n_test=n_test) for t in range(ntrials)]
    th = data.theta0("CP", trials[0]["X"])
    th[1:-1] -= 1.0
    rng = np.random.default_rng(seed)
    thetas = [np.tile(th, (4, 1)) + 0.05 * rng.standard_normal((4, th.size)) for _ in trials]
    gps = []
    for tr, tt in zip(trials, thetas):
        for k in range(4):
            gps.append(gprb.GPE(tr["X"], tr["Y"][k], gprb.MeanZero(), gprb.SEArd(tt[k][1:-1], tt[k][-1]), logNoise=tt[k][0]))
    return gprb.GPBatch(gps), trials, np.concatenate(thetas)


def test_failed_gp_is_masked_at_predict_time(gprb):
    """One GP without a state (info = -2) gets NaN rows; every other GP of the batch is predicted normally - on the tiled
    path (value-only state, any m), the split GEMV path (m <= 8 with V resident) and the mean-only path
    (/root/reference/examples/parallel/core.jl:41-46 swallows a failed trial and carries on)."""
    batch, trials, theta = _cp_batch(gprb, 3, 200, seed=40, n_test=12)
    theta[5, 3] = np.nan
    good = [b for b in range(12) if b != 5]
    Xs = trials[0]["Xtest"]
    for with_grad, m in [(False, 12), (True, 5), (True, 1), (True, 12)]:
        mll, _, info = batch.eval(theta=theta, grad=with_grad)
        assert info[5] == -2 and mll[5] == -np.inf and np.all(info[good] == 0)
        mu, var = batch.predict_y(Xs[:, :m])
        mu_m, none = batch.predict_y(Xs[:, :m], var=False)
        assert none is None
        assert np.all(np.isnan(mu[5])) and np.all(np.isnan(var[5])) and np.all(np.isnan(mu_m[5]))
        for b in good:
            tr = trials[b // 4]
            X = np.ascontiguousarray(tr["X"].T)
            r = go.eval_mll(X, tr["Y"][b % 4], theta[b], with_grad=False, return_state=True)
            m_o, v_o = go.predict(X, theta[b], r["state"], np.ascontiguousarray(Xs[:, :m].T))
            assert rel(mu[b], m_o) <= 1e-9 and rel(mu_m[b], m_o) <= 1e-9, (with_grad, m, b)
            np.testing.assert_allclose(var[b], v_o, rtol=1e-9, atol=1e-13)
    batch.close()


def test_split_gemv_predict_is_batch_size_invariant(gprb):
    """The m <= 8 variance path cuts the rows of V into 16 fixed chunks shared by 1..16 CTAs depending on the batch size;
    the partials are always summed in chunk order, so one GP alone (16 CTAs) and the same GP among 40 (fewer CTAs per GP)
    give bit-identical results, at every column-chunk width (m = 1, 2, 3, 4, 7, 8)."""
    big, trials, theta = _cp_batch(gprb, 10, 300, seed=60, n_test=8)
    big.eval(theta=theta, grad=True)
    one = gprb.GPBatch([gprb.GPE(trials[2]["X"], trials[2]["Y"][1], gprb.MeanZero(),
                                 gprb.SEArd(theta[9][1:-1], theta[9][-1]), logNoise=theta[9][0])])
    one.eval(grad=True)
    X = np.ascontiguousarray(trials[2]["X"].T)
    r = go.eval_mll(X, trials[2]["Y"][1], theta[9], with_grad=False, return_state=True)
    for m in (1, 2, 3, 4, 7, 8):
        Xs = trials[0]["Xtest"][:, :m]
        mu_b, var_b = big.predict_y(Xs)
        mu_1, var_1 = one.predict_y(Xs)
        assert np.array_equal(mu_b[9], mu_1[0]) and np.array_equal(var_b[9], var_1[0]), m
        m_o, v_o = go.predict(X, theta[9], r["state"], np.ascontiguousarray(Xs.T))
        assert rel(mu_1[0], m_o) <= 1e-9
        np.testing.assert_allclose(var_1[0], v_o, rtol=1e-9, atol=1e-13)
    big.close()
    one.close()


def test_async_predict_slots_equal_sync(gprb):
    """gprb_predict_async / gprb_predict_wait on GP sub-ranges, both pipelines in flight at once, shared per-trial test
    blocks (gps_per_block = G) - identical to one synchronous gprb_predict with per-GP blocks."""
    batch, trials, theta = _cp_batch(gprb, 6, 200, seed=70, n_test=9)
    batch.eval(theta=theta, grad=False)
    blocks = [tr["Xtest"] for tr in trials]
    per_gp = [blocks[b // 4] for b in range(24)]
    mu_s, var_s = batch.predict_y(per_gp, per_gp=True)
    batch.predict_async(0, 0, 12, blocks[:3], var=True, gps_per_block=4)
    batch.predict_async(1, 12, 24, blocks[3:], var=True, gps_per_block=4)
    mu1, var1 = batch.predict_wait(1)
    mu0, var0 = batch.predict_wait(0)
    assert np.array_equal(np.concatenate([mu0, mu1]), mu_s) and np.array_equal(np.concatenate([var0, var1]), var_s)
    assert batch.last_predict_ms(0) > 0 and batch.last_predict_ms(1) > 0
    # mean only (what the rollout asks for: predictdynamics.jl:13 discards the variance), odd split
    batch.predict_async(0, 0, 8, blocks[:2], var=False, gps_per_block=4)
    batch.predict_async(1, 8, 24, blocks[2:], var=False, gps_per_block=4)
    m0, v0 = batch.predict_wait(0)
    m1, v1 = batch.predict_wait(1)
    assert v0 is None and v1 is None
    np.testing.assert_allclose(np.concatenate([m0, m1]), mu_s, rtol=1e-13, atol=1e-15)
    # misuse: a slot cannot take a second prediction before the first is collected
    batch.predict_async(0, 0, 4, blocks[:1], var=False, gps_per_block=4)
    with pytest.raises(gprb.GprbError):
        batch.predict_async(0, 0, 4, blocks[:1], var=False, gps_per_block=4)
    batch.predict_wait(0)
    batch.close()


def test_overlapped_rollout_equals_serial(gprb):
    """experiment.predictdynamics with the two alternating trial groups (device predict of one group under the host
    projection of the other) gives bit-identical rollouts to the serial per-step loop."""
    from gpr_jl_b200 import experiment
    batch, trials, theta = _cp_batch(gprb, 5, 160, seed=80, n_test=6)
    batch.eval(theta=theta, grad=False)
    idx = np.array([9, 22, 23, 24]) - 1  # CPnoise.jl:28

    def step_fn(t, states, mu):  # stand-in for getvomega + projectv! + updatestate!
        nxt = states.copy()
        nxt[idx, :] = mu
        nxt[1, :] += 0.01 * nxt[8, :]
        return nxt
    starts = [tr["Xtest"] for tr in trials]
    tm = {}
    a = experiment.predictdynamics(batch, 4, starts, 4, step_fn, overlap=True, timing=tm)
    b = experiment.predictdynamics(batch, 4, starts, 4, step_fn, overlap=False)
    assert all(np.array_equal(x, y) for x, y in zip(a, b))
    assert tm["total_s"] > 0 and tm["host_s"] > 0
    batch.close()


def test_dataset_slab_updates(gprb):
    """All trial datasets of a batch share one allocation (gprb_datasets_create).  A contiguous host block re-uploads in
    one copy + one transpose launch, scattered host matrices take the per-dataset path; both must give the evaluation
    of a freshly built batch."""
    batch, trials, theta = _cp_batch(gprb, 4, 150, seed=90)
    mll0, _, _ = batch.eval(theta=theta, grad=False)
    Xn = [np.asfortranarray(tr["X"] * (1.0 + 1e-3 * (t + 1))) for t, tr in enumerate(trials)]
    fresh = gprb.GPBatch([gprb.GPE(Xn[b // 4], trials[b // 4]["Y"][b % 4], gprb.MeanZero(),
                                   gprb.SEArd(theta[b][1:-1], theta[b][-1]), logNoise=theta[b][0]) for b in range(16)])
    want, _, _ = fresh.eval(grad=False)
    ctx = gprb.gp.context()
    l0 = ctx.launch_count()
    batch.update_data(trials_X=Xn)                      # scattered host arrays: per-dataset copies
    l1 = ctx.launch_count()
    got, _, _ = batch.eval(theta=theta, grad=False)
    assert np.array_equal(got, want) and not np.array_equal(got, mll0)
    block = np.empty((4, 150, 26))
    for t in range(4):
        block[t] = trials[t]["X"].T
    l2 = ctx.launch_count()
    batch.update_data(trials_X=[block[t].T for t in range(4)])   # one contiguous (T, n, d) block: one copy, one launch
    l3 = ctx.launch_count()
    back, _, _ = batch.eval(theta=theta, grad=False)
    assert np.array_equal(back, mll0)
    assert l1 - l0 == 4 and l3 - l2 == 1
    batch.close()
    fresh.close()


def test_two_contexts_in_one_process(gprb):
    """A second gprb_ctx in the same process (VERDICT r01 #11: process-wide `configured` flags broke it on a second
    device) - on the same device here, and on a second device when the box has one."""
    import torch
    from gpr_jl_b200 import data
    lib = gprb.load_library()
    tr = data.make_trial("P1", 130, seed=3)
    th = data.theta0("P1", tr["X"])
    th[1:-1] -= 1.0
    ref = go.eval_mll(np.ascontiguousarray(tr["X"].T), tr["Y"][0], th)
    devs = [0] + ([1] if torch.cuda.device_count() > 1 else [])
    for dev in devs:
        h = C.c_void_p()
        lib.check(lib.dll.gprb_init(C.byref(h), dev))
        Xc = np.ascontiguousarray(tr["X"].T)
        ds = C.c_void_p()
        lib.check(lib.dll.gprb_dataset_create(h, 130, 13, Xc.ctypes.data_as(C.POINTER(C.c_double)), 13, C.byref(ds)))
        dsa = (C.c_void_p * 1)(ds.value)
        y = np.ascontiguousarray(tr["Y"][0])
        bh = C.c_void_p()
        lib.check(lib.dll.gprb_batch_create(h, 1, dsa, y.ctypes.data_as(C.POINTER(C.c_double)), 0, C.byref(bh)))
        mll, grad, info = np.zeros(1), np.zeros(15), np.zeros(1, dtype=np.int32)
        lib.check(lib.dll.gprb_eval(bh, th.ctypes.data_as(C.POINTER(C.c_double)), None, mll.ctypes.data_as(C.POINTER(C.c_double)),
                                    grad.ctypes.data_as(C.POINTER(C.c_double)), info.ctypes.data_as(C.POINTER(C.c_int32))))
        assert info[0] == 0 and abs(mll[0] - ref["mll"]) <= 1e-8 * abs(ref["mll"]) and rel(grad, ref["grad"]) <= 1e-8
        lib.dll.gprb_batch_destroy(bh)
        lib.dll.gprb_dataset_destroy(ds)
        lib.dll.gprb_destroy(h)
    if len(devs) > 1:
        torch.cuda.set_device(0)


def test_gather_single_rank_scatter(gprb):
    """gprb_gather without a communicator degenerates to the local scatter by row id (NaN where nobody contributed)."""
    ctx = gprb.gp.context()
    local = {3: np.arange(5.0), 0: np.arange(5.0) + 10, 6: np.arange(5.0) + 20}
    out = ctx.gather(local, 7, 5)
    assert out.shape == (7, 5)
    for t, row in local.items():
        assert np.array_equal(out[t], row)
    assert np.all(np.isnan(out[[1, 2, 4, 5]]))


def test_gather_multi_two_gpus(gprb):
    """gprb_init_multi + gprb_gather_multi: one process, two B200s, one NCCL all-gather inside the library; two batches
    (one per device) evaluate trials round-robin and the gathered table equals the single-GPU results bit for bit."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    from gpr_jl_b200 import data
    lib = gprb.load_library()
    hs = (C.c_void_p * 2)()
    lib.check(lib.dll.gprb_init_multi(hs, 2, None))
    dp = C.POINTER(C.c_double)
    trials = [data.make_trial("P1", 140, seed=200 + t) for t in range(5)]
    th = data.theta0("P1", trials[0]["X"])
    th[1:-1] -= 1.0
    single, _, _ = gprb.GPBatch([gprb.GPE(tr["X"], tr["Y"][0], gprb.MeanZero(), gprb.SEArd(th[1:-1], th[-1]), logNoise=th[0])
                                 for tr in trials]).eval(grad=True)
    rows, ids = [], []
    for g in range(2):
        mine = list(range(g, 5, 2))
        res = np.zeros((len(mine), 2))
        for k, t in enumerate(mine):
            Xc = np.ascontiguousarray(trials[t]["X"].T)
            ds = C.c_void_p()
            lib.check(lib.dll.gprb_dataset_create(hs[g], 140, 13, Xc.ctypes.data_as(dp), 13, C.byref(ds)))
            dsa = (C.c_void_p * 1)(ds.value)
            y = np.ascontiguousarray(trials[t]["Y"][0])
            bh = C.c_void_p()
            lib.check(lib.dll.gprb_batch_create(hs[g], 1, dsa, y.ctypes.data_as(dp), 0, C.byref(bh)))
            mll, grad, info = np.zeros(1), np.zeros(15), np.zeros(1, dtype=np.int32)
            lib.check(lib.dll.gprb_eval(bh, th.ctypes.data_as(dp), None, mll.ctypes.data_as(dp), grad.ctypes.data_as(dp),
                                        info.ctypes.data_as(C.POINTER(C.c_int32))))
            res[k] = [mll[0], float(info[0])]
            lib.dll.gprb_batch_destroy(bh)
            lib.dll.gprb_dataset_destroy(ds)
        rows.append(np.ascontiguousarray(res))
        ids.append(np.ascontiguousarray(mine, dtype=np.int32))
    ip = C.POINTER(C.c_int32)
    counts = (C.c_int32 * 2)(len(ids[0]), len(ids[1]))
    idp = (ip * 2)(ids[0].ctypes.data_as(ip), ids[1].ctypes.data_as(ip))
    rp = (dp * 2)(rows[0].ctypes.data_as(dp), rows[1].ctypes.data_as(dp))
    out = np.zeros((5, 2))
    lib.check(lib.dll.gprb_gather_multi(hs, 2, 5, 2, counts, idp, rp, out.ctypes.data_as(dp)))
    assert np.array_equal(out[:, 0], single) and np.all(out[:, 1] == 0)
    for g in range(2):
        lib.dll.gprb_destroy(hs[g])
    torch.cuda.set_device(0)


def test_optimize_per_gp_virtual_time_limit(gprb):
    """Optim.Options(time_limit=10.) is 10 s of CPU time PER GP on the reference (CPnoise.jl:41).  With evaluation costs
    set, every GP runs on its own deterministic virtual clock: GPs whose line searches need more trials stop after fewer
    iterations, exactly like the scalar restatement with the same costs."""
    from gpr_jl_b200 import data
    from oracle.lbfgs_oracle import LBFGSOptions, lbfgs
    tr = data.make_trial("P1", 96, seed=17)
    tr = {"X": tr["X"], "Y": tr["Y"] + 0.05 * np.random.default_rng(96).standard_normal(tr["Y"].shape)}  # well-conditioned optimum, see test_optimize_matches_scalar_oracle
    th = data.theta0("P1", tr["X"])
    gps = [gprb.GPE(tr["X"], tr["Y"][k], gprb.MeanZero(), gprb.SEArd(th[1:-1], th[-1]), logNoise=th[0]) for k in range(3)]
    batch = gprb.GPBatch(gps)
    opt = gprb.Options(time_limit=10.0, cost_value=0.4, cost_grad=1.1)
    res = batch.optimize(gprb.LBFGS(linesearch=gprb.BackTracking(order=2)), opt)
    X = np.ascontiguousarray(tr["X"].T)
    for k in range(3):
        y = tr["Y"][k]
        f = lambda t: -go.eval_mll(X, y, t, with_grad=False)["mll"]

        def fg(t):
            r = go.eval_mll(X, y, t)
            return (-r["mll"], -r["grad"]) if r["info"] >= 0 else (np.inf, np.full(t.size, np.nan))
        o = lbfgs(f, fg, th, LBFGSOptions(time_limit=10.0, cost_value=0.4, cost_grad=1.1))
        assert o.stopped_by == "time_limit"
        assert (res[k]["iterations"], res[k]["f_calls"], res[k]["g_calls"]) == (o.iterations, o.f_calls, o.fg_calls)
        assert res[k]["f_calls"] * 0.4 + res[k]["g_calls"] * 1.1 > 10.0          # stopped at the first iteration past 10 s
        assert abs(res[k]["minimum"] - o.f) <= 1e-6 * abs(o.f)
    batch.close()


@pytest.mark.parametrize("system,n", [("CP", 300), ("P2", 1000), ("CP", 2000)])
def test_cluster_substitution_is_bit_identical(gprb, system, n, monkeypatch):
    """k_solve_cluster (one thread-block cluster of up to 8 CTAs per GP, used when a pass has fewer GPs than SMs) adds its
    terms in exactly the order of the one-CTA k_solve: alpha, mll and everything downstream are bit-identical, so a GP's
    results still do not depend on the batch it is evaluated in.  J = 3 (ragged last block), 8 and 16 block rows."""
    from gpr_jl_b200 import data
    tr = data.make_trial(system, n, seed=7 + n, n_test=5)
    th = data.theta0(system, tr["X"])
    th[1:-1] -= 0.5
    G = min(3, tr["Y"].shape[0])
    thetas = np.tile(th, (G, 1)) + 0.05 * np.random.default_rng(n).standard_normal((G, th.size))

    def run(below):
        monkeypatch.setenv("GPRB200_SOLVE_CLUSTER_BELOW", below)  # read when the batch is created
        gps = [gprb.GPE(tr["X"], tr["Y"][k], gprb.MeanZero(), gprb.SEArd(thetas[k][1:-1], thetas[k][-1]), logNoise=thetas[k][0])
               for k in range(G)]
        b = gprb.GPBatch(gps)
        mll, grad, info = b.eval(grad=True)
        al = np.stack([b.alpha(k) for k in range(G)])
        mu, var = b.predict_y(tr["Xtest"])
        b.close()
        return mll, grad, info, al, mu, var
    one = run("0")
    clu = run("100000")
    for a, c in zip(one, clu):
        assert np.array_equal(a, c)
    X = np.ascontiguousarray(tr["X"].T)
    r = go.eval_mll(X, tr["Y"][0], thetas[0], with_grad=True, return_state=True)
    assert abs(clu[0][0] - r["mll"]) <= 1e-8 * abs(r["mll"]) and rel(clu[3][0], r["state"]["alpha"]) <= 1e-8
