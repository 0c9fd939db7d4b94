"""CPU: the leave-one-out oracle (oracle/loo_oracle.py) against brute-force refits on n - 1 points, its textbook gradient
against central differences, and the rewrite the device uses (alpha = 0, -Q' in the K^-1 slot, pushed through the
evaluation gradient's 1/2 tr(Q dK_j) contraction) against the textbook form."""
import numpy as np
import pytest

from oracle import gp_oracle as go
from oracle import loo_oracle as lo

KINDS = ["se", "mat12", "mat32", "mat52"]


def _problem(n, kind, seed, d=3):
    rng = np.random.default_rng(seed)
    X = rng.standard_normal((n, d))
    y = np.sin(X[:, 0]) + 0.5 * X[:, 1] + 0.1 * rng.standard_normal(n)
    th = np.concatenate([[-1.5], np.log(np.full(d, 1.2)), [0.2]]) + 0.1 * rng.standard_normal(d + 2)
    return X, y, th


def _jitter_offset(X, th, kind, k):
    """Diagonal offset that makes make_posdef! add exactly k jitters (the construction of the evaluation ladder test)."""
    K = go.assemble_K(X, th, kind)
    n = K.shape[0]
    lam = float(np.linalg.eigvalsh(K)[0])
    T = float(np.trace(K)) / n
    delta = 1e-6 * (T - lam) / (1.0 + 1e-6 * (k - 0.5))
    return -(lam + (k - 0.5) * delta)


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("n", [12, 40, 60])
@pytest.mark.parametrize("case", ["plain", "offset", "jitter"])
def test_oracle_matches_brute_force(kind, n, case):
    X, y, th = _problem(n, kind, seed=n + len(kind))
    off = {"plain": 0.0, "offset": 0.05, "jitter": None}[case]
    if off is None:
        th = th.copy()
        th[0] = -4.0  # small noise: the offset that needs one jitter leaves cond(K) moderate
        off = _jitter_offset(X, th, kind, 1)
    r = lo.loo(X, y, th, kind, diag_offset=off, with_grad=False)
    assert r["info"] == (1 if case == "jitter" else 0)
    lp, mu, var = lo.brute_force_loo(r["K"], y)
    cond = go.cond_estimate(r["K"])
    tol = max(1e-12, 10 * cond * go.EPS)
    assert abs(r["logp"] - lp) <= tol * abs(lp), (r["logp"], lp, cond)
    assert np.max(np.abs(r["mu"] - mu)) <= tol * np.max(np.abs(mu))
    assert np.max(np.abs(r["var"] - var)) <= tol * np.max(np.abs(var))


@pytest.mark.parametrize("kind", KINDS)
def test_textbook_gradient_matches_central_differences(kind):
    X, y, th = _problem(30, kind, seed=3)
    r = lo.loo(X, y, th, kind)
    assert r["info"] == 0
    h = 1e-6
    fd = np.empty(th.size)
    for j in range(th.size):
        e = np.zeros(th.size)
        e[j] = h
        fd[j] = (lo.loo(X, y, th + e, kind, with_grad=False)["logp"] - lo.loo(X, y, th - e, kind, with_grad=False)["logp"]) / (2 * h)
    assert np.max(np.abs(r["grad"] - fd)) <= 1e-6 * np.max(np.abs(fd)), (r["grad"], fd)


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("off", [0.0, 0.05])
def test_rewrite_matches_textbook(kind, off):
    X, y, th = _problem(40, kind, seed=11)
    f = lo.factorise(X, y, th, kind, diag_offset=off)
    dKs = lo.dK(X, th, kind)
    g_text = lo.textbook_grad(f["Kinv"], f["alpha"], dKs)
    slot = lo.rewrite_slot(f["Kinv"], f["alpha"])
    g_rew = lo.contract(np.zeros_like(f["alpha"]), slot, dKs)
    assert np.max(np.abs(g_rew - g_text)) <= 1e-12 * np.max(np.abs(g_text)), (g_rew, g_text)
    # and the contraction with the evaluation's own Q gives the evaluation gradient (the same kernel, other inputs)
    r = go.eval_mll(X, y, th, kind=kind, diag_offset=off)
    g_mll = lo.contract(f["alpha"], f["Kinv"], dKs)
    assert np.max(np.abs(g_mll - r["grad"])) <= 1e-10 * np.max(np.abs(r["grad"]))


def test_failed_factorisation_is_minus_inf():
    X, y, th = _problem(20, "se", seed=5)
    r = lo.loo(X, y, th, "se", diag_offset=-100.0)
    assert r["info"] == -1 and r["logp"] == -np.inf and np.all(np.isnan(r["grad"])) and np.all(np.isnan(r["mu"]))
