"""CPU: the feature-map VJP of tests/grad_oracle_features.py equals torch float64 autograd of scale * act(W x + b) to 1e-12 for
every activation, and composed with the closed-form ∂ℓ/∂ϕ(x) of tests/grad_oracle.py it equals torch autograd through the
reference's literal logpdf (test_oracle_grad.literal_logpdf) over the torch map to 1e-12, and central differences of
oracle.blr_oracle.logpdf in W, b and x."""
import math

import numpy as np
import pytest
import torch

from oracle import blr_oracle as ref
from tests import grad_oracle as go
from tests import grad_oracle_features as gof
from tests.test_oracle_grad import literal_logpdf


def rel_inf(a, b):
    """max |a - b| / max |b|; 0 when both are exactly zero (relu with every z <= 0)"""
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return float(np.max(np.abs(a - b)) / max(np.max(np.abs(b)), np.finfo(np.float64).tiny))


TORCH_ACTS = {"cos": torch.cos, "tanh": torch.tanh, "relu": torch.relu, "identity": lambda t: t, "sin": torch.sin}


def feature_problem(din, D, N, seed, act):
    rng = np.random.default_rng(seed)
    x = rng.standard_normal((din, N))
    W = rng.standard_normal((D, din)) / math.sqrt(din)
    b = rng.uniform(0.0, 2.0 * math.pi, D)
    scale = math.sqrt(2.0 / D) if act == "cos" else 0.7
    return x, W, b, scale


def torch_map(xt, Wt, bt, act, scale):
    return scale * TORCH_ACTS[act](Wt @ xt + bt[:, None])


@pytest.mark.parametrize("act", gof.ACTS)
@pytest.mark.parametrize("din,D,N", [(1, 1, 1), (3, 7, 17), (32, 65, 40)])
def test_vjp_matches_autograd(act, din, D, N):
    x, W, b, scale = feature_problem(din, D, N, din + D + N, act)
    dphi = np.random.default_rng(1).standard_normal((D, N))
    t = lambda a: torch.tensor(a, dtype=torch.float64, requires_grad=True)
    xt, Wt, bt = t(x), t(W), t(b)
    torch_map(xt, Wt, bt, act, scale).backward(torch.tensor(dphi))
    got = gof.features_vjp(x, W, b, act, scale, dphi)
    assert np.allclose(gof.features(x, W, b, act, scale), torch_map(*(torch.tensor(a) for a in (x, W, b)), act, scale).numpy(),
                       rtol=1e-14, atol=1e-14)
    for key, want in (("W", Wt.grad), ("b", bt.grad), ("xin", xt.grad)):
        assert rel_inf(got[key], want.numpy()) <= 1e-12, (act, key)


def test_relu_derivative_is_zero_at_zero():
    x, W, b, scale = feature_problem(3, 6, 9, 0, "relu")
    b[:] = 0.0
    x[:, ::2] = 0.0
    dphi = np.random.default_rng(2).standard_normal((6, 9))
    t = lambda a: torch.tensor(a, dtype=torch.float64, requires_grad=True)
    xt, Wt, bt = t(x), t(W), t(b)
    torch_map(xt, Wt, bt, "relu", scale).backward(torch.tensor(dphi))
    got = gof.features_vjp(x, W, b, "relu", scale, dphi)
    for key, want in (("W", Wt.grad), ("b", bt.grad), ("xin", xt.grad)):
        assert np.array_equal(got[key] == 0.0, want.numpy() == 0.0) and rel_inf(got[key], want.numpy()) <= 1e-12, key
    assert np.all(got["xin"][:, ::2] == 0.0)


def chain_problem(act, din=4, D=12, N=30, seed=3):
    x, W, b, scale = feature_problem(din, D, N, seed, act)
    rng = np.random.default_rng(seed + 1)
    Phi = gof.features(x, W, b, act, scale)
    y = Phi.T @ rng.standard_normal(D) + 0.3 * rng.standard_normal(N)
    mw = rng.standard_normal(D)
    lam = np.exp(rng.standard_normal(D))
    σ2 = 0.5 + np.exp(0.5 * rng.standard_normal(N))
    return x, W, b, scale, y, mw, lam, σ2


def chain_oracle(x, W, b, act, scale, y, mw, lam, σ2):
    Phi = gof.features(x, W, b, act, scale)
    fx = ref.BayesianLinearRegressor(mw, ref.Diagonal(lam))(ref.ColVecs(Phi), σ2)
    dPhi = go.logpdf_grad(fx, y)["X"]
    return ref.logpdf(fx, y), gof.features_vjp(x, W, b, act, scale, dPhi)


@pytest.mark.parametrize("act", gof.ACTS)
def test_chain_matches_autograd_through_literal_logpdf(act):
    x, W, b, scale, y, mw, lam, σ2 = chain_problem(act)
    t = lambda a: torch.tensor(a, dtype=torch.float64, requires_grad=True)
    xt, Wt, bt = t(x), t(W), t(b)
    c = lambda a: torch.tensor(a, dtype=torch.float64)
    lp = literal_logpdf(torch_map(xt, Wt, bt, act, scale), c(y), c(mw), torch.diag(c(lam)), c(σ2))
    lp.backward()
    lpo, got = chain_oracle(x, W, b, act, scale, y, mw, lam, σ2)
    assert abs(float(lp) - lpo) <= 1e-12 * abs(lpo)
    for key, want in (("W", Wt.grad), ("b", bt.grad), ("xin", xt.grad)):
        assert rel_inf(got[key], want.numpy()) <= 1e-12, (act, key)


@pytest.mark.parametrize("act", ["cos", "tanh", "sin", "identity"])
def test_chain_matches_central_differences(act):
    x, W, b, scale, y, mw, lam, σ2 = chain_problem(act)
    _, got = chain_oracle(x, W, b, act, scale, y, mw, lam, σ2)

    def lp(x_, W_, b_):
        Phi = gof.features(x_, W_, b_, act, scale)
        return ref.logpdf(ref.BayesianLinearRegressor(mw, ref.Diagonal(lam))(ref.ColVecs(Phi), σ2), y)

    h = 1e-6
    for key, arr, idx in (("W", W, (2, 1)), ("W", W, (7, 3)), ("b", b, (5,)), ("xin", x, (1, 11)), ("xin", x, (3, 0))):
        up, dn = arr.copy(), arr.copy()
        up[idx] += h
        dn[idx] -= h
        args_up = {"xin": (up, W, b), "W": (x, up, b), "b": (x, W, up)}[key]
        args_dn = {"xin": (dn, W, b), "W": (x, dn, b), "b": (x, W, dn)}[key]
        fd = (lp(*args_up) - lp(*args_dn)) / (2 * h)
        assert abs(fd - got[key][idx]) <= 1e-6 * max(1.0, abs(fd)), (act, key, idx, fd, got[key][idx])
