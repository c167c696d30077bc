"""CPU: the closed-form gradients of logpdf (tests/grad_oracle.py) equal torch float64 autograd through the reference's literal
op sequence (src/bayesian_linear_regression.jl:72-89 and :55-58: `Uw' \\ X`, `Σy.U' \\ ...`, `chol(Bt'Bt + I)`, the logdet and
the quadratic form) to 1e-12, and agree with central finite differences of oracle.blr_oracle.logpdf."""
import math

import numpy as np
import pytest
import torch

from oracle import blr_oracle as ref
from tests import grad_oracle as go

LOG2PI = math.log(2.0 * math.pi)


def literal_logpdf(X, y, mw, Λ, σ2):
    """The reference's logpdf in torch (X: D x N; Λ: D x D; σ2: N), differentiable in every argument."""
    D, N = X.shape
    Uw = torch.linalg.cholesky(Λ).mT                                                    # :78
    sd = torch.sqrt(σ2)                                                                 # :79  Uy = Diagonal(sqrt(σ²))
    Bt = torch.linalg.solve_triangular(Uw.mT, X, upper=False).T / sd[:, None]           # :81  Uy' \ (Uw' \ X)'
    δy = (y - X.T @ mw) / sd                                                            # :82
    lp_δy = -(N * LOG2PI + 2.0 * torch.sum(torch.log(sd)) + δy @ δy) / 2                # :84
    U = torch.linalg.cholesky(Bt.T @ Bt + torch.eye(D, dtype=X.dtype)).mT               # :86
    v = torch.linalg.solve_triangular(U.mT, (Bt.T @ δy)[:, None], upper=False)[:, 0]
    return -(2.0 * torch.sum(torch.log(torch.diagonal(U))) - v @ v) / 2 + lp_δy         # :57


def problem(D, N, seed, prior, noise, zero_mean, layout):
    rng = np.random.default_rng(seed)
    X = rng.standard_normal((D, N))
    y = X.T @ rng.standard_normal(D) + 0.5 * rng.standard_normal(N)
    mw = np.zeros(D) if zero_mean else rng.standard_normal(D)
    B = rng.standard_normal((D, D)) / math.sqrt(D)
    Λd = B @ B.T + np.eye(D)
    lam = np.exp(rng.standard_normal(D))
    Λw = {"diag": ref.Diagonal(lam), "dense": Λd, "pdmat": ref.PDMat.from_matrix(Λd)}[prior]
    σ2 = 0.7 if noise == "scalar" else np.exp(0.5 * rng.standard_normal(N))
    x = ref.ColVecs(X) if layout == "col" else ref.RowVecs(np.ascontiguousarray(X.T))
    return ref.BayesianLinearRegressor(mw, Λw)(x, σ2), y


def autograd(fx, y):
    X = ref.x_as_colvecs(fx.x)
    N = X.shape[1]
    t = lambda a: torch.tensor(np.asarray(a, dtype=np.float64), requires_grad=True)
    Xt, yt, mwt = t(X), t(y), t(fx.f.mw)
    diag = isinstance(fx.f.Λw, ref.Diagonal)
    if diag:
        lt = t(fx.f.Λw.diag)
        Λt = torch.diag(lt)
    else:
        lt = t(ref.dense(fx.f.Λw))
        Λt = (lt + lt.T) / 2  # dℓ = <G, dΛ> over symmetric dΛ: the gradient in B of ℓ((B + B')/2) at B = Λ is G
    scalar = np.ndim(fx.Σy) == 0
    st = t(fx.Σy)
    σ2t = st * torch.ones(N, dtype=torch.float64) if scalar else st
    lp = literal_logpdf(Xt, yt, mwt, Λt, σ2t)
    lp.backward()
    gX = Xt.grad.numpy()
    return float(lp.detach()), {
        "X": gX.T if isinstance(fx.x, ref.RowVecs) else gX, "y": yt.grad.numpy(),
        "σ²": float(st.grad) if scalar else st.grad.numpy(), "mw": mwt.grad.numpy(), "Λw": lt.grad.numpy(),
    }


def rel_inf(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return float(np.max(np.abs(a - b)) / np.max(np.abs(b)))


CASES = [(prior, noise, zero_mean, layout) for prior in ("diag", "dense", "pdmat") for noise in ("scalar", "vector")
         for zero_mean in (True, False) for layout in ("col", "row")]


@pytest.mark.parametrize("prior,noise,zero_mean,layout", CASES)
def test_closed_forms_equal_autograd_through_the_reference_sequence(prior, noise, zero_mean, layout):
    fx, y = problem(7, 40, 11, prior, noise, zero_mean, layout)
    lp, want = autograd(fx, y)
    assert abs(lp - ref.logpdf(fx, y)) <= 1e-12 * abs(lp)
    got = go.logpdf_grad(fx, y)
    for k in want:
        assert np.shape(got[k]) == np.shape(want[k]), k
        assert rel_inf(got[k], want[k]) <= 1e-12, (k, rel_inf(got[k], want[k]))


def test_doctest_sized_toy():
    """D = 2, N = 10 (the size of the reference's basis_function_regression.jl doctest)."""
    fx, y = problem(2, 10, 3, "dense", "vector", False, "col")
    _, want = autograd(fx, y)
    got = go.logpdf_grad(fx, y)
    for k in want:
        assert rel_inf(got[k], want[k]) <= 1e-12, k


@pytest.mark.parametrize("prior,noise,layout", [("diag", "vector", "col"), ("dense", "scalar", "row"), ("pdmat", "vector", "row")])
def test_closed_forms_agree_with_central_differences(prior, noise, layout):
    fx, y = problem(5, 30, 7, prior, noise, False, layout)
    g = go.logpdf_grad(fx, y)
    h = 1e-6

    def fd(make):
        return (ref.logpdf(*make(+h)) - ref.logpdf(*make(-h))) / (2 * h)

    def check(approx, exact):
        assert abs(approx - exact) <= 1e-6 * max(1.0, abs(exact)), (approx, exact)

    X = fx.x.X
    for (i, j) in [(0, 0), (2, 3), (4, 1)]:
        def mk(d, i=i, j=j):
            Xp = X.copy()
            Xp[i, j] += d
            return fx.f(type(fx.x)(Xp), fx.Σy), y
        check(fd(mk), g["X"][i, j])
    for n in (0, 17):
        def mk(d, n=n):
            yp = y.copy()
            yp[n] += d
            return fx, yp
        check(fd(mk), g["y"][n])
    if noise == "scalar":
        check(fd(lambda d: (fx.f(fx.x, fx.Σy + d), y)), g["σ²"])
    else:
        for n in (1, 29):
            def mk(d, n=n):
                s = np.array(fx.Σy, copy=True)
                s[n] += d
                return fx.f(fx.x, s), y
            check(fd(mk), g["σ²"][n])
    for i in (0, 3):
        def mk(d, i=i):
            mw = fx.f.mw.copy()
            mw[i] += d
            return ref.BayesianLinearRegressor(mw, fx.f.Λw)(fx.x, fx.Σy), y
        check(fd(mk), g["mw"][i])
    for (i, j) in [(1, 1), (0, 3)]:
        def mk(d, i=i, j=j):
            if isinstance(fx.f.Λw, ref.Diagonal):
                lam = fx.f.Λw.diag.copy()
                lam[i] += d
                Λ = ref.Diagonal(lam)
            else:
                A = ref.dense(fx.f.Λw).copy()
                A[i, j] += d / (1 if i == j else 2)  # a symmetric perturbation E with <G, E> = G_ij
                A[j, i] += 0 if i == j else d / 2
                Λ = A
            return ref.BayesianLinearRegressor(fx.f.mw, Λ)(fx.x, fx.Σy), y
        if isinstance(fx.f.Λw, ref.Diagonal):
            if i == j:
                check(fd(mk), g["Λw"][i])
        else:
            check(fd(mk), g["Λw"][i, j])
