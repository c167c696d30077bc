"""CPU: the closed-form gradients of L = Σ_j c_j logpdf(fx, Y[:, j]) (tests/grad_oracle_multi.py) equal torch float64
autograd of the same weighted sum through the reference's literal op sequence (src/bayesian_linear_regression.jl:72-89 and
:55-58) to 1e-12, agree with central finite differences of oracle.blr_oracle.logpdf, and reduce to logpdf_grad for k = 1."""
import numpy as np
import pytest
import torch

from oracle import blr_oracle as ref
from tests import grad_oracle as go
from tests import grad_oracle_multi as gom
from tests.test_oracle_grad import literal_logpdf, problem, rel_inf


def targets(fx, k, seed):
    X = ref.x_as_colvecs(fx.x)
    D, N = X.shape
    rng = np.random.default_rng(seed)
    return X.T @ rng.standard_normal((D, k)) + 0.5 * rng.standard_normal((N, k))


def autograd(fx, Y, c):
    X = ref.x_as_colvecs(fx.x)
    N = X.shape[1]
    t = lambda a: torch.tensor(np.asarray(a, dtype=np.float64), requires_grad=True)
    Xt, Yt, mwt = t(X), t(Y), t(fx.f.mw)
    if isinstance(fx.f.Λw, ref.Diagonal):
        lt = t(fx.f.Λw.diag)
        Λt = torch.diag(lt)
    else:
        lt = t(ref.dense(fx.f.Λw))
        Λt = (lt + lt.T) / 2  # the gradient in B of L((B + B')/2) at B = Λ is the symmetric G with dL = <G, dΛ>
    scalar = np.ndim(fx.Σy) == 0
    st = t(fx.Σy)
    σ2t = st * torch.ones(N, dtype=torch.float64) if scalar else st
    lps = torch.stack([literal_logpdf(Xt, Yt[:, j], mwt, Λt, σ2t) for j in range(Y.shape[1])])
    (torch.tensor(c) @ lps).backward()
    gX = Xt.grad.numpy()
    return lps.detach().numpy(), {
        "X": gX.T if isinstance(fx.x, ref.RowVecs) else gX, "y": Yt.grad.numpy(),
        "σ²": float(st.grad) if scalar else st.grad.numpy(), "mw": mwt.grad.numpy(), "Λw": lt.grad.numpy(),
    }


WEIGHTS = {
    1: [np.array([1.0]), np.array([-0.7])],
    3: [np.array([1.0, 1.0, 1.0]), np.array([0.5, -2.0, 0.0])],
    5: [np.array([1.0, -1.0, 0.25, 0.0, -0.25])],  # c̄ = 0: the -c̄ Q and -c̄ s terms vanish
}
CASES = [(prior, noise, zero_mean, layout) for prior in ("diag", "dense", "pdmat") for noise in ("scalar", "vector")
         for zero_mean in (True, False) for layout in ("col", "row")]


@pytest.mark.parametrize("prior,noise,zero_mean,layout", CASES)
@pytest.mark.parametrize("k", sorted(WEIGHTS))
def test_closed_forms_equal_autograd_through_the_reference_sequence(prior, noise, zero_mean, layout, k):
    fx, _ = problem(7, 40, 11, prior, noise, zero_mean, layout)
    Y = targets(fx, k, 3 + k)
    for c in WEIGHTS[k]:
        lps, want = autograd(fx, Y, c)
        for j in range(k):
            assert abs(lps[j] - ref.logpdf(fx, Y[:, j])) <= 1e-12 * abs(lps[j])
        got = gom.logpdf_multi_grad(fx, Y, c)
        for key in want:
            assert np.shape(got[key]) == np.shape(want[key]), key
            scale = max(np.max(np.abs(want[key])), 1e-300)
            err = float(np.max(np.abs(np.asarray(got[key]) - want[key])) / scale)
            assert err <= 1e-12, (key, c, err)


@pytest.mark.parametrize("prior,noise,layout", [("diag", "vector", "col"), ("dense", "scalar", "row"), ("pdmat", "vector", "row")])
def test_k1_reproduces_logpdf_grad(prior, noise, layout):
    fx, y = problem(6, 33, 5, prior, noise, False, layout)
    single = go.logpdf_grad(fx, y)
    for c in (1.0, -2.5):
        multi = gom.logpdf_multi_grad(fx, y[:, None], [c])
        for key in single:
            want = c * np.asarray(single[key])
            got = multi[key][:, 0] if key == "y" else multi[key]
            assert rel_inf(got, want) <= 1e-13, key


@pytest.mark.parametrize("prior,noise,layout", [("diag", "vector", "col"), ("dense", "scalar", "row"), ("pdmat", "vector", "row")])
def test_closed_forms_agree_with_central_differences(prior, noise, layout):
    fx, _ = problem(5, 30, 7, prior, noise, False, layout)
    Y = targets(fx, 3, 9)
    c = np.array([0.8, -1.3, 2.0])
    g = gom.logpdf_multi_grad(fx, Y, c)
    h = 1e-6

    def L(f, Yv):
        return sum(c[j] * ref.logpdf(f, Yv[:, j]) for j in range(Y.shape[1]))

    def fd(make):
        return (L(*make(+h)) - L(*make(-h))) / (2 * h)

    def check(approx, exact):
        assert abs(approx - exact) <= 1e-6 * max(1.0, abs(exact)), (approx, exact)

    X = fx.x.X
    for (i, j) in [(0, 0), (2, 3), (4, 1)]:
        def mk(d, i=i, j=j):
            Xp = X.copy()
            Xp[i, j] += d
            return fx.f(type(fx.x)(Xp), fx.Σy), Y
        check(fd(mk), g["X"][i, j])
    for (n, j) in [(0, 0), (17, 2), (29, 1)]:
        def mk(d, n=n, j=j):
            Yp = Y.copy()
            Yp[n, j] += d
            return fx, Yp
        check(fd(mk), g["y"][n, j])
    if noise == "scalar":
        check(fd(lambda d: (fx.f(fx.x, fx.Σy + d), Y)), g["σ²"])
    else:
        for n in (1, 29):
            def mk(d, n=n):
                s = np.array(fx.Σy, copy=True)
                s[n] += d
                return fx.f(fx.x, s), Y
            check(fd(mk), g["σ²"][n])
    for i in (0, 3):
        def mk(d, i=i):
            mw = fx.f.mw.copy()
            mw[i] += d
            return ref.BayesianLinearRegressor(mw, fx.f.Λw)(fx.x, fx.Σy), Y
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
            return ref.BayesianLinearRegressor(fx.f.mw, Λ)(fx.x, fx.Σy), Y
        if isinstance(fx.f.Λw, ref.Diagonal):
            if i == j:
                check(fd(mk), g["Λw"][i])
        else:
            check(fd(mk), g["Λw"][i, j])
