"""CPU: pins for the extended-precision gradient truth of tests/highprec_grad.py and for the error criteria that
tests/test_gpu_grad_highprec.py holds the CUDA gradient kernels to.

  * The longdouble gradients of logpdf (single and rank k), and of the feature-map VJP, equal 50-digit mpmath closed forms to
    5e-16 -- the same pin tests/test_highprec_pins.py puts on the forward evaluator.  (The closed forms themselves are checked
    against autograd and finite differences in tests/test_oracle_grad*.py.)
  * Every criterion is achievable in fp64.  At a CPU-sized N of every stress regime, the fp64 yardsticks are finite, and an
    fp64 evaluation outside the yardstick set (the closed form on the same problem with its features permuted and its points
    reversed: the same math, other roundings) meets each criterion.  The per-point and per-coordinate criteria it meets with at
    least 100× margin wherever cond(Λw) is moderate (every regime but cond(Λw) = 1e10 and 1e13).  The norm-wise criteria, and
    every criterion at cond(Λw) >= 1e10, follow fp64's own error (cond · eps); their margin, printed, is what fp64 allows
    (4× to 30× where the yardstick sets the bound).  For the feature VJP a stable fp64 evaluation (sech² as 1/cosh²) meets
    |err| <= 1e-9 M with 100× margin.  So a failure of a GPU test points at the kernel, not at the criterion.
  * 1 - tanh² fails the per-row criterion of dW on saturated tanh units, and sech² passes it.
"""
import math

import mpmath as mp
import numpy as np
import pytest

from oracle import blr_oracle as ref
from tests import grad_oracle as go
from tests import grad_oracle_multi as gom
from tests import highprec_grad as hg
from tests.highprec import LD
from tests.test_oracle_grad import autograd
from tests.test_oracle_grad_multi import autograd as autograd_multi

RTOL, SLACK, MARGIN = 1e-9, 4.0, 100.0
DPS = 50


# ----------------------------------------------------------------------------------------------- 50-digit closed forms
def _mpm(a):
    a = np.asarray(a, dtype=np.float64)
    return mp.matrix(a.tolist()) if a.ndim == 2 else mp.matrix([mp.mpf(float(v)) for v in a])


def _to_ld(m, shape):
    """an mpmath matrix / list of mpf -> longdouble array (through decimal strings: every longdouble digit kept)"""
    flat = [m[i] for i in range(len(m))] if not isinstance(m, mp.matrix) else \
        [m[i, j] for i in range(m.rows) for j in range(m.cols)]
    return np.array([LD(mp.nstr(v, 30)) for v in flat], dtype=LD).reshape(shape)


def mp_logpdf_multi_grad(X, Y, σ2, mw, Λw, c):
    """The closed forms of tests/highprec_grad.py (k columns, weights c) at DPS digits, with explicit inverses."""
    mp.mp.dps = DPS
    D, N = X.shape
    Y = np.asarray(Y).reshape(N, -1)
    k = Y.shape[1]
    Xm = _mpm(X)
    s = [1 / mp.mpf(float(v)) for v in np.broadcast_to(np.asarray(σ2, dtype=np.float64), (N,))]
    Λ = mp.diag([mp.mpf(float(v)) for v in Λw]) if np.ndim(Λw) == 1 else _mpm(Λw)
    XS = Xm.copy()
    for n in range(N):
        for d in range(D):
            XS[d, n] *= s[n]
    P = Λ + XS * Xm.T
    Q = mp.inverse(P)
    Λi = mp.inverse(Λ)
    mwm = _mpm(mw)
    cbar = sum(mp.mpf(float(v)) for v in c)
    QX = Q * Xm
    h = [sum(Xm[d, n] * QX[d, n] for d in range(D)) for n in range(N)]
    dX = mp.matrix(D, N) - cbar * QX
    for n in range(N):
        for d in range(D):
            dX[d, n] *= s[n]
    dY, dσ2 = mp.matrix(N, k), [-cbar * s[n] + cbar * s[n] ** 2 * h[n] for n in range(N)]
    dmw, G = mp.matrix(D, 1), -cbar * (Q - Λi)
    for j in range(k):
        cj = mp.mpf(float(c[j]))
        yj = _mpm(Y[:, j])
        u = Q * (XS * (yj - Xm.T * mwm))
        mpj = mwm + u
        e = yj - Xm.T * mpj
        for n in range(N):
            dY[n, j] = -cj * s[n] * e[n]
            dσ2[n] += cj * s[n] ** 2 * e[n] ** 2
            for d in range(D):
                dX[d, n] += cj * s[n] * e[n] * mpj[d]
        dmw += cj * (Λ * u)
        G -= cj * (u * u.T)
    G = G / 2
    dσ2 = [v / 2 for v in dσ2]
    out = {"X": _to_ld(dX, (D, N)), "y": _to_ld(dY, (N, k)), "mw": _to_ld(dmw, (D,)),
           "σ²": _to_ld(dσ2, (N,)) if np.ndim(σ2) else np.sum(_to_ld(dσ2, (N,)))}
    Gl = _to_ld(G, (D, D))
    out["Λw"] = np.diag(Gl).copy() if np.ndim(Λw) == 1 else Gl
    return out


def mp_features_vjp(x, W, b, act, scale, dphi):
    mp.mp.dps = DPS
    din, N = x.shape
    D = W.shape[0]
    fn = {"tanh": lambda z: 1 / mp.cosh(z) ** 2, "cos": lambda z: -mp.sin(z), "sin": mp.cos}[act]
    g = [[mp.mpf(float(dphi[d, n])) * mp.mpf(scale) *
          fn(mp.fsum(mp.mpf(float(W[d, i])) * mp.mpf(float(x[i, n])) for i in range(din)) + mp.mpf(float(b[d])))
          for n in range(N)] for d in range(D)]
    gm = mp.matrix(g)
    xm, Wm = _mpm(x), _mpm(W)
    db = [mp.fsum(g[d]) for d in range(D)]
    return {"W": _to_ld(gm * xm.T, (D, din)), "b": _to_ld(db, (D,)), "xin": _to_ld(Wm.T * gm, (din, N))}


def toy(D, N, seed, prior, noise, k=None):
    rng = np.random.default_rng(seed)
    X = rng.standard_normal((D, N))
    B = rng.standard_normal((D, D)) / math.sqrt(D)
    Λd = B @ B.T + np.eye(D)
    Λ = {"diag": np.exp(rng.standard_normal(D)), "dense": Λd, "pdmat": ref.PDMat.from_matrix(Λd).mat}[prior]
    σ2 = 0.6 if noise == "scalar" else np.exp(rng.standard_normal(N))
    shape = (N,) if k is None else (N, k)
    y = X.T @ rng.standard_normal((D,) + shape[1:]) + 0.5 * rng.standard_normal(shape)
    return X, y, σ2, rng.standard_normal(D), Λ


@pytest.mark.parametrize("prior", ["diag", "dense", "pdmat"])
@pytest.mark.parametrize("noise", ["scalar", "vector"])
@pytest.mark.parametrize("D,N", [(7, 13), (24, 60)])
def test_longdouble_gradients_against_mpmath(D, N, prior, noise):
    X, y, σ2, mw, Λ = toy(D, N, 10 * D + N, prior, noise)
    ld = hg.ld_logpdf_grad(X, y, σ2, mw, Λ)
    want = mp_logpdf_multi_grad(X, y, σ2, mw, Λ, [1.0])
    want["y"] = want["y"][:, 0]
    for key in want:
        assert hg.rel(ld[key], want[key]) < 5e-16, key


@pytest.mark.parametrize("prior,noise", [("diag", "vector"), ("dense", "scalar"), ("pdmat", "vector")])
def test_longdouble_multi_gradients_against_mpmath(prior, noise):
    X, Y, σ2, mw, Λ = toy(24, 60, 7, prior, noise, k=3)
    c = np.array([1.0, -0.5, 2.0])
    ld = hg.ld_logpdf_multi_grad(X, Y, σ2, mw, Λ, c)
    want = mp_logpdf_multi_grad(X, Y, σ2, mw, Λ, c)
    for key in want:
        assert hg.rel(ld[key], want[key]) < 5e-16, key


@pytest.mark.parametrize("act", ["tanh", "cos", "sin"])
def test_longdouble_features_vjp_against_mpmath(act):
    rng = np.random.default_rng(3)
    din, D, N = 3, 9, 40
    x = rng.standard_normal((din, N))
    W = rng.standard_normal((D, din)) / (1e-3 if act != "tanh" else 1.0)
    b = rng.uniform(-16.0, 16.0, D) if act == "tanh" else rng.uniform(0.0, 2 * math.pi, D)  # tanh: |z| up to ~20
    dphi = rng.standard_normal((D, N))
    ld = hg.ld_features_vjp(x, W, b, act, 0.7, dphi)
    want = mp_features_vjp(x, W, b, act, 0.7, dphi)
    for key in want:
        assert hg.rel(ld[key], want[key]) < 5e-16, key
    for d in range(W.shape[0] if act == "tanh" else 0):  # row by row too: a saturated row is ~1e-14 of the norm
        assert hg.rel(ld["W"][d], want["W"][d]) < 5e-16 and hg.rel(ld["b"][d], want["b"][d]) < 5e-16, d


# ----------------------------------------------------------------------------------------------- achievable in fp64
def permuted_closed_form(p, k=None, c=None):
    """grad_oracle(_multi) on the same problem with the features permuted and the points reversed, mapped back: the same
    mathematics in other roundings -- a correct fp64 implementation that is not one of the yardsticks."""
    X, Λ, mw = p["X"], p["Λw"], p["mw"]
    D, N = X.shape
    pf = np.random.default_rng(0).permutation(D)
    pn = np.arange(N)[::-1]
    Λp = Λ[pf] if np.ndim(Λ) == 1 else Λ[np.ix_(pf, pf)]
    σ2p = p["σ2"] if np.ndim(p["σ2"]) == 0 else p["σ2"][pn]
    fo = ref.BayesianLinearRegressor(mw[pf], ref.Diagonal(Λp) if np.ndim(Λ) == 1 else Λp)(ref.ColVecs(X[np.ix_(pf, pn)]), σ2p)
    g = go.logpdf_grad(fo, p["y"][pn]) if k is None else gom.logpdf_multi_grad(fo, p["y"][pn], c)
    inv = np.argsort(pf)
    out = {"X": g["X"][np.ix_(inv, np.argsort(pn))], "y": g["y"][np.argsort(pn)], "mw": g["mw"][inv],
           "σ²": g["σ²"] if np.ndim(p["σ2"]) == 0 else g["σ²"][np.argsort(pn)],
           "Λw": g["Λw"][inv] if np.ndim(Λ) == 1 else g["Λw"][np.ix_(inv, inv)]}
    return out


def yardsticks(p, k=None, c=None):
    """The fp64 evaluations the GPU tests widen their bound by: the closed form and torch autograd through the reference's
    literal op sequence (of Σ_j c_j ℓ_j for rank k)."""
    Λo = ref.Diagonal(p["Λw"]) if np.ndim(p["Λw"]) == 1 else p["Λw"]
    fo = ref.BayesianLinearRegressor(p["mw"], Λo)(ref.ColVecs(p["X"]), p["σ2"])
    if k is None:
        return {"oracle": go.logpdf_grad(fo, p["y"]), "autograd": autograd(fo, p["y"])[1]}
    return {"oracle": gom.logpdf_multi_grad(fo, p["y"], c), "autograd": autograd_multi(fo, p["y"], c)[1]}


CPU_REGIMES = [
    # regime, D, N (the GPU cases' regimes at a CPU-sized N; D = 1024 and 600 stand in at 256 and 130), conditioning-limited
    ("cond1e6", 64, 300, False), ("cond1e10", 64, 300, True), ("cond1e13", 256, 300, True), ("ard", 130, 300, False),
    ("interp", 256, 100, False), ("wide-noise", 130, 400, False), ("scaled-rows", 96, 300, False),
    ("pdmat-cond1e10", 127, 300, True),
]


@pytest.mark.parametrize("regime,D,N,limited", CPU_REGIMES, ids=[f"{r[0]}-D{r[1]}" for r in CPU_REGIMES])
@pytest.mark.parametrize("k", [None, 9])
def test_criteria_achievable_in_fp64(regime, D, N, limited, k):
    p = hg.logpdf_problem(regime, D, N, seed=D + N)
    c = None
    if k is not None:
        p["y"] = hg.multi_targets(p, k)
        c = hg.zero_sum_weights(k, k)
        t = hg.ld_logpdf_multi_grad(p["X"], p["y"], p["σ2"], p["mw"], p["Λw"], c)
    else:
        t = hg.ld_logpdf_grad(p["X"], p["y"], p["σ2"], p["mw"], p["Λw"])
    vec, diag = np.ndim(p["σ2"]) == 1, np.ndim(p["Λw"]) == 1
    ys = {name: hg.logpdf_errors(g, t, vec, diag) for name, g in yardsticks(p, k, c).items()}
    alt = hg.logpdf_errors(permuted_closed_form(p, k, c), t, vec, diag)
    rows = []
    for crit, e_alt in alt.items():
        worst = max(e[crit] for e in ys.values())
        assert all(math.isfinite(e[crit]) for e in ys.values()), (crit, ys)
        bound = max(RTOL, SLACK * worst)
        margin = bound / max(e_alt, 1e-300)
        rows.append(f"{crit} {e_alt:.1e} (x{margin:.0f})")
        assert margin >= (MARGIN if "/" in crit and not limited else 1.0), (crit, e_alt, bound)
    print(f"[fp64] {regime} D={D} N={N} k={k}: " + " | ".join(rows))


def fp64_vjp(x, W, b, act, scale, dphi, tanh_grad):
    z = W @ x + b[:, None]
    a = {"tanh": tanh_grad, "cos": lambda t: -np.sin(t), "sin": np.cos, "relu": lambda t: (t > 0.0).astype(np.float64),
         "identity": np.ones_like}[act](z)
    g = dphi * scale * a
    return {"W": g @ x.T, "b": g.sum(axis=1), "xin": W.T @ g}


def sech2(z):
    return 1.0 / np.cosh(z) ** 2


def one_minus_tanh2(z):
    return 1.0 - np.tanh(z) ** 2


@pytest.mark.parametrize("tag", ["tanh-saturated", "cos-short-lengthscale", "sin-short-lengthscale", "relu",
                                 "identity-scaled-cotangent"])
def test_features_criterion_achievable_in_fp64(tag):
    x, W, b, act, scale, dphi = hg.feature_cases(3001)[tag]
    t = hg.ld_features_vjp(x, W, b, act, scale, dphi)
    e = hg.features_vjp_errors(fp64_vjp(x, W, b, act, scale, dphi, sech2), t, x, W)
    print(f"[fp64] {tag}: " + " | ".join(f"{k} {v:.1e}" for k, v in e.items()))
    assert all(v <= RTOL / MARGIN for v in e.values()), e


def test_one_minus_tanh_squared_fails_the_row_criterion_when_saturated():
    x, W, b, scale, dphi, sat = hg.saturated_tanh_problem(3001)
    t = hg.ld_features_vjp(x, W, b, "tanh", scale, dphi)
    naive = hg.features_vjp_row_errors(fp64_vjp(x, W, b, "tanh", scale, dphi, one_minus_tanh2), t, x)
    stable = hg.features_vjp_row_errors(fp64_vjp(x, W, b, "tanh", scale, dphi, sech2), t, x)
    print(f"[fp64] saturated tanh, worst dW row: 1 - tanh² {naive:.1e}, sech² {stable:.1e}")
    assert naive > RTOL and stable <= RTOL / MARGIN
