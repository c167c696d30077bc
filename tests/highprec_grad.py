"""Independent extended-precision truth for the gradients of logpdf and of the feature-map VJP -- TEST INFRASTRUCTURE.

numpy ``longdouble`` (x87 80-bit, eps 1.08e-19) with the hand-written factorisations of tests/highprec.py.  Nothing here is
shared with the fp64 closed forms of tests/grad_oracle*.py, which the CUDA kernels are otherwise checked against: those restate
the same formulas in the same rounding, so a formula that loses digits loses them in both.  tests/test_highprec_grad_pins.py
pins these functions against 50-digit mpmath.

With S = diag(s), s_n = 1/σ²_n, P = Λw + X S X', Q = P⁻¹, m' the posterior mean, u = m' - mw, e_n = y_n - x_n'm' and
h_n = x_n'Q x_n:

    ∂ℓ/∂x_n = s_n (e_n m' - Q x_n)     ∂ℓ/∂y_n = -s_n e_n      ∂ℓ/∂σ²_n = ½ (s_n² (h_n + e_n²) - s_n)
    ∂ℓ/∂mw  = Λw u                     ∂ℓ/∂Λw  = -½ (Q - Λw⁻¹ + u u')

Besides the gradients, ``ld_logpdf_grad`` returns the magnitudes the per-point and per-coordinate error criteria of
tests/test_gpu_grad_highprec.py divide by (``magnitudes``): the size of the terms before they cancel.
"""
from __future__ import annotations

import math

import numpy as np

from tests.highprec import LD, ld_cholesky, ld_solve_lower, ld_solve_upper

_CACHE: dict = {}


def cached(key, fn):
    """fn() once per key: the truth of one data set is reused by every test that reads it."""
    if key not in _CACHE:
        _CACHE[key] = fn()
    return _CACHE[key]


def _inverse_factor(A):
    """(L, L⁻¹) for the lower Cholesky factor L of A."""
    Lc = ld_cholesky(A)
    return Lc, ld_solve_lower(Lc, np.eye(A.shape[0], dtype=LD))


def _posterior(X, Y, σ2, mw, Λw):
    """Shared longdouble core: -> X, Y (N x k), s, Λ (dense), Q, Λw⁻¹, M' (D x k), U, E (N x k), QX, h."""
    X = np.asarray(X, dtype=LD)
    D, N = X.shape
    Y = np.asarray(Y, dtype=LD).reshape(N, -1)
    s = 1 / np.broadcast_to(np.asarray(σ2, dtype=LD), (N,))
    mw = np.asarray(mw, dtype=LD)
    Λ = np.asarray(Λw, dtype=LD)
    Λ = np.diag(Λ) if Λ.ndim == 1 else (Λ + Λ.T) / 2
    Xs = X * s
    G = Xs @ X.T
    P = Λ + (G + G.T) / 2
    Lp, Wp = _inverse_factor(P)
    Q = Wp.T @ Wp
    if np.asarray(Λw).ndim == 1:
        Λinv = np.diag(1 / np.asarray(Λw, dtype=LD))
    else:
        _, Ww = _inverse_factor(Λ)
        Λinv = Ww.T @ Ww
    R = Xs @ (Y - (X.T @ mw)[:, None])
    U = ld_solve_upper(Lp.T, ld_solve_lower(Lp, R))
    Mp = mw[:, None] + U
    E = Y - X.T @ Mp
    V = Wp @ X
    QX = Wp.T @ V
    h = np.sum(V * V, axis=0)
    return dict(X=X, Y=Y, s=s, Λ=Λ, Q=Q, Λinv=Λinv, Mp=Mp, U=U, E=E, QX=QX, h=h)


def ld_logpdf_grad(X, y, σ2, mw, Λw):
    """Gradients of logpdf for ColVecs X (D x N), vector y, scalar or vector σ², and a Diagonal (Λw a vector) or dense prior:
    the keys and shapes of tests/grad_oracle.logpdf_grad, in longdouble, plus "magnitudes" -- a dict with Q, m' ("mp"),
    u, e, h, |y| ("ay") and Σ_d |x_dn||m'_d| ("xm")."""
    c = _posterior(X, y, σ2, mw, Λw)
    s, Q, Mp, U, E, QX, h = c["s"], c["Q"], c["Mp"], c["U"], c["E"], c["QX"], c["h"]
    mp, u, e = Mp[:, 0], U[:, 0], E[:, 0]
    dσ2 = (s * s * (h + e * e) - s) / 2
    G = -(Q - c["Λinv"] + np.outer(u, u)) / 2
    diag = np.asarray(Λw).ndim == 1
    return {
        "X": np.outer(mp, s * e) - QX * s,
        "y": -s * e,
        "σ²": np.sum(dσ2) if np.ndim(σ2) == 0 else dσ2,
        "mw": c["Λ"] @ u,
        "Λw": np.diag(G).copy() if diag else (G + G.T) / 2,
        "magnitudes": {"Q": Q, "mp": mp, "u": u, "e": e, "h": h, "s": s, "ay": np.abs(c["Y"][:, 0]),
                       "xm": np.abs(c["X"]).T @ np.abs(mp), "qx": np.sqrt(np.sum(QX * QX, axis=0)),
                       "Λinv_diag": np.diag(c["Λinv"]).copy(), "c": np.ones(1, dtype=LD)},
    }


def ld_logpdf_multi_grad(X, Y, σ2, mw, Λw, c=None):
    """Gradients of L = Σ_j c_j logpdf(X, Y[:, j]) (c = None: all ones), the keys and shapes of
    tests/grad_oracle_multi.logpdf_multi_grad ("y" N x k), in longdouble, plus "magnitudes" as in ld_logpdf_grad with
    per-column mp, u, e, ay and xm (D x k, D x k, N x k, N x k, N x k) and the weights."""
    p = _posterior(X, Y, σ2, mw, Λw)
    s, Q, Mp, U, E, QX, h = p["s"], p["Q"], p["Mp"], p["U"], p["E"], p["QX"], p["h"]
    k = E.shape[1]
    c = np.ones(k, dtype=LD) if c is None else np.asarray(c, dtype=LD).reshape(k)
    cbar = np.sum(c)
    dσ2 = (s * s * (cbar * h + (E * E) @ c) - cbar * s) / 2
    G = -(cbar * (Q - p["Λinv"]) + (U * c) @ U.T) / 2
    diag = np.asarray(Λw).ndim == 1
    return {
        "X": (Mp * c) @ (E.T * s) - cbar * QX * s,
        "y": -(E * c) * s[:, None],
        "σ²": np.sum(dσ2) if np.ndim(σ2) == 0 else dσ2,
        "mw": p["Λ"] @ (U @ c),
        "Λw": np.diag(G).copy() if diag else (G + G.T) / 2,
        "magnitudes": {"Q": Q, "mp": Mp, "u": U, "e": E, "h": h, "s": s, "ay": np.abs(p["Y"]),
                       "xm": np.abs(p["X"]).T @ np.abs(Mp), "qx": np.sqrt(np.sum(QX * QX, axis=0)),
                       "Λinv_diag": np.diag(p["Λinv"]).copy(), "c": c},
    }


def ld_act_grad(z, act):
    """act'(z) in longdouble, stably: sech² z = 4e / (1 + e)² with e = exp(-2|z|) for tanh."""
    z = np.asarray(z, dtype=LD)
    if act == "cos":
        return -np.sin(z)
    if act == "sin":
        return np.cos(z)
    if act == "tanh":
        e = np.exp(-2 * np.abs(z))
        return 4 * e / (1 + e) ** 2
    if act == "relu":
        return (z > 0).astype(LD)
    return np.ones_like(z)


def ld_features_vjp(x, W, b, act, scale, dphi):
    """The VJP of ϕ(x) = scale * act(W x + b) for the cotangent dphi (D x N), with z formed from the exact fp64 inputs in
    longdouble: -> {"W": D x d_in, "b": D, "xin": d_in x N, "g": D x N}."""
    x, W = np.asarray(x, dtype=LD), np.asarray(W, dtype=LD)
    z = W @ x + np.asarray(b, dtype=LD)[:, None]
    g = np.asarray(dphi, dtype=LD) * LD(scale) * ld_act_grad(z, act)
    return {"W": g @ x.T, "b": g.sum(axis=1), "xin": W.T @ g, "g": g}


# ----------------------------------------------------------------------------------------------- error criteria
def _f64(a):
    return np.asarray(a, dtype=np.float64)


def _ld(a):
    return np.asarray(a, dtype=LD)


def rel(a, b) -> float:
    """norm-wise relative error of a (any precision) against the longdouble b (0 when both are 0)."""
    a, b = _ld(a), _ld(b)
    num, den = np.sqrt(np.sum((a - b) ** 2)), np.sqrt(np.sum(b * b))
    return float(num / den) if den > 0 else (0.0 if num == 0 else float("inf"))


def _ratio(err, M):
    """err / M elementwise, 0 where both are 0 and inf where only M is."""
    err, M = _ld(err), _ld(M)
    out = np.where(M > 0, err / np.where(M > 0, M, 1), np.where(err == 0, 0, np.inf))
    return float(np.max(out)) if out.size else 0.0


def point_magnitudes(t):
    """The size of the terms before they cancel, per point n (and column j), from a truth of ld_logpdf_grad or
    ld_logpdf_multi_grad; with a = Σ_j |c_j| and r_jn = |y_jn| + Σ_d |x_dn||m'_jd|:
        dX column  s_n (Σ_j |c_j| r_jn ‖m'_j‖ + a ‖Q x_n‖)        dY[n, j]  |c_j| s_n r_jn
        dσ²_n      ½ (s_n² (a h_n + Σ_j |c_j| r_jn²) + a s_n)     dλ_i      ½ (a (Q_ii + 1/λ_i) + Σ_j |c_j| u_ji²)
    (k = 1, c = 1: the single-column terms s_n ((|y_n| + Σ|x||m'|) ‖m'‖ + ‖Q x_n‖) and so on)."""
    m = t["magnitudes"]
    s, h, ac = m["s"], m["h"], np.abs(m["c"])
    N = s.shape[0]
    r = (m["ay"] + m["xm"]).reshape(N, -1)
    mpn = np.sqrt(np.sum(m["mp"].reshape(m["mp"].shape[0], -1) ** 2, axis=0))
    U = m["u"].reshape(m["u"].shape[0], -1)
    a = np.sum(ac)
    return {
        "X": s * ((r * ac) @ mpn + a * m["qx"]),
        "y": (r * ac) * s[:, None],
        "σ²": (s * s * (a * h + (r * r) @ ac) + a * s) / 2,
        "Λw": (a * (np.diag(m["Q"]) + m["Λinv_diag"]) + (U * U) @ ac) / 2,
    }


def logpdf_errors(g, t, vector_noise, diag_prior):
    """Distances of the fp64 gradients g (the keys of grad_oracle.logpdf_grad / logpdf_multi_grad, ColVecs layout) from the
    truth t: norm-wise for every output, and per point ("X/pt", "y/pt", "σ²/pt") and per coordinate of a Diagonal dΛw
    ("Λw/coord") relative to point_magnitudes(t)."""
    e = {k: rel(g[k], t[k]) for k in ("X", "y", "σ²", "mw", "Λw")}
    M = point_magnitudes(t)
    N = M["X"].shape[0]
    dX = _ld(g["X"]) - t["X"]
    e["X/pt"] = _ratio(np.sqrt(np.sum(dX * dX, axis=0)), M["X"])
    e["y/pt"] = _ratio(np.abs(_ld(g["y"]).reshape(N, -1) - t["y"].reshape(N, -1)), M["y"])
    if vector_noise:
        e["σ²/pt"] = _ratio(np.abs(_ld(g["σ²"]) - t["σ²"]), M["σ²"])
    if diag_prior:
        e["Λw/coord"] = _ratio(np.abs(_ld(g["Λw"]) - t["Λw"]), M["Λw"])
    return e


def features_vjp_errors(got, t, x, W):
    """Per entry |got - t| / M for the feature VJP, with g from the truth: M = Σ_n |g_dn||x_jn| for dW, Σ_n |g_dn| for db and
    Σ_d |W_dj||g_dn| for dx.  Returns the largest ratio per output."""
    ag = np.abs(_f64(t["g"]))
    M = {"W": ag @ np.abs(_f64(x)).T, "b": ag.sum(axis=1), "xin": np.abs(_f64(W)).T @ ag}
    return {k: _ratio(np.abs(_ld(got[k]) - t[k]), M[k]) for k in got}


def features_vjp_row_errors(got, t, x):
    """Per row d of dW: ‖dW_d - t_d‖ / Σ_{n,j} |g_dn||x_jn| -- what a wrong act' for one saturated unit shows up as."""
    ag = np.abs(_f64(t["g"]))
    M = np.sum(ag @ np.abs(_f64(x)).T, axis=1)
    d = _ld(got["W"]) - t["W"]
    return _ratio(np.sqrt(np.sum(d * d, axis=1)), M)


# ----------------------------------------------------------------------------------------------- the stress regimes
def spectrum_prior(rng, D, lo, hi):
    """Q diag(geomspace(lo, hi)) Q' for a random orthogonal Q: cond = hi / lo."""
    Q, _ = np.linalg.qr(rng.standard_normal((D, D)))
    Λ = (Q * np.geomspace(lo, hi, D)) @ Q.T
    return (Λ + Λ.T) / 2


REGIMES = ("cond1e6", "cond1e10", "cond1e13", "ard", "interp", "wide-noise", "scaled-rows", "pdmat-cond1e10")


def logpdf_problem(regime, D, N, seed):
    """The data of one stress regime -> dict X (D x N), y, σ2 (float or N), mw, Λw (a vector for a Diagonal prior, else D x D):
        cond1e6 / 1e10 / 1e13  dense Λw with that condition number, heteroscedastic noise exp(N(0, 1))
        ard                    Diagonal Λw = geomspace(1e-2, 1e12), heteroscedastic noise
        interp                 σ² = 1e-8 (scalar), dense Λw with cond 10; meant for N < D
        wide-noise             σ²_n = 10^U(-6, 6), dense Λw with cond 100
        scaled-rows            feature rows scaled by geomspace(1e-3, 1e3), dense Λw with cond 100, heteroscedastic noise
        pdmat-cond1e10         dense Λw with cond 1e10 (the test wraps it in a PDMat), heteroscedastic noise"""
    rng = np.random.default_rng(seed)
    X = rng.standard_normal((D, N))
    if regime == "scaled-rows":
        X *= np.geomspace(1e-3, 1e3, D)[:, None]
    if regime == "interp":
        σ2 = 1e-8
    elif regime == "wide-noise":
        σ2 = 10.0 ** rng.uniform(-6.0, 6.0, N)
    else:
        σ2 = np.exp(rng.standard_normal(N))
    if regime.startswith("cond") or regime == "pdmat-cond1e10":
        Λ = spectrum_prior(rng, D, 1.0, float(regime[regime.index("cond") + 4:]))
    elif regime == "ard":
        Λ = np.geomspace(1e-2, 1e12, D)
    else:
        Λ = spectrum_prior(rng, D, 1.0, 10.0 if regime == "interp" else 100.0)
    y = X.T @ rng.standard_normal(D) + np.sqrt(σ2) * rng.standard_normal(N)
    return {"X": X, "y": y, "σ2": σ2, "mw": rng.standard_normal(D), "Λw": Λ}


def multi_targets(p, k):
    """N x k targets for a logpdf_problem: its y, then k - 1 fresh draws from the same model."""
    X, σ2 = p["X"], p["σ2"]
    D, N = X.shape
    rng = np.random.default_rng(k)
    cols = [X.T @ rng.standard_normal(D) + np.sqrt(σ2) * rng.standard_normal(N) for _ in range(k - 1)]
    return np.stack([p["y"]] + cols, axis=1)


def zero_sum_weights(k, seed):
    """k non-zero weights, multiples of 1/4, summing to exactly 0 in fp64 (c̄ = 0: the Q and s terms of the rank-k gradients
    vanish and only the per-column terms remain)."""
    rng = np.random.default_rng(seed)
    c = rng.integers(1, 9, k) * rng.choice([-1.0, 1.0], k) / 4.0
    c[-1] = -np.sum(c[:-1])
    if c[-1] == 0.0:
        c[-1], c[0] = 0.25, c[0] - 0.25
    assert np.sum(c) == 0.0 and np.all(c != 0.0)
    return c


def saturated_tanh_problem(N, seed=1):
    """d_in = 33, D = 160, a third of the rows saturated: |b_d| in [8, 16], so |z| reaches about 20."""
    rng = np.random.default_rng(seed)
    din, D = 33, 160
    x = rng.standard_normal((din, N))
    W = rng.standard_normal((D, din)) / math.sqrt(din)
    b = rng.uniform(-2.0, 2.0, D)
    sat = np.arange(D) % 3 == 0
    b[sat] = rng.uniform(8.0, 16.0, sat.sum()) * rng.choice([-1.0, 1.0], sat.sum())
    return x, W, b, 0.7, rng.standard_normal((D, N)), sat


def feature_cases(N):
    """The feature-VJP cases of tests/test_gpu_grad_highprec.py at N points -> {tag: (x, W, b, act, scale, dphi)}."""
    x, W, b, scale, dphi, _ = saturated_tanh_problem(N)
    out = {"tanh-saturated": (x, W, b, "tanh", scale, dphi)}
    rng = np.random.default_rng(2)
    din, D = 3, 65
    xs = rng.standard_normal((din, N))
    Ω = rng.standard_normal((D, din))
    bs = rng.uniform(0.0, 2 * math.pi, D)
    dps = rng.standard_normal((D, N))
    for act in ("cos", "sin"):
        out[f"{act}-short-lengthscale"] = (xs, Ω / 1e-3, bs, act, math.sqrt(2.0 / D), dps)
    out["relu"] = relu_problem(N)
    rng = np.random.default_rng(4)
    din, D = 33, 160
    out["identity-scaled-cotangent"] = (rng.standard_normal((din, N)), rng.standard_normal((D, din)), rng.standard_normal(D),
                                        "identity", 0.7, rng.standard_normal((D, N)) * np.geomspace(1e-6, 1e6, D)[:, None])
    return out


def relu_problem(N, seed=3):
    """relu with every z at least 1e-12 (|W||x| + |b|) away from 0, apart from exact zeros: b_d = 0 on every fifth row and
    x_n = 0 on every seventh point."""
    rng = np.random.default_rng(seed)
    din, D = 33, 160
    x = rng.standard_normal((din, N))
    W = rng.standard_normal((D, din)) / math.sqrt(din)
    b = rng.standard_normal(D)
    b[::5] = 0.0
    x[:, ::7] = 0.0
    while True:
        z = W.astype(LD) @ x.astype(LD) + b.astype(LD)[:, None]
        scale_z = np.abs(W) @ np.abs(x) + np.abs(b)[:, None]
        near = (np.abs(z) < 1e-12 * scale_z) & (z != 0)
        if not near.any():
            return x, W, b, "relu", 0.7, rng.standard_normal((D, N))
        cols = np.unique(np.nonzero(near)[1])
        x[:, cols] = rng.standard_normal((din, cols.size))
