"""CPU reference for the gradients of logpdf (blr_logpdf_grad), in closed form with numpy / scipy.

With S = diag(s), s_n = 1/σ²_n, P = Λw + X S X' the posterior precision, Q = P⁻¹, m' the posterior mean, u = m' - mw,
e_n = y_n - x_n'm' and h_n = x_n'Q x_n:

    ∂ℓ/∂x_n = s_n (e_n m' - Q x_n)     ∂ℓ/∂y_n = -s_n e_n      ∂ℓ/∂σ²_n = ½ (s_n² (h_n + e_n²) - s_n)
    ∂ℓ/∂mw  = Λw u                     ∂ℓ/∂Λw  = -½ (Q - Λw⁻¹ + u u')  (symmetric; its diagonal for a Diagonal prior)

Scalar noise gets the sum of ∂ℓ/∂σ²_n.  tests/test_oracle_grad.py pins these against torch autograd through the reference's
literal op sequence (oracle.blr_oracle.logpdf) and against central finite differences.
"""
import numpy as np
import scipy.linalg as sl

from oracle import blr_oracle as ref


def logpdf_grad(fx, y):
    """-> dict with keys "X" (shaped like fx.x.X: D x N for ColVecs / a bare matrix, N x D for RowVecs), "y", "σ²" (float for
    scalar noise, else N), "mw", "Λw" (D for a Diagonal prior, else D x D)."""
    X = ref.x_as_colvecs(fx.x)
    D, N = X.shape
    y = np.asarray(y, dtype=np.float64)
    Σ = fx.noise(N)
    if not isinstance(Σ, ref.Diagonal):
        raise ValueError("closed-form gradients are defined for scalar / diagonal observation noise")
    s = 1.0 / np.asarray(Σ.diag, dtype=np.float64)
    Λ = ref.dense(fx.f.Λw)
    mw = fx.f.mw
    P = Λ + (X * s) @ X.T
    cP = sl.cho_factor(P, lower=False)
    Q = sl.cho_solve(cP, np.eye(D))
    mp = mw + sl.cho_solve(cP, (X * s) @ (y - X.T @ mw))
    u = mp - mw
    e = y - X.T @ mp
    QX = Q @ X
    h = np.sum(X * QX, axis=0)
    dX = np.outer(mp, s * e) - QX * s
    dσ2 = 0.5 * (s * s * (h + e * e) - s)
    G = -0.5 * (Q - sl.cho_solve(sl.cho_factor(Λ, lower=False), np.eye(D)) + np.outer(u, u))
    scalar = np.ndim(fx.Σy) == 0 and not isinstance(fx.Σy, (ref.Diagonal, ref.Symmetric, ref.PDMat))
    return {
        "X": dX.T.copy() if isinstance(fx.x, ref.RowVecs) else dX,
        "y": -s * e,
        "σ²": float(np.sum(dσ2)) if scalar else dσ2,
        "mw": Λ @ u,
        "Λw": np.diag(G).copy() if isinstance(fx.f.Λw, ref.Diagonal) else 0.5 * (G + G.T),
    }
