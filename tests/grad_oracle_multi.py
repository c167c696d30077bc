"""CPU reference for the gradients of the matrix form of logpdf (blr_logpdf_multi_grad), in closed form with numpy / scipy: the
single-column formulas of tests/grad_oracle.py summed over the columns with weights c.  tests/test_oracle_grad_multi.py pins them
against torch autograd through the reference's literal op sequence and against central finite differences.
"""
import numpy as np
import scipy.linalg as sl

from oracle import blr_oracle as ref


def logpdf_multi_grad(fx, Y, c=None):
    """Gradients of L = Σ_j c_j ℓ_j, ℓ_j = logpdf(fx, Y[:, j]) (blr_logpdf_multi_grad); c = None means all ones.  With c̄ = Σ_j c_j,
    M' = [m'_1 .. m'_k], U = M' - mw and E[n, j] = y_jn - x_n'm'_j, each line the single-column formula summed over the columns:

        ∂L/∂x_n = s_n (Σ_j c_j e_jn m'_j - c̄ Q x_n)     ∂L/∂Y[n, j] = -c_j s_n e_jn
        ∂L/∂σ²_n = ½ (s_n² (c̄ h_n + Σ_j c_j e_jn²) - c̄ s_n)
        ∂L/∂mw  = Λw U c                                ∂L/∂Λw = -½ (c̄ (Q - Λw⁻¹) + U diag(c) U')

    -> the same keys and shapes as logpdf_grad, "y" N x k."""
    X = ref.x_as_colvecs(fx.x)
    D, N = X.shape
    Y = np.asarray(Y, dtype=np.float64).reshape(N, -1)
    k = Y.shape[1]
    c = np.ones(k) if c is None else np.asarray(c, dtype=np.float64).reshape(k)
    cbar = float(np.sum(c))
    Σ = fx.noise(N)
    if not isinstance(Σ, ref.Diagonal):
        raise ValueError("closed-form gradients are defined for scalar / diagonal observation noise")
    s = 1.0 / np.asarray(Σ.diag, dtype=np.float64)
    Λ = ref.dense(fx.f.Λw)
    mw = fx.f.mw
    P = Λ + (X * s) @ X.T
    cP = sl.cho_factor(P, lower=False)
    Q = sl.cho_solve(cP, np.eye(D))
    Mp = mw[:, None] + sl.cho_solve(cP, (X * s) @ (Y - (X.T @ mw)[:, None]))
    U = Mp - mw[:, None]
    E = Y - X.T @ Mp
    QX = Q @ X
    h = np.sum(X * QX, axis=0)
    dX = (Mp * c) @ E.T * s - cbar * QX * s
    dσ2 = 0.5 * (s * s * (cbar * h + (E * E) @ c) - cbar * s)
    G = -0.5 * (cbar * (Q - sl.cho_solve(sl.cho_factor(Λ, lower=False), np.eye(D))) + (U * c) @ U.T)
    scalar = np.ndim(fx.Σy) == 0 and not isinstance(fx.Σy, (ref.Diagonal, ref.Symmetric, ref.PDMat))
    return {
        "X": dX.T.copy() if isinstance(fx.x, ref.RowVecs) else dX,
        "y": -(E * c) * s[:, None],
        "σ²": float(np.sum(dσ2)) if scalar else dσ2,
        "mw": Λ @ (U @ c),
        "Λw": np.diag(G).copy() if isinstance(fx.f.Λw, ref.Diagonal) else 0.5 * (G + G.T),
    }
