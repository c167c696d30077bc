"""CPU reference for the vector-Jacobian product of the device feature maps ϕ(x) = scale * act(W x + b) (blr_x_features_vjp),
in numpy.  With z = W x + b (D x N) and g = dΦ * scale * act'(z):

    dW = g x'      db = Σ_n g_n      dx = W' g

act' is -sin, 1 - tanh², 1[z > 0] (0 at z = 0, as torch and Flux define it), 1 and cos for "cos", "tanh", "relu", "identity" and
"sin".  tests/test_oracle_grad_features.py pins this against torch autograd and, composed with tests/grad_oracle.py, against
central differences of the log marginal likelihood.
"""
import numpy as np

ACTS = ("cos", "tanh", "relu", "identity", "sin")


def features(x, W, b, act, scale):
    """ϕ(x) for x d_in x N, W D x d_in, b D."""
    z = W @ x + b[:, None]
    a = {"cos": np.cos, "tanh": np.tanh, "relu": lambda t: np.maximum(t, 0.0), "identity": lambda t: t, "sin": np.sin}[act](z)
    return scale * a


def act_grad(z, act):
    if act == "cos":
        return -np.sin(z)
    if act == "sin":
        return np.cos(z)
    if act == "tanh":
        return 1.0 - np.tanh(z) ** 2
    if act == "relu":
        return (z > 0.0).astype(np.float64)
    return np.ones_like(z)


def features_vjp(x, W, b, act, scale, dphi):
    """-> {"W": D x d_in, "b": D, "xin": d_in x N} for the cotangent dphi (D x N)."""
    z = W @ x + b[:, None]
    g = dphi * scale * act_grad(z, act)
    return {"W": g @ x.T, "b": g.sum(axis=1), "xin": W.T @ g}
