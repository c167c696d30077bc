"""GPU: the gradient kernels (blr_logpdf_grad, blr_logpdf_multi_grad in csrc/grad.cu; blr_x_features_vjp in
csrc/features_grad.cu) against the extended-precision truth of tests/highprec_grad.py, on ill-conditioned, wide-range and
saturated inputs: the regimes where an ML-II optimiser runs and where fp64 closed forms lose digits.

Criteria (t the longdouble truth; Y the fp64 yardsticks: tests/grad_oracle*.py and torch autograd through the reference's
literal op sequence, of Σ_j c_j ℓ_j for rank k):
  * norm-wise, every output:      rel(dev, t) <= max(1e-9, 4 max_Y rel(y, t))                       (as tests/test_gpu_illcond.py)
  * per point, dX / dy / dσ²:     max_n |dev_n - t_n| / M_n, the same rule, M_n the size of the terms before they cancel
                                  (highprec_grad.point_magnitudes); per coordinate of a Diagonal dΛw likewise
  * feature VJP, per entry:       |dev - t| <= 1e-9 M, M = Σ_n |g_dn||x_jn| (dW), Σ_n |g_dn| (db), Σ_d |W_dj||g_dn| (dx)
tests/test_highprec_grad_pins.py shows on the CPU that each is met by fp64 (the per-point ones and the feature VJP with 100×
margin where the conditioning allows), so a failure here is a kernel defect.  Every test prints its error table.
"""
import math

import numpy as np
import pytest

import blr_b200 as blr
from oracle import blr_oracle as ref
from tests import highprec_grad as hg
from tests.test_gpu_features_grad import raw_vjp
from tests.test_highprec_grad_pins import yardsticks

pytestmark = pytest.mark.gpu
RTOL, SLACK = 1e-9, 4.0


def device_fx(p, layout="col", pdmat=False):
    X, Λ = p["X"], p["Λw"]
    if np.ndim(Λ) == 1:
        prior = blr.Diagonal(Λ)
    elif pdmat:
        po = ref.PDMat.from_matrix(Λ)
        prior = blr.PDMat(po.mat, po.U)
    else:
        prior = Λ
    x = blr.ColVecs(X) if layout == "col" else blr.RowVecs(np.ascontiguousarray(X.T))
    return blr.BayesianLinearRegressor(p["mw"], prior)(x, p["σ2"])


def device_grad(p, layout="col", pdmat=False, form="direct", c=None):
    ctx = blr.default_context()
    ctx.set_form(form)
    try:
        _, g = blr.logpdf_and_grad(device_fx(p, layout, pdmat), p["y"], weights=c)
    finally:
        ctx.set_form("direct")
    g = dict(g)
    if layout == "row":
        g["X"] = np.asarray(g["X"]).T
    return g


def check(tag, t, g_dev, ys, vec, diag):
    """the norm-wise, per-point and per-coordinate rules against the yardsticks ys (name -> gradients)"""
    e_dev = hg.logpdf_errors(g_dev, t, vec, diag)
    e_y = {name: hg.logpdf_errors(g, t, vec, diag) for name, g in ys.items()}
    rows, bad = [], {}
    for crit, e in e_dev.items():
        worst = max(ey[crit] for ey in e_y.values())
        bound = max(RTOL, SLACK * worst)
        rows.append(f"{crit} gpu {e:.1e} ref {worst:.1e}")
        if not e <= bound:
            bad[crit] = (e, bound)
    print(f"[grad-highprec] {tag}: " + " | ".join(rows))
    assert not bad, (tag, bad)
    return e_dev


def problem(regime, D, N):
    return hg.cached(("data", regime, D, N), lambda: hg.logpdf_problem(regime, D, N, seed=D + N))


def truth(regime, D, N, k=None):
    p = problem(regime, D, N)
    if k is None:
        return hg.cached(("truth", regime, D, N), lambda: hg.ld_logpdf_grad(p["X"], p["y"], p["σ2"], p["mw"], p["Λw"]))
    Y, c = multi(regime, D, N, k)
    return hg.cached(("truth", regime, D, N, k), lambda: hg.ld_logpdf_multi_grad(p["X"], Y, p["σ2"], p["mw"], p["Λw"], c))


def multi(regime, D, N, k):
    return hg.cached(("multi", regime, D, N, k), lambda: (hg.multi_targets(problem(regime, D, N), k), hg.zero_sum_weights(k, k)))


CASES = [
    # regime, D, N, layout, form -- and the kernel path it reaches (api.cu / grad.cu dispatch)
    ("cond1e6", 64, 500, "col", "direct"),         # grad_x fast path, one pass
    ("cond1e10", 64, 500, "col", "direct"),
    ("cond1e13", 64, 500, "col", "direct"),
    ("cond1e6", 256, 1500, "col", "direct"),       # grad_x fast path, one pass
    ("cond1e10", 256, 1500, "col", "direct"),
    ("cond1e13", 256, 1500, "col", "direct"),
    ("cond1e6", 1024, 1100, "col", "direct"),      # grad_x fast path, four passes
    ("cond1e10", 1024, 1100, "col", "direct"),
    ("cond1e13", 1024, 1100, "col", "direct"),
    ("ard", 130, 1500, "col", "direct"),           # TMA Gram, ragged rows; Diagonal dΛw
    ("interp", 256, 100, "col", "direct"),         # σ² = 1e-8, N < D, scalar noise
    ("wide-noise", 600, 2000, "col", "direct"),    # grad_x fast path, three passes, ragged last one
    ("scaled-rows", 96, 1031, "row", "direct"),    # RowVecs: K1m, staged
    ("pdmat-cond1e10", 127, 1100, "col", "direct"),  # odd D: generic grad_x
    ("cond1e10", 256, 1500, "col", "whitened"),
    ("wide-noise", 130, 1500, "col", "whitened"),
]


@pytest.mark.parametrize("regime,D,N,layout,form", CASES, ids=[f"{c[0]}-D{c[1]}-{c[4]}" for c in CASES])
def test_logpdf_gradients_against_extended_precision(regime, D, N, layout, form):
    p = problem(regime, D, N)
    t = truth(regime, D, N)
    pdmat = regime.startswith("pdmat")
    g = device_grad(p, layout, pdmat, form)
    vec, diag = np.ndim(p["σ2"]) == 1, np.ndim(p["Λw"]) == 1
    check(f"{regime} D={D} N={N} {layout} {form}", t, g, yardsticks(p), vec, diag)
    if diag:
        # Diagonal dλ_i = -½(Q_ii - 1/λ_i + u_i²) cancels where λ_i >> G_ii; recorded relative to each coordinate's value
        err = np.abs(np.asarray(g["Λw"], dtype=hg.LD) - t["Λw"]) / np.abs(t["Λw"])
        print(f"[grad-highprec] {regime} D={D}: Diagonal dΛw, largest error relative to the coordinate's value {float(np.max(err)):.1e}")


MULTI = [("cond1e10", 256, 1500), ("wide-noise", 600, 2000)]


@pytest.mark.parametrize("regime,D,N", MULTI, ids=[f"{m[0]}-D{m[1]}" for m in MULTI])
@pytest.mark.parametrize("k", [9, 17])
def test_multi_gradients_against_extended_precision(regime, D, N, k):
    p = dict(problem(regime, D, N))
    Y, c = multi(regime, D, N, k)
    p["y"] = Y
    t = truth(regime, D, N, k)
    g = device_grad(p, c=c)
    assert np.shape(g["y"]) == (N, k)
    check(f"{regime} D={D} N={N} k={k} c̄=0", t, g, yardsticks(p, k, c), np.ndim(p["σ2"]) == 1, False)


def test_duplicated_and_zero_points():
    """Duplicated points get bit-identical dX columns, dy and dσ²; a point at x = 0 gets dX = s e m' and dσ² = ½(s² e² - s)
    to within the per-point bound."""
    D, N = 130, 1500
    p = dict(hg.logpdf_problem("wide-noise", D, N, seed=11))
    X, y, σ2 = p["X"].copy(), p["y"].copy(), p["σ2"].copy()
    dup = [(10, 500), (63, 64), (700, N - 1)]  # other tiles, a tile boundary, the ragged last tile
    for a, b in dup:
        X[:, b], y[b], σ2[b] = X[:, a], y[a], σ2[a]
    z = 333
    X[:, z] = 0.0
    p.update(X=X, y=y, σ2=σ2)
    g = device_grad(p)
    dX, dy, ds = np.asarray(g["X"]), np.asarray(g["y"]), np.asarray(g["σ²"])
    for a, b in dup:
        assert np.array_equal(dX[:, a], dX[:, b]) and dy[a] == dy[b] and ds[a] == ds[b], (a, b)
    t = hg.ld_logpdf_grad(X, y, σ2, p["mw"], p["Λw"])
    m = t["magnitudes"]
    M = hg.point_magnitudes(t)
    s, e = m["s"][z], m["e"][z]
    d = np.asarray(dX[:, z], dtype=hg.LD) - s * e * m["mp"]
    eX = float(np.sqrt(np.sum(d * d)) / M["X"][z])
    eS = float(abs(hg.LD(ds[z]) - (s * s * e * e - s) / 2) / M["σ²"][z])
    print(f"[grad-highprec] x_n = 0: dX column {eX:.1e}, dσ² {eS:.1e} of the per-point magnitude")
    assert eX <= RTOL and eS <= RTOL


FEATURE_N = (1 << 15) + 1  # the per-range partials and the fixed-order reduce both run; ragged last tile


@pytest.mark.parametrize("tag", ["tanh-saturated", "cos-short-lengthscale", "sin-short-lengthscale", "relu",
                                 "identity-scaled-cotangent"])
def test_features_vjp_against_extended_precision(tag):
    x, W, b, act, scale, dphi = hg.cached("features", lambda: hg.feature_cases(FEATURE_N))[tag]
    t = hg.cached(("features-truth", tag), lambda: hg.ld_features_vjp(x, W, b, act, scale, dphi))
    got = raw_vjp(x, W, b, act, scale, dphi)
    e = hg.features_vjp_errors(got, t, x, W)
    rows = hg.features_vjp_row_errors(got, t, x)
    print(f"[grad-highprec] features {tag} d_in={x.shape[0]} D={W.shape[0]} N={x.shape[1]}: " +
          " | ".join(f"{k} {v:.1e}" for k, v in e.items()) + f" | worst dW row {rows:.1e}")
    assert all(v <= RTOL for v in e.values()), e


def test_logpdf_and_grad_through_saturated_tanh_features():
    """logpdf_and_grad(bfr, y, wrt=("W", "b", "xin")) through tanh AffineFeatures with a third of the units saturated, against
    ld_logpdf_grad at the features chained into ld_features_vjp."""
    rng = np.random.default_rng(17)
    din, D, N = 5, 80, 2000
    x = rng.standard_normal((din, N))
    W = rng.standard_normal((D, din)) / math.sqrt(din)
    b = rng.uniform(-2.0, 2.0, D)
    sat = np.arange(D) % 3 == 0
    b[sat] = rng.uniform(8.0, 16.0, sat.sum()) * rng.choice([-1.0, 1.0], sat.sum())
    scale = 0.8
    z = W.astype(hg.LD) @ x.astype(hg.LD) + b.astype(hg.LD)[:, None]
    Phi = np.asarray(scale * np.tanh(z), dtype=np.float64)
    mw, lam = 0.1 * rng.standard_normal(D), np.exp(rng.standard_normal(D))
    σ2 = np.exp(0.3 * rng.standard_normal(N))
    y = Phi.T @ rng.standard_normal(D) + 0.5 * rng.standard_normal(N)
    ϕ = blr.AffineFeatures(W, b, "tanh", scale)
    fx = blr.BasisFunctionRegressor(blr.BayesianLinearRegressor(mw, blr.Diagonal(lam)), ϕ)(blr.ColVecs(x), σ2)
    _, g = blr.logpdf_and_grad(fx, y, wrt=("W", "b", "xin"))
    dPhi = hg.ld_logpdf_grad(Phi, y, σ2, mw, lam)["X"]
    t = hg.ld_features_vjp(x, W, b, "tanh", scale, dPhi)
    e = hg.features_vjp_errors({k: g[k] for k in ("W", "b", "xin")}, t, x, W)
    rows = hg.features_vjp_row_errors(g, t, x)
    print("[grad-highprec] logpdf_and_grad through saturated tanh: " + " | ".join(f"{k} {v:.1e}" for k, v in e.items()) +
          f" | worst dW row {rows:.1e}")
    assert all(v <= RTOL for v in e.values()), e
