"""GPU: the feature-map VJP (blr_x_features_vjp, csrc/features_grad.cu; AffineFeatures.vjp / RandomFourierFeatures.vjp,
logpdf_and_grad with "W", "b", "xin" and torch_features in the package) against the numpy VJP of tests/grad_oracle_features.py,
‖g_dev - g_ref‖∞ / ‖g_ref‖∞ <= 1e-9 for every output, over every activation, d_in from 1 to 384, D from 1 to 4096, N from 0 to
2^15 (one tile, tile ± 1), padded leading dimensions and each output requested alone.  Also: bit-identical repeated calls,
launch counts, the error contract, logpdf gradients through RFF and affine regressors (vector y and a weighted matrix Y),
torch_features composed with torch_logpdf, a random-Fourier-feature lengthscale fitted by Adam, one full-size shape and two
ranks."""
import ctypes as C
import math
import os
import socket
import subprocess
import sys
import textwrap

import numpy as np
import pytest

import blr_b200 as blr
from blr_b200 import _lib as L
from oracle import blr_oracle as ref
from tests import grad_oracle as go
from tests import grad_oracle_features as gof
from tests import grad_oracle_multi as gom

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
RTOL = 1e-9
ACT = {"cos": 0, "tanh": 1, "relu": 2, "identity": 3, "sin": 4}
TILE = 64  # points per tile of features_vjp_x_kernel / features_vjp_w_kernel


def rel_inf(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    if a.size == 0 and b.size == 0:
        return 0.0
    return float(np.max(np.abs(a - b)) / max(np.max(np.abs(b)), np.finfo(np.float64).tiny))


def problem(din, D, N, act, seed):
    rng = np.random.default_rng(seed)
    x = rng.standard_normal((din, N))
    W = rng.standard_normal((D, din)) / math.sqrt(din)
    b = rng.uniform(0.0, 2.0 * math.pi, D)
    scale = math.sqrt(2.0 / D) if act == "cos" else 0.7
    dphi = rng.standard_normal((D, N))
    return x, W, b, scale, dphi


def raw_vjp(x, W, b, act, scale, dphi, want=("W", "b", "xin"), pad_phi=0, pad_x=0):
    """One blr_x_features_vjp call through the C ABI with leading dimensions D + pad_phi and d_in + pad_x."""
    import torch

    ctx = blr.default_context()
    din, N = x.shape
    D = W.shape[0]
    xin = blr.DeviceMatrix.upload(ctx, x, L.COLVECS)
    ldp, ldx = D + pad_phi, din + pad_x
    dp = torch.zeros((max(N, 1), ldp), dtype=torch.float64, device="cuda")
    dp[:N, :D] = torch.from_numpy(dphi.T.copy())
    dx = torch.full((max(N, 1), ldx), 7.0, dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    Wf, bf = np.asfortranarray(W), np.ascontiguousarray(b)
    dW = np.full((D, din), np.nan, order="F") if "W" in want else None
    db = np.full(D, np.nan) if "b" in want else None
    ctx.check(ctx.lib.blr_x_features_vjp(ctx.handle, xin.handle, Wf.ctypes.data_as(C.c_void_p), bf.ctypes.data_as(C.c_void_p), D,
                                         ACT[act], scale, C.c_void_p(dp.data_ptr()), ldp,
                                         None if dW is None else dW.ctypes.data_as(C.c_void_p),
                                         None if db is None else db.ctypes.data_as(C.c_void_p),
                                         C.c_void_p(dx.data_ptr()) if "xin" in want else None, ldx))
    ctx.sync()
    out = {}
    if dW is not None:
        out["W"] = dW
    if db is not None:
        out["b"] = db
    if "xin" in want:
        h = dx.cpu().numpy()
        out["xin"] = h[:N, :din].T.copy()
        if pad_x:
            assert np.all(h[:N, din:] == 7.0), "dxin padding written"
    return out


def check(got, want, tag):
    for key in got:
        assert np.shape(got[key]) == np.shape(want[key]), (tag, key)
        err = rel_inf(got[key], want[key])
        assert err <= RTOL, (tag, key, err)


@pytest.mark.parametrize("act", list(ACT))
@pytest.mark.parametrize("din", [1, 3, 32, 33, 384])
def test_every_activation_and_input_width(act, din):
    x, W, b, scale, dphi = problem(din, 65, TILE + 1, act, din)
    check(raw_vjp(x, W, b, act, scale, dphi), gof.features_vjp(x, W, b, act, scale, dphi), (act, din))


@pytest.mark.parametrize("D", [1, 7, 64, 65, 160])
@pytest.mark.parametrize("N", [0, 1, 17, TILE - 1, TILE + 1, 1 << 15])
def test_shapes(D, N):
    for act, din in (("cos", 32), ("tanh", 33)):
        x, W, b, scale, dphi = problem(din, D, N, act, D + N)
        got = raw_vjp(x, W, b, act, scale, dphi)
        want = gof.features_vjp(x, W, b, act, scale, dphi)
        if N == 0:
            assert np.all(got["W"] == 0.0) and np.all(got["b"] == 0.0) and got["xin"].shape == (din, 0)
        else:
            check(got, want, (act, din, D, N))


def test_wide_output_small_n():
    x, W, b, scale, dphi = problem(32, 4096, 17, "cos", 9)
    check(raw_vjp(x, W, b, "cos", scale, dphi), gof.features_vjp(x, W, b, "cos", scale, dphi), "D=4096")


def test_relu_derivative_is_zero_at_zero():
    """b = 0 and every third input column 0 give z = 0 exactly there: relu' = 0 (torch, Flux), so those points add nothing"""
    x, W, b, scale, dphi = problem(5, 40, 90, "relu", 13)
    b[:] = 0.0
    x[:, ::3] = 0.0
    got = raw_vjp(x, W, b, "relu", scale, dphi)
    want = gof.features_vjp(x, W, b, "relu", scale, dphi)
    check(got, want, "relu at 0")
    assert np.all(got["xin"][:, ::3] == 0.0)
    keep = np.ones(90, dtype=bool)
    keep[::3] = False
    rest = gof.features_vjp(x[:, keep], W, b, "relu", scale, dphi[:, keep])
    assert rel_inf(got["b"], rest["b"]) <= RTOL and rel_inf(got["W"], rest["W"]) <= RTOL


@pytest.mark.parametrize("act,din", [("sin", 3), ("relu", 40)])
def test_padded_leading_dimensions(act, din):
    x, W, b, scale, dphi = problem(din, 70, 300, act, 5)
    got = raw_vjp(x, W, b, act, scale, dphi, pad_phi=5, pad_x=3)
    check(got, gof.features_vjp(x, W, b, act, scale, dphi), "padded")


@pytest.mark.parametrize("key", ["W", "b", "xin"])
def test_each_output_alone(key):
    x, W, b, scale, dphi = problem(33, 100, 500, "tanh", 11)
    got = raw_vjp(x, W, b, "tanh", scale, dphi, want=(key,))
    assert list(got) == [key]
    want = gof.features_vjp(x, W, b, "tanh", scale, dphi)
    check(got, {key: want[key]}, key)
    full = raw_vjp(x, W, b, "tanh", scale, dphi)
    assert np.array_equal(got[key], full[key])


def test_repeated_calls_bit_identical():
    x, W, b, scale, dphi = problem(32, 300, 5000, "cos", 2)
    a, c = raw_vjp(x, W, b, "cos", scale, dphi), raw_vjp(x, W, b, "cos", scale, dphi)
    for key in a:
        assert np.array_equal(a[key], c[key]), key


def test_launch_counts():
    ctx = blr.default_context()
    x, W, b, scale, dphi = problem(8, 96, 400, "cos", 4)
    n0 = ctx.launch_count()
    raw_vjp(x, W, b, "cos", scale, dphi, want=())
    assert ctx.launch_count() == n0  # nothing requested: nothing launched
    n0 = ctx.launch_count()
    raw_vjp(x, W, b, "cos", scale, dphi, want=("xin",))
    assert ctx.launch_count() - n0 == 1  # the dx kernel alone, no dW work
    n0 = ctx.launch_count()
    raw_vjp(x, W, b, "cos", scale, dphi, want=("W", "b"))
    assert ctx.launch_count() - n0 == 2  # the dW kernel and its fixed-order reduction
    n0 = ctx.launch_count()
    raw_vjp(x[:, :0], W, b, "cos", scale, dphi[:, :0], want=("W", "b", "xin"))
    assert ctx.launch_count() == n0  # N = 0: zeros, no kernel


def test_error_contract():
    import torch

    ctx = blr.default_context()
    din, D, N = 4, 16, 10
    x, W, b, scale, dphi = problem(din, D, N, "cos", 1)
    Wf = np.asfortranarray(W)
    dp = torch.zeros((N, D), dtype=torch.float64, device="cuda")
    dx = torch.zeros((N, din), dtype=torch.float64, device="cuda")
    xin = blr.DeviceMatrix.upload(ctx, x, L.COLVECS)
    xrow = blr.DeviceMatrix.upload(ctx, x.T.copy(), L.ROWVECS)
    xwide = blr.DeviceMatrix.upload(ctx, np.zeros((385, 2)), L.COLVECS)
    dW, db = np.empty((D, din), order="F"), np.empty(D)
    p = lambda a: None if a is None else a.ctypes.data_as(C.c_void_p)
    vp = lambda t: C.c_void_p(t.data_ptr())

    def call(xh=xin, Wp=p(Wf), bp=p(b), D_=D, act=0, dphi=vp(dp), ldp=D, ldx=din, out=True):
        return ctx.lib.blr_x_features_vjp(ctx.handle, xh.handle, Wp, bp, D_, act, scale, dphi, ldp, p(dW), p(db),
                                          vp(dx) if out else None, ldx)

    assert call() == 0
    assert call(xh=xrow) == L.E_INVALID
    assert call(xh=xwide) == L.E_INVALID
    assert call(act=5) == L.E_INVALID and call(act=-1) == L.E_INVALID
    assert call(Wp=None) == L.E_INVALID and call(bp=None) == L.E_INVALID and call(dphi=None) == L.E_INVALID
    assert call(D_=0) == L.E_INVALID
    assert call(ldp=D - 1) == L.E_INVALID
    assert call(ldx=din - 1) == L.E_INVALID
    assert call(ldx=0, out=False) == 0  # ld_dxin is only checked when dxin is requested
    ϕ = blr.AffineFeatures(W, b, "cos", scale)
    with pytest.raises(blr.BLRError):
        ϕ.vjp(blr.ColVecs(x), dphi, wrt=("W", "nope"))
    tf = blr.TorchFeatureMap(lambda t: torch.cos(t @ torch.from_numpy(W.T.copy()).cuda()))
    f = blr.BayesianLinearRegressor(np.zeros(D), blr.Diagonal(np.ones(D)))
    with pytest.raises(blr.BLRError, match="torch autograd"):
        blr.logpdf_and_grad(blr.BasisFunctionRegressor(f, tf)(blr.ColVecs(x), 0.5), np.zeros(N), wrt=("W",))
    with pytest.raises(blr.BLRError, match="torch autograd"):
        blr.logpdf_and_grad(f(blr.ColVecs(np.zeros((D, N))), 0.5), np.zeros(N), wrt=("xin",))


def test_methods_on_both_maps():
    import torch

    x, W, b, scale, dphi = problem(6, 50, 200, "cos", 8)
    want = gof.features_vjp(x, W, b, "cos", math.sqrt(2.0 / 50), dphi)
    for ϕ in (blr.RandomFourierFeatures(W, b), blr.AffineFeatures(W, b, "cos", math.sqrt(2.0 / 50))):
        check(ϕ.vjp(blr.ColVecs(x), dphi), want, type(ϕ).__name__)
        xt = torch.from_numpy(x.T.copy()).cuda()
        g = ϕ.vjp(blr.ColVecs(xt), torch.from_numpy(dphi.T.copy()).cuda())
        assert isinstance(g["xin"], torch.Tensor) and g["xin"].shape == (200, 6)
        check({"W": g["W"], "b": g["b"], "xin": g["xin"].cpu().numpy().T}, want, type(ϕ).__name__ + " torch")


def regression_problem(mapname, act, seed, k=None):
    rng = np.random.default_rng(seed)
    din, D, N = 5, 80, 700
    x = rng.standard_normal((din, N))
    W = rng.standard_normal((D, din)) / math.sqrt(din)
    b = rng.uniform(0.0, 2.0 * math.pi, D)
    scale = math.sqrt(2.0 / D) if mapname == "rff" else 0.8
    ϕ = blr.RandomFourierFeatures(W, b) if mapname == "rff" else blr.AffineFeatures(W, b, act, scale)
    mw, lam = 0.1 * rng.standard_normal(D), np.exp(rng.standard_normal(D))
    σ2 = np.exp(0.3 * rng.standard_normal(N))
    Phi = gof.features(x, W, b, "cos" if mapname == "rff" else act, scale)
    shape = (N,) if k is None else (N, k)
    y = Phi.T @ rng.standard_normal((D,) + shape[1:]) + 0.5 * rng.standard_normal(shape)
    return x, W, b, scale, ϕ, mw, lam, σ2, Phi, y


@pytest.mark.parametrize("mapname,act", [("rff", "cos"), ("affine", "tanh"), ("affine", "relu")])
def test_logpdf_and_grad_through_feature_maps(mapname, act):
    x, W, b, scale, ϕ, mw, lam, σ2, Phi, y = regression_problem(mapname, act, 3)
    fx = blr.BasisFunctionRegressor(blr.BayesianLinearRegressor(mw, blr.Diagonal(lam)), ϕ)(blr.ColVecs(x), σ2)
    lp, g = blr.logpdf_and_grad(fx, y, wrt=("W", "b", "xin", "mw"))
    fxo = ref.BayesianLinearRegressor(mw, ref.Diagonal(lam))(ref.ColVecs(Phi), σ2)
    go_ = go.logpdf_grad(fxo, y)
    want = gof.features_vjp(x, W, b, "cos" if mapname == "rff" else act, scale, go_["X"])
    assert set(g) == {"W", "b", "xin", "mw"}
    check({k: g[k] for k in ("W", "b", "xin")}, want, mapname)
    assert rel_inf(g["mw"], go_["mw"]) <= RTOL
    assert abs(lp - ref.logpdf(fxo, y)) <= RTOL * abs(lp)
    lp2, g2 = blr.logpdf_and_grad(fx, y, wrt=("X", "W"))
    assert rel_inf(g2["X"], go_["X"]) <= RTOL and np.array_equal(g2["W"], g["W"]) and lp2 == lp


@pytest.mark.parametrize("mapname,act", [("rff", "cos"), ("affine", "sin")])
def test_logpdf_and_grad_matrix_targets(mapname, act):
    k = 4
    x, W, b, scale, ϕ, mw, lam, σ2, Phi, Y = regression_problem(mapname, act, 5, k=k)
    c = np.array([1.0, -0.5, 0.0, 2.0])
    fx = blr.BasisFunctionRegressor(blr.BayesianLinearRegressor(mw, blr.Diagonal(lam)), ϕ)(blr.ColVecs(x), σ2)
    lps, g = blr.logpdf_and_grad(fx, Y, wrt=("W", "b", "xin"), weights=c)
    fxo = ref.BayesianLinearRegressor(mw, ref.Diagonal(lam))(ref.ColVecs(Phi), σ2)
    dPhi = gom.logpdf_multi_grad(fxo, Y, c)["X"]
    want = gof.features_vjp(x, W, b, "cos" if mapname == "rff" else act, scale, dPhi)
    check(g, want, mapname)
    assert lps.shape == (k,)


def test_torch_features_composes_with_torch_logpdf():
    import torch

    rng = np.random.default_rng(12)
    din, D, N = 7, 96, 900
    dev = "cuda"
    t = lambda a, rg=False: torch.tensor(a, dtype=torch.float64, device=dev, requires_grad=rg)
    x = t(rng.standard_normal((N, din)), True)
    W = t(rng.standard_normal((D, din)) / math.sqrt(din), True)
    b = t(rng.uniform(0, 2 * math.pi, D), True)
    y, mw, lam, σ2 = t(rng.standard_normal(N)), t(0.1 * rng.standard_normal(D)), t(np.exp(rng.standard_normal(D))), t(0.4)
    for act, scale in (("cos", math.sqrt(2.0 / D)), ("tanh", 0.9)):
        lp = blr.torch_logpdf(blr.torch_features(x, W, b, act, scale), y, mw, lam, σ2)
        gx, gW, gb = torch.autograd.grad(lp, (x, W, b))
        fn = {"cos": torch.cos, "tanh": torch.tanh}[act]
        lp_ref = blr.torch_logpdf(scale * fn(x @ W.T + b), y, mw, lam, σ2)
        rx, rW, rb = torch.autograd.grad(lp_ref, (x, W, b))
        assert abs(float(lp) - float(lp_ref)) <= RTOL * abs(float(lp_ref))
        for a, r, name in ((gx, rx, "x"), (gW, rW, "W"), (gb, rb, "b")):
            assert rel_inf(a.cpu().numpy(), r.cpu().numpy()) <= RTOL, (act, name)


def test_rff_lengthscale():
    import torch

    rng = np.random.default_rng(21)
    din, D, N = 3, 128, 4000
    X = rng.standard_normal((N, din))
    yv = np.sin(X @ np.array([1.5, -0.7, 0.4])) + 0.1 * rng.standard_normal(N)
    Ω = torch.tensor(rng.standard_normal((D, din)), device="cuda")
    b = torch.tensor(rng.uniform(0, 2 * math.pi, D), device="cuda")
    x, y = torch.tensor(X, device="cuda"), torch.tensor(yv, device="cuda")
    mw, lam, σ2 = torch.zeros(D, dtype=torch.float64, device="cuda"), torch.ones(D, dtype=torch.float64, device="cuda"), \
        torch.tensor(0.05, dtype=torch.float64, device="cuda")
    scale = math.sqrt(2.0 / D)

    def lp_of(logℓ):
        return blr.torch_logpdf(blr.torch_features(x, Ω / torch.exp(logℓ), b, "cos", scale), y, mw, lam, σ2)

    logℓ = torch.tensor(1.2, dtype=torch.float64, device="cuda", requires_grad=True)
    (g,) = torch.autograd.grad(lp_of(logℓ), logℓ)
    h = 1e-5
    with torch.no_grad():
        fd = (float(lp_of(logℓ + h)) - float(lp_of(logℓ - h))) / (2 * h)
    assert abs(float(g) - fd) <= 1e-6 * abs(fd), (float(g), fd)
    opt = torch.optim.Adam([logℓ], lr=0.1)
    start = float(lp_of(logℓ.detach()))
    for _ in range(5):
        opt.zero_grad()
        (-lp_of(logℓ)).backward()
        opt.step()
    assert float(lp_of(logℓ.detach())) > start


def test_full_size_cfg5_share():
    import torch

    din, D, N = 32, 4096, 1 << 19
    rng = np.random.default_rng(0)
    x = rng.standard_normal((din, N))
    W = rng.standard_normal((D, din)) / math.sqrt(din)
    b = rng.uniform(0, 2 * math.pi, D)
    scale = math.sqrt(2.0 / D)
    ctx = blr.default_context()
    xt = torch.tensor(x.T.copy(), device="cuda")  # (N, d_in) == d_in x N ColVecs
    g = torch.Generator(device="cuda").manual_seed(1)
    dphi = torch.randn((N, D), dtype=torch.float64, device="cuda", generator=g)  # 16 GiB
    out = blr.AffineFeatures(W, b, "cos", scale).vjp(blr.ColVecs(xt), dphi)
    Wt, bt = torch.tensor(W, device="cuda"), torch.tensor(b, device="cuda")
    dW = torch.zeros((D, din), dtype=torch.float64, device="cuda")
    db = torch.zeros(D, dtype=torch.float64, device="cuda")
    for lo in range(0, N, 1 << 15):
        xs = xt[lo:lo + (1 << 15)]
        gs = dphi[lo:lo + (1 << 15)] * scale * -torch.sin(xs @ Wt.T + bt)  # (n, D)
        dW += gs.T @ xs
        db += gs.sum(0)
    assert rel_inf(out["W"], dW.cpu().numpy()) <= RTOL
    assert rel_inf(out["b"], db.cpu().numpy()) <= RTOL
    idx = np.sort(rng.choice(N, 64, replace=False))
    ds = dphi[torch.tensor(idx, device="cuda")].cpu().numpy().T
    want = gof.features_vjp(x[:, idx], W, b, "cos", scale, ds)["xin"]
    assert rel_inf(out["xin"][torch.tensor(idx, device="cuda")].cpu().numpy().T, want) <= RTOL
    del dphi
    ctx.sync()


WORKER = textwrap.dedent(
    """
    import os, sys
    import numpy as np
    sys.path.insert(0, %(root)r)
    import torch, torch.distributed as dist
    import blr_b200 as blr
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    ctx = blr.Context(local); blr.set_default_context(ctx); ctx.init_comm_from_torch()
    sys.path.insert(0, os.path.join(%(root)r, "tests"))
    from test_gpu_features_grad import two_rank_problem
    x, W, b, dphi = two_rank_problem()
    lo, hi = blr.ShardPlan(x.shape[1], world).bounds(rank)
    g = blr.AffineFeatures(W, b, "tanh", 0.5).vjp(blr.ColVecs(x[:, lo:hi]), dphi[:, lo:hi])
    np.savez(os.path.join(%(out)r, f"rank{rank}.npz"), dW=g["W"], db=g["b"], dx=g["xin"])
    dist.barrier(); dist.destroy_process_group()
    """
)


def two_rank_problem():
    rng = np.random.default_rng(4)
    din, D, N = 9, 150, 20011
    return rng.standard_normal((din, N)), rng.standard_normal((D, din)) / 3.0, rng.standard_normal(D), rng.standard_normal((D, N))


def test_two_rank_dW_db_equal_single_rank(tmp_path):
    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    script = tmp_path / "worker.py"
    script.write_text(WORKER % {"root": ROOT, "out": str(tmp_path)})
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", str(port), str(script)]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-3000:]
    r0, r1 = np.load(tmp_path / "rank0.npz"), np.load(tmp_path / "rank1.npz")
    assert np.array_equal(r0["dW"], r1["dW"]) and np.array_equal(r0["db"], r1["db"])  # replicated
    x, W, b, dphi = two_rank_problem()
    g = blr.AffineFeatures(W, b, "tanh", 0.5).vjp(blr.ColVecs(x), dphi)
    assert rel_inf(r0["dW"], g["W"]) <= RTOL and rel_inf(r0["db"], g["b"]) <= RTOL
    assert rel_inf(np.concatenate([r0["dx"], r1["dx"]], axis=1), g["xin"]) <= RTOL
