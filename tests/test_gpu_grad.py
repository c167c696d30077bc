"""GPU: gradients of logpdf (blr_logpdf_grad, csrc/grad.cu; logpdf_and_grad / torch_logpdf in the package) against the closed
forms of tests/grad_oracle.py, ‖g_dev - g_ref‖∞ / ‖g_ref‖∞ <= 1e-9 for every output, over every Gram regime (tiny, small fused,
K1s, K1m, staged odd D, TMA with ragged rows, the grad_x fast path with several row passes, D = 1024), both layouts, zero and
non-zero prior mean, scalar and vector noise, Diagonal / dense / PDMat priors and the whitened form.  Also: the value is
bit-identical to logpdf, repeated calls are bit-identical, the observation pass and grad_x only run when asked for, the error
contract, torch autograd integration (down to an MLP feature map), one full-size shape, and two ranks."""
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

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
RTOL = 1e-9
LOG2PI = math.log(2.0 * math.pi)


def rel_inf(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return float(np.max(np.abs(a - b)) / np.max(np.abs(b)))


def problem(D, N, seed, prior, noise, zero_mean, layout):
    """-> (product fx, oracle fx, y)"""
    rng = np.random.default_rng(seed)
    X = rng.standard_normal((D, N))
    y = X.T @ rng.standard_normal(D) / math.sqrt(D) + 0.5 * rng.standard_normal(N)
    mw = np.zeros(D) if zero_mean else rng.standard_normal(D) / math.sqrt(D)
    B = rng.standard_normal((D, D)) / math.sqrt(D)
    Λd = B @ B.T + np.eye(D)
    lam = np.exp(rng.standard_normal(D))
    σ2 = 0.7 if noise == "scalar" else np.exp(0.5 * rng.standard_normal(N))
    if prior == "diag":
        Λ, Λo = blr.Diagonal(lam), ref.Diagonal(lam)
    elif prior == "dense":
        Λ, Λo = Λd, Λd
    else:
        po = ref.PDMat.from_matrix(Λd)
        Λ, Λo = blr.PDMat(po.mat, po.U), po
    if layout == "col":
        x, xo = blr.ColVecs(X), ref.ColVecs(X)
    else:
        Xr = np.ascontiguousarray(X.T)
        x, xo = blr.RowVecs(Xr), ref.RowVecs(Xr)
    return blr.BayesianLinearRegressor(mw, Λ)(x, σ2), ref.BayesianLinearRegressor(mw, Λo)(xo, σ2), y


def check_all(got, want, tag):
    for k in want:
        assert np.shape(got[k]) == np.shape(want[k]), (tag, k)
        err = rel_inf(got[k], want[k])
        print(f"[grad] {tag} {k}: {err:.1e}")
        assert err <= RTOL, (tag, k, err)


CASES = [
    # D, N, layout, prior, noise, zero_mean
    (2, 301, "col", "dense", "vector", False),      # tiny Gram
    (12, 517, "row", "diag", "scalar", False),      # small fused Gram
    (40, 1003, "col", "pdmat", "vector", True),     # K1s
    (66, 999, "col", "diag", "vector", False),      # K1m
    (96, 1031, "row", "dense", "scalar", False),    # K1m (staged RowVecs)
    (127, 1100, "col", "dense", "vector", False),   # staged odd D; generic grad_x (odd leading dimension)
    (130, 1500, "col", "diag", "vector", False),    # TMA Gram, ragged rows; grad_x fast path, one pass
    (600, 2000, "col", "dense", "vector", False),   # grad_x fast path, three 256-row passes, ragged last one
    (600, 1200, "row", "diag", "vector", True),     # RowVecs: generic grad_x
    (1024, 3001, "col", "pdmat", "scalar", False),  # four passes
]


@pytest.mark.parametrize("D,N,layout,prior,noise,zero_mean", CASES)
def test_gradients_match_oracle(D, N, layout, prior, noise, zero_mean):
    fx, fo, y = problem(D, N, D + N, prior, noise, zero_mean, layout)
    lp, g = blr.logpdf_and_grad(fx, y)
    # bit-identical to logpdf on the same device-resident inputs (host inputs would take logpdf's streaming path)
    assert lp == blr.logpdf(fx, blr.DeviceVector.upload(blr.default_context(), y))
    check_all(g, go.logpdf_grad(fo, y), f"D={D} N={N} {layout} {prior} {noise} mw0={zero_mean}")


def test_whitened_form():
    ctx = blr.default_context()
    fx, fo, y = problem(130, 1500, 5, "dense", "vector", False, "col")
    ctx.set_form("whitened")
    try:
        lp, g = blr.logpdf_and_grad(fx, y)
        assert lp == blr.logpdf(fx, blr.DeviceVector.upload(ctx, y))
    finally:
        ctx.set_form("direct")
    check_all(g, go.logpdf_grad(fo, y), "whitened")


def test_repeated_calls_bit_identical_and_subsets():
    fx, fo, y = problem(256, 4099, 9, "dense", "scalar", False, "col")
    lp1, g1 = blr.logpdf_and_grad(fx, y)
    lp2, g2 = blr.logpdf_and_grad(fx, y)
    assert lp1 == lp2
    for k in g1:
        assert np.array_equal(np.asarray(g1[k]), np.asarray(g2[k])), k
    _, gs = blr.logpdf_and_grad(fx, y, wrt=("mw", "σ²"))
    assert sorted(gs) == ["mw", "σ²"]
    assert np.array_equal(gs["mw"], g1["mw"]) and gs["σ²"] == g1["σ²"]


def test_torch_inputs_get_torch_outputs():
    import torch

    fx, fo, y = problem(256, 2048, 4, "diag", "vector", False, "col")
    Xt = torch.tensor(fx.x.X.T, device="cuda").contiguous()
    yt = torch.tensor(y, device="cuda")
    st = torch.tensor(fx.Σy, device="cuda")
    _, g = blr.logpdf_and_grad(fx.f(blr.ColVecs(Xt), st), yt)
    assert all(isinstance(g[k], torch.Tensor) and g[k].is_cuda for k in ("X", "y", "σ²"))
    assert tuple(g["X"].shape) == (2048, 256)
    want = go.logpdf_grad(fo, y)
    assert rel_inf(g["X"].cpu().numpy().T, want["X"]) <= RTOL
    assert rel_inf(g["y"].cpu().numpy(), want["y"]) <= RTOL
    assert rel_inf(g["σ²"].cpu().numpy(), want["σ²"]) <= RTOL


def test_prior_only_request_skips_the_observation_pass_and_grad_x():
    ctx = blr.default_context()
    fx, _, y = problem(130, 1500, 8, "diag", "vector", False, "col")
    fx = fx.f(blr.ColVecs(blr.DeviceMatrix.upload(ctx, fx.x.X, L.COLVECS)), blr.DeviceVector.upload(ctx, fx.Σy))
    y = blr.DeviceVector.upload(ctx, y)

    def launches(fn):
        n0 = ctx.launch_count()
        fn()
        return ctx.launch_count() - n0

    n_lp = launches(lambda: blr.logpdf(fx, y))
    n_mw = launches(lambda: blr.logpdf_and_grad(fx, y, wrt=("mw",)))
    n_prior = launches(lambda: blr.logpdf_and_grad(fx, y, wrt=("mw", "Λw")))
    n_obs = launches(lambda: blr.logpdf_and_grad(fx, y, wrt=("mw", "Λw", "y")))
    n_all = launches(lambda: blr.logpdf_and_grad(fx, y))
    print(f"[grad] launches: logpdf {n_lp}, mw {n_mw}, mw + Λw {n_prior}, + y {n_obs}, all {n_all}")
    assert n_mw == n_lp + 1  # Diagonal prior: one assembly kernel on top of logpdf's launches
    assert n_prior > n_mw  # + the inverse factor for diag(Q)
    assert n_obs - n_prior >= 2  # + the predict pass and grad_obs_kernel
    assert n_all - n_obs >= 2  # + Q = W'W and grad_x


def test_errors():
    fx, _, y = problem(64, 200, 1, "diag", "vector", False, "col")
    C_dense = np.eye(200) + 0.01
    with pytest.raises(blr.BLRError):
        blr.logpdf_and_grad(fx.f(fx.x, C_dense), y)
    σ2 = np.array(fx.Σy, copy=True)
    σ2[5] = -1.0
    with pytest.raises(blr.PosDefException) as ei:
        blr.logpdf_and_grad(fx.f(fx.x, σ2), y)
    assert ei.value.info == 6  # cholesky(Diagonal(σ²)) fails at the first non-positive entry
    with pytest.raises(blr.PosDefException) as ei:
        blr.logpdf_and_grad(fx.f(fx.x, -0.5), y)
    assert ei.value.info == 1
    f_bad = blr.BayesianLinearRegressor(np.zeros(65), blr.Diagonal(np.ones(65)))
    with pytest.raises(blr.DimensionMismatch):
        blr.logpdf_and_grad(f_bad(fx.x, fx.Σy), y)
    with pytest.raises(blr.BLRError):
        blr.logpdf_and_grad(fx, y, wrt=("Σy",))
    # the C ABI itself: prior.D mismatch, short ld_dX, dsigma2 of the wrong kind
    ctx = blr.default_context()
    X = blr.DeviceMatrix.upload(ctx, fx.x.X, L.COLVECS)
    yv = blr.DeviceVector.upload(ctx, y)
    noise, keep = blr.runtime.make_noise(ctx, fx.Σy, 200)
    prior, keep_p = fx.f._prior_struct()
    dX = blr.DeviceVector.alloc(ctx, 64 * 200)
    lp = C.c_double()

    def call(g, pr=prior):
        return ctx.lib.blr_logpdf_grad(ctx.handle, C.byref(pr), X.handle, yv.handle, C.byref(noise), C.byref(lp), C.byref(g))

    assert call(L.LogpdfGrads(dX_dev=dX.device_ptr(), ld_dX=63)) == L.E_INVALID
    assert call(L.LogpdfGrads(dX_dev=dX.device_ptr(), ld_dX=64)) == 0
    s = C.c_double()
    assert call(L.LogpdfGrads(dsigma2=C.pointer(s))) == L.E_INVALID  # vector noise: dsigma2_dev, not the scalar
    pr2 = L.Prior(prior.mw, prior.lambda_kind, prior.lambda_, prior.ld, 63)
    assert call(L.LogpdfGrads(), pr2) == L.E_DIM


def torch_literal_logpdf(X, y, mw, Λ, σ2):
    """The reference's logpdf (:72-89, :55-58) as a torch graph; X is D x N."""
    import torch

    D, N = X.shape
    Uw = torch.linalg.cholesky(Λ).mT
    sd = torch.sqrt(σ2)
    Bt = torch.linalg.solve_triangular(Uw.mT, X, upper=False).T / sd[:, None]
    δy = (y - X.T @ mw) / sd
    lp_δy = -(N * LOG2PI + 2.0 * torch.sum(torch.log(sd)) + δy @ δy) / 2
    U = torch.linalg.cholesky(Bt.T @ Bt + torch.eye(D, dtype=X.dtype, device=X.device)).mT
    v = torch.linalg.solve_triangular(U.mT, (Bt.T @ δy)[:, None], upper=False)[:, 0]
    return -(2.0 * torch.sum(torch.log(torch.diagonal(U))) - v @ v) / 2 + lp_δy


@pytest.mark.parametrize("dense,scalar", [(True, False), (False, True)])
def test_torch_logpdf_matches_all_torch_graph(dense, scalar):
    import torch

    rng = np.random.default_rng(21)
    D, N = 96, 700
    dev = "cuda"
    X = torch.tensor(rng.standard_normal((N, D)), device=dev, requires_grad=True)
    y = torch.tensor(rng.standard_normal(N), device=dev, requires_grad=True)
    mw = torch.tensor(rng.standard_normal(D) * 0.1, device=dev, requires_grad=True)
    B = rng.standard_normal((D, D)) / math.sqrt(D)
    lam0 = B @ B.T + np.eye(D) if dense else np.exp(rng.standard_normal(D))
    lam = torch.tensor(lam0, device=dev, requires_grad=True)
    s2 = torch.tensor(0.8 if scalar else np.exp(0.5 * rng.standard_normal(N)), device=dev, requires_grad=True)

    lp = blr.torch_logpdf(X, y, mw, lam, s2)
    (2.5 * lp).backward()
    got = [t.grad.clone() for t in (X, y, mw, lam, s2)]
    for t in (X, y, mw, lam, s2):
        t.grad = None
    Λ = (lam + lam.T) / 2 if dense else torch.diag(lam)
    σ2v = s2 * torch.ones(N, dtype=torch.float64, device=dev) if scalar else s2
    lp_ref = torch_literal_logpdf(X.T, y, mw, Λ, σ2v)
    (2.5 * lp_ref).backward()
    assert abs(lp.item() - lp_ref.item()) <= RTOL * abs(lp_ref.item())
    for name, a, t in zip(("X", "y", "mw", "Λw", "σ²"), got, (X, y, mw, lam, s2)):
        err = rel_inf(a.cpu().numpy(), t.grad.cpu().numpy())
        print(f"[torch_logpdf] dense={dense} scalar={scalar} {name}: {err:.1e}")
        assert err <= RTOL, name


def test_mlp_feature_map_end_to_end():
    """examples/nn-blr.jl: an MLP's last-layer features, a BLR on top, type-II maximum likelihood -- the MLP's parameter
    gradients through TorchFeatureMap and torch_logpdf equal the all-torch graph."""
    import torch

    torch.manual_seed(0)
    rng = np.random.default_rng(2)
    d_in, D, N = 3, 80, 1500
    mlp = torch.nn.Sequential(torch.nn.Linear(d_in, 64), torch.nn.Tanh(), torch.nn.Linear(64, D), torch.nn.Tanh()).double().cuda()
    xin = torch.tensor(rng.standard_normal((N, d_in)), device="cuda")
    y = torch.tensor(np.sin(rng.standard_normal(N)), device="cuda")
    mw = torch.zeros(D, dtype=torch.float64, device="cuda")
    lam = torch.ones(D, dtype=torch.float64, device="cuda")
    s2 = torch.tensor(0.1, dtype=torch.float64, device="cuda")

    phi = blr.TorchFeatureMap(mlp)
    Xf = phi(blr.ColVecs(xin)).X
    lp = blr.torch_logpdf(Xf, y, mw, lam, s2)
    lp.backward()
    got = [p.grad.clone() for p in mlp.parameters()]
    mlp.zero_grad()
    lp_ref = torch_literal_logpdf(mlp(xin).T, y, mw, torch.diag(lam), s2 * torch.ones(N, dtype=torch.float64, device="cuda"))
    lp_ref.backward()
    assert abs(lp.item() - lp_ref.item()) <= RTOL * abs(lp_ref.item())
    for a, p in zip(got, mlp.parameters()):
        assert rel_inf(a.cpu().numpy(), p.grad.cpu().numpy()) <= RTOL


def test_full_size_sampled_columns():
    """D = 1024, N = 2^20 on the grad_x fast path: 64 sampled columns of dX against the closed form evaluated from the
    downloaded posterior precision."""
    import torch

    ctx = blr.default_context()
    D, N = 1024, 1 << 20
    X = blr.DeviceMatrix.alloc(ctx, D, N).synth_(7)
    s2 = blr.DeviceVector.alloc(ctx, N)
    ctx.check(ctx.lib.blr_vec_synth_noise(ctx.handle, s2.handle, 7, 0))
    y = blr.DeviceVector.alloc(ctx, N)
    ctx.check(ctx.lib.blr_vec_synth_targets(ctx.handle, X.handle, s2.handle, 7, 0, y.handle))
    rng = np.random.default_rng(1)
    mw = rng.standard_normal(D) * 0.1
    lam = np.exp(rng.standard_normal(D))
    f = blr.BayesianLinearRegressor(mw, blr.Diagonal(lam))
    fx = f(blr.ColVecs(X), s2)
    post, lp0 = blr.posterior_and_logpdf(fx, y)
    Xt = X.as_torch()  # (N, D) view
    lp, g = blr.logpdf_and_grad(blr.FiniteGP(f, blr.ColVecs(Xt), s2), y, wrt=("X", "σ²"))
    assert lp == lp0
    cols = np.sort(rng.choice(N, 64, replace=False))
    cols[-1] = N - 1  # the last, partial point tile
    idx = torch.tensor(cols, device="cuda")
    Xs = Xt[idx].cpu().numpy().T  # D x 64
    ys, ss = y.download()[cols], s2.download()[cols]
    P = post.Λw.dense()
    Q = np.linalg.inv(P)
    mp = post.mw
    e = ys - Xs.T @ mp
    want = np.outer(mp, e / ss) - (Q @ Xs) / ss
    got = g["X"][idx].cpu().numpy().T
    err = rel_inf(got, want)
    print(f"[grad] full size: dX sampled columns {err:.1e}")
    assert err <= RTOL
    h = np.sum(Xs * (Q @ Xs), axis=0)
    want_s = 0.5 * ((h + e * e) / ss**2 - 1.0 / ss)
    assert rel_inf(g["σ²"][idx].cpu().numpy(), want_s) <= RTOL


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
    from test_gpu_grad import two_rank_problem
    X, y, s2, mw, Lam = two_rank_problem()
    lo, hi = blr.ShardPlan(X.shape[1], world).bounds(rank)
    f = blr.BayesianLinearRegressor(mw, Lam)
    lp, g = blr.logpdf_and_grad(f(blr.ColVecs(X[:, lo:hi]), s2[lo:hi]), y[lo:hi])
    lp_s, gs = blr.logpdf_and_grad(f(blr.ColVecs(X[:, lo:hi]), 0.9), y[lo:hi], wrt=("σ²", "mw"))
    np.savez(os.path.join(%(out)r, f"rank{rank}.npz"), lp=lp, dX=g["X"], dy=g["y"], ds=g["σ²"], dmw=g["mw"], dlam=g["Λw"],
             lp_s=lp_s, ds_s=gs["σ²"], dmw_s=gs["mw"])
    dist.barrier(); dist.destroy_process_group()
    """
)


def two_rank_problem():
    rng = np.random.default_rng(3)
    D, N = 192, 20011
    X = rng.standard_normal((D, N))
    s2 = np.exp(rng.standard_normal(N))
    mw = rng.standard_normal(D) * 0.1
    B = rng.standard_normal((D, D)) / math.sqrt(D)
    Lam = B @ B.T + np.eye(D)
    y = X.T @ rng.standard_normal(D) / math.sqrt(D) + np.sqrt(s2) * rng.standard_normal(N)
    return X, y, s2, mw, Lam


def test_two_rank_sharded_gradients(tmp_path):
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
    for k in ("lp", "dmw", "dlam", "lp_s", "ds_s", "dmw_s"):  # replicated: bit-identical on every rank
        assert np.array_equal(r0[k], r1[k]), k
    X, y, s2, mw, Lam = two_rank_problem()
    f = blr.BayesianLinearRegressor(mw, Lam)
    lp, g = blr.logpdf_and_grad(f(blr.ColVecs(X), s2), y)
    assert abs(float(r0["lp"]) - lp) <= RTOL * abs(lp)
    for k, key in (("dX", "X"), ("dy", "y"), ("ds", "σ²")):
        cat = np.concatenate([r0[k], r1[k]], axis=-1)
        assert rel_inf(cat, g[key]) <= RTOL, k
    assert rel_inf(r0["dmw"], g["mw"]) <= RTOL and rel_inf(r0["dlam"], g["Λw"]) <= RTOL
    lp_s, gs = blr.logpdf_and_grad(f(blr.ColVecs(X), 0.9), y, wrt=("σ²", "mw"))
    assert abs(float(r0["ds_s"]) - gs["σ²"]) <= RTOL * abs(gs["σ²"])
    assert rel_inf(r0["dmw_s"], gs["mw"]) <= RTOL
