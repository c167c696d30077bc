"""GPU: gradients of Σ_j c_j logpdf(fx, Y[:, j]) (blr_logpdf_multi_grad, csrc/grad.cu; logpdf_and_grad / torch_logpdf with an
(N, k) Y in the package) against the closed forms of tests/grad_oracle_multi.py, ‖g_dev - g_ref‖∞ / ‖g_ref‖∞ <= 1e-9 for every output,
over the Gram regimes of test_gpu_grad.CASES, k from 1 to 33 (one, several and a ragged last 16-column block of E), weights with
zeros, negatives and c̄ = 0, and the whitened form.  Also: the k values are bit-identical to blr_logpdf_multi, the gradients equal
Σ_j c_j blr_logpdf_grad(column j), repeated calls are bit-identical, the fast and generic ∂/∂X paths agree, a prior-only request
runs no extra pass over the observations, the error contract, torch autograd integration, one full-size shape and two ranks."""
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
from tests import grad_oracle_multi as gom
from tests.test_gpu_grad import CASES, RTOL, problem, rel_inf, torch_literal_logpdf

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KS = (1, 2, 9, 17, 33)


def targets(fx, k, seed):
    X = np.asarray(fx.x.X) if isinstance(fx.x, blr.ColVecs) else np.asarray(fx.x.X).T
    D, N = X.shape
    rng = np.random.default_rng(seed)
    return X.T @ rng.standard_normal((D, k)) / math.sqrt(D) + 0.5 * rng.standard_normal((N, k))


def weights(k, seed):
    """negatives, zeros (k > 2) and c̄ = 0 (k = 2 and k = 17)"""
    if k == 1:
        return np.array([-1.3])
    if k == 2:
        return np.array([0.8, -0.8])
    c = np.random.default_rng(seed).standard_normal(k)
    c[0] = 0.0
    if k == 17:
        c[-1] = -np.sum(c[:-1])
    return c


def check_all(got, want, tag):
    for key in want:
        assert np.shape(got[key]) == np.shape(want[key]), (tag, key)
        err = rel_inf(got[key], want[key])
        print(f"[grad_multi] {tag} {key}: {err:.1e}")
        assert err <= RTOL, (tag, key, err)


@pytest.mark.parametrize("k", KS)
@pytest.mark.parametrize("D,N,layout,prior,noise,zero_mean", CASES)
def test_gradients_match_oracle(D, N, layout, prior, noise, zero_mean, k):
    fx, fo, _ = problem(D, N, D + N, prior, noise, zero_mean, layout)
    Y = targets(fx, k, D + k)
    c = weights(k, N + k)
    lps, g = blr.logpdf_and_grad(fx, Y, weights=c)
    assert np.array_equal(lps, blr.logpdf(fx, Y))  # bit-identical to blr_logpdf_multi
    check_all(g, gom.logpdf_multi_grad(fo, Y, c), f"D={D} N={N} {layout} {prior} {noise} mw0={zero_mean} k={k}")


def test_whitened_form():
    ctx = blr.default_context()
    fx, fo, _ = problem(130, 1500, 5, "dense", "vector", False, "col")
    Y = targets(fx, 9, 1)
    c = weights(9, 2)
    ctx.set_form("whitened")
    try:
        lps, g = blr.logpdf_and_grad(fx, Y, weights=c)
        assert np.array_equal(lps, blr.logpdf(fx, Y))
    finally:
        ctx.set_form("direct")
    check_all(g, gom.logpdf_multi_grad(fo, Y, c), "whitened")


@pytest.mark.parametrize("D,N,layout,prior,noise", [(256, 4099, "col", "dense", "scalar"), (96, 1031, "row", "diag", "vector")])
def test_equals_weighted_sum_of_single_column_calls(D, N, layout, prior, noise):
    fx, _, _ = problem(D, N, 17, prior, noise, False, layout)
    Y = targets(fx, 9, 4)
    c = weights(9, 5)
    lps, g = blr.logpdf_and_grad(fx, Y, weights=c)
    acc = {}
    ctx = blr.default_context()
    for j in range(9):
        lp_j, g_j = blr.logpdf_and_grad(fx, blr.DeviceVector.upload(ctx, np.ascontiguousarray(Y[:, j])))
        assert abs(lp_j - lps[j]) <= 1e-12 * abs(lp_j)
        for key, v in g_j.items():
            v = np.asarray(v)
            acc[key] = acc.get(key, 0.0) + c[j] * v if key != "y" else acc.get(key, []) + [c[j] * v]
    acc["y"] = np.stack(acc["y"], axis=1)
    for key in acc:
        err = rel_inf(g[key], acc[key])
        print(f"[grad_multi] Σ_j c_j single-column {key}: {err:.1e}")
        assert err <= 1e-11, key


def test_repeated_calls_bit_identical_and_subsets():
    fx, _, _ = problem(256, 4099, 9, "dense", "scalar", False, "col")
    Y = targets(fx, 17, 3)
    c = weights(17, 4)
    lp1, g1 = blr.logpdf_and_grad(fx, Y, weights=c)
    lp2, g2 = blr.logpdf_and_grad(fx, Y, weights=c)
    assert np.array_equal(lp1, lp2)
    for key in g1:
        assert np.array_equal(np.asarray(g1[key]), np.asarray(g2[key])), key
    _, gs = blr.logpdf_and_grad(fx, Y, wrt=("mw", "σ²"), weights=c)
    assert sorted(gs) == ["mw", "σ²"]
    assert np.array_equal(gs["mw"], g1["mw"]) and gs["σ²"] == g1["σ²"]
    _, g_ones = blr.logpdf_and_grad(fx, Y)
    _, g_ones2 = blr.logpdf_and_grad(fx, Y, weights=np.ones(17))
    for key in g_ones:
        assert np.array_equal(np.asarray(g_ones[key]), np.asarray(g_ones2[key])), key


@pytest.mark.parametrize("k", (1, 9, 33))
def test_fast_and_generic_dx_paths_agree(k):
    """The same data through the tensor-map kernel (aligned base) and through gemm_generic (base offset by one double)."""
    import torch

    D, N = 256, 3001
    fx, _, _ = problem(D, N, 31, "diag", "vector", False, "col")
    Y = targets(fx, k, 6)
    c = weights(k, 7)
    Xh = np.ascontiguousarray(fx.x.X.T)  # (N, D) row-major == ColVecs D x N
    aligned = torch.tensor(Xh, device="cuda")
    store = torch.empty(N * D + 1, dtype=torch.float64, device="cuda")
    offset = store[1:].view(N, D)
    offset.copy_(aligned)
    assert offset.data_ptr() % 16 == 8
    gs = []
    for Xt in (aligned, offset):
        _, g = blr.logpdf_and_grad(fx.f(blr.ColVecs(Xt), fx.Σy), Y, wrt=("X",), weights=c)
        gs.append(g["X"].cpu().numpy())
    err = rel_inf(gs[1], gs[0])
    print(f"[grad_multi] k={k} fast vs generic dX: {err:.1e}")
    assert err <= 1e-12


def test_prior_only_request_runs_no_pass_over_the_observations():
    ctx = blr.default_context()

    def launches(fn):
        n0 = ctx.launch_count()
        fn()
        return ctx.launch_count() - n0

    extra = []
    for N in (1500, 6000):
        fx, _, _ = problem(130, N, 8, "diag", "vector", False, "col")
        Y = blr.DeviceVector.upload(ctx, targets(fx, 9, 1).T.reshape(-1))
        fx = fx.f(blr.ColVecs(blr.DeviceMatrix.upload(ctx, fx.x.X, L.COLVECS)), blr.DeviceVector.upload(ctx, fx.Σy))
        X = fx.x.X
        noise, keep = blr.runtime.make_noise(ctx, fx.Σy, N)
        prior, keep_p = fx.f._prior_struct()
        out = np.empty(9)
        dmw, dlam = np.empty(130), np.empty(130)

        def multi():
            ctx.check(ctx.lib.blr_logpdf_multi(ctx.handle, C.byref(prior), X.handle, C.c_void_p(Y.device_ptr()), N, 9,
                                               C.byref(noise), out.ctypes.data_as(C.c_void_p)))

        def prior_only():
            g = L.LogpdfGrads(dmw=dmw.ctypes.data_as(L.c_double_p), dlambda=dlam.ctypes.data_as(L.c_double_p))
            ctx.check(ctx.lib.blr_logpdf_multi_grad(ctx.handle, C.byref(prior), X.handle, C.c_void_p(Y.device_ptr()), N, 9,
                                                    C.byref(noise), None, out.ctypes.data_as(L.c_double_p), C.byref(g)))

        n_lp, n_prior = launches(multi), launches(prior_only)
        print(f"[grad_multi] N={N}: logpdf_multi {n_lp} launches, + dmw, dΛw {n_prior}")
        extra.append(n_prior - n_lp)
    assert extra[0] == extra[1] and extra[0] > 0


def test_zero_columns_write_zeros():
    ctx = blr.default_context()
    fx, _, _ = problem(64, 200, 1, "dense", "scalar", False, "col")
    X = blr.DeviceMatrix.upload(ctx, fx.x.X, L.COLVECS)
    noise, keep = blr.runtime.make_noise(ctx, fx.Σy, 200)
    prior, keep_p = fx.f._prior_struct()
    dX = blr.DeviceVector.upload(ctx, np.full(64 * 200, 7.0))
    dmw, dlam, ds = np.full(64, 7.0), np.full((64, 64), 7.0), C.c_double(7.0)
    g = L.LogpdfGrads(dmw=dmw.ctypes.data_as(L.c_double_p), dlambda=dlam.ctypes.data_as(L.c_double_p), dsigma2=C.pointer(ds),
                      dX_dev=dX.device_ptr(), ld_dX=64)
    assert ctx.lib.blr_logpdf_multi_grad(ctx.handle, C.byref(prior), X.handle, None, 200, 0, C.byref(noise), None, None,
                                         C.byref(g)) == 0
    assert not dmw.any() and not dlam.any() and ds.value == 0.0 and not dX.download().any()


def test_errors():
    fx, _, _ = problem(64, 200, 1, "diag", "vector", False, "col")
    Y = targets(fx, 3, 1)
    with pytest.raises(blr.BLRError):
        blr.logpdf_and_grad(fx.f(fx.x, np.eye(200) + 0.01), Y)  # dense Σy
    σ2 = np.array(fx.Σy, copy=True)
    σ2[5] = -1.0
    with pytest.raises(blr.PosDefException) as ei:
        blr.logpdf_and_grad(fx.f(fx.x, σ2), Y)
    assert ei.value.info == 6  # cholesky(Diagonal(σ²)) fails at the first non-positive entry
    with pytest.raises(blr.PosDefException) as ei:
        blr.logpdf_and_grad(fx.f(fx.x, -0.5), Y)
    assert ei.value.info == 1
    f_bad = blr.BayesianLinearRegressor(np.zeros(65), blr.Diagonal(np.ones(65)))
    with pytest.raises(blr.DimensionMismatch):
        blr.logpdf_and_grad(f_bad(fx.x, fx.Σy), Y)
    with pytest.raises(blr.DimensionMismatch):
        blr.logpdf_and_grad(fx, Y[:150])
    with pytest.raises(blr.DimensionMismatch):
        blr.logpdf_and_grad(fx, Y, weights=np.ones(2))
    with pytest.raises(blr.BLRError):
        blr.logpdf_and_grad(fx, Y, wrt=("Σy",))
    # the C ABI itself
    ctx = blr.default_context()
    X = blr.DeviceMatrix.upload(ctx, fx.x.X, L.COLVECS)
    Yd = blr.DeviceVector.upload(ctx, Y.T.reshape(-1))
    noise, keep = blr.runtime.make_noise(ctx, fx.Σy, 200)
    prior, keep_p = fx.f._prior_struct()
    dX = blr.DeviceVector.alloc(ctx, 64 * 200)
    lp = np.empty(3)

    def call(g, pr=prior, ldy=200, y=Yd.device_ptr(), nz=noise, x=X.handle):
        return ctx.lib.blr_logpdf_multi_grad(ctx.handle, C.byref(pr) if pr is not None else None, x, C.c_void_p(y), ldy, 3,
                                             C.byref(nz) if nz is not None else None, None, lp.ctypes.data_as(L.c_double_p),
                                             C.byref(g))

    assert call(L.LogpdfGrads(dX_dev=dX.device_ptr(), ld_dX=63)) == L.E_INVALID
    assert call(L.LogpdfGrads(dX_dev=dX.device_ptr(), ld_dX=64)) == 0
    s = C.c_double()
    assert call(L.LogpdfGrads(dsigma2=C.pointer(s))) == L.E_INVALID  # vector noise: dsigma2_dev, not the scalar
    assert call(L.LogpdfGrads(), ldy=199) == L.E_DIM
    assert call(L.LogpdfGrads(), pr=L.Prior(prior.mw, prior.lambda_kind, prior.lambda_, prior.ld, 63)) == L.E_DIM
    assert call(L.LogpdfGrads(), y=None) == L.E_INVALID
    assert call(L.LogpdfGrads(), nz=None) == L.E_INVALID
    assert call(L.LogpdfGrads(), pr=None) == L.E_INVALID
    noise_s, keep_s = blr.runtime.make_noise(ctx, 0.5, 200)
    dsd = blr.DeviceVector.alloc(ctx, 200)
    assert call(L.LogpdfGrads(dsigma2_dev=dsd.device_ptr()), nz=noise_s) == L.E_INVALID  # scalar noise: dsigma2, not the vector


def test_torch_gradcheck():
    import torch

    rng = np.random.default_rng(0)
    D, N, k = 3, 11, 2
    t = lambda a: torch.tensor(a, device="cuda", requires_grad=True)
    X = t(rng.standard_normal((N, D)))
    Y = t(rng.standard_normal((N, k)))
    mw = t(rng.standard_normal(D) * 0.1)
    lam = t(np.exp(rng.standard_normal(D)))
    s2 = t(np.exp(0.3 * rng.standard_normal(N)))
    assert torch.autograd.gradcheck(blr.torch_logpdf, (X, Y, mw, lam, s2), eps=1e-6, atol=1e-7, rtol=1e-6)


@pytest.mark.parametrize("dense,scalar", [(True, False), (False, True)])
def test_torch_logpdf_matches_all_torch_graph(dense, scalar):
    """A loss non-linear in the k values, so that the cotangent differs from column to column."""
    import torch

    rng = np.random.default_rng(21)
    D, N, k = 96, 700, 5
    dev = "cuda"
    X = torch.tensor(rng.standard_normal((N, D)), device=dev, requires_grad=True)
    Y = torch.tensor(rng.standard_normal((N, k)), device=dev, requires_grad=True)
    mw = torch.tensor(rng.standard_normal(D) * 0.1, device=dev, requires_grad=True)
    B = rng.standard_normal((D, D)) / math.sqrt(D)
    lam0 = B @ B.T + np.eye(D) if dense else np.exp(rng.standard_normal(D))
    lam = torch.tensor(lam0, device=dev, requires_grad=True)
    s2 = torch.tensor(0.8 if scalar else np.exp(0.5 * rng.standard_normal(N)), device=dev, requires_grad=True)
    wts = torch.linspace(-1.0, 2.0, k, dtype=torch.float64, device=dev)

    def loss(lps):
        return torch.sum(wts * lps) + 1e-3 * torch.sum(lps**2)

    lps = blr.torch_logpdf(X, Y, mw, lam, s2)
    assert tuple(lps.shape) == (k,)
    loss(lps).backward()
    got = [t.grad.clone() for t in (X, Y, mw, lam, s2)]
    for t in (X, Y, mw, lam, s2):
        t.grad = None
    Λ = (lam + lam.T) / 2 if dense else torch.diag(lam)
    σ2v = s2 * torch.ones(N, dtype=torch.float64, device=dev) if scalar else s2
    lps_ref = torch.stack([torch_literal_logpdf(X.T, Y[:, j], mw, Λ, σ2v) for j in range(k)])
    loss(lps_ref).backward()
    assert rel_inf(lps.detach().cpu().numpy(), lps_ref.detach().cpu().numpy()) <= RTOL
    for name, a, t in zip(("X", "Y", "mw", "Λw", "σ²"), got, (X, Y, mw, lam, s2)):
        err = rel_inf(a.cpu().numpy(), t.grad.cpu().numpy())
        print(f"[torch_logpdf multi] dense={dense} scalar={scalar} {name}: {err:.1e}")
        assert err <= RTOL, name


def test_mlp_feature_map_with_k_outputs_trains():
    """examples/nn-blr.jl with vector outputs: an MLP feature map shared by k target series, a few Adam steps on -Σ_j ℓ_j through
    torch_logpdf with an (N, k) Y raise the summed log marginal likelihood; the first step's parameter gradients equal the
    all-torch graph's."""
    import torch

    torch.manual_seed(0)
    rng = np.random.default_rng(2)
    d_in, D, N, k = 3, 80, 1500, 4
    mlp = torch.nn.Sequential(torch.nn.Linear(d_in, 64), torch.nn.Tanh(), torch.nn.Linear(64, D), torch.nn.Tanh()).double().cuda()
    xin = torch.tensor(rng.standard_normal((N, d_in)), device="cuda")
    Y = torch.tensor(np.sin(rng.standard_normal((N, k)) + rng.standard_normal(k)), device="cuda")
    mw = torch.zeros(D, dtype=torch.float64, device="cuda")
    lam = torch.ones(D, dtype=torch.float64, device="cuda")
    s2 = torch.tensor(0.1, dtype=torch.float64, device="cuda")
    phi = blr.TorchFeatureMap(mlp)

    lp = blr.torch_logpdf(phi(blr.ColVecs(xin)).X, Y, mw, lam, s2).sum()
    lp.backward()
    got = [p.grad.clone() for p in mlp.parameters()]
    mlp.zero_grad()
    σ2v = s2 * torch.ones(N, dtype=torch.float64, device="cuda")
    lp_ref = sum(torch_literal_logpdf(mlp(xin).T, Y[:, j], mw, torch.diag(lam), σ2v) for j in range(k))
    lp_ref.backward()
    assert abs(lp.item() - lp_ref.item()) <= RTOL * abs(lp_ref.item())
    for a, p in zip(got, mlp.parameters()):
        assert rel_inf(a.cpu().numpy(), p.grad.cpu().numpy()) <= RTOL
    mlp.zero_grad()

    opt = torch.optim.Adam(mlp.parameters(), lr=1e-2)
    history = []
    for _ in range(6):
        opt.zero_grad()
        lp = blr.torch_logpdf(phi(blr.ColVecs(xin)).X, Y, mw, lam, s2).sum()
        (-lp).backward()
        opt.step()
        history.append(lp.item())
    print(f"[grad_multi] MLP Σ_j ℓ_j over Adam steps: {history}")
    assert history[-1] > history[0]


def test_full_size_sampled_columns():
    """D = 1024, N = 2^20, k = 8 on the rank-k grad_x fast path: 64 sampled points of dX and ∂/∂σ² against the closed form
    evaluated from the downloaded posterior precision."""
    import torch

    ctx = blr.default_context()
    D, N, k = 1024, 1 << 20, 8
    X = blr.DeviceMatrix.alloc(ctx, D, N).synth_(7)
    s2 = blr.DeviceVector.alloc(ctx, N)
    ctx.check(ctx.lib.blr_vec_synth_noise(ctx.handle, s2.handle, 7, 0))
    y = blr.DeviceVector.alloc(ctx, N)
    ctx.check(ctx.lib.blr_vec_synth_targets(ctx.handle, X.handle, s2.handle, 7, 0, y.handle))
    rng = np.random.default_rng(1)
    mw = rng.standard_normal(D) * 0.1
    lam = np.exp(rng.standard_normal(D))
    f = blr.BayesianLinearRegressor(mw, blr.Diagonal(lam))
    Xt = X.as_torch()  # (N, D) view
    y0 = torch.tensor(y.download(), device="cuda")
    Yt = torch.stack([y0 * (1.0 + 0.1 * j) + 0.05 * j for j in range(k)], dim=1)  # (N, k)
    c = np.linspace(-1.0, 1.5, k)
    fx = blr.FiniteGP(f, blr.ColVecs(Xt), s2)
    post, lp0 = blr.posterior_and_logpdf(fx, y)
    lps, g = blr.logpdf_and_grad(fx, Yt, wrt=("X", "σ²"), weights=c)
    assert lps[0] == lp0
    cols = np.sort(rng.choice(N, 64, replace=False))
    cols[-1] = N - 1  # the last, partial point tile
    idx = torch.tensor(cols, device="cuda")
    Xs = Xt[idx].cpu().numpy().T  # D x 64
    Ys, ss = Yt[idx].cpu().numpy(), s2.download()[cols]
    P = post.Λw.dense()
    Q = np.linalg.inv(P)
    # m'_j from the statistics: P m'_j = Λw mw + X S y_j  (X S y_j on the device, as a column of the Gram pass)
    XSY = (Xt.T @ (Yt / torch.tensor(s2.download(), device="cuda")[:, None])).cpu().numpy()
    Mp = np.linalg.solve(P, (lam * mw)[:, None] + XSY)
    E = Ys - Xs.T @ Mp  # 64 x k
    cbar = float(np.sum(c))
    want = (Mp * c) @ E.T / ss - cbar * (Q @ Xs) / ss
    got = g["X"][idx].cpu().numpy().T
    err = rel_inf(got, want)
    print(f"[grad_multi] full size k={k}: dX sampled columns {err:.1e}")
    assert err <= RTOL
    h = np.sum(Xs * (Q @ Xs), axis=0)
    want_s = 0.5 * ((cbar * h + (E * E) @ c) / ss**2 - cbar / ss)
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
    from test_gpu_grad_multi import two_rank_problem
    X, Y, s2, mw, Lam, c = two_rank_problem()
    lo, hi = blr.ShardPlan(X.shape[1], world).bounds(rank)
    f = blr.BayesianLinearRegressor(mw, Lam)
    lp, g = blr.logpdf_and_grad(f(blr.ColVecs(X[:, lo:hi]), s2[lo:hi]), Y[lo:hi], weights=c)
    lp_s, gs = blr.logpdf_and_grad(f(blr.ColVecs(X[:, lo:hi]), 0.9), Y[lo:hi], wrt=("σ²", "mw"), weights=c)
    np.savez(os.path.join(%(out)r, f"rank{rank}.npz"), lp=lp, dX=g["X"], dy=g["y"], ds=g["σ²"], dmw=g["mw"], dlam=g["Λw"],
             lp_s=lp_s, ds_s=gs["σ²"], dmw_s=gs["mw"])
    dist.barrier(); dist.destroy_process_group()
    """
)


def two_rank_problem():
    rng = np.random.default_rng(3)
    D, N, k = 192, 20011, 5
    X = rng.standard_normal((D, N))
    s2 = np.exp(rng.standard_normal(N))
    mw = rng.standard_normal(D) * 0.1
    B = rng.standard_normal((D, D)) / math.sqrt(D)
    Lam = B @ B.T + np.eye(D)
    Y = X.T @ rng.standard_normal((D, k)) / math.sqrt(D) + np.sqrt(s2)[:, None] * rng.standard_normal((N, k))
    return X, Y, s2, mw, Lam, np.array([1.0, -0.5, 0.0, 2.0, 0.3])


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
    for key in ("lp", "dmw", "dlam", "lp_s", "ds_s", "dmw_s"):  # replicated: bit-identical on every rank
        assert np.array_equal(r0[key], r1[key]), key
    X, Y, s2, mw, Lam, c = two_rank_problem()
    f = blr.BayesianLinearRegressor(mw, Lam)
    lp, g = blr.logpdf_and_grad(f(blr.ColVecs(X), s2), Y, weights=c)
    assert rel_inf(r0["lp"], lp) <= RTOL
    for key, name, axis in (("dX", "X", -1), ("dy", "y", 0), ("ds", "σ²", -1)):
        cat = np.concatenate([r0[key], r1[key]], axis=axis)
        assert rel_inf(cat, g[name]) <= RTOL, key
    assert rel_inf(r0["dmw"], g["mw"]) <= RTOL and rel_inf(r0["dlam"], g["Λw"]) <= RTOL
    lp_s, gs = blr.logpdf_and_grad(f(blr.ColVecs(X), 0.9), Y, wrt=("σ²", "mw"), weights=c)
    assert abs(float(r0["ds_s"]) - gs["σ²"]) <= RTOL * abs(gs["σ²"])
    assert rel_inf(r0["dmw_s"], gs["mw"]) <= RTOL
