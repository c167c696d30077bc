"""Host-side mirror of BayesianLinearRegressors.jl's public API for the FiniteBLR inference path.

Same names, argument meaning and error behaviour as the reference (file:line cited per function); every method
body is a call into libblr_cuda through the C ABI (`_lib.py`) -- the role the `ccall`s of `julia/src/` play on the
Julia side.  No arithmetic on the path runs on the host and there is no CPU fallback.

    f  = BayesianLinearRegressor(mw, Λw)          # src/bayesian_linear_regression.jl:11-14
    fx = f(ColVecs(X), Σy)                         # AbstractGPs FiniteGP construction
    logpdf(fx, y); posterior(fx, y); mean_and_var(fx); marginals(fx); rand(rng, fx, S)
    BasisFunctionRegressor(f, ϕ)                   # src/basis_function_regression.jl:34-37
    rand(rng, f) / rand(rng, f, dims)              # src/sampling_functions.jl:27-38
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, field
from typing import Callable, Optional, Sequence, Tuple, Union

import numpy as np

from . import _lib as L
from .runtime import (Context, DeviceMatrix, DevicePosterior, DeviceVector, Stats, _f64, _ptr, default_context,
                      make_noise)


# ------------------------------------------------------------------------------------------------
# Input wrappers and matrix kinds
# ------------------------------------------------------------------------------------------------
def _is_torch_cuda(a) -> bool:
    try:
        import torch

        return isinstance(a, torch.Tensor) and a.is_cuda
    except ImportError:  # pragma: no cover
        return False


@dataclass(frozen=True)
class ColVecs:
    """D x N matrix, each column one input (README.md:24).  `X` may be a numpy array (uploaded per call, as the
    reference re-reads its arguments per call), a CUDA tensor of shape (N, D) (= the column-major D x N matrix,
    borrowed), or a DeviceMatrix (already resident: synthetic / RFF outputs)."""

    X: object

    def __len__(self) -> int:
        if isinstance(self.X, DeviceMatrix):
            return self.X.N
        return self.X.shape[0] if _is_torch_cuda(self.X) else self.X.shape[1]

    def __getitem__(self, idx) -> "ColVecs":
        return ColVecs(self.X[:, idx])


@dataclass(frozen=True)
class RowVecs:
    """N x D matrix, each row one input (README.md:25)."""

    X: object

    def __len__(self) -> int:
        if isinstance(self.X, DeviceMatrix):
            return self.X.N
        return self.X.shape[1] if _is_torch_cuda(self.X) else self.X.shape[0]

    def __getitem__(self, idx) -> "RowVecs":
        return RowVecs(self.X[idx, :])


@dataclass(frozen=True)
class Diagonal:
    diag: object

    def dense(self) -> np.ndarray:
        return np.diag(np.asarray(self.diag, dtype=np.float64))


@dataclass(frozen=True)
class Symmetric:
    data: np.ndarray

    def dense(self) -> np.ndarray:
        return self.data


@dataclass(frozen=True)
class PDMat:
    """PDMats.PDMat: matrix + its upper Cholesky factor."""

    mat: np.ndarray
    U: Optional[np.ndarray] = None

    def dense(self) -> np.ndarray:
        return self.mat


def _dense(A) -> np.ndarray:
    return np.asarray(A, dtype=np.float64) if isinstance(A, np.ndarray) else A.dense()


def x_as_colvecs(ctx: Context, x) -> DeviceMatrix:
    """src/bayesian_linear_regression.jl:20-31.  ColVecs pass through; RowVecs are read in place as the
    feature-major layout (the reference's lazy adjoint: no copy); anything else is an error."""
    if isinstance(x, (ColVecs, RowVecs)):
        layout = L.COLVECS if isinstance(x, ColVecs) else L.ROWVECS
        if isinstance(x.X, DeviceMatrix):
            if x.X.layout != layout:
                raise L.BLRError(L.E_INVALID, "DeviceMatrix layout does not match its wrapper")
            return x.X
        if _is_torch_cuda(x.X):
            return DeviceMatrix.wrap_torch(ctx, x.X, layout)
        return DeviceMatrix.upload(ctx, np.asarray(x.X, dtype=np.float64), layout)
    raise RuntimeError(
        f"{type(x).__name__} is not a subtype of AbstractVector that is known. Please provide either a"
        "ColVecs or RowVecs."
    )


def _wrap_inputs(x):
    if isinstance(x, np.ndarray) and x.ndim == 2:  # a bare Matrix is D x N ColVecs (README.md:26)
        return ColVecs(x)
    return x


# ------------------------------------------------------------------------------------------------
# Model types
# ------------------------------------------------------------------------------------------------
class BayesianLinearRegressor:
    """w ~ N(mw, inv(Λw)), f(x) = dot(x, w)   (src/bayesian_linear_regression.jl:11-14).

    `_post` caches the device-resident factorisation (the reference re-runs `_cholesky(Λw)` on every predict
    call, :36,:41,:51)."""

    def __init__(self, mw, Λw, _post: Optional[DevicePosterior] = None):
        self.mw = np.asarray(mw, dtype=np.float64).reshape(-1)
        self.Λw = Λw
        self._post = _post

    def __call__(self, x, Σy=1e-18) -> "FiniteGP":
        return FiniteGP(self, _wrap_inputs(x), Σy)

    # -- C-ABI views ----------------------------------------------------------------------------
    def _prior_struct(self):
        """-> (Prior struct, keepalive list)."""
        D = self.mw.shape[0]
        mw = _f64(self.mw)
        if isinstance(self.Λw, Diagonal):
            lam = _f64(np.asarray(self.Λw.diag, dtype=np.float64).reshape(-1))
            if lam.shape[0] != D:
                raise L.BLRError(L.E_INVALID, "size(Λw) does not match length(mw)")
            kind, ld = L.LAMBDA_DIAGONAL, D
        else:
            lam = _f64(_dense(self.Λw), "F")
            if lam.shape != (D, D):
                raise L.BLRError(L.E_INVALID, "size(Λw) does not match length(mw)")
            kind, ld = L.LAMBDA_DENSE, D
        p = L.Prior(mw.ctypes.data_as(L.c_double_p), kind, lam.ctypes.data_as(L.c_double_p), ld, D)
        return p, [mw, lam]

    def _device(self, ctx: Context) -> DevicePosterior:
        if self._post is None or self._post.ctx is not ctx:
            p, keep = self._prior_struct()
            h = C.c_void_p()
            ctx.check(ctx.lib.blr_post_create(ctx.handle, C.byref(p), self.mw.shape[0], C.byref(h)))
            self._post = DevicePosterior(ctx, h, self.mw.shape[0])
        return self._post


@dataclass
class BasisFunctionRegressor:
    """blr(ϕ(x))   (src/basis_function_regression.jl:34-37).  ϕ maps ColVecs / RowVecs / Matrix to one of those
    types; a device-native map (RandomFourierFeatures) keeps ϕ(x) resident on the GPU."""

    blr: BayesianLinearRegressor
    ϕ: Callable

    def __call__(self, x, Σy=1e-18) -> "FiniteGP":
        return FiniteGP(self, _wrap_inputs(x), Σy)


@dataclass
class FiniteGP:
    """AbstractGPs.FiniteGP{f,x,Σy}: fields .f .x .Σy."""

    f: Union[BayesianLinearRegressor, BasisFunctionRegressor]
    x: object
    Σy: object
    ctx: Optional[Context] = field(default=None, repr=False)

    def _context(self) -> Context:
        return self.ctx if self.ctx is not None else default_context()


def _to_finite_blr(fx: FiniteGP) -> FiniteGP:
    """src/basis_function_regression.jl:41 -- ϕ is evaluated per call, exactly as the reference does."""
    if isinstance(fx.f, BasisFunctionRegressor):
        return FiniteGP(fx.f.blr, _wrap_inputs(fx.f.ϕ(fx.x)), fx.Σy, fx.ctx)
    return fx


FEATURE_GRAD_KEYS = ("W", "b", "xin")


class _DeviceAffineMap:
    """What the two device-native maps ϕ(x) = scale * act(W x + b) share: input staging and the vector-Jacobian product."""

    ACTS = {"cos": 0, "tanh": 1, "relu": 2, "identity": 3, "sin": 4}

    def _context(self) -> Context:
        return self.ctx if self.ctx is not None else default_context()

    def _device_inputs(self, ctx: Context, x) -> DeviceMatrix:
        x = _wrap_inputs(x)
        if isinstance(x, RowVecs):
            x = ColVecs(np.ascontiguousarray(np.asarray(x.X).T)) if isinstance(x.X, np.ndarray) else x
        return x_as_colvecs(ctx, x)

    def vjp(self, x, dΦ, wrt=FEATURE_GRAD_KEYS):
        """Vector-Jacobian product of ϕ at x for the cotangent dΦ (blr_x_features_vjp): with z = W x + b and
        g = dΦ * scale * act'(z), "W" = g x' (D x d_in numpy), "b" = Σ_n g_n (length D), "xin" = W'g (d_in x N numpy for host
        x, an (N, d_in) CUDA tensor for a torch x).  dΦ is D x N numpy or an (N, D) CUDA tensor (ϕ(x)'s ColVecs convention)."""
        ctx = self._context()
        xin = self._device_inputs(ctx, x)
        if _is_torch_cuda(dΦ):
            import torch

            if not (dΦ.dim() == 2 and dΦ.stride(1) == 1):
                dΦ = dΦ.contiguous()
            d = dΦ.to(torch.float64)
            if tuple(d.shape) != (xin.N, self.W.shape[0]):
                raise L.DimensionMismatch(L.E_DIM, "dΦ must be an (N, D) tensor")
            ctx.wait_torch_stream(d)
            return _features_vjp(ctx, self, xin, d.data_ptr(), max(d.stride(0), 1), wrt, _torch_of(x))
        Φd = DeviceMatrix.upload(ctx, np.asarray(dΦ, dtype=np.float64), L.COLVECS)
        if Φd.D != self.W.shape[0] or Φd.N != xin.N:
            raise L.DimensionMismatch(L.E_DIM, "size(dΦ) != (D, N)")
        ptr, ld = Φd.device_ptr()
        return _features_vjp(ctx, self, xin, ptr, ld, wrt, _torch_of(x))


class RandomFourierFeatures(_DeviceAffineMap):
    """Device-native feature map ϕ(x) = sqrt(2/D) cos(W x + b) for BasisFunctionRegressor (BASELINE config 5).
    W is D x d_in, b has length D; input ColVecs (d_in x N) -> output ColVecs (D x N) resident on the device."""

    def __init__(self, W, b, ctx: Optional[Context] = None):
        self.W = _f64(np.asarray(W, dtype=np.float64), "F")
        self.b = _f64(np.asarray(b, dtype=np.float64).reshape(-1))
        self.ctx = ctx
        self.act, self.scale = "cos", float(np.sqrt(2.0 / max(self.W.shape[0], 1)))

    def __call__(self, x):
        ctx = self._context()
        xin = self._device_inputs(ctx, x)
        h = C.c_void_p()
        ctx.check(ctx.lib.blr_x_rff(ctx.handle, xin.handle, _ptr(self.W), _ptr(self.b), self.W.shape[0], C.byref(h)))
        return ColVecs(DeviceMatrix(ctx, h, self.W.shape[0], xin.N, L.COLVECS))


class AffineFeatures(_DeviceAffineMap):
    """Device-native one-layer feature map ϕ(x) = scale * act(W x + b) (blr_x_features): random Fourier features are
    act = "cos", scale = sqrt(2/D); "tanh" / "relu" give the last-layer features of examples/nn-blr.jl style models;
    "identity" a linear projection.  Output resident on the device like RandomFourierFeatures."""

    def __init__(self, W, b, act: str = "tanh", scale: float = 1.0, ctx: Optional[Context] = None):
        if act not in self.ACTS:
            raise L.BLRError(L.E_INVALID, f"unknown activation {act!r}")
        self.W = _f64(np.asarray(W, dtype=np.float64), "F")
        self.b = _f64(np.asarray(b, dtype=np.float64).reshape(-1))
        self.act, self.scale, self.ctx = act, float(scale), ctx

    def __call__(self, x):
        ctx = self._context()
        xin = self._device_inputs(ctx, x)
        if xin.D != self.W.shape[1]:
            raise L.DimensionMismatch(L.E_DIM, "size(W, 2) != size(x, 1)")
        h = C.c_void_p()
        ctx.check(ctx.lib.blr_x_features(ctx.handle, xin.handle, _ptr(self.W), _ptr(self.b), self.W.shape[0], self.ACTS[self.act],
                                         self.scale, C.byref(h)))
        return ColVecs(DeviceMatrix(ctx, h, self.W.shape[0], xin.N, L.COLVECS))


def _torch_of(x):
    """The CUDA tensor behind inputs x, or None."""
    x = _wrap_inputs(x)
    X = x.X if isinstance(x, (ColVecs, RowVecs)) else x
    return X if _is_torch_cuda(X) else None


def _features_vjp(ctx: Context, ϕ: _DeviceAffineMap, xin: DeviceMatrix, dphi_ptr: int, ld_dphi: int, wrt, x_torch=None):
    """One blr_x_features_vjp call for the cotangent at device address dphi_ptr (D x N, leading dimension ld_dphi)."""
    wrt = tuple(wrt)
    bad = [k for k in wrt if k not in FEATURE_GRAD_KEYS]
    if bad:
        raise L.BLRError(L.E_INVALID, f"unknown feature-map gradient keys {bad}; expected a subset of {FEATURE_GRAD_KEYS}")
    D, din, N = ϕ.W.shape[0], ϕ.W.shape[1], xin.N
    if xin.D != din:
        raise L.DimensionMismatch(L.E_DIM, "size(W, 2) != size(x, 1)")
    out = {}
    if "W" in wrt:
        out["W"] = np.empty((D, din), order="F")
    if "b" in wrt:
        out["b"] = np.empty(D)
    dx, dx_ptr = None, None
    if "xin" in wrt and N > 0:
        if x_torch is not None:
            import torch

            dx = torch.empty((N, din), dtype=torch.float64, device=x_torch.device)  # (N, d_in) row-major == d_in x N ColVecs
            ctx.wait_torch_stream(dx)
            dx_ptr = dx.data_ptr()
        else:
            dx = DeviceVector.alloc(ctx, N * din)
            dx_ptr = dx.device_ptr()
    ctx.check(ctx.lib.blr_x_features_vjp(ctx.handle, xin.handle, _ptr(ϕ.W), _ptr(ϕ.b), D, ϕ.ACTS[ϕ.act], ϕ.scale,
                                         C.c_void_p(dphi_ptr), ld_dphi, _ptr(out.get("W")), _ptr(out.get("b")),
                                         None if dx_ptr is None else C.c_void_p(dx_ptr), max(din, 1)))
    if "xin" in wrt:
        if x_torch is not None:
            import torch

            ctx.release_to_torch_stream(x_torch.device)
            out["xin"] = dx if dx is not None else torch.empty((0, din), dtype=torch.float64, device=x_torch.device)
        else:
            out["xin"] = dx.download().reshape((din, N), order="F") if dx is not None else np.empty((din, 0))
    return out


class TorchFeatureMap:
    """Generic device-resident feature-map protocol (src/basis_function_regression.jl:34-37: ϕ is any callable): `fn` is
    user code in torch that maps the (N, d_in) CUDA tensor of inputs to an (N, D) CUDA tensor of features.  Inputs arrive as
    a zero-copy view of the library's device matrix (or are uploaded once if they live on the host), the result is borrowed
    back as a ColVecs design matrix -- ϕ(x) never visits the host, whatever ϕ is.  Stream ordering between torch's stream and
    the library's is handled on both sides (blr_stream_wait_ctx / blr_ctx_wait_stream).  The Julia counterpart wraps CUDA.jl
    arrays with blr_x_wrap_device (INTEGRATION.md)."""

    def __init__(self, fn: Callable, ctx: Optional[Context] = None):
        self.fn, self.ctx = fn, ctx

    def __call__(self, x):
        import torch

        ctx = self.ctx if self.ctx is not None else default_context()
        x = _wrap_inputs(x)
        if isinstance(x, RowVecs) and not isinstance(x.X, DeviceMatrix) and not _is_torch_cuda(x.X):
            x = ColVecs(np.ascontiguousarray(np.asarray(x.X).T))
        if _is_torch_cuda(x.X):
            xin = x.X if isinstance(x, ColVecs) else x.X.T
        else:
            xd = x_as_colvecs(ctx, x)
            xin = xd.as_torch() if xd.layout == L.COLVECS else xd.as_torch().T
        out = self.fn(xin)
        if not (isinstance(out, torch.Tensor) and out.is_cuda and out.dim() == 2 and out.shape[0] == xin.shape[0]):
            raise L.BLRError(L.E_INVALID, "a TorchFeatureMap must return an (N, D) CUDA tensor")
        out = out.to(torch.float64).contiguous()
        return ColVecs(out)  # borrowed by x_as_colvecs -> DeviceMatrix.wrap_torch (orders the library after torch's stream)


# ------------------------------------------------------------------------------------------------
# Inference: logpdf / posterior  (src/bayesian_linear_regression.jl:55-93)
# ------------------------------------------------------------------------------------------------
def _as_device_vector(ctx: Context, y) -> DeviceVector:
    if isinstance(y, DeviceVector):
        return y
    if _is_torch_cuda(y):
        return DeviceVector.wrap_torch(ctx, y)
    return DeviceVector.upload(ctx, y)


def _build_Λ(prior_Λw, Λ_post: np.ndarray, T: Optional[np.ndarray]):
    """src/bayesian_linear_regression.jl:92-93: PDMat prior -> PDMat(Cholesky(UpperTriangular(T))), else Symmetric."""
    if isinstance(prior_Λw, PDMat):
        return PDMat(Λ_post, T)
    return Symmetric(Λ_post)


def _infer(fx: FiniteGP, y, want_logpdf: bool, want_post: bool):
    fx = _to_finite_blr(fx)
    ctx = fx._context()
    blr = fx.f
    D = blr.mw.shape[0]
    if isinstance(fx.x, (ColVecs, RowVecs)) and isinstance(fx.x.X, np.ndarray) and fx.x.X.ndim == 2 and not isinstance(y, DeviceVector) \
            and not _is_torch_cuda(y):
        layout = L.COLVECS if isinstance(fx.x, ColVecs) else L.ROWVECS
        hn = _host_noise(fx.Σy, len(fx.x))
        if hn is not None:  # host data + diagonal noise: stream it (no staging copy of X on the device)
            return _infer_host(ctx, blr, fx.x.X, layout, y, hn, 1 << 16, want_logpdf, want_post)
    X = x_as_colvecs(ctx, fx.x)
    if X.D != D:  # `X' * mw` (:33) throws DimensionMismatch in the reference; the C ABI checks prior.D as well
        raise L.DimensionMismatch(L.E_DIM, "size(X, 1) != length(mw)")
    yv = _as_device_vector(ctx, y)
    if yv.n != X.N:  # src/bayesian_linear_regression.jl:74
        raise L.DimensionMismatch(L.E_DIM, "length(y) != size(fx.x.X, 2)")
    noise, keep_noise = make_noise(ctx, fx.Σy, X.N)
    prior, keep_prior = blr._prior_struct()
    lp = C.c_double()
    m_post = np.empty(D) if want_post else None
    Λ_post = ctx.empty_pinned((D, D)) if want_post else None
    T_post = ctx.empty_pinned((D, D)) if (want_post and isinstance(blr.Λw, PDMat)) else None
    h = C.c_void_p()
    ctx.check(
        ctx.lib.blr_infer(ctx.handle, C.byref(prior), X.handle, yv.handle, C.byref(noise),
                          C.byref(lp) if want_logpdf else None, _ptr(m_post), _ptr(T_post), _ptr(Λ_post),
                          C.byref(h) if want_post else None)
    )
    post = None
    if want_post:
        post = BayesianLinearRegressor(m_post, _build_Λ(blr.Λw, Λ_post, T_post), _post=DevicePosterior(ctx, h, D))
    return (lp.value if want_logpdf else None), post


def logpdf(fx: FiniteGP, y):
    """src/bayesian_linear_regression.jl:55-58 / basis_function_regression.jl:60.  A matrix `Y` (N x k, one
    observation vector per column) returns the k log densities, as AbstractGPs' `logpdf(fx, Y::AbstractMatrix)`."""
    if (isinstance(y, np.ndarray) or _is_torch_cuda(y)) and y.ndim == 2:
        return _logpdf_multi(fx, y)
    return _infer(fx, y, True, False)[0]


def _logpdf_multi(fx: FiniteGP, Y) -> np.ndarray:
    """logpdf(fx, Y::AbstractMatrix): one Gram pass, one factorisation, k right-hand sides (blr_logpdf_multi).  Y is a host
    array or a CUDA tensor of shape (N, k).  Dense Σy (the small-N side path) loops over the columns."""
    fx = _to_finite_blr(fx)
    ctx = fx._context()
    blr = fx.f
    k = int(Y.shape[1])
    if k == 0:
        return np.empty(0)
    if isinstance(fx.Σy, (Symmetric, PDMat)) or (isinstance(fx.Σy, np.ndarray) and fx.Σy.ndim == 2):
        cols = Y.T.contiguous() if _is_torch_cuda(Y) else np.ascontiguousarray(np.asarray(Y, dtype=np.float64).T)
        return np.array([_infer(fx, cols[j], True, False)[0] for j in range(k)])
    X = x_as_colvecs(ctx, fx.x)
    if X.D != blr.mw.shape[0]:
        raise L.DimensionMismatch(L.E_DIM, "size(X, 1) != length(mw)")
    if Y.shape[0] != X.N:  # src/bayesian_linear_regression.jl:74
        raise L.DimensionMismatch(L.E_DIM, "length(y) != size(fx.x.X, 2)")
    if _is_torch_cuda(Y):
        import torch

        Yt = Y.to(torch.float64).T.contiguous()  # (k, N) row-major == N x k column-major
        ctx.wait_torch_stream()
        y_ptr, keep = C.c_void_p(Yt.data_ptr()), Yt
    else:
        Yd = DeviceVector.upload(ctx, np.asarray(Y, dtype=np.float64).T.reshape(-1))  # column-major N x k, flattened
        y_ptr, keep = C.c_void_p(Yd.device_ptr()), Yd
    noise, keep_noise = make_noise(ctx, fx.Σy, X.N)
    prior, keep_prior = blr._prior_struct()
    out = np.empty(k)
    ctx.check(ctx.lib.blr_logpdf_multi(ctx.handle, C.byref(prior), X.handle, y_ptr, max(X.N, 1), k, C.byref(noise), _ptr(out)))
    del keep
    return out


GRAD_KEYS = ("X", "y", "σ²", "mw", "Λw")


def _logpdf_grad_call(ctx: Context, blr: BayesianLinearRegressor, X: DeviceMatrix, yv, Σy, wrt, out_like=None, k=None,
                      weights=None, keep_dX=False):
    """One blr_logpdf_grad call, or with `k` one blr_logpdf_multi_grad call: then yv is the device address of Y (N x k,
    column-major, ld = N), the value is the k log densities and the gradients are those of Σ_j weights_j ℓ_j (weights: None for
    all ones).  Per-observation gradients are written into CUDA tensors on out_like's device when `out_like` (a CUDA tensor) is
    given -- dX with the shape torch sees x in, (N, D) for ColVecs; "y" (N, k) -- else downloaded into numpy arrays (dX with the
    Julia-side shape; with keep_dX the device buffer itself, ColVecs only).  Keys of `wrt` not in GRAD_KEYS are an error; keys
    left out get NULL."""
    wrt = tuple(wrt)
    bad = [k for k in wrt if k not in GRAD_KEYS]
    if bad:
        raise L.BLRError(L.E_INVALID, f"unknown gradient keys {bad}; expected a subset of {GRAD_KEYS}")
    D = blr.mw.shape[0]
    if X.D != D:  # `X' * mw` (:33) throws DimensionMismatch in the reference
        raise L.DimensionMismatch(L.E_DIM, "size(X, 1) != length(mw)")
    if k is None and yv.n != X.N:  # src/bayesian_linear_regression.jl:74
        raise L.DimensionMismatch(L.E_DIM, "length(y) != size(fx.x.X, 2)")
    noise, keep_noise = make_noise(ctx, Σy, X.N)
    prior, keep_prior = blr._prior_struct()
    N, colv = X.N, X.layout == L.COLVECS
    vector_noise = noise.kind == L.NOISE_VECTOR
    g = L.LogpdfGrads()
    out, dev = {}, {}
    if "mw" in wrt:
        out["mw"] = np.empty(D)
        g.dmw = out["mw"].ctypes.data_as(L.c_double_p)
    if "Λw" in wrt:
        out["Λw"] = np.empty(D) if isinstance(blr.Λw, Diagonal) else np.empty((D, D), order="F")
        g.dlambda = out["Λw"].ctypes.data_as(L.c_double_p)
    dσ2_host = C.c_double()
    if "σ²" in wrt and not vector_noise:
        g.dsigma2 = C.pointer(dσ2_host)
    if out_like is not None:
        import torch

        def buf(*shape):
            return torch.empty(shape, dtype=torch.float64, device=out_like.device)
    else:
        def buf(*shape):
            return DeviceVector.alloc(ctx, int(np.prod(shape)))

    def addr(b):
        return b.data_ptr() if out_like is not None else b.device_ptr()

    if "y" in wrt:
        dev["y"] = buf(N) if k is None else buf(k, N)  # (k, N) row-major == N x k column-major
        g.dy_dev = addr(dev["y"])
    if "σ²" in wrt and vector_noise:
        dev["σ²"] = buf(N)
        g.dsigma2_dev = addr(dev["σ²"])
    if "X" in wrt:
        dev["X"] = buf(N, D) if colv else buf(D, N)  # torch row-major (N, D) == column-major D x N (ColVecs); (D, N) for RowVecs
        g.dX_dev = addr(dev["X"])
        g.ld_dX = max(D if colv else N, 1)
    if out_like is not None:  # the output tensors were just allocated on torch's stream
        ctx.wait_torch_stream(out_like)
    if k is None:
        lp = C.c_double()
        ctx.check(ctx.lib.blr_logpdf_grad(ctx.handle, C.byref(prior), X.handle, yv.handle, C.byref(noise), C.byref(lp), C.byref(g)))
        lp = lp.value
    else:
        lp = np.empty(k)
        c = None if weights is None else np.ascontiguousarray(weights, dtype=np.float64).reshape(k)
        ctx.check(ctx.lib.blr_logpdf_multi_grad(ctx.handle, C.byref(prior), X.handle, yv, max(N, 1), k, C.byref(noise),
                                                None if c is None else c.ctypes.data_as(L.c_double_p), lp.ctypes.data_as(L.c_double_p),
                                                C.byref(g)))
    if "σ²" in wrt and not vector_noise:
        out["σ²"] = dσ2_host.value
    if out_like is not None:
        ctx.release_to_torch_stream(out_like.device)
        if k is not None and "y" in dev:
            dev["y"] = dev["y"].T
        out.update(dev)
    else:
        for key, v in dev.items():
            if key == "X" and keep_dX:
                out[key] = v
                continue
            a = v.download()
            if key == "X":
                a = a.reshape((D, N) if colv else (N, D), order="F")
            elif key == "y" and k is not None:
                a = a.reshape((N, k), order="F")
            out[key] = a
    return lp, out


def logpdf_and_grad(fx: FiniteGP, y, wrt=GRAD_KEYS, weights=None):
    """logpdf(fx, y) and its gradients with respect to the keys of `wrt` -- "X" (the inputs; ϕ(x) for a BasisFunctionRegressor),
    "y", "σ²" (a scalar for scalar noise, else one per observation), "mw" and "Λw" (D values for a Diagonal prior, else the
    symmetric D x D G with dℓ = <G, dΛw>) -- in closed form on the device (blr_logpdf_grad).  Returns (logpdf, dict).
    Per-observation gradients of inputs given as CUDA tensors come back as CUDA tensors (dX with x's tensor shape, (N, D) for
    ColVecs); otherwise everything is numpy (dX D x N for ColVecs, N x D for RowVecs).
    A matrix `Y` (N x k, a host array or a CUDA tensor; one observation vector per column) returns the k log densities and the
    gradients of Σ_j weights_j ℓ_j (weights: k values, None for all ones) from ONE call (blr_logpdf_multi_grad): the Gram pass and
    the O(N D²) product run once for all k columns.  "y" then has Y's shape.
    For a BasisFunctionRegressor over AffineFeatures or RandomFourierFeatures, `wrt` may also hold "W" and "b" (the gradients
    with respect to ϕ's parameters, D x d_in and D numpy) and "xin" (with respect to ϕ's input, shaped as vjp returns it):
    ∂ℓ/∂ϕ(x) stays on the device and goes through one blr_x_features_vjp call."""
    if any(k in FEATURE_GRAD_KEYS for k in wrt):
        return _logpdf_and_feature_grad(fx, y, tuple(wrt), weights)
    fx = _to_finite_blr(fx)
    ctx = fx._context()
    out_like = None
    for cand in (fx.x.X, y):
        if _is_torch_cuda(cand):
            out_like = cand
            break
    if (isinstance(y, np.ndarray) or _is_torch_cuda(y)) and y.ndim == 2:
        return _logpdf_multi_grad(ctx, fx, y, wrt, weights, out_like)
    X = x_as_colvecs(ctx, fx.x)
    yv = _as_device_vector(ctx, y)
    return _logpdf_grad_call(ctx, fx.f, X, yv, fx.Σy, wrt, out_like)


def _logpdf_and_feature_grad(fx: FiniteGP, y, wrt, weights):
    """logpdf_and_grad through a device feature map: x uploaded and ϕ(x) evaluated once, ∂ℓ/∂ϕ(x) written by blr_logpdf_grad
    (blr_logpdf_multi_grad for a matrix Y) into a device buffer, then one VJP call."""
    ϕ = fx.f.ϕ if isinstance(fx.f, BasisFunctionRegressor) else None
    if not isinstance(ϕ, _DeviceAffineMap):
        raise L.BLRError(L.E_INVALID, "gradients with respect to \"W\", \"b\" and \"xin\" need a BasisFunctionRegressor over "
                                      "AffineFeatures or RandomFourierFeatures; differentiate a TorchFeatureMap with torch autograd "
                                      "(torch_logpdf)")
    ctx = ϕ._context()
    xin = ϕ._device_inputs(ctx, fx.x)
    Φ = ϕ(ColVecs(xin))
    inner = tuple(k for k in wrt if k not in FEATURE_GRAD_KEYS) + (() if "X" in wrt else ("X",))
    ffx = FiniteGP(fx.f.blr, Φ, fx.Σy, ctx)
    out_like = y if _is_torch_cuda(y) else None
    if (isinstance(y, np.ndarray) or _is_torch_cuda(y)) and y.ndim == 2:
        lp, g = _logpdf_multi_grad(ctx, ffx, y, inner, weights, out_like, keep_dX=True)
    else:
        lp, g = _logpdf_grad_call(ctx, ffx.f, Φ.X, _as_device_vector(ctx, y), fx.Σy, inner, out_like, keep_dX=True)
    dΦ = g.pop("X")
    D, N = Φ.X.D, Φ.X.N
    ptr = dΦ.data_ptr() if out_like is not None else dΦ.device_ptr()
    if out_like is not None:
        ctx.wait_torch_stream(dΦ)
    g.update(_features_vjp(ctx, ϕ, xin, ptr, max(D, 1), [k for k in wrt if k in FEATURE_GRAD_KEYS], _torch_of(fx.x)))
    if "X" in wrt:
        g["X"] = dΦ if out_like is not None else dΦ.download().reshape((D, N), order="F")
    return lp, g


def _logpdf_multi_grad(ctx: Context, fx: FiniteGP, Y, wrt, weights, out_like, keep_dX=False):
    X = x_as_colvecs(ctx, fx.x)
    k = int(Y.shape[1])
    if X.D != fx.f.mw.shape[0]:
        raise L.DimensionMismatch(L.E_DIM, "size(X, 1) != length(mw)")
    if Y.shape[0] != X.N:  # src/bayesian_linear_regression.jl:74
        raise L.DimensionMismatch(L.E_DIM, "length(y) != size(fx.x.X, 2)")
    if weights is not None and np.size(weights) != k:
        raise L.DimensionMismatch(L.E_DIM, "length(weights) != size(Y, 2)")
    if _is_torch_cuda(Y):
        import torch

        Yt = Y.to(torch.float64).T.contiguous()  # (k, N) row-major == N x k column-major
        ctx.wait_torch_stream()
        return _logpdf_grad_call(ctx, fx.f, X, C.c_void_p(Yt.data_ptr()), fx.Σy, wrt, out_like, k, weights, keep_dX)
    Yd = DeviceVector.upload(ctx, np.asarray(Y, dtype=np.float64).T.reshape(-1))  # column-major N x k, flattened
    return _logpdf_grad_call(ctx, fx.f, X, C.c_void_p(Yd.device_ptr()), fx.Σy, wrt, out_like, k, weights, keep_dX)


def _torch_logpdf_function():
    import torch

    class TorchLogpdf(torch.autograd.Function):
        """ℓ(X, y, mw, Λw, σ²) as a differentiable torch op; forward computes the gradients the backward needs in the same call
        (blr_logpdf_grad), backward only scales them by grad_output."""

        @staticmethod
        def forward(fctx, X, y, mw, Λw, σ2):
            ctx = default_context()
            if not (X.is_cuda and X.dtype == torch.float64 and X.dim() == 2):
                raise L.BLRError(L.E_INVALID, "torch_logpdf: X must be an (N, D) float64 CUDA tensor")
            mw_h = mw.detach().to("cpu", torch.float64).numpy()
            lam_h = Λw.detach().to("cpu", torch.float64).numpy()
            blr = BayesianLinearRegressor(mw_h, Diagonal(lam_h) if lam_h.ndim == 1 else lam_h)
            Xc = X.detach().contiguous()
            Xd = DeviceMatrix.wrap_torch(ctx, Xc, L.COLVECS)
            yv = DeviceVector.wrap_torch(ctx, y.detach().to(torch.float64).contiguous())
            Σy = float(σ2) if σ2.dim() == 0 else σ2.detach().to(torch.float64).contiguous()
            need = fctx.needs_input_grad
            wrt = [k for k, n in zip(GRAD_KEYS, (need[0], need[1], need[4], need[2], need[3])) if n]
            lp, g = _logpdf_grad_call(ctx, blr, Xd, yv, Σy, wrt, out_like=Xc)
            grads = []
            for k, like in (("X", X), ("y", y), ("mw", mw), ("Λw", Λw), ("σ²", σ2)):
                v = g.get(k)
                if v is not None and not isinstance(v, torch.Tensor):
                    v = torch.as_tensor(np.asarray(v), dtype=torch.float64, device=like.device).reshape(like.shape)
                grads.append(v)
            fctx.save_for_backward(*[v if v is not None else torch.empty(0) for v in grads])
            fctx.present = [v is not None for v in grads]
            return torch.tensor(lp, dtype=torch.float64, device=X.device)

        @staticmethod
        def backward(fctx, grad_out):
            saved = fctx.saved_tensors
            return tuple(grad_out * v if present else None for v, present in zip(saved, fctx.present))

    class TorchLogpdfMulti(torch.autograd.Function):
        """The k log densities of the columns of an (N, k) Y as a differentiable torch op.  The cotangent is not known in the
        forward call, so forward runs blr_logpdf_multi alone and backward makes one blr_logpdf_multi_grad call with the
        cotangent as the weights: the backward re-runs the Gram pass and the factorisation."""

        @staticmethod
        def forward(fctx, X, Y, mw, Λw, σ2):
            if not (X.is_cuda and X.dtype == torch.float64 and X.dim() == 2):
                raise L.BLRError(L.E_INVALID, "torch_logpdf: X must be an (N, D) float64 CUDA tensor")
            fx = _torch_finite_gp(X, mw, Λw, σ2)
            fctx.save_for_backward(X, Y, mw, Λw, σ2)
            return torch.as_tensor(_logpdf_multi(fx, Y.detach()), dtype=torch.float64, device=X.device)

        @staticmethod
        def backward(fctx, grad_out):
            X, Y, mw, Λw, σ2 = fctx.saved_tensors
            need = fctx.needs_input_grad
            wrt = [k for k, n in zip(GRAD_KEYS, (need[0], need[1], need[4], need[2], need[3])) if n]
            if not wrt:
                return (None,) * 5
            fx = _torch_finite_gp(X, mw, Λw, σ2)
            c = grad_out.detach().to("cpu", torch.float64).numpy()
            _, g = logpdf_and_grad(fx, Y.detach(), wrt=wrt, weights=c)
            grads = []
            for k, like in (("X", X), ("y", Y), ("mw", mw), ("Λw", Λw), ("σ²", σ2)):
                v = g.get(k)
                if v is not None and not isinstance(v, torch.Tensor):
                    v = torch.as_tensor(np.asarray(v), dtype=torch.float64, device=like.device).reshape(like.shape)
                grads.append(v)
            return tuple(grads)

    return TorchLogpdf, TorchLogpdfMulti


def _torch_finite_gp(X, mw, Λw, σ2):
    """BayesianLinearRegressor(mw, Λw)(ColVecs(X), σ²) over detached tensors: the prior on the host, X and a vector σ² on the
    device."""
    import torch

    mw_h = mw.detach().to("cpu", torch.float64).numpy()
    lam_h = Λw.detach().to("cpu", torch.float64).numpy()
    blr = BayesianLinearRegressor(mw_h, Diagonal(lam_h) if lam_h.ndim == 1 else lam_h)
    Σy = float(σ2) if σ2.dim() == 0 else σ2.detach().to(torch.float64).contiguous()
    return blr(ColVecs(X.detach().contiguous()), Σy)


_TORCH_LOGPDF = None


def torch_logpdf(X, y, mw, Λw, σ2):
    """Differentiable logpdf of y under BayesianLinearRegressor(mw, Λw)(ColVecs(X), σ²) for float64 CUDA tensors: X is (N, D),
    Λw is (D,) (Diagonal prior) or (D, D), σ² is 0-d (scalar noise) or (N,).  The gradients of the inputs that require them are
    computed on the device in the forward call; this is what makes a TorchFeatureMap's network trainable by type-II maximum
    likelihood (the reference's examples/nn-blr.jl).
    An (N, k) y (k target series sharing one feature map) returns the (k,) log densities.  Its forward is blr_logpdf_multi; its
    backward is one blr_logpdf_multi_grad call weighted by the incoming gradient, which re-runs the Gram pass (about the cost of
    one single-column gradient call, whatever k)."""
    global _TORCH_LOGPDF
    if _TORCH_LOGPDF is None:
        _TORCH_LOGPDF = _torch_logpdf_function()
    return _TORCH_LOGPDF[1 if y.dim() == 2 else 0].apply(X, y, mw, Λw, σ2)


def _torch_features_function():
    import torch

    class TorchFeatures(torch.autograd.Function):
        """ϕ(x) = scale * act(W x + b) as a differentiable torch op: forward is blr_x_features, returned as a zero-copy (N, D)
        view of the library's matrix; only x, W and b are saved; backward is one blr_x_features_vjp call."""

        @staticmethod
        def forward(fctx, x, W, b, act, scale):
            if not (x.is_cuda and x.dtype == torch.float64 and x.dim() == 2):
                raise L.BLRError(L.E_INVALID, "torch_features: x must be an (N, d_in) float64 CUDA tensor")
            ϕ = _torch_affine_map(W, b, act, scale)
            fctx.save_for_backward(x, W, b)
            fctx.act, fctx.scale = act, scale
            return ϕ(ColVecs(x.detach().contiguous())).X.as_torch()

        @staticmethod
        def backward(fctx, gΦ):
            x, W, b = fctx.saved_tensors
            need = fctx.needs_input_grad
            wrt = [k for k, n in zip(("xin", "W", "b"), need[:3]) if n]
            if not wrt:
                return (None,) * 5
            ϕ = _torch_affine_map(W, b, fctx.act, fctx.scale)
            g = ϕ.vjp(ColVecs(x.detach().contiguous()), gΦ.to(torch.float64).contiguous(), wrt)
            dx = g.get("xin")
            dW = None if "W" not in g else torch.as_tensor(g["W"], dtype=W.dtype, device=W.device)
            db = None if "b" not in g else torch.as_tensor(g["b"], dtype=b.dtype, device=b.device)
            return dx, dW, db, None, None

    return TorchFeatures


def _torch_affine_map(W, b, act, scale) -> AffineFeatures:
    import torch

    return AffineFeatures(W.detach().to("cpu", torch.float64).numpy(), b.detach().to("cpu", torch.float64).numpy(), act, float(scale))


_TORCH_FEATURES = None


def torch_features(x, W, b, act: str = "cos", scale: float = 1.0):
    """ϕ(x) = scale * act(W x + b) for an (N, d_in) float64 CUDA tensor x, W (D, d_in) and b (D,), as an (N, D) CUDA tensor that
    torch autograd differentiates with respect to x, W and b on the device (blr_x_features / blr_x_features_vjp).  Composes with
    torch_logpdf: torch_logpdf(torch_features(x, Ω / ℓ, b, "cos", (2 / D) ** 0.5), y, mw, Λw, σ²).backward() gives ∂/∂ℓ of
    a random-Fourier-feature regressor.
    Against torch autograd of the same map in fp64 this saves memory, not time: it keeps no N x D temporaries (torch's
    holds several), but its backward is currently about 2x slower (DESIGN.md, K10)."""
    global _TORCH_FEATURES
    if _TORCH_FEATURES is None:
        _TORCH_FEATURES = _torch_features_function()
    return _TORCH_FEATURES.apply(x, W, b, act, scale)


def posterior(fx: FiniteGP, y):
    """src/bayesian_linear_regression.jl:60-69 / basis_function_regression.jl:62-65."""
    post = _infer(fx, y, False, True)[1]
    if isinstance(fx.f, BasisFunctionRegressor):
        return BasisFunctionRegressor(post, fx.f.ϕ)
    return post


def posterior_and_logpdf(fx: FiniteGP, y):
    """Both results from ONE pass over the data (the reference runs __compute_inference_quantities twice,
    src/bayesian_linear_regression.jl:56,:61).  Returns (posterior, logpdf)."""
    lp, post = _infer(fx, y, True, True)
    if isinstance(fx.f, BasisFunctionRegressor):
        post = BasisFunctionRegressor(post, fx.f.ϕ)
    return post, lp


def _host_noise(Σy, N: int):
    """-> (kind, scalar, vector-or-None) for scalar / diagonal host noise, or None if Σy is anything else."""
    if isinstance(Σy, Diagonal):
        Σy = Σy.diag
    if isinstance(Σy, (DeviceVector, Symmetric, PDMat)) or _is_torch_cuda(Σy):
        return None
    s2 = np.asarray(Σy, dtype=np.float64)
    if s2.ndim == 0:
        return L.NOISE_SCALAR, float(s2), None
    if s2.ndim == 1:
        if s2.shape[0] != N:
            raise L.DimensionMismatch(L.E_DIM, "length(diag(Σy)) != number of inputs")
        return L.NOISE_VECTOR, 0.0, _f64(s2)
    return None


def _infer_host(ctx: Context, f: BayesianLinearRegressor, X, layout: int, y, noise, chunk: int, want_logpdf: bool,
                want_post: bool):
    """Inference from HOST arrays: the observations are streamed through blr_stats_accumulate_host in chunks (H2D on a
    copy stream overlapped with the Gram kernel, no second full copy of X on the device), then one all-reduce and the
    replicated solve."""
    D = f.mw.shape[0]
    Xf = _f64(np.asarray(X, dtype=np.float64), "F")
    Dx, N = Xf.shape if layout == L.COLVECS else Xf.shape[::-1]
    yv = _f64(np.asarray(y, dtype=np.float64).reshape(-1))
    if Dx != D:
        raise L.BLRError(L.E_INVALID, "size(X, 1) != length(mw)")
    if yv.shape[0] != N:  # src/bayesian_linear_regression.jl:74
        raise L.DimensionMismatch(L.E_DIM, "length(y) != size(fx.x.X, 2)")
    kind, scalar, s2 = noise
    st = Stats(ctx, D)
    mw = _f64(f.mw)
    ctx.check(ctx.lib.blr_stats_accumulate_host(ctx.handle, st.handle, _ptr(mw), _ptr(Xf), D, N, max(Xf.shape[0], 1), layout,
                                                _ptr(yv), kind, scalar, _ptr(s2), int(chunk)))
    st.allreduce()
    prior, keep = f._prior_struct()
    lp = C.c_double()
    m_post = np.empty(D) if want_post else None
    Λ_post = ctx.empty_pinned((D, D)) if want_post else None
    T_post = ctx.empty_pinned((D, D)) if (want_post and isinstance(f.Λw, PDMat)) else None
    h = C.c_void_p()
    try:
        ctx.check(ctx.lib.blr_infer_from_stats(ctx.handle, C.byref(prior), st.handle, C.byref(lp) if want_logpdf else None,
                                               _ptr(m_post), _ptr(T_post), _ptr(Λ_post), C.byref(h) if want_post else None))
    except L.PosDefException:
        if s2 is not None and not np.all(s2 > 0):  # cholesky(Diagonal(σ²)) fails at the first non-positive entry (:79)
            raise L.PosDefException(int(np.argmax(~(s2 > 0))) + 1) from None
        raise
    post = None
    if want_post:
        post = BayesianLinearRegressor(m_post, _build_Λ(f.Λw, Λ_post, T_post), _post=DevicePosterior(ctx, h, D))
    return (lp.value if want_logpdf else None), post


def posterior_and_logpdf_streamed(f: BayesianLinearRegressor, X, y, Σy, chunk: int = 1 << 16, ctx: Optional[Context] = None,
                                  layout: int = L.COLVECS):
    """posterior + logpdf for HOST arrays too large (or too transient) to keep on the device; X is the D x N matrix
    (ColVecs; Fortran order is sent without a copy) or the N x D matrix with layout=ROWVECS.  Returns
    (posterior, logpdf).  `posterior` / `logpdf` on numpy inputs take the same path."""
    ctx = ctx or default_context()
    Xa = np.asarray(X)
    N = Xa.shape[1] if layout == L.COLVECS else Xa.shape[0]
    noise = _host_noise(Σy, N)
    if noise is None:
        raise L.BLRError(L.E_INVALID, "noise must be a scalar or a length-N vector of variances")
    lp, post = _infer_host(ctx, f, Xa, layout, y, noise, chunk, True, True)
    return post, lp


# ------------------------------------------------------------------------------------------------
# Prediction: mean / var / cov / marginals  (src/bayesian_linear_regression.jl:33-47)
# ------------------------------------------------------------------------------------------------
def _predict(fx: FiniteGP, want_mean: bool, want_var: bool):
    fx = _to_finite_blr(fx)
    ctx = fx._context()
    X = x_as_colvecs(ctx, fx.x)
    if X.D != fx.f.mw.shape[0]:
        raise L.BLRError(L.E_INVALID, "size(X, 1) != length(mw)")
    post = fx.f._device(ctx)
    noise, keep = make_noise(ctx, fx.Σy, X.N)
    m = ctx.empty_pinned((X.N,)) if want_mean else None
    v = ctx.empty_pinned((X.N,)) if want_var else None
    ctx.check(ctx.lib.blr_mean_var(ctx.handle, post.handle, X.handle, C.byref(noise), _ptr(m), _ptr(v)))
    return m, v


def mean(fx: FiniteGP) -> np.ndarray:
    return _predict(fx, True, False)[0]


def var(fx: FiniteGP) -> np.ndarray:
    return _predict(fx, False, True)[1]


def mean_and_var(fx: FiniteGP) -> Tuple[np.ndarray, np.ndarray]:
    return _predict(fx, True, True)


def std(fx: FiniteGP) -> np.ndarray:
    return np.sqrt(var(fx))


def marginals(fx: FiniteGP) -> Tuple[np.ndarray, np.ndarray]:
    """AbstractGPs.marginals: Normal.(mean, sqrt.(var)); returned as (mean, std) arrays."""
    m, v = mean_and_var(fx)
    return m, np.sqrt(v)


def cov(fx: FiniteGP) -> np.ndarray:
    """src/bayesian_linear_regression.jl:35-38 (N x N; small-N path)."""
    fx = _to_finite_blr(fx)
    ctx = fx._context()
    X = x_as_colvecs(ctx, fx.x)
    post = fx.f._device(ctx)
    noise, keep = make_noise(ctx, fx.Σy, X.N)
    Cm = np.empty((X.N, X.N), order="F")
    ctx.check(ctx.lib.blr_cov(ctx.handle, post.handle, X.handle, C.byref(noise), _ptr(Cm)))
    return Cm


def mean_and_cov(fx: FiniteGP):
    return mean(fx), cov(fx)


# ------------------------------------------------------------------------------------------------
# Sampling  (src/bayesian_linear_regression.jl:49-53, src/sampling_functions.jl)
# ------------------------------------------------------------------------------------------------
def _randn_colmajor(rng: np.random.Generator, rows: int, cols: int) -> np.ndarray:
    """randn(rng, rows, cols) with Julia's column-major fill order."""
    return np.asfortranarray(rng.standard_normal((cols, rows)).T)


@dataclass(frozen=True)
class DeviceRNG:
    """Draw the standard normals on the device (Philox4x32-10) instead of shipping them from the host."""

    seed: int = 0


@dataclass(frozen=True)
class BLRFunctionSample:
    """src/sampling_functions.jl:12-19: a fixed weight sample; calling it evaluates ϕ(X)'w on the device."""

    w: np.ndarray
    ϕ: Callable

    def __call__(self, X):
        ctx = default_context()
        Z = _wrap_inputs(self.ϕ(_wrap_inputs(X)))
        Xd = x_as_colvecs(ctx, Z)
        if Xd.D != self.w.shape[0]:
            raise L.BLRError(L.E_INVALID, "size(ϕ(X), 1) != length(w)")
        out = np.empty(Xd.N)
        w = _f64(self.w)
        ctx.check(ctx.lib.blr_apply_weights(ctx.handle, Xd.handle, _ptr(w), _ptr(out)))
        return out


def _identity(x):
    return x


def _blr_and_mapping(b):
    """src/sampling_functions.jl:51-52."""
    if isinstance(b, BasisFunctionRegressor):
        return b.blr, b.ϕ
    return b, _identity


def _rand_weights(blr: BayesianLinearRegressor, rng, S: int, ctx: Optional[Context] = None) -> np.ndarray:
    ctx = ctx or default_context()
    D = blr.mw.shape[0]
    post = blr._device(ctx)
    W = np.empty((D, S), order="F")
    if isinstance(rng, DeviceRNG):
        Z, seed = None, rng.seed
    else:
        Z, seed = _randn_colmajor(rng, D, S), 0
    ctx.check(ctx.lib.blr_rand_weights(ctx.handle, post.handle, S, _ptr(Z), seed, _ptr(W)))
    return W


def rand(rng, target, *dims):
    """Julia's `rand` methods on this path, dispatched on the target:

    rand(rng, fx::FiniteGP, samples::Int) -> N x samples matrix     (src/bayesian_linear_regression.jl:49-53)
    rand(rng, fx::FiniteGP)               -> N vector               (AbstractGPs generic -> rand(rng, fx, 1))
    rand(rng, b)                          -> BLRFunctionSample      (src/sampling_functions.jl:27-31)
    rand(rng, b, dims...)                 -> array of samples       (src/sampling_functions.jl:33-38)

    `rng` is a numpy Generator (draws Zw = randn(D, S) FIRST, then Zy = randn(N, S), as :51-52) or a DeviceRNG.
    """
    if rng is None:  # Julia's `rand(fx)` / `rand(b)`: the global default RNG
        rng = np.random.default_rng()
    if isinstance(target, FiniteGP):
        S = int(dims[0]) if dims else 1
        Y = _rand_finite(rng, target, S)
        return Y if dims else Y[:, 0]
    blr, ϕ = _blr_and_mapping(target)
    if not dims:
        return BLRFunctionSample(_rand_weights(blr, rng, 1)[:, 0].copy(), ϕ)
    shape = tuple(int(d) for d in (dims[0] if len(dims) == 1 and isinstance(dims[0], (tuple, list)) else dims))
    ws = _rand_weights(blr, rng, int(np.prod(shape)))
    flat = np.empty(ws.shape[1], dtype=object)
    for i in range(ws.shape[1]):
        flat[i] = BLRFunctionSample(ws[:, i].copy(), ϕ)
    return flat.reshape(shape, order="F")


def rand_into(rng, A: np.ndarray, b):
    """Random.rand!(rng, A, b)  (src/sampling_functions.jl:40-49)."""
    blr, ϕ = _blr_and_mapping(b)
    ws = _rand_weights(blr, rng, A.size)
    flat = A.reshape(-1, order="F")
    for i in range(A.size):
        flat[i] = BLRFunctionSample(ws[:, i].copy(), ϕ)
    A[...] = flat.reshape(A.shape, order="F")
    return A


def _rand_finite(rng, fx: FiniteGP, S: int, Zw=None, Zy=None) -> np.ndarray:
    fx = _to_finite_blr(fx)
    ctx = fx._context()
    X = x_as_colvecs(ctx, fx.x)
    D = fx.f.mw.shape[0]
    if X.D != D:
        raise L.BLRError(L.E_INVALID, "size(X, 1) != length(mw)")
    post = fx.f._device(ctx)
    noise, keep = make_noise(ctx, fx.Σy, X.N)
    seed = 0
    if Zw is None and Zy is None:
        if isinstance(rng, DeviceRNG):
            seed = rng.seed
        else:
            Zw = _randn_colmajor(rng, D, S)  # :51 first
            Zy = _randn_colmajor(rng, X.N, S)  # :52 second
    if Zw is not None:
        Zw = _f64(np.asarray(Zw, dtype=np.float64).reshape(D, S), "F")
    if Zy is not None:
        Zy = _f64(np.asarray(Zy, dtype=np.float64).reshape(X.N, S), "F")
    Y = ctx.empty_pinned((X.N, S))
    ctx.check(ctx.lib.blr_rand_finite(ctx.handle, post.handle, X.handle, C.byref(noise), S, _ptr(Zw), _ptr(Zy), seed, _ptr(Y)))
    return Y


def rand_with_draws(fx: FiniteGP, Zw, Zy) -> np.ndarray:
    """rand with the standard-normal draws supplied (parity mode of BASELINE.json: 'same standard-normal draws')."""
    Zw = np.asarray(Zw, dtype=np.float64)
    S = 1 if Zw.ndim == 1 else Zw.shape[1]
    return _rand_finite(None, fx, S, Zw=Zw, Zy=Zy)
