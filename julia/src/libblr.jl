# Low-level ccall bindings of libblr_cuda (include/blr_cuda.h).
#
# UNEXECUTED: there is no Julia toolchain in the build image or on the GPU box (SURVEY.md section 8c); this file
# documents the binding a maintainer adds to BayesianLinearRegressors.jl.  The same symbols are exercised end
# to end through the Python ctypes binding (bayesianlinearregressors.jl_b200/_lib.py).
module LibBLR

using LinearAlgebra: PosDefException
using FillArrays: FillArrays

const libblr = get(ENV, "LIBBLR_CUDA", "libblr_cuda")

const COLVECS, ROWVECS = Cint(0), Cint(1)
const LAMBDA_DIAGONAL, LAMBDA_DENSE = Cint(0), Cint(1)
const NOISE_SCALAR, NOISE_VECTOR, NOISE_DENSE = Cint(0), Cint(1), Cint(2)
const E_DIM = Cint(-4)

struct Prior
    mw::Ptr{Float64}
    lambda_kind::Cint
    lambda::Ptr{Float64}
    ld::Int64
    D::Int64                # length(mw) = size(Λw, 1): validated by the library against size(X, 1) (BLR_E_DIM)
end

struct Noise
    kind::Cint
    scalar::Float64
    vec::Ptr{Cvoid}
    dense::Ptr{Float64}     # host N x N matrix when kind == NOISE_DENSE
    dense_ld::Int64
end
Noise(kind, scalar, vec) = Noise(kind, scalar, vec, C_NULL, 0)

mutable struct Context
    ptr::Ptr{Cvoid}
    function Context(device::Integer=0)
        r = Ref{Ptr{Cvoid}}(C_NULL)
        rc = ccall((:blr_ctx_create, libblr), Cint, (Ref{Ptr{Cvoid}}, Cint), r, device)
        rc == 0 || error("blr_ctx_create failed with code $rc (no sm_100 device? libblr_cuda has no CPU fallback)")
        ctx = new(r[])
        finalizer(c -> ccall((:blr_ctx_destroy, libblr), Cint, (Ptr{Cvoid},), c.ptr), ctx)
        return ctx
    end
end

const _ctx = Ref{Union{Nothing,Context}}(nothing)
default_context() = something(_ctx[], (_ctx[] = Context(); _ctx[]))

# Numerical form of the D x D phase and the factor applications (include/blr_cuda.h, blr_ctx_set_form):
#   :direct   -- chol(Λw + G), inverse-factor GEMMs in var / rand (default);
#   :whitened -- the package's own evaluation order (chol(Uw⁻ᵀ G Uw⁻¹ + I), T = Λεy.U * Uw, triangular solves in var / cov / rand).
const FORMS = Dict(:direct => Cint(0), :whitened => Cint(1))
function set_form!(ctx::Context, form::Symbol)
    check(ctx, ccall((:blr_ctx_set_form, libblr), Cint, (Ptr{Cvoid}, Cint), ctx.ptr, FORMS[form]))
    return ctx
end
function form(ctx::Context)
    r = Ref{Cint}(0)
    check(ctx, ccall((:blr_ctx_get_form, libblr), Cint, (Ptr{Cvoid}, Ref{Cint}), ctx.ptr, r))
    return r[] == 0 ? :direct : :whitened
end

# status -> Julia exception, preserving the reference's error behaviour
function check(ctx::Context, rc::Cint)
    rc == 0 && return nothing
    rc > 0 && throw(PosDefException(Int(rc)))                    # LAPACK-style info from the device Cholesky
    msg = unsafe_string(ccall((:blr_last_error, libblr), Cstring, (Ptr{Cvoid},), ctx.ptr))
    rc == E_DIM && occursin("length(y)", msg) && error("length(y) != size(fx.x.X, 2)")      # ErrorException (:74)
    rc == E_DIM && throw(DimensionMismatch(msg))                                             # X' * mw (:33)
    error("libblr_cuda error $rc: $msg")
end

# ---- device handles with finalizers ---------------------------------------------------------------
mutable struct DeviceX
    ptr::Ptr{Cvoid}
    ctx::Context
    D::Int
    N::Int
end
function upload_x(ctx::Context, X::StridedMatrix{Float64}, layout::Cint)
    D, N = layout == COLVECS ? size(X) : reverse(size(X))
    r = Ref{Ptr{Cvoid}}(C_NULL)
    GC.@preserve X check(ctx, ccall((:blr_x_upload, libblr), Cint,
        (Ptr{Cvoid}, Ptr{Float64}, Int64, Int64, Int64, Cint, Ref{Ptr{Cvoid}}),
        ctx.ptr, pointer(X), D, N, stride(X, 2), layout, r))
    x = DeviceX(r[], ctx, D, N)
    finalizer(h -> ccall((:blr_x_free, libblr), Cint, (Ptr{Cvoid}, Ptr{Cvoid}), h.ctx.ptr, h.ptr), x)
    return x
end

mutable struct DeviceVec
    ptr::Ptr{Cvoid}
    ctx::Context
end
function upload_vec(ctx::Context, v::StridedVector{Float64})
    r = Ref{Ptr{Cvoid}}(C_NULL)
    GC.@preserve v check(ctx, ccall((:blr_vec_upload, libblr), Cint,
        (Ptr{Cvoid}, Ptr{Float64}, Int64, Ref{Ptr{Cvoid}}), ctx.ptr, pointer(v), length(v), r))
    h = DeviceVec(r[], ctx)
    finalizer(h -> ccall((:blr_vec_free, libblr), Cint, (Ptr{Cvoid}, Ptr{Cvoid}), h.ctx.ptr, h.ptr), h)
    return h
end

mutable struct DevicePost
    ptr::Ptr{Cvoid}
    ctx::Context
end
_post(ctx, p) = (h = DevicePost(p, ctx);
    finalizer(h -> ccall((:blr_post_free, libblr), Cint, (Ptr{Cvoid}, Ptr{Cvoid}), h.ctx.ptr, h.ptr), h); h)

# fused posterior + logpdf  (replaces src/bayesian_linear_regression.jl:55-89)
function infer(ctx::Context, prior::Prior, x::DeviceX, y::DeviceVec, noise::Noise;
               want_T::Bool=false, want_post::Bool=true)
    D = x.D
    lp = Ref{Float64}(NaN)
    m = Vector{Float64}(undef, D)
    Λ = Matrix{Float64}(undef, D, D)
    T = want_T ? Matrix{Float64}(undef, D, D) : nothing
    h = Ref{Ptr{Cvoid}}(C_NULL)
    check(ctx, ccall((:blr_infer, libblr), Cint,
        (Ptr{Cvoid}, Ref{Prior}, Ptr{Cvoid}, Ptr{Cvoid}, Ref{Noise}, Ref{Float64}, Ptr{Float64}, Ptr{Float64},
         Ptr{Float64}, Ref{Ptr{Cvoid}}),
        ctx.ptr, prior, x.ptr, y.ptr, noise, lp, m, want_T ? T : C_NULL, Λ, h))
    return lp[], m, Λ, T, _post(ctx, h[])
end

# logpdf of the k columns of Y under one fx (AbstractGPs' logpdf(fx, Y::AbstractMatrix)): one Gram pass, one factorisation
function logpdf_multi(ctx::Context, prior::Prior, x::DeviceX, Y::Matrix{Float64}, noise::Noise)
    N, k = size(Y)
    Yd = upload_vec(ctx, vec(Y))                       # column-major N x k, ld = N
    p = Ref{Ptr{Float64}}(C_NULL)
    check(ctx, ccall((:blr_vec_device_ptr, libblr), Cint, (Ptr{Cvoid}, Ptr{Cvoid}, Ref{Ptr{Float64}}), ctx.ptr, Yd.ptr, p))
    out = Vector{Float64}(undef, k)
    GC.@preserve Yd check(ctx, ccall((:blr_logpdf_multi, libblr), Cint,
        (Ptr{Cvoid}, Ref{Prior}, Ptr{Cvoid}, Ptr{Float64}, Int64, Int64, Ref{Noise}, Ptr{Float64}),
        ctx.ptr, prior, x.ptr, p[], max(N, 1), k, noise, out))
    return out
end

# gradients of logpdf (blr_logpdf_grad): the per-observation ones land in library-owned device vectors and are downloaded;
# returns (logpdf, dX (shaped like the input matrix), dy, dσ² (a number for scalar noise), dmw, dΛw (vector for a Diagonal prior))
struct LogpdfGrads
    dmw::Ptr{Float64}
    dlambda::Ptr{Float64}
    dsigma2::Ptr{Float64}       # host, scalar noise
    dsigma2_dev::Ptr{Float64}   # device, vector noise
    dy_dev::Ptr{Float64}
    dX_dev::Ptr{Float64}
    ld_dX::Int64
end
function _alloc_vec(ctx::Context, n::Integer)
    r = Ref{Ptr{Cvoid}}(C_NULL)
    check(ctx, ccall((:blr_vec_alloc, libblr), Cint, (Ptr{Cvoid}, Int64, Ref{Ptr{Cvoid}}), ctx.ptr, n, r))
    h = DeviceVec(r[], ctx)
    finalizer(h -> ccall((:blr_vec_free, libblr), Cint, (Ptr{Cvoid}, Ptr{Cvoid}), h.ctx.ptr, h.ptr), h)
    p = Ref{Ptr{Float64}}(C_NULL)
    check(ctx, ccall((:blr_vec_device_ptr, libblr), Cint, (Ptr{Cvoid}, Ptr{Cvoid}, Ref{Ptr{Float64}}), ctx.ptr, h.ptr, p))
    return h, p[]
end
function _download(ctx::Context, h::DeviceVec, n::Integer)
    out = Vector{Float64}(undef, n)
    check(ctx, ccall((:blr_vec_download, libblr), Cint, (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Float64}), ctx.ptr, h.ptr, out))
    return out
end
function logpdf_grad(ctx::Context, prior::Prior, x::DeviceX, layout::Cint, y::DeviceVec, noise::Noise; diagonal::Bool)
    D, N = x.D, x.N
    lp, hX, _, dy, dσ², dmw, dΛ = logpdf_grad_dev(ctx, prior, x, layout, y, noise; diagonal=diagonal)
    dX = reshape(_download(ctx, hX, D * N), layout == COLVECS ? (D, N) : (N, D))
    return lp, dX, dy, dσ², dmw, dΛ
end

# the same with ∂/∂X left on the device: returns (logpdf, hX (the library-owned vector, keeps the buffer alive), pX (its device
# address, leading dimension D for ColVecs), dy, dσ², dmw, dΛw) -- what a feature-map rule hands to features_vjp
function logpdf_grad_dev(ctx::Context, prior::Prior, x::DeviceX, layout::Cint, y::DeviceVec, noise::Noise; diagonal::Bool)
    D, N = x.D, x.N
    dmw = Vector{Float64}(undef, D)
    dΛ = diagonal ? Vector{Float64}(undef, D) : Matrix{Float64}(undef, D, D)
    dσ²_host = Ref{Float64}(NaN)
    vector_noise = noise.kind == NOISE_VECTOR
    hX, pX = _alloc_vec(ctx, D * N)
    hy, py = _alloc_vec(ctx, N)
    hs, ps = vector_noise ? _alloc_vec(ctx, N) : (nothing, Ptr{Float64}(C_NULL))
    lp = Ref{Float64}(NaN)
    GC.@preserve dmw dΛ dσ²_host begin
        g = LogpdfGrads(pointer(dmw), pointer(dΛ), vector_noise ? C_NULL : Base.unsafe_convert(Ptr{Float64}, dσ²_host), ps, py, pX,
                        max(layout == COLVECS ? D : N, 1))
        check(ctx, ccall((:blr_logpdf_grad, libblr), Cint,
            (Ptr{Cvoid}, Ref{Prior}, Ptr{Cvoid}, Ptr{Cvoid}, Ref{Noise}, Ref{Float64}, Ref{LogpdfGrads}),
            ctx.ptr, prior, x.ptr, y.ptr, noise, lp, g))
    end
    dσ² = vector_noise ? _download(ctx, hs, N) : dσ²_host[]
    return lp[], hX, pX, _download(ctx, hy, N), dσ², dmw, dΛ
end

# vector-Jacobian product of ϕ(x) = scale * act(W x + b) (blr_x_features_vjp) for the cotangent at device address pdphi (D x N,
# leading dimension ld_dphi): returns (dW (D x d_in), db (D), dx (d_in x N))
function features_vjp(ctx::Context, xin::DeviceX, W::Matrix{Float64}, b::Vector{Float64}, act::Integer, scale::Float64,
                      pdphi::Ptr{Float64}, ld_dphi::Integer)
    D, din, N = size(W, 1), size(W, 2), xin.N
    dW = Matrix{Float64}(undef, D, din)
    db = Vector{Float64}(undef, D)
    hx, px = _alloc_vec(ctx, din * N)
    check(ctx, ccall((:blr_x_features_vjp, libblr), Cint,
        (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}, Int64, Cint, Float64, Ptr{Float64}, Int64, Ptr{Float64}, Ptr{Float64},
         Ptr{Float64}, Int64),
        ctx.ptr, xin.ptr, W, b, D, act, scale, pdphi, ld_dphi, dW, db, N > 0 ? px : C_NULL, max(din, 1)))
    dx = N > 0 ? reshape(_download(ctx, hx, din * N), din, N) : zeros(din, 0)
    return dW, db, dx
end

# gradients of Σ_j Δ_j logpdf(fx, Y[:, j]) (blr_logpdf_multi_grad): one call for all k columns; Δ is the cotangent of the k
# log densities.  Returns (dX (shaped like the input matrix), dY (N x k), dσ², dmw, dΛw), as logpdf_grad without the value.
function logpdf_multi_grad(ctx::Context, prior::Prior, x::DeviceX, layout::Cint, Y::Matrix{Float64}, noise::Noise,
                           Δ::Vector{Float64}; diagonal::Bool)
    D, N = x.D, x.N
    k = size(Y, 2)
    length(Δ) == k || throw(DimensionMismatch("length(Δ) != size(Y, 2)"))
    Yd = upload_vec(ctx, vec(Y))                       # column-major N x k, ld = N
    pY = Ref{Ptr{Float64}}(C_NULL)
    check(ctx, ccall((:blr_vec_device_ptr, libblr), Cint, (Ptr{Cvoid}, Ptr{Cvoid}, Ref{Ptr{Float64}}), ctx.ptr, Yd.ptr, pY))
    dmw = Vector{Float64}(undef, D)
    dΛ = diagonal ? Vector{Float64}(undef, D) : Matrix{Float64}(undef, D, D)
    dσ²_host = Ref{Float64}(NaN)
    vector_noise = noise.kind == NOISE_VECTOR
    hX, pX = _alloc_vec(ctx, D * N)
    hy, py = _alloc_vec(ctx, N * k)
    hs, ps = vector_noise ? _alloc_vec(ctx, N) : (nothing, Ptr{Float64}(C_NULL))
    GC.@preserve Yd Δ dmw dΛ dσ²_host begin
        g = LogpdfGrads(pointer(dmw), pointer(dΛ), vector_noise ? C_NULL : Base.unsafe_convert(Ptr{Float64}, dσ²_host), ps, py, pX,
                        max(layout == COLVECS ? D : N, 1))
        check(ctx, ccall((:blr_logpdf_multi_grad, libblr), Cint,
            (Ptr{Cvoid}, Ref{Prior}, Ptr{Cvoid}, Ptr{Float64}, Int64, Int64, Ref{Noise}, Ptr{Float64}, Ptr{Float64}, Ref{LogpdfGrads}),
            ctx.ptr, prior, x.ptr, pY[], max(N, 1), k, noise, Δ, C_NULL, g))
    end
    dX = reshape(_download(ctx, hX, D * N), layout == COLVECS ? (D, N) : (N, D))
    dσ² = vector_noise ? _download(ctx, hs, N) : dσ²_host[]
    return dX, reshape(_download(ctx, hy, N * k), N, k), dσ², dmw, dΛ
end

# the same from host arrays: blr_stats_create -> blr_stats_accumulate_host -> blr_stats_allreduce -> blr_infer_from_stats
function infer_host(ctx::Context, prior::Prior, X::StridedMatrix{Float64}, layout::Cint, y::Vector{Float64}, Σy;
                    want_T::Bool=false, chunk::Integer=1 << 16)
    D, N = layout == COLVECS ? size(X) : reverse(size(X))
    st = Ref{Ptr{Cvoid}}(C_NULL)
    check(ctx, ccall((:blr_stats_create, libblr), Cint, (Ptr{Cvoid}, Int64, Ref{Ptr{Cvoid}}), ctx.ptr, D, st))
    try
        d = Σy.diag
        scalar = d isa FillArrays.Fill
        σ² = scalar ? Float64[] : collect(Float64, d)
        mw = unsafe_wrap(Array, prior.mw, D)
        GC.@preserve X y σ² check(ctx, ccall((:blr_stats_accumulate_host, libblr), Cint,
            (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}, Int64, Int64, Int64, Cint, Ptr{Float64}, Cint, Float64,
             Ptr{Float64}, Int64),
            ctx.ptr, st[], mw, X, D, N, stride(X, 2), layout, y, scalar ? NOISE_SCALAR : NOISE_VECTOR,
            scalar ? Float64(first(d)) : 0.0, scalar ? C_NULL : pointer(σ²), chunk))
        check(ctx, ccall((:blr_stats_allreduce, libblr), Cint, (Ptr{Cvoid}, Ptr{Cvoid}), ctx.ptr, st[]))
        lp = Ref{Float64}(NaN)
        m = Vector{Float64}(undef, D)
        Λ = Matrix{Float64}(undef, D, D)
        T = want_T ? Matrix{Float64}(undef, D, D) : nothing
        h = Ref{Ptr{Cvoid}}(C_NULL)
        check(ctx, ccall((:blr_infer_from_stats, libblr), Cint,
            (Ptr{Cvoid}, Ref{Prior}, Ptr{Cvoid}, Ref{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ref{Ptr{Cvoid}}),
            ctx.ptr, prior, st[], lp, m, want_T ? T : C_NULL, Λ, h))
        return lp[], m, Λ, T, _post(ctx, h[])
    finally
        ccall((:blr_stats_free, libblr), Cint, (Ptr{Cvoid}, Ptr{Cvoid}), ctx.ptr, st[])
    end
end

function post_create(ctx::Context, prior::Prior, D::Integer)
    h = Ref{Ptr{Cvoid}}(C_NULL)
    check(ctx, ccall((:blr_post_create, libblr), Cint, (Ptr{Cvoid}, Ref{Prior}, Int64, Ref{Ptr{Cvoid}}),
        ctx.ptr, prior, D, h))
    return _post(ctx, h[])
end

function mean_var(ctx::Context, p::DevicePost, x::DeviceX, noise::Noise; mean::Bool=true, var::Bool=true)
    m = mean ? Vector{Float64}(undef, x.N) : nothing
    v = var ? Vector{Float64}(undef, x.N) : nothing
    check(ctx, ccall((:blr_mean_var, libblr), Cint,
        (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Cvoid}, Ref{Noise}, Ptr{Float64}, Ptr{Float64}),
        ctx.ptr, p.ptr, x.ptr, noise, mean ? m : C_NULL, var ? v : C_NULL))
    return m, v
end

function cov(ctx::Context, p::DevicePost, x::DeviceX, noise::Noise)
    C = Matrix{Float64}(undef, x.N, x.N)
    check(ctx, ccall((:blr_cov, libblr), Cint, (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Cvoid}, Ref{Noise}, Ptr{Float64}),
        ctx.ptr, p.ptr, x.ptr, noise, C))
    return C
end

function rand_finite(ctx::Context, p::DevicePost, x::DeviceX, noise::Noise, Zw::Matrix{Float64}, Zy::Matrix{Float64})
    S = size(Zw, 2)
    Y = Matrix{Float64}(undef, x.N, S)
    check(ctx, ccall((:blr_rand_finite, libblr), Cint,
        (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Cvoid}, Ref{Noise}, Int64, Ptr{Float64}, Ptr{Float64}, UInt64, Ptr{Float64}),
        ctx.ptr, p.ptr, x.ptr, noise, S, Zw, Zy, 0, Y))
    return Y
end

function rand_weights(ctx::Context, p::DevicePost, Z::Matrix{Float64})
    W = similar(Z)
    check(ctx, ccall((:blr_rand_weights, libblr), Cint,
        (Ptr{Cvoid}, Ptr{Cvoid}, Int64, Ptr{Float64}, UInt64, Ptr{Float64}), ctx.ptr, p.ptr, size(Z, 2), Z, 0, W))
    return W
end

function apply_weights(ctx::Context, x::DeviceX, w::Vector{Float64})
    out = Vector{Float64}(undef, x.N)
    check(ctx, ccall((:blr_apply_weights, libblr), Cint, (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}),
        ctx.ptr, x.ptr, w, out))
    return out
end




# ------------------------------------------------------------------------------------------------ several GPUs, one process
# (inside the module: uses Context, check, libblr, Prior, COLVECS, NOISE_VECTOR unqualified)
# One Context per device; observations are sharded over them (contiguous column blocks), each device accumulates the
# statistics of its shard, ONE grouped all-reduce sums them, every device then holds the same posterior
# (SURVEY.md section 8e).  UNEXECUTED -- see INTEGRATION.md.
struct MultiContext
    ctxs::Vector{Context}
end

function MultiContext(devices::AbstractVector{<:Integer})
    ctxs = [Context(Cint(d)) for d in devices]
    ptrs = [c.ptr for c in ctxs]
    rc = ccall((:blr_comm_init_all, libblr), Cint, (Ptr{Ptr{Cvoid}}, Cint), ptrs, length(ptrs))
    check(ctxs[1], rc)
    return MultiContext(ctxs)
end

"contiguous shard of 1:N owned by rank r (0-based) of P -- the same split as sharding.py / bench.py"
function shard_bounds(N::Integer, P::Integer, r::Integer)
    q, rem = divrem(N, P)
    lo = r * q + min(r, rem)
    return lo + 1, lo + q + (r < rem ? 1 : 0)
end

"posterior + logpdf of ColVecs data X (D x N) sharded over the devices of `mc`; returns (logpdf, m′, Λ′) from device 1.\nblr_stats_accumulate_host only ENQUEUES (it returns without synchronising), so the devices' copies and kernels overlap."
function infer_sharded(mc::MultiContext, prior::Prior, X::StridedMatrix{Float64}, y::Vector{Float64}, σ²::Vector{Float64},
                       mw::Vector{Float64})
    D, N = size(X)
    P = length(mc.ctxs)
    stats = Vector{Ptr{Cvoid}}(undef, P)
    for (r, ctx) in enumerate(mc.ctxs)
        lo, hi = shard_bounds(N, P, r - 1)
        st = Ref{Ptr{Cvoid}}(C_NULL)
        check(ctx, ccall((:blr_stats_create, libblr), Cint, (Ptr{Cvoid}, Int64, Ref{Ptr{Cvoid}}), ctx.ptr, D, st))
        Xr, yr, sr = view(X, :, lo:hi), view(y, lo:hi), view(σ², lo:hi)
        GC.@preserve X y σ² mw check(ctx, ccall((:blr_stats_accumulate_host, libblr), Cint,
            (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}, Int64, Int64, Int64, Cint, Ptr{Float64}, Cint, Float64,
             Ptr{Float64}, Int64),
            ctx.ptr, st[], mw, Xr, D, hi - lo + 1, stride(X, 2), COLVECS, yr, NOISE_VECTOR, 0.0, sr, 1 << 16))
        stats[r] = st[]
    end
    ptrs = [c.ptr for c in mc.ctxs]
    check(mc.ctxs[1], ccall((:blr_stats_allreduce_all, libblr), Cint, (Ptr{Ptr{Cvoid}}, Ptr{Ptr{Cvoid}}, Cint), ptrs, stats, P))
    lp = Ref{Float64}(NaN); m = Vector{Float64}(undef, D); Λ = Matrix{Float64}(undef, D, D)
    ctx = mc.ctxs[1]
    check(ctx, ccall((:blr_infer_from_stats, libblr), Cint,
        (Ptr{Cvoid}, Ref{Prior}, Ptr{Cvoid}, Ref{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Cvoid}),
        ctx.ptr, prior, stats[1], lp, m, C_NULL, Λ, C_NULL))
    for (r, c) in enumerate(mc.ctxs)
        ccall((:blr_stats_free, libblr), Cint, (Ptr{Cvoid}, Ptr{Cvoid}), c.ptr, stats[r])
    end
    return lp[], m, Λ
end

# ---- stream ordering for borrowed device buffers (CUDA.jl arrays wrapped with blr_x_wrap_device)
wait_stream(ctx::Context, stream::Ptr{Cvoid}) = check(ctx, ccall((:blr_ctx_wait_stream, libblr), Cint, (Ptr{Cvoid}, Ptr{Cvoid}), ctx.ptr, stream))
release_to_stream(ctx::Context, stream::Ptr{Cvoid}) = check(ctx, ccall((:blr_stream_wait_ctx, libblr), Cint, (Ptr{Cvoid}, Ptr{Cvoid}), ctx.ptr, stream))

end # module
