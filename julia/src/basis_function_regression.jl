# src/basis_function_regression.jl needs NO change: every FiniteBFR method forwards through
# `_to_finite_blr(fx) = fx.f.blr(fx.f.ϕ(fx.x), fx.Σy)` (:41) to the FiniteBLR methods replaced in
# bayesian_linear_regression.jl.  The only addition is a device-native feature map whose output stays resident
# on the GPU (BASELINE config 5): a ϕ that returns a ColVecs wrapping a device handle instead of a host matrix.
# UNEXECUTED -- see INTEGRATION.md.
struct RandomFourierFeatures
    W::Matrix{Float64}   # D x d_in
    b::Vector{Float64}   # D
end

struct DeviceColVecs <: AbstractVector{Vector{Float64}}
    x::LibBLR.DeviceX
end
Base.size(x::DeviceColVecs) = (x.x.N,)
_device_x(ctx, x::DeviceColVecs) = x.x

function (ϕ::RandomFourierFeatures)(x::ColVecs)
    ctx = LibBLR.default_context()
    xin = LibBLR.upload_x(ctx, x.X, LibBLR.COLVECS)
    r = Ref{Ptr{Cvoid}}(C_NULL)
    LibBLR.check(ctx, ccall((:blr_x_rff, LibBLR.libblr), Cint,
        (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}, Int64, Ref{Ptr{Cvoid}}),
        ctx.ptr, xin.ptr, ϕ.W, ϕ.b, size(ϕ.W, 1), r))
    h = LibBLR.DeviceX(r[], ctx, size(ϕ.W, 1), xin.N)
    finalizer(h -> ccall((:blr_x_free, LibBLR.libblr), Cint, (Ptr{Cvoid}, Ptr{Cvoid}), h.ctx.ptr, h.ptr), h)
    return DeviceColVecs(h)
end

# Any one-layer map  ϕ(x) = scale * act(W x + b)  evaluated by the library (blr_x_features); RandomFourierFeatures is
# act = :cos, scale = sqrt(2 / D).  `act` ∈ (:cos, :tanh, :relu, :identity, :sin).
struct AffineFeatures
    W::Matrix{Float64}   # D x d_in
    b::Vector{Float64}   # D
    act::Symbol
    scale::Float64
end
const _ACT = Dict(:cos => 0, :tanh => 1, :relu => 2, :identity => 3, :sin => 4)

function (ϕ::AffineFeatures)(x::ColVecs)
    ctx = LibBLR.default_context()
    size(ϕ.W, 2) == size(x.X, 1) || throw(DimensionMismatch("size(W, 2) != size(x, 1)"))
    xin = LibBLR.upload_x(ctx, x.X, LibBLR.COLVECS)
    r = Ref{Ptr{Cvoid}}(C_NULL)
    LibBLR.check(ctx, ccall((:blr_x_features, LibBLR.libblr), Cint,
        (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}, Int64, Cint, Float64, Ref{Ptr{Cvoid}}),
        ctx.ptr, xin.ptr, ϕ.W, ϕ.b, size(ϕ.W, 1), _ACT[ϕ.act], ϕ.scale, r))
    h = LibBLR.DeviceX(r[], ctx, size(ϕ.W, 1), xin.N)
    finalizer(h -> ccall((:blr_x_free, LibBLR.libblr), Cint, (Ptr{Cvoid}, Ptr{Cvoid}), h.ctx.ptr, h.ptr), h)
    return DeviceColVecs(h)
end

# An arbitrary ϕ written on CUDA.jl arrays: borrow its output (D x N CuMatrix{Float64}, column-major = ColVecs) without a copy.
# `stream` is the CUDA.jl stream ϕ ran on (CUDA.stream().handle): the library's stream is ordered after it before reading.
function device_colvecs(Φ_ptr::Ptr{Float64}, D::Integer, N::Integer, ld::Integer, stream::Ptr{Cvoid}; keep=nothing)
    ctx = LibBLR.default_context()
    r = Ref{Ptr{Cvoid}}(C_NULL)
    LibBLR.check(ctx, ccall((:blr_x_wrap_device, LibBLR.libblr), Cint,
        (Ptr{Cvoid}, Ptr{Float64}, Int64, Int64, Int64, Cint, Ref{Ptr{Cvoid}}), ctx.ptr, Φ_ptr, D, N, ld, LibBLR.COLVECS, r))
    LibBLR.wait_stream(ctx, stream)
    h = LibBLR.DeviceX(r[], ctx, D, N)
    finalizer(h -> (keep; ccall((:blr_x_free, LibBLR.libblr), Cint, (Ptr{Cvoid}, Ptr{Cvoid}), h.ctx.ptr, h.ptr)), h)  # `keep` pins the CuArray
    return DeviceColVecs(h)
end

# Gradients through the device feature maps: logpdf of a BasisFunctionRegressor over AffineFeatures / RandomFourierFeatures
# (what Zygote does through ϕ in the reference, e.g. RFF lengthscales W = Ω / ℓ by type-II maximum likelihood).  x is uploaded
# and ϕ(x) evaluated once; ∂ℓ/∂ϕ(x) stays on the device (LibBLR.logpdf_grad_dev) and one blr_x_features_vjp call maps it to
# ϕ.W, ϕ.b and x.X.  Tangents also for the regressor's mw and Λw, Σy and y, as the FiniteBLR rule.  UNEXECUTED, like the rest
# of this glue.
const _DeviceMap = Union{RandomFourierFeatures,AffineFeatures}
_act_scale(ϕ::RandomFourierFeatures) = (_ACT[:cos], sqrt(2.0 / size(ϕ.W, 1)))
_act_scale(ϕ::AffineFeatures) = (_ACT[ϕ.act], ϕ.scale)

function _features(ctx, ϕ::_DeviceMap, xin::LibBLR.DeviceX)
    act, scale = _act_scale(ϕ)
    r = Ref{Ptr{Cvoid}}(C_NULL)
    LibBLR.check(ctx, ccall((:blr_x_features, LibBLR.libblr), Cint,
        (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}, Int64, Cint, Float64, Ref{Ptr{Cvoid}}),
        ctx.ptr, xin.ptr, ϕ.W, ϕ.b, size(ϕ.W, 1), act, scale, r))
    h = LibBLR.DeviceX(r[], ctx, size(ϕ.W, 1), xin.N)
    finalizer(h -> ccall((:blr_x_free, LibBLR.libblr), Cint, (Ptr{Cvoid}, Ptr{Cvoid}), h.ctx.ptr, h.ptr), h)
    return h
end

function ChainRulesCore.rrule(::typeof(AbstractGPs.logpdf), fx::AbstractGPs.FiniteGP{<:BasisFunctionRegressor{<:Any,<:_DeviceMap},<:ColVecs},
                              y::AbstractVector{<:Real})
    ctx = LibBLR.default_context()
    ϕ, blr = fx.f.ϕ, fx.f.blr
    length(y) == length(fx.x) || throw(error("length(y) != size(fx.x.X, 2)"))
    size(ϕ.W, 2) == size(fx.x.X, 1) || throw(DimensionMismatch("size(W, 2) != size(x, 1)"))
    xin = LibBLR.upload_x(ctx, fx.x.X, LibBLR.COLVECS)
    Φ = _features(ctx, ϕ, xin)
    prior, keep1 = _prior(blr)
    yv = LibBLR.upload_vec(ctx, collect(Float64, y))
    noise, keep2 = _noise(ctx, fx.Σy)
    lp, hΦ, pΦ, dy, dσ², dmw, dΛ = GC.@preserve keep1 keep2 Φ yv LibBLR.logpdf_grad_dev(ctx, prior, Φ, LibBLR.COLVECS, yv, noise;
                                                                                          diagonal=blr.Λw isa Diagonal)
    act, scale = _act_scale(ϕ)
    dW, db, dx = GC.@preserve hΦ xin LibBLR.features_vjp(ctx, xin, ϕ.W, ϕ.b, act, scale, pΦ, size(ϕ.W, 1))
    function logpdf_features_pullback(Δ)
        Δ = ChainRulesCore.unthunk(Δ)
        Λ̄ = blr.Λw isa Diagonal ? ChainRulesCore.Tangent{typeof(blr.Λw)}(diag=Δ .* dΛ) : Δ .* dΛ
        Σ̄ = fx.Σy isa Diagonal{<:Real,<:FillArrays.Fill} ?
            ChainRulesCore.Tangent{typeof(fx.Σy)}(diag=ChainRulesCore.Tangent{typeof(fx.Σy.diag)}(value=Δ * dσ²)) :
            ChainRulesCore.Tangent{typeof(fx.Σy)}(diag=Δ .* dσ²)
        blr̄ = ChainRulesCore.Tangent{typeof(blr)}(mw=Δ .* dmw, Λw=Λ̄)
        ϕ̄ = ChainRulesCore.Tangent{typeof(ϕ)}(W=Δ .* dW, b=Δ .* db)
        f̄ = ChainRulesCore.Tangent{typeof(fx.f)}(blr=blr̄, ϕ=ϕ̄)
        x̄ = ChainRulesCore.Tangent{typeof(fx.x)}(X=Δ .* dx)
        return ChainRulesCore.NoTangent(), ChainRulesCore.Tangent{typeof(fx)}(f=f̄, x=x̄, Σy=Σ̄), Δ .* dy
    end
    return lp, logpdf_features_pullback
end
