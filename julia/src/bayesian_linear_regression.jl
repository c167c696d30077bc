# Drop-in replacement for the method bodies of BayesianLinearRegressors.jl/src/bayesian_linear_regression.jl:33-93.
# The struct, the FiniteBLR alias, x_as_colvecs and every signature are unchanged; only the bodies dispatch to
# libblr_cuda.  UNEXECUTED (no Julia in the build image) -- see INTEGRATION.md.
using .LibBLR: LibBLR
using ChainRulesCore: ChainRulesCore      # a dependency of AbstractGPs

# layout + device upload of whatever x_as_colvecs accepts (:20-31); errors for unknown vectors are preserved.
_device_x(ctx, x::ColVecs) = LibBLR.upload_x(ctx, x.X, LibBLR.COLVECS)
_device_x(ctx, x::RowVecs) = LibBLR.upload_x(ctx, x.X, LibBLR.ROWVECS)      # feature-major read in place: no transpose copy
_device_x(ctx, x::AbstractVector) = x_as_colvecs(x)                           # -> the reference's ErrorException

# Λw kinds (:11-14): Diagonal is sent as its diagonal, everything else as the dense symmetric matrix.
_prior(f::BayesianLinearRegressor{<:Any,<:Diagonal}) =
    (mw = collect(Float64, f.mw); λ = collect(Float64, f.Λw.diag);
     (LibBLR.Prior(pointer(mw), LibBLR.LAMBDA_DIAGONAL, pointer(λ), length(mw), length(mw)), (mw, λ)))
_prior(f::BayesianLinearRegressor) =
    (mw = collect(Float64, f.mw); Λ = Matrix{Float64}(f.Λw);
     (LibBLR.Prior(pointer(mw), LibBLR.LAMBDA_DENSE, pointer(Λ), size(Λ, 1), length(mw)), (mw, Λ)))

# Device-resident factorisation cached per regressor (the reference re-runs `_cholesky(Λw)` on every predict call, :36,:41,:51;
# model.py keeps the handle in the Python object).  The Julia struct is immutable and unchanged, so the handle lives in a
# weak-keyed side table: key = the (mutable) array behind Λw, value = (copy of mw, DevicePost).  `posterior` registers the
# handle blr_infer returned, so mean / var / cov / rand on a posterior never factorise again.
const _POST_CACHE = WeakKeyDict{Any,Tuple{Vector{Float64},LibBLR.DevicePost}}()
_cache_key(Λ::Diagonal) = Λ.diag
_cache_key(Λ::Symmetric) = parent(Λ)
_cache_key(Λ::AbstractPDMat) = Λ.mat
_cache_key(Λ::AbstractMatrix) = Λ
function _device_post(ctx, f::BayesianLinearRegressor)
    key = _cache_key(f.Λw)
    hit = get(_POST_CACHE, key, nothing)
    hit !== nothing && hit[2].ctx === ctx && hit[1] == f.mw && return hit[2]
    prior, keep = _prior(f)
    p = GC.@preserve keep LibBLR.post_create(ctx, prior, length(f.mw))
    ismutable(key) && (_POST_CACHE[key] = (collect(Float64, f.mw), p))
    return p
end

# Σy kinds of FiniteGP: Diagonal(Fill) -> scalar, Diagonal(v) -> device vector, dense -> small-N whitening side path.
function _noise(ctx, Σy::AbstractMatrix)
    S = Matrix{Float64}(Σy)
    return LibBLR.Noise(LibBLR.NOISE_DENSE, 0.0, C_NULL, pointer(S), size(S, 1)), S
end
_noise(ctx, Σy::Diagonal{<:Real,<:FillArrays.Fill}) = (LibBLR.Noise(LibBLR.NOISE_SCALAR, first(Σy.diag), C_NULL), nothing)
function _noise(ctx, Σy::Diagonal)
    v = LibBLR.upload_vec(ctx, collect(Float64, Σy.diag))
    return LibBLR.Noise(LibBLR.NOISE_VECTOR, 0.0, v.ptr), v
end

function _infer(fx::FiniteBLR, y::AbstractVector{<:Real}; want_T::Bool)
    ctx = LibBLR.default_context()
    length(y) == length(fx.x) || throw(error("length(y) != size(fx.x.X, 2)"))            # :74
    prior, keep1 = _prior(fx.f)
    if fx.Σy isa Diagonal && fx.x isa Union{ColVecs,RowVecs} && fx.x.X isa StridedMatrix{Float64}
        # host arrays are streamed to the device in chunks (PCIe overlapped with the Gram kernel); no second copy of X
        return GC.@preserve keep1 LibBLR.infer_host(ctx, prior, fx.x.X, fx.x isa ColVecs ? LibBLR.COLVECS : LibBLR.ROWVECS,
                                                    collect(Float64, y), fx.Σy; want_T=want_T)
    end
    x = _device_x(ctx, fx.x)                                                              # dense Σy, lazy / non-strided inputs
    yv = LibBLR.upload_vec(ctx, collect(Float64, y))
    noise, keep2 = _noise(ctx, fx.Σy)
    GC.@preserve keep1 keep2 x yv LibBLR.infer(ctx, prior, x, yv, noise; want_T=want_T)
end

AbstractGPs.logpdf(fx::FiniteBLR, y::AbstractVector{<:Real}) = _infer(fx, y; want_T=false)[1]     # :55-58
# AbstractGPs' generic `logpdf(fx, Y::AbstractMatrix)` maps the vector method over the columns, i.e. one full
# __compute_inference_quantities (:72-89) per column; only δy (:84) depends on y, so the device runs the Gram pass and the
# factorisation once for all columns (blr_logpdf_multi).  Dense Σy keeps the per-column loop (small-N side path).
function AbstractGPs.logpdf(fx::FiniteBLR, Y::AbstractMatrix{<:Real})
    size(Y, 1) == length(fx.x) || throw(error("length(y) != size(fx.x.X, 2)"))            # :74
    fx.Σy isa Diagonal || return [AbstractGPs.logpdf(fx, collect(Float64, c)) for c in eachcol(Y)]
    ctx = LibBLR.default_context()
    x = _device_x(ctx, fx.x)
    prior, keep1 = _prior(fx.f)
    noise, keep2 = _noise(ctx, fx.Σy)
    GC.@preserve keep1 keep2 x LibBLR.logpdf_multi(ctx, prior, x, Matrix{Float64}(Y), noise)
end

# Reverse-mode rule for logpdf (:55-58): Zygote cannot enter the ccall above, so the gradients come in closed form from the
# device (blr_logpdf_grad, one call for the value and every tangent).  Tangents for fx.f.mw, fx.f.Λw (the diagonal of a
# Diagonal, else the symmetric D x D G with dℓ = <G, dΛw>), fx.x.X (ColVecs or RowVecs), fx.Σy (Diagonal(Fill) or Diagonal)
# and y.  Dense Σy has no rule (the library returns an error).
function ChainRulesCore.rrule(::typeof(AbstractGPs.logpdf), fx::FiniteBLR, y::AbstractVector{<:Real})
    ctx = LibBLR.default_context()
    length(y) == length(fx.x) || throw(error("length(y) != size(fx.x.X, 2)"))            # :74
    prior, keep1 = _prior(fx.f)
    x = _device_x(ctx, fx.x)
    yv = LibBLR.upload_vec(ctx, collect(Float64, y))
    noise, keep2 = _noise(ctx, fx.Σy)
    layout = fx.x isa ColVecs ? LibBLR.COLVECS : LibBLR.ROWVECS
    lp, dX, dy, dσ², dmw, dΛ = GC.@preserve keep1 keep2 x yv LibBLR.logpdf_grad(ctx, prior, x, layout, yv, noise;
                                                                                  diagonal=fx.f.Λw isa Diagonal)
    function logpdf_pullback(Δ)
        Δ = ChainRulesCore.unthunk(Δ)
        Λ̄ = fx.f.Λw isa Diagonal ? ChainRulesCore.Tangent{typeof(fx.f.Λw)}(diag=Δ .* dΛ) : Δ .* dΛ
        Σ̄ = fx.Σy isa Diagonal{<:Real,<:FillArrays.Fill} ?
            ChainRulesCore.Tangent{typeof(fx.Σy)}(diag=ChainRulesCore.Tangent{typeof(fx.Σy.diag)}(value=Δ * dσ²)) :
            ChainRulesCore.Tangent{typeof(fx.Σy)}(diag=Δ .* dσ²)
        f̄ = ChainRulesCore.Tangent{typeof(fx.f)}(mw=Δ .* dmw, Λw=Λ̄)
        x̄ = ChainRulesCore.Tangent{typeof(fx.x)}(X=Δ .* dX)
        return ChainRulesCore.NoTangent(), ChainRulesCore.Tangent{typeof(fx)}(f=f̄, x=x̄, Σy=Σ̄), Δ .* dy
    end
    return lp, logpdf_pullback
end

# The same rule for the matrix method above (k observation vectors, one per column of Y): the primal is that method
# (blr_logpdf_multi); the cotangent Δ of the k values is not known until the pullback, which makes ONE blr_logpdf_multi_grad
# call with the weights Δ (re-running the Gram pass) -- the gradients of Σ_j Δ_j logpdf_j, in the tangent structure of the
# vector rule.  Dense Σy: the pullback raises the library's error.
function ChainRulesCore.rrule(::typeof(AbstractGPs.logpdf), fx::FiniteBLR, Y::AbstractMatrix{<:Real})
    lps = AbstractGPs.logpdf(fx, Y)
    function logpdf_multi_pullback(Δ)
        Δ = collect(Float64, ChainRulesCore.unthunk(Δ))
        ctx = LibBLR.default_context()
        prior, keep1 = _prior(fx.f)
        x = _device_x(ctx, fx.x)
        noise, keep2 = _noise(ctx, fx.Σy)
        layout = fx.x isa ColVecs ? LibBLR.COLVECS : LibBLR.ROWVECS
        dX, dY, dσ², dmw, dΛ = GC.@preserve keep1 keep2 x LibBLR.logpdf_multi_grad(ctx, prior, x, layout, Matrix{Float64}(Y), noise,
                                                                                      Δ; diagonal=fx.f.Λw isa Diagonal)
        Λ̄ = fx.f.Λw isa Diagonal ? ChainRulesCore.Tangent{typeof(fx.f.Λw)}(diag=dΛ) : dΛ
        Σ̄ = fx.Σy isa Diagonal{<:Real,<:FillArrays.Fill} ?
            ChainRulesCore.Tangent{typeof(fx.Σy)}(diag=ChainRulesCore.Tangent{typeof(fx.Σy.diag)}(value=dσ²)) :
            ChainRulesCore.Tangent{typeof(fx.Σy)}(diag=dσ²)
        f̄ = ChainRulesCore.Tangent{typeof(fx.f)}(mw=dmw, Λw=Λ̄)
        x̄ = ChainRulesCore.Tangent{typeof(fx.x)}(X=dX)
        return ChainRulesCore.NoTangent(), ChainRulesCore.Tangent{typeof(fx)}(f=f̄, x=x̄, Σy=Σ̄), dY
    end
    return lps, logpdf_multi_pullback
end

function AbstractGPs.posterior(fx::FiniteBLR, y::AbstractVector{<:Real})                           # :60-69
    _, m′, Λ′, T, p = _infer(fx, y; want_T=fx.f.Λw isa AbstractPDMat)
    _POST_CACHE[Λ′] = (copy(m′), p)          # the returned regressor carries its device factor (keyed by its Λ′ array)
    return BayesianLinearRegressor(m′, __build_Λ(typeof(fx.f.Λw), Λ′, T))
end
__build_Λ(_, Λ′, _) = Symmetric(Λ′)                                                                # :92
__build_Λ(::Type{<:AbstractPDMat}, Λ′, T) = PDMat(Λ′, Cholesky(UpperTriangular(T)))                 # :93

function _predict(fx::FiniteBLR; mean::Bool, var::Bool)
    ctx = LibBLR.default_context()
    x = _device_x(ctx, fx.x)
    size(fx.x isa RowVecs ? fx.x.X' : fx.x.X, 1) == length(fx.f.mw) || throw(DimensionMismatch("size(X, 1) != length(mw)"))
    noise, keep2 = _noise(ctx, fx.Σy)
    GC.@preserve keep2 LibBLR.mean_var(ctx, _device_post(ctx, fx.f), x, noise; mean=mean, var=var)
end
AbstractGPs.mean(fx::FiniteBLR) = _predict(fx; mean=true, var=false)[1]                            # :33
AbstractGPs.var(fx::FiniteBLR) = _predict(fx; mean=false, var=true)[2]                             # :40-43
AbstractGPs.mean_and_var(fx::FiniteBLR) = _predict(fx; mean=true, var=true)                        # :47

function AbstractGPs.cov(fx::FiniteBLR)                                                            # :35-38
    ctx = LibBLR.default_context()
    x = _device_x(ctx, fx.x)
    noise, keep2 = _noise(ctx, fx.Σy)
    GC.@preserve keep2 Symmetric(LibBLR.cov(ctx, _device_post(ctx, fx.f), x, noise))
end
AbstractGPs.mean_and_cov(fx::FiniteBLR) = (mean(fx), cov(fx))                                      # :45

function AbstractGPs.rand(rng::AbstractRNG, fx::FiniteBLR, samples::Int)                           # :49-53
    ctx = LibBLR.default_context()
    x = _device_x(ctx, fx.x)
    Zw = randn(rng, length(fx.f.mw), samples)          # drawn FIRST (:51)
    Zy = randn(rng, length(fx.x), samples)             # drawn SECOND (:52)
    noise, keep2 = _noise(ctx, fx.Σy)
    GC.@preserve keep2 LibBLR.rand_finite(ctx, _device_post(ctx, fx.f), x, noise, Zw, Zy)
end
