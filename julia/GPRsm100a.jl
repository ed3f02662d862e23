# GPRsm100a.jl -- Julia glue binding libgpr_sm100a.so (include/gpr_sm100a.h) into
# srinix007/GaussianProcessRegression.jl.  EXPERIMENTAL, SOURCE ONLY: no `julia` binary exists in the build image, so
# this file has never been executed (it is desk-checked against the reference's type definitions, see the notes at
# each definition); the executed bindings of the same C ABI are the ctypes layer
# gaussianprocessregression.jl_b200/gpr_sm100a/_ffi.py, which mirrors it call for call, and the plain-C caller
# tests/cabi/test_cabi.c.
#
# Seam (SURVEY.md 8b): the reference's callers (train, update_sample!, cv_step!, predict*) only ever touch the
# non-allocating, cache-based API.  New cache types hold an opaque model handle; the methods below overload
#     update_cache!(tc, hp, md)                 src/cost.jl:74-111
#     loss(::MarginalLikelihood, md, tc)        src/cost.jl:113-117
#     grad!(dL, ::MarginalLikelihood, md, tc)   src/cost.jl:119-127
#     loss_grad! / log_loss_grad!               src/cost.jl:50-70   (one fused ccall)
#     update_cache!(pc, md)                     src/predict.jl:29-34
#     predict_mean! / predict!                  src/predict.jl:36-71, src/split_predict.jl:5-53
# and `loss_cache / grad_cache / loss_grad_cache / predict_cache` route a wrapped model to them, so
# `train(SM100(md), MarginalLikelihood(); method = ...)` and `predict(SM100(md), xp)` run unchanged.
module GPRsm100a

using GaussianProcessRegression
using LinearAlgebra
using Random
import GaussianProcessRegression: update_cache!, loss, grad!, loss_grad!, log_loss_grad!, loss_cache, grad_cache,
    loss_grad_cache, predict_cache, predict_mean!, predict!, AbstractGPRModel, AbstractLossCache, AbstractGradCache,
    AbstractPredictCache, AbstractKernel, MarginalLikelihood, SquaredExp, WhiteNoise, ComposedKernel, GPRModel, Cmap, get_sample

const LIB = get(ENV, "GPR_SM100A_LIB", "libgpr_sm100a")
const GPR_KERN_SE, GPR_KERN_NOISE = Cint(1), Cint(2)
const GPR_FETCH_U, GPR_FETCH_ALPHA, GPR_FETCH_KINV, GPR_FETCH_WT = Cint(0), Cint(1), Cint(2), Cint(3)

mutable struct Ctx
    h::Ptr{Cvoid}
    function Ctx(device::Integer = 0)
        r = Ref{Ptr{Cvoid}}(C_NULL)
        rc = ccall((:gpr_ctx_create, LIB), Cint, (Cint, Ref{Ptr{Cvoid}}), device, r)
        rc == 0 || error("gpr_ctx_create: ", unsafe_string(ccall((:gpr_last_error, LIB), Cstring, (Ptr{Cvoid},), C_NULL)))
        c = new(r[])
        finalizer(x -> ccall((:gpr_ctx_destroy, LIB), Cint, (Ptr{Cvoid},), x.h), c)
    end
end
const DEFAULT_CTX = Ref{Union{Nothing,Ctx}}(nothing)
ctx() = (DEFAULT_CTX[] === nothing && (DEFAULT_CTX[] = Ctx(0)); DEFAULT_CTX[])

function check(c::Ctx, rc::Cint, info::Int64 = 0)
    rc == 0 && return nothing
    rc == 1 && throw(PosDefException(info))          # cholesky!(...; check = true), src/cost.jl:77
    error("libgpr_sm100a: ", unsafe_string(ccall((:gpr_last_error, LIB), Cstring, (Ptr{Cvoid},), c.h)))
end

comp_types(::SquaredExp) = Cint[GPR_KERN_SE]
comp_types(K::ComposedKernel) = Cint[k isa WhiteNoise ? GPR_KERN_NOISE : GPR_KERN_SE for k in K.kernels]

"""
Wrapper that routes a GPRModel to the sm_100a caches (every field access is forwarded to the wrapped model).

The supertype carries the wrapped model's own parameters: `AbstractGPRModel{K<:AbstractKernel,T,P<:AbstractArray{T},
X<:AbstractArray{T}}` (src/models.jl:3-4) -- so the reference's trait dispatch works unaided on the wrapper:
`islog(::MarginalLikelihood, ::AbstractGPRModel{<:SquaredExp})` and `islog(::MarginalLikelihood,
md::AbstractGPRModel{<:ComposedKernel})` (src/cost.jl:4-8; the latter reads `md.covar.kernels`, forwarded below),
`train(md::AbstractModel, ...)` (src/train.jl:9-12), `predict(md::AbstractGPRModel, xp)` (src/predict.jl:6-25).
"""
struct SM100{K<:AbstractKernel,T,P<:AbstractArray{T},X<:AbstractArray{T,2},M<:GPRModel{K,T,P,X}} <: AbstractGPRModel{K,T,P,X}
    md::M
end
SM100(md::GPRModel{K,T,P,X}) where {K,T,P,X} = SM100{K,T,P,X,typeof(md)}(md)
Base.getproperty(s::SM100, f::Symbol) = f === :md ? getfield(s, :md) : getproperty(getfield(s, :md), f)
Base.propertynames(s::SM100) = (:md, propertynames(getfield(s, :md))...)
GaussianProcessRegression.get_sample(s::SM100) = get_sample(s.md)      # src/models.jl:39-45 is typed on GPRModel
# src/models.jl:6-16 prints size(getfield(md, f)) for every field and src/models.jl:47-49 calls typeof(md)(covar, hp, x, y):
# neither works on a one-field wrapper, so both are forwarded (cv_batch / cv_step build their fold models with `similar`)
Base.show(io::IO, m::MIME"text/plain", s::SM100) = (println(io, "SM100 wrapper of"); show(io, m, s.md))
Base.similar(s::SM100, hp, x, y) = SM100(similar(s.md, hp, x, y))

mutable struct Handle
    c::Ctx
    h::Ptr{Cvoid}
    x::Matrix{Float64}      # what the device holds: the reference reads md.x / md.y afresh at every call, and its callers
    y::Matrix{Float64}      # mutate them in place between calls (md.y .+= dy, src/update_model.jl:36; mdt.x .= ..., src/crossval.jl:27-30)
end
_ymat(y) = y isa AbstractVector ? reshape(y, :, 1) : y
function Handle(md)
    c = ctx()
    t = comp_types(md.covar)
    x = Matrix{Float64}(md.x)
    y = Matrix{Float64}(_ymat(md.y))
    r = Ref{Ptr{Cvoid}}(C_NULL)
    rc = ccall((:gpr_model_create, LIB), Cint,
        (Ptr{Cvoid}, Ptr{Cint}, Cint, Cint, Int64, Ptr{Float64}, Ptr{Float64}, Cint, Cint, Ref{Ptr{Cvoid}}),
        c.h, t, length(t), size(x, 1), size(x, 2), x, y, size(y, 2), md.train_axis, r)
    check(c, rc)
    h = Handle(c, r[], x, y)
    # The Handle keeps its Ctx reachable, but at process exit finalizers run in no particular order: the library
    # tolerates that (gpr_ctx_destroy releases the models it still owns; gpr_model_destroy on such a handle is a no-op).
    finalizer(o -> ccall((:gpr_model_destroy, LIB), Cint, (Ptr{Cvoid},), o.h), h)
end
"re-upload x / y when the caller changed them since the last call (O(N D) host compare; gpr_model_set_* drop the cached factor)"
function _sync!(h::Handle, md)
    if md.x != h.x
        copyto!(h.x, md.x)
        check(h.c, ccall((:gpr_model_set_x, LIB), Cint, (Ptr{Cvoid}, Ptr{Float64}), h.h, h.x))
    end
    y = _ymat(md.y)
    if y != h.y
        copyto!(h.y, y)
        check(h.c, ccall((:gpr_model_set_y, LIB), Cint, (Ptr{Cvoid}, Ptr{Float64}), h.h, h.y))
    end
    return nothing
end

struct SM100LossCache <: AbstractLossCache;    hp::Vector{Float64}; h::Handle; end
struct SM100GradCache <: AbstractGradCache;    hp::Vector{Float64}; h::Handle; end
struct SM100PredictCache <: AbstractPredictCache; h::Handle; end
struct SM100SplitPredictCache <: AbstractPredictCache; h::Handle; var_range::UnitRange{Int64}; end
SM100LossCache(md::SM100) = SM100LossCache(copy(md.params), Handle(md))
SM100GradCache(md::SM100) = SM100GradCache(copy(md.params), Handle(md))

# trait functions (src/cost.jl:10-12, src/predict.jl:1, src/split_predict.jl:1) dispatch on the wrapped model
# through the cache constructors: loss_cache(cost)(md) in src/train.jl:16,38,49,60,74 calls SM100*Cache(md::SM100)
GaussianProcessRegression.MllLossCache(md::SM100) = SM100LossCache(md)
GaussianProcessRegression.MllGradCache(md::SM100) = SM100GradCache(md)
predict_cache(::SM100, ::AbstractArray) = (md, xp) -> SM100PredictCache(Handle(md))
predict_cache(::SM100, ::Cmap) = (md, xp) -> SM100SplitPredictCache(Handle(md), 1:3)

function _update!(h::Handle, hp, want_inverse::Bool; ϵ = 1e-8)
    info = Ref{Int64}(0)
    rc = ccall((:gpr_update_cache, LIB), Cint, (Ptr{Cvoid}, Ptr{Float64}, Cint, Cdouble, Cint, Ref{Int64}),
        h.h, hp, length(hp), ϵ, want_inverse, info)
    check(h.c, rc, info[])
end
update_cache!(tc::SM100LossCache, hp, md) = (tc.hp .= hp; _sync!(tc.h, md); _update!(tc.h, tc.hp, false))
update_cache!(tc::SM100GradCache, hp, md) = (tc.hp .= hp; _sync!(tc.h, md); _update!(tc.h, tc.hp, true))
# md::AbstractGPRModel, not Any: an untyped md would be ambiguous with update_cache!(::AbstractPredictCache, ::AbstractGPRModel) (src/predict.jl:29)
update_cache!(pc::Union{SM100PredictCache,SM100SplitPredictCache}, md::AbstractGPRModel) =
    (_sync!(pc.h, md); _update!(pc.h, Vector{Float64}(md.params), false))

function loss(::MarginalLikelihood, md::SM100, tc::Union{SM100LossCache,SM100GradCache})
    F = Ref{Float64}(0.0)
    check(tc.h.c, ccall((:gpr_loss, LIB), Cint, (Ptr{Cvoid}, Ref{Float64}), tc.h.h, F))
    return F[]
end
function grad!(∇L, ::MarginalLikelihood, md::SM100, tc::SM100GradCache)
    check(tc.h.c, ccall((:gpr_grad, LIB), Cint, (Ptr{Cvoid}, Cint, Ptr{Float64}), tc.h.h, 0, ∇L))
    return nothing
end
# fused single-call forms of src/cost.jl:50-70 (Optim only_fg! contract: F / G may be `nothing`)
function _fg!(F, G, v, md, tc::SM100GradCache, logscale::Bool)
    _sync!(tc.h, md)
    f = Ref{Float64}(0.0); info = Ref{Int64}(0)
    rc = ccall((:gpr_nlml_grad, LIB), Cint,
        (Ptr{Cvoid}, Ptr{Float64}, Cint, Cint, Cdouble, Ptr{Float64}, Ptr{Float64}, Ref{Int64}),
        tc.h.h, v, length(v), logscale, 1e-8, F === nothing ? C_NULL : f, G === nothing ? C_NULL : G, info)
    check(tc.h.c, rc, info[])
    F === nothing ? nothing : f[]
end
loss_grad!(::MarginalLikelihood, F, G, hp, md::SM100, tc::SM100GradCache) = _fg!(F, G, hp, md, tc, false)
log_loss_grad!(::MarginalLikelihood, F, G, log_hp, md::SM100, tc::SM100GradCache) = _fg!(F, G, log_hp, md, tc, true)

"tc.kchol_base / tc.α / tc.K⁻¹ of the reference caches (test/test_loss.jl:46-48)"
function fetch(h::Handle, which::Cint, dims...)
    out = Array{Float64}(undef, dims...)
    check(h.c, ccall((:gpr_fetch, LIB), Cint, (Ptr{Cvoid}, Cint, Ptr{Float64}), h.h, which, out))
    out
end

function predict_mean!(μₚ, md::SM100, xp::AbstractMatrix, pc::SM100PredictCache)
    rc = ccall((:gpr_predict, LIB), Cint, (Ptr{Cvoid}, Ptr{Float64}, Int64, Cint, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}),
        pc.h.h, xp, size(xp, 2), xp === md.x, μₚ, C_NULL, C_NULL)
    check(pc.h.c, rc)
end
function predict!(μₚ, Σₚ::Diagonal, md::SM100, xp::AbstractMatrix, pc::SM100PredictCache)
    rc = ccall((:gpr_predict, LIB), Cint, (Ptr{Cvoid}, Ptr{Float64}, Int64, Cint, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}),
        pc.h.h, xp, size(xp, 2), xp === md.x, μₚ, Σₚ.diag, C_NULL)
    check(pc.h.c, rc)
end
function predict!(μₚ, Σₚ::AbstractMatrix, md::SM100, xp::AbstractMatrix, pc::SM100PredictCache)
    rc = ccall((:gpr_predict, LIB), Cint, (Ptr{Cvoid}, Ptr{Float64}, Int64, Cint, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}),
        pc.h.h, xp, size(xp, 2), xp === md.x, μₚ, C_NULL, Σₚ)
    check(pc.h.c, rc)
end
function predict_mean!(μₚ, md::SM100, xeq::Cmap, pc::SM100SplitPredictCache)       # src/split_predict.jl:5-19
    rc = ccall((:gpr_split_predict, LIB), Cint,
        (Ptr{Cvoid}, Ptr{Float64}, Int64, Ptr{Float64}, Int64, Int64, Int64, Ptr{Float64}, Ptr{Float64}),
        pc.h.h, xeq.xe, size(xeq.xe, 2), xeq.xq, size(xeq.xq, 2), 1, 0, μₚ, C_NULL)
    check(pc.h.c, rc)
end
function predict!(μₚ, Σₚ::Diagonal, md::SM100, xeq::Cmap, pc::SM100SplitPredictCache)
    rc = ccall((:gpr_split_predict, LIB), Cint,
        (Ptr{Cvoid}, Ptr{Float64}, Int64, Ptr{Float64}, Int64, Int64, Int64, Ptr{Float64}, Ptr{Float64}),
        pc.h.h, xeq.xe, size(xeq.xe, 2), xeq.xq, size(xeq.xq, 2), first(pc.var_range), last(pc.var_range), μₚ, Σₚ.diag)
    check(pc.h.c, rc)
end

# ---------------------------------------------------------------------------------------------------------
# Multi-GPU gradient cache (BASELINE.json config 5: N = 131072, 137 GB of FP64 K): K / U / K^-1 block-cyclic over
# `devices`, one Julia process drives all of them (gpr_mgpu_*, include/gpr_sm100a.h).  Drop-in for
# SM100GradCache in loss_grad! / log_loss_grad!; `train(SM100Multi(md; devices = 0:7), ...)` builds it (wrapper below).
# ---------------------------------------------------------------------------------------------------------
mutable struct MultiHandle
    mg::Ptr{Cvoid}
    h::Ptr{Cvoid}
end
struct SM100MultiGradCache <: AbstractGradCache
    hp::Vector{Float64}
    h::MultiHandle
    x::Matrix{Float64}      # snapshots: the distributed model is immutable, a changed md.x / md.y is an error, not a silent stale result
    y::Matrix{Float64}
end
function mcheck(h::MultiHandle, rc::Cint, info::Int64 = 0)
    rc == 0 && return nothing
    rc == 1 && throw(PosDefException(info))
    error("libgpr_sm100a: ", unsafe_string(ccall((:gpr_mgpu_last_error, LIB), Cstring, (Ptr{Cvoid},), h.mg)))
end
default_nb(md) = size(md.x, 2) >= 65536 ? 2048 : 1024      # block-column width (DESIGN.md 7: 2048 feeds the INT8 route at large N)
all_devices() = 0:(ccall((:gpr_device_count, LIB), Cint, ()) - 1)
"distributed model of `md` over `devices`: (handle, x snapshot, y snapshot)"
function _multi_model(md::GPRModel, devices, nb::Integer)
    devs = Cint.(collect(devices))
    mg = Ref{Ptr{Cvoid}}(C_NULL)
    rc = ccall((:gpr_mgpu_create, LIB), Cint, (Cint, Ptr{Cint}, Int64, Ref{Ptr{Cvoid}}), length(devs), devs, nb, mg)
    rc == 0 || error("gpr_mgpu_create: ", unsafe_string(ccall((:gpr_mgpu_last_error, LIB), Cstring, (Ptr{Cvoid},), C_NULL)))
    t = comp_types(md.covar)
    x = Matrix{Float64}(md.x)
    y = Matrix{Float64}(_ymat(md.y))
    h = Ref{Ptr{Cvoid}}(C_NULL)
    mh = MultiHandle(mg[], C_NULL)
    finalizer(mh) do o           # registered before the model exists: a failed model creation still releases the devices
        o.h == C_NULL || ccall((:gpr_mgpu_model_destroy, LIB), Cint, (Ptr{Cvoid},), o.h)
        ccall((:gpr_mgpu_destroy, LIB), Cint, (Ptr{Cvoid},), o.mg)
    end
    rc = ccall((:gpr_mgpu_model_create, LIB), Cint,
        (Ptr{Cvoid}, Ptr{Cint}, Cint, Cint, Int64, Ptr{Float64}, Ptr{Float64}, Cint, Cint, Ref{Ptr{Cvoid}}),
        mg[], t, length(t), size(x, 1), size(x, 2), x, y, size(y, 2), md.train_axis, h)
    mcheck(mh, rc)
    mh.h = h[]
    mh, x, y
end
SM100MultiGradCache(md::GPRModel; devices = all_devices(), nb::Integer = default_nb(md)) =
    SM100MultiGradCache(Vector{Float64}(md.params), _multi_model(md, devices, nb)...)
function _fg!(F, G, v, md, tc::SM100MultiGradCache, logscale::Bool)
    (md.x == tc.x && _ymat(md.y) == tc.y) || error("SM100MultiGradCache: x / y changed; build a new cache")
    f = Ref{Float64}(0.0); info = Ref{Int64}(0)
    rc = ccall((:gpr_mgpu_nlml_grad, LIB), Cint,
        (Ptr{Cvoid}, Ptr{Float64}, Cint, Cint, Cdouble, Ptr{Float64}, Ptr{Float64}, Ref{Int64}),
        tc.h.h, v, length(v), logscale, 1e-8, F === nothing ? C_NULL : f, G === nothing ? C_NULL : G, info)
    mcheck(tc.h, rc, info[])
    F === nothing ? nothing : f[]
end
loss_grad!(::MarginalLikelihood, F, G, hp, md, tc::SM100MultiGradCache) = _fg!(F, G, hp, md, tc, false)
log_loss_grad!(::MarginalLikelihood, F, G, log_hp, md, tc::SM100MultiGradCache) = _fg!(F, G, log_hp, md, tc, true)

"""
Wrapper that makes `train(SM100Multi(md; devices = 0:7), MarginalLikelihood(); method = LBFGS())` build the multi-GPU gradient
cache: `loss_grad_cache(cost)(md)` (src/train.jl:38,49) is `MllGradCache(md)`, overloaded below.  Same supertype parameters as
`SM100`, so `islog` (src/cost.jl:4-8) dispatches on the wrapped kernel.  First-order methods only (the distributed handle has no
loss-only path; use `SM100` for that).  `predict(SM100Multi(md; devices = 0:7), xp)` predicts on the same devices
(SM100MultiPredictCache below; SM100MultiSplitPredictCache for `xp::Cmap`).
"""
struct SM100Multi{K<:AbstractKernel,T,P<:AbstractArray{T},X<:AbstractArray{T,2},M<:GPRModel{K,T,P,X}} <: AbstractGPRModel{K,T,P,X}
    md::M
    devices::Vector{Cint}
    nb::Int
end
SM100Multi(md::GPRModel{K,T,P,X}; devices = all_devices(), nb::Integer = default_nb(md)) where {K,T,P,X} =
    SM100Multi{K,T,P,X,typeof(md)}(md, Cint.(collect(devices)), Int(nb))
Base.getproperty(s::SM100Multi, f::Symbol) = f in (:md, :devices, :nb) ? getfield(s, f) : getproperty(getfield(s, :md), f)
Base.propertynames(s::SM100Multi) = (:md, :devices, :nb, propertynames(getfield(s, :md))...)
Base.show(io::IO, m::MIME"text/plain", s::SM100Multi) = (println(io, "SM100Multi wrapper (devices ", Int.(s.devices), ") of"); show(io, m, s.md))
GaussianProcessRegression.get_sample(s::SM100Multi) = get_sample(s.md)
GaussianProcessRegression.MllGradCache(s::SM100Multi) = SM100MultiGradCache(s.md; devices = s.devices, nb = s.nb)

# Prediction on the distributed model (src/predict.jl:14-102): update_cache! forms K^-1 block-cyclic over the devices,
# gpr_mgpu_predict evaluates mean, Diagonal variance or dense covariance from it without a triangular solve.
struct SM100MultiPredictCache <: AbstractPredictCache
    h::MultiHandle
    x::Matrix{Float64}
    y::Matrix{Float64}
end
predict_cache(s::SM100Multi, ::AbstractArray) = (md, xp) -> SM100MultiPredictCache(_multi_model(s.md, s.devices, s.nb)...)
# split prediction on Cmap(+, xe, xq) grids (src/split_predict.jl:5-53): gpr_mgpu_split_predict shards the q columns over the devices
struct SM100MultiSplitPredictCache <: AbstractPredictCache
    h::MultiHandle
    x::Matrix{Float64}
    y::Matrix{Float64}
    var_range::UnitRange{Int64}
end
predict_cache(s::SM100Multi, ::Cmap) = (md, xp) -> SM100MultiSplitPredictCache(_multi_model(s.md, s.devices, s.nb)..., 1:3)
function update_cache!(pc::Union{SM100MultiPredictCache,SM100MultiSplitPredictCache}, md::AbstractGPRModel)
    (md.x == pc.x && _ymat(md.y) == pc.y) || error("SM100MultiPredictCache: x / y changed; build a new cache")
    hp = Vector{Float64}(md.params); info = Ref{Int64}(0)
    rc = ccall((:gpr_mgpu_update_cache, LIB), Cint, (Ptr{Cvoid}, Ptr{Float64}, Cint, Cdouble, Ref{Int64}),
        pc.h.h, hp, length(hp), 1e-8, info)
    mcheck(pc.h, rc, info[])
end
function _mpredict!(pc::SM100MultiPredictCache, md, xp, μₚ, var, Σ)
    rc = ccall((:gpr_mgpu_predict, LIB), Cint, (Ptr{Cvoid}, Ptr{Float64}, Int64, Cint, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}),
        pc.h.h, xp, size(xp, 2), xp === md.x, μₚ, var, Σ)
    mcheck(pc.h, rc)
end
function predict_mean!(μₚ, md::SM100Multi, xp::AbstractMatrix, pc::SM100MultiPredictCache)
    _mpredict!(pc, md, xp, μₚ, C_NULL, C_NULL)
end
function predict!(μₚ, Σₚ::Diagonal, md::SM100Multi, xp::AbstractMatrix, pc::SM100MultiPredictCache)
    _mpredict!(pc, md, xp, μₚ, Σₚ.diag, C_NULL)
end
function predict!(μₚ, Σₚ::AbstractMatrix, md::SM100Multi, xp::AbstractMatrix, pc::SM100MultiPredictCache)
    _mpredict!(pc, md, xp, μₚ, C_NULL, Σₚ)
end
function _msplit!(pc::SM100MultiSplitPredictCache, xeq::Cmap, e_lo, e_hi, μₚ, var)
    rc = ccall((:gpr_mgpu_split_predict, LIB), Cint,
        (Ptr{Cvoid}, Ptr{Float64}, Int64, Ptr{Float64}, Int64, Int64, Int64, Ptr{Float64}, Ptr{Float64}),
        pc.h.h, xeq.xe, size(xeq.xe, 2), xeq.xq, size(xeq.xq, 2), e_lo, e_hi, μₚ, var)
    mcheck(pc.h, rc)
end
function predict_mean!(μₚ, md::SM100Multi, xeq::Cmap, pc::SM100MultiSplitPredictCache)
    _msplit!(pc, xeq, 1, 0, μₚ, C_NULL)
end
function predict!(μₚ, Σₚ::Diagonal, md::SM100Multi, xeq::Cmap, pc::SM100MultiSplitPredictCache)
    _msplit!(pc, xeq, first(pc.var_range), last(pc.var_range), μₚ, Σₚ.diag)
end

# ---------------------------------------------------------------------------------------------------------
# sample(N::NormalDistribution) on the device (src/distributions.jl:30-35): the draws stay on the Julia side (rng),
# the factorization of `Sigma .+ 1e-7` and the product L * s + mu run in gpr_sample_mvn.
# update_sample! (src/update_model.jl), cv_batch / cv_step! (src/crossval.jl) need no binding of their own: they only
# call log_loss_grad! / update_cache! / predict! on the caches above.
# ---------------------------------------------------------------------------------------------------------
function sample_sm100(cov, θ::Vector{Float64}, x::Matrix{Float64}, μ::Vector{Float64}; rng = Xoshiro(1), c::Ctx = ctx())
    n = size(x, 2)
    z = randn(rng, n)
    out = Vector{Float64}(undef, n)
    t = comp_types(cov)
    info = Ref{Int64}(0)
    rc = ccall((:gpr_sample_mvn, LIB), Cint,
        (Ptr{Cvoid}, Ptr{Cint}, Cint, Cint, Ptr{Float64}, Ptr{Float64}, Int64, Cdouble, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ref{Int64}),
        c.h, t, length(t), size(x, 1), θ, x, n, 1e-7, z, μ, out, info)
    check(c, rc, info[])
    out
end

# ---------------------------------------------------------------------------------------------------------
# integrate(md, hp, a, b; sample_noise) on the device (src/integrate.jl:45-62,103-160).  sample_noise === nothing: one
# factorization.  Scalar / vector noise: the same mu_i, var_i from one shifted factorization per distinct noise level
# (the shift rides in the jitter argument of gpr_update_cache, divided by the number of non-noise components because
# every such component adds its own jitter, src/compose_covar.jl:53-55) instead of the eigendecomposition of :72-80.
# ---------------------------------------------------------------------------------------------------------
# The noise-level bookkeeping of both methods below: once(eps) factors at jitter eps and integrates every box, returning
# Iout (nbox x ny) and var (nbox).  Each distinct noise level is factored once; vectors a, b (single) give the shapes of the
# reference's integrate, matrices Iout nbox x ny and var nbox (nbox x ny with sample_noise).
function _integrate_levels(once, covar, nbox::Int, ny::Int, single::Bool, sample_noise)
    if sample_noise === nothing
        I, v = once(1e-8)
        return single ? (I[1, :], v) : (I, v)
    end
    nk = count(k -> !(k isa WhiteNoise), covar isa ComposedKernel ? covar.kernels : (covar,))
    if sample_noise isa Real
        I, v = once(1e-8 + sample_noise / nk)
        return single ? (I[1, :], fill(v[1], ny)) : (I, repeat(v, 1, ny))
    end
    Iout = Matrix{Float64}(undef, nbox, ny); var = similar(Iout)
    levels = Dict{Float64,Tuple{Matrix{Float64},Vector{Float64}}}()
    for (i, e) in enumerate(sample_noise)
        haskey(levels, e) || (levels[e] = once(1e-8 + e / nk))
        I, v = levels[e]
        Iout[:, i] = I[:, i]; var[:, i] = v
    end
    single ? (Iout[1, :], var[1, :]) : (Iout, var)
end

# a, b vectors: gpr_integrate for the one box; D x nbox matrices (box i = column i): gpr_integrate_batch for all boxes at
# once, one triangular solve per tile of boxes instead of one per box.
function _integrate_once(h::Handle, hp::Vector{Float64}, a::VecOrMat{Float64}, b::VecOrMat{Float64}, eps::Float64, ny::Int)
    info = Ref{Int64}(0)
    check(h.c, ccall((:gpr_update_cache, LIB), Cint, (Ptr{Cvoid}, Ptr{Float64}, Cint, Cdouble, Cint, Ref{Int64}),
        h.h, hp, length(hp), eps, 0, info), info[])
    nbox = size(a, 2)
    Iout = Matrix{Float64}(undef, nbox, ny); v = Vector{Float64}(undef, nbox)
    if a isa Vector
        check(h.c, ccall((:gpr_integrate, LIB), Cint, (Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}),
            h.h, a, b, Iout, v))
    else
        check(h.c, ccall((:gpr_integrate_batch, LIB), Cint,
            (Ptr{Cvoid}, Int64, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}), h.h, nbox, a, b, Iout, v))
    end
    Iout, v
end
function integrate_sm100(md::GPRModel, hp, a, b; sample_noise = nothing)
    h = Handle(md)                       # device model (x, y uploaded once), freed by its finalizer
    ny = size(md.y, 2)
    single = a isa AbstractVector
    hpv = Vector{Float64}(hp)
    av, bv = single ? (Vector{Float64}(a), Vector{Float64}(b)) : (Matrix{Float64}(a), Matrix{Float64}(b))
    _integrate_levels(eps -> _integrate_once(h, hpv, av, bv, eps, ny), md.covar, size(av, 2), ny, single, sample_noise)
end

# The same on the distributed model of SM100Multi: one gpr_mgpu_update_cache per distinct noise level, then
# gpr_mgpu_integrate for all boxes at once (a, b: vectors or D x nbox matrices, box i = column i) in one pass over K^-1.
# Vectors give the results of the single-device method; matrices give Iout nbox x ny and var nbox (nbox x ny with sample_noise).
function _mintegrate_once(h::MultiHandle, hp::Vector{Float64}, a::Matrix{Float64}, b::Matrix{Float64}, eps::Float64, ny::Int)
    info = Ref{Int64}(0)
    mcheck(h, ccall((:gpr_mgpu_update_cache, LIB), Cint, (Ptr{Cvoid}, Ptr{Float64}, Cint, Cdouble, Ref{Int64}),
        h.h, hp, length(hp), eps, info), info[])
    nbox = size(a, 2)
    Iout = Matrix{Float64}(undef, nbox, ny); v = Vector{Float64}(undef, nbox)
    mcheck(h, ccall((:gpr_mgpu_integrate, LIB), Cint, (Ptr{Cvoid}, Int64, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}),
        h.h, nbox, a, b, Iout, v))
    Iout, v
end
function integrate_sm100(s::SM100Multi, hp, a, b; sample_noise = nothing)
    h, _, _ = _multi_model(s.md, s.devices, s.nb)
    ny = size(s.md.y, 2)
    hpv = Vector{Float64}(hp)
    am = Matrix{Float64}(reshape(a, size(a, 1), :)); bm = Matrix{Float64}(reshape(b, size(b, 1), :))
    _integrate_levels(eps -> _mintegrate_once(h, hpv, am, bm, eps, ny), s.md.covar, size(am, 2), ny, a isa AbstractVector,
                      sample_noise)
end

end # module
