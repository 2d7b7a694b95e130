# GPB200.jl -- the reference-side binding: a `CovarianceStrategy` whose methods `ccall` libgpb200.so.
#
# Drop-in behind GaussianProcesses.jl's own strategy seam (src/GP.jl:10); no edit to the reference's
# source is needed.  Usage:
#
#     using GaussianProcesses, GPB200
#     gp = GPE(x, y, MeanConst(0.0), SEIso(0.3, 0.3), 0.3, B200Covariance())   # src/GPE.jl:68
#     optimize!(gp); predict_f(gp, xtest)
#
# Julia is not installed in the build image, so this file is the *specification* of the binding a
# maintainer adds (INTEGRATION.md); the executable twin used by the tests is
# gaussianprocesses.jl_b200/gpb200/{capi,gpe}.py, which drives the identical C ABI (include/gpb200.h).
module GPB200

using GaussianProcesses
using LinearAlgebra
using PDMats
import Random
import GaussianProcesses: CovarianceStrategy, KernelData, EmptyData, alloc_cK, update_cK!, init_precompute,
                          precompute!, dmll_kern!, dmll_noise, predictMVN, predict_f, predict_full,
                          AbstractGradientPrecompute, Kernel, Mean, GPE, get_params, num_params, mean,
                          SumKernel, ProdKernel, Masked, FixedKernel, update_target!, get_value,
                          predict_LOO, predict_CVfold, dlogpdθ_LOO, dlogpdθ_CVfold, Folds
using ElasticArrays: ElasticArray
import PDMats: AbstractPDMat, dim
import Base: \, size, Matrix
import LinearAlgebra: logdet, tr

const LIB = get(ENV, "GPB200_LIB", "libgpb200.so")

# opcodes of include/gpb200.h
const OP = Dict(SEIso => 1, SEArd => 2, Mat12Iso => 3, Mat32Iso => 4, Mat52Iso => 5, Mat12Ard => 6, Mat32Ard => 7,
                Mat52Ard => 8, RQIso => 9, RQArd => 10, Periodic => 11, LinIso => 12, LinArd => 13, Poly => 14,
                Noise => 15, Const => 16)
const OP_SUM, OP_PROD = 32, 33

struct B200Covariance <: CovarianceStrategy
    device::Int
    capacity::Int                 # rows reserved on the device for append! (0: exactly nobs) -- ElasticCovStrat, GPEelastic.jl:3-6
    stepsize::Int                 # extra rows reserved whenever append! outgrows the reservation
end
B200Covariance(device::Int = 0; capacity::Int = 0, stepsize::Int = 10^3) = B200Covariance(device, capacity, stepsize)

mutable struct B200PDMat <: AbstractPDMat{Float64}
    handle::Ptr{Cvoid}
    n::Int
    exposed::Vector{Int}          # positions of get_params(kernel) inside the device's full theta
    ntheta::Int                   # length of the device's full parameter vector (FixedKernel may hide some)
    xid::UInt                     # objectid of the x last uploaded (skip the H2D copy while it is unchanged)
    xsize::Tuple{Int,Int}
    ops::Vector{Int32}            # kernel program last sent (skip gpb200_set_kernel while the tree shape is unchanged)
    dims::Vector{Int32}
    capacity::Int                 # rows reserved on the device (option "capacity"); append! extends in place below it
    function B200PDMat(device::Int, n::Int, capacity::Int = 0)
        h = Ref{Ptr{Cvoid}}(C_NULL)
        rc = ccall((:gpb200_create, LIB), Cint, (Ref{Ptr{Cvoid}}, Cint), h, device)
        rc == 0 || error("gpb200_create: ", unsafe_string(ccall((:gpb200_last_error, LIB), Cstring, (Ptr{Cvoid},), C_NULL)))
        obj = new(h[], n, Int[], 0, UInt(0), (0, 0), Int32[], Int32[], capacity)
        if capacity > 0
            ccall((:gpb200_set_option, LIB), Cint, (Ptr{Cvoid}, Cstring, Int64), h[], "capacity", capacity)
        end
        finalizer(o -> ccall((:gpb200_destroy, LIB), Cvoid, (Ptr{Cvoid},), o.handle), obj)
        return obj
    end
end

# precompute!(pre, gp) runs the inverse AND the fused trace once; dmll_kern! / dmll_noise read the cached result
mutable struct B200Precompute <: AbstractGradientPrecompute
    g::Vector{Float64}            # full kernel gradient (device parameter order)
    trA::Float64                  # tr(alpha alpha' - K_y^-1)
    exposed::Vector{Int}
end
B200Precompute() = B200Precompute(Float64[], NaN, Int[])

# error convention of include/gpb200.h -> the exceptions optimize!/mcmc filter (src/optimize.jl:46-87)
function check(cK::B200PDMat, rc::Integer, what)
    rc == 0 && return
    rc > 0 && throw(PosDefException(rc))
    msg = unsafe_string(ccall((:gpb200_last_error, LIB), Cstring, (Ptr{Cvoid},), cK.handle))
    (rc == -1 || rc == -4) && throw(ArgumentError("$what: $msg"))
    error("$what failed ($rc): $msg")
end

# ---- kernel tree -> post-order program (Masked folded into dims, FixedKernel into `exposed`) ----
function emit!(ops, dims, theta, k::Kernel, active::Vector{Int})
    if k isa SumKernel || k isa ProdKernel
        el = emit!(ops, dims, theta, k.kleft, active)
        er = emit!(ops, dims, theta, k.kright, active)
        append!(ops, Int32[k isa SumKernel ? OP_SUM : OP_PROD, 0, 0, 0, 0, 0])
        return vcat(el, er)
    elseif k isa Masked
        return emit!(ops, dims, theta, k.kernel, active[collect(k.active_dims)])
    elseif k isa FixedKernel
        e = emit!(ops, dims, theta, k.kernel, active)
        return e[collect(k.free)]
    else
        p = get_params(k)
        toff, doff = length(theta), length(dims)
        append!(theta, p); append!(dims, Int32.(active .- 1))
        extra = k isa Poly ? k.deg : 0
        append!(ops, Int32[OP[Base.typename(typeof(k)).wrapper], toff, length(p), doff, length(active), extra])
        return collect(toff+1:toff+length(p))
    end
end

function flatten(kernel::Kernel, d::Int)
    ops, dims, theta = Int32[], Int32[], Float64[]
    exposed = emit!(ops, dims, theta, kernel, collect(1:d))
    return ops, dims, theta, exposed
end

# ---- strategy methods (SURVEY.md §8(b); exemplar src/sparse/subsetofregressors.jl) --------------
KernelData(k::Kernel, X1::AbstractMatrix, X2::AbstractMatrix, ::B200Covariance) = EmptyData()   # no N x N host cache

alloc_cK(cs::B200Covariance, nobs) = B200PDMat(cs.device, nobs, cs.capacity)                               # src/GP.jl:14-20

size(a::B200PDMat) = (a.n, a.n)
size(a::B200PDMat, i::Int) = a.n
dim(a::B200PDMat) = a.n

# update_cK! (src/GPE.jl:169-186).  Two methods, typed like the reference's pair (logNoise::Real / ::AbstractVector)
# so that they are strictly more specific than update_cK!(::AbstractPDMat, ..., ::CovarianceStrategy).
function b200_update!(cK::B200PDMat, x::AbstractMatrix, kernel::Kernel, ln::Vector{Float64})
    d, n = size(x)
    if objectid(x) != cK.xid || (d, n) != cK.xsize       # fit!/push!/append! replace or grow x; optimiser steps do not
        X = Matrix{Float64}(x)                   # Adjoint / SubArray / ElasticArray -> dense d x N (gotcha 1)
        check(cK, ccall((:gpb200_set_data, LIB), Cint, (Ptr{Cvoid}, Int64, Int32, Ptr{Float64}, Int64), cK.handle, n, d, X, d), "set_data")
        cK.xid = objectid(x); cK.xsize = (d, n); cK.n = n
        empty!(cK.ops)
    end
    ops, dims, theta, exposed = flatten(kernel, d)
    if ops != cK.ops || dims != cK.dims
        check(cK, ccall((:gpb200_set_kernel, LIB), Cint, (Ptr{Cvoid}, Int32, Ptr{Int32}, Int32, Ptr{Int32}, Int32),
                        cK.handle, length(ops) ÷ 6, ops, length(dims), dims, length(theta)), "set_kernel")
        cK.ops = ops; cK.dims = dims
    end
    cK.exposed = exposed; cK.ntheta = length(theta)
    check(cK, ccall((:gpb200_factorize, LIB), Cint, (Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}, Int64, Float64),
                    cK.handle, theta, ln, length(ln), 0.0), "factorize")          # rc > 0 -> PosDefException
    return cK
end
update_cK!(cK::B200PDMat, x::AbstractMatrix, kernel::Kernel, logNoise::Real, data::KernelData, ::B200Covariance) =
    b200_update!(cK, x, kernel, Float64[logNoise])
update_cK!(cK::B200PDMat, x::AbstractMatrix, kernel::Kernel, logNoise::AbstractVector, data::KernelData, ::B200Covariance) =
    b200_update!(cK, x, kernel, Vector{Float64}(logNoise))

function \(cK::B200PDMat, y::AbstractVector)                                      # src/GPE.jl:208
    out = Vector{Float64}(undef, cK.n)
    check(cK, ccall((:gpb200_solve, LIB), Cint, (Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}), cK.handle, Vector{Float64}(y), out), "solve")
    return out
end

function logdet(cK::B200PDMat)                                                    # src/GPE.jl:210
    out = Ref{Float64}(0.0)
    check(cK, ccall((:gpb200_logdet, LIB), Cint, (Ptr{Cvoid}, Ref{Float64}), cK.handle, out), "logdet")
    return out[]
end

function Matrix(cK::B200PDMat)                                                    # debug only
    K = Matrix{Float64}(undef, cK.n, cK.n)
    check(cK, ccall((:gpb200_get_gram, LIB), Cint, (Ptr{Cvoid}, Ptr{Float64}), cK.handle, K), "get_gram")
    return K
end
tr(cK::B200PDMat) = tr(Matrix(cK))

init_precompute(::B200Covariance, X, y, k) = B200Precompute()                      # src/GPE.jl:256-260: no N x N host buffer

function precompute!(pre::B200Precompute, gp)                                     # src/GPE.jl:262-264
    cK = gp.cK
    check(cK, ccall((:gpb200_grad_prepare, LIB), Cint, (Ptr{Cvoid},), cK.handle), "grad_prepare")
    g = Vector{Float64}(undef, max(cK.ntheta, 1)); trA = Ref{Float64}(0.0)
    check(cK, ccall((:gpb200_grad_kernel, LIB), Cint, (Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}, Ref{Float64}),
                    cK.handle, gp.alpha, g, trA), "grad_kernel")                   # one fused pass: P gradients + tr(A)
    pre.g = g; pre.trA = trA[]; pre.exposed = cK.exposed
    return pre
end

function dmll_kern!(dmll::AbstractVector, gp, pre::B200Precompute, ::B200Covariance)   # src/GPE.jl:265-267
    dmll .= pre.g[pre.exposed]                    # FixedKernel selection (fixed_kernel.jl:64-66)
    return dmll
end

dmll_noise(gp::GPE, pre::B200Precompute, ::B200Covariance) =                      # src/GPE.jl:273-281
    exp(2 * GaussianProcesses.get_value(gp.logNoise)) * pre.trA

# leave-one-out predictions (src/crossvalidation.jl:8-13) without materialising inv(Σ) on the host
function GaussianProcesses.predict_LOO(cK::B200PDMat, alpha::AbstractVector{<:Real}, y::AbstractVector{<:Real})
    check(cK, ccall((:gpb200_grad_prepare, LIB), Cint, (Ptr{Cvoid},), cK.handle), "grad_prepare")
    d = Vector{Float64}(undef, cK.n)
    check(cK, ccall((:gpb200_get_inverse_diag, LIB), Cint, (Ptr{Cvoid}, Ptr{Float64}), cK.handle, d), "get_inverse_diag")
    σi2 = 1 ./ d
    return -alpha .* σi2 .+ y, σi2
end

# ---- cross-validation on the device's resident inverse (src/crossvalidation.jl:67-341) -------------------------------
# The reference forms inv(Σ) and, per hyper-parameter j, Z_j = inv(Σ) ∂K_j and Z_j inv(Σ) on the host (three N x N
# matrices, two N^3 products).  Here K_y^-1 is already resident after gpb200_grad_prepare: gpb200_cv_param returns the two
# N-vectors every formula needs (Z_j α and diag(Z_j inv(Σ)); j = -1 is the noise direction, Z = inv(Σ)) and gpb200_cv_block
# reads the principal sub-blocks the fold formulas index.  The O(N) / per-fold assembly below is the reference's, line by line.
function cv_param(cK::B200PDMat, j::Integer, alpha::AbstractVector)
    Zjα = Vector{Float64}(undef, cK.n); dg = Vector{Float64}(undef, cK.n)
    check(cK, ccall((:gpb200_cv_param, LIB), Cint, (Ptr{Cvoid}, Int32, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}),
                    cK.handle, j, Vector{Float64}(alpha), Zjα, dg), "cv_param")
    return Zjα, dg
end

# which = 0: inv(Σ)[V,V];  which = 1: (Z_j inv(Σ))[V,V] of the last cv_param call.  Both are symmetric, so the row-major
# block the device writes is the column-major matrix Julia reads.
function cv_block(cK::B200PDMat, which::Integer, V::AbstractVector{Int})
    idx = Vector{Int64}(V .- 1); B = Matrix{Float64}(undef, length(V), length(V))
    check(cK, ccall((:gpb200_cv_block, LIB), Cint, (Ptr{Cvoid}, Int32, Int64, Ptr{Int64}, Ptr{Float64}),
                    cK.handle, which, length(V), idx, B), "cv_block")
    return B
end

# one parameter of dlogpdθ_LOO_kern! / dlogpdσ2_LOO (crossvalidation.jl:86-101, 119-131), before the factor -1/2
function loo_component(y, alpha, σi2, μi, Zjα, ZjΣinv)
    ∂σ2 = ZjΣinv .* (σi2 .^ 2)
    ∂μ = Zjα .* σi2 .- alpha .* ∂σ2
    return -sum(2 .* (y .- μi) ./ σi2 .* ∂μ) - sum((y .- μi) .^ 2 .* ZjΣinv) + sum(ZjΣinv .* σi2)
end

function dlogpdθ_LOO(gp::GPE{X,Y,M,K,CS,D,P}; noise::Bool, domean::Bool, kern::Bool) where {X,Y,M,K,CS<:B200Covariance,D,P}
    cK = gp.cK; y = gp.y; alpha = gp.alpha
    n_mean_params = num_params(gp.mean)
    domean && n_mean_params > 0 && throw("I don't know how to do means yet")       # crossvalidation.jl:162
    μi, σi2 = predict_LOO(cK, alpha, y)                                             # runs gpb200_grad_prepare
    out = Float64[]
    if noise                                                                        # crossvalidation.jl:157-160
        Zjα, dg = cv_param(cK, -1, alpha)
        push!(out, -loo_component(y, alpha, σi2, μi, Zjα, dg) / 2 * 2 * exp(2 * get_value(gp.logNoise)))
    end
    if kern
        for j in cK.exposed                                                         # FixedKernel selection, fixed_kernel.jl:64-66
            Zjα, dg = cv_param(cK, j - 1, alpha)
            push!(out, -loo_component(y, alpha, σi2, μi, Zjα, dg) / 2)
        end
    end
    return out
end

function predict_CVfold(cK::B200PDMat, alpha::AbstractVector{<:Real}, y::AbstractVector{<:Real}, folds::Folds)   # crossvalidation.jl:180-191
    check(cK, ccall((:gpb200_grad_prepare, LIB), Cint, (Ptr{Cvoid},), cK.handle), "grad_prepare")
    μ = Vector{Float64}[]; Σ = Matrix{Float64}[]
    for V in folds
        ΣVT = inv(Symmetric(cv_block(cK, 0, V)))
        push!(μ, y[V] - ΣVT * alpha[V]); push!(Σ, Matrix(ΣVT))
    end
    return μ, Σ
end

# gradient_fold (crossvalidation.jl:250-261) with the two sub-blocks read off the device
function fold_component(cK::B200PDMat, alpha, Zjα, V, ΣVTinv)
    ZVV = cv_block(cK, 1, V)
    C = cholesky(Symmetric(ΣVTinv))
    ΣVTα = C \ alpha[V]
    return -2 * dot(ΣVTα, Zjα[V]) + dot(ΣVTα, ZVV * ΣVTα) + tr(C \ ZVV)
end

function dlogpdθ_CVfold(gp::GPE{X,Y,M,K,CS,D,P}, folds::Folds; noise::Bool, domean::Bool, kern::Bool) where {X,Y,M,K,CS<:B200Covariance,D,P}
    cK = gp.cK; alpha = gp.alpha
    n_mean_params = num_params(gp.mean)
    domean && n_mean_params > 0 && throw("I don't know how to do means yet")       # crossvalidation.jl:330
    check(cK, ccall((:gpb200_grad_prepare, LIB), Cint, (Ptr{Cvoid},), cK.handle), "grad_prepare")
    blocks = [cv_block(cK, 0, V) for V in folds]                                    # inv(Σ)[V,V], shared by every parameter
    out = Float64[]
    if noise
        Zjα, _ = cv_param(cK, -1, alpha)
        push!(out, -sum(fold_component(cK, alpha, Zjα, V, B) for (V, B) in zip(folds, blocks)) / 2 * 2 * exp(2 * get_value(gp.logNoise)))
    end
    if kern
        for j in cK.exposed
            Zjα, _ = cv_param(cK, j - 1, alpha)
            push!(out, -sum(fold_component(cK, alpha, Zjα, V, B) for (V, B) in zip(folds, blocks)) / 2)
        end
    end
    return out
end

# ---- ElasticGPE on the device (src/GPEelastic.jl:13-22, 38-47) ------------------------------------------------------
# B200Covariance(device; capacity, stepsize) reserves rows on the device so that append! extends the Cholesky factor in place
# (gpb200_append: O(k N^2)) instead of refitting; beyond the reservation the data is refitted with `stepsize` more rows
# reserved, which is what ElasticPDMats' resize! amounts to.
function B200ElasticGPE(x::AbstractMatrix, y::AbstractVector, mean::Mean, kernel::Kernel, logNoise::Real = -2.0;
                        device::Int = 0, capacity::Int = 10^3, stepsize::Int = 10^3)
    return GPE(ElasticArray(Matrix{Float64}(x)), ElasticArray(Vector{Float64}(y)), mean, kernel, logNoise,
               B200Covariance(device; capacity = capacity, stepsize = stepsize))
end

Base.append!(gp::GPE{X,Y,M,K,CS,D,P}, x::AbstractVector, y::Float64) where {X,Y,M,K,CS<:B200Covariance,D,P<:B200PDMat} =
    append!(gp, reshape(x, :, 1), [y])
function Base.append!(gp::GPE{X,Y,M,K,CS,D,P}, x::AbstractMatrix, y::AbstractVector) where {X,Y,M,K,CS<:B200Covariance,D,P<:B200PDMat}
    size(x, 2) == length(y) || error("$(size(x, 2)) observations, but $(length(y)) targets.")       # GPEelastic.jl:14
    cK = gp.cK; k = length(y)
    Xn = Matrix{Float64}(x)
    inplace = get_value(gp.logNoise) isa Real && cK.n + k <= cK.capacity
    append!(gp.x, Xn); append!(gp.y, y); gp.nobs += k
    if inplace
        check(cK, ccall((:gpb200_append, LIB), Cint, (Ptr{Cvoid}, Int64, Ptr{Float64}, Int64), cK.handle, k, Xn, size(Xn, 1)), "append")
        cK.n += k; cK.xid = objectid(gp.x); cK.xsize = size(gp.x)
        return update_target!(gp, kern = false, noise = false)                                      # GPEelastic.jl:21
    end
    cK.capacity = gp.nobs + gp.covstrat.stepsize
    check(cK, ccall((:gpb200_set_option, LIB), Cint, (Ptr{Cvoid}, Cstring, Int64), cK.handle, "capacity", cK.capacity), "set_option")
    cK.xid = UInt(0)                                                                                # force the upload of the grown x
    return update_target!(gp)
end

# batched prediction instead of the per-column loop of src/GP.jl:72-76
function predict_raw(cK::B200PDMat, x::AbstractMatrix, alpha::AbstractVector, full_cov::Bool)
    X = Matrix{Float64}(x); M = size(X, 2)
    mu = Vector{Float64}(undef, M)
    var = full_cov ? Float64[] : Vector{Float64}(undef, M)
    cov = full_cov ? Matrix{Float64}(undef, M, M) : Matrix{Float64}(undef, 0, 0)
    check(cK, ccall((:gpb200_predict, LIB), Cint,
                    (Ptr{Cvoid}, Int64, Ptr{Float64}, Int64, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}),
                    cK.handle, M, X, size(X, 1), Vector{Float64}(alpha), mu,
                    full_cov ? Ptr{Float64}(C_NULL) : pointer(var), full_cov ? pointer(cov) : Ptr{Float64}(C_NULL)), "predict")
    return mu, (full_cov ? cov : var)
end

function predict_f(gp::GPE{X,Y,M,K,CS,D,P}, x::AbstractMatrix; full_cov::Bool=false) where {X,Y,M,K,CS<:B200Covariance,D,P}
    size(x, 1) == gp.dim || throw(ArgumentError("Gaussian Process object and input observations do not have consistent dimensions"))
    full_cov && return predict_full(gp, x)                                         # -> predictMVN below (src/GPE.jl:399)
    mu, s = predict_raw(gp.cK, x, gp.alpha, false)
    return mu .+ mean(gp.mean, Matrix{Float64}(x)), max.(s, 0.0)                   # src/GP.jl:75
end

# predictMVN (src/GP.jl:39-49): mean + FULL predictive covariance through gpb200_predict(cov != NULL); this is what
# predict_full / predict_f(full_cov=true) / rand(gp, X) reach.
function predictMVN(xpred::AbstractMatrix, xtrain::AbstractMatrix, ytrain::AbstractVector, kernel::Kernel, meanf::Mean,
                    alpha::AbstractVector, ::B200Covariance, Ktrain::B200PDMat)
    mu, Sigma_raw = predict_raw(Ktrain, xpred, alpha, true)
    return mu .+ mean(meanf, Matrix{Float64}(xpred)), Sigma_raw
end

# rand(gp, X, n) (src/GP.jl:120-146) on the device: predictive covariance, make_posdef!(Σ; nugget), unwhiten!
function Random.rand!(gp::GPE{X,Y,M,K,CS,D,P}, x::AbstractMatrix, A::DenseMatrix; nugget=1e-10) where {X,Y,M,K,CS<:B200Covariance,D,P}
    Xs = Matrix{Float64}(x); Ms = size(Xs, 2); n = size(A, 2)
    Z = randn(Ms, n); mu = Vector{Float64}(undef, Ms); S = Matrix{Float64}(undef, Ms, n)
    check(gp.cK, ccall((:gpb200_rand, LIB), Cint,
                       (Ptr{Cvoid}, Int64, Ptr{Float64}, Int64, Ptr{Float64}, Int64, Ptr{Float64}, Float64, Ptr{Float64}, Ptr{Float64}),
                       gp.cK.handle, Ms, Xs, size(Xs, 1), Vector{Float64}(gp.alpha), n, Z, Float64(nugget), mu, S), "rand")
    A .= S .+ mean(gp.mean, Xs)
    return A
end

# =====================================================================================================
# Latent-variable GP (src/GPA.jl) on the device.  The reference's GPA hard-codes cK::PDMat{Float64,Matrix{Float64}}, so
# the binding is a GPBase of its own with GPA's fields and methods; mcmc / ess / optimize! drive it unchanged.  The
# device keeps the factor: update_cK! (GPA.jl:111-114), unwhiten (f = L v) and the gradient's reverse-mode Cholesky
# contracted with dK/dθ (gpb200_gpa_grad) never bring an N x N matrix to the host.
import GaussianProcesses: GPBase, Likelihood, log_dens, dlog_dens_df, dlog_dens_dθ, predict_obs, predict_y,
                          initialise_target!, update_dtarget!, update_target_and_dtarget!, set_params!, grad_stack,
                          prior_logpdf, prior_gradlogpdf, get_params_kwargs

mutable struct B200GPA{L<:Likelihood} <: GPBase
    x::Matrix{Float64}
    y::AbstractVector
    mean::Mean
    kernel::Kernel
    lik::L
    dim::Int
    nobs::Int
    v::Vector{Float64}
    μ::Vector{Float64}
    cK::B200PDMat
    ll::Float64
    dll::Vector{Float64}
    target::Float64
    dtarget::Vector{Float64}
    function B200GPA(x::AbstractMatrix, y::AbstractVector, mean::Mean, kernel::Kernel, lik::L; device::Int = 0) where {L<:Likelihood}
        dim, nobs = size(x)
        length(y) == nobs || throw(ArgumentError("Input and output observations must have consistent dimensions."))
        gp = new{L}(Matrix{Float64}(x), y, mean, kernel, lik, dim, nobs, zeros(nobs), zeros(nobs), B200PDMat(device, nobs),
                    NaN, Float64[], NaN, Float64[])
        return initialise_target!(gp)
    end
end

function b200_unwhiten(cK::B200PDMat, v::Vector{Float64})                      # unwhiten(cK, v), GPA.jl:106
    f = Vector{Float64}(undef, cK.n)
    check(cK, ccall((:gpb200_unwhiten, LIB), Cint, (Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}), cK.handle, v, f), "unwhiten")
    return f
end

function gpa_set_target!(gp::B200GPA)                                           # GPA.jl:247-248, 263-264
    gp.μ = mean(gp.mean, gp.x)
    gp.ll = sum(log_dens(gp.lik, b200_unwhiten(gp.cK, gp.v) + gp.μ, gp.y))
    gp.target = gp.ll - (sum(abs2, gp.v) + log(2π) * gp.nobs) / 2 +
        prior_logpdf(gp.lik) + prior_logpdf(gp.mean) + prior_logpdf(gp.kernel)
    return gp
end

function initialise_target!(gp::B200GPA)                                        # GPA.jl:101-109: Σ + 1e-6 I
    b200_update!(gp.cK, gp.x, gp.kernel, [0.5 * log(1e-6)])
    return gpa_set_target!(gp)
end

function update_target!(gp::B200GPA; process::Bool=true, lik::Bool=true, domean::Bool=true, kern::Bool=true)   # GPA.jl:261-266
    kern && b200_update!(gp.cK, gp.x, gp.kernel, [-20.0])                   # update_cK!, GPA.jl:111-114
    return gpa_set_target!(gp)
end

function update_dtarget!(gp::B200GPA; process::Bool=true, lik::Bool=true, domean::Bool=true, kern::Bool=true)  # GPA.jl:183-228, 268-272
    f = b200_unwhiten(gp.cK, gp.v) + gp.μ
    dl_df = Vector{Float64}(dlog_dens_df(gp.lik, f, gp.y))
    dv = Vector{Float64}(undef, gp.nobs); g = Vector{Float64}(undef, max(gp.cK.ntheta, 1))
    if process || kern                                                          # L' dl_df and dll_kern! in one device call
        check(gp.cK, ccall((:gpb200_gpa_grad, LIB), Cint, (Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}),
                           gp.cK.handle, gp.v, dl_df, dv, g), "gpa_grad")
    end
    dll = Float64[]
    process && append!(dll, dv)
    lik && num_params(gp.lik) > 0 && append!(dll, vec(sum(dlog_dens_dθ(gp.lik, f, gp.y), dims=1)))
    domean && num_params(gp.mean) > 0 && append!(dll, grad_stack(gp.mean, gp.x)' * dl_df)
    kern && append!(dll, g[gp.cK.exposed])
    gp.dll = dll
    gp.dtarget = dll + prior_gradlogpdf(gp; process=process, lik=lik, domean=domean, kern=kern)
    return gp
end

function update_target_and_dtarget!(gp::B200GPA; kwargs...)                      # GPA.jl:283-291
    update_target!(gp; kwargs...)
    return update_dtarget!(gp; kwargs...)
end
update_target_and_dtarget!(gp::B200GPA, ::AbstractGradientPrecompute; kwargs...) = update_target_and_dtarget!(gp; kwargs...)
init_precompute(gp::B200GPA) = B200Precompute()
get_params_kwargs(::B200GPA; kwargs...) = delete!(Dict(kwargs), :noise)          # src/optimize.jl:2

function prior_gradlogpdf(gp::B200GPA; process::Bool=true, lik::Bool=true, domean::Bool=true, kern::Bool=true)  # GPA.jl:383-399
    grad = process ? -gp.v : Float64[]
    lik && append!(grad, prior_gradlogpdf(gp.lik))
    domean && append!(grad, prior_gradlogpdf(gp.mean))
    kern && append!(grad, prior_gradlogpdf(gp.kernel))
    return grad
end

function get_params(gp::B200GPA; lik::Bool=true, domean::Bool=true, kern::Bool=true)   # GPA.jl:336-349
    params = copy(gp.v)
    lik && num_params(gp.lik) > 0 && append!(params, get_params(gp.lik))
    domean && num_params(gp.mean) > 0 && append!(params, get_params(gp.mean))
    kern && append!(params, get_params(gp.kernel))
    return params
end
num_params(gp::B200GPA; lik::Bool=true, domean::Bool=true, kern::Bool=true) =      # GPA.jl:351-357
    gp.nobs + (lik ? num_params(gp.lik) : 0) + (domean ? num_params(gp.mean) : 0) + (kern ? num_params(gp.kernel) : 0)

function set_params!(gp::B200GPA, hyp::AbstractVector; process::Bool=true, lik::Bool=true, domean::Bool=true, kern::Bool=true)  # GPA.jl:359-381
    nl, nm, nk = num_params(gp.lik), num_params(gp.mean), num_params(gp.kernel)
    i = 1
    if process
        gp.v = hyp[1:gp.nobs]; i += gp.nobs
    end
    if lik && nl > 0
        set_params!(gp.lik, hyp[i:i+nl-1]); i += nl
    end
    if domean && nm > 0
        set_params!(gp.mean, hyp[i:i+nm-1]); i += nm
    end
    kern && set_params!(gp.kernel, hyp[i:i+nk-1])
end

function predict_f(gp::B200GPA, x::AbstractMatrix; full_cov::Bool=false)          # predict_full, GPA.jl:294
    size(x, 1) == gp.dim || throw(ArgumentError("Gaussian Process object and input observations do not have consistent dimensions"))
    alpha = gp.cK \ b200_unwhiten(gp.cK, gp.v)
    mu, s = predict_raw(gp.cK, x, alpha, full_cov)
    mu = mu .+ mean(gp.mean, Matrix{Float64}(x))
    return full_cov ? (mu, s) : (mu, max.(s, 0.0))                                   # src/GP.jl:75
end

function predict_y(gp::B200GPA, x::AbstractMatrix; full_cov::Bool=false)          # GPA.jl:303-306
    μ, σ2 = predict_f(gp, x; full_cov=full_cov)
    return predict_obs(gp.lik, μ, σ2)
end

# =====================================================================================================
# Sparse strategies on the device: FITC / DTC / SoR (src/sparse/*.jl) -> gpb200_fitc_* (one streaming engine)
#     gp = GPE(x, y, mean, kernel, logNoise, B200Sparse(Xu, :FITC))
# =====================================================================================================
import GaussianProcesses: SparseStrategy

struct B200Sparse{M<:AbstractMatrix} <: SparseStrategy
    inducing::M
    mode::Symbol              # :FITC (fully_indep_train_conditional.jl), :DTC (determ_train_conditional.jl), :SoR
    device::Int
end
B200Sparse(Xu::AbstractMatrix, mode::Symbol=:FITC) = B200Sparse(Xu, mode, 0)
const SPARSE_MODE = Dict(:FITC => 0, :DTC => 1, :SoR => 2)

mutable struct B200SparsePDMat <: AbstractPDMat{Float64}
    handle::Ptr{Cvoid}
    n::Int
    exposed::Vector{Int}
    ntheta::Int
    alpha::Vector{Float64}     # Sigma^-1 r of the last `\`
    logdet::Float64
    function B200SparsePDMat(cs::B200Sparse, n::Int)
        h = Ref{Ptr{Cvoid}}(C_NULL)
        rc = ccall((:gpb200_fitc_create, LIB), Cint, (Ref{Ptr{Cvoid}}, Cint), h, cs.device)
        rc == 0 || error("gpb200_fitc_create failed ($rc)")
        ccall((:gpb200_fitc_set_mode, LIB), Cint, (Ptr{Cvoid}, Cint), h[], SPARSE_MODE[cs.mode])
        obj = new(h[], n, Int[], 0, Float64[], NaN)
        finalizer(o -> ccall((:gpb200_fitc_destroy, LIB), Cvoid, (Ptr{Cvoid},), o.handle), obj)
        return obj
    end
end
size(a::B200SparsePDMat) = (a.n, a.n)
dim(a::B200SparsePDMat) = a.n

function checks(cK::B200SparsePDMat, rc::Integer, what)
    rc == 0 && return
    rc > 0 && throw(PosDefException(rc))
    msg = unsafe_string(ccall((:gpb200_fitc_last_error, LIB), Cstring, (Ptr{Cvoid},), cK.handle))
    (rc == -1 || rc == -4) && throw(ArgumentError("$what: $msg"))
    error("$what failed ($rc): $msg")
end

KernelData(k::Kernel, X1::AbstractMatrix, X2::AbstractMatrix, ::B200Sparse) = EmptyData()
alloc_cK(cs::B200Sparse, nobs) = B200SparsePDMat(cs, nobs)

# update_cK!(::FullyIndepPDMat) fitc.jl:134-156 / update_cK!(::SubsetOfRegsPDMat) sor.jl:96-106
function update_cK!(cK::B200SparsePDMat, x::AbstractMatrix, kernel::Kernel, logNoise::Real, data::KernelData, cs::B200Sparse)
    X = Matrix{Float64}(x); Xu = Matrix{Float64}(cs.inducing)
    d, n = size(X)
    checks(cK, ccall((:gpb200_fitc_set_data, LIB), Cint,
                     (Ptr{Cvoid}, Int64, Int32, Ptr{Float64}, Int64, Int64, Ptr{Float64}, Int64),
                     cK.handle, n, d, X, d, size(Xu, 2), Xu, d), "fitc_set_data")
    ops, dims, theta, exposed = flatten(kernel, d)
    cK.exposed = exposed; cK.ntheta = length(theta)
    checks(cK, ccall((:gpb200_fitc_set_kernel, LIB), Cint, (Ptr{Cvoid}, Int32, Ptr{Int32}, Int32, Ptr{Int32}, Int32),
                     cK.handle, length(ops) ÷ 6, ops, length(dims), dims, length(theta)), "fitc_set_kernel")
    checks(cK, ccall((:gpb200_fitc_factorize, LIB), Cint, (Ptr{Cvoid}, Ptr{Float64}, Float64),
                     cK.handle, theta, Float64(logNoise)), "fitc_factorize")
    return cK
end

# `\` (fitc.jl:33-36, sor.jl:50) and logdet (fitc.jl:77, sor.jl:53) come from one device pass
function \(cK::B200SparsePDMat, y::AbstractVector)
    alpha = Vector{Float64}(undef, cK.n); mll = Ref{Float64}(0.0); ld = Ref{Float64}(0.0)
    checks(cK, ccall((:gpb200_fitc_mll, LIB), Cint, (Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}, Ref{Float64}, Ref{Float64}),
                     cK.handle, Vector{Float64}(y), alpha, mll, ld), "fitc_mll")
    cK.alpha = alpha; cK.logdet = ld[]
    return alpha
end
logdet(cK::B200SparsePDMat) = cK.logdet

struct B200SparsePrecompute <: AbstractGradientPrecompute end
init_precompute(::B200Sparse, X, y, k) = B200SparsePrecompute()
precompute!(::B200SparsePrecompute, gp) = nothing

function dmll_noise(gp::GPE, ::B200SparsePrecompute, ::B200Sparse)                 # fitc.jl:243-257, sor.jl:159-166
    g = Ref{Float64}(0.0)
    checks(gp.cK, ccall((:gpb200_fitc_grad_noise, LIB), Cint, (Ptr{Cvoid}, Ref{Float64}), gp.cK.handle, g), "fitc_grad_noise")
    return g[]
end
function dmll_kern!(dmll::AbstractVector, gp, ::B200SparsePrecompute, ::B200Sparse)    # fitc.jl:200-234, sor.jl:219-253
    g = Vector{Float64}(undef, max(gp.cK.ntheta, 1))
    checks(gp.cK, ccall((:gpb200_fitc_grad_kernel, LIB), Cint, (Ptr{Cvoid}, Ptr{Float64}), gp.cK.handle, g), "fitc_grad_kernel")
    dmll .= g[gp.cK.exposed]
    return dmll
end
function predict_f(gp::GPE{X,Y,M,K,CS,D,P}, x::AbstractMatrix; full_cov::Bool=false) where {X,Y,M,K,CS<:B200Sparse,D,P}
    size(x, 1) == gp.dim || throw(ArgumentError("Gaussian Process object and input observations do not have consistent dimensions"))
    Xs = Matrix{Float64}(x); Ms = size(Xs, 2)
    if full_cov                                                                    # predictMVN: fitc.jl:324-332, dtc.jl:41-59, sor.jl:302-321
        mu = Vector{Float64}(undef, Ms); Σ = Matrix{Float64}(undef, Ms, Ms)
        checks(gp.cK, ccall((:gpb200_fitc_predict_cov, LIB), Cint, (Ptr{Cvoid}, Int64, Ptr{Float64}, Int64, Ptr{Float64}, Ptr{Float64}),
                            gp.cK.handle, Ms, Xs, size(Xs, 1), mu, Σ), "fitc_predict_cov")
        return mu .+ mean(gp.mean, Xs), Σ
    end
    mu = Vector{Float64}(undef, Ms); var = Vector{Float64}(undef, Ms)
    checks(gp.cK, ccall((:gpb200_fitc_predict, LIB), Cint, (Ptr{Cvoid}, Int64, Ptr{Float64}, Int64, Ptr{Float64}, Ptr{Float64}),
                        gp.cK.handle, Ms, Xs, size(Xs, 1), mu, var), "fitc_predict")
    return mu .+ mean(gp.mean, Xs), max.(var, 0.0)
end

export B200Covariance, B200Sparse, B200ElasticGPE, B200GPA

end # module
