# GPRB200.jl - routes the GP calls of GPR.jl's experiments to libgprb200.so WITHOUT changing their types.
#
# NOT EXECUTED IN THIS REPOSITORY'S CI: the build image has no Julia toolchain.  The tested contract is the C ABI
# (include/gprb200.h, exercised through ctypes by tests/); every ccall below mirrors one prototype of that header
# one-to-one (tests/test_julia_shim_signatures.py parses this file and checks every ccall tuple against the header),
# and gpr.jl_b200/lib.py + gp.py are the executable twin.  Names and signatures of GaussianProcesses.jl 0.12.4
# internals (GPE type parameters, alloc_cK, the 8-argument GPE constructor, init_precompute) are written from the
# published source of that version (Manifest.toml:409-413) and could not be compiled here.
#
# Drop-in mechanism: GaussianProcesses.jl's own extension point for the linear-algebra back end is the covariance
# strategy (`GPE(...; covstrat)`, used by its sparse approximations).  `B200Covariance <: CovarianceStrategy` keeps the
# object a real `GaussianProcesses.GPE`, so the reference's typed call sites work unchanged:
#     gps = Vector{GPE}()                                              examples/maximal_coordinates/CPnoise.jl:35
#     predictdynamics(mechanism, gps::Vector{<:GPE}, x0, steps, getvω)   examples/utils/predictdynamics.jl:7
# Nothing is exported that GaussianProcesses / Optim export (`using GaussianProcesses, GPRB200` has no clashes).
#
# Per-GP flavour - the ONLY edit in an experiment body (CPnoise.jl:40): the constructor gets the strategy
#     kernel = SEArd(log.(params[2:end]), log(params[1]))                          # :38 unchanged
#     gp = GP(xtrain_old, yi, mean, kernel, B200Covariance())                      # :40  (+ one argument)
#     GaussianProcesses.optimize!(gp, LBFGS(linesearch = BackTracking(order=2)), Optim.Options(time_limit=10.))   # :41 unchanged
#     μ = predict_y(gp, obs)[1][1]                                                 # predictdynamics.jl:13 unchanged
# Batched flavour (what replaces the `Threads.@threads for jobid` loop of examples/parallel/core.jl:28):
#     gps = [GPE(X_t, y_tk, mean_tk, SEArd(...), -2.0, B200Covariance()) for t in trials for k in outputs]   # no evaluation yet
#     GaussianProcesses.optimize!(gps, LBFGS(linesearch = BackTracking(order=2)), Optim.Options(time_limit=10.))  # ONE gprb_optimize
#     predictdynamics(mechanism, gps[(t-1)*G+1:t*G], x0, steps, getvω)            # unchanged; the G predict_y calls of a step share one device call
module GPRB200

using Libdl
import Random
import GaussianProcesses
import GaussianProcesses: GPE, Mean, MeanZero, Kernel, SEArd, Mat12Ard, Mat32Ard, Mat52Ard, CovarianceStrategy, KernelData, EmptyData,
                          get_params, set_params!, num_params
import Optim
import PDMats

export B200Covariance, GPBatch, params_to_theta, theta_to_params, gather_results, predict_cov, sample_posterior!

const LIB = get(ENV, "GPRB200_LIB", joinpath(@__DIR__, "..", "libgprb200.so"))

# ---- status handling (no exceptions cross the C boundary; we raise on the Julia side) --------------------------------
struct GprbError <: Exception
    code::Cint
    msg::String
end
last_error() = unsafe_string(ccall((:gprb_last_error, LIB), Cstring, ()))
check(rc::Cint) = rc == 0 ? nothing : throw(GprbError(rc, last_error()))

# ---- context: one per process and GPU --------------------------------------------------------------------------------
const CTX = Ref{Ptr{Cvoid}}(C_NULL)
function context()
    if CTX[] == C_NULL
        h = Ref{Ptr{Cvoid}}(C_NULL)
        dev = parse(Cint, get(ENV, "GPRB200_DEVICE", get(ENV, "LOCAL_RANK", "0")))
        check(ccall((:gprb_init, LIB), Cint, (Ref{Ptr{Cvoid}}, Cint), h, dev))     # fails without a B200: no CPU fallback
        CTX[] = h[]
    end
    CTX[]
end

kernel_kind(::SEArd) = Cint(0)
kernel_kind(::Mat12Ard) = Cint(1)
kernel_kind(::Mat32Ard) = Cint(2)
kernel_kind(::Mat52Ard) = Cint(3)

# ---- the covariance strategy -----------------------------------------------------------------------------------------
"Covariance strategy that keeps K, its factor and alpha in HBM (libgprb200.so) instead of a host PDMat."
struct B200Covariance <: CovarianceStrategy end

# gp.cK is never read by the reference's callers; a 1-byte placeholder satisfies the field type (no n x n host allocation,
# no n x n x d distance stack: KernelData is EmptyData)
GaussianProcesses.alloc_cK(::B200Covariance, nobs::Int) = PDMats.ScalMat(nobs, 1.0)

const B200GPE = GPE{<:AbstractMatrix,<:AbstractVector,<:Mean,<:Kernel,<:B200Covariance}

"`GPE(X, y, mean, kernel, logNoise, B200Covariance())`: a GaussianProcesses.GPE whose linear algebra lives on the B200 (no evaluation yet)."
GaussianProcesses.GPE(x::AbstractMatrix, y::AbstractVector, mean::Mean, kernel::Kernel, logNoise::Real, cs::B200Covariance) =
    GPE(Matrix{Float64}(x), Vector{Float64}(y), mean, kernel, Float64(logNoise), cs, EmptyData(), GaussianProcesses.alloc_cK(cs, length(y)))

"`GP(X, y, mean, kernel, B200Covariance())`: construct + initial update_mll!, like GaussianProcesses.GP (CPnoise.jl:40)."
function GaussianProcesses.GP(x::AbstractMatrix, y::AbstractVector, mean::Mean, kernel::Kernel, cs::B200Covariance; logNoise::Real = -2.0)
    gp = GPE(x, y, mean, kernel, logNoise, cs)
    GaussianProcesses.update_mll!(gp)
    gp
end

# GaussianProcesses.get_params order: [logNoise; mean params; kernel params] - the reference's means have none (src/mDynamics.jl:29-31)
theta_of(gp::GPE) = Vector{Float64}(get_params(gp))

# ---- GPBatch: the device residence of one or many GPEs ----------------------------------------------------------------
mutable struct GPBatch
    gps::Vector{GPE}
    handle::Ptr{Cvoid}
    datasets::Vector{Ptr{Cvoid}}
    B::Int; n::Int; d::Int; P::Int
    # shared prediction cache of one rollout step: the G predict_y(gp, obs) calls of predictdynamics.jl:13 hit one device call
    cache_key::Matrix{Float64}
    cache_mu::Matrix{Float64}
    cache_var::Matrix{Float64}
end

# gp -> (batch, slot); weak, so dropping the GPEs frees the device memory through the batch finalizer
const RESIDENT = WeakKeyDict{GPE,Tuple{GPBatch,Int}}()

function GPBatch(gps::Vector{<:GPE})
    ctx = context()
    d, n = gps[1].dim, gps[1].nobs
    B = length(gps)
    # all distinct training sets of the batch in ONE device allocation, uploaded as one contiguous block
    uniq = IdDict{Any,Int}()
    for gp in gps
        get!(uniq, gp.x, length(uniq) + 1)
    end
    T = length(uniq)
    block = Array{Float64,3}(undef, d, n, T)
    for (x, t) in uniq
        block[:, :, t] = x
    end
    ptrs = [pointer(block, (t - 1) * d * n + 1) for t in 1:T]
    dsh = Vector{Ptr{Cvoid}}(undef, T)
    GC.@preserve block begin
        check(ccall((:gprb_datasets_create, LIB), Cint, (Ptr{Cvoid}, Int32, Int64, Int32, Ptr{Ptr{Float64}}, Int64, Ptr{Ptr{Cvoid}}),
                    ctx, T, n, d, ptrs, d, dsh))
    end
    handles = [dsh[uniq[gp.x]] for gp in gps]
    # m(X) does not depend on θ: evaluate once per training set, column by column across the GPs of a trial so the shared
    # MDCache (src/mDynamics.jl:6-11,42) hits for the other G-1 outputs.  Only y - m(X) goes to the device.
    ymm = Matrix{Float64}(undef, n, B)
    for (x, _) in uniq
        members = [b for b in 1:B if gps[b].x === x]
        for j in 1:n, b in members
            ymm[j, b] = gps[b].y[j] - GaussianProcesses.mean(gps[b].mean, gps[b].x[:, j])
        end
    end
    h = Ref{Ptr{Cvoid}}(C_NULL)
    check(ccall((:gprb_batch_create, LIB), Cint, (Ptr{Cvoid}, Int32, Ptr{Ptr{Cvoid}}, Ptr{Float64}, Int32, Ref{Ptr{Cvoid}}),
                ctx, B, handles, ymm, kernel_kind(gps[1].kernel), h))
    batch = GPBatch(Vector{GPE}(gps), h[], dsh, B, n, d, d + 2, zeros(0, 0), zeros(0, 0), zeros(0, 0))
    for (b, gp) in enumerate(gps)
        RESIDENT[gp] = (batch, b)
    end
    finalizer(batch) do bt
        ccall((:gprb_batch_destroy, LIB), Cint, (Ptr{Cvoid},), bt.handle)
        foreach(ds -> ccall((:gprb_dataset_destroy, LIB), Cint, (Ptr{Cvoid},), ds), bt.datasets)
    end
    batch
end

"The batch a GPE lives in (a batch of one is created on demand: the reference's per-GP call pattern)."
function residence(gp::GPE)
    haskey(RESIDENT, gp) || GPBatch(GPE[gp])
    RESIDENT[gp]
end

thetas(batch::GPBatch) = reduce(hcat, theta_of.(batch.gps))          # P × B, column per GP: the layout gprb_eval takes

"One objective evaluation per active GP of the batch; writes mll / dmll / alpha back into the GPE fields the callers read."
function evaluate!(batch::GPBatch; θ::Matrix{Float64} = thetas(batch), grad::Bool = true, active::Union{Nothing,Vector{UInt8}} = nothing)
    mll = fill(NaN, batch.B)
    g = grad ? fill(NaN, batch.P, batch.B) : nothing
    info = zeros(Int32, batch.B)
    GC.@preserve θ mll g info active begin
        check(ccall((:gprb_eval, LIB), Cint, (Ptr{Cvoid}, Ptr{Float64}, Ptr{UInt8}, Ptr{Float64}, Ptr{Float64}, Ptr{Int32}),
                    batch.handle, θ, active === nothing ? C_NULL : pointer(active), mll, grad ? pointer(g) : C_NULL, info))
    end
    for (b, gp) in enumerate(batch.gps)
        (active === nothing || active[b] != 0) || continue
        gp.mll = mll[b]; gp.target = mll[b]                       # no priors are set anywhere in the reference
        if grad
            gp.dmll = g[:, b]; gp.dtarget = g[:, b]
        end
        info[b] < 0 && throw(PDMats.PosDefException(Int(info[b])))   # get_optim_target's catch branch turns this into +Inf
    end
    batch.cache_key = zeros(0, 0)
    mll, g, info
end

function only_active(batch::GPBatch, slot::Int)
    a = zeros(UInt8, batch.B)
    a[slot] = 1
    a
end

# the two evaluation entry points GaussianProcesses.optimize! / GP(...) reach (GPE.jl: update_mll!, update_mll_and_dmll!)
function GaussianProcesses.update_mll!(gp::B200GPE; kwargs...)
    batch, slot = residence(gp)
    evaluate!(batch; grad = false, active = batch.B == 1 ? nothing : only_active(batch, slot))
    gp
end
function GaussianProcesses.update_mll_and_dmll!(gp::B200GPE, precomp...; kwargs...)
    batch, slot = residence(gp)
    evaluate!(batch; grad = true, active = batch.B == 1 ? nothing : only_active(batch, slot))
    gp
end
GaussianProcesses.init_precompute(gp::B200GPE) = nothing     # no n x n host work buffer

"gp.alpha on demand (the field is filled lazily: the rollout never reads it)."
function alpha!(gp::B200GPE)
    batch, slot = residence(gp)
    a = Vector{Float64}(undef, batch.n)
    check(ccall((:gprb_get_alpha, LIB), Cint, (Ptr{Cvoid}, Int32, Ptr{Float64}), batch.handle, slot - 1, a))
    gp.alpha = a
end

# ---- optimize! -------------------------------------------------------------------------------------------------------
struct LbfgsOpts                 # gprb_lbfgs_opts
    m::Int32; iterations::Int32; max_evals::Int32; ls_iterations::Int32
    g_abstol::Float64; time_limit::Float64; c_1::Float64; rho_hi::Float64; rho_lo::Float64
    cost_value::Float64; cost_grad::Float64
end
struct OptResult                 # gprb_opt_result
    mll::Float64; g_norm::Float64
    iterations::Int32; f_calls::Int32; fg_calls::Int32; converged::Int32; ls_failed::Int32; info::Int32
end

"""
    GaussianProcesses.optimize!(gps::Vector{<:GPE}, method::Optim.LBFGS, options::Optim.Options; max_evals, cost_value, cost_grad)

Batched form of the reference's `GaussianProcesses.optimize!(gp, LBFGS(linesearch=BackTracking(order=2)),
Optim.Options(time_limit=10.))` (CPnoise.jl:41): all GPs advance in lock-step inside ONE gprb_optimize call.
`options.time_limit` is the reference's per-GP 10 s: with `cost_value` / `cost_grad` (seconds one value-only / value+gradient
evaluation takes on the CPU being emulated) it runs on a deterministic per-GP virtual clock; without them it is the wall
clock of the whole batch.  `max_evals` is a per-GP evaluation cap.
"""
function GaussianProcesses.optimize!(gps::Vector{<:GPE}, method::Optim.LBFGS = Optim.LBFGS(), options::Optim.Options = Optim.Options();
                                     max_evals::Integer = 0, cost_value::Real = 0.0, cost_grad::Real = 0.0)
    batch = (haskey(RESIDENT, gps[1]) && RESIDENT[gps[1]][1].gps == gps) ? RESIDENT[gps[1]][1] : GPBatch(gps)
    ls = method.linesearch!
    o = LbfgsOpts(method.m, options.iterations, max_evals, ls.iterations, options.g_abstol,
                  isfinite(options.time_limit) ? options.time_limit : 0.0, ls.c_1, ls.ρ_hi, ls.ρ_lo, cost_value, cost_grad)
    θ = thetas(batch)
    res = Vector{OptResult}(undef, batch.B)
    check(ccall((:gprb_optimize, LIB), Cint, (Ptr{Cvoid}, Ptr{Float64}, Ref{LbfgsOpts}, Ptr{OptResult}), batch.handle, θ, o, res))
    for (b, gp) in enumerate(batch.gps)
        set_params!(gp, θ[:, b])
        gp.mll = res[b].mll; gp.target = res[b].mll
    end
    batch.cache_key = zeros(0, 0)
    res
end
# the reference's per-GP call (CPnoise.jl:41) on a B200-resident GPE: a batch of one through the same driver
GaussianProcesses.optimize!(gp::B200GPE, method::Optim.LBFGS = Optim.LBFGS(), options::Optim.Options = Optim.Options(); kw...) =
    GaussianProcesses.optimize!(GPE[gp], method, options; kw...)[1]

# ---- predict_y -------------------------------------------------------------------------------------------------------
"predict_y(batch, Xstar::d×m) -> (μ::m×B, σ²::m×B | nothing); `var=false` skips the variance the reference discards. GPs without state give NaN columns."
function GaussianProcesses.predict_y(batch::GPBatch, Xstar::AbstractMatrix; var::Bool = true)
    Xs = Matrix{Float64}(Xstar)
    m = size(Xs, 2)
    mstar = nothing
    if !all(gp -> gp.mean isa MeanZero, batch.gps)
        mstar = Matrix{Float64}(undef, m, batch.B)
        for j in 1:m, b in 1:batch.B            # column-major over GPs: MDCache semantics of src/mDynamics.jl:41-55
            mstar[j, b] = GaussianProcesses.mean(batch.gps[b].mean, Xs[:, j])
        end
    end
    μ = Matrix{Float64}(undef, m, batch.B)
    σ2 = var ? Matrix{Float64}(undef, m, batch.B) : nothing
    GC.@preserve Xs mstar μ σ2 begin
        check(ccall((:gprb_predict, LIB), Cint, (Ptr{Cvoid}, Int64, Ptr{Float64}, Int64, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}),
                    batch.handle, m, Xs, 0, mstar === nothing ? C_NULL : pointer(mstar), μ, var ? pointer(σ2) : C_NULL))
    end
    μ, σ2
end

# The reference's call `predict_y(gp, obs)[1][1]` (predictdynamics.jl:13), once per GP of the trial with the SAME obs:
# the first call predicts every GP of the batch on the device, the other G-1 calls are served from the step cache
# (the device-side twin of MDCache, src/mDynamics.jl:6-11).  `full_cov=true` returns the joint m×m predictive covariance.
function GaussianProcesses.predict_y(gp::B200GPE, Xstar::AbstractMatrix; full_cov::Bool = false)
    batch, slot = residence(gp)
    if full_cov
        μ, Σ = predict_cov(batch, Xstar; add_noise = true)
        return μ[:, slot], Σ[:, :, slot]
    end
    if size(batch.cache_key) != size(Xstar) || batch.cache_key != Xstar
        μ, σ2 = GaussianProcesses.predict_y(batch, Xstar; var = true)
        batch.cache_key, batch.cache_mu, batch.cache_var = Matrix{Float64}(Xstar), μ, σ2
    end
    batch.cache_mu[:, slot], batch.cache_var[:, slot]
end

# ---- predict_f / full_cov / rand (GaussianProcesses 0.12.4 GP.jl, GPE.jl) ------------------------------------------------
# Without these methods the generic predictMVN / rand! of GaussianProcesses would read gp.cK (a placeholder here) and
# gp.alpha (filled on demand): every call below goes to the device instead.
prior_means(batch::GPBatch, Xs::Matrix{Float64}) = all(gp -> gp.mean isa MeanZero, batch.gps) ? nothing :
    [GaussianProcesses.mean(batch.gps[b].mean, Xs[:, j]) for j in 1:size(Xs, 2), b in 1:batch.B]

"predict_cov(batch, Xstar) -> (μ::m×B, Σ::m×m×B): Σ_f = K** - K*'K⁻¹K* (`add_noise=false`) or Σ_y = Σ_f + σ²_n I."
function predict_cov(batch::GPBatch, Xstar::AbstractMatrix; add_noise::Bool)
    Xs = Matrix{Float64}(Xstar)
    m = size(Xs, 2)
    mstar = prior_means(batch, Xs)
    μ = Matrix{Float64}(undef, m, batch.B)
    Σ = Array{Float64,3}(undef, m, m, batch.B)
    GC.@preserve Xs mstar μ Σ begin
        check(ccall((:gprb_predict_cov, LIB), Cint, (Ptr{Cvoid}, Int64, Ptr{Float64}, Int64, Ptr{Float64}, Int32, Ptr{Float64}, Ptr{Float64}),
                    batch.handle, m, Xs, 0, mstar === nothing ? C_NULL : pointer(mstar), add_noise ? 1 : 0, μ, Σ))
    end
    μ, Σ
end

"predict_f(batch, Xstar; full_cov) -> (μ::m×B, σ²_f::m×B | Σ_f::m×m×B): the latent posterior (no observation noise)."
function predict_f(batch::GPBatch, Xstar::AbstractMatrix; full_cov::Bool = false)
    full_cov && return predict_cov(batch, Xstar; add_noise = false)
    μ, σ2 = GaussianProcesses.predict_y(batch, Xstar; var = true)
    for b in 1:batch.B
        σ2[:, b] .= max.(σ2[:, b] .- exp(2 * batch.gps[b].logNoise), 0.0)
    end
    μ, σ2
end

function GaussianProcesses.predict_f(gp::B200GPE, Xstar::AbstractMatrix; full_cov::Bool = false)
    batch, slot = residence(gp)
    μ, v = predict_f(batch, Xstar; full_cov = full_cov)
    full_cov ? (μ[:, slot], v[:, :, slot]) : (μ[:, slot], v[:, slot])
end

"""
    sample_posterior!(batch, Xstar, A::Array{Float64,3}, Z::Array{Float64,3}) -> info::Vector{Int32}

Draws of every GP's latent posterior at Xstar: A[:, :, b] = μ_b + L_b Z[:, :, b], L_b the lower factor of
make_posdef!(Σ_f).  info[b]: jitter rung 0..10, -1 indefinite after 10 jitters, -2 non-finite Σ_f / no state (NaN draws).
"""
function sample_posterior!(batch::GPBatch, Xstar::AbstractMatrix, A::Array{Float64,3}, Z::Array{Float64,3})
    Xs = Matrix{Float64}(Xstar)
    m, ns = size(Xs, 2), size(A, 2)
    size(A) == size(Z) == (m, ns, batch.B) || throw(DimensionMismatch("A and Z must be m × n × B"))
    mstar = prior_means(batch, Xs)
    info = zeros(Int32, batch.B)
    GC.@preserve Xs mstar A Z info begin
        check(ccall((:gprb_sample_posterior, LIB), Cint,
                    (Ptr{Cvoid}, Int64, Ptr{Float64}, Int64, Ptr{Float64}, Int32, Ptr{Float64}, Ptr{Float64}, Ptr{Int32}),
                    batch.handle, m, Xs, 0, mstar === nothing ? C_NULL : pointer(mstar), ns, Z, A, info))
    end
    info
end

"Batched `rand`: draws m × n × B with Z = randn(m, n) per GP (the order GaussianProcesses' rand! draws them in)."
function Random.rand(batch::GPBatch, Xstar::AbstractMatrix, n::Integer = 1)
    m = size(Xstar, 2)
    Z = Array{Float64,3}(undef, m, n, batch.B)
    for b in 1:batch.B
        Z[:, :, b] = randn(m, n)
    end
    A = similar(Z)
    sample_posterior!(batch, Xstar, A, Z), A
end

# `rand!(gp, X, A)` (GPE.jl): Z = randn(nobs, n_sample) on the host exactly as GaussianProcesses draws it, then
# A = μ + chol_lower(make_posdef!(Σ_f)) Z on the device.  A factorisation that fails raises PosDefException.
function Random.rand!(gp::B200GPE, x::AbstractMatrix, A::DenseMatrix)
    batch, slot = residence(gp)
    m, ns = size(x, 2), size(A, 2)
    Zb = zeros(m, ns, batch.B)
    Zb[:, :, slot] = randn(m, ns)
    Ab = similar(Zb)
    info = sample_posterior!(batch, x, Ab, Zb)
    info[slot] < 0 && throw(PDMats.PosDefException(Int(info[slot])))
    A .= view(Ab, :, :, slot)
end
Random.rand(gp::B200GPE, x::AbstractMatrix, n::Int) = Random.rand!(gp, x, Matrix{Float64}(undef, size(x, 2), n))
Random.rand(gp::B200GPE, x::AbstractMatrix) = vec(Random.rand(gp, x, 1))

# ---- leave-one-out cross-validation (GaussianProcesses crossvalidation.jl: predict_LOO, logp_CVLOO, dlogpdθ_CVLOO) --------
# The generic methods work from gp.cK (a placeholder here) and gp.alpha (filled on demand): these go to the device.  The
# GaussianProcesses function is extended where the installed version defines it; otherwise GPRB200 defines and exports
# its own, so the module loads either way.
for name in (:predict_LOO, :logp_CVLOO, :dlogpdθ_CVLOO)
    if isdefined(GaussianProcesses, name)
        @eval import GaussianProcesses: $name
    else
        @eval function $name end
        @eval export $name
    end
end

"""
    eval_loo!(batch; grad=true, mu_var=false, active=nothing) -> (logp::B, ∇::P×B | nothing, info::B, μ::n×B | nothing, σ²::n×B | nothing)

One evaluation with gradient per active GP (gp.mll / gp.dmll are written back as by update_mll_and_dmll!), then the
leave-one-out terms on the factorised K.  μ is the LOO mean of y - m(X).  A GP with info < 0 gets logp = -Inf and NaN rows.
"""
function eval_loo!(batch::GPBatch; grad::Bool = true, mu_var::Bool = false, active::Union{Nothing,Vector{UInt8}} = nothing)
    θ = thetas(batch)
    mll = fill(NaN, batch.B)
    g = fill(NaN, batch.P, batch.B)
    logp = fill(NaN, batch.B)
    gl = grad ? fill(NaN, batch.P, batch.B) : nothing
    μ = mu_var ? fill(NaN, batch.n, batch.B) : nothing
    σ2 = mu_var ? fill(NaN, batch.n, batch.B) : nothing
    info = zeros(Int32, batch.B)
    GC.@preserve θ mll g logp gl μ σ2 info active begin
        check(ccall((:gprb_eval_loo, LIB), Cint,
                    (Ptr{Cvoid}, Ptr{Float64}, Ptr{UInt8}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Int32}),
                    batch.handle, θ, active === nothing ? C_NULL : pointer(active), mll, g, logp, grad ? pointer(gl) : C_NULL,
                    mu_var ? pointer(μ) : C_NULL, mu_var ? pointer(σ2) : C_NULL, info))
    end
    for (b, gp) in enumerate(batch.gps)
        (active === nothing || active[b] != 0) || continue
        gp.mll = mll[b]; gp.target = mll[b]
        gp.dmll = g[:, b]; gp.dtarget = g[:, b]
    end
    batch.cache_key = zeros(0, 0)
    logp, gl, info, μ, σ2
end

loo_active(batch::GPBatch, slot::Int) = batch.B == 1 ? nothing : only_active(batch, slot)
loo_rows(P::Int, noise::Bool, kern::Bool) = vcat(noise ? [1] : Int[], kern ? collect(2:P) : Int[])   # [logNoise; kernel]: means have no parameters

"predict_LOO(batch) -> (μ::n×B, σ²::n×B): leave-one-out predictive mean (m(X) included) and variance at the training inputs."
function predict_LOO(batch::GPBatch)
    _, _, _, μ, σ2 = eval_loo!(batch; grad = false, mu_var = true)
    for (b, gp) in enumerate(batch.gps)
        gp.mean isa MeanZero && continue
        μ[:, b] .+= [GaussianProcesses.mean(gp.mean, gp.x[:, i]) for i in 1:batch.n]
    end
    μ, σ2
end
"logp_CVLOO(batch) -> logp::B (-Inf for a GP whose factorisation failed)."
logp_CVLOO(batch::GPBatch) = eval_loo!(batch; grad = false)[1]
"dlogpdθ_CVLOO(batch; noise, domean, kern) -> ∇::rows×B, rows of [logNoise; kernel params] selected by the flags."
dlogpdθ_CVLOO(batch::GPBatch; noise::Bool = true, domean::Bool = true, kern::Bool = true) =
    eval_loo!(batch; grad = true)[2][loo_rows(batch.P, noise, kern), :]

function predict_LOO(gp::B200GPE)
    batch, slot = residence(gp)
    _, _, info, μ, σ2 = eval_loo!(batch; grad = false, mu_var = true, active = loo_active(batch, slot))
    info[slot] < 0 && throw(PDMats.PosDefException(Int(info[slot])))
    mX = gp.mean isa MeanZero ? 0.0 : [GaussianProcesses.mean(gp.mean, gp.x[:, i]) for i in 1:batch.n]
    μ[:, slot] .+ mX, σ2[:, slot]
end
function logp_CVLOO(gp::B200GPE)
    batch, slot = residence(gp)
    logp, _, info = eval_loo!(batch; grad = false, active = loo_active(batch, slot))
    info[slot] < 0 && throw(PDMats.PosDefException(Int(info[slot])))
    logp[slot]
end
function dlogpdθ_CVLOO(gp::B200GPE; noise::Bool = true, domean::Bool = true, kern::Bool = true)
    batch, slot = residence(gp)
    _, ∇, info = eval_loo!(batch; grad = true, active = loo_active(batch, slot))
    info[slot] < 0 && throw(PDMats.PosDefException(Int(info[slot])))
    ∇[loo_rows(batch.P, noise, kern), slot]
end

# ---- predictive gradients: Jacobians of the posterior mean and variance with respect to the test inputs ---------------
# For the linearisation of a learned one-step map (stability analysis, Σₜ₊₁ = Jₜ Σₜ Jₜᵀ + diag σ²(xₜ), LQR / MPC).  ∂σ² is
# the gradient of the unclamped K** - K*ᵀK⁻¹K* (the same for σ²_f and σ²_y; predict_f's floor at 0 is not differentiated).
# A prior mean other than MeanZero needs its Jacobian from the caller (`mean_jacobian`): ForwardDiff cannot pass a ccall.
for name in (:predict_grad,)
    if isdefined(GaussianProcesses, name)
        @eval import GaussianProcesses: $name
    else
        @eval function $name end
        @eval export $name
    end
end

"""
    predict_grad(batch, Xstar::d×m; var=true, mean_jacobian=nothing) -> (μ::m×B, σ²::m×B | nothing, ∂μ::d×m×B, ∂σ²::d×m×B | nothing)

∂μ[p, j, b] = ∂μ_bj/∂x*_pj.  `var=false`: the mean and its Jacobian only (no triangular substitution on the device).
`mean_jacobian(b, x) -> d-vector` is the Jacobian of GP b's prior mean; required when a GP's mean is not MeanZero.
GPs without state give NaN columns.
"""
function predict_grad(batch::GPBatch, Xstar::AbstractMatrix; var::Bool = true, mean_jacobian = nothing)
    for gp in batch.gps
        gp.mean isa MeanZero || mean_jacobian !== nothing ||
            throw(ArgumentError("predict_grad: the prior mean $(typeof(gp.mean)) needs `mean_jacobian`"))
    end
    Xs = Matrix{Float64}(Xstar)
    d, m = size(Xs)
    mstar = prior_means(batch, Xs)
    dmstar = nothing
    if mstar !== nothing
        dmstar = zeros(d, m, batch.B)
        for b in 1:batch.B, j in 1:m
            batch.gps[b].mean isa MeanZero || (dmstar[:, j, b] .= mean_jacobian(b, Xs[:, j]))
        end
    end
    μ = Matrix{Float64}(undef, m, batch.B)
    σ2 = var ? Matrix{Float64}(undef, m, batch.B) : nothing
    ∂μ = Array{Float64,3}(undef, d, m, batch.B)
    ∂σ2 = var ? Array{Float64,3}(undef, d, m, batch.B) : nothing
    GC.@preserve Xs mstar dmstar μ σ2 ∂μ ∂σ2 begin
        check(ccall((:gprb_predict_grad, LIB), Cint,
                    (Ptr{Cvoid}, Int64, Ptr{Float64}, Int64, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}),
                    batch.handle, m, Xs, 0, mstar === nothing ? C_NULL : pointer(mstar), dmstar === nothing ? C_NULL : pointer(dmstar),
                    μ, var ? pointer(σ2) : C_NULL, ∂μ, var ? pointer(∂σ2) : C_NULL))
    end
    μ, σ2, ∂μ, ∂σ2
end

"predict_grad(gp, x::d×m; var=true, mean_jacobian=nothing) -> (μ::m, σ²::m, ∂μ::d×m, ∂σ²::d×m); `mean_jacobian(x) -> d-vector`."
function predict_grad(gp::B200GPE, x::AbstractMatrix; var::Bool = true, mean_jacobian = nothing)
    gp.mean isa MeanZero || mean_jacobian !== nothing ||
        throw(ArgumentError("predict_grad: the prior mean $(typeof(gp.mean)) needs `mean_jacobian`"))
    batch, slot = residence(gp)
    mj = mean_jacobian === nothing ? nothing : (b, xj) -> b == slot ? mean_jacobian(xj) : zeros(length(xj))
    if mj === nothing && !all(g -> g.mean isa MeanZero, batch.gps)
        mj = (b, xj) -> zeros(length(xj))  # the other GPs of the batch: their rows are not returned
    end
    μ, σ2, ∂μ, ∂σ2 = predict_grad(batch, x; var = var, mean_jacobian = mj)
    μ[:, slot], var ? σ2[:, slot] : nothing, ∂μ[:, :, slot], var ? ∂σ2[:, :, slot] : nothing
end

# ---- append! (ElasticGPE): new samples on resident GPs, only the block rows they reach refactorised ---------------------
# Base.append! is extended, nothing is exported.  The other GPs of the batch read the same device datasets, so a GPE that
# shares its batch moves to a batch of its own first (like optimize!).
"""
    append!(batch::GPBatch, xs::Vector{<:AbstractMatrix}, ys::AbstractMatrix) -> (mll::Vector{Float64}, info::Vector{Int32})

`xs`: one d × k block per distinct training set of the batch, in order of first use by GP index; `ys`: k × B raw targets
(m(x) is subtracted here).  Every GP with a resident state is conditioned on its enlarged data at the θ of that state;
GPs without a state get NaN and stay without one.
"""
function Base.append!(batch::GPBatch, xs::AbstractVector{<:AbstractMatrix}, ys::AbstractMatrix)
    uniq = IdDict{Any,Int}()
    for gp in batch.gps
        get!(uniq, gp.x, length(uniq) + 1)
    end
    length(xs) == length(uniq) || throw(ArgumentError("append!: expected $(length(uniq)) input blocks, got $(length(xs))"))
    d, k = batch.d, size(xs[1], 2)
    all(x -> size(x) == (d, k), xs) || throw(DimensionMismatch("append!: every input block must be $d × $k"))
    size(ys) == (k, batch.B) || throw(DimensionMismatch("append!: ys must be $k × $(batch.B)"))
    blocks = [Matrix{Float64}(x) for x in xs]
    ymm = Matrix{Float64}(undef, k, batch.B)
    for (x, t) in uniq
        members = [b for b in 1:batch.B if batch.gps[b].x === x]
        for j in 1:k, b in members
            ymm[j, b] = ys[j, b] - GaussianProcesses.mean(batch.gps[b].mean, blocks[t][:, j])
        end
    end
    mll = fill(NaN, batch.B)
    info = zeros(Int32, batch.B)
    ptrs = [pointer(x) for x in blocks]
    GC.@preserve blocks ymm mll info begin
        check(ccall((:gprb_batch_append, LIB), Cint, (Ptr{Cvoid}, Int64, Ptr{Ptr{Float64}}, Int64, Ptr{Float64}, Ptr{Float64}, Ptr{Int32}),
                    batch.handle, k, ptrs, d, ymm, mll, info))
    end
    grown = IdDict{Any,Matrix{Float64}}(x => hcat(x, blocks[t]) for (x, t) in uniq)
    for (b, gp) in enumerate(batch.gps)
        gp.x = grown[gp.x]
        gp.y = vcat(gp.y, ys[:, b])
        gp.nobs += k
        isnan(mll[b]) || (gp.mll = mll[b]; gp.target = mll[b])
    end
    batch.n += k
    batch.cache_key = zeros(0, 0)
    mll, info
end

"`append!(gp, x::d×k, y::k)`: ElasticGPE's append! on a B200-resident GPE; the GP ends evaluated at its current parameters."
function Base.append!(gp::B200GPE, x::AbstractMatrix, y::AbstractVector)
    batch, _ = residence(gp)
    if batch.B != 1
        batch = GPBatch(GPE[gp])
        evaluate!(batch; grad = false)
    end
    append!(batch, [x], reshape(Vector{Float64}(y), :, 1))
    gp
end

# ---- asynchronous rollout step (two trial groups alternate: device predict of one under the host projectv! of the other) -----
"Enqueue the mean prediction of GPs gp0:gp1 (1-based, inclusive) at the per-trial state blocks `states` (d × m × trials) on pipeline `slot`."
function predict_async!(batch::GPBatch, slot::Integer, gp0::Integer, gp1::Integer, states::Array{Float64,3}, G::Integer; var::Bool = false)
    d, m, _ = size(states)
    GC.@preserve states begin
        check(ccall((:gprb_predict_async, LIB), Cint,
                    (Ptr{Cvoid}, Int32, Int32, Int32, Int64, Ptr{Float64}, Int64, Int32, Ptr{Float64}, Int32),
                    batch.handle, slot, gp0 - 1, gp1, m, states, d * m, G, C_NULL, var ? 1 : 0))
    end
end
function predict_wait!(batch::GPBatch, slot::Integer, count::Integer, m::Integer; var::Bool = false)
    μ = Matrix{Float64}(undef, m, count)
    σ2 = var ? Matrix{Float64}(undef, m, count) : nothing
    check(ccall((:gprb_predict_wait, LIB), Cint, (Ptr{Cvoid}, Int32, Ptr{Float64}, Ptr{Float64}),
                batch.handle, slot, μ, var ? pointer(σ2) : C_NULL))
    μ, σ2
end

# ---- glue the experiment drivers need ---------------------------------------------------------------------------------
"config.json order `[σ_f, ℓ_1..ℓ_d]` (examples/config/README) -> GaussianProcesses order `[logNoise, ll_1..ll_d, lσ]` (CPnoise.jl:38)."
params_to_theta(params::AbstractVector; logNoise::Real = -2.0) = vcat(Float64(logNoise), log.(params[2:end]), log(params[1]))
"Inverse of params_to_theta: what parallelsearch stores in `config[\"params\"]` / the JSON checkpoints (core.jl:94-112, utils.jl:48-63)."
theta_to_params(θ::AbstractVector) = vcat(exp(θ[end]), exp.(θ[2:end-1]))

"""
    gather_results(local_rows::Dict{Int,Vector{Float64}}, ntrials, width) -> Matrix (width × ntrials)

The final gather of per-trial results across ranks (replaces the lock-guarded result callbacks of core.jl:47-56 when the
trials are sharded over GPUs): one ncclAllGather inside libgprb200.so.  Ranks join with `comm_init_rank!` (the 128-byte id
from `comm_unique_id()` on rank 0 travels through Distributed.jl / MPI / a file).  Rows are `kstep_mse`, `projectionerror`,
`params` ... in whatever layout `resultcallback!` needs; trial ids are 1-based here, 0-based in the C ABI.
"""
function gather_results(local_rows::Dict{Int,Vector{Float64}}, ntrials::Integer, width::Integer)
    ids = Int32[t - 1 for t in sort(collect(keys(local_rows)))]
    rows = isempty(ids) ? zeros(width, 0) : reduce(hcat, [local_rows[t + 1] for t in ids])     # width × count = row-major count × width
    out = Matrix{Float64}(undef, width, ntrials)
    check(ccall((:gprb_gather, LIB), Cint, (Ptr{Cvoid}, Int32, Int32, Int32, Ptr{Int32}, Ptr{Float64}, Ptr{Float64}),
                context(), ntrials, width, length(ids), ids, rows, out))
    out
end
function comm_unique_id()
    id = Vector{UInt8}(undef, 128)
    check(ccall((:gprb_comm_unique_id, LIB), Cint, (Ptr{Cvoid},), id))
    id
end
comm_init_rank!(nranks::Integer, rank::Integer, id::Vector{UInt8}) =
    check(ccall((:gprb_comm_init_rank, LIB), Cint, (Ptr{Cvoid}, Int32, Int32, Ptr{Cvoid}), context(), nranks, rank, id))

end # module
