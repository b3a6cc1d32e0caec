# Julia binding of libbnr for BayesianNetworkRegression.jl  --  the stub a maintainer adds to the package.
#
# It replaces the chain generation behind `Fit!` (generate_samples! / generate_samples_dbl!, src/gibbs.jl:897-1198:
# the pmap over initialize_and_run!, run!, the PSRF loops and return_psrf_VOI) with ONE `ccall` of `bnr_fit`
# (include/bnr.h).  Everything else of Fit! stays as it is: keyword handling, parameters.log, seed choice, setup_X!,
# Results / Summary.  NOT EXECUTED in the build image (no julia binary there); the identical C entry points are
# exercised by the Python/ctypes mirror and by the plain-C client tests/c/fit_client.c.
module BNRB200

using TypedTables

const libbnr = get(ENV, "LIBBNR", joinpath(@__DIR__, "..", "bayesiannetworkregression.jl_b200", "libbnr.so"))

# struct bnr_params (include/bnr.h) -- field for field
struct BnrParams
    n::Int32; V::Int32; R::Int32; num_chains::Int32; chain_offset::Int32; device::Int32
    trace_full_chains::Int32; trace_gamma_xi_all::Int32
    trace_rows::Int64; seed::UInt64
    eta::Float64; zeta::Float64; iota::Float64; a_delta::Float64; b_delta::Float64; nu::Float64
    gig_inject_len::Int32; gamma_mode::Int32; chain_groups::Int32; trace_gamma_xi_chains::Int32
end

# struct bnr_fit_params
struct BnrFitParams
    base::BnrParams
    nburn::Int64; nsamples::Int64; mingen::Int64; maxgen::Int64
    psrf_cutoff::Float64
    purge_burn::Int64
    return_state::Int32; n_devices::Int32; interval::Int32; ess_max_lag::Int32; verbose::Int32
    ext_world::Int32; ext_rank::Int32
    allgather::Ptr{Cvoid}; allgather_ctx::Ptr{Cvoid}
end

# struct bnr_fit_info
struct BnrFitInfo
    tot_generated::Int64; burn_in::Int64; sampled::Int64; rows::Int64; n_psrf::Int64
    streamed::Int32; summary_ok::Int32; ess_ok::Int32; gamma_mode::Int32; status_or::Int32
    total_chains::Int32; n_devices::Int32; exchange::Int32
end

const STATE_FULL = Int32(2)
# state variables in the order of the reference's Table (src/gibbs.jl:835-841) with their BNR_VAR_* ids
const VARS = ((:τ², 0), (:u, 1), (:ξ, 2), (:γ, 3), (:S, 4), (:θ, 5), (:Δ, 6), (:M, 7), (:μ, 8), (:λ, 9), (:πᵥ, 10))

fit_error() = unsafe_string(ccall((:bnr_fit_last_error, libbnr), Cstring, ()))
check(rc) = rc == 0 || error("libbnr error $rc: " * fit_error())

const PRED_MEAN = Int32(0)
const PRED_PREDICTIVE = Int32(1)

"""
    fit_b200(Xv, y, R; η, ζ, ι, aΔ, bΔ, ν, nburn, nsamp, mingen, maxgen, psrf_cutoff, num_chains, seed, purge_burn,
             n_devices = 1, X_new = nothing, predictive = false, loo = false)
        -> (state::Table, rhatξ::Vector, rhatγ::Vector, burn_in, sampled, prediction, loo)

Drop-in for the body of generate_samples! / generate_samples_dbl! after `setup_X!`: `Xv` is the n x q
`Matrix{Float64}`; the returned arrays have the reference's (iteration, d1, d2) layout, so
`Results(state, Table(ξ = rhatξ), Table(γ = rhatγ), burn_in, sampled)` is the same object `Fit!` returns today.
`num_chains` chains run on EACH of the `n_devices` GPUs (the reference runs one chain per Distributed.jl worker).
`X_new` (m x q, new networks vectorised by `setup_X!` like `Xv`) runs `bnr_fit_predict`: `prediction` is then
`(mean, lower, upper)` of μ + X_new γ (+ √τ² z with `predictive = true`) pooled over the retained draws of all chains
(95 % interval), else `nothing`.  `loo = true` runs `bnr_fit_loo` (with or without `X_new`): `loo` is then the
pointwise `(elpd_loo, p_loo, pareto_k, elpd_waic, p_waic)` (vectors of n) of PSIS-LOO and WAIC over the retained draws
of all chains (`nothing` when fewer than 2 draws were kept), else `nothing`.
"""
function fit_b200(Xv::Matrix{Float64}, y::Vector{Float64}, R::Integer; η = 1.01, ζ = 1.0, ι = 1.0, aΔ = 1.0, bΔ = 1.0,
                  ν = 10, nburn = 30000, nsamp = 20000, mingen = 0, maxgen = 0, psrf_cutoff = 1.01, num_chains = 2,
                  seed = 1, purge_burn = nothing, n_devices = 1, device = 0, verbose = false,
                  X_new::Union{Nothing,Matrix{Float64}} = nothing, predictive = false, loo = false)
    n, q = size(Xv)
    V = Int((-1 + sqrt(1 + 8q)) / 2)
    base = BnrParams(n, V, R, num_chains, 0, device, 1, 0, 0, UInt64(seed), η, ζ, ι, aΔ, bΔ, Float64(ν), 64, 0, 0, 1)
    p = Ref(BnrFitParams(base, nburn, nsamp, mingen, maxgen, psrf_cutoff, isnothing(purge_burn) ? 0 : purge_burn,
                         STATE_FULL, n_devices, 95, 0, verbose ? 1 : 0, 0, 0, C_NULL, C_NULL))
    res = Ref{Ptr{Cvoid}}(C_NULL)
    X_new === nothing || size(X_new, 2) == q || error("X_new must have the q = $q columns of Xv")
    if loo
        m = X_new === nothing ? 0 : size(X_new, 1)
        check(ccall((:bnr_fit_loo, libbnr), Cint,
                    (Ref{BnrFitParams}, Ptr{Float64}, Ptr{Float64}, Int32, Ptr{Float64}, Int32, Ref{Ptr{Cvoid}}),
                    p, Xv, y, Int32(m), X_new === nothing ? Ptr{Float64}(C_NULL) : X_new,
                    predictive ? PRED_PREDICTIVE : PRED_MEAN, res))
    elseif X_new === nothing
        check(ccall((:bnr_fit, libbnr), Cint, (Ref{BnrFitParams}, Ptr{Float64}, Ptr{Float64}, Ref{Ptr{Cvoid}}), p, Xv, y, res))
    else
        check(ccall((:bnr_fit_predict, libbnr), Cint,
                    (Ref{BnrFitParams}, Ptr{Float64}, Ptr{Float64}, Int32, Ptr{Float64}, Int32, Ref{Ptr{Cvoid}}),
                    p, Xv, y, Int32(size(X_new, 1)), X_new, predictive ? PRED_PREDICTIVE : PRED_MEAN, res))
    end
    try
        info = Ref{BnrFitInfo}()
        check(ccall((:bnr_fit_get_info, libbnr), Cint, (Ptr{Cvoid}, Ref{BnrFitInfo}), res[], info))
        rows = Int(info[].rows)
        dims = Dict(:τ² => (1, 1), :u => (R, V), :ξ => (V, 1), :γ => (q, 1), :S => (q, 1), :θ => (1, 1), :Δ => (1, 1),
                    :M => (R, R), :μ => (1, 1), :λ => (R, 1), :πᵥ => (R, 3))
        cols = Dict{Symbol,Array{Float64,3}}()
        for (name, id) in VARS
            a = Array{Float64,3}(undef, rows, dims[name]...)          # iteration is the fastest index, as in the reference
            check(ccall((:bnr_fit_state, libbnr), Cint, (Ptr{Cvoid}, Int32, Ptr{Float64}), res[], Int32(id), a))
            cols[name] = a
        end
        rξ = Vector{Float64}(undef, V); rγ = Vector{Float64}(undef, q)
        check(ccall((:bnr_fit_rhat, libbnr), Cint, (Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}), res[], rξ, rγ))
        state = Table(τ² = cols[:τ²], u = cols[:u], ξ = cols[:ξ], γ = cols[:γ], S = cols[:S], θ = cols[:θ], Δ = cols[:Δ],
                      M = cols[:M], μ = cols[:μ], λ = cols[:λ], πᵥ = cols[:πᵥ])
        prediction = nothing
        if X_new !== nothing
            m = size(X_new, 1)
            pm = Vector{Float64}(undef, m); pl = Vector{Float64}(undef, m); ph = Vector{Float64}(undef, m)
            check(ccall((:bnr_fit_prediction, libbnr), Cint, (Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}),
                        res[], pm, pl, ph))
            prediction = (mean = pm, lower = pl, upper = ph)
        end
        pointwise = nothing
        if loo
            pw = ntuple(_ -> Vector{Float64}(undef, n), 5)
            rc = ccall((:bnr_fit_loo_pointwise, libbnr), Cint,
                       (Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}), res[], pw...)
            rc == -4 || check(rc)           # BNR_ESTATE: fewer than 2 retained draws
            rc == 0 && (pointwise = (elpd_loo = pw[1], p_loo = pw[2], pareto_k = pw[3], elpd_waic = pw[4], p_waic = pw[5]))
        end
        return state, rξ, rγ, Int(info[].burn_in), Int(info[].sampled), prediction, pointwise
    finally
        ccall((:bnr_fit_free, libbnr), Cint, (Ptr{Cvoid},), res[])
    end
end

end # module
