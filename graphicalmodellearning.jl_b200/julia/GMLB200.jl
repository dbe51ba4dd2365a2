# GMLB200.jl -- reference-side binding of libgml_b200.so.
#
# Drop this file next to src/GraphicalModelLearning.jl and `include("GMLB200.jl")` it from the module
# (after the GMLMethod / formulation definitions, src/GraphicalModelLearning.jl:20-65), then add
# `export B200` next to `export GMLMethod, NLP` (src/GraphicalModelLearning.jl:6).  Nothing else in the
# package changes: `learn(samples, RISE(), B200())` dispatches here, `learn(samples)` and
# `learn(samples, formulation)` keep selecting NLP() (:69-70), and Adjoint inputs reach these methods
# through the existing shim at :73.
#
# NOTE: the build image has no Julia toolchain, so this file is not executed by the test-suite; the
# ctypes mirror (graphicalmodellearning.jl_b200/api.py) calls the same C symbols with the same memory
# layout and is what tests/ exercise.  Keep the two in sync.

const _libgml_b200 = get(ENV, "GML_B200_LIB", "libgml_b200.so")

# struct gml_b200_opts (include/gml_b200.h)
mutable struct _GMLB200Opts
    tol::Cdouble
    barrier_mu::Cdouble
    max_iter::Int32
    solver::Int32
    device::Int32
    node_begin::Int32
    node_end::Int32
    verbose::Int32
    stream::Ptr{Cvoid}
    reserved::NTuple{8,Int32}
end

# struct gml_b200_stats (include/gml_b200.h)
mutable struct GMLB200Stats
    solver_used::Int32
    iterations::Int32
    n_fg_passes::Int32
    n_f_passes::Int32
    n_unconverged::Int32
    n_stalled::Int32
    kernel_launches::Int64
    evals::Cdouble
    pack_ms::Cdouble
    h2d_ms::Cdouble
    solve_ms::Cdouble
    d2h_ms::Cdouble
    total_ms::Cdouble
    max_residual::Cdouble
    reserved_d::NTuple{4,Cdouble}
    GMLB200Stats() = new(0, 0, 0, 0, 0, 0, 0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, (0.0, 0.0, 0.0, 0.0))
end

"""
    B200(; tol=0.0, max_iter=0, solver=:auto, barrier_mu=0.0, device=0, devices=1, verbose=0)

Batched GPU method.  `tol`: stopping tolerance (max-norm of the proximal-gradient mapping for the
FISTA solvers, Newton step for the small-problem solver; 0 selects 1e-6 / 1e-12).  `barrier_mu > 0`
returns the log-barrier point Ipopt stops at instead of the exact L1 minimiser (1e-9 reproduces the
stored test fixtures to ~1e-9; available for problems with at most 64 features per node).  `devices > 1` splits
the work over that many GPUs (device, device+1, ...) from this one Julia process: histogram rows when every device keeps
at least 65536 of them (sample-sharded solve, NCCL all-reduce per pass), node shards otherwise.
"""
mutable struct B200 <: GMLMethod
    tol::Float64
    max_iter::Int
    solver::Symbol
    barrier_mu::Float64
    device::Int
    devices::Int
    verbose::Int
    stats::GMLB200Stats
end
B200(; tol=0.0, max_iter=0, solver=:auto, barrier_mu=0.0, device=0, devices=1, verbose=0) =
    B200(tol, max_iter, solver, barrier_mu, device, devices, verbose, GMLB200Stats())

const _gml_b200_solver_id = Dict(:auto => 0, :newton => 1, :fista_cc => 2, :fista_tc => 3)

function _gml_b200_opts(m::B200)
    _GMLB200Opts(m.tol, m.barrier_mu, Int32(m.max_iter), Int32(_gml_b200_solver_id[m.solver]), Int32(m.device),
                 Int32(0), Int32(0), Int32(m.verbose), C_NULL,
                 (Int32(0), Int32(0), Int32(0), Int32(0), Int32(m.devices), Int32(0), Int32(0), Int32(0)))   # reserved[4] = devices
end

function _gml_b200_check(rc::Integer)
    rc == 0 && return
    msg = unsafe_string(ccall((:gml_b200_last_error, _libgml_b200), Cstring, ()))
    # same caller-visible behaviour as the reference's @assert LOCALLY_SOLVED (:180): an exception
    error("gml_b200 error $(rc): $(msg)")
end

# element types the library ingests directly from the reference's K x (N+1) `samples` matrix (include/gml_b200.h:
# GML_B200_DTYPE_*); any other Real is converted to Float64 first
const _gml_b200_dtype = Dict(Float64 => 0, Int64 => 1, Float32 => 2, Int32 => 3, Int8 => 4)
_gml_b200_native(samples::Array{T,2}) where T <: Real = haskey(_gml_b200_dtype, T) ? samples : Float64.(samples)

function _gml_b200_pairwise(samples::Array{T,2}, formulation_id::Integer, regularizer::Real,
                            symmetrization::Bool, method::B200) where T <: Real
    # `samples` goes to the library AS IS (column-major, ld = num_conf): data_info (:76-81), lambda (:157), the narrowing of
    # the spins to bytes (threaded, validated) and the transfer all happen inside the call
    native = _gml_b200_native(samples)
    num_conf, num_spins = size(native, 1), size(native, 2) - 1
    reconstruction = Array{Float64}(undef, num_spins, num_spins)                            # :159
    opts = _gml_b200_opts(method)
    GC.@preserve native reconstruction begin
        rc = ccall((:gml_b200_learn_pairwise_matrix, _libgml_b200), Cint,
                   (Ptr{Cvoid}, Int32, Int64, Int32, Int64, Int32, Cdouble, Int32,
                    Ref{_GMLB200Opts}, Ptr{Cdouble}, Ptr{Cdouble}, Ref{GMLB200Stats}),
                   native, _gml_b200_dtype[eltype(native)], num_conf, num_spins, num_conf, formulation_id,
                   Float64(regularizer), symmetrization ? 1 : 0, opts, reconstruction, C_NULL, method.stats)
    end
    _gml_b200_check(rc)
    return reconstruction          # column-major N x N, row u = node u, diagonal = fields (:181-188)
end

learn(samples::Array{T,2}, formulation::RISE, method::B200) where T <: Real =
    _gml_b200_pairwise(samples, 0, formulation.regularizer, formulation.symmetrization, method)
learn(samples::Array{T,2}, formulation::logRISE, method::B200) where T <: Real =
    _gml_b200_pairwise(samples, 1, formulation.regularizer, formulation.symmetrization, method)
learn(samples::Array{T,2}, formulation::RPLE, method::B200) where T <: Real =
    _gml_b200_pairwise(samples, 2, formulation.regularizer, formulation.symmetrization, method)

function learn(samples::Array{T,2}, formulation::multiRISE, method::B200) where T <: Real
    native = _gml_b200_native(samples)
    num_conf, num_spins = size(native, 1), size(native, 2) - 1
    inter_order = formulation.interaction_order
    n_keys = ccall((:gml_b200_multibody_num_keys, _libgml_b200), Int64, (Int32, Int32), num_spins, inter_order)
    vals = Array{Float64}(undef, n_keys, num_spins)      # vals[f, u] == out_vals[u*n_keys + f] of the C side
    opts = _gml_b200_opts(method)
    GC.@preserve native vals begin
        rc = ccall((:gml_b200_learn_multibody_matrix, _libgml_b200), Cint,
                   (Ptr{Cvoid}, Int32, Int64, Int32, Int64, Int32, Cdouble,
                    Ref{_GMLB200Opts}, Ptr{Cdouble}, Ptr{Cdouble}, Ref{GMLB200Stats}),
                   native, _gml_b200_dtype[eltype(native)], num_conf, num_spins, num_conf, inter_order,
                   Float64(formulation.regularizer), opts, vals, C_NULL, method.stats)      # lambda of :86 inside
    end
    _gml_b200_check(rc)

    # rebuild the reference's Dict with the reference's own key enumeration (:91-109, models.jl:228-246)
    reconstruction = Dict{Tuple,Real}()
    for current_spin = 1:num_spins
        nodal_keys = Tuple[(current_spin,)]
        neighbours = [i for i=1:num_spins if i!=current_spin]
        for p = 2:inter_order
            perm = permutations(neighbours, p - 1)
            append!(nodal_keys, [(current_spin, perm[i]...) for i=1:length(perm)])
        end
        for (f, key) in enumerate(nodal_keys)
            reconstruction[key] = vals[f, current_spin]
        end
    end

    if formulation.symmetrization      # mean over the per-node estimates of each sorted key (:135-149)
        groups = Dict{Tuple,Vector{Float64}}()
        for (k, v) in reconstruction
            push!(get!(groups, Tuple(sort(collect(k))), Float64[]), v)
        end
        reconstruction = Dict{Tuple,Real}(k => mean(v) for (k, v) in groups)
    end

    return FactorGraph(inter_order, num_spins, :spin, reconstruction)                       # :151
end

"""
    B200Exact(; seed=0, device=0)

Exact iid sampler on the GPU: the distribution of the reference's `sample` (src/sampling.jl:58-106), drawn by enumerating
all 2^N configurations in blocks on the device, for N <= 40.  The draws depend only on (model, number_sample, replicates,
seed); rows come out in increasing configuration index.
"""
struct B200Exact <: GMLSampler
    seed::UInt64
    device::Int
end
B200Exact(; seed=0, device=0) = B200Exact(UInt64(seed), device)

# the term lists of the sampler entry points: n_terms x order 0-based spin ids (-1 padded) and fp64 weights
function _gml_b200_terms(gm::FactorGraph)
    if gm.alphabet != :spin                                                                 # src/sampling.jl:95-97
        error("sampling is only supported for spin alphabets, not $(gm.alphabet)")
    end
    order = maximum(length(k) for k in keys(gm.terms); init=1)
    n_terms = length(gm.terms)
    term_idx = fill(Int32(-1), order, max(n_terms, 1))     # column t = term t: the C side's n_terms x order row-major array
    term_weight = zeros(Float64, max(n_terms, 1))
    for (t, (key, weight)) in enumerate(gm.terms)
        for (m, i) in enumerate(key)
            term_idx[m, t] = Int32(i - 1)
        end
        term_weight[t] = Float64(weight)
    end
    return order, n_terms, term_idx, term_weight
end

# the replicates' [count, s_1..s_N] matrices (src/sampling.jl:53-54) from the rows the library wrote at consecutive offsets
function _gml_b200_replicates(counts, spins, out_K)
    out = Vector{Array{Int64,2}}(undef, length(out_K))
    first = 1
    for r in eachindex(out_K)
        last = first + out_K[r] - 1
        out[r] = hcat(Int64.(counts[first:last]), Int64.(spins[first:last, :]))
        first = last + 1
    end
    return out
end

function sample(gm::FactorGraph{T}, number_sample::Integer, replicates::Integer, sampler::B200Exact) where T <: Real
    num_spins = gm.varible_count
    order, n_terms, term_idx, term_weight = _gml_b200_terms(gm)
    rows = replicates * min(number_sample, 2^min(num_spins, 62))
    out_K = zeros(Int64, replicates)
    # host buffers of the largest possible size (min(n, 2^N) rows per replicate); the library stages them on the device
    counts = Array{Float64}(undef, rows)
    spins = Array{Int8}(undef, rows, num_spins)              # column-major: spins[:, i] == the C side's row i (ld = rows)
    GC.@preserve term_idx term_weight out_K counts spins begin
        rc = ccall((:gml_b200_sample_exact_device, _libgml_b200), Cint,
                   (Int32, Int32, Int32, Int32, Ptr{Int32}, Ptr{Cdouble}, Int64, Int32, UInt64, Ptr{Int64}, Ptr{Cdouble},
                    Ptr{Cdouble}, Ptr{Int8}, Int64, Ptr{Cvoid}),
                   sampler.device, num_spins, order, n_terms, term_idx, term_weight, number_sample, replicates, sampler.seed,
                   out_K, C_NULL, counts, spins, rows, C_NULL)
    end
    _gml_b200_check(rc)
    return _gml_b200_replicates(counts, spins, out_K)
end

sample(gm::FactorGraph, number_sample::Integer, sampler::B200Exact) = sample(gm, number_sample, 1, sampler)[1]

"""
    B200Gibbs(; seed=0, device=0, chains=0, burn_in=200, thin=10)

Multi-sample Gibbs sampler on the GPU for N <= 4096 spins and terms of order <= 8.  Each of `chains` chains (0 selects
min(round_up(number_sample, 32), 2^17)) runs `burn_in` systematic-scan sweeps from a random start, then records its
configuration after every `thin`-th sweep.  The draws depend only on (model, number_sample, replicates, seed, chains,
burn_in, thin).  Up to 64 spins each replicate is a histogram in increasing configuration index; beyond, one row of count 1
per draw.  `rhat` receives, per replicate of the last call, the split-R-hat (energy, magnetisation) over the chains' halves.
"""
mutable struct B200Gibbs <: GMLSampler
    seed::UInt64
    device::Int
    chains::Int
    burn_in::Int
    thin::Int
    rhat::Vector{NTuple{2,Float64}}
end
B200Gibbs(; seed=0, device=0, chains=0, burn_in=200, thin=10) =
    B200Gibbs(UInt64(seed), device, chains, burn_in, thin, NTuple{2,Float64}[])

function sample(gm::FactorGraph{T}, number_sample::Integer, replicates::Integer, sampler::B200Gibbs) where T <: Real
    num_spins = gm.varible_count
    order, n_terms, term_idx, term_weight = _gml_b200_terms(gm)
    rows = replicates * (num_spins <= 62 ? min(number_sample, 2^num_spins) : number_sample)
    out_K = zeros(Int64, replicates)
    rhat = zeros(Float64, 2, replicates)
    counts = Array{Float64}(undef, rows)
    spins = Array{Int8}(undef, rows, num_spins)
    GC.@preserve term_idx term_weight out_K rhat counts spins begin
        rc = ccall((:gml_b200_sample_mcmc_device, _libgml_b200), Cint,
                   (Int32, Int32, Int32, Int32, Ptr{Int32}, Ptr{Cdouble}, Int64, Int32, Int64, Int32, Int32, UInt64, Ptr{Int64},
                    Ptr{Cdouble}, Ptr{Cdouble}, Ptr{Int8}, Int64, Ptr{Cvoid}),
                   sampler.device, num_spins, order, n_terms, term_idx, term_weight, number_sample, replicates, sampler.chains,
                   sampler.burn_in, sampler.thin, sampler.seed, out_K, rhat, counts, spins, rows, C_NULL)
    end
    _gml_b200_check(rc)
    sampler.rhat = [(rhat[1, r], rhat[2, r]) for r in 1:replicates]
    return _gml_b200_replicates(counts, spins, out_K)
end

sample(gm::FactorGraph, number_sample::Integer, sampler::B200Gibbs) = sample(gm, number_sample, 1, sampler)[1]

const GML_B200_TEMPERING_DEFAULT_RUNGS = 16   # include/gml_b200.h

"""
    B200Tempering(; seed=0, device=0, chains=0, burn_in=200, thin=10, betas=Float64[])

Replica-exchange (parallel tempering) sampler on the GPU for models whose B200Gibbs chains do not mix; N <= 4096 spins,
terms of order <= 8.  Each chain is a ladder of replicas at the inverse temperatures `betas` (betas[1] = 1, strictly
decreasing, non-negative; 2, 4, 8, 16 or 32 rungs; empty selects the library's default, 16 rungs geometric from 1 to 0.1)
that exchange states between adjacent rungs after every sweep; only the beta = 1 replica records.  `chains` = 0 selects
min(round_up(number_sample, 32/R), 2^17/R) ladders of R rungs; a draw costs about R times a B200Gibbs draw.  `rhat`
receives, per replicate of the last call, the split-R-hat (energy, magnetisation); `swap_rate` the fraction of accepted
swaps of each adjacent pair of rungs after burn_in.
"""
mutable struct B200Tempering <: GMLSampler
    seed::UInt64
    device::Int
    chains::Int
    burn_in::Int
    thin::Int
    betas::Vector{Float64}
    rhat::Vector{NTuple{2,Float64}}
    swap_rate::Vector{Vector{Float64}}
end
B200Tempering(; seed=0, device=0, chains=0, burn_in=200, thin=10, betas=Float64[]) =
    B200Tempering(UInt64(seed), device, chains, burn_in, thin, Float64.(betas), NTuple{2,Float64}[], Vector{Float64}[])

function sample(gm::FactorGraph{T}, number_sample::Integer, replicates::Integer, sampler::B200Tempering) where T <: Real
    num_spins = gm.varible_count
    order, n_terms, term_idx, term_weight = _gml_b200_terms(gm)
    rows = replicates * (num_spins <= 62 ? min(number_sample, 2^num_spins) : number_sample)
    n_rungs = length(sampler.betas)
    pairs = (n_rungs == 0 ? GML_B200_TEMPERING_DEFAULT_RUNGS : n_rungs) - 1
    betas = sampler.betas
    out_K = zeros(Int64, replicates)
    rhat = zeros(Float64, 2, replicates)
    swap = zeros(Float64, pairs, replicates)
    counts = Array{Float64}(undef, rows)
    spins = Array{Int8}(undef, rows, num_spins)
    GC.@preserve term_idx term_weight betas out_K rhat swap counts spins begin
        rc = ccall((:gml_b200_sample_tempering_device, _libgml_b200), Cint,
                   (Int32, Int32, Int32, Int32, Ptr{Int32}, Ptr{Cdouble}, Int32, Ptr{Cdouble}, Int64, Int32, Int64, Int32, Int32,
                    UInt64, Ptr{Int64}, Ptr{Cdouble}, Ptr{Cdouble}, Ptr{Cdouble}, Ptr{Int8}, Int64, Ptr{Cvoid}),
                   sampler.device, num_spins, order, n_terms, term_idx, term_weight, n_rungs,
                   n_rungs == 0 ? Ptr{Cdouble}(C_NULL) : pointer(betas), number_sample, replicates, sampler.chains,
                   sampler.burn_in, sampler.thin, sampler.seed, out_K, rhat, swap, counts, spins, rows, C_NULL)
    end
    _gml_b200_check(rc)
    sampler.rhat = [(rhat[1, r], rhat[2, r]) for r in 1:replicates]
    sampler.swap_rate = [swap[:, r] for r in 1:replicates]
    return _gml_b200_replicates(counts, spins, out_K)
end

sample(gm::FactorGraph, number_sample::Integer, sampler::B200Tempering) = sample(gm, number_sample, 1, sampler)[1]
