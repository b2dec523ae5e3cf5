# NHPB200.jl -- the reference-side binding a maintainer adds to NetworkHawkesProcesses.jl so that its event-history hot
# path runs in libnhp.so (include/nhp.h) on B200s.  The package API is unchanged and so are its callers: `mle!`, `mcmc!`, `vb!`,
# `resample!`, `update!` and `plot` run exactly the code they run today.  Every method below carries a name the reference
# already has; it is either
#   (R) a REDEFINITION of a hot-path method for the reference's own argument types (loglikelihood, intensity,
#       resample_parents, update_parents, convolve, resample_adjacency_matrix!, rand), or
#   (E) an EXTENSION of a reference function to the lazy device-side result types defined here (FusedParents, FusedCounts,
#       FusedVB, DeviceConvolved), which is how the fused statistics reach the unchanged `resample!` / `update!` bodies:
#       `resample_parents` returns a FusedParents, the reference hands it on to `resample!(process.weights, data, parents)`,
#       whose first line is `sufficient_statistics(model, data, parents)` -- and that call lands on the method below, which
#       reads the statistics the sweep already accumulated instead of re-scanning the parent vectors.
# A FusedParents still destructures as `parents, parentnodes = resample_parents(process, data)` (the vectors are exported from
# the device on first use), and a DeviceConvolved is an AbstractArray{Float64,3} (exported on first indexing), so user code
# that looks inside them keeps working.
#
# This file cannot be executed in the build image (no Julia toolchain, SURVEY.md section 8c); the Python mirror
# (networkhawkesprocesses.jl_b200/nhp_b200) binds the same symbols with ctypes and is what the tests drive.
#
# Usage:   using NetworkHawkesProcesses; include("NHPB200.jl"); NHPB200.init!("/path/to/libnhp.so")
#          multi-GPU (one Julia process per GPU): NHPB200.init_comm!(id, rank, nranks) with id = NHPB200.unique_id() of rank 0
module NHPB200

using NetworkHawkesProcesses
import NetworkHawkesProcesses: loglikelihood, intensity, rand, resample_parents, update_parents, resample_adjacency_matrix!, convolve,
    sufficient_statistics, parent_counts, resample!, update!,
    ContinuousHawkesProcess, ContinuousStandardHawkesProcess, ContinuousNetworkHawkesProcess,
    DiscreteHawkesProcess, DiscreteStandardHawkesProcess, DiscreteNetworkHawkesProcess,
    HomogeneousProcess, DiscreteHomogeneousProcess, Weights, DenseWeightModel,
    ExponentialImpulseResponse, LogitNormalImpulseResponse, DiscreteGaussianImpulseResponse,
    BernoulliNetworkModel, link_probability, ndims, basis, fillna!, variational_log_expectation
using Distributions: Gamma, Dirichlet
using LinearAlgebra: cholesky, Symmetric

const LIB = Ref{String}("libnhp")
const CTX = Ref{Ptr{Cvoid}}(C_NULL)
const SWEEP = Ref{UInt64}(0)     # Philox counter: one value per sweep; the seed is drawn from Julia's RNG per call

function check(rc::Cint)
    rc == 0 && return
    msg = unsafe_string(ccall((:nhp_last_error, LIB[]), Cstring, (Ptr{Cvoid},), CTX[]))
    error("libnhp error $rc: $msg")          # the reference throws `error(...)` / DomainError at the same places
end

function init!(lib::String="libnhp"; device::Integer=0)
    LIB[] = lib
    ctx = Ref{Ptr{Cvoid}}(C_NULL)
    rc = ccall((:nhp_create, LIB[]), Cint, (Cint, Ref{Ptr{Cvoid}}), device, ctx)
    rc == 0 || error("nhp_create failed ($rc): " * unsafe_string(ccall((:nhp_last_error, LIB[]), Cstring, (Ptr{Cvoid},), C_NULL)))
    CTX[] = ctx[]
    atexit(() -> ccall((:nhp_destroy, LIB[]), Cint, (Ptr{Cvoid},), CTX[]))
    return nothing
end

# ---- multi-GPU: the 128-byte id of rank 0 travels by whatever the host has (MPI.jl, Distributed.jl, a file) ------------------------
function unique_id()
    id = Vector{UInt8}(undef, 128)
    check(ccall((:nhp_comm_unique_id, LIB[]), Cint, (Ptr{UInt8},), id))
    return id
end
init_comm!(id::Vector{UInt8}, rank::Integer, nranks::Integer) =
    check(ccall((:nhp_comm_init, LIB[]), Cint, (Ptr{Cvoid}, Ptr{UInt8}, Cint, Cint), CTX[], id, rank, nranks))
function comm_rank()
    r = Ref{Cint}(0); n = Ref{Cint}(1)
    ccall((:nhp_comm_rank, LIB[]), Cint, (Ptr{Cvoid}, Ref{Cint}, Ref{Cint}), CTX[], r, n)
    return Int(r[]), Int(n[])
end
allreduce!(x::Vector{Float64}) = (check(ccall((:nhp_comm_allreduce_host, LIB[]), Cint, (Ptr{Cvoid}, Ptr{Float64}, Int64), CTX[], x, length(x))); x)

# ---- device-resident data: upload once, reuse across the thousands of mle!/mcmc! evaluations ----------------------------------------
# Cache keyed by the IDENTITY of the caller's array (objectid) and holding it through a WeakRef only: the handle is freed by its
# finalizer once the caller drops the data, and a cheap fingerprint catches in-place mutation (ADVICE r1: an IdDict keyed on a fresh
# `Matrix{Int64}(data)` copy never hit and pinned every upload for ever).
mutable struct DeviceEvents
    h::Ptr{Cvoid}          # this rank's time shard (the whole stream on one GPU)
    full::Ptr{Cvoid}       # the unsharded stream (adjacency sampler: columns are partitioned, not time); == h on one GPU
    n::Int
    duration::Float64
end
mutable struct DeviceCounts
    h::Ptr{Cvoid}
    N::Int
    T::Int
    convolved::Bool
end
struct CacheEntry{H}
    key::WeakRef
    fingerprint::UInt
    handle::H
end
const EVENT_CACHE = Dict{UInt,CacheEntry{DeviceEvents}}()
const COUNT_CACHE = Dict{UInt,CacheEntry{DeviceCounts}}()
fingerprint(a::AbstractArray) = isempty(a) ? UInt(0) : hash((length(a), first(a), last(a), a[cld(length(a), 2)], sum(@view a[1:max(1, length(a) ÷ 1024):end])))
function cached(make::Function, cache::Dict{UInt,CacheEntry{H}}, key) where {H}
    for (k, e) in cache                      # drop the entries whose data died
        e.key.value === nothing && delete!(cache, k)
    end
    id, fp = objectid(key), fingerprint(key)
    e = get(cache, id, nothing)
    (e !== nothing && e.key.value === key && e.fingerprint == fp) && return e.handle
    h = make()
    cache[id] = CacheEntry{H}(WeakRef(key), fp, h)
    return h
end

function upload_events(events, nodes::Vector{Int64}, first::Int, last::Int, halo::Int, duration, K, flags)
    h = Ref{Ptr{Cvoid}}(C_NULL)
    lo = first - halo
    check(ccall((:nhp_events_upload, LIB[]), Cint,
        (Ptr{Cvoid}, Ptr{Float64}, Ptr{Int64}, Int64, Float64, Int64, Int64, Int64, Cint, Ref{Ptr{Cvoid}}),
        CTX[], pointer(events, lo), pointer(nodes, lo), last - lo + 1, Float64(duration), K, halo, lo - 1, flags, h))
    return h[]
end

function device_events(process, data)
    events, nodes, duration = data
    cached(EVENT_CACHE, events) do
        nodes64 = convert(Vector{Int64}, nodes)            # a no-op when the type already matches
        n, K = length(events), ndims(process)
        rank, nranks = comm_rank()
        full = upload_events(events, nodes64, 1, n, 0, duration, K, 1)
        if nranks == 1 || n == 0
            shard = full
        else                                               # contiguous time shard + the predecessors within the look-back horizon
            push_params!(process)
            hz = Ref{Float64}(0.0)
            check(ccall((:nhp_cont_horizon, LIB[]), Cint, (Ptr{Cvoid}, Int64, Cint, Ref{Float64}), CTX[], n, 1, hz))
            i0, i1 = rank * n ÷ nranks + 1, (rank + 1) * n ÷ nranks
            lo = rank == 0 ? i0 : searchsortedlast(events, events[i0] - hz[]) + 1
            shard = upload_events(events, nodes64, i0, i1, i0 - min(lo, i0), duration, K, rank == 0 ? 1 : 0)
        end
        ev = DeviceEvents(shard, full, n, Float64(duration))
        finalizer(ev) do e
            e.h != e.full && ccall((:nhp_events_free, LIB[]), Cint, (Ptr{Cvoid}, Ptr{Cvoid}), CTX[], e.h)
            ccall((:nhp_events_free, LIB[]), Cint, (Ptr{Cvoid}, Ptr{Cvoid}), CTX[], e.full)
        end
        ev
    end
end

kind(::ExponentialImpulseResponse) = Cint(0)
kind(::LogitNormalImpulseResponse) = Cint(1)
p1(i::ExponentialImpulseResponse) = convert(Matrix{Float64}, i.θ)
p1(i::LogitNormalImpulseResponse) = convert(Matrix{Float64}, i.μ)
p2(i::ExponentialImpulseResponse) = C_NULL
p2(i::LogitNormalImpulseResponse) = convert(Matrix{Float64}, i.τ)
adjacency(p::ContinuousStandardHawkesProcess) = C_NULL
adjacency(p::ContinuousNetworkHawkesProcess) = Matrix{Float64}(p.adjacency_matrix)   # Bool / Int64 / Float64 -> Float64

function push_params!(process::ContinuousHawkesProcess)
    K = ndims(process)
    check(ccall((:nhp_cont_params_set, LIB[]), Cint,
        (Ptr{Cvoid}, Cint, Int64, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Float64),
        CTX[], kind(process.impulses), K, baseline_rates(process.baseline), convert(Matrix{Float64}, process.weights.W),
        adjacency(process), p1(process.impulses), p2(process.impulses), Float64(process.impulses.Δtmax)))
    push_baseline!(process)   # LogGaussianCoxProcess: the curves replace the homogeneous rates inside the sweeps
end
baseline_rates(b::HomogeneousProcess) = convert(Vector{Float64}, b.λ)
baseline_rates(b::LogGaussianCoxProcess) = Float64[sum(l) / length(l) for l in b.λ]   # placeholder rates; the grid takes over

# ================================================== continuous path =============================================================
# (R) continuous.jl:210 / :360.  On several GPUs every rank computes its shard's share and the shares are summed (NCCL).
function loglikelihood(process::ContinuousHawkesProcess, data; recursive=true)
    ev = device_events(process, data)
    push_params!(process)
    ll = Ref{Float64}(0.0)
    check(ccall((:nhp_cont_loglik, LIB[]), Cint, (Ptr{Cvoid}, Ptr{Cvoid}, Cint, Ref{Float64}), CTX[], ev.h, recursive ? 1 : 0, ll))
    return allreduce!([ll[]])[1]
end

# extension for mle! (Optim.only_fg!): objective + analytic gradient in the layout of params(process), continuous.jl:116-119
function loglikelihood_gradient(process::ContinuousStandardHawkesProcess, data; recursive=true)
    ev = device_events(process, data)
    push_params!(process)
    K = ndims(process)
    ll = Ref{Float64}(0.0)
    dλ = Vector{Float64}(undef, K); dW = Matrix{Float64}(undef, K, K); d1 = Matrix{Float64}(undef, K, K); d2 = Matrix{Float64}(undef, K, K)
    check(ccall((:nhp_cont_loglik_grad, LIB[]), Cint,
        (Ptr{Cvoid}, Ptr{Cvoid}, Cint, Ref{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}),
        CTX[], ev.h, recursive ? 1 : 0, ll, dλ, dW, d1, d2))
    impulse_grad = process.impulses isa ExponentialImpulseResponse ? vec(d1) : [vec(d1); vec(d2)]
    g = allreduce!([ll[]; dλ; impulse_grad; vec(dW)])
    return g[1], g[2:end]
end

# (R) continuous.jl:76 / :84.  Query times are partitioned over the ranks (SURVEY 8e); a single GPU answers them all.
function intensity(process::ContinuousHawkesProcess, data, times::Vector{Float64})
    ev = device_events(process, data)
    push_params!(process)
    out = Matrix{Float64}(undef, length(times), ndims(process))          # column-major [q + nq*k]
    check(ccall((:nhp_cont_intensity, LIB[]), Cint, (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Float64}, Int64, Ptr{Float64}),
        CTX[], ev.full, times, length(times), out))
    return out
end
intensity(process::ContinuousHawkesProcess, data, time::Float64) = vec(intensity(process, data, [time]))

# (R) continuous.jl:16-37: the branching simulator on the device; the sample comes back in the reference's format
function rand(process::ContinuousHawkesProcess, duration::Float64)
    push_params!(process)
    K = ndims(process)
    Weff = process isa ContinuousNetworkHawkesProcess ? process.adjacency_matrix .* process.weights.W : process.weights.W
    expected = sum(process.baseline.λ) * duration / max(0.05, 1 - min(0.95, maximum(sum(Weff, dims=2))))
    h = Ref{Ptr{Cvoid}}(C_NULL)
    check(ccall((:nhp_cont_rand, LIB[]), Cint, (Ptr{Cvoid}, Float64, UInt64, Int64, Ref{Ptr{Cvoid}}),
        CTX[], duration, Base.rand(UInt64), ceil(Int64, 2expected + 10sqrt(expected) + 1000), h))
    n = ccall((:nhp_events_count, LIB[]), Int64, (Ptr{Cvoid},), h[])
    events = Vector{Float64}(undef, n); nodes = Vector{Int64}(undef, n)
    check(ccall((:nhp_events_download, LIB[]), Cint, (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Float64}, Ptr{Int64}, Ptr{Float64}), CTX[], h[], events, nodes, C_NULL))
    ccall((:nhp_events_free, LIB[]), Cint, (Ptr{Cvoid}, Ptr{Cvoid}), CTX[], h[])
    return events, nodes, duration
end

# ---- parents.jl:1: the sweep and what it leaves behind ---------------------------------------------------------------------------
"""Result of `resample_parents(::ContinuousHawkesProcess, data)`: the assignment stays on the device together with the fused
statistics (counts, baseline attributions, impulse statistics; all-reduced over the ranks).  Destructuring it
(`parents, parentnodes = ...`) exports the two `Vector{Int64}` of the reference on demand."""
mutable struct FusedParents
    ev::DeviceEvents
    K::Int
    stats::Union{Nothing,NamedTuple}
    vectors::Union{Nothing,Tuple{Vector{Int64},Vector{Int64}}}
end

# (R) parents.jl:1
function resample_parents(process::ContinuousHawkesProcess, data)
    ev = device_events(process, data)
    push_params!(process)
    SWEEP[] += 1
    check(ccall((:nhp_cont_resample_parents, LIB[]), Cint,
        (Ptr{Cvoid}, Ptr{Cvoid}, UInt64, UInt64, Ptr{Float64}, Ptr{Int64}, Ptr{Int64}),
        CTX[], ev.h, Base.rand(UInt64), SWEEP[], C_NULL, C_NULL, C_NULL))
    check(ccall((:nhp_comm_allreduce_stats, LIB[]), Cint, (Ptr{Cvoid}, Cint), CTX[], 0))
    check(ccall((:nhp_cont_suffstats_second_pass, LIB[]), Cint, (Ptr{Cvoid}, Ptr{Cvoid}), CTX[], ev.h))
    check(ccall((:nhp_comm_allreduce_stats, LIB[]), Cint, (Ptr{Cvoid}, Cint), CTX[], 1))
    return FusedParents(ev, ndims(process), nothing, nothing)
end

function statistics(p::FusedParents)
    if p.stats === nothing
        K = p.K
        M0 = zeros(K); Mn = zeros(K); Mnm = zeros(K, K); S1 = zeros(K, K); S2 = zeros(K, K)
        check(ccall((:nhp_cont_suffstats_read, LIB[]), Cint,
            (Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}), CTX[], M0, Mn, Mnm, S1, S2))
        p.stats = (M0=M0, Mn=Mn, Mnm=Mnm, S1=S1, S2=S2)
    end
    return p.stats
end
function vectors(p::FusedParents)            # single GPU: the reference's (parents, parentnodes)
    if p.vectors === nothing
        parents = Vector{Int64}(undef, p.ev.n); parentnodes = Vector{Int64}(undef, p.ev.n)
        check(ccall((:nhp_cont_parents_get, LIB[]), Cint, (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Int64}, Ptr{Int64}), CTX[], p.ev.h, parents, parentnodes))
        p.vectors = (parents, parentnodes)
    end
    return p.vectors
end
Base.iterate(p::FusedParents, state=1) = state > 2 ? nothing : (vectors(p)[state], state + 1)
Base.getindex(p::FusedParents, i::Int) = vectors(p)[i]
Base.length(::FusedParents) = 2

# (E) weights.jl:29-43, impulses.jl:75-82 / 216-226, baselines.jl:79-85: the statistics the unchanged resample! bodies ask for
sufficient_statistics(model::Weights, data::Tuple, parents::FusedParents) = (s = statistics(parents); (s.Mn, s.Mnm))
function sufficient_statistics(impulse::ExponentialImpulseResponse, data, parents::FusedParents)
    s = statistics(parents)
    return s.Mnm, fillna!(s.S1 ./ s.Mnm, 0)                               # duration_mean (impulses.jl:84-96)
end
function sufficient_statistics(impulse::LogitNormalImpulseResponse, data, parents::FusedParents)
    s = statistics(parents)
    return s.Mnm, s.S1 ./ s.Mnm, s.S2                                     # log_duration_sum ./ Mnm (NaN kept), log_duration_variation
end
sufficient_statistics(process::HomogeneousProcess, data, parents::FusedParents) = (statistics(parents).M0, data[3])

# (R) continuous.jl:444.  Columns c % nranks == rank are resampled on this GPU, the columns are all-gathered.
function resample_adjacency_matrix!(process::ContinuousNetworkHawkesProcess, data)
    ev = device_events(process, data)
    push_params!(process)
    K = ndims(process)
    rank, nranks = comm_rank()
    SWEEP[] += 1
    seed = Base.rand(UInt64)
    if process.network isa BernoulliNetworkModel
        check(ccall((:nhp_cont_resample_adjacency_dev, LIB[]), Cint, (Ptr{Cvoid}, Ptr{Cvoid}, Float64, UInt64, UInt64, Int64, Int64, Cint),
            CTX[], ev.full, Float64(process.network.ρ), seed, SWEEP[], rank, nranks, 0))
        check(ccall((:nhp_comm_allgather_adjacency, LIB[]), Cint, (Ptr{Cvoid},), CTX[]))
        A = Matrix{Float64}(undef, K, K)
        check(ccall((:nhp_cont_params_get, LIB[]), Cint, (Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}),
            CTX[], C_NULL, C_NULL, A, C_NULL, C_NULL))
    else                                                                   # any other network model: per-link probabilities from the host
        A = Matrix{Float64}(process.adjacency_matrix)
        rho = Matrix{Float64}(link_probability(process.network))
        check(ccall((:nhp_cont_resample_adjacency, LIB[]), Cint,
            (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Float64}, UInt64, UInt64, Ptr{Float64}, Ptr{Float64}), CTX[], ev.full, rho, seed, SWEEP[], C_NULL, A))
    end
    process.adjacency_matrix .= A
    return nothing
end

# LogGaussianCoxProcess baselines (baselines.jl:187-336) inside the sweeps: push_params! sends the curves after the parameters, and the
# elliptical-slice likelihood of resample!(::LogGaussianCoxProcess, data, parents) (baselines.jl:247-254) is evaluated for all nodes at
# once from the device-resident parent assignment -- split_extract never materialises.
function push_baseline!(process::ContinuousHawkesProcess)
    b = process.baseline
    b isa LogGaussianCoxProcess || return nothing
    vals = reduce(hcat, b.λ)                                   # [grid, node]: values[g + n_grid*k]
    check(ccall((:nhp_cont_baseline_grid, LIB[]), Cint, (Ptr{Cvoid}, Int64, Ptr{Float64}, Ptr{Float64}), CTX[], length(b.x), b.x, vals))
end
function loglikelihood(process::LogGaussianCoxProcess, data::FusedParents, y::Matrix{Float64})  # y[grid, node]: all nodes at once
    vals = exp.(process.m .+ y)
    ll = Vector{Float64}(undef, size(y, 2))
    check(ccall((:nhp_cont_baseline_loglik, LIB[]), Cint, (Ptr{Cvoid}, Ptr{Cvoid}, Int64, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}),
        CTX[], data.ev.h, length(process.x), process.x, vals, ll))
    return ll
end

# The elliptical-slice update of the curves on the device (nhp_cont_resample_baseline): the GP prior goes up as cholesky(Σ).L and m
# (nhp_cont_baseline_prior; push_params! drops it, so it follows every push), the curves come back with nhp_cont_baseline_get.
function push_baseline_prior!(b::LogGaussianCoxProcess)
    L = Matrix{Float64}(cholesky(Symmetric(Matrix{Float64}(b.Σ))).L)   # column-major: L[g + n_grid*h]
    check(ccall((:nhp_cont_baseline_prior, LIB[]), Cint, (Ptr{Cvoid}, Int64, Ptr{Float64}, Float64), CTX[], length(b.x), L, Float64(b.m)))
end
function pull_baseline!(b::LogGaussianCoxProcess)
    vals = Matrix{Float64}(undef, length(b.x), length(b.λ))             # [grid, node]
    check(ccall((:nhp_cont_baseline_get, LIB[]), Cint, (Ptr{Cvoid}, Ptr{Float64}), CTX[], vals))
    b.λ = [vals[:, k] for k in axes(vals, 2)]
    return nothing
end
# resample!(process::LogGaussianCoxProcess, data, parents) for the parents of the last parent sweep on `data`, without a host round
# trip per attempt; Philox keyed by (seed, counter).  Returns the candidates each node evaluated.
function resample_baseline_on_device!(process::ContinuousHawkesProcess, data; seed::UInt64=Base.rand(UInt64), counter::UInt64=UInt64(0))
    b = process.baseline
    ev = device_events(process, data)
    push_baseline_prior!(b)
    attempts = Vector{Int64}(undef, length(b.λ))
    check(ccall((:nhp_cont_resample_baseline, LIB[]), Cint, (Ptr{Cvoid}, Ptr{Cvoid}, UInt64, UInt64, Ptr{Float64}, Ptr{Float64}, Ptr{Int64}),
        CTX[], ev.h, seed, counter, C_NULL, C_NULL, attempts))
    pull_baseline!(b)
    return attempts
end
gibbs_hyper(b, w, imp) = begin
    a0, b0 = b isa LogGaussianCoxProcess ? (1.0, 1.0) : (b.α0, b.β0)   # the curves replace the homogeneous draw these feed
    imp isa ExponentialImpulseResponse ? Float64[a0, b0, w.κ, w.ν, imp.α, imp.β] : Float64[a0, b0, w.κ, w.ν, imp.μμ, imp.κμ, imp.α0, imp.β0]
end

# optional: the whole `resample!(process, data)` (continuous.jl:202-208 / 350-358) in one call that never leaves the device
# A LogGaussianCoxProcess baseline needs `baseline_on_device=true`: the sweep then runs the elliptical-slice update of the curves
# on the device after the conjugate draws (nhp_cont_gibbs_sweep with the prior set).
function resample_on_device!(process::ContinuousHawkesProcess, data; baseline_on_device::Bool=false)
    lgcp = process.baseline isa LogGaussianCoxProcess
    lgcp && !baseline_on_device &&
        throw(ArgumentError("resample_on_device!: a LogGaussianCoxProcess baseline takes resample! (elliptical-slice update of the curves on the host) unless baseline_on_device=true"))
    ev = device_events(process, data)
    push_params!(process)
    lgcp && push_baseline_prior!(process.baseline)
    SWEEP[] += 1
    b, w, imp = process.baseline, process.weights, process.impulses
    hyper = gibbs_hyper(b, w, imp)
    net = process isa ContinuousNetworkHawkesProcess
    bern = net && process.network isa BernoulliNetworkModel
    bern && check(ccall((:nhp_cont_network_set, LIB[]), Cint, (Ptr{Cvoid}, Float64), CTX[], Float64(process.network.ρ)))
    check(ccall((:nhp_cont_gibbs_sweep, LIB[]), Cint,
        (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Cvoid}, UInt64, UInt64, Float64, Ptr{Float64}, Cint, Float64, Float64),
        CTX[], ev.h, ev.full, Base.rand(UInt64), SWEEP[], Float64(data[3]), hyper, length(hyper),
        bern ? Float64(process.network.α) : 0.0, bern ? Float64(process.network.β) : 0.0))
    K = ndims(process)
    λ = Vector{Float64}(undef, K); W = Matrix{Float64}(undef, K, K); A = Matrix{Float64}(undef, K, K)
    q1 = Matrix{Float64}(undef, K, K); q2 = Matrix{Float64}(undef, K, K)
    check(ccall((:nhp_cont_params_get, LIB[]), Cint, (Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}),
        CTX[], λ, W, net ? A : C_NULL, q1, imp isa ExponentialImpulseResponse ? C_NULL : q2))
    lgcp ? pull_baseline!(b) : (b.λ = λ); w.W = W
    if imp isa ExponentialImpulseResponse; imp.θ = q1 else imp.μ = q1; imp.τ = q2 end
    net && (process.adjacency_matrix .= A)
    if bern
        ρ = Ref{Float64}(0.0)
        ccall((:nhp_cont_network_get, LIB[]), Cint, (Ptr{Cvoid}, Ref{Float64}), CTX[], ρ)
        process.network.ρ = ρ[]
    end
    return NetworkHawkesProcesses.params(process)
end

# `mcmc!` (inference.jl:49-70) with the chain and its sample trace on the device: the parameters go up once, every sweep is one
# nhp_cont_gibbs_sweep (which appends its sample to the device-side trace, adjacency bit-packed), one read at the end.  A
# LogGaussianCoxProcess baseline needs `baseline_on_device=true`: the trace then also keeps the curves of every sample.
function mcmc_on_device!(process::ContinuousHawkesProcess, data; nsteps=1000, baseline_on_device::Bool=false)
    lgcp = process.baseline isa LogGaussianCoxProcess
    lgcp && !baseline_on_device &&
        throw(ArgumentError("mcmc_on_device!: a LogGaussianCoxProcess baseline takes mcmc! (elliptical-slice update of the curves on the host) unless baseline_on_device=true"))
    ev = device_events(process, data)
    push_params!(process)
    lgcp && push_baseline_prior!(process.baseline)
    b, w, imp = process.baseline, process.weights, process.impulses
    hyper = gibbs_hyper(b, w, imp)
    net = process isa ContinuousNetworkHawkesProcess
    bern = net && process.network isa BernoulliNetworkModel
    bern && check(ccall((:nhp_cont_network_set, LIB[]), Cint, (Ptr{Cvoid}, Float64), CTX[], Float64(process.network.ρ)))
    check(ccall((:nhp_cont_trace_begin, LIB[]), Cint, (Ptr{Cvoid}, Int64), CTX[], nsteps))
    seed = Base.rand(UInt64)
    start = time()
    for step in 1:nsteps
        check(ccall((:nhp_cont_gibbs_sweep, LIB[]), Cint,
            (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Cvoid}, UInt64, UInt64, Float64, Ptr{Float64}, Cint, Float64, Float64),
            CTX[], ev.h, ev.full, seed, UInt64(step), Float64(data[3]), hyper, length(hyper),
            bern ? Float64(process.network.α) : 0.0, bern ? Float64(process.network.β) : 0.0))
    end
    K = ndims(process); ln = !(imp isa ExponentialImpulseResponse)
    ρ = Vector{Float64}(undef, nsteps); λ = Matrix{Float64}(undef, K, nsteps); W = Array{Float64}(undef, K, K, nsteps)
    q1 = Array{Float64}(undef, K, K, nsteps); q2 = Array{Float64}(undef, K, K, nsteps); A = Array{Float64}(undef, K, K, nsteps)
    check(ccall((:nhp_cont_trace_read, LIB[]), Cint,
        (Ptr{Cvoid}, Int64, Int64, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}),
        CTX[], 0, nsteps, ρ, λ, W, net ? A : C_NULL, q1, ln ? q2 : C_NULL))
    if lgcp   # curves[g, k, sample]: they take the baseline's place in the samples
        G = length(b.x)
        C = Array{Float64}(undef, G, K, nsteps)
        check(ccall((:nhp_cont_trace_read_curves, LIB[]), Cint, (Ptr{Cvoid}, Int64, Int64, Ptr{Float64}), CTX[], 0, nsteps, C))
    end
    check(ccall((:nhp_cont_trace_free, LIB[]), Cint, (Ptr{Cvoid},), CTX[]))
    samples = Vector{Vector{Float64}}(undef, nsteps)
    for k in 1:nsteps   # the order of params(process): continuous.jl:116-119 / 325-333
        impv = ln ? [vec(q1[:, :, k]); vec(q2[:, :, k])] : vec(q1[:, :, k])
        base = lgcp ? vec(C[:, :, k]) : λ[:, k]
        samples[k] = net ? [bern ? [ρ[k]] : Float64[]; base; vec(W[:, :, k]); impv; vec(A[:, :, k])] : [base; impv; vec(W[:, :, k])]
    end
    lgcp ? (b.λ = [C[:, j, end] for j in 1:K]) : (b.λ = λ[:, end]); w.W = W[:, :, end]
    if ln; imp.μ = q1[:, :, end]; imp.τ = q2[:, :, end] else imp.θ = q1[:, :, end] end
    net && (process.adjacency_matrix .= A[:, :, end])
    bern && (process.network.ρ = ρ[end])
    return NetworkHawkesProcesses.MarkovChainMonteCarlo(samples, time() - start)
end

# ================================================== discrete path ===============================================================
function device_counts(data::AbstractMatrix)
    cached(COUNT_CACHE, data) do
        d64 = convert(Matrix{Int64}, data)                  # a no-op for the Matrix{Int64} the reference produces
        h = Ref{Ptr{Cvoid}}(C_NULL)
        N, T = size(d64)
        check(ccall((:nhp_disc_upload, LIB[]), Cint, (Ptr{Cvoid}, Ptr{Int64}, Int64, Int64, Int64, Ref{Ptr{Cvoid}}), CTX[], d64, N, T, 0, h))
        d = DeviceCounts(h[], N, T, false)
        finalizer(x -> ccall((:nhp_disc_free, LIB[]), Cint, (Ptr{Cvoid}, Ptr{Cvoid}), CTX[], x.h), d)
        d
    end
end

"""`convolve(process, data)`: the T x N x B array stays on the device inside the count handle; it behaves as the reference's
`Array{Float64,3}` (exported on first indexing) and is what the methods below dispatch on."""
mutable struct DeviceConvolved <: AbstractArray{Float64,3}
    d::DeviceCounts
    B::Int
    host::Union{Nothing,Array{Float64,3}}
end
Base.size(c::DeviceConvolved) = (c.d.T, c.d.N, c.B)
function host(c::DeviceConvolved)
    if c.host === nothing
        out = Array{Float64,3}(undef, c.d.T, c.d.N, c.B)     # conv[t + T*(n + N*b)]
        check(ccall((:nhp_disc_conv_export, LIB[]), Cint, (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Float64}), CTX[], c.d.h, out))
        c.host = out
    end
    return c.host
end
Base.getindex(c::DeviceConvolved, i::Int...) = host(c)[i...]

function ensure_convolved!(process::DiscreteHawkesProcess, d::DeviceCounts)
    d.convolved && return
    ϕ = hcat(basis(process.impulses)...)                     # L x B, column-major phi[l + L*b]
    L, B = size(ϕ)
    check(ccall((:nhp_disc_convolve, LIB[]), Cint, (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Float64}, Int64, Int64, Ptr{Float64}), CTX[], d.h, ϕ, L, B, C_NULL))
    d.convolved = true
end

# (R) discrete.jl:146
function convolve(process::DiscreteHawkesProcess, data)
    d = device_counts(data)
    ensure_convolved!(process, d)
    return DeviceConvolved(d, size(process.impulses.θ, 3), nothing)
end

adjacency(p::DiscreteStandardHawkesProcess) = C_NULL
adjacency(p::DiscreteNetworkHawkesProcess) = Matrix{Float64}(p.adjacency_matrix)
function push_params!(process::DiscreteHawkesProcess)
    N = ndims(process); B = size(process.impulses.θ, 3)
    check(ccall((:nhp_disc_params_set, LIB[]), Cint,
        (Ptr{Cvoid}, Int64, Int64, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Float64),
        CTX[], N, B, convert(Vector{Float64}, process.baseline.λ), convert(Matrix{Float64}, process.weights.W), adjacency(process),
        convert(Array{Float64,3}, process.impulses.θ), process.dt))
end

# (R) discrete.jl:20-38: the cluster simulator on the device (nhp_disc_rand).  The sample comes back as the reference's
# Matrix{Int64}, and its live device handle is registered in COUNT_CACHE under that matrix, so a following mcmc!, mcmc_on_device! or
# vb_on_device! on it uploads nothing.
function rand(process::DiscreteHawkesProcess, T::Integer)
    push_params!(process)
    N = ndims(process); B = size(process.impulses.θ, 3)
    ϕ = hcat(basis(process.impulses)...)                     # L x B
    Weff = process isa DiscreteNetworkHawkesProcess ? process.adjacency_matrix .* process.weights.W : process.weights.W
    e = Weff .* dropdims(sum(process.impulses.θ .* reshape(vec(sum(ϕ, dims=1)) .* process.dt, 1, 1, B), dims=3), dims=3)
    expected = sum(process.baseline.λ) * process.dt * T / max(0.05, 1 - min(0.95, maximum(sum(e, dims=2))))
    h = Ref{Ptr{Cvoid}}(C_NULL)
    check(ccall((:nhp_disc_rand, LIB[]), Cint, (Ptr{Cvoid}, Int64, Int64, UInt64, Int64, Ref{Ptr{Cvoid}}),
        CTX[], T, size(ϕ, 1), Base.rand(UInt64), ceil(Int64, min(2.1e9, 2expected + 10sqrt(expected) + 1000)), h))
    d = DeviceCounts(h[], N, Int(T), false)
    finalizer(x -> ccall((:nhp_disc_free, LIB[]), Cint, (Ptr{Cvoid}, Ptr{Cvoid}), CTX[], x.h), d)
    data = Matrix{Int64}(undef, N, T)                        # data[n + N*t]
    check(ccall((:nhp_disc_download, LIB[]), Cint, (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Int64}), CTX[], d.h, data))
    COUNT_CACHE[objectid(data)] = CacheEntry{DeviceCounts}(WeakRef(data), fingerprint(data), d)
    return data
end

# (E) discrete.jl:115
function intensity(process::DiscreteHawkesProcess, convolved::DeviceConvolved)
    push_params!(process)
    lam = Matrix{Float64}(undef, convolved.d.T, convolved.d.N)            # lam[t + T*c]
    check(ccall((:nhp_disc_intensity, LIB[]), Cint, (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Float64}), CTX[], convolved.d.h, lam))
    return lam
end

# (E) discrete.jl:91 and (R) :86
function loglikelihood(process::DiscreteHawkesProcess, data, convolved::DeviceConvolved)
    push_params!(process)
    ll = Ref{Float64}(0.0)
    check(ccall((:nhp_disc_loglik, LIB[]), Cint, (Ptr{Cvoid}, Ptr{Cvoid}, Ref{Float64}), CTX[], convolved.d.h, ll))
    return ll[]
end
loglikelihood(process::DiscreteHawkesProcess, data) = loglikelihood(process, data, convolve(process, data))

"""Result of `resample_parents(::DiscreteHawkesProcess, data, convolved)`: `counts[c, k] = sum_t parents[t, c, k]`, the only form
the reference consumes (impulses.jl:341, parents.jl:130, baselines.jl:414); the dense T x N x (1 + N B) array is never built."""
struct FusedCounts
    counts::Matrix{Float64}     # N x (1 + N B)
    T::Int
    rowsum::Vector{Float64}     # sum_t data[n, t]
end
Base.size(p::FusedCounts) = (p.T, size(p.counts, 1), size(p.counts, 2))
Base.sum(p::FusedCounts; dims=1) = (dims == 1 || error("FusedCounts only holds the sum over time"); reshape(p.counts, 1, size(p.counts)...))

# (E) parents.jl:82
function resample_parents(process::DiscreteHawkesProcess, data, convolved::DeviceConvolved)
    push_params!(process)
    N = ndims(process); B = convolved.B
    counts = zeros(N, 1 + N * B)
    SWEEP[] += 1
    check(ccall((:nhp_disc_gibbs_counts, LIB[]), Cint, (Ptr{Cvoid}, Ptr{Cvoid}, UInt64, UInt64, Ptr{Float64}, Int64, Ptr{Float64}),
        CTX[], convolved.d.h, Base.rand(UInt64), SWEEP[], C_NULL, 0, counts))
    return FusedCounts(counts, convolved.d.T, vec(sum(data, dims=2)))
end
# (E) parents.jl:124-134, weights.jl:29-43
function parent_counts(parents::FusedCounts, ndims, nbasis)
    M = zeros(ndims, ndims)
    for p = 1:ndims, c = 1:ndims
        M[p, c] = sum(@view parents.counts[c, (2+(p-1)*nbasis):(1+p*nbasis)])
    end
    return M
end
function sufficient_statistics(model::Weights, data::Matrix, parents::FusedCounts)
    N = size(data, 1)
    return parents.rowsum, parent_counts(parents, N, div(size(parents.counts, 2) - 1, N))
end
# (E) baselines.jl:413-419 in its intended form (quirk Q2: the reference passes a T x N slice to a function that wants N x T)
function resample!(p::DiscreteHomogeneousProcess, parents::FusedCounts)
    α = p.α0 .+ parents.counts[:, 1]
    β = p.β0 + parents.T * p.dt
    p.λ = vec(Base.rand.(Gamma.(α, 1 ./ β)))
    return copy(p.λ)
end
# resample!(::DenseWeightModel, data, parents) (weights.jl:59-64) and resample!(::DiscreteGaussianImpulseResponse, parents)
# (impulses.jl:337-353) run UNCHANGED: the first through the sufficient_statistics method above, the second through
# `sum(parents, dims=1)` and `size(parents)`.

"""Result of `update_parents(::DiscreteHawkesProcess, convolved)`: the three reductions `update!` needs (baselines.jl:444-452,
weights.jl:70-91, impulses.jl:355-371) instead of the dense T x N x (1 + N B) responsibilities."""
struct FusedVB
    alpha_sum::Vector{Float64}
    kappa_sum::Matrix{Float64}
    nu_sum::Matrix{Float64}
    gamma_sum::Array{Float64,3}
    T::Int
end
# (E) parents.jl:136
function update_parents(process::DiscreteHawkesProcess, convolved::DeviceConvolved)
    N = ndims(process); B = convolved.B
    e0 = [exp(variational_log_expectation(process.baseline, c)) for c = 1:N]
    E = Array{Float64,3}(undef, N, N, B)
    for p = 1:N, c = 1:N
        E[p, c, :] .= exp.(variational_log_expectation(process.impulses, p, c) .+ variational_log_expectation(process.weights, p, c))
    end
    a = zeros(N); k = zeros(N, N); nu = zeros(N, N); g = zeros(N, N, B)
    check(ccall((:nhp_disc_vb_stats, LIB[]), Cint,
        (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}),
        CTX[], convolved.d.h, e0, E, a, k, nu, g))
    return FusedVB(a, k, nu, g, convolved.d.T)
end
# (E) the three VB updates on the fused reductions
function update!(process::DiscreteHomogeneousProcess, data, parents::FusedVB)
    N, T = size(data)
    process.αv = process.α0 .+ parents.alpha_sum
    process.βv = 1 ./ process.β0 .+ T .* process.dt .* ones(N)
    return vec(process.αv), copy(process.βv)
end
function update!(model::DenseWeightModel, data, parents::FusedVB)
    model.κv = model.κ .+ parents.kappa_sum
    model.νv = model.ν .+ parents.nu_sum
    return copy(model.κv), copy(model.νv)
end
function update!(impulse::DiscreteGaussianImpulseResponse, data, parents::FusedVB)
    impulse.γv = impulse.γ .+ parents.gamma_sum
    return copy(impulse.γv)
end

# (E) discrete.jl:426
# optional extension for the discrete `mle!` (discrete.jl:211-296 differentiates numerically): log-likelihood + analytic gradient
function loglikelihood_gradient(process::DiscreteHawkesProcess, data, convolved::DeviceConvolved)
    push_params!(process)
    N = ndims(process); B = size(process.impulses.θ, 3)
    ll = Ref{Float64}(0.0)
    dλ = Vector{Float64}(undef, N); dW = Matrix{Float64}(undef, N, N); dθ = Array{Float64}(undef, N, N, B)
    check(ccall((:nhp_disc_loglik_grad, LIB[]), Cint, (Ptr{Cvoid}, Ptr{Cvoid}, Ref{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}),
        CTX[], convolved.d.h, ll, dλ, dW, dθ))
    return ll[], (λ=dλ, W=dW, θ=dθ)
end

# optional: the conjugate draws of the discrete `resample!` (discrete.jl:361-367 / 416-424) on the device, from the counts the last
# resample_parents left there (baseline Gamma, weight Gamma, Dirichlet theta; Philox keyed by the sweep counter)
function resample_params_on_device!(process::DiscreteHawkesProcess, data::Matrix{Int64}, convolved::DeviceConvolved)
    N = ndims(process); B = size(process.impulses.θ, 3)
    b, w, imp = process.baseline, process.weights, process.impulses
    Mn = Float64.(vec(sum(data, dims=2)))
    hyper = Float64[b.α0, b.β0, w.κ, w.ν, imp.γ]
    λ = Vector{Float64}(undef, N); W = Matrix{Float64}(undef, N, N); θ = Array{Float64}(undef, N, N, B)
    SWEEP[] += 1
    check(ccall((:nhp_disc_resample_params, LIB[]), Cint,
        (Ptr{Cvoid}, Ptr{Cvoid}, UInt64, UInt64, Ptr{Float64}, Ptr{Float64}, Cint, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}),
        CTX[], convolved.d.h, Base.rand(UInt64), SWEEP[], Mn, hyper, 5, λ, W, θ))
    b.λ = λ; w.W = W; imp.θ = θ
    return nothing
end

function resample_adjacency_matrix!(process::DiscreteNetworkHawkesProcess, data, convolved::DeviceConvolved)
    push_params!(process)
    A = Matrix{Float64}(process.adjacency_matrix)
    rho = Matrix{Float64}(link_probability(process.network))
    SWEEP[] += 1
    check(ccall((:nhp_disc_resample_adjacency, LIB[]), Cint,
        (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Float64}, UInt64, UInt64, Ptr{Float64}, Ptr{Float64}), CTX[], convolved.d.h, rho, Base.rand(UInt64), SWEEP[], C_NULL, A))
    process.adjacency_matrix .= A
    return copy(process.adjacency_matrix)
end

# `mcmc!` (inference.jl:49-70) of a discrete process with the chain and its sample trace on the device: the parameters (and ρ of a
# BernoulliNetworkModel) go up once, every sweep is one nhp_disc_gibbs_sweep (which appends its sample to the discrete trace,
# adjacency bit-packed), one read at the end.  Samples in the order of params(process): discrete.jl:178-182 / 406-414.
function mcmc_on_device!(process::DiscreteHawkesProcess, data; nsteps=1000)
    d = device_counts(data)
    ensure_convolved!(process, d)
    push_params!(process)
    b, w, imp = process.baseline, process.weights, process.impulses
    hyper = Float64[b.α0, b.β0, w.κ, w.ν, imp.γ]
    net = process isa DiscreteNetworkHawkesProcess
    bern = net && process.network isa BernoulliNetworkModel
    bern && check(ccall((:nhp_disc_network_set, LIB[]), Cint, (Ptr{Cvoid}, Float64), CTX[], Float64(process.network.ρ)))
    check(ccall((:nhp_disc_trace_begin, LIB[]), Cint, (Ptr{Cvoid}, Int64), CTX[], nsteps))
    seed = Base.rand(UInt64)
    start = time()
    for step in 1:nsteps
        check(ccall((:nhp_disc_gibbs_sweep, LIB[]), Cint,
            (Ptr{Cvoid}, Ptr{Cvoid}, UInt64, UInt64, Ptr{Float64}, Cint, Float64, Float64),
            CTX[], d.h, seed, UInt64(step), hyper, length(hyper),
            bern ? Float64(process.network.α) : 0.0, bern ? Float64(process.network.β) : 0.0))
    end
    N = ndims(process); B = size(imp.θ, 3)
    ρ = Vector{Float64}(undef, nsteps); λ = Matrix{Float64}(undef, N, nsteps); W = Array{Float64}(undef, N, N, nsteps)
    θ = Array{Float64}(undef, N, N, B, nsteps); A = Array{Float64}(undef, N, N, nsteps)
    check(ccall((:nhp_disc_trace_read, LIB[]), Cint,
        (Ptr{Cvoid}, Int64, Int64, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}),
        CTX[], 0, nsteps, ρ, λ, W, net ? A : C_NULL, θ))
    check(ccall((:nhp_disc_trace_free, LIB[]), Cint, (Ptr{Cvoid},), CTX[]))
    samples = Vector{Vector{Float64}}(undef, nsteps)
    for k in 1:nsteps
        samples[k] = net ? [bern ? [ρ[k]] : Float64[]; λ[:, k]; vec(W[:, :, k]); vec(θ[:, :, :, k]); vec(A[:, :, k])] :
                           [λ[:, k]; vec(W[:, :, k] .* θ[:, :, :, k])]
    end
    b.λ = λ[:, end]; w.W = W[:, :, end]; imp.θ = θ[:, :, :, end]
    net && (process.adjacency_matrix .= A[:, :, end])
    bern && (process.network.ρ = ρ[end])
    return NetworkHawkesProcesses.MarkovChainMonteCarlo(samples, time() - start)
end

# `vb!` (inference.jl:153-181) of a discrete standard process with the loop and its trace on the device: variational_params(process)
# (discrete.jl:204-209) and the hyper-parameters go up once, every step is one nhp_disc_vb_step (`update!`, discrete.jl:369-375, with
# digamma on the device; it appends the new state to the VB trace), one read at the end.  With `rtol`, the loop stops after the first
# step whose largest relative change of a variational parameter is <= rtol (this package's criterion: the reference's test is
# commented out, inference.jl:163-176).  Returns the trace, one variational_params vector per step; the process holds the last one.
function vb_on_device!(process::DiscreteStandardHawkesProcess, data; max_steps=100, rtol=nothing)
    d = device_counts(data)
    ensure_convolved!(process, d)
    b, w, imp = process.baseline, process.weights, process.impulses
    N = ndims(process); B = size(imp.θ, 3)
    q = Vector{Float64}(NetworkHawkesProcesses.variational_params(process))
    hyper = Float64[b.α0, b.β0, w.κ, w.ν, imp.γ]
    check(ccall((:nhp_disc_vb_set, LIB[]), Cint, (Ptr{Cvoid}, Int64, Int64, Float64, Ptr{Float64}, Cint, Ptr{Float64}),
        CTX[], N, B, process.dt, hyper, length(hyper), q))
    check(ccall((:nhp_disc_vb_trace_begin, LIB[]), Cint, (Ptr{Cvoid}, Int64), CTX[], max_steps))
    change = Ref{Float64}(0.0)
    steps = 0
    for step in 1:max_steps
        check(ccall((:nhp_disc_vb_step, LIB[]), Cint, (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Float64}), CTX[], d.h,
            rtol === nothing ? C_NULL : change))
        steps = step
        rtol !== nothing && change[] <= rtol && break
    end
    Q = Matrix{Float64}(undef, length(q), steps)
    check(ccall((:nhp_disc_vb_trace_read, LIB[]), Cint, (Ptr{Cvoid}, Int64, Int64, Ptr{Float64}), CTX[], 0, steps, Q))
    check(ccall((:nhp_disc_vb_trace_free, LIB[]), Cint, (Ptr{Cvoid},), CTX[]))
    trace = [Q[:, k] for k in 1:steps]
    last = trace[end]; o = 2N + N * N * B
    b.αv = last[1:N]; b.βv = last[N+1:2N]
    imp.γv = reshape(last[2N+1:o], N, N, B); w.κv = reshape(last[o+1:o+N*N], N, N); w.νv = reshape(last[o+N*N+1:end], N, N)
    return trace
end

# Stochastic variational inference (the reference's `svi!`, inference.jl:183-190, is an empty stub) with the loop and its trace on
# the device, modelled on vb_on_device!: step s = 1 … nsteps is one nhp_disc_svi_step on the batch_bins bins (t + j) mod T from a
# t uniform on 0 … T-1 (a window may wrap around the end, which keeps the scaled statistics unbiased), with step size (s + τ0)^(-κ);
# it moves the state to (1 - step) q + step q*, q* being the VB update from the window's statistics scaled by T / batch_bins.  The
# windows come from Julia's own RNG, so a run does not reproduce the Python svi_device_ bit for bit.  Returns the trace, one
# variational_params vector per step; the process holds the last one.
function svi_on_device!(process::DiscreteStandardHawkesProcess, data; nsteps, batch_bins, τ0=1.0, κ=0.75)
    T = size(data, 2)
    1 <= batch_bins <= T || throw(ArgumentError("batch_bins = $batch_bins outside 1 … T = $T"))
    0.5 < κ <= 1 || throw(ArgumentError("κ = $κ outside (0.5, 1]"))
    (τ0 >= 0 && isfinite(τ0)) || throw(ArgumentError("τ0 = $τ0 must be finite and >= 0"))
    nsteps >= 0 || throw(ArgumentError("nsteps = $nsteps is negative"))
    nsteps == 0 && return Vector{Vector{Float64}}()
    d = device_counts(data)
    ensure_convolved!(process, d)
    b, w, imp = process.baseline, process.weights, process.impulses
    N = ndims(process); B = size(imp.θ, 3)
    q = Vector{Float64}(NetworkHawkesProcesses.variational_params(process))
    hyper = Float64[b.α0, b.β0, w.κ, w.ν, imp.γ]
    check(ccall((:nhp_disc_vb_set, LIB[]), Cint, (Ptr{Cvoid}, Int64, Int64, Float64, Ptr{Float64}, Cint, Ptr{Float64}),
        CTX[], N, B, process.dt, hyper, length(hyper), q))
    check(ccall((:nhp_disc_vb_trace_begin, LIB[]), Cint, (Ptr{Cvoid}, Int64), CTX[], nsteps))
    for s in 1:nsteps
        check(ccall((:nhp_disc_svi_step, LIB[]), Cint, (Ptr{Cvoid}, Ptr{Cvoid}, Int64, Int64, Float64, Ptr{Float64}), CTX[], d.h,
            rand(0:T-1), batch_bins, (s + τ0)^(-κ), C_NULL))
    end
    Q = Matrix{Float64}(undef, length(q), nsteps)
    check(ccall((:nhp_disc_vb_trace_read, LIB[]), Cint, (Ptr{Cvoid}, Int64, Int64, Ptr{Float64}), CTX[], 0, nsteps, Q))
    check(ccall((:nhp_disc_vb_trace_free, LIB[]), Cint, (Ptr{Cvoid},), CTX[]))
    trace = [Q[:, k] for k in 1:nsteps]
    last = trace[end]; o = 2N + N * N * B
    b.αv = last[1:N]; b.βv = last[N+1:2N]
    imp.γv = reshape(last[2N+1:o], N, N, B); w.κv = reshape(last[o+1:o+N*N], N, N); w.νv = reshape(last[o+N*N+1:end], N, N)
    return trace
end

end # module
