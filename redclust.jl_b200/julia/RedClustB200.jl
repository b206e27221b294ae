# RedClustB200.jl -- `ccall` host layer over librcb200.so (include/rcb200.h).
#
# This is the Julia twin of redclust.jl_b200/host.py: it keeps RedClust.jl's API surface
# (MCMCData / MCMCOptionsList / PriorHyperparamsList / runsampler / MCMCResult / getpointestimate,
# /root/reference/src/RedClust.jl:32-66) and replaces the bodies of the hot-path functions by calls into the
# sm_100a library.
#
# STATUS: EXPERIMENTAL, NEVER EXECUTED.  Julia is not installed in the build image or on the GPU boxes, so this file
# has been read against the reference and against include/rcb200.h but not run; the same ABI is exercised by the Python
# mirror in the test-suite.  Use it with RedClust.jl installed: `include("RedClustB200.jl"); using .RedClustB200`
# (it reuses RedClust's own MCMCOptionsList / PriorHyperparamsList / MCMCResult types).
module RedClustB200

import RedClust
import Clustering
using RedClust: MCMCOptionsList, PriorHyperparamsList, MCMCResult, MCMCState, ClustLabelVector, fitprior
using RedClust: iac_ess_acf, sortlabels
using StatsBase: mean_and_var, mean
import Libdl

const LIB = Ref{String}(get(ENV, "RCB200_LIB", joinpath(@__DIR__, "..", "librcb200.so")))

struct rc_options
    numiters::Int64; burnin::Int64; thin::Int64; numGibbs::Int64; numMH::Int64
end
struct rc_params
    delta1::Float64; delta2::Float64; alpha::Float64; beta::Float64; zeta::Float64; gamma::Float64
    eta::Float64; sigma::Float64; proposalsd_r::Float64; u::Float64; v::Float64
    K_initial::Int64; maxK::Int64; repulsion::Int32; _pad::Int32
end
rc_options(o::MCMCOptionsList) = rc_options(o.numiters, o.burnin, o.thin, o.numGibbs, o.numMH)
rc_params(p::PriorHyperparamsList) = rc_params(p.δ1, p.δ2, p.α, p.β, p.ζ, p.γ, p.η, p.σ, p.proposalsd_r, p.u, p.v,
                                               p.K_initial, p.maxK, Int32(p.repulsion), Int32(0))

lasterror() = unsafe_string(ccall((:rc_last_error, LIB[]), Cstring, ()))
check(st::Integer) = st == 0 ? nothing : error(lasterror())      # ErrorException, as error(...) in src/types.jl

"""
NCCL communicator of the exchange steps (rc_comm_* of include/rcb200.h), one per process / GPU.  Rank 0 calls
`comm_unique_id()`, the launcher (Distributed, MPI.jl, ...) hands the 128 bytes to every rank, every rank builds `Comm`.
"""
mutable struct Comm
    handle::Ptr{Cvoid}
    rank::Int; world::Int; device::Int
    function Comm(id::Vector{UInt8}, rank::Integer, world::Integer; device::Integer = 0)
        length(id) == 128 || error("the NCCL unique id has 128 bytes")
        h = Ref{Ptr{Cvoid}}(C_NULL)
        GC.@preserve id check(ccall((:rc_comm_init, LIB[]), Int32, (Ptr{UInt8}, Int32, Int32, Int32, Ref{Ptr{Cvoid}}), id, rank, world, device, h))
        x = new(h[], rank, world, device)
        finalizer(c -> ccall((:rc_comm_destroy, LIB[]), Cvoid, (Ptr{Cvoid},), c.handle), x)
    end
end
function comm_unique_id()
    id = Vector{UInt8}(undef, 128)
    check(ccall((:rc_comm_unique_id, LIB[]), Int32, (Ptr{UInt8},), id))
    return id
end

"Device-resident MCMCData (src/types.jl:145-162)."
mutable struct MCMCData
    handle::Ptr{Cvoid}
    n::Int
    function MCMCData(D::AbstractMatrix{Float64}; device::Integer = 0)
        size(D, 1) == size(D, 2) || error("D must be a square matrix.")
        Dm = Matrix(D)
        h = Ref{Ptr{Cvoid}}(C_NULL)
        GC.@preserve Dm check(ccall((:rc_data_from_dist, LIB[]), Int32, (Ptr{Float64}, Int64, Int32, Ref{Ptr{Cvoid}}),
                                    Dm, size(Dm, 1), device, h))
        x = new(h[], size(Dm, 1))
        finalizer(d -> ccall((:rc_data_destroy, LIB[]), Cvoid, (Ptr{Cvoid},), d.handle), x)
    end
    function MCMCData(pnts::AbstractVector{<:AbstractVector{<:Float64}}; device::Integer = 0, comm::Union{Comm,Nothing} = nothing)
        X = [pnts[i][j] for j in 1:length(pnts[1]), i in 1:length(pnts)]      # dim x n, makematrix (src/utils.jl:154-156)
        h = Ref{Ptr{Cvoid}}(C_NULL)
        if isnothing(comm)
            GC.@preserve X check(ccall((:rc_data_from_points, LIB[]), Int32, (Ptr{Float64}, Int64, Int64, Int32, Ref{Ptr{Cvoid}}),
                                       X, size(X, 1), size(X, 2), device, h))
        else                                                                   # row blocks over the ranks + ncclAllGather
            GC.@preserve X check(ccall((:rc_comm_data_from_points, LIB[]), Int32, (Ptr{Cvoid}, Ptr{Float64}, Int64, Int64, Ref{Ptr{Cvoid}}),
                                       comm.handle, X, size(X, 1), size(X, 2), h))
        end
        x = new(h[], size(X, 2))
        finalizer(d -> ccall((:rc_data_destroy, LIB[]), Cvoid, (Ptr{Cvoid},), d.handle), x)
    end
end
function Base.getproperty(d::MCMCData, s::Symbol)
    if s === :D || s === :logD
        out = Matrix{Float64}(undef, d.n, d.n)
        check(s === :D ? ccall((:rc_data_copy_dist, LIB[]), Int32, (Ptr{Cvoid}, Ptr{Float64}), getfield(d, :handle), out) :
                         ccall((:rc_data_copy_logdist, LIB[]), Int32, (Ptr{Cvoid}, Ptr{Float64}), getfield(d, :handle), out))
        return out
    end
    return getfield(d, s)
end

"""
    runsampler(data, options = MCMCOptionsList(), params = nothing, init = nothing; verbose = true,
               nchains = 1, seed = rand(UInt64), slot_cap = 0) -> MCMCResult (or Vector{MCMCResult})

Same contract as RedClust.runsampler (src/mcmc.jl:501-590); the iteration loop runs in one persistent CUDA kernel.
"""
function runsampler(data::MCMCData, options::MCMCOptionsList = MCMCOptionsList(),
                    params::Union{PriorHyperparamsList,Nothing} = nothing, init::Union{MCMCState,Nothing} = nothing;
                    verbose = true, nchains::Integer = 1, seed::UInt64 = rand(UInt64), slot_cap::Integer = 0,
                    comm::Union{Comm,Nothing} = nothing, chain_offset::Integer = isnothing(comm) ? 0 : comm.rank * nchains)
    if isnothing(params)
        params = fitprior(data.D, "k-medoids", true; verbose = verbose)                      # :516-518
    end
    n = data.n
    cp = rc_params(params)
    labels = Matrix{Int64}(undef, n, nchains); r0 = Vector{Float64}(undef, nchains); p0 = similar(r0)
    if isnothing(init)                                                                       # :519-527
        k0 = params.maxK > 0 ? min(params.maxK, params.K_initial) : params.K_initial
        lab0 = Clustering.kmedoids(data.D, k0; maxiter = 1000).assignments
        for c in 1:nchains
            labels[:, c] .= lab0
            r = Ref(0.0); p = Ref(0.0)
            check(ccall((:rc_init_rp, LIB[]), Int32, (Ref{rc_params}, UInt64, Int64, Ref{Float64}, Ref{Float64}), cp, seed, chain_offset + c - 1, r, p))
            r0[c] = r[]; p0[c] = p[]
        end
    else
        for c in 1:nchains
            labels[:, c] .= sortlabels(init.clusts); r0[c] = init.r; p0[c] = init.p
        end
    end
    co = rc_options(options)
    h = Ref{Ptr{Cvoid}}(C_NULL)
    GC.@preserve labels r0 p0 check(ccall((:rc_sampler_create, LIB[]), Int32,
        (Ptr{Cvoid}, Ref{rc_options}, Ref{rc_params}, Int64, Int64, Ptr{Int64}, Ptr{Float64}, Ptr{Float64}, UInt64, Int32, Ref{Ptr{Cvoid}}),
        data.handle, co, cp, nchains, chain_offset, labels, r0, p0, seed, slot_cap, h))
    s = h[]
    try
        check(ccall((:rc_sampler_run, LIB[]), Int32, (Ptr{Cvoid}, Int64), s, -1))
        iters = Ref{Int64}(0); secs = Ref(0.0)
        check(ccall((:rc_sampler_progress, LIB[]), Int32, (Ptr{Cvoid}, Ref{Int64}, Ref{Float64}), s, iters, secs))
        S = options.numsamples
        results = MCMCResult[]
        # PSM over the chains of EVERY rank (src/mcmc.jl:560 across chain shards): int32 counts + one ncclAllReduce
        psm_all = nothing
        if !isnothing(comm)
            psm_all = Matrix{Float64}(undef, n, n)
            check(ccall((:rc_comm_sampler_psm, LIB[]), Int32, (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Float64}, Ptr{Cvoid}), comm.handle, s, psm_all, C_NULL))
        end
        for c in 0:(nchains - 1)
            if ccall((:rc_sampler_chain_status, LIB[]), Int32, (Ptr{Cvoid}, Int64), s, c) != 0
                @warn "chain $(c + 1) needed more than slot_cap simultaneously live clusters and was stopped; it is skipped"
                continue
            end
            # MCMCResult's only constructor takes a RedClust.MCMCData and reads size(data.D, 1) (src/types.jl:225-247):
            # build it on a 1 x 1 matrix and size the two point-indexed fields here
            res = MCMCResult(RedClust.MCMCData(zeros(1, 1)), options, params)
            res.clusts = [Vector{Int}(undef, n) for _ in 1:S]
            lab = Matrix{Int64}(undef, n, S)
            racc = Vector{UInt8}(undef, options.numiters); sacc = Vector{UInt8}(undef, options.numiters * options.numMH); sspl = similar(sacc)
            GC.@preserve lab check(ccall((:rc_sampler_copy_samples, LIB[]), Int32,
                (Ptr{Cvoid}, Int64, Ptr{Int64}, Ptr{Int64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}),
                s, c, lab, res.K, res.r, res.p, res.loglik, res.logposterior))
            check(ccall((:rc_sampler_copy_acceptances, LIB[]), Int32, (Ptr{Cvoid}, Int64, Ptr{UInt8}, Ptr{UInt8}, Ptr{UInt8}), s, c, racc, sacc, sspl))
            for j in 1:S
                res.clusts[j] .= @view lab[:, j]
            end
            res.r_acceptances .= racc .!= 0; res.splitmerge_acceptances .= sacc .!= 0; res.splitmerge_splits .= sspl .!= 0
            if isnothing(psm_all)
                psm = Matrix{Float64}(undef, n, n)
                check(ccall((:rc_sampler_psm, LIB[]), Int32, (Ptr{Cvoid}, Int64, Int64, Ptr{Float64}), s, c, 1, psm))   # :560
                res.posterior_coclustering = psm
            else
                res.posterior_coclustering = psm_all
            end
            res.K_iac, res.K_ess, res.K_acf = iac_ess_acf(res.K); res.K_mean, res.K_variance = mean_and_var(res.K)   # :564-573
            res.r_iac, res.r_ess, res.r_acf = iac_ess_acf(res.r); res.r_mean, res.r_variance = mean_and_var(res.r)
            res.p_iac, res.p_ess, res.p_acf = iac_ess_acf(res.p); res.p_mean, res.p_variance = mean_and_var(res.p)
            res.splitmerge_acceptance_rate = options.numMH > 0 ? mean(res.splitmerge_acceptances) : 0
            res.r_acceptance_rate = mean(res.r_acceptances)
            res.runtime = secs[]; res.mean_iter_time = secs[] / options.numiters
            push!(results, res)
        end
        return nchains == 1 ? results[1] : results
    finally
        ccall((:rc_sampler_destroy, LIB[]), Cvoid, (Ptr{Cvoid},), s)
    end
end

"MPEL search of getpointestimate (src/pointestimate.jl:34-59) on the GPU; loss in (\"binder\", \"omARI\", \"VI\", \"ID\")."
function mpel(clusts::Vector{ClustLabelVector}, loss::String; device::Integer = 0)
    code = Dict("binder" => 0, "omARI" => 1, "VI" => 2, "ID" => 3)[loss]
    S = length(clusts); n = length(clusts[1])
    L = Matrix{Int64}(undef, n, S)
    for j in 1:S; L[:, j] .= clusts[j]; end
    sums = Vector{Float64}(undef, S); best = Ref{Int64}(0)
    GC.@preserve L check(ccall((:rc_mpel, LIB[]), Int32, (Ptr{Int64}, Int64, Int64, Int32, Int32, Ptr{Float64}, Ref{Int64}), L, S, n, code, device, sums, best))
    return sums, best[] + 1
end

"Clustering.kmedoids(dissM, k) on the resident matrix (src/prior.jl:55-71, src/mcmc.jl:519-527); init: 1-based medoids."
function kmedoids_device(data::MCMCData, k::Integer, init::Vector{Int}; maxiter::Integer = 1000)
    n = getfield(data, :n)
    assign = Vector{Int64}(undef, n); med = Vector{Int64}(undef, k)
    cost = Ref{Float64}(0); conv = Ref{Int32}(0); its = Ref{Int64}(0)
    init0 = Int64.(init .- 1)
    GC.@preserve init0 check(ccall((:rc_kmedoids, LIB[]), Int32,
        (Ptr{Cvoid}, Int64, Ptr{Int64}, Int64, Ptr{Int64}, Ptr{Int64}, Ref{Float64}, Ref{Int32}, Ref{Int64}),
        getfield(data, :handle), k, init0, maxiter, assign, med, cost, conv, its))
    return (assignments = assign, medoids = med .+ 1, totalcost = cost[], converged = conv[] != 0, iterations = its[])
end

"k-medoids++ seeding on the resident matrix (Clustering.jl's default init of kmedoids): 1-based medoids for kmedoids_device."
function kmedoids_seed(data::MCMCData, k::Integer)
    u = rand(k); med = Vector{Int64}(undef, k)
    GC.@preserve u check(ccall((:rc_kmedoids_seed, LIB[]), Int32, (Ptr{Cvoid}, Int64, Ptr{Float64}, Ptr{Int64}), getfield(data, :handle), k, u, med))
    return Int.(med .+ 1)
end

"Clustering.kmeans(x, k; maxiter) on the device (src/prior.jl:63-69): x is dim x n (a point per column, the C side's n x dim row-major)."
function kmeans_device(x::Matrix{Float64}, k::Integer; maxiter::Integer = 1000, tol::Float64 = 1e-6, device::Integer = 0)
    dim, n = size(x)
    u = rand(k)
    assign = Vector{Int64}(undef, n); cent = Matrix{Float64}(undef, dim, k)
    cost = Ref{Float64}(0); conv = Ref{Int32}(0); its = Ref{Int64}(0)
    GC.@preserve x u check(ccall((:rc_kmeans, LIB[]), Int32,
        (Ptr{Float64}, Int64, Int64, Int64, Ptr{Int64}, Ptr{Float64}, Int64, Float64, Int32, Ptr{Int64}, Ptr{Float64}, Ref{Float64}, Ref{Int32}, Ref{Int64}),
        x, n, dim, k, C_NULL, u, maxiter, tol, device, assign, cent, cost, conv, its))
    return (assignments = assign, centers = cent, totalcost = cost[], converged = conv[] != 0, iterations = its[])
end

"Counts, sums and log-sums of the within / between cluster dissimilarities (A and B of src/prior.jl:73-75)."
function pairstats(data::MCMCData, labels::Vector{Int})
    n = getfield(data, :n)
    rows = Matrix{Int64}(undef, 5, n)                       # column i = row i of the C layout (n x 5 row-major)
    qD = Ref{Int32}(0); qL = Ref{Int32}(0)
    GC.@preserve labels check(ccall((:rc_pair_stats, LIB[]), Int32, (Ptr{Cvoid}, Ptr{Int64}, Ptr{Int64}), getfield(data, :handle), Int64.(labels), rows))
    check(ccall((:rc_data_scales, LIB[]), Int32, (Ptr{Cvoid}, Ref{Int32}, Ref{Int32}), getfield(data, :handle), qD, qL))
    t = [sum(big.(rows[c, :])) for c in 1:5]
    nA = Int(t[5]); nB = n * (n - 1) ÷ 2 - nA
    return (nA = nA, sA = Float64(t[1] / big(2)^qD[]), lA = Float64(t[2] / big(2)^qL[]),
            nB = nB, sB = Float64((t[3] - t[1]) / big(2)^qD[]), lB = Float64((t[4] - t[2]) / big(2)^qL[]))
end

"sample_rp(clustsizes, options, params) (src/mcmc.jl:592-636) on the device: the (r, p)-only chain of fitprior."
function sample_rp(clustsizes::Vector{Int}, options::MCMCOptionsList = MCMCOptionsList(), params::PriorHyperparamsList = PriorHyperparamsList();
                   seed::UInt64 = rand(UInt64), device::Integer = 0)
    S = options.numsamples
    r = Vector{Float64}(undef, S); p = Vector{Float64}(undef, S)
    cs = Int64.(clustsizes)
    GC.@preserve cs check(ccall((:rc_sample_rp, LIB[]), Int32,
        (Ptr{Int64}, Int64, Ref{rc_options}, Ref{rc_params}, UInt64, Int32, Ptr{Float64}, Ptr{Float64}, Ptr{UInt8}),
        cs, length(cs), rc_options(options), rc_params(params), seed, device, r, p, C_NULL))
    return (r = r, p = p)
end

# ---- posterior predictive allocation of new observations (no reference equivalent): the conditional of the full Gibbs
# scan (src/mcmc.jl:193-247) for a point that is not in the data, normalised as sample_logweights draws from it
# (src/utils.jl:2-6), averaged over the samples.  newdist is m x n (a row per new point); the C side is row-major.

"Euclidean distances (m x n) of new points to the training points, bit-equal to the stacked MCMCData(points) rows."
function crossdistances(pnts::AbstractVector{<:AbstractVector{<:Float64}}, newpnts::AbstractVector{<:AbstractVector{<:Float64}}; device::Integer = 0)
    dim = length(pnts[1])
    all(length(v) == dim for v in newpnts) || throw(ArgumentError("points and newpoints must have the same dimension."))
    X = [pnts[i][j] for j in 1:dim, i in 1:length(pnts)]          # dim x n column-major = n x dim row-major
    Y = [newpnts[i][j] for j in 1:dim, i in 1:length(newpnts)]
    out = Matrix{Float64}(undef, length(pnts), length(newpnts))   # n x m column-major = m x n row-major
    GC.@preserve X Y check(ccall((:rc_crossdist, LIB[]), Int32, (Ptr{Float64}, Int64, Ptr{Float64}, Int64, Int64, Int32, Ptr{Float64}),
                                 X, length(pnts), Y, length(newpnts), dim, device, out))
    return permutedims(out)
end

function _predict(data::MCMCData, newdist::AbstractMatrix{Float64}, clusts::Vector{<:AbstractVector{<:Integer}},
                  r::Vector{Float64}, p::Vector{Float64}, params::PriorHyperparamsList)
    n = getfield(data, :n); m = size(newdist, 1); S = length(clusts)
    size(newdist, 2) == n || throw(ArgumentError("newdist must be an m × $n matrix: one row per new point, one column per training point."))
    all(length(c) == n for c in clusts) || throw(ArgumentError("the samples must label the $n points of data."))
    Dt = Matrix{Float64}(permutedims(newdist))                     # n x m column-major = m x n row-major
    L = Matrix{Int64}(undef, n, S)
    for s in 1:S; L[:, s] .= clusts[s]; end
    cocl = Matrix{Float64}(undef, n, m); newcl = Vector{Float64}(undef, m)
    GC.@preserve Dt L r p check(ccall((:rc_predict, LIB[]), Int32,
        (Ptr{Cvoid}, Ref{rc_params}, Ptr{Float64}, Int64, Ptr{Int64}, Ptr{Float64}, Ptr{Float64}, Int64, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}),
        getfield(data, :handle), rc_params(params), Dt, m, L, r, p, S, cocl, newcl, C_NULL))
    return (coclustering = permutedims(cocl), newcluster = newcl)
end

"""
    predictivecoclustering(samples, data, newdist) -> (coclustering = m x n, newcluster = m)

coclustering[x, j]: posterior probability that new point x joins the cluster of training point j; newcluster[x]: that
it opens a cluster of its own.  `samples` is an MCMCResult or a vector of them sampled with the same hyperparameters.
"""
function predictivecoclustering(samples::Union{MCMCResult,Vector{MCMCResult}}, data::MCMCData, newdist::AbstractMatrix{Float64})
    res = samples isa MCMCResult ? [samples] : samples
    isempty(res) && throw(ArgumentError("samples must hold at least one MCMCResult."))
    all(x.params == res[1].params for x in res) || throw(ArgumentError("the results to pool were sampled with different hyperparameters."))
    return _predict(data, newdist, [c for x in res for c in x.clusts], vcat([x.r for x in res]...), vcat([x.p for x in res]...), res[1].params)
end

"Allocation probabilities (m x (K + 1)) of new points for one partition: column k for the k-th distinct label in ascending order, the last for a new cluster."
function allocationprobabilities(data::MCMCData, newdist::AbstractMatrix{Float64}, clusts::AbstractVector{<:Integer}, r::Float64, p::Float64,
                                 params::PriorHyperparamsList)
    out = _predict(data, newdist, [clusts], [r], [p], params)
    first = [findfirst(==(u), clusts) for u in sort(unique(clusts))]
    return hcat(out.coclustering[:, first], out.newcluster)
end

function getpointestimate(samples::MCMCResult; method::String = "MAP", loss::Union{String,Function} = "VI")
    if method == "MPEL" && loss isa String && loss ∉ ["binder", "omARI", "VI", "ID"]
        throw(ArgumentError("Invalid loss function specifier."))
    end
    method ∉ ["MAP", "MLE", "MPEL"] && throw(ArgumentError("Invalid method specifier."))
    if method == "MAP"
        i = argmax(samples.logposterior)
    elseif method == "MLE"
        i = argmax(samples.loglik)
    elseif loss isa String
        _, i = mpel(samples.clusts, loss)
    else
        return RedClust.getpointestimate(samples; method = method, loss = loss)   # user-supplied loss: host loop
    end
    return (samples.clusts[i], i)
end

"""
    binder_loss_sums(clusts) -> (sums, best, totals)

Expected Binder loss of every sample against all of them (src/pointestimate.jl:34-59,68-76) from their co-clustering
counts on the GPU (rc_binder_mpel): totals are the exact integer counts of disagreeing pairs summed over the samples,
sums = totals / binomial(n, 2), best the first argmin (1-based).  No S x S matrix, so it takes pooled chains.  (The
sampler-resident entry points rc_sampler_binder_mpel / rc_comm_sampler_binder_mpel need the sampler handle, which this
runsampler releases before it returns.)
"""
function binder_loss_sums(clusts::Vector{<:AbstractVector{<:Integer}}; device::Integer = 0)
    S = length(clusts); n = length(clusts[1])
    all(length(c) == n for c in clusts) || throw(ArgumentError("the samples to pool label different numbers of points."))
    L = Matrix{Int64}(undef, n, S)
    for j in 1:S; L[:, j] .= clusts[j]; end
    sums = Vector{Float64}(undef, S); totals = Vector{Int64}(undef, S); best = Ref{Int64}(0)
    GC.@preserve L check(ccall((:rc_binder_mpel, LIB[]), Int32, (Ptr{Int64}, Int64, Int64, Int32, Ptr{Float64}, Ref{Int64}, Ptr{Int64}),
                               L, S, n, device, sums, best, totals))
    return sums, best[] + 1, totals
end

"""
    getpointestimate(results::Vector{MCMCResult}; method, loss) -> (clust, i)

The samples of several chains (runsampler with nchains > 1) pooled in vector order; i indexes the concatenation.  MPEL
with loss = "binder" runs from the pooled co-clustering counts (binder_loss_sums); the other losses build the pairwise
S x S loss matrix, refused beyond 64 GiB.
"""
function getpointestimate(results::Vector{MCMCResult}; method::String = "MAP", loss::Union{String,Function} = "VI")
    if method == "MPEL" && loss isa String && loss ∉ ["binder", "omARI", "VI", "ID"]
        throw(ArgumentError("Invalid loss function specifier."))
    end
    method ∉ ["MAP", "MLE", "MPEL"] && throw(ArgumentError("Invalid method specifier."))
    isempty(results) && throw(ArgumentError("samples must hold at least one MCMCResult."))
    clusts = [c for r in results for c in r.clusts]
    all(length(c) == length(clusts[1]) for c in clusts) || throw(ArgumentError("the results to pool label different numbers of points."))
    if method == "MAP"
        i = argmax(vcat([r.logposterior for r in results]...))
    elseif method == "MLE"
        i = argmax(vcat([r.loglik for r in results]...))
    elseif loss == "binder"
        _, i, _ = binder_loss_sums(clusts)
    else
        S = length(clusts)
        8 * S^2 > 64 * 2^30 && throw(ArgumentError("$S pooled samples need a pairwise loss matrix above 64 GiB for loss = $loss; loss = \"binder\" takes pooled samples without one."))
        if loss isa String
            _, i = mpel(clusts, loss)
        else                                                # user-supplied loss: host loop, as the reference
            M = zeros(S, S)
            for a in 1:S, b in (a + 1):S
                M[a, b] = M[b, a] = loss(clusts[a], clusts[b])
            end
            i = argmin(vec(sum(M, dims = 1)))
        end
    end
    return (clusts[i], i)
end

end # module
