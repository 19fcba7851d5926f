# DPMMSubClustersB200.jl -- ccall binding of libdpmm_b200.so (include/dpmm_b200.h).
#
# UNEXERCISED IN THIS REPOSITORY'S CI: Julia is not installed in the build container or on the GPU
# box.  The identical ABI is driven from Python (dpmmsubclusters.jl_b200/sweep.py), which is what the
# parity tests run.  This file is what a maintainer of DPMMSubClusters.jl would load to redirect the
# worker side of the sampler to the GPU; INTEGRATION.md lists the call sites.
module DPMMSubClustersB200

const lib = get(ENV, "DPMM_B200_LIB", "libdpmm_b200.so")

const PRIOR_NIW = Cint(0)
const PRIOR_MULTINOMIAL = Cint(1)

mutable struct Ctx
    ptr::Ptr{Cvoid}
    n::Int
    d::Int
    prior::Cint
end

last_error(c::Ptr{Cvoid}) = unsafe_string(ccall((:dpmm_last_error, lib), Cstring, (Ptr{Cvoid},), c))
function check(rc::Cint, c::Ptr{Cvoid} = C_NULL)
    rc == 0 || error("libdpmm_b200 error $rc: $(last_error(c))")
    nothing
end

"""
    create(points::Matrix{Float32}, prior; device=0, seed=0, global_offset=0)

`points` is D x N (each column one point), exactly `local_group.points` (ds.jl:53).  Replaces
`distribute(all_data)` for one shard (dp-parallel-sampling.jl:42-44).
"""
function create(points::Matrix{Float32}, prior::Cint; device::Integer = 0, seed::Integer = 0, global_offset::Integer = 0)
    out = Ref{Ptr{Cvoid}}(C_NULL)
    d, n = size(points)
    GC.@preserve points check(ccall((:dpmm_create, lib), Cint,
        (Ref{Ptr{Cvoid}}, Ptr{Cfloat}, Int64, Int32, Int32, Int32, UInt64, Int64),
        out, points, n, d, prior, device, UInt64(seed), global_offset))
    c = Ctx(out[], n, d, prior)
    finalizer(x -> (x.ptr == C_NULL || ccall((:dpmm_destroy, lib), Cint, (Ptr{Cvoid},), x.ptr); x.ptr = C_NULL), c)
    return c
end

init_labels!(c::Ctx, init_clusters::Integer, outlier::Bool = false) =
    check(ccall((:dpmm_init_labels, lib), Cint, (Ptr{Cvoid}, Int32, Int32), c.ptr, init_clusters, outlier), c.ptr)

function randomize_sublabels!(c::Ctx, indices::Union{Nothing,Vector{Int64}} = nothing)
    if indices === nothing
        check(ccall((:dpmm_randomize_sublabels, lib), Cint, (Ptr{Cvoid}, Ptr{Int64}, Int32), c.ptr, C_NULL, 0), c.ptr)
    else
        GC.@preserve indices check(ccall((:dpmm_randomize_sublabels, lib), Cint, (Ptr{Cvoid}, Ptr{Int64}, Int32),
            c.ptr, indices, length(indices)), c.ptr)
    end
end

function labels(c::Ctx)
    out = Vector{Int64}(undef, c.n)
    check(ccall((:dpmm_get_labels, lib), Cint, (Ptr{Cvoid}, Ptr{Int64}), c.ptr, out), c.ptr)
    out
end
function sublabels(c::Ctx)
    out = Vector{Int64}(undef, c.n)
    check(ccall((:dpmm_get_sublabels, lib), Cint, (Ptr{Cvoid}, Ptr{Int64}), c.ptr, out), c.ptr)
    out
end
set_labels!(c::Ctx, l::Vector{Int64}) = check(ccall((:dpmm_set_labels, lib), Cint, (Ptr{Cvoid}, Ptr{Int64}), c.ptr, l), c.ptr)
set_sublabels!(c::Ctx, l::Vector{Int64}) = check(ccall((:dpmm_set_sublabels, lib), Cint, (Ptr{Cvoid}, Ptr{Int64}), c.ptr, l), c.ptr)

"""
    set_params!(c, clusters::Vector{<:thin_cluster_params}, weights::Vector{Float32})

Replaces `broadcast_cluster_params` (local_clusters_actions.jl:518-549).  Packs, for every cluster,
(cluster_dist, l_dist, r_dist): mv_gaussian fields mu, invSigma, logdetSigma (mv_gaussian.jl:12-18) or
multinomial_dist.alpha (multinomial_dist.jl:8-10).
"""
function set_params!(c::Ctx, clusters, weights::Vector{Float32})
    K = length(clusters)
    lr = Vector{Float32}(undef, 2K)
    for (k, cl) in enumerate(clusters)
        lr[2k-1] = cl.lr_weights[1]; lr[2k] = cl.lr_weights[2]
    end
    dists(cl) = (cl.cluster_dist, cl.l_dist, cl.r_dist)
    if c.prior == PRIOR_NIW
        D = c.d
        mu = Array{Float32}(undef, D, 3, K); inv = Array{Float32}(undef, D, D, 3, K); ld = Array{Float32}(undef, 3, K)
        for (k, cl) in enumerate(clusters), (s, dist) in enumerate(dists(cl))
            mu[:, s, k] .= dist.μ; inv[:, :, s, k] .= dist.invΣ; ld[s, k] = dist.logdetΣ
        end
        GC.@preserve mu inv ld weights lr check(ccall((:dpmm_set_params_niw, lib), Cint,
            (Ptr{Cvoid}, Int32, Ptr{Cfloat}, Ptr{Cfloat}, Ptr{Cfloat}, Ptr{Cfloat}, Ptr{Cfloat}),
            c.ptr, K, mu, inv, ld, weights, lr), c.ptr)
    else
        D = c.d
        lp = Array{Float32}(undef, D, 3, K)
        for (k, cl) in enumerate(clusters), (s, dist) in enumerate(dists(cl))
            lp[:, s, k] .= dist.α
        end
        GC.@preserve lp weights lr check(ccall((:dpmm_set_params_multinomial, lib), Cint,
            (Ptr{Cvoid}, Int32, Ptr{Cfloat}, Ptr{Cfloat}, Ptr{Cfloat}), c.ptr, K, lp, weights, lr), c.ptr)
    end
end

sample_labels!(c::Ctx, final::Bool) = check(ccall((:dpmm_sample_labels, lib), Cint, (Ptr{Cvoid}, Int32), c.ptr, final), c.ptr)
sample_sublabels!(c::Ctx) = check(ccall((:dpmm_sample_sublabels, lib), Cint, (Ptr{Cvoid},), c.ptr), c.ptr)

"""
    suff_stats(c, indices) -> (counts[3,m], sum_x[D,3,m], sum_xx[D,D,3,m])

Replaces `update_suff_stats_posterior!`'s remote part (local_clusters_actions.jl:206-236): the caller
builds niw_sufficient_statistics / multinomial_sufficient_statistics from the three arrays and runs
calc_posterior unchanged (:237-251).
"""
function suff_stats(c::Ctx, indices::Vector{Int64})
    m = length(indices); D = c.d
    counts = Array{Int64}(undef, 3, m); sx = Array{Float64}(undef, D, 3, m)
    sxx = c.prior == PRIOR_NIW ? Array{Float64}(undef, D, D, 3, m) : Array{Float64}(undef, 0, 0, 0, 0)
    GC.@preserve indices counts sx sxx check(ccall((:dpmm_suff_stats, lib), Cint,
        (Ptr{Cvoid}, Ptr{Int64}, Int32, Ptr{Int64}, Ptr{Cdouble}, Ptr{Cdouble}),
        c.ptr, indices, m, counts, sx, c.prior == PRIOR_NIW ? pointer(sxx) : C_NULL), c.ptr)
    counts, sx, sxx
end

apply_split!(c::Ctx, idx::Vector{Int64}, new_idx::Vector{Int64}) = check(ccall((:dpmm_apply_split, lib), Cint,
    (Ptr{Cvoid}, Ptr{Int64}, Ptr{Int64}, Int32), c.ptr, idx, new_idx, length(idx)), c.ptr)
apply_merge!(c::Ctx, idx::Vector{Int64}, new_idx::Vector{Int64}) = check(ccall((:dpmm_apply_merge, lib), Cint,
    (Ptr{Cvoid}, Ptr{Int64}, Ptr{Int64}, Int32), c.ptr, idx, new_idx, length(idx)), c.ptr)
remove_empty!(c::Ctx, pts_count::Vector{Int64}) = check(ccall((:dpmm_remove_empty, lib), Cint,
    (Ptr{Cvoid}, Ptr{Int64}, Int32), c.ptr, pts_count, length(pts_count)), c.ptr)

# ---- device-side parameter step (NIW and multinomial; include/dpmm_b200.h "device-side parameter step") ----
# With these the master keeps only the Hastings decisions: posterior hyper-parameters, log marginal
# likelihoods, the 3K posterior draws and the Dirichlet weights are produced next to the statistics.

"""
    set_hyper!(c, h::niw_hyperparams, α)   (niw.jl:6-11, ds.jl:9)
"""
function set_hyper!(c::Ctx, κ::Real, m::Vector{Float64}, ν::Real, ψ::Matrix{Float64}, α::Real)
    GC.@preserve m ψ check(ccall((:dpmm_set_hyper_niw, lib), Cint,
        (Ptr{Cvoid}, Cdouble, Ptr{Cdouble}, Cdouble, Ptr{Cdouble}, Cdouble), c.ptr, κ, m, ν, ψ, α), c.ptr)
end

"""
    set_hyper!(c, h::multinomial_hyper, α)   (multinomial_prior.jl:6-8, ds.jl:9)
"""
set_hyper!(c::Ctx, α_prior::Vector{Float32}, α::Real) =
    GC.@preserve α_prior check(ccall((:dpmm_set_hyper_multinomial, lib), Cint,
        (Ptr{Cvoid}, Ptr{Cfloat}, Cdouble), c.ptr, α_prior, α), c.ptr)

"""
    posterior_step(c, indices; splittable=nothing, from_table=false) -> (counts[3,m], logml[3,m], merge[K,K] or nothing)

update_suff_stats_posterior! (local_clusters_actions.jl:206-254) kept on the device.  `indices === nothing`
means every cluster.  `merge[j, i]` (column-major view of the C row-major table) holds the log marginal
likelihood of clusters i < j merged (should_merge!, shared_actions.jl:21-38).
"""
function posterior_step(c::Ctx, indices::Union{Nothing,Vector{Int64}}; splittable::Union{Nothing,Vector{UInt8}} = nothing,
                        from_table::Bool = false)
    m = indices === nothing ? Int(ccall((:dpmm_num_clusters, lib), Cint, (Ptr{Cvoid},), c.ptr)) : length(indices)
    counts = Array{Int64}(undef, 3, m); logml = Array{Float64}(undef, 3, m)
    km = splittable === nothing ? 0 : length(splittable)
    merge = km > 1 ? Array{Float64}(undef, km, km) : nothing
    GC.@preserve indices splittable counts logml merge check(ccall((:dpmm_posterior_step, lib), Cint,
        (Ptr{Cvoid}, Ptr{Int64}, Int32, Int32, Ptr{UInt8}, Int32, Ptr{Int64}, Ptr{Cdouble}, Ptr{Cdouble}),
        c.ptr, indices === nothing ? C_NULL : pointer(indices), m, from_table,
        km > 1 ? pointer(splittable) : C_NULL, km > 1 ? km : 0, counts, logml,
        merge === nothing ? C_NULL : pointer(merge)), c.ptr)
    counts, logml, merge
end

"sample_clusters! + broadcast_cluster_params on the device (local_clusters_actions.jl:417-437, 518-549)."
sample_params!(c::Ctx, K::Integer; from_prior::Bool = false, unit_weights::Bool = false) =
    check(ccall((:dpmm_sample_params, lib), Cint, (Ptr{Cvoid}, Int32, Int32, Int32), c.ptr, K, from_prior, unit_weights), c.ptr)
"merge_clusters_to_splittable on the statistics table (shared_actions.jl:12-18); i, j 1-based."
params_merge!(c::Ctx, i::Integer, j::Integer) =
    check(ccall((:dpmm_params_merge, lib), Cint, (Ptr{Cvoid}, Int64, Int64), c.ptr, i, j), c.ptr)

"(mu[D,3,K], L[D,D,3,K] with invΣ = L*L' (stored row-major: read it transposed), logdetΣ[3,K], weights[K], lr[2,K])"
function get_params(c::Ctx, K::Integer)
    D = c.d
    mu = Array{Float32}(undef, D, 3, K); lf = Array{Float64}(undef, D, D, 3, K); ld = Array{Float32}(undef, 3, K)
    w = Vector{Float32}(undef, K); lr = Array{Float32}(undef, 2, K)
    GC.@preserve mu lf ld w lr check(ccall((:dpmm_get_params_niw, lib), Cint,
        (Ptr{Cvoid}, Int32, Ptr{Cfloat}, Ptr{Cdouble}, Ptr{Cfloat}, Ptr{Cfloat}, Ptr{Cfloat}), c.ptr, K, mu, lf, ld, w, lr), c.ptr)
    mu, lf, ld, w, lr
end

"(log_p[D,3,K] = multinomial_dist.α of the 3K distributions, weights[K], lr[2,K])"
function get_params_multinomial(c::Ctx, K::Integer)
    lp = Array{Float32}(undef, c.d, 3, K); w = Vector{Float32}(undef, K); lr = Array{Float32}(undef, 2, K)
    GC.@preserve lp w lr check(ccall((:dpmm_get_params_multinomial, lib), Cint,
        (Ptr{Cvoid}, Int32, Ptr{Cfloat}, Ptr{Cfloat}, Ptr{Cfloat}), c.ptr, K, lp, w, lr), c.ptr)
    lp, w, lr
end

"""
    predict_multinomial(c, logp::Matrix{Float64}, logw::Vector{Float32}) -> (labels[n], probs[K,n])

predict_points (local_clusters_actions.jl:23-40) on this context's points: `logp[:, k] = log.(α′ₖ ./ sum(α′ₖ))`
(multinomial_prior.jl:45-48), `logw = log.(weights)`.
"""
function predict_multinomial(c::Ctx, logp::Matrix{Float64}, logw::Vector{Float32})
    K = length(logw)
    labels = Vector{Int64}(undef, c.n); probs = Array{Float32}(undef, K, c.n)
    GC.@preserve logp logw labels probs check(ccall((:dpmm_predict_multinomial, lib), Cint,
        (Ptr{Cvoid}, Int32, Ptr{Cdouble}, Ptr{Cfloat}, Ptr{Int64}, Ptr{Cfloat}), c.ptr, K, logp, logw, labels, probs), c.ptr)
    labels, probs
end

# ---- host-type shim ------------------------------------------------------------------------------------
# local_group.points / labels / labels_subcluster are typed AbstractArray (ds.jl:53-55).  These wrappers over the
# context implement what fit / run_model / save_model / calculate_posterior touch -- size and Array(...) --
# so those functions run unmodified (size(points, 2) at dp-parallel-sampling.jl:459; Array(group.labels) at
# :218, :276, :371 and ds.jl:85-87).
struct DevicePoints <: AbstractArray{Float32,2}
    c::Ctx
end
Base.size(p::DevicePoints) = (p.c.d, p.c.n)
Base.getindex(::DevicePoints, ::Int...) = error("the points live on the GPU; they are not read back element-wise")

struct DeviceLabels <: AbstractArray{Int64,1}
    c::Ctx
    sub::Bool
end
Base.size(l::DeviceLabels) = (l.c.n,)
Base.Array(l::DeviceLabels) = l.sub ? sublabels(l.c) : labels(l.c)
Base.collect(l::DeviceLabels) = Array(l)
Base.getindex(l::DeviceLabels, i::Int) = Array(l)[i]   # (debugging only: one device->host copy per call)
# e.g.  local_group(model_hyperparams, DevicePoints(ctx), DeviceLabels(ctx, false), DeviceLabels(ctx, true), [], Float32[])

# smart splits: the three worker calls of smart_cluster_init! (local_clusters_actions.jl:570-624); the eigen-decomposition
# (:557-569) and the k-means bookkeeping stay in the Julia host
function smart_project(c::Ctx, cluster::Integer, v::Vector{Float64}, μ::Vector{Float64})
    lohi = Vector{Float64}(undef, 2); cnt = Ref{Int64}(0)
    GC.@preserve v μ lohi check(ccall((:dpmm_smart_project, lib), Cint,
        (Ptr{Cvoid}, Int64, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Int64}), c.ptr, cluster, v, μ, lohi, cnt), c.ptr)
    lohi[1], lohi[2], cnt[]
end
function smart_kmeans_iter(c::Ctx, min_mean::Real, max_mean::Real)
    out = Vector{Float64}(undef, 4)      # (sum_1, count_1, sum_2, count_2) over all shards
    check(ccall((:dpmm_smart_kmeans_iter, lib), Cint, (Ptr{Cvoid}, Float64, Float64, Ptr{Float64}), c.ptr, min_mean, max_mean, out), c.ptr)
    out
end
smart_set_sublabels!(c::Ctx, cluster::Integer) =
    check(ccall((:dpmm_smart_set_sublabels, lib), Cint, (Ptr{Cvoid}, Int64), c.ptr, cluster), c.ptr)

# multi-GPU: one Julia process per GPU; rank 0 creates the id and ships it (e.g. over Distributed)
function nccl_unique_id()
    id = Vector{UInt8}(undef, 128)
    check(ccall((:dpmm_nccl_unique_id, lib), Cint, (Ptr{UInt8},), id))
    id
end
comm_init!(c::Ctx, id::Vector{UInt8}, rank::Integer, world::Integer) =
    check(ccall((:dpmm_comm_init, lib), Cint, (Ptr{Cvoid}, Ptr{UInt8}, Int32, Int32), c.ptr, id, rank, world), c.ptr)

end # module
