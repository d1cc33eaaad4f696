# PGBPB200.jl -- reference-side binding of libpgbp_b200.so (include/pgbp_b200.h).
#
# This is the host code a maintainer of PhyloGaussianBeliefProp.jl adds to use the B200 library
# as a drop-in for the message-passing path: a batched belief container plus methods of the
# package's own function names (`calibrate!`, `propagate_1traversal_postorder!`,
# `propagate_belief!`, `integratebelief!`, `factored_energy`, `assignfactors!` /
# `init_factors_frommodel!`, `regularizebeliefs_*!`, `init_beliefs_reset_fromfactors!`, ...), each
# a thin `ccall`.  Everything graph-related (cluster graphs, spanning-tree schedules, models,
# optimisers) stays what the package already does.
#
# STATUS: Julia is not available in the image this repository is built and tested in, so this file
# has never been executed here.  The same boundary is exercised by the Python ctypes mirror
# (phylogaussianbeliefprop.jl_b200/api.py), which the parity tests drive; this module is a
# line-for-line counterpart of that mirror.  `PGBPB200.dumpplan(...)` writes the plan arrays as
# JSON so they can be diffed against `workloads/*.json` wherever Julia exists.
module PGBPB200

import PhyloGaussianBeliefProp as PGBP
using PhyloGaussianBeliefProp: ClusterGraphBelief, CanonicalBelief, nclusters, nsepsets, scopeindex,
    sepsetindex, clusterindex
import PhyloNetworks as PN
import Tables
import Optim
import LinearAlgebra as LA
using MetaGraphsNext: labels, edge_labels, MetaGraph

const LIB = get(ENV, "PGBP_B200_LIB", joinpath(@__DIR__, "..", "phylogaussianbeliefprop.jl_b200", "lib", "libpgbp_b200.so"))

# ---------------------------------------------------------------- error handling
struct PgbpError <: Exception
    code::Int32
    msg::String
end
function check(rc::Int32)
    rc == 0 && return nothing
    buf = Vector{UInt8}(undef, 512)
    ccall((:pgbp_last_error, LIB), Int32, (Ptr{UInt8}, Csize_t), buf, 512)
    throw(PgbpError(rc, unsafe_string(pointer(buf))))
end

# flags (mirror include/pgbp_b200.h)
const BATCH_FACTORS = UInt32(1); const BATCH_RESIDUALS = UInt32(2)
const CAL_POSTORDER = UInt32(1); const CAL_PREORDER = UInt32(2); const CAL_BOTH = UInt32(3)
const CAL_RESIDNORM = UInt32(4); const CAL_RESIDKLDIV = UInt32(8); const CAL_AUTO = UInt32(16)
const CAL_REFORDER = UInt32(32)   # validation mode: every message in the reference's LAPACK-style operation order
const PAIR_ZIP = Int32(0); const PAIR_PRODUCT = Int32(1)

# ---------------------------------------------------------------- C structs
struct FamilyTableC
    nnodes::Int32
    ntips::Int32
    node_cluster::Ptr{Int32}
    mem_off::Ptr{Int32}
    mem_pos::Ptr{Int32}
    mem_length::Ptr{Float64}
    mem_gamma::Ptr{Float64}
    mem_color::Ptr{Int32}
    node_datarow::Ptr{Int32}
    root_fixed::Int32
    mem_tpos::Ptr{Int32}     # trait-level scopes (missing data); C_NULL = full scopes
    tip_missing::Ptr{UInt8}
end
struct PlanDescC
    nclusters::Int32
    nsepsets::Int32
    ntraits::Int32
    belief_dim::Ptr{Int32}
    sepset_clusters::Ptr{Int32}
    upind_off::Ptr{Int32}
    upind::Ptr{Int32}
    ntrees::Int32
    tree_off::Ptr{Int32}
    tree_parent::Ptr{Int32}
    tree_child::Ptr{Int32}
    families::Ptr{FamilyTableC}
end

# ---------------------------------------------------------------- plan (static index work, once per graph)
"""
    PlanArrays(beliefs, nclusters, cgraph, schedule; families=nothing)

Index data of one cluster graph, exactly as the package produces it:
`beliefs` from `allocatebeliefs` (clusters then sepsets), `schedule` from
`spanningtree(s)_clusterlist`.  All indices converted to 0-based Int32.
"""
struct PlanArrays
    nclusters::Int32
    ntraits::Int32
    belief_dim::Vector{Int32}
    sepset_clusters::Vector{Int32}
    upind_off::Vector{Int32}
    upind::Vector{Int32}
    tree_off::Vector{Int32}
    tree_parent::Vector{Int32}
    tree_child::Vector{Int32}
    families::Union{Nothing,NamedTuple}
end

function PlanArrays(beliefs::AbstractVector, nclu::Integer, cgraph, schedule::AbstractVector; families=nothing)
    lab2idx = Dict(l => Int32(i - 1) for (i, l) in enumerate(labels(cgraph)))
    dims = Int32[PGBP.dimension(b) for b in beliefs]  # sum(inscope), src/beliefs.jl:291
    sc = Int32[]; off = Int32[0]; up = Int32[]
    for s in beliefs[nclu+1:end]
        (l1, l2) = s.metadata
        a, b = lab2idx[l1], lab2idx[l2]
        push!(sc, a, b)
        append!(up, Int32.(scopeindex(s, beliefs[a+1]) .- 1)); push!(off, length(up))
        append!(up, Int32.(scopeindex(s, beliefs[b+1]) .- 1)); push!(off, length(up))
    end
    toff = Int32[0]; tp = Int32[]; tc = Int32[]
    for spt in schedule            # (parent_labels, child_labels, parent_indices, child_indices)
        append!(tp, Int32.(spt[3] .- 1)); append!(tc, Int32.(spt[4] .- 1)); push!(toff, length(tp))
    end
    PlanArrays(nclu, beliefs[1].ntraits, dims, sc, off, up, toff, tp, tc, families)
end

"""
    familiestable(prenodes, node2cluster, node2family, node2fixed, beliefs, taxa; edgecolor = e -> 0, rootfixed, tbl = nothing)

Node-family table for device-side `assignfactors!` (Brownian-motion models).  With `tbl` (the column
table the beliefs were allocated from) the missingness pattern of the tips is recorded; whenever a
value is missing or a belief has a partial trait scope the table carries trait-level scope positions
and the library runs the reference's absorb / marginalise sequence per node family on the device.
"""
function familiestable(prenodes, node2cluster, node2family, node2fixed, beliefs, taxa; edgecolor = e -> 0, rootfixed::Bool, tbl = nothing)
    p = beliefs[1].ntraits
    mem_off = Int32[0]; mem_pos = Int32[]; mem_len = Float64[]; mem_gam = Float64[]; mem_col = Int32[]; row = Int32[]
    mem_tpos = Int32[]; partial = false
    for (v, node) in enumerate(prenodes)
        be = beliefs[node2cluster[v]]
        nd = vec(sum(be.inscope, dims=1)); cs = cumsum(vcat(0, nd))
        for (k, q) in enumerate(node2family[v])
            if node2fixed[q]
                push!(mem_pos, -1); append!(mem_tpos, fill(Int32(-1), p))
            else
                jj = findfirst(isequal(q), be.nodelabel)
                nd[jj] == p || (partial = true)
                push!(mem_pos, cs[jj])
                run = cs[jj]
                for t in 1:p
                    if be.inscope[t, jj]; push!(mem_tpos, run); run += 1 else push!(mem_tpos, -1) end
                end
            end
            if k == 1
                push!(mem_len, 0.0); push!(mem_gam, 1.0); push!(mem_col, 0)
            else
                e = first(e for e in node.edge if PN.getchild(e) === node && PN.getparent(e) === prenodes[q])
                push!(mem_len, e.length); push!(mem_gam, e.gamma); push!(mem_col, edgecolor(e))
            end
        end
        push!(mem_off, length(mem_pos))
        push!(row, node.leaf ? findfirst(isequal(node.name), taxa) - 1 : -1)
    end
    # tip_missing[row, trait] (row-major, like a tip-data record)
    miss = tbl === nothing ? zeros(UInt8, p * length(taxa)) :
           UInt8[ismissing(col[i]) for i in eachindex(taxa) for col in tbl]
    scoped = partial || any(!iszero, miss)
    (nnodes = Int32(length(prenodes)), ntips = Int32(length(taxa)), root_fixed = Int32(rootfixed),
     node_cluster = Int32.(node2cluster .- 1), mem_off = mem_off, mem_pos = mem_pos, mem_length = mem_len,
     mem_gamma = mem_gam, mem_color = mem_col, node_datarow = row,
     mem_tpos = scoped ? mem_tpos : Int32[], tip_missing = scoped ? miss : UInt8[])
end

mutable struct Plan
    handle::Ptr{Cvoid}
    arrays::PlanArrays
    function Plan(a::PlanArrays)
        h = Ref{Ptr{Cvoid}}(C_NULL)
        f = a.families
        GC.@preserve a begin
            famref = Ref{FamilyTableC}()
            famptr = Ptr{FamilyTableC}(C_NULL)
            if f !== nothing
                famref[] = FamilyTableC(f.nnodes, f.ntips, pointer(f.node_cluster), pointer(f.mem_off), pointer(f.mem_pos),
                                        pointer(f.mem_length), pointer(f.mem_gamma), pointer(f.mem_color),
                                        pointer(f.node_datarow), f.root_fixed,
                                        isempty(f.mem_tpos) ? Ptr{Int32}(C_NULL) : pointer(f.mem_tpos),
                                        isempty(f.tip_missing) ? Ptr{UInt8}(C_NULL) : pointer(f.tip_missing))
                famptr = Base.unsafe_convert(Ptr{FamilyTableC}, famref)
            end
            d = Ref(PlanDescC(a.nclusters, length(a.belief_dim) - a.nclusters, a.ntraits, pointer(a.belief_dim),
                              pointer(a.sepset_clusters), pointer(a.upind_off), pointer(a.upind),
                              length(a.tree_off) - 1, pointer(a.tree_off), pointer(a.tree_parent), pointer(a.tree_child), famptr))
            GC.@preserve famref d check(ccall((:pgbp_plan_create, LIB), Int32, (Ref{PlanDescC}, Ref{Ptr{Cvoid}}), d, h))
        end
        p = new(h[], a)
        finalizer(x -> ccall((:pgbp_plan_destroy, LIB), Int32, (Ptr{Cvoid},), x.handle), p)
    end
end

# ---------------------------------------------------------------- batched beliefs
"""
    BatchedClusterGraphBelief(plan, B; device=0, factors=true, residuals=true)

`B` independent replicas (trait replicates and/or parameter vectors) of a
`ClusterGraphBelief` (src/clustergraphbeliefs.jl:26-53), resident on one GPU.
"""
mutable struct BatchedClusterGraphBelief
    handle::Ptr{Cvoid}
    plan::Plan
    B::Int
    schedule::Vector            # the spanning trees the plan was built with (for tree ids)
    template::Union{Nothing,ClusterGraphBelief}   # optional: a ClusterGraphBelief of the same graph (scopes for index programs)
    # sharedgroup = g > 1: the g consecutive elements of a group are trait replicates under one parameter
    # vector; their (identical) precisions J are stored and updated once per group
    function BatchedClusterGraphBelief(plan::Plan, B::Integer, schedule; device::Integer=0, factors=true, residuals=true,
                                       sharedgroup::Integer=0)
        h = Ref{Ptr{Cvoid}}(C_NULL)
        fl = (factors ? BATCH_FACTORS : UInt32(0)) | (residuals ? BATCH_RESIDUALS : UInt32(0))
        check(ccall((:pgbp_batch_create_shared, LIB), Int32, (Ptr{Cvoid}, Int64, Int64, Int32, UInt32, Ref{Ptr{Cvoid}}),
                    plan.handle, B, sharedgroup, device, fl, h))
        b = new(h[], plan, B, collect(schedule), nothing)
        finalizer(x -> ccall((:pgbp_batch_destroy, LIB), Int32, (Ptr{Cvoid},), x.handle), b)
    end
end
PGBP.nclusters(b::BatchedClusterGraphBelief) = Int(b.plan.arrays.nclusters)
PGBP.nsepsets(b::BatchedClusterGraphBelief) = length(b.plan.arrays.belief_dim) - PGBP.nclusters(b)
dimension(b::BatchedClusterGraphBelief, j::Integer) = Int(b.plan.arrays.belief_dim[j])

treeid(b::BatchedClusterGraphBelief, spt) = Int32(findfirst(t -> t[3] == spt[3] && t[4] == spt[4], b.schedule) - 1)

# belief access: J (m,m,B), h (m,B), g (B,) -- Julia's column-major arrays map directly
function setbelief!(b::BatchedClusterGraphBelief, j::Integer, J::Array{Float64,3}, h::Matrix{Float64}, g::Vector{Float64})
    GC.@preserve J h g check(ccall((:pgbp_set_belief, LIB), Int32, (Ptr{Cvoid}, Int32, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}),
                                   b.handle, j - 1, J, h, g))
end
function getbelief(b::BatchedClusterGraphBelief, j::Integer)
    m = dimension(b, j)
    J = Array{Float64}(undef, m, m, b.B); h = Matrix{Float64}(undef, m, b.B); g = Vector{Float64}(undef, b.B)
    GC.@preserve J h g check(ccall((:pgbp_get_belief, LIB), Int32, (Ptr{Cvoid}, Int32, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}),
                                   b.handle, j - 1, J, h, g))
    return J, h, g
end
function status(b::BatchedClusterGraphBelief)
    st = Vector{Int32}(undef, b.B)
    GC.@preserve st check(ccall((:pgbp_get_status, LIB), Int32, (Ptr{Cvoid}, Ptr{Int32}), b.handle, st))
    st
end

# ---------------------------------------------------------------- the package's API, batched
"""
    assignfactors!(b, params, tipdata; ncolors=1, pairing=:zip)

Device-side `assignfactors!` (src/beliefs.jl:786-861) for Brownian-motion models.
`params`: (ncolors*p*p + p + p*p, nparamsets) -- rates `R_c`, root mean, root variance per column;
`tipdata`: (p, ntips, ndatasets).
"""
function PGBP.assignfactors!(b::BatchedClusterGraphBelief, params::Matrix{Float64}, tipdata::Array{Float64,3};
                             ncolors::Integer=1, pairing::Symbol=:zip)
    GC.@preserve params tipdata check(ccall((:pgbp_assign_factors, LIB), Int32,
        (Ptr{Cvoid}, Int32, Ptr{Float64}, Int64, Ptr{Float64}, Int64, Int32),
        b.handle, ncolors, params, size(params, 2), tipdata, size(tipdata, 3), pairing === :product ? PAIR_PRODUCT : PAIR_ZIP))
end
const init_factors_frommodel! = PGBP.assignfactors!   # spelling of the revision named in BASELINE.json

"pack one Brownian-motion parameter set (`R` per colour, root mean, root variance; 0 = fixed root)"
bmparams(rates::Vector{<:AbstractMatrix}, μ::AbstractVector, v::AbstractMatrix=zeros(length(μ), length(μ))) =
    vcat((vec(Matrix{Float64}(R)) for R in rates)..., Float64.(μ), vec(Matrix{Float64}(v)))
bmparams(m::PGBP.MvFullBrownianMotion) = bmparams([Matrix(m.R)], m.μ, Matrix(m.v))
bmparams(m::PGBP.MvDiagBrownianMotion) = bmparams([Matrix(PGBP.LA.Diagonal(m.R))], m.μ, Matrix(PGBP.LA.Diagonal(m.v)))
bmparams(m::PGBP.UnivariateBrownianMotion) = bmparams([fill(m.σ2, 1, 1)], [m.μ], fill(m.v, 1, 1))

function _flags(update_residualnorm, update_residualkldiv, auto, reference_order=false)
    (update_residualnorm ? CAL_RESIDNORM : UInt32(0)) | (update_residualkldiv ? CAL_RESIDKLDIV : UInt32(0)) |
    (auto ? CAL_AUTO : UInt32(0)) | (reference_order ? CAL_REFORDER : UInt32(0))
end

"""
    calibrate!(b::BatchedClusterGraphBelief, schedule, niter=1; auto, info, update_residualnorm, update_residualkldiv)

Same semantics as `calibrate!` (src/calibration.jl:35-60), per batch element:
returns `(succ::BitVector, iscal::BitVector)`.
"""
function PGBP.calibrate!(b::BatchedClusterGraphBelief, schedule::AbstractVector, niter::Integer=1;
                         auto::Bool=false, info::Bool=false, verbose::Bool=true,
                         update_residualnorm::Bool=true, update_residualkldiv::Bool=false, direction::UInt32=CAL_BOTH,
                         reference_order::Bool=false)
    ids = Int32[treeid(b, spt) for spt in schedule]
    succ = Vector{Int32}(undef, b.B); iscal = Vector{Int32}(undef, b.B)
    it = info ? Matrix{Int32}(undef, 2, b.B) : nothing
    GC.@preserve ids succ iscal it check(ccall((:pgbp_calibrate, LIB), Int32,
        (Ptr{Cvoid}, Ptr{Int32}, Int32, Int32, UInt32, Ptr{Int32}, Ptr{Int32}, Ptr{Int32}),
        b.handle, ids, length(ids), niter, direction | _flags(update_residualnorm, update_residualkldiv, auto, reference_order),
        succ, iscal, info ? pointer(it) : C_NULL))
    if info
        for e in 1:b.B
            it[1, e] > 0 && verbose && @info "element $e: calibration reached: iteration $(it[1,e]), schedule tree $(it[2,e])"
        end
    end
    return succ .!= 0, iscal .!= 0
end
PGBP.propagate_1traversal_postorder!(b::BatchedClusterGraphBelief, spt...; kw...) =
    PGBP.calibrate!(b, [spt]; direction=CAL_POSTORDER, kw...)[1]
PGBP.propagate_1traversal_preorder!(b::BatchedClusterGraphBelief, spt...; kw...) =
    PGBP.calibrate!(b, [spt]; direction=CAL_PREORDER, kw...)[1]

"`propagate_belief!(cluster_to, sepset, cluster_from, residual)` (src/beliefupdates.jl:634) by belief index"
PGBP.propagate_belief!(b::BatchedClusterGraphBelief, to::Integer, sepset::Integer, from::Integer) =
    check(ccall((:pgbp_propagate, LIB), Int32, (Ptr{Cvoid}, Int32, Int32, Int32, UInt32), b.handle, from - 1, sepset - 1, to - 1, 0))

"`integratebelief!(beliefs, j)` -> `(μ::Matrix (m,B), norm::Vector (B))` (src/clustergraphbeliefs.jl:194)"
function PGBP.integratebelief!(b::BatchedClusterGraphBelief, j::Integer)
    μ = Matrix{Float64}(undef, dimension(b, j), b.B); nrm = Vector{Float64}(undef, b.B)
    GC.@preserve μ nrm check(ccall((:pgbp_integrate, LIB), Int32, (Ptr{Cvoid}, Int32, Ptr{Float64}, Ptr{Float64}), b.handle, j - 1, μ, nrm))
    return μ, nrm
end

"`integratebelief!` + `inv(J)`: `(μ (m,B), cov (m,m,B), norm (B))`, the conditional moments of calibrate_exact_cliquetree!"
function integratebelief_cov!(b::BatchedClusterGraphBelief, j::Integer)
    m = dimension(b, j)
    μ = Matrix{Float64}(undef, m, b.B); cov = Array{Float64}(undef, m, m, b.B); nrm = Vector{Float64}(undef, b.B)
    GC.@preserve μ cov nrm check(ccall((:pgbp_integrate_cov, LIB), Int32, (Ptr{Cvoid}, Int32, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}),
                                       b.handle, j - 1, μ, cov, nrm))
    return μ, cov, nrm
end

# (belief j, positions) queries -> 0-based C arrays (positions are 1-based here, as Julia indices)
function _marginal_queries(queries)
    qb = Int32[j - 1 for (j, _) in queries]
    off = Int32[0]; pos = Int32[]
    for (_, p) in queries
        append!(pos, Int32.(p) .- Int32(1)); push!(off, length(pos))
    end
    return qb, off, pos
end

"""
    marginal_moments!(b, queries) -> [(μ (k,B), cov (k,k,B)) per query]

Posterior moments of position subsets: query `(j, positions)` (1-based belief index and 1-based scope positions) is
the marginal of belief j on those positions, `μ = (J \\ h)[pos]`, `cov = inv(J)[pos, pos]` (`integratebelief!` +
`inv(J)`, src/beliefupdates.jl:168-200), for every element; each belief is factorised once however many queries name
it.  Entries equal those of `integratebelief_cov!` bit for bit.
"""
function marginal_moments!(b::BatchedClusterGraphBelief, queries::AbstractVector)
    qb, off, pos = _marginal_queries(queries)
    ks = diff(off)
    μ = Matrix{Float64}(undef, sum(ks), b.B); cov = Matrix{Float64}(undef, sum(ks .^ 2), b.B)
    GC.@preserve qb off pos μ cov check(ccall((:pgbp_marginal_moments, LIB), Int32,
        (Ptr{Cvoid}, Int32, Ptr{Int32}, Ptr{Int32}, Ptr{Int32}, Ptr{Float64}, Ptr{Float64}),
        b.handle, length(qb), qb, off, pos, μ, cov))
    m0 = cumsum([0; ks]); c0 = cumsum([0; ks .^ 2])
    return [(μ[m0[q]+1:m0[q+1], :], reshape(cov[c0[q]+1:c0[q+1], :], ks[q], ks[q], b.B)) for q in eachindex(ks)]
end

"`factored_energy(beliefs)` -> (3,B) matrix: average energy, approximate entropy, factored energy (src/score.jl:151)"
function PGBP.factored_energy(b::BatchedClusterGraphBelief)
    out = Matrix{Float64}(undef, 3, b.B)
    GC.@preserve out check(ccall((:pgbp_factored_energy, LIB), Int32, (Ptr{Cvoid}, Ptr{Float64}), b.handle, out))
    out
end
function PGBP.free_energy(b::BatchedClusterGraphBelief)
    out = PGBP.factored_energy(b); out[3, :] .*= -1; out
end

PGBP.regularizebeliefs_bycluster!(b::BatchedClusterGraphBelief, cgraph=nothing) =
    check(ccall((:pgbp_regularize_bycluster, LIB), Int32, (Ptr{Cvoid},), b.handle))
PGBP.regularizebeliefs_onschedule!(b::BatchedClusterGraphBelief, cgraph=nothing) =
    check(ccall((:pgbp_regularize_onschedule, LIB), Int32, (Ptr{Cvoid},), b.handle))
PGBP.init_beliefs_reset_fromfactors!(b::BatchedClusterGraphBelief) =
    check(ccall((:pgbp_reset_from_factors, LIB), Int32, (Ptr{Cvoid},), b.handle))
PGBP.init_factors_frombeliefs!(b::BatchedClusterGraphBelief) =
    check(ccall((:pgbp_factors_from_beliefs, LIB), Int32, (Ptr{Cvoid},), b.handle))
PGBP.init_messagecalibrationflags_reset!(b::BatchedClusterGraphBelief, reset_kl::Bool=true) =
    check(ccall((:pgbp_reset_calibration_flags, LIB), Int32, (Ptr{Cvoid}, Int32), b.handle, reset_kl))

"""
    regularizebeliefs_bynodesubtree!(b, cgraph)

Index program of the loop at src/clustergraphbeliefs.jl:314-340 (which clusters define a node's ϵ,
which (cluster, sepset) pairs and diagonal positions it is added to), then one library call.
"""
function PGBP.regularizebeliefs_bynodesubtree!(b::BatchedClusterGraphBelief, beliefs::ClusterGraphBelief, cgraph)
    eo = Int32[0]; ec = Int32[]; so = Int32[0]; sc = Int32[]; ss = Int32[]; io = Int32[0]; ic = Int32[]; is = Int32[]
    for (node_ind, (nodelab, clusterlabs)) in enumerate(PGBP.get_nodesymbols2index(cgraph) |> pairs)
        # follows the reference: clusters containing the node, then its node subtree in preorder
        sch = PGBP.nodesubtree_clusterlist(PGBP.nodesubtree(cgraph, nodelab, node_ind)[1], nodelab)
        isempty(sch[3]) && (push!(eo, length(ec)); push!(so, length(sc)); continue)
        cl = unique(vcat(sch[3], sch[4]))
        append!(ec, Int32.(cl .- 1)); push!(eo, length(ec))
        for (pl, chl) in zip(sch[1], sch[2])
            ci = clusterindex(chl, beliefs); si = sepsetindex(pl, chl, beliefs)
            (s_ind, c_ind) = scopeindex(node_ind, beliefs.belief[si], beliefs.belief[ci])
            push!(sc, ci - 1); push!(ss, si - 1 - PGBP.nclusters(beliefs))
            append!(ic, Int32.(c_ind .- 1)); append!(is, Int32.(s_ind .- 1)); push!(io, length(ic))
        end
        push!(so, length(sc))
    end
    GC.@preserve eo ec so sc ss io ic is check(ccall((:pgbp_regularize_bynodesubtree, LIB), Int32,
        (Ptr{Cvoid}, Int32, Ptr{Int32}, Ptr{Int32}, Ptr{Int32}, Ptr{Int32}, Ptr{Int32}, Ptr{Int32}, Ptr{Int32}, Ptr{Int32}),
        b.handle, length(eo) - 1, eo, ec, so, sc, ss, io, ic, is))
end


# ---------------------------------------------------------------- reference-signature methods
# The methods above take pre-packed arrays; the ones below take what the package's own functions take, so that a
# call site written for `ClusterGraphBelief` works on a `BatchedClusterGraphBelief` unchanged.  A batch holds B
# elements: `model` / `tbl` may be ONE object (shared by all elements) or a vector (one per element, or per
# factor of the :product pairing).

ncolors(m::PGBP.EvolutionaryModel) = 1
ncolors(m::PGBP.HeterogeneousBrownianMotion) = PGBP.ncolors(m.variancerate)
bmparams(m::PGBP.HeterogeneousBrownianMotion) = bmparams([Matrix(R) for R in m.variancerate.parameter], m.μ, Matrix(m.v))
"colour (0-based) of an edge under a painted model; 0 for homogeneous models (families table: `edgecolor`)"
edgecolor(m::PGBP.EvolutionaryModel) = e -> Int32(0)
edgecolor(m::PGBP.HeterogeneousBrownianMotion) = e -> Int32(m.variancerate.color[e.number] - 1)

"tip data of one or several column tables as the (p, ntips, ndatasets) array of the ABI; `missing` -> NaN"
function tipdata(tbls::AbstractVector, ntips::Integer)
    p = length(first(tbls))
    out = Array{Float64}(undef, p, ntips, length(tbls))
    for (d, tbl) in enumerate(tbls), (t, col) in enumerate(tbl), i in 1:ntips
        out[t, i, d] = ismissing(col[i]) ? NaN : Float64(col[i])
    end
    out
end

"""
    assignfactors!(b::BatchedClusterGraphBelief, model, tbl, taxa, prenodes, node2cluster, node2family, node2fixed; pairing=:zip)

The reference's signature (src/beliefs.jl:786-795).  The plan of `b` was compiled from the same
`node2cluster / node2family / node2fixed` (`familiestable`), so they are only checked for length here.
Brownian-motion models (homogeneous, heterogeneous) and the univariate Ornstein-Uhlenbeck model are assigned on the
device; for any other model assign on the host with the package's method and upload with `setbelief!`.
"""
function PGBP.assignfactors!(b::BatchedClusterGraphBelief,
                             model::Union{PGBP.EvolutionaryModel,AbstractVector{<:PGBP.EvolutionaryModel}},
                             tbl::Union{Tables.ColumnTable,AbstractVector{<:Tables.ColumnTable}},
                             taxa::AbstractVector, prenodes::Vector{PN.Node}, node2cluster, node2family, node2fixed;
                             pairing::Symbol=:zip)
    f = b.plan.arrays.families
    f === nothing && error("the plan was built without a families table (PlanArrays(...; families = familiestable(...)))")
    length(node2cluster) == f.nnodes == length(prenodes) || error("node2cluster does not match the plan")
    models = model isa AbstractVector ? model : [model]
    tbls = tbl isa AbstractVector ? tbl : [tbl]
    tips = tipdata(tbls, length(taxa))
    if first(models) isa PGBP.UnivariateOrnsteinUhlenbeck
        params = Float64[getfield(m, k) for k in (:γ2, :α, :θ, :μ, :v), m in models]
        params[1, :] .*= 2 .* params[2, :]                       # σ2 = 2 α γ2
        return assignfactors_ou!(b, params, tips; pairing)
    end
    params = reduce(hcat, (bmparams(m) for m in models))
    PGBP.assignfactors!(b, params, tips; ncolors=ncolors(first(models)), pairing)
end

"`assignfactors!` for the univariate Ornstein-Uhlenbeck model: `params` (5, nparamsets) = (σ2, α, θ, μ, v) per column"
function assignfactors_ou!(b::BatchedClusterGraphBelief, params::Matrix{Float64}, tipdata::Array{Float64,3}; pairing::Symbol=:zip)
    GC.@preserve params tipdata check(ccall((:pgbp_assign_factors_ou, LIB), Int32,
        (Ptr{Cvoid}, Ptr{Float64}, Int64, Ptr{Float64}, Int64, Int32),
        b.handle, params, size(params, 2), tipdata, size(tipdata, 3), pairing === :product ? PAIR_PRODUCT : PAIR_ZIP))
end

"""
    assignfactors_device!(b, d_params::Ptr{Float64}, nparamsets, d_tipdata::Ptr{Float64}, ndatasets; ncolors, pairing)

Same records already resident in HBM (e.g. `CUDA.CuArray` pointers): enqueue only -- the optimiser inner loop that
keeps its parameter grid on the GPU.  Companions: `calibrate_async!`, `integratebelief_device!`,
`factored_energy_device!`, `setstream!`, `synchronize`.
"""
assignfactors_device!(b::BatchedClusterGraphBelief, d_params::Ptr{Float64}, nparamsets::Integer, d_tipdata::Ptr{Float64},
                      ndatasets::Integer; ncolors::Integer=1, pairing::Symbol=:zip) =
    check(ccall((:pgbp_assign_factors_device, LIB), Int32, (Ptr{Cvoid}, Int32, Ptr{Float64}, Int64, Ptr{Float64}, Int64, Int32),
                b.handle, ncolors, d_params, nparamsets, d_tipdata, ndatasets, pairing === :product ? PAIR_PRODUCT : PAIR_ZIP))
function calibrate_async!(b::BatchedClusterGraphBelief, schedule::AbstractVector, niter::Integer=1; auto::Bool=false,
                          update_residualnorm::Bool=true, direction::UInt32=CAL_BOTH)
    ids = Int32[treeid(b, spt) for spt in schedule]
    GC.@preserve ids check(ccall((:pgbp_calibrate_async, LIB), Int32, (Ptr{Cvoid}, Ptr{Int32}, Int32, Int32, UInt32),
                                 b.handle, ids, length(ids), niter, direction | _flags(update_residualnorm, false, auto)))
end
integratebelief_device!(b::BatchedClusterGraphBelief, j::Integer, d_norm::Ptr{Float64}, d_mu::Ptr{Float64}=Ptr{Float64}(C_NULL)) =
    check(ccall((:pgbp_integrate_device, LIB), Int32, (Ptr{Cvoid}, Int32, Ptr{Float64}, Ptr{Float64}), b.handle, j - 1, d_mu, d_norm))
"`marginal_moments!` into device arrays, enqueue only: μ rows [sum k][ld], cov rows [sum k(k+1)/2][ld] (packed upper per query)"
function marginal_moments_device!(b::BatchedClusterGraphBelief, queries::AbstractVector, d_mu::Ptr{Float64},
                                  d_cov::Ptr{Float64}=Ptr{Float64}(C_NULL))
    qb, off, pos = _marginal_queries(queries)
    GC.@preserve qb off pos check(ccall((:pgbp_marginal_moments_device, LIB), Int32,
        (Ptr{Cvoid}, Int32, Ptr{Int32}, Ptr{Int32}, Ptr{Int32}, Ptr{Float64}, Ptr{Float64}),
        b.handle, length(qb), qb, off, pos, d_mu, d_cov))
end
factored_energy_device!(b::BatchedClusterGraphBelief, d_out::Ptr{Float64}) =
    check(ccall((:pgbp_factored_energy_device, LIB), Int32, (Ptr{Cvoid}, Ptr{Float64}), b.handle, d_out))
"run the batch on an externally owned `cudaStream_t` (e.g. `CUDA.stream().handle`)"
setstream!(b::BatchedClusterGraphBelief, stream::Ptr{Cvoid}) =
    check(ccall((:pgbp_batch_set_stream, LIB), Int32, (Ptr{Cvoid}, Ptr{Cvoid}), b.handle, stream))
synchronize(b::BatchedClusterGraphBelief) = check(ccall((:pgbp_batch_synchronize, LIB), Int32, (Ptr{Cvoid},), b.handle))
clearstatus!(b::BatchedClusterGraphBelief) = check(ccall((:pgbp_clear_status, LIB), Int32, (Ptr{Cvoid},), b.handle))
"rows (h first row, g row; 0-based) of belief j in the device view: plan slots, or compact rows of a shared-precision batch"
function beliefrows(b::BatchedClusterGraphBelief, j::Integer)
    h = Ref{Int64}(0); g = Ref{Int64}(0)
    check(ccall((:pgbp_batch_belief_rows, LIB), Int32, (Ptr{Cvoid}, Int32, Ref{Int64}, Ref{Int64}), b.handle, j - 1, h, g))
    h[], g[]
end

"`integratebelief!(beliefs, cgraph, prenodes)` (src/clustergraphbeliefs.jl:190): at the default root cluster"
PGBP.integratebelief!(b::BatchedClusterGraphBelief, cgraph::MetaGraph, prenodes) =
    PGBP.integratebelief!(b, PGBP.default_rootcluster(cgraph, prenodes))
"`integratebelief!(beliefs)`: at the first sepset with a single node (valid after a full calibration)"
function PGBP.integratebelief!(b::BatchedClusterGraphBelief)
    a = b.plan.arrays
    j = findnext(j -> a.belief_dim[j] == a.ntraits, 1:length(a.belief_dim), PGBP.nclusters(b) + 1)
    isnothing(j) && error("no sepset with a single node")
    PGBP.integratebelief!(b, j)
end

"""
    regularizebeliefs_bynodesubtree!(b::BatchedClusterGraphBelief, cgraph)

The reference's signature (src/clustergraphbeliefs.jl:306-311).  The index program of its loop (:314-340) only needs
scopes, which the batch's plan holds as belief dimensions and `upind` maps; they are rebuilt here from a template
`ClusterGraphBelief` the caller keeps (`b.template`), set by `attach_template!`.
"""
function PGBP.regularizebeliefs_bynodesubtree!(b::BatchedClusterGraphBelief, cgraph::MetaGraph)
    b.template === nothing && error("attach_template!(b, beliefs::ClusterGraphBelief) first: the index program needs the scopes")
    PGBP.regularizebeliefs_bynodesubtree!(b, b.template, cgraph)
end
attach_template!(b::BatchedClusterGraphBelief, beliefs::ClusterGraphBelief) = (b.template = beliefs; b)

# ---------------------------------------------------------------- drivers (src/calibration.jl:163-517), batched
# The reference evaluates its objective one parameter vector at a time and lets Optim difference it.  Here every
# objective AND its central-difference gradient are ONE batched device call: the batch holds the 2n+1 parameter
# vectors of the stencil (n = number of optimised parameters).

function _stencil(θ::AbstractVector, h::Float64)
    n = length(θ)
    S = repeat(θ, 1, 2n + 1)
    for k in 1:n
        S[k, 2k] += h; S[k, 2k+1] -= h
    end
    S
end

"""
    calibrate_optimize_cliquetree!(b::BatchedClusterGraphBelief, cgraph, prenodes, tbl, taxa, evomodelfun, evomodelparams,
                                   optimoptions = Optim.Options(iterations=30); fdstep = 1e-6)

Mirror of `calibrate_optimize_cliquetree!` (src/calibration.jl:182-234): `b` must hold `2n+1` elements, n =
`length(params_optimize(model))`.  Returns `(bestmodel, loglikscore, opt)` like the reference.
"""
function PGBP.calibrate_optimize_cliquetree!(b::BatchedClusterGraphBelief, cgraph, prenodes::Vector{PN.Node},
        tbl::Tables.ColumnTable, taxa::AbstractVector, evomodelfun, evomodelparams,
        optimoptions=Optim.Options(iterations=30); fdstep::Float64=1e-6)
    spt = PGBP.spanningtree_clusterlist(cgraph, prenodes)
    rootj = spt[3][1]
    mod = evomodelfun(evomodelparams...)
    θ0 = PGBP.params_optimize(mod)
    n = length(θ0)
    b.B == 2n + 1 || error("the batch must hold 2n+1 = $(2n+1) elements (central-difference stencil)")
    tips = tipdata([tbl], length(taxa))
    function scores(S)                      # S: (n, 2n+1) unconstrained parameter vectors -> -loglik per column
        out = fill(Inf, size(S, 2))
        models = Vector{Any}(undef, size(S, 2)); ok = trues(size(S, 2))
        for c in axes(S, 2)
            try models[c] = evomodelfun(PGBP.params_original(mod, S[:, c])...)
            catch ex
                ex isa LA.PosDefException || rethrow(ex)
                ok[c] = false; models[c] = mod
            end
        end
        clearstatus!(b)
        PGBP.assignfactors!(b, reduce(hcat, (bmparams(m) for m in models)), tips; ncolors=ncolors(mod))
        PGBP.init_messagecalibrationflags_reset!(b, false)
        succ = PGBP.propagate_1traversal_postorder!(b, spt...; update_residualnorm=false)
        _, ll = PGBP.integratebelief!(b, rootj)
        st = status(b)
        for c in axes(S, 2)
            ok[c] && succ[c] && st[c] == 0 && isfinite(ll[c]) && (out[c] = -ll[c])
        end
        out
    end
    fg!(F, G, θ) = begin
        f = scores(_stencil(θ, fdstep))
        G === nothing || (G .= (f[2:2:end] .- f[3:2:end]) ./ (2fdstep))
        F === nothing ? nothing : f[1]
    end
    opt = Optim.optimize(Optim.only_fg!(fg!), θ0, Optim.LBFGS(), optimoptions)
    bestmodel = evomodelfun(PGBP.params_original(mod, Optim.minimizer(opt))...)
    return bestmodel, -Optim.minimum(opt), opt
end

"""
    calibrate_optimize_clustergraph!(b::BatchedClusterGraphBelief, cgraph, prenodes, tbl, taxa, evomodelfun, evomodelparams,
                                     maxiter = 100, regfun = regularizebeliefs_bycluster!, optimoptions; fdstep)

Mirror of `calibrate_optimize_clustergraph!` (src/calibration.jl:309-359): objective = free energy after
`assignfactors!` -> factor snapshot -> `regfun` -> `calibrate!(sch, maxiter, auto=true)`, per stencil element.
"""
function PGBP.calibrate_optimize_clustergraph!(b::BatchedClusterGraphBelief, cgraph, prenodes::Vector{PN.Node},
        tbl::Tables.ColumnTable, taxa::AbstractVector, evomodelfun, evomodelparams, maxiter::Integer=100,
        regfun=PGBP.regularizebeliefs_bycluster!, optimoptions=Optim.Options(iterations=30); fdstep::Float64=1e-6)
    sch = PGBP.spanningtrees_clusterlist(cgraph, prenodes)
    mod = evomodelfun(evomodelparams...)
    θ0 = PGBP.params_optimize(mod)
    n = length(θ0)
    b.B == 2n + 1 || error("the batch must hold 2n+1 = $(2n+1) elements (central-difference stencil)")
    tips = tipdata([tbl], length(taxa))
    function scores(S)
        out = fill(Inf, size(S, 2))
        models = [evomodelfun(PGBP.params_original(mod, S[:, c])...) for c in axes(S, 2)]
        clearstatus!(b)
        PGBP.assignfactors!(b, reduce(hcat, (bmparams(m) for m in models)), tips; ncolors=ncolors(mod))  # + factor snapshot
        PGBP.init_messagecalibrationflags_reset!(b, true)
        regfun(b, cgraph)
        succ, _ = PGBP.calibrate!(b, sch, maxiter; auto=true)
        fe = PGBP.free_energy(b)[3, :]
        st = status(b)
        for c in axes(S, 2)
            succ[c] && st[c] == 0 && isfinite(fe[c]) && (out[c] = fe[c])
        end
        out
    end
    fg!(F, G, θ) = begin
        f = scores(_stencil(θ, fdstep))
        G === nothing || (G .= (f[2:2:end] .- f[3:2:end]) ./ (2fdstep))
        F === nothing ? nothing : f[1]
    end
    opt = Optim.optimize(Optim.only_fg!(fg!), θ0, Optim.LBFGS(), optimoptions)
    bestmodel = evomodelfun(PGBP.params_original(mod, Optim.minimizer(opt))...)
    return bestmodel, -Optim.minimum(opt), opt
end

"""
    calibrate_exact_cliquetree!(b_improper, b_fixed, spt_improper, spt_fixed, prenodes, tbls, taxa, evomodelfun)

Mirror of `calibrate_exact_cliquetree!` (src/calibration.jl:404-517) for `B` data sets at once (`tbls`: vector of
column tables, no missing values): REML rate matrix and ML root mean from the conditional moments of every node
family (`integratebelief_cov!`), then the likelihood at the optimum with a fixed root.  `b_improper` / `b_fixed`:
batches on plans of the same clique tree allocated for a random and for a fixed root.
Returns `(models::Vector, loglik::Vector)`.
"""
function PGBP.calibrate_exact_cliquetree!(bi::BatchedClusterGraphBelief, bf::BatchedClusterGraphBelief, spt_i, spt_f,
        prenodes::Vector{PN.Node}, tbls::AbstractVector, taxa::AbstractVector, evomodelfun)
    B = bi.B; f = bi.plan.arrays.families
    td = tipdata(tbls, length(taxa)); p = size(td, 1)
    PGBP.assignfactors!(bi, reshape(bmparams([Matrix(1.0LA.I, p, p)], zeros(p), Matrix(LA.Diagonal(fill(Inf, p)))), :, 1), td)
    succ, _ = PGBP.calibrate!(bi, [spt_i])
    moments = Dict{Int,Any}()
    mom(c) = get!(() -> integratebelief_cov!(bi, c + 1)[1:2], moments, c)
    rootpos = f.mem_pos[f.mem_off[1]+1]
    rootpos < 0 && error("the improper-root plan must have the root in scope")
    μhat = mom(f.node_cluster[1])[1][rootpos+1:rootpos+p, :]
    num = zeros(p, p, B); den = zeros(B)
    for v in 2:f.nnodes
        k0 = f.mem_off[v] + 1; k1 = f.mem_off[v+1]
        par = (k0+1):k1
        t = sum(f.mem_gamma[k]^2 * f.mem_length[k] for k in par)
        t == 0 && continue
        μ, cov = mom(f.node_cluster[v])
        if f.node_datarow[v] >= 0
            pa = f.mem_pos[k0+1]; pa < 0 && continue
            d = μ[pa+1:pa+p, :] .- td[:, f.node_datarow[v]+1, :]
            for e in 1:B
                num[:, :, e] .+= d[:, e] * d[:, e]' ./ t
                den[e] += 1 - cov[pa+1, pa+1, e] / t
            end
        else
            ch = f.mem_pos[k0]
            for e in 1:B
                d = μ[ch+1:ch+p, e]; dv = cov[ch+1, ch+1, e]
                for k in par
                    d .-= f.mem_gamma[k] .* μ[f.mem_pos[k]+1:f.mem_pos[k]+p, e]
                    dv -= 2f.mem_gamma[k] * cov[ch+1, f.mem_pos[k]+1, e]
                    for k2 in par
                        dv += f.mem_gamma[k] * f.mem_gamma[k2] * cov[f.mem_pos[k]+1, f.mem_pos[k2]+1, e]
                    end
                end
                num[:, :, e] .+= d * d' ./ t
                den[e] += 1 - dv / t
            end
        end
    end
    σ2 = [num[:, :, e] ./ den[e] for e in 1:B]
    models = [evomodelfun(p == 1 ? σ2[e][1] : σ2[e], p == 1 ? μhat[1, e] : μhat[:, e]) for e in 1:B]
    PGBP.assignfactors!(bf, reduce(hcat, (bmparams(m) for m in models)), td)
    succ2, _ = PGBP.calibrate!(bf, [spt_f])
    _, ll = PGBP.integratebelief!(bf, spt_f[3][1])
    ll[.!(succ .& succ2)] .= NaN
    return models, ll
end

# ---------------------------------------------------------------- multi-GPU gather over NVLink peer windows
"""
    PeerGather(device, rank, nranks, ld; nbuffers = 2)

One process per GPU; `handle(pg)` is the 64-byte CUDA IPC handle of this rank's window, to be exchanged by the host
(e.g. `MPI.Allgather`) and passed to `connect!` in rank order; `integrate_gather!(b, j, pg, k)` then runs
`integratebelief!` and stores every log-likelihood into row `rank` of buffer `k` on every rank.
"""
mutable struct PeerGather
    handle::Ptr{Cvoid}
    nranks::Int
    ld::Int
    function PeerGather(device::Integer, rank::Integer, nranks::Integer, ld::Integer; nbuffers::Integer=2)
        h = Ref{Ptr{Cvoid}}(C_NULL)
        check(ccall((:pgbp_comm_create, LIB), Int32, (Int32, Int32, Int32, Int64, Int32, Ref{Ptr{Cvoid}}), device, rank, nranks, ld, nbuffers, h))
        new(h[], nranks, ld)
    end
end
function handle(pg::PeerGather)
    buf = Vector{UInt8}(undef, 64)
    GC.@preserve buf check(ccall((:pgbp_comm_handle, LIB), Int32, (Ptr{Cvoid}, Ptr{UInt8}), pg.handle, buf))
    buf
end
connect!(pg::PeerGather, handles::Vector{UInt8}) =
    GC.@preserve handles check(ccall((:pgbp_comm_connect, LIB), Int32, (Ptr{Cvoid}, Ptr{UInt8}), pg.handle, handles))
integrate_gather!(b::BatchedClusterGraphBelief, j::Integer, pg::PeerGather, buffer::Integer) =
    check(ccall((:pgbp_integrate_gather, LIB), Int32, (Ptr{Cvoid}, Int32, Ptr{Cvoid}, Int32), b.handle, j - 1, pg.handle, buffer))
put!(pg::PeerGather, b::BatchedClusterGraphBelief, buffer::Integer, d_src::Ptr{Float64}) =
    check(ccall((:pgbp_comm_put, LIB), Int32, (Ptr{Cvoid}, Ptr{Cvoid}, Int32, Ptr{Float64}), pg.handle, b.handle, buffer, d_src))
wait!(pg::PeerGather, b::BatchedClusterGraphBelief, buffer::Integer; timeout_ms::Integer=2000) =
    check(ccall((:pgbp_comm_wait, LIB), Int32, (Ptr{Cvoid}, Ptr{Cvoid}, Int32, Int32), pg.handle, b.handle, buffer, timeout_ms))
function read(pg::PeerGather, b::BatchedClusterGraphBelief, buffer::Integer)
    out = Matrix{Float64}(undef, pg.ld, pg.nranks)
    GC.@preserve out check(ccall((:pgbp_comm_read, LIB), Int32, (Ptr{Cvoid}, Ptr{Cvoid}, Int32, Ptr{Float64}), pg.handle, b.handle, buffer, out))
    out
end
checkwait(pg::PeerGather, b::BatchedClusterGraphBelief) =
    check(ccall((:pgbp_comm_check, LIB), Int32, (Ptr{Cvoid}, Ptr{Cvoid}), pg.handle, b.handle))
"teardown: every rank `disconnect!`s, the ranks synchronise (e.g. `MPI.Barrier`), every rank `destroy!`s"
disconnect!(pg::PeerGather) = check(ccall((:pgbp_comm_disconnect, LIB), Int32, (Ptr{Cvoid},), pg.handle))
destroy!(pg::PeerGather) = (check(ccall((:pgbp_comm_destroy, LIB), Int32, (Ptr{Cvoid},), pg.handle)); pg.handle = C_NULL; nothing)

# ---------------------------------------------------------------- plan dump, for diffing against workloads/*.json
function dumpplan(io::IO, a::PlanArrays)
    println(io, "{\"nclusters\": $(a.nclusters), \"ntraits\": $(a.ntraits), \"belief_dim\": $(a.belief_dim), ",
            "\"sepset_clusters\": $(a.sepset_clusters), \"upind_off\": $(a.upind_off), \"upind\": $(a.upind), ",
            "\"tree_off\": $(a.tree_off), \"tree_parent\": $(a.tree_parent), \"tree_child\": $(a.tree_child)}")
end

end # module
