# CMFsm100.jl -- the Julia-side binding a CMF.jl maintainer would add to run the MU / HALS fit on
# libcmf_sm100 (B200).  NOT EXECUTED in this repository's CI: Julia is not installed in the build
# image; the Python mirror in cmf.jl_b200/ binds exactly the same C symbols and is what the tests run.
#
# Drop-in points (reference file:line):
#   * `SM100MultUpdate <: CMF.AbstractCFUpdate`, `SM100HALSUpdate` -- the update-rule plugin interface
#     (src/algs/alternating.jl:8, constructor call at src/model.jl:79, method calls at alternating.jl:52,54)
#   * `fit_cnmf_sm100` -- replaces the whole `fit_cnmf` (src/model.jl:58-85) with ONE ccall for the loop.
#   * every rule constructor and both fit functions also take `SparseMatrixCSC{T,Int64}` data: its colptr / rowval / nzval
#     go to cmf_set_data_csc as they are (index_base = 1, no copy) and the dense X is never formed.
module CMFsm100

using LinearAlgebra
using SparseArrays
import Random

const LIB = get(ENV, "LIBCMF_SM100", "libcmf_sm100")
const CMF_F64, CMF_F32 = Cint(0), Cint(1)
const CMF_MULT, CMF_HALS, CMF_PGD = Cint(0), Cint(1), Cint(2)

struct CMFError <: Exception
    code::Cint
    msg::String
end

function check(code::Cint)
    code == 0 && return
    msg = unsafe_string(ccall((:cmf_last_error, LIB), Cstring, ()))
    throw(CMFError(code, msg))
end

dtype_code(::Type{Float64}) = CMF_F64
dtype_code(::Type{Float32}) = CMF_F32

"""Opaque device handle; the finalizer releases all device memory (ownership rule of include/cmf_sm100.h)."""
mutable struct Handle
    ptr::Ptr{Cvoid}
    function Handle(N, T, K, L, dtype::Cint, alg::Cint, device::Integer=0; ngpu::Integer=1, devices=nothing, sparse::Bool=false)
        out = Ref{Ptr{Cvoid}}(C_NULL)
        if sparse
            ngpu > 1 && throw(CMFError(3, "sparse data run on one GPU"))
            check(ccall((:cmf_create_sparse, LIB), Cint,
                        (Ref{Ptr{Cvoid}}, Int64, Int64, Int64, Int64, Cint, Cint, Cint),
                        out, N, T, K, L, dtype, alg, device))
        elseif ngpu > 1
            # the fit spans `ngpu` GPUs: time axis sharded INSIDE the library (NCCL communicators, one worker thread and one
            # stream per device), driven from this one Julia task -- no `Distributed`, same calls as a single-GPU handle
            devs = devices === nothing ? C_NULL : convert(Vector{Cint}, devices)
            GC.@preserve devs check(ccall((:cmf_create_multi, LIB), Cint,
                        (Ref{Ptr{Cvoid}}, Int64, Int64, Int64, Int64, Cint, Cint, Cint, Ptr{Cint}),
                        out, N, T, K, L, dtype, alg, ngpu, devs))
        else
        check(ccall((:cmf_create, LIB), Cint,
                    (Ref{Ptr{Cvoid}}, Int64, Int64, Int64, Int64, Cint, Cint, Cint),
                    out, N, T, K, L, dtype, alg, device))
        end
        h = new(out[])
        finalizer(h) do x
            x.ptr == C_NULL || ccall((:cmf_destroy, LIB), Cint, (Ptr{Cvoid},), x.ptr)
            x.ptr = C_NULL
        end
        return h
    end
end

const SparseData{T} = SparseMatrixCSC{T,Int64}

"""X as compressed sparse columns: Julia's own arrays, 1-based, passed without a copy (cmf_set_data_csc)."""
function set_csc!(h::Ptr{Cvoid}, data::SparseData{T}) where {T}
    GC.@preserve data check(ccall((:cmf_set_data_csc, LIB), Cint, (Ptr{Cvoid}, Int64, Ptr{Int64}, Ptr{Int64}, Ptr{Cvoid}, Cint),
                                  h, nnz(data), data.colptr, data.rowval, data.nzval, 1))
end

# ---- update rules behind CMF.jl's own interface ------------------------------------------------
# In CMF.jl these would be declared `<: CMF.AbstractCFUpdate`; the abstract type is re-declared here
# only so that this file parses stand-alone.
abstract type AbstractCFUpdate end

mutable struct SM100Update{ALG} <: AbstractCFUpdate
    h::Handle
    elty::DataType
    sync_host::Bool   # copy W/H back after every half-step (reference in-place semantics)
end
const SM100MultUpdate = SM100Update{:mult}
const SM100HALSUpdate = SM100Update{:hals}
const SM100PGDUpdate = SM100Update{:pgd}    # src/algs/pgd.jl, SquareLoss; l2W/l1W = Square/Absolute penalty weights
alg_code(::Type{SM100Update{:mult}}) = CMF_MULT
alg_code(::Type{SM100Update{:hals}}) = CMF_HALS
alg_code(::Type{SM100Update{:pgd}}) = CMF_PGD

"""`Rule(data, W, H)` -- src/model.jl:79, src/algs/mult.jl:11-20, src/algs/hals.jl:18-28."""
function (::Type{R})(data::Union{Matrix{T},SparseData{T}}, W::Array{T,3}, H::Matrix{T}; sync_host=true, device=0, ngpu=1,
                     devices=nothing, loss_func=:square, mask=nothing, constrW=:nonneg,
                     constrH=:nonneg) where {R<:SM100Update,T<:Union{Float32,Float64}}
    K, N, L = size(W)
    @assert size(data) == (N, size(H, 2)) && size(H, 1) == K
    sparse = data isa SparseData
    sparse && R === SM100PGDUpdate && throw(CMFError(3, "sparse data serve MultUpdate and HALSUpdate"))
    h = Handle(N, size(data, 2), K, L, dtype_code(T), alg_code(R), device; ngpu=ngpu, devices=devices, sparse=sparse)
    if R === SM100PGDUpdate && (loss_func != :square || mask !== nothing)
        # PGD's pluggable losses (src/algs/pgd.jl:28-70): AbsoluteLoss and / or a MaskedLoss around it, on the device
        m = mask === nothing ? nothing : convert(Matrix{T}, mask)
        GC.@preserve m check(ccall((:cmf_set_pgd_loss, LIB), Cint, (Ptr{Cvoid}, Cint, Ptr{Cvoid}),
                                   h.ptr, loss_func == :absolute ? 1 : 0, m === nothing ? C_NULL : pointer(m)))
    end
    if R === SM100PGDUpdate && (constrW != :nonneg || constrH != :nonneg)     # UnitNormConstraint, src/algs/pgd.jl:98-110
        check(ccall((:cmf_set_pgd_constraints, LIB), Cint, (Ptr{Cvoid}, Cint, Cint), h.ptr, constrW == :unitnorm ? 1 : 0, constrH == :unitnorm ? 1 : 0))
    end
    sparse ? set_csc!(h.ptr, data) :
        GC.@preserve data check(ccall((:cmf_set_data, LIB), Cint, (Ptr{Cvoid}, Ptr{Cvoid}, Int64), h.ptr, data, 0))
    GC.@preserve W H check(ccall((:cmf_set_factors, LIB), Cint, (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Cvoid}, Int64), h.ptr, W, H, 0))
    return R(h, T, sync_host)
end

function pull!(rule::SM100Update, W, H)
    GC.@preserve W H check(ccall((:cmf_get_factors, LIB), Cint, (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Cvoid}),
                                 rule.h.ptr, W === nothing ? C_NULL : pointer(W), H === nothing ? C_NULL : pointer(H)))
end

"""`update_motifs!(rule, data, W, H; l1W, l2W)` -- src/algs/mult.jl:23-39 / hals.jl:31-34."""
function update_motifs!(rule::SM100Update, data, W, H; l1W=0, l2W=0, kwargs...)
    check(ccall((:cmf_update_motifs, LIB), Cint, (Ptr{Cvoid}, Cdouble, Cdouble), rule.h.ptr, l1W, l2W))
    rule.sync_host && pull!(rule, W, nothing)
end

"""`loss = update_feature_maps!(rule, data, W, H; l1H, l2H)` -- mult.jl:42-58 / hals.jl:37-42."""
function update_feature_maps!(rule::SM100Update, data, W, H; l1H=0, l2H=0, kwargs...)
    loss = Ref{Cdouble}(0)
    check(ccall((:cmf_update_feature_maps, LIB), Cint, (Ptr{Cvoid}, Cdouble, Cdouble, Ref{Cdouble}),
                rule.h.ptr, l1H, l2H, loss))
    rule.sync_host && pull!(rule, nothing, H)
    return loss[]
end

# ---- coarse entry: the whole alternating loop in one ccall -------------------------------------
struct CNMF_results   # src/model.jl:11-17
    data; W; H; time_hist; loss_hist
end

const ALGS = Dict(:mult => SM100MultUpdate, :hals => SM100HALSUpdate, :pgd => SM100PGDUpdate)

"""src/model.jl:113-125 (kept in Julia so the random stream is the reference's own)."""
function init_rand(data, L, K, tensor_conv)
    N, T = size(data)
    W = rand(K, N, L); H = rand(K, T)
    est = tensor_conv(W, H)
    alpha = dot(vec(data), vec(est)) / norm(est)^2
    return W * sqrt(abs(alpha)), H * sqrt(abs(alpha))
end

"""init_rand for sparse data: the same draws, the alpha rescale on the device through <X, est> = <numH, H> and
||est||^2 = <W W', Htilde Htilde'> (cmf_init_scale_partials), so est is never formed."""
function init_rand(data::SparseData{T}, L, K) where {T}
    N, Tt = size(data)
    W = convert(Array{T,3}, rand(K, N, L)); H = convert(Matrix{T}, rand(K, Tt))
    rule = SM100MultUpdate(data, W, H; sync_host=false)
    part = zeros(Cdouble, 2)
    check(ccall((:cmf_init_scale_partials, LIB), Cint, (Ptr{Cvoid}, Ptr{Cdouble}), rule.h.ptr, part))
    s = sqrt(abs(part[1] / part[2]))
    return W * s, H * s
end
init_rand(data::SparseData, L, K, tensor_conv) = init_rand(data, L, K)

"""tensor_conv(W, H) on the device -- src/common.jl:17-34."""
function tensor_conv(W::Array{T,3}, H::Matrix{T}) where {T}
    K, N, L = size(W); Tt = size(H, 2)
    est = zeros(T, N, Tt)
    GC.@preserve W H est check(ccall((:cmf_tensor_conv, LIB), Cint,
        (Int64, Int64, Int64, Int64, Cint, Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Cvoid}), N, Tt, K, L, dtype_code(T), W, H, est))
    return est
end

"""compute_resids(data, W, H) = tensor_conv(W, H) - data on the device -- src/common.jl:58-59."""
function compute_resids(data::Matrix{T}, W::Array{T,3}, H::Matrix{T}) where {T}
    K, N, L = size(W); Tt = size(H, 2)
    out = zeros(T, N, Tt)
    GC.@preserve data W H out check(ccall((:cmf_compute_resids, LIB), Cint,
        (Int64, Int64, Int64, Int64, Cint, Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Cvoid}), N, Tt, K, L, dtype_code(T), data, W, H, out))
    return out
end

"""shift_and_stack(H, L) on the device -- src/common.jl:133-142 (the fit itself never materialises it)."""
function shift_and_stack(H::Matrix{T}, L::Integer) where {T}
    K, Tt = size(H)
    out = zeros(T, K * L, Tt)
    GC.@preserve H out check(ccall((:cmf_shift_and_stack, LIB), Cint,
        (Int64, Int64, Int64, Cint, Ptr{Cvoid}, Ptr{Cvoid}), K, Tt, L, dtype_code(T), H, out))
    return out
end

"""
    fit_cnmf_sm100(data; L=10, K=5, alg=:mult, max_itr=100, max_time=Inf, ngpu=1, kwargs...)

`ngpu > 1` runs the same fit T-sharded over that many GPUs inside the same single `cmf_fit` call (MultUpdate, HALSUpdate).
`data` may be a `SparseMatrixCSC{T,Int64}` (MultUpdate, HALSUpdate, one GPU; cmf_create_sparse): X is never densified.

Drop-in for `CMF.fit_cnmf` (src/model.jl:58-85).  Accepts both API generations (SURVEY.md Appendix C):
`alg` as `:mult`/`:hals` or a rule type, regularisers as `l1_H…` (README) or `l1H…` (current src),
inits as `W_init/H_init` (or `initW/initH`).  `layout=:LNK` (default, README layout) or `:KNL`.
"""
function fit_cnmf_sm100(data::Union{Matrix{T},SparseData{T}}; L::Integer=10, K::Integer=5, alg=:mult, max_itr=100, max_time=Inf,
                        layout=:LNK, kwargs...) where {T<:Union{Float32,Float64}}
    kw = Dict{Symbol,Any}(kwargs)
    for (a, b) in ((:l1_W, :l1W), (:l2_W, :l2W), (:l1_H, :l1H), (:l2_H, :l2H), (:initW, :W_init), (:initH, :H_init))
        haskey(kw, a) && (kw[b] = pop!(kw, a))
    end
    known = (:l1W, :l2W, :l1H, :l2H, :seed, :W_init, :H_init, :check_convergence, :patience, :eval_mode, :tol, :verbose,
             :engine, :loss_mode, :loss_guard, :ngpu, :devices, :loss_func, :mask)      # sm100 extras (include/cmf_sm100.h): contraction engine 0/1/2, loss
                                                                            # evaluation 0/1, GPUs of the fit, PGD loss (pgd.jl:160,183)
    for k in keys(kw)
        k in known || @warn "fit_cnmf_sm100: unknown keyword $k ignored (CMF.jl ignores it silently)"
    end
    seed = get(kw, :seed, nothing)
    seed === nothing || Random.seed!(seed)                       # model.jl:64-67
    W0, H0 = init_rand(data, L, K, tensor_conv)                  # model.jl:70
    W0 = convert(Array{T,3}, get(kw, :W_init, W0)); H0 = convert(Matrix{T}, get(kw, :H_init, H0))   # model.jl:72-73
    R = alg isa Symbol ? ALGS[alg] : alg
    rule = R(data, W0, H0; sync_host=false, ngpu=get(kw, :ngpu, 1), devices=get(kw, :devices, nothing),
             loss_func=get(kw, :loss_func, :square), mask=get(kw, :mask, nothing))   # model.jl:79
    haskey(kw, :engine) && check(ccall((:cmf_set_engine, LIB), Cint, (Ptr{Cvoid}, Cint), rule.h.ptr, kw[:engine]))
    haskey(kw, :loss_mode) && check(ccall((:cmf_set_loss_mode, LIB), Cint, (Ptr{Cvoid}, Cint), rule.h.ptr, kw[:loss_mode]))
    haskey(kw, :loss_guard) && check(ccall((:cmf_set_loss_guard, LIB), Cint, (Ptr{Cvoid}, Cdouble, Cint), rule.h.ptr, kw[:loss_guard], 16))
    cap = isfinite(max_itr) ? Int(max_itr) + 1 : 1_000_001
    loss_hist = zeros(Cdouble, cap); time_hist = zeros(Cdouble, cap)
    n = Ref{Int64}(0); early = Ref{Cint}(0)
    check(ccall((:cmf_fit, LIB), Cint,
        (Ptr{Cvoid}, Int64, Cdouble, Cint, Cint, Cint, Cdouble, Cdouble, Cdouble, Cdouble, Cdouble,
         Ptr{Cdouble}, Ptr{Cdouble}, Int64, Ref{Int64}, Ref{Cint}),
        rule.h.ptr, isfinite(max_itr) ? Int(max_itr) : -1, Float64(max_time),
        get(kw, :eval_mode, false), get(kw, :check_convergence, true), get(kw, :patience, 3), get(kw, :tol, 1e-4),
        get(kw, :l1W, 0), get(kw, :l2W, R === SM100PGDUpdate ? 1 : 0), get(kw, :l1H, 0), get(kw, :l2H, 0),   # pgd.jl:161 default SquarePenalty(1)
        loss_hist, time_hist, cap, n, early))
    early[] != 0 && println("Converged early.")                 # alternating.jl:64
    W = similar(W0); H = similar(H0)
    pull!(rule, W, H)
    layout == :LNK && (W = permutedims(W, (3, 2, 1)))            # W_LNK[l,n,k] = W_KNL[k,n,l]
    return CNMF_results(data, W, H, time_hist[1:n[]], loss_hist[1:n[]])
end

per_restart(v, R) = v isa Number ? fill(Cdouble(v), R) : (length(v) == R ? convert(Vector{Cdouble}, v) :
                                                          throw(ArgumentError("need a scalar or one value per restart ($R)")))

"""
    fit_cnmf_batch_sm100(data; L=10, K=5, max_itr=100, max_time=Inf, seeds=nothing, W_init=nothing, H_init=nothing, kwargs...)

R MultUpdate fits of the same data in ONE batch handle and ONE `cmf_fit_batch` call (include/cmf_sm100.h).  Restart r
equals `fit_cnmf_sm100(data; seed=seeds[r], l1W=l1W[r], ...)` -- or the fit from `W_init[:,:,:,r]`, `H_init[:,:,r]`
(stacks K x N x L x R and K x T x R, restart last, which is the library's restart-major host layout) -- with every other
keyword the same.  `l1W`, `l2W`, `l1H`, `l2H` are scalars or length-R vectors.  A restart that meets the early stop is
frozen while the others go on; `max_time` and `time_hist` use the batch's own clock (shared by all restarts).  Returns a
vector of R `CNMF_results`.  MultUpdate only, one GPU.  `data` may be a `SparseMatrixCSC{T,Int64}` (cmf_create_batch_sparse).

`K` may be a vector of R ranks (a rank sweep in one handle, `cmf_create_batch_ranks`): restart r then has rank `K[r]`,
`seeds` has R entries, and `W_init` / `H_init` are vectors of R arrays of sizes `K[r] x N x L` and `K[r] x T`.
"""
function fit_cnmf_batch_sm100(data::Union{Matrix{T},SparseData{T}}; L::Integer=10, K::Union{Integer,AbstractVector{<:Integer}}=5, max_itr=100,
                              max_time=Inf, seeds=nothing,
                              W_init=nothing, H_init=nothing, layout=:LNK, device::Integer=0, kwargs...) where {T<:Union{Float32,Float64}}
    kw = Dict{Symbol,Any}(kwargs)
    for (a, b) in ((:l1_W, :l1W), (:l2_W, :l2W), (:l1_H, :l1H), (:l2_H, :l2H))
        haskey(kw, a) && (kw[b] = pop!(kw, a))
    end
    N, Tt = size(data)
    ranks = K isa AbstractVector ? collect(Int64, K) : nothing
    if ranks !== nothing
        (!isempty(ranks) && all(>=(1), ranks)) || throw(ArgumentError("K must hold one rank >= 1 per restart"))
        R = length(ranks)
        if seeds !== nothing
            (W_init === nothing && H_init === nothing) || throw(ArgumentError("give seeds or the W_init / H_init arrays, not both"))
            length(seeds) == R || throw(ArgumentError("need one seed per rank ($R)"))
            Ws, Hs = Array{T,3}[], Matrix{T}[]
            for (k, s) in zip(ranks, seeds)                        # the draws and rescale of fit_cnmf_sm100 (model.jl:64-70)
                Random.seed!(s)
                Wr, Hr = init_rand(data, L, k, tensor_conv)
                push!(Ws, convert(Array{T,3}, Wr)); push!(Hs, convert(Matrix{T}, Hr))
            end
        else
            (W_init === nothing || H_init === nothing) && throw(ArgumentError("need seeds, or both W_init and H_init"))
            (length(W_init) == R && length(H_init) == R) || throw(ArgumentError("need one W_init and one H_init per rank ($R)"))
            Ws = [convert(Array{T,3}, w) for w in W_init]; Hs = [convert(Matrix{T}, x) for x in H_init]
            all(size(Ws[r]) == (ranks[r], N, L) && size(Hs[r]) == (ranks[r], Tt) for r in 1:R) ||
                throw(ArgumentError("W_init[r] must be K[r] x N x L and H_init[r] K[r] x T"))
        end
        W0 = reduce(vcat, vec.(Ws)); H0 = reduce(vcat, vec.(Hs))    # restart-major host layout (include/cmf_sm100.h)
    elseif seeds !== nothing
        (W_init === nothing && H_init === nothing) || throw(ArgumentError("give seeds or the W_init / H_init stacks, not both"))
        R = length(seeds)
        W0 = zeros(T, K, N, L, R); H0 = zeros(T, K, Tt, R)
        for (r, s) in enumerate(seeds)                             # the draws and rescale of fit_cnmf_sm100 (model.jl:64-70)
            Random.seed!(s)
            Wr, Hr = init_rand(data, L, K, tensor_conv)
            W0[:, :, :, r] .= Wr; H0[:, :, r] .= Hr
        end
    else
        (W_init === nothing || H_init === nothing) && throw(ArgumentError("need seeds, or both W_init and H_init"))
        W0 = convert(Array{T,4}, W_init); H0 = convert(Array{T,3}, H_init)
        R = size(W0, 4)
        (size(W0)[1:3] == (K, N, L) && size(H0) == (K, Tt, R)) || throw(ArgumentError("W_init must be K x N x L x R, H_init K x T x R"))
    end
    regs = [per_restart(get(kw, k, 0), R) for k in (:l1W, :l2W, :l1H, :l2H)]
    out = Ref{Ptr{Cvoid}}(C_NULL)
    if data isa SparseData
        rk = ranks === nothing ? fill(Int64(K), R) : ranks
        check(ccall((:cmf_create_batch_sparse, LIB), Cint, (Ref{Ptr{Cvoid}}, Int64, Int64, Ptr{Int64}, Int64, Cint, Cint, Int64, Cint),
                    out, N, Tt, rk, L, dtype_code(T), CMF_MULT, R, device))
    elseif ranks === nothing
        check(ccall((:cmf_create_batch, LIB), Cint, (Ref{Ptr{Cvoid}}, Int64, Int64, Int64, Int64, Cint, Cint, Int64, Cint),
                    out, N, Tt, K, L, dtype_code(T), CMF_MULT, R, device))
    else
        check(ccall((:cmf_create_batch_ranks, LIB), Cint, (Ref{Ptr{Cvoid}}, Int64, Int64, Ptr{Int64}, Int64, Cint, Cint, Int64, Cint),
                    out, N, Tt, ranks, L, dtype_code(T), CMF_MULT, R, device))
    end
    h = out[]
    try
        data isa SparseData ? set_csc!(h, data) : check(ccall((:cmf_set_data, LIB), Cint, (Ptr{Cvoid}, Ptr{Cvoid}, Int64), h, data, 0))
        check(ccall((:cmf_set_factors_batch, LIB), Cint, (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Cvoid}), h, W0, H0))
        cap = isfinite(max_itr) ? Int(max_itr) + 1 : 1_000_001
        loss_hist = zeros(Cdouble, cap, R); time_hist = zeros(Cdouble, cap)
        n = zeros(Int64, R); early = zeros(Cint, R)
        check(ccall((:cmf_fit_batch, LIB), Cint,
            (Ptr{Cvoid}, Int64, Cdouble, Cint, Cint, Cint, Cdouble, Ptr{Cdouble}, Ptr{Cdouble}, Ptr{Cdouble}, Ptr{Cdouble},
             Ptr{Cdouble}, Ptr{Cdouble}, Int64, Ptr{Int64}, Ptr{Cint}),
            h, isfinite(max_itr) ? Int(max_itr) : -1, Float64(max_time),
            get(kw, :eval_mode, false), get(kw, :check_convergence, true), get(kw, :patience, 3), get(kw, :tol, 1e-4),
            regs[1], regs[2], regs[3], regs[4], loss_hist, time_hist, cap, n, early))
        for r in 1:R
            early[r] != 0 && println("Converged early.")          # alternating.jl:64, once per restart that stopped early
        end
        W = similar(W0); H = similar(H0)
        check(ccall((:cmf_get_factors_batch, LIB), Cint, (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Cvoid}), h, W, H))
        if ranks !== nothing
            offs = [0; cumsum(ranks)]
            res = CNMF_results[]
            for r in 1:R
                k, o = ranks[r], offs[r]
                Wr = reshape(W[N*L*o+1:N*L*(o+k)], k, N, L); Hr = reshape(H[Tt*o+1:Tt*(o+k)], k, Tt)
                push!(res, CNMF_results(data, layout == :LNK ? permutedims(Wr, (3, 2, 1)) : Wr, Hr, time_hist[1:n[r]],
                                        loss_hist[1:n[r], r]))
            end
            return res
        end
        return [CNMF_results(data, layout == :LNK ? permutedims(W[:, :, :, r], (3, 2, 1)) : W[:, :, :, r], H[:, :, r],
                             time_hist[1:n[r]], loss_hist[1:n[r], r]) for r in 1:R]
    finally
        ccall((:cmf_destroy, LIB), Cint, (Ptr{Cvoid},), h)
    end
end

end # module
