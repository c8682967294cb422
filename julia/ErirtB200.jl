# ErirtB200.jl -- reference-side binding of liberirt_b200.so (include/erirt_b200.h).
#
# This file is what a maintainer of ExtendedRtIrtModeling.jl adds to the package (INTEGRATION.md): it keeps the
# package's API (setCond, InputData, the Gibbs* constructors, sample!, MCMC.Post.mean, coef, precis) and replaces
# only the BODY of the `sample!` methods (src/GibbsRtIrt.pl.jl:210-257, :278-346, :367-426,
# src/GibbsRtIrtLatent.pl.jl:168-233, :271-337) by ccalls.  Julia is not installed in the build container, so this
# shim is delivered as source and has not been executed; the same C ABI is exercised by the Python ctypes mirror
# (extendedrtirtmodeling.jl_b200/engine.py) in the test-suite.
module ErirtB200

using ExtendedRtIrtModeling
import ExtendedRtIrtModeling: sample!, InputPara, GibbsMlIrt, GibbsRtIrt, GibbsRtIrtNull, GibbsRtIrtCross, GibbsRtIrtCrossQr,
                               GibbsRtIrtLatent, GibbsRtIrtLatentQr

export GibbsRtIrtQuantile, lean, LeanGibbs, LeanPost, Shard, sample_sharded!, sample_batch!, ess_rhat_gpu, checkConvergence_gpu

const LIB = get(ENV, "ERIRT_B200_LIB", joinpath(@__DIR__, "..", "extendedrtirtmodeling.jl_b200", "liberirt_b200.so"))

# struct erirt_config (include/erirt_b200.h) -- field order and C alignment must match
struct ErirtConfig
    abi_version::Int32
    model::Int32
    n_subj::Int64
    n_subj_total::Int64
    subj_offset::Int64
    n_item::Int32
    n_feat::Int32
    n_iter::Int32
    n_chain::Int32
    n_burnin::Int32
    q_rt::Float64
    intercept::Int32
    itemtype_1pl::Int32
    cov2one::Int32
    dtype::Int32
    seed::UInt64
    chain::UInt32
    compat::Int32
    person_trace::Int32
    device::Int32
    use_graph::Int32
    time_kernels::Int32
    nu_cell_moments::Int32
    reserved::NTuple{6,Int32}
end

const MODEL_ID = Dict(GibbsMlIrt => 0, GibbsRtIrt => 1, GibbsRtIrtNull => 2, GibbsRtIrtCross => 3, GibbsRtIrtCrossQr => 4,
                      GibbsRtIrtLatent => 5, GibbsRtIrtLatentQr => 6)
const F_THETA, F_ZETA, F_A, F_B, F_LAMBDA, F_SIGMA2, F_BETA, F_RHO, F_SIGMA_P, F_NU = Int32.(0:9)
const T_RA, T_RT, T_QR, T_LL = Int32.(0:3)

lasterror() = unsafe_string(ccall((:erirt_last_error, LIB), Cstring, ()))
check(rc) = rc == 0 ? nothing : error("erirt_b200: " * lasterror())

"README.md:95 names GibbsRtIrtQuantile; the package ships that sampler as GibbsRtIrtLatentQr (export commented out at src/ExtendedRtIrtModeling.jl:65)."
GibbsRtIrtQuantile(Cond; kwargs...) = GibbsRtIrtLatentQr(Cond; kwargs...)

function _set_state(h, field, v)
    isempty(v) && return
    x = Vector{Float64}(vec(v))
    GC.@preserve x check(ccall((:erirt_set_state, LIB), Cint, (Ptr{Cvoid}, Int32, Ptr{Float64}, Int64), h, field, x, length(x)))
end

function _trace!(h, which, out::Array{Float64,3}, first_col)
    GC.@preserve out check(ccall((:erirt_get_trace, LIB), Cint, (Ptr{Cvoid}, Int32, Int64, Int64, Ptr{Float64}),
                                 h, which, first_col, size(out, 2), out))
end

# Person columns of Post.ra / rt / qr are kept on the device (and copied back) only when nIter*nChain*3*nSubj reals fit this budget;
# beyond it only the item / structural columns are traced and θ, ζ, ν come back as post-burn-in means and SDs (erirt_get_moments),
# which is all Post.mean needs (SURVEY 0.10: at nSubj = 1M the reference's own trace would be 160 TB).
const PERSON_TRACE_BUDGET_MB = parse(Int, get(ENV, "ERIRT_PERSON_TRACE_MB", "8192"))
person_trace_fits(Cond, dtype) = 3 * Cond.nIter * Cond.nChain * Cond.nSubj * (dtype == 0 ? 4 : 8) <= PERSON_TRACE_BUDGET_MB * 2^20

struct Shard                      # one rank of a person-sharded chain (INTEGRATION.md section 2)
    rank::Int32
    world::Int32
    offset::Int64                 # global id of this rank's first person
    total::Int64                  # persons of the whole chain
    allgather::Function           # bytes::Vector{UInt8} -> concatenation over the ranks, in rank order (e.g. MPI.Allgather)
    barrier::Function             # () -> nothing, host barrier over the ranks
end

function _moments(h, field, n)
    m, sd = Vector{Float64}(undef, n), Vector{Float64}(undef, n)
    GC.@preserve m sd check(ccall((:erirt_get_moments, LIB), Cint, (Ptr{Cvoid}, Int32, Ptr{Float64}, Ptr{Float64}, Int64), h, field, m, sd, n))
    return m, sd
end

# item / structural columns [first_col, first_col + ncols) of Post.<which> into dest[:, dest_cols, :]
function _trace_cols!(h, which, dest::AbstractArray{Float64,3}, dest_cols, first_col)
    tmp = Array{Float64}(undef, size(dest, 1), length(dest_cols), size(dest, 3))
    _trace!(h, which, tmp, first_col)
    dest[:, dest_cols, :] .= tmp
end

"""
Body of every `sample!` method.  `Post` is any object with `ra`, `rt`, `qr`, `logLike` arrays: the reference's OutputPost* (person
columns present, width nSubj + 2 nItem) or a `LeanPost` (item / structural columns only).  Returns a NamedTuple with the person-level
posterior means / SDs when the person trace was off (`nothing` entries otherwise) and CrossQr's mean weights.
"""
function _sample_gpu!(MCMC; intercept=false, itemtype="2pl", cov2one=true, dtype=1, seed=rand(UInt64), device=0,
                      person_trace::Union{Bool,Nothing}=nothing, shard::Union{Shard,Nothing}=nothing, modeltype=typeof(MCMC))
    if !(itemtype in ["1pl", "2pl"])
        error("Invalid input: the item type must be '1pl' or '2pl'.")     # src/GibbsRtIrt.pl.jl:212-214
    end
    Cond, Data, Para, Post = MCMC.Cond, MCMC.Data, MCMC.Para, MCMC.Post
    N, J, F = Cond.nSubj, Cond.nItem, Cond.nFeat      # N = persons held by THIS process (the shard's, when sharded)
    has_rt = !(modeltype === GibbsMlIrt)
    cqr = modeltype === GibbsRtIrtCrossQr
    lqr = modeltype === GibbsRtIrtLatentQr
    lean = Post isa LeanPost
    ptrace = lean ? false : (person_trace === nothing ? person_trace_fits(Cond, dtype) : person_trace)
    total, offset = shard === nothing ? (N, 0) : (shard.total, shard.offset)
    cfg = ErirtConfig(1, MODEL_ID[modeltype], N, total, offset, J, F, Cond.nIter, Cond.nChain, Cond.nBurnin, Cond.qRt,
                      intercept, itemtype == "1pl", cov2one, dtype, seed, 0, 0, ptrace, device, 1, 0, cqr, ntuple(_ -> Int32(0), 6))
    νmean = Float64[]   # CrossQr: post-burn-in mean of the N*J weights
    person = (θ=nothing, θsd=nothing, ζ=nothing, ζsd=nothing, ν=nothing, νsd=nothing)
    href = Ref{Ptr{Cvoid}}(C_NULL)
    check(ccall((:erirt_create, LIB), Cint, (Ref{ErirtConfig}, Ref{Ptr{Cvoid}}), cfg, href))
    h = href[]
    try
        if shard !== nothing      # rank / world, then the fused exchange over NVLink peer memory (no NCCL communicator)
            check(ccall((:erirt_comm_init, LIB), Cint, (Ptr{Cvoid}, Int32, Int32, Ptr{Cvoid}), h, shard.rank, shard.world, C_NULL))
            mine = Vector{UInt8}(undef, 64)
            GC.@preserve mine check(ccall((:erirt_peer_export, LIB), Cint, (Ptr{Cvoid}, Ptr{UInt8}), h, mine))
            all = shard.allgather(mine)::Vector{UInt8}
            GC.@preserve all check(ccall((:erirt_peer_attach, LIB), Cint, (Ptr{Cvoid}, Ptr{UInt8}), h, all))
        end
        logT = has_rt ? Matrix{Float64}(Data.logT) : zeros(0, 0)
        X = F > 0 ? Matrix{Float64}(Data.X) : zeros(0, 0)
        if Data.Y isa Matrix{Bool}   # rand.(BernoulliLogit…) of src/SimTools.jl:165: one byte per response, passed as it lies in memory
            Y8 = Data.Y
            GC.@preserve Y8 logT X check(ccall((:erirt_set_data_y8, LIB), Cint,
                (Ptr{Cvoid}, Ptr{Bool}, Int64, Ptr{Float64}, Int64, Ptr{Float64}, Int64),
                h, Y8, N, has_rt ? pointer(logT) : C_NULL, N, F > 0 ? pointer(X) : C_NULL, N))
        else                         # Int from CSV (src/Base.pl.jl:84-95) or Float64
            Y = Matrix{Float64}(Data.Y)
            GC.@preserve Y logT X check(ccall((:erirt_set_data, LIB), Cint,
                (Ptr{Cvoid}, Ptr{Float64}, Int64, Ptr{Float64}, Int64, Ptr{Float64}, Int64),
                h, Y, N, has_rt ? pointer(logT) : C_NULL, N, F > 0 ? pointer(X) : C_NULL, N))
        end
        _set_state(h, F_THETA, Para.θ); _set_state(h, F_A, Para.a); _set_state(h, F_B, Para.b)
        if has_rt
            _set_state(h, F_ZETA, Para.ζ); _set_state(h, F_LAMBDA, Para.λ); _set_state(h, F_SIGMA2, Para.σ²t)
            _set_state(h, F_SIGMA_P, Matrix{Float64}(Para.Σp))
        end
        _set_state(h, F_BETA, Para.β)
        (modeltype === GibbsRtIrtCross || cqr) && _set_state(h, F_RHO, Para.ρ)
        check(ccall((:erirt_sample, LIB), Cint, (Ptr{Cvoid}, Int64), h, Cond.nIter * Cond.nChain))
        qw = Int(ccall((:erirt_trace_width, LIB), Int64, (Ptr{Cvoid}, Int32), h, T_QR)) - (lqr ? N : 0)   # item / structural width of qr
        if ptrace
            # fill the pre-allocated Post arrays (same layouts, src/GibbsRtIrt.pl.jl:63-69)
            _trace!(h, T_RA, Post.ra, 0)
            has_rt && _trace!(h, T_RT, Post.rt, 0)
            if cqr
                # the reference traces all N*J weights per sweep (src/GibbsRtIrtCross.pl.jl:65, :297); the engine keeps their running
                # mean instead, so only the [ρ; vec Σp] columns of Post.qr are filled and Post.mean.ν comes from erirt_get_moments
                _trace_cols!(h, T_QR, Post.qr, 1:(J + 4), 0)
            else
                _trace!(h, T_QR, Post.qr, 0)
            end
        else
            # person trace off: item / structural columns only.  A reference OutputPost keeps its width (person columns stay
            # unset: `undef` as allocated); a LeanPost has exactly the item / structural columns.
            c0 = lean ? 0 : N
            _trace_cols!(h, T_RA, Post.ra, (c0 + 1):(c0 + 2J), N)
            has_rt && _trace_cols!(h, T_RT, Post.rt, (c0 + 1):(c0 + 2J), N)
            _trace_cols!(h, T_QR, Post.qr, 1:qw, 0)
            θ, θsd = _moments(h, F_THETA, N)
            ζ, ζsd = has_rt ? _moments(h, F_ZETA, N) : (nothing, nothing)
            ν, νsd = lqr ? _moments(h, F_NU, N) : (nothing, nothing)
            person = (θ=θ, θsd=θsd, ζ=ζ, ζsd=ζsd, ν=ν, νsd=νsd)
        end
        if cqr
            νmean = Vector{Float64}(undef, N * J)
            GC.@preserve νmean check(ccall((:erirt_get_moments, LIB), Cint, (Ptr{Cvoid}, Int32, Ptr{Float64}, Ptr{Float64}, Int64),
                                           h, F_NU, νmean, C_NULL, N * J))
        end
        _trace!(h, T_LL, Post.logLike, 0)
        if shard !== nothing      # unmap the peers' exchange buffers on every rank before anybody frees its own
            check(ccall((:erirt_peer_detach, LIB), Cint, (Ptr{Cvoid},), h))
            shard.barrier()
        end
    finally
        ccall((:erirt_destroy, LIB), Cint, (Ptr{Cvoid},), h)
    end
    return (person=person, νcell=νmean)
end

_pm(A, r, nb) = vec(ExtendedRtIrtModeling.mean(A[(nb + 1):end, r, :], dims=(1, 3)))
_or(x, f) = x === nothing ? f() : x     # person means from the moments when the trace was off, else from the trace columns

# ---- the sample! methods: same signatures as the reference (plus the engine's keyword options), body replaced ----
function sample!(MCMC::GibbsMlIrt; intercept=false, itemtype::Union{String}="2pl", kw...)
    r = _sample_gpu!(MCMC; intercept, itemtype, kw...)
    C, P = MCMC.Cond, MCMC.Post
    P.mean = InputPara(θ=_or(r.person.θ, () -> _pm(P.ra, 1:C.nSubj, C.nBurnin)), a=_pm(P.ra, (C.nSubj + 1):(C.nSubj + C.nItem), C.nBurnin),
                       b=_pm(P.ra, (C.nSubj + C.nItem + 1):size(P.ra, 2), C.nBurnin), β=_pm(P.qr, 1:(C.nFeat + 1), C.nBurnin))
    return MCMC
end

function _rt_mean!(MCMC, nβ, r; with_ν=false)
    C, P = MCMC.Cond, MCMC.Post
    nb, N, J = C.nBurnin, C.nSubj, C.nItem
    c0 = size(P.ra, 2) - 2J      # N for the reference's OutputPost, 0 for a LeanPost
    P.mean = InputPara(β=_pm(P.qr, 1:nβ, nb), Σp=_pm(P.qr, (nβ + 1):(nβ + 4), nb),
                       ν=with_ν ? _or(r.person.ν, () -> _pm(P.qr, (nβ + 5):size(P.qr, 2), nb)) : Float64[],
                       θ=_or(r.person.θ, () -> _pm(P.ra, 1:N, nb)), a=_pm(P.ra, (c0 + 1):(c0 + J), nb), b=_pm(P.ra, (c0 + J + 1):(c0 + 2J), nb),
                       ζ=_or(r.person.ζ, () -> _pm(P.rt, 1:N, nb)), λ=_pm(P.rt, (c0 + 1):(c0 + J), nb), σ²t=_pm(P.rt, (c0 + J + 1):(c0 + 2J), nb))
    return MCMC
end

function sample!(MCMC::GibbsRtIrt; intercept=false, itemtype::Union{String}="2pl", cov2one=true, kw...)
    r = _sample_gpu!(MCMC; intercept, itemtype, cov2one, kw...); _rt_mean!(MCMC, 2 * (MCMC.Cond.nFeat + 1), r)
end
function sample!(MCMC::GibbsRtIrtNull; itemtype::Union{String}="2pl", cov2one=true, kw...)
    r = _sample_gpu!(MCMC; itemtype, cov2one, kw...); _rt_mean!(MCMC, 2 * (MCMC.Cond.nFeat + 1), r)
end
function _cross_mean!(MCMC, r)
    C, P = MCMC.Cond, MCMC.Post
    nb, N, J = C.nBurnin, C.nSubj, C.nItem
    c0 = size(P.ra, 2) - 2J
    P.mean = InputPara(ρ=_pm(P.qr, 1:J, nb), Σp=_pm(P.qr, (J + 1):(J + 4), nb), ν=r.νcell,
                       θ=_or(r.person.θ, () -> _pm(P.ra, 1:N, nb)), a=_pm(P.ra, (c0 + 1):(c0 + J), nb), b=_pm(P.ra, (c0 + J + 1):(c0 + 2J), nb),
                       ζ=_or(r.person.ζ, () -> _pm(P.rt, 1:N, nb)), λ=_pm(P.rt, (c0 + 1):(c0 + J), nb), σ²t=_pm(P.rt, (c0 + J + 1):(c0 + 2J), nb))
    return MCMC
end
function sample!(MCMC::GibbsRtIrtCross; itemtype::Union{String}="2pl", cov2one=true, kw...)      # src/GibbsRtIrtCross.pl.jl:176
    r = _sample_gpu!(MCMC; itemtype, cov2one, kw...); _cross_mean!(MCMC, r)
end
function sample!(MCMC::GibbsRtIrtCrossQr; itemtype::Union{String}="2pl", cov2one=true, kw...)    # src/GibbsRtIrtCross.pl.jl:265
    r = _sample_gpu!(MCMC; itemtype, cov2one, kw...); _cross_mean!(MCMC, r)                       # Post.mean.ν, :310
end
function sample!(MCMC::GibbsRtIrtLatent; intercept=false, itemtype::Union{String}="2pl", cov2one=false, kw...)
    r = _sample_gpu!(MCMC; intercept, itemtype, cov2one, kw...); _rt_mean!(MCMC, MCMC.Cond.nFeat + 2, r)
end
function sample!(MCMC::GibbsRtIrtLatentQr; intercept=false, itemtype::Union{String}="2pl", cov2one=false, kw...)
    r = _sample_gpu!(MCMC; intercept, itemtype, cov2one, kw...); _rt_mean!(MCMC, MCMC.Cond.nFeat + 2, r; with_ν=true)
end

# ---- large nSubj: a lean model object.  The reference's constructors allocate Post.ra / rt as nIter x (nSubj + 2 nItem) x nChain
#      (src/GibbsRtIrt.pl.jl:63-69; 160 TB at nSubj = 1M, nIter = 5000, nChain = 4) inside an inner constructor, so a model of that
#      size cannot even be constructed.  `lean(GibbsRtIrtLatentQr, Cond; Data)` builds the same five fields with a LeanPost that holds
#      the item / structural columns only; `sample!` fills Post.mean.θ / ζ / ν (and Post.sd) from the engine's running moments. ----
mutable struct LeanPost
    ra::Array{Float64,3}        # [nIter, 2 nItem, nChain]  a, b
    rt::Array{Float64,3}        # [nIter, 2 nItem, nChain]  λ, σ²t
    qr::Array{Float64,3}        # [nIter, qw, nChain]       β / ρ, vec Σp  (no ν block)
    logLike::Array{Float64,3}
    mean
    sd                          # (θ, ζ, ν) posterior SDs from erirt_get_moments
end
mutable struct LeanGibbs
    modeltype::DataType         # GibbsMlIrt, GibbsRtIrt, ..., GibbsRtIrtLatentQr
    Cond
    Data
    truePara
    Para
    Post::LeanPost
end
_qw(T, J, F) = T === GibbsMlIrt ? F + 1 : (T === GibbsRtIrt || T === GibbsRtIrtNull) ? 2 * (F + 1) + 4 :
               (T === GibbsRtIrtCross || T === GibbsRtIrtCrossQr) ? J + 4 : F + 2 + 4
function lean(T::DataType, Cond; Data, truePara=Float64[], Para=nothing)
    N, J, F = Cond.nSubj, Cond.nItem, Cond.nFeat
    nβ = T === GibbsMlIrt ? (F + 1,) : (T === GibbsRtIrt || T === GibbsRtIrtNull) ? (F + 1, 2) : (F + 2,)
    if Para === nothing        # setInitialValues of the reference (src/GibbsRtIrt.pl.jl:84-133, Cross :77-147, Latent :70-137)
        Para = InputPara(θ=randn(N), a=ones(J), b=zeros(J), ζ=randn(N), λ=zeros(J), σ²t=ones(J),
                         β=T === GibbsRtIrtNull ? zeros(nβ...) : randn(nβ...), ρ=randn(J), Σp=[1.0 0.0; 0.0 1.0])
    end
    post = LeanPost(Array{Float64}(undef, Cond.nIter, 2J, Cond.nChain), Array{Float64}(undef, Cond.nIter, 2J, Cond.nChain),
                    Array{Float64}(undef, Cond.nIter, _qw(T, J, F), Cond.nChain), Array{Float64}(undef, Cond.nIter, 1, Cond.nChain),
                    Float64[], nothing)
    return LeanGibbs(T, Cond, Data, truePara, Para, post)
end
function sample!(MCMC::LeanGibbs; intercept=false, itemtype::Union{String}="2pl",
                 cov2one=!(MCMC.modeltype === GibbsRtIrtLatent || MCMC.modeltype === GibbsRtIrtLatentQr), kw...)
    T = MCMC.modeltype
    r = _sample_gpu!(MCMC; intercept, itemtype, cov2one, modeltype=T, kw...)
    F = MCMC.Cond.nFeat
    if T === GibbsMlIrt
        C, P = MCMC.Cond, MCMC.Post
        P.mean = InputPara(θ=r.person.θ, a=_pm(P.ra, 1:C.nItem, C.nBurnin), b=_pm(P.ra, (C.nItem + 1):(2 * C.nItem), C.nBurnin),
                           β=_pm(P.qr, 1:(F + 1), C.nBurnin))
    elseif T === GibbsRtIrtCross || T === GibbsRtIrtCrossQr
        _cross_mean!(MCMC, r)
    else
        _rt_mean!(MCMC, (T === GibbsRtIrt || T === GibbsRtIrtNull) ? 2 * (F + 1) : F + 2, r; with_ν=T === GibbsRtIrtLatentQr)
    end
    MCMC.Post.sd = (θ=r.person.θsd, ζ=r.person.ζsd, ν=r.person.νsd)
    return MCMC
end

"""
    sample_sharded!(MCMC::LeanGibbs, shard::Shard; kw...)

One rank of a person-sharded chain (BASELINE configs[4]; INTEGRATION.md section 2): this process holds the rows `shard.offset + 1 :
shard.offset + MCMC.Cond.nSubj` of Y, logT, X (its `Data`) and their initial θ, ζ, one GPU (`device`), and calls this on every rank
with the SAME `seed`.  Item / structural traces are identical on every rank; Post.mean.θ / ζ / ν are this rank's persons.
"""
sample_sharded!(MCMC::LeanGibbs, shard::Shard; kw...) = sample!(MCMC; shard=shard, kw...)

# ---- replica batches (erirt_create_batch, DESIGN.md 6.6): B replications of one model, e.g. the nRep data sets of runSimulation
#      (src/SimTools.jl:457-495), sampled by ONE handle with one person launch and one global launch per sweep ----
function _trace4!(h, which, out::Array{Float64,4}, first_col)   # [nIter, ncols, nChain, B]
    GC.@preserve out check(ccall((:erirt_get_trace, LIB), Cint, (Ptr{Cvoid}, Int32, Int64, Int64, Ptr{Float64}),
                                 h, which, first_col, size(out, 2), out))
end

"""
    sample_batch!(MCMCs::AbstractVector; intercept=false, itemtype="2pl", cov2one, dtype=1, seed=rand(UInt64), device=0)

`sample!(MCMCs[r]; seed=seed + r - 1, person_trace=false)` for every r, as one replica batch on one GPU.  The model objects are of one
of the five one-launch types (GibbsMlIrt, GibbsRtIrt, GibbsRtIrtNull, GibbsRtIrtLatent, GibbsRtIrtLatentQr) with equal Cond; each has
its own Data and initial Para.  Replica r's chain is the one its own `sample!` with that seed would draw (same Philox stream), so
Post (item / structural traces, logLike) and Post.mean (θ, ζ, ν from the running moments) are filled as that call fills them.
"""
function sample_batch!(MCMCs::AbstractVector; intercept=false, itemtype::Union{String}="2pl", cov2one=nothing, dtype=1,
                       seed=rand(UInt64), device=0)
    T, B = typeof(MCMCs[1]), length(MCMCs)
    Cond = MCMCs[1].Cond
    all(M -> typeof(M) === T && M.Cond == Cond, MCMCs) || error("sample_batch!: the model objects must share one type and one Cond")
    (T === GibbsRtIrtCross || T === GibbsRtIrtCrossQr) && error("sample_batch!: the Cross family is not batched")
    itemtype in ["1pl", "2pl"] || error("Invalid input: the item type must be '1pl' or '2pl'.")
    cov2one === nothing && (cov2one = !(T === GibbsRtIrtLatent || T === GibbsRtIrtLatentQr))
    N, J, F, nb = Cond.nSubj, Cond.nItem, Cond.nFeat, Cond.nBurnin
    has_rt, lqr = !(T === GibbsMlIrt), T === GibbsRtIrtLatentQr
    cfg = ErirtConfig(1, MODEL_ID[T], N, N, 0, J, F, Cond.nIter, Cond.nChain, nb, Cond.qRt, intercept, itemtype == "1pl", cov2one,
                      dtype, seed, 0, 0, 0, device, 1, 0, 0, ntuple(_ -> Int32(0), 6))
    href = Ref{Ptr{Cvoid}}(C_NULL)
    check(ccall((:erirt_create_batch, LIB), Cint, (Ref{ErirtConfig}, Int32, Ref{Ptr{Cvoid}}), cfg, Int32(B), href))
    h = href[]
    try
        # person-indexed matrices stack the replicas along the rows; every other field is B consecutive blocks
        Y = reduce(vcat, [Matrix{Float64}(M.Data.Y) for M in MCMCs])
        logT = has_rt ? reduce(vcat, [Matrix{Float64}(M.Data.logT) for M in MCMCs]) : zeros(0, 0)
        X = F > 0 ? reduce(vcat, [Matrix{Float64}(M.Data.X) for M in MCMCs]) : zeros(0, 0)
        GC.@preserve Y logT X check(ccall((:erirt_set_data, LIB), Cint,
            (Ptr{Cvoid}, Ptr{Float64}, Int64, Ptr{Float64}, Int64, Ptr{Float64}, Int64),
            h, Y, B * N, has_rt ? pointer(logT) : C_NULL, B * N, F > 0 ? pointer(X) : C_NULL, B * N))
        stacked(f) = reduce(vcat, [vec(Matrix{Float64}(reshape(f(M.Para), :, 1))) for M in MCMCs])
        _set_state(h, F_THETA, stacked(p -> p.θ)); _set_state(h, F_A, stacked(p -> p.a)); _set_state(h, F_B, stacked(p -> p.b))
        if has_rt
            _set_state(h, F_ZETA, stacked(p -> p.ζ)); _set_state(h, F_LAMBDA, stacked(p -> p.λ)); _set_state(h, F_SIGMA2, stacked(p -> p.σ²t))
            _set_state(h, F_SIGMA_P, stacked(p -> p.Σp))
        end
        _set_state(h, F_BETA, stacked(p -> p.β))
        check(ccall((:erirt_sample, LIB), Cint, (Ptr{Cvoid}, Int64), h, Cond.nIter * Cond.nChain))
        qw = Int(ccall((:erirt_trace_width, LIB), Int64, (Ptr{Cvoid}, Int32), h, T_QR)) - (lqr ? N : 0)
        shape(w) = Array{Float64}(undef, Cond.nIter, w, Cond.nChain, B)
        ra, rt, qr, ll = shape(2J), shape(has_rt ? 2J : 0), shape(qw), shape(1)
        _trace4!(h, T_RA, ra, N); has_rt && _trace4!(h, T_RT, rt, N); _trace4!(h, T_QR, qr, 0); _trace4!(h, T_LL, ll, 0)
        θ, θsd = _moments(h, F_THETA, B * N)
        ζ, ζsd = has_rt ? _moments(h, F_ZETA, B * N) : (nothing, nothing)
        ν, νsd = lqr ? _moments(h, F_NU, B * N) : (nothing, nothing)
        for (r, M) in enumerate(MCMCs)
            P, rows = M.Post, ((r - 1) * N + 1):(r * N)
            c0 = size(P.ra, 2) - 2J
            P.ra[:, (c0 + 1):(c0 + 2J), :] .= ra[:, :, :, r]
            has_rt && (P.rt[:, (c0 + 1):(c0 + 2J), :] .= rt[:, :, :, r])
            P.qr[:, 1:qw, :] .= qr[:, :, :, r]
            P.logLike .= ll[:, :, :, r]
            sel(v) = v === nothing ? nothing : v[rows]
            res = (person=(θ=sel(θ), θsd=sel(θsd), ζ=sel(ζ), ζsd=sel(ζsd), ν=sel(ν), νsd=sel(νsd)), νcell=Float64[])
            if T === GibbsMlIrt
                P.mean = InputPara(θ=res.person.θ, a=_pm(P.ra, (c0 + 1):(c0 + J), nb), b=_pm(P.ra, (c0 + J + 1):(c0 + 2J), nb),
                                   β=_pm(P.qr, 1:(F + 1), nb))
            else
                _rt_mean!(M, (T === GibbsRtIrt || T === GibbsRtIrtNull) ? 2 * (F + 1) : F + 2, res; with_ν=lqr)
            end
        end
    finally
        ccall((:erirt_destroy, LIB), Cint, (Ptr{Cvoid},), h)
    end
    return MCMCs
end

# ---- simulated data generated on the device (erirt_generate_data): the N x J part of setData* (src/SimTools.jl:117-368) never exists on
#      the host.  `truePara` holds the person-level draws θ (and ζ) made by the caller as in setData*, X the covariates (or nothing);
#      errortype: 0 truncated normal (Null / RtIrt), 1 N(0,1) (Latent*), 2 / 3 / 4 = "norm" / "tail" / "skew" (Cross) ----
function generate_data!(h, truePara, X, errortype::Integer; seed::UInt64=rand(UInt64))
    ptr(v) = isempty(v) ? Ptr{Float64}(C_NULL) : pointer(v)
    θ, ζ = Vector{Float64}(vec(truePara.θ)), Vector{Float64}(vec(truePara.ζ))
    a, b, λ = Vector{Float64}(vec(truePara.a)), Vector{Float64}(vec(truePara.b)), Vector{Float64}(vec(truePara.λ))
    σ², ρ = Vector{Float64}(vec(truePara.σ²t)), Vector{Float64}(vec(truePara.ρ))
    Xm = X === nothing ? zeros(0, 0) : Matrix{Float64}(X)
    GC.@preserve θ ζ a b λ σ² ρ Xm check(ccall((:erirt_generate_data, LIB), Cint,
        (Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Int64, Int32, UInt64),
        h, θ, ptr(ζ), a, b, ptr(λ), ptr(σ²), ptr(ρ), ptr(Xm), max(size(Xm, 1), 1), errortype, seed))
end

# ---- checkpoint / resume of a running chain (erirt_checkpoint_*): `h` is the handle of a chain driven in chunks ----
function checkpoint(h)::Vector{UInt8}
    n = ccall((:erirt_checkpoint_size, LIB), Int64, (Ptr{Cvoid},), h)
    n < 0 && error("erirt_b200: " * lasterror())
    buf = Vector{UInt8}(undef, n)
    GC.@preserve buf check(ccall((:erirt_checkpoint_save, LIB), Cint, (Ptr{Cvoid}, Ptr{UInt8}, Int64), h, buf, n))
    return buf      # write(io, buf) to persist it
end
restore!(h, buf::Vector{UInt8}) =
    GC.@preserve buf check(ccall((:erirt_checkpoint_load, LIB), Cint, (Ptr{Cvoid}, Ptr{UInt8}, Int64), h, buf, length(buf)))

# ---- convergence diagnostics on the device (erirt_ess_rhat, csrc/diagnostics.cuh): the estimator behind `Chains(...) |> ess_rhat` in
#      checkConvergence (src/SimTools.jl:419-443), one CTA per column.  `post` is any Post.ra / Post.rt / Post.qr block
#      [nIter, P, nChain]; returns (ess, rhat), NaN for constant columns (MCMCChains gives missing / NaN there as well) ----
function ess_rhat_gpu(post::Array{Float64,3}; skip::Integer=0, device::Integer=0)
    ess, rhat = Vector{Float64}(undef, size(post, 2)), Vector{Float64}(undef, size(post, 2))
    GC.@preserve post ess rhat check(ccall((:erirt_ess_rhat, LIB), Cint,
        (Ptr{Float64}, Int64, Int64, Int64, Int64, Int32, Ptr{Float64}, Ptr{Float64}),
        post, size(post, 1), size(post, 2), size(post, 3), skip, device, ess, rhat))
    return ess, rhat
end
# the same on the traces of a live handle, without copying them to the host: columns first_col+1 ... first_col+ncols of Post.<which>
function ess_rhat_gpu(h::Ptr{Cvoid}, which::Integer, first_col::Integer, ncols::Integer; skip::Integer=0)
    ess, rhat = Vector{Float64}(undef, ncols), Vector{Float64}(undef, ncols)
    GC.@preserve ess rhat check(ccall((:erirt_trace_ess_rhat, LIB), Cint,
        (Ptr{Cvoid}, Int32, Int64, Int64, Int64, Ptr{Float64}, Ptr{Float64}), h, which, first_col, ncols, skip, ess, rhat))
    return ess, rhat
end
"""
    checkConvergence(MCMC; device=0)

src/SimTools.jl:419-443 with the ESS / R-hat of every traced column computed on the GPU: share of the columns of Post.ra / rt / qr
(after nBurnin) with ESS > 400 and R-hat < 1.1.
"""
function checkConvergence_gpu(MCMC; device::Integer=0)
    nb = MCMC.Cond.nBurnin
    essOk = rhatOk = n = 0
    for post in (MCMC.Post.ra, MCMC.Post.rt, MCMC.Post.qr)
        (post === nothing || isempty(post)) && continue
        ess, rhat = ess_rhat_gpu(Array{Float64,3}(post); skip=nb, device=device)
        keep = .!isnan.(ess)
        n += count(keep)
        essOk += count(ess[keep] .> 400)
        rhatOk += count(rhat[keep] .< 1.1)
    end
    return (ess=100 * essOk / max(n, 1), rhat=100 * rhatOk / max(n, 1), essN="$(essOk) / $(n)", rhatN="$(rhatOk) / $(n)")
end

end # module
