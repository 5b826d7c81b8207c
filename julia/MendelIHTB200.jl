# MendelIHTB200.jl — Julia shim that routes MendelIHT's IHT hot path to libihtb200.so through ccall.
#
# NOT EXECUTED IN THIS REPOSITORY'S CI: Julia is not installed in the build image.  The Python mirror
# (mendeliht.jl_b200/api.py) binds the very same C entry points and is what the tests run; this file shows the
# reference-side binding a maintainer adds (see INTEGRATION.md).  Entry points: include/ihtb200.h.
module MendelIHTB200

using MendelIHT, SnpArrays, Distributions, GLM, LinearAlgebra
import MendelIHT: fit_iht, cv_iht, IHTResult, pve

const LIB = get(ENV, "IHTB200_LIB", "libihtb200")

# ---- status codes -> the exception types the reference throws -------------------------------------------------
function last_error()
    buf = Vector{UInt8}(undef, 1024)
    ccall((:ihtb_last_error, LIB), Int32, (Ptr{UInt8}, Int64), buf, 1024)
    unsafe_string(pointer(buf))
end
function check(status::Int32)
    status == 0 && return
    msg = last_error()
    status == -1 && throw(ArgumentError(msg))          # @assert / ArgumentError (src/fit.jl:87-90)
    status == -2 && throw(DimensionMismatch(msg))      # src/data_structures.jl:63-85
    status == -3 && throw(DomainError(msg))            # src/utilities.jl:554
    status == -4 && error(msg)                         # "Loglikelihood function is NaN, aborting..." (src/fit.jl:259)
    error("libihtb200: $msg (status $status)")
end

# ---- SnpLinAlg replacement -------------------------------------------------------------------------------------
"Device-resident genotype operator; drop-in for `SnpLinAlg{Float64}(s; center, scale, impute)` (src/wrapper.jl:68)."
mutable struct B200SnpLinAlg <: AbstractMatrix{Float64}
    handle::Ptr{Cvoid}
    n::Int
    p::Int
    center::Bool
    scale::Bool
    impute::Bool
    function B200SnpLinAlg(s::SnpArray; model=ADDITIVE_MODEL, center::Bool=true, scale::Bool=true, impute::Bool=true)
        model == ADDITIVE_MODEL || error("only ADDITIVE_MODEL is supported")
        n, p = size(s)
        h = Ref{Ptr{Cvoid}}(C_NULL)
        # s.data is the mmapped packed matrix, ceil(n/4) x p bytes, SNP-major: exactly bed_cols
        check(ccall((:ihtb_geno_create, LIB), Int32,
                    (Ptr{UInt8}, Int64, Int64, Int64, Int32, Int32, Int32, Ref{Ptr{Cvoid}}),
                    s.data, n, p, size(s.data, 1), center, scale, impute, h))
        x = new(h[], n, p, center, scale, impute)
        finalizer(x -> ccall((:ihtb_geno_destroy, LIB), Int32, (Ptr{Cvoid},), x.handle), x)
        return x
    end
end
Base.size(x::B200SnpLinAlg) = (x.n, x.p)
function Base.getindex(x::B200SnpLinAlg, i::Int, j::Int)    # bit-exact with SnpLinAlg getindex (src/utilities.jl:102)
    out = Ref{Float64}(0.0)
    check(ccall((:ihtb_geno_decode, LIB), Int32, (Ptr{Cvoid}, Int64, Int64, Int64, Int64, Ref{Float64}),
                x.handle, i - 1, i, j - 1, j, out))
    out[]
end
"mul!(out, Transpose(x), v)  (src/utilities.jl:133, src/multivariate.jl:85)"
function LinearAlgebra.mul!(out::AbstractVecOrMat{Float64}, xt::Transpose{Float64,B200SnpLinAlg},
                            v::AbstractVecOrMat{Float64})
    x = xt.parent
    check(ccall((:ihtb_xt_v, LIB), Int32, (Ptr{Cvoid}, Ptr{Float64}, Int64, Ptr{Float64}, Int32),
                x.handle, v, size(v, 2), out, 1))       # 1 = IHTB_SWEEP_EXACT for stand-alone products
    out
end

# ---- several GPUs driven by this Julia process (include/ihtb200.h, ihtb_mgeno) -----------------------------------
"""
    B200MultiSnpLinAlg(s::SnpArray; ngpu, mode = :shard, devices = nothing)

The genotype operator over `ngpu` GPUs of the box.  `mode = :shard` splits the SNP columns over the devices and
`fit_iht` runs ONE fit over all of them (X*beta partials all-reduced and top-k candidates all-gathered by peer-memory
kernels over NVLink inside the library); `mode = :replicate` puts the whole matrix on every device and `cv_iht` farms
its (fold, k) grid over them -- the GPU counterpart of the reference's `Threads.@threads` loop
(src/cross_validation.jl:98-121).  No torchrun, no second process: one `ccall` per API call.
"""
mutable struct B200MultiSnpLinAlg <: AbstractMatrix{Float64}
    handle::Ptr{Cvoid}
    n::Int
    p::Int
    ngpu::Int
    mode::Symbol
    function B200MultiSnpLinAlg(s::SnpArray; ngpu::Int, mode::Symbol=:shard, devices::Union{Nothing,Vector{Int}}=nothing,
                                center::Bool=true, scale::Bool=true, impute::Bool=true)
        mode in (:shard, :replicate) || throw(ArgumentError("mode must be :shard or :replicate"))
        n, p = size(s)
        h = Ref{Ptr{Cvoid}}(C_NULL)
        devs = devices === nothing ? C_NULL : Int32.(devices)
        check(ccall((:ihtb_mgeno_create, LIB), Int32,
                    (Ptr{UInt8}, Int64, Int64, Int64, Int32, Int32, Int32, Int32, Ptr{Int32}, Int32, Ref{Ptr{Cvoid}}),
                    s.data, n, p, size(s.data, 1), center, scale, impute, ngpu, devs, mode == :shard ? 0 : 1, h))
        x = new(h[], n, p, ngpu, mode)
        finalizer(x -> ccall((:ihtb_mgeno_destroy, LIB), Int32, (Ptr{Cvoid},), x.handle), x)
        return x
    end
end
Base.size(x::B200MultiSnpLinAlg) = (x.n, x.p)

# ---- dense design matrix (include/ihtb200.h ihtb_geno_create_dense) ----------------------------------------------
"""Device-resident dense predictors: `fit_iht(y, x::AbstractMatrix{T}, z)` (src/fit.jl:62) for T = Float64 / Float32,
e.g. the dosages `convert_gt` / `convert_bgen_gt` produce (src/wrapper.jl:406-485).  `standardize = true` runs
`standardize_genotypes!` on the device (NaN = missing).  Stored as T, computed on in Float64; univariate fits only.

`dosage_denominator = D` (Float64 input, 1 <= D <= 65534): dosages on the grid 1/D (PLINK 2: 16384, VCF DS with d
decimals: 10^d, BGEN 8-bit: 255) are stored losslessly as 16-bit codes c = round(x D), 2 bytes per entry; every entry
must satisfy 0 <= c <= 65534 and c / D == x (ArgumentError otherwise), NaN is missing with `standardize = true`.  Results
equal those of the Float64 storage of the same values (include/ihtb200.h ihtb_geno_create_dosage16)."""
mutable struct B200DenseLinAlg{T<:Union{Float32,Float64}} <: AbstractMatrix{T}
    handle::Ptr{Cvoid}
    n::Int
    p::Int
    function B200DenseLinAlg(x::Matrix{T}; standardize::Bool=false,
                             dosage_denominator::Union{Nothing,Integer}=nothing) where {T<:Union{Float32,Float64}}
        n, p = size(x)
        h = Ref{Ptr{Cvoid}}(C_NULL)
        if dosage_denominator === nothing
            check(ccall((:ihtb_geno_create_dense, LIB), Int32,
                        (Ptr{Cvoid}, Int32, Int64, Int64, Int64, Int32, Ref{Ptr{Cvoid}}),
                        x, T === Float32 ? 1 : 0, n, p, n, standardize, h))
        else
            codes = encode_dosages(x, dosage_denominator, standardize)
            check(ccall((:ihtb_geno_create_dosage16, LIB), Int32,
                        (Ptr{UInt16}, Int64, Int64, Int64, Int32, Int32, Ref{Ptr{Cvoid}}),
                        codes, n, p, n, dosage_denominator, standardize, h))
        end
        g = new{T}(h[], n, p)
        finalizer(g -> ccall((:ihtb_geno_destroy, LIB), Int32, (Ptr{Cvoid},), g.handle), g)
        return g
    end
end
Base.size(x::B200DenseLinAlg) = (x.n, x.p)

# codes c = round(x D) of dosages on the grid 1/D; the first entry (column-major) that is not c / D names the error
function encode_dosages(x::Matrix{T}, D::Integer, standardize::Bool) where {T}
    T === Float64 || throw(ArgumentError("dosage codes need Float64 input"))
    1 <= D <= 65534 || throw(ArgumentError("dosage_denominator must be in [1, 65534], got $D"))
    codes = Matrix{UInt16}(undef, size(x))
    @inbounds for j in axes(x, 2), i in axes(x, 1)
        v = x[i, j]
        if isnan(v)
            standardize || throw(DomainError(v, "x[$i, $j] is NaN: missing dosages need standardize = true"))
            codes[i, j] = 0xffff
            continue
        end
        c = round(v * D)
        (0 <= c <= 65534 && c / D == v) ||
            throw(ArgumentError("x[$i, $j] = $v is not a dosage c / $D with an integer 0 <= c <= 65534"))
        codes[i, j] = UInt16(c)
    end
    codes
end
function Base.getindex(x::B200DenseLinAlg{T}, i::Int, j::Int) where {T}     # the stored value
    out = Ref{Float64}(0.0)
    check(ccall((:ihtb_geno_decode, LIB), Int32, (Ptr{Cvoid}, Int64, Int64, Int64, Int64, Ref{Float64}),
                x.handle, i - 1, i, j - 1, j, out))
    T(out[])
end
function LinearAlgebra.mul!(out::AbstractVecOrMat{Float64}, xt::Transpose{<:Any,<:B200DenseLinAlg},
                            v::AbstractVecOrMat{Float64})
    check(ccall((:ihtb_xt_v, LIB), Int32, (Ptr{Cvoid}, Ptr{Float64}, Int64, Ptr{Float64}, Int32),
                xt.parent.handle, v, size(v, 2), out, 1))
    out
end

const AnyB200 = Union{B200SnpLinAlg,B200MultiSnpLinAlg,B200DenseLinAlg}
# the single-device and the multi-device calls have the same argument lists (ihtb_fit_* / ihtb_mfit_*)
fitsym(::Union{B200SnpLinAlg,B200DenseLinAlg}, name::Symbol) = Symbol(:ihtb_fit_, name)
fitsym(::B200MultiSnpLinAlg, name::Symbol) = Symbol(:ihtb_mfit_, name)
mvsym(::B200SnpLinAlg, name::Symbol) = Symbol(:ihtb_mvfit_, name)          # multivariate: ihtb_mvfit_* / ihtb_mmvfit_*
mvsym(::B200MultiSnpLinAlg, name::Symbol) = Symbol(:ihtb_mmvfit_, name)

# ---- fit_iht on the device -----------------------------------------------------------------------------------
struct Cfg
    dist::Int32; link::Int32; k::Int64; nb_r::Float64; tol::Float64
    max_iter::Int32; min_iter::Int32; max_step::Int32; sweep_mode::Int32; est_r::Int32; debias::Int32
end
mutable struct CResult
    time::Float64; logl::Float64; iter::Int64; sigma_g::Float64; n_sweeps::Int64; n_backtracks::Int64
    sweep_seconds::Float64; n_launches::Int64; n_steps::Int64
    CResult() = new(0, 0, 0, 0, 0, 0, 0, 0, 0)
end
struct CIterTrace        # one line of the verbose trace (include/ihtb200.h ihtb_iter_trace)
    logl::Float64; tol::Float64; eta::Float64; backtracks::Int32; n_candidates::Int32
end
# keywords of the reference that this path does not implement must fail loudly, not be swallowed by kwargs...
reject_unknown(kw) = isempty(kw) || throw(ArgumentError("unsupported keyword(s) for the B200 path: $(collect(keys(kw)))"))
distcode(::Normal) = Int32(0); distcode(::Bernoulli) = Int32(1); distcode(::Poisson) = Int32(2)
distcode(::NegativeBinomial) = Int32(3)
linkcode(::IdentityLink) = Int32(0); linkcode(::LogitLink) = Int32(1); linkcode(::LogLink) = Int32(2)
linkcode(::ProbitLink) = Int32(3); linkcode(::CloglogLink) = Int32(4); linkcode(::CauchitLink) = Int32(5)
linkcode(::SqrtLink) = Int32(6); linkcode(::InverseLink) = Int32(7); linkcode(::InverseSquareLink) = Int32(8)

"SnpArrays.maf / MendelIHT.maf_weights (src/utilities.jl:692-697) from the device-side allele counts."
function maf(x::B200SnpLinAlg)
    out = Vector{Float64}(undef, x.p)
    check(ccall((:ihtb_geno_maf, LIB), Int32, (Ptr{Cvoid}, Ptr{Float64}), x.handle, out))
    out
end
function MendelIHT.maf_weights(x::B200SnpLinAlg; max_weight::Float64=Inf)
    p = maf(x)
    clamp!(p .= 1 ./ (2 .* sqrt.(p .* (1 .- p))), 1.0, max_weight)
end

# weight / group / per-group k are attached to the fit handle before ihtb_fit_init
function attach_options(x::AnyB200, fh, p::Int, k::Union{Int,Vector{Int}}, J::Int, group::AbstractVector{Int},
                        weight::AbstractVector{Float64})
    if length(group) > 0
        length(group) == p || throw(DimensionMismatch("group must have length $p but was $(length(group))"))
        ks = k isa Vector ? Int64.(k) : Int64[]
        check(ccall((fitsym(x, :set_groups), LIB), Int32, (Ptr{Cvoid}, Ptr{Int32}, Int32, Ptr{Int64}, Int64),
                    fh, Int32.(group), J, k isa Vector ? ks : C_NULL, length(ks)))
    end
    if length(weight) > 0
        length(weight) == p || throw(DimensionMismatch("weight must have length $p but was $(length(weight))"))
        check(ccall((fitsym(x, :set_weights), LIB), Int32, (Ptr{Cvoid}, Ptr{Float64}), fh, weight))
    end
end
function fit_init(x::Union{B200SnpLinAlg,B200DenseLinAlg}, fh, mask, init_beta::Bool)
    check(ccall((init_beta ? :ihtb_fit_init_beta : :ihtb_fit_init, LIB), Int32, (Ptr{Cvoid}, Ptr{UInt8}), fh, mask))
end
function fit_init(x::B200MultiSnpLinAlg, fh, mask, init_beta::Bool)
    check(ccall((:ihtb_mfit_init, LIB), Int32, (Ptr{Cvoid}, Ptr{UInt8}, Int32), fh, mask, init_beta))
end

"""
Same signature and return type as MendelIHT.fit_iht (src/fit.jl:60-118) for `x::B200SnpLinAlg`, or for a
`B200MultiSnpLinAlg` in `:shard` mode (one fit over several GPUs).  `verbose` / `io` print the reference's
per-iteration line (src/fit.jl:194-196) from the trace the library records.
"""
function fit_iht(y::AbstractVector{Float64}, x::AnyB200, z::AbstractVecOrMat{Float64};
                 k::Union{Int,Vector{Int}}=10, J::Int=1, d::Distribution=Normal(), l::Link=IdentityLink(),
                 group::AbstractVector{Int}=Int[], weight::AbstractVector{Float64}=Float64[],
                 zkeep::BitVector=trues(size(z, 2)), est_r::Symbol=:None, debias::Bool=false, init_beta::Bool=false,
                 use_maf::Bool=false, tol::Float64=1e-4, max_iter::Int=200,
                 min_iter::Int=5, max_step::Int=3, verbose::Bool=false, io::IO=stdout, kwargs...)
    reject_unknown(kwargs)
    est = est_r == :None ? Int32(0) : est_r == :MM ? Int32(1) : est_r == :Newton ? Int32(2) :
          throw(ArgumentError("Only support method is Newton or MM, but got $est_r"))
    x isa B200SnpLinAlg && !x.center &&
        error("x is not centered! Please construct SnpLinAlg{Float64}(::SnpArray, center=true, scale=true)")
    x isa B200MultiSnpLinAlg && x.mode != :shard && throw(ArgumentError("fit_iht over several GPUs needs mode = :shard"))
    zm = z isa AbstractVector ? reshape(z, :, 1) : Matrix(z)
    r = d isa NegativeBinomial ? d.r : 1.0
    MendelIHT.check_group(k, group)                                       # src/utilities.jl:902-915
    kscalar = k isa Vector ? 0 : k                                         # src/data_structures.jl:75-81
    cfg = Ref(Cfg(distcode(d), linkcode(l), kscalar, r, tol, max_iter, min_iter, max_step, 0, est, debias))
    fh = Ref{Ptr{Cvoid}}(C_NULL)
    keep = UInt8.(zkeep)
    check(ccall((fitsym(x, :create), LIB), Int32,
                (Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}, Int64, Ptr{UInt8}, Ref{Cfg}, Ref{Ptr{Cvoid}}),
                x.handle, y, zm, size(zm, 2), keep, cfg, fh))
    try
        attach_options(x, fh[], x.p, k, J, group, weight)
        fit_init(x, fh[], C_NULL, init_beta)
        res = CResult()
        trace = Vector{CIterTrace}(undef, verbose ? max_iter : 0)
        check(ccall((fitsym(x, :run), LIB), Int32, (Ptr{Cvoid}, Ref{CResult}, Ptr{CIterTrace}, Int64),
                    fh[], res, verbose ? trace : C_NULL, length(trace)))
        if verbose                                                         # src/fit.jl:194-196
            for i in 1:min(res.n_steps, length(trace))
                t = trace[i]
                println(io, "Iteration $i: loglikelihood = $(t.logl), backtracks = $(t.backtracks), tol = $(t.tol)")
            end
        end
        beta = zeros(x.p); c = zeros(size(zm, 2))
        check(ccall((fitsym(x, :get), LIB), Int32, (Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}),
                    fh[], beta, c, C_NULL, C_NULL))
        return IHTResult(res.time, res.logl, res.iter, beta, c, J, k, collect(group), d, res.sigma_g)
    finally
        ccall((fitsym(x, :destroy), LIB), Int32, (Ptr{Cvoid},), fh[])
    end
end

"""
Multivariate (MvNormal) fit: same call as the reference, `fit_iht(Y, Transpose(xla), Z; k)` with Y r x n and Z q x n
(src/fit.jl:60-118, src/multivariate.jl); returns `mIHTResult`.  The library wants samples as rows (n x r, n x q).
"""
function fit_iht(Y::AbstractMatrix{Float64}, xt::Transpose{Float64,<:AnyB200}, Z::AbstractVecOrMat{Float64};
                 k::Int=10, zkeep::BitVector=trues(size(Z, 1)), init_beta::Bool=false, debias::Bool=false,
                 tol::Float64=1e-4, max_iter::Int=200, min_iter::Int=5, max_step::Int=3, verbose::Bool=false,
                 io::IO=stdout, kwargs...)
    reject_unknown(kwargs)            # J / group / weight do not exist for MvNormal in the reference either
    debias && error("Currently the debiasing routine for multivariate IHT is broken, sorry!")   # src/multivariate.jl:570
    x = xt.parent
    r, n = size(Y)
    Zm = Z isa AbstractVector ? reshape(Z, 1, :) : Matrix(Z)
    q = size(Zm, 1)
    (n == x.n == size(Zm, 2)) || throw(DimensionMismatch("number of samples in y, x, and z = $n, $(x.n), $(size(Zm, 2)) are not equal"))
    all(zkeep) || error("multivariate zkeep with false entries is not supported")
    Yc = Matrix(transpose(Y)); Zc = Matrix(transpose(Zm))                  # n x r, n x q column-major
    # sweep_mode 2 = IHTB_SWEEP_PAIR: the skinny X'R reads the matrix once per two traits (src/multivariate.jl:85)
    cfg = Ref(Cfg(0, 0, k, 1.0, tol, max_iter, min_iter, max_step, 2, 0, 0))
    fh = Ref{Ptr{Cvoid}}(C_NULL)
    check(ccall((mvsym(x, :create), LIB), Int32,
                (Ptr{Cvoid}, Ptr{Float64}, Int64, Ptr{Float64}, Int64, Ref{Cfg}, Ref{Ptr{Cvoid}}),
                x.handle, Yc, r, Zc, q, cfg, fh))
    try
        if x isa B200MultiSnpLinAlg
            check(ccall((:ihtb_mmvfit_init, LIB), Int32, (Ptr{Cvoid}, Ptr{UInt8}, Int32), fh[], C_NULL, init_beta ? 1 : 0))
        else
            check(ccall((init_beta ? :ihtb_mvfit_init_beta : :ihtb_mvfit_init, LIB), Int32, (Ptr{Cvoid}, Ptr{UInt8}), fh[], C_NULL))
        end
        res = CResult()
        trace = Vector{CIterTrace}(undef, verbose ? max_iter : 0)
        check(ccall((mvsym(x, :run), LIB), Int32, (Ptr{Cvoid}, Ref{CResult}, Ptr{CIterTrace}, Int64),
                    fh[], res, verbose ? trace : C_NULL, length(trace)))
        if verbose
            for i in 1:min(res.n_steps, length(trace))
                t = trace[i]
                println(io, "Iteration $i: loglikelihood = $(t.logl), backtracks = $(t.backtracks), tol = $(t.tol)")
            end
        end
        B = zeros(r, x.p); C = zeros(r, q); Σ = zeros(r, r); σg = zeros(r)
        check(ccall((mvsym(x, :get), LIB), Int32, (Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}),
                    fh[], B, C, Σ, σg))
        return MendelIHT.mIHTResult(res.time, res.logl, res.iter, B, C, k, r, Σ, σg)   # field order: src/data_structures.jl:263-273
    finally
        ccall((mvsym(x, :destroy), LIB), Int32, (Ptr{Cvoid},), fh[])
    end
end

"""
cv_iht (src/cross_validation.jl:60-131).  The plain grid is ONE library call: `ihtb_cv_run` on one GPU,
`ihtb_mcv_run` over the replicas of a `B200MultiSnpLinAlg(...; mode = :replicate)` (shared work queue, largest k
first).  Groups, `init_beta` and `est_r` take the per-fit loop on one device, where the NegativeBinomial estimate is
carried from fit to fit like the reference's per-thread `IHTVariable` (src/cross_validation.jl:105).
"""
function cv_iht(y::AbstractVector{Float64}, x::AnyB200, z::AbstractVecOrMat{Float64};
                d::Distribution=Normal(), l::Link=IdentityLink(), path::AbstractVector{<:Integer}=1:20, q::Int=5,
                folds::AbstractVector{Int}=rand(1:q, size(x, 1)), zkeep::BitVector=trues(size(z, 2)),
                J::Int=1, group::AbstractVector{Int}=Int[], weight::AbstractVector{Float64}=Float64[],
                est_r::Symbol=:None, debias::Bool=false, init_beta::Bool=false, tol::Float64=1e-4,
                max_iter::Int=100, min_iter::Int=5, max_step::Int=3, verbose::Bool=false, kwargs...)
    reject_unknown(kwargs)
    maximum(path) > size(x, 2) && error("Sparsity level in `path` cannot be larger than total number of variables")
    zm = z isa AbstractVector ? reshape(z, :, 1) : Matrix(z)
    r = d isa NegativeBinomial ? d.r : 1.0
    est = est_r == :None ? Int32(0) : est_r == :MM ? Int32(1) : est_r == :Newton ? Int32(2) :
          throw(ArgumentError("Only support method is Newton or MM, but got $est_r"))
    cfg = Ref(Cfg(distcode(d), linkcode(l), maximum(path), r, tol, max_iter, min_iter, max_step, 0, est, debias))
    combos = MendelIHT.allocate_fold_and_k(q, path)
    mses = zeros(length(combos))
    pathv = Int64.(collect(path)); foldv = Int32.(folds)
    w = length(weight) > 0 ? weight : C_NULL
    if length(group) == 0 && !init_beta
        if x isa B200MultiSnpLinAlg
            x.mode == :replicate || throw(ArgumentError("cv_iht over several GPUs needs mode = :replicate"))
            check(ccall((:ihtb_mcv_run, LIB), Int32,
                        (Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}, Int64, Ptr{UInt8}, Ref{Cfg}, Ptr{Int32}, Int32, Ptr{Int64},
                         Int64, Ptr{Float64}, Ptr{Float64}, Ptr{Int64}, Ptr{Float64}),
                        x.handle, y, zm, size(zm, 2), UInt8.(zkeep), cfg, foldv, q, pathv, length(pathv), w, mses, C_NULL, C_NULL))
        else
            check(ccall((:ihtb_cv_run, LIB), Int32,
                        (Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}, Int64, Ptr{UInt8}, Ref{Cfg}, Ptr{Int32}, Int32, Ptr{Int64},
                         Int64, Ptr{Float64}, Ptr{Float64}, Ptr{Int64}),
                        x.handle, y, zm, size(zm, 2), UInt8.(zkeep), cfg, foldv, q, pathv, length(pathv), w, mses, C_NULL))
        end
        return MendelIHT.meanloss(mses, q, folds)
    end
    x isa Union{B200SnpLinAlg,B200DenseLinAlg} ||
        throw(ArgumentError("group / init_beta cross-validation runs on a single-device operator"))
    fh = Ref{Ptr{Cvoid}}(C_NULL)
    check(ccall((:ihtb_fit_create, LIB), Int32,
                (Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}, Int64, Ptr{UInt8}, Ref{Cfg}, Ref{Ptr{Cvoid}}),
                x.handle, y, zm, size(zm, 2), UInt8.(zkeep), cfg, fh))
    try
        attach_options(x, fh[], x.p, maximum(path), J, group, weight)
        for (i, (fold, k)) in enumerate(combos)
            test = UInt8.(folds .== fold); train = UInt8.(folds .!= fold)
            check(ccall((:ihtb_fit_set_k, LIB), Int32, (Ptr{Cvoid}, Int64), fh[], k))
            fit_init(x, fh[], train, init_beta)
            check(ccall((:ihtb_fit_run, LIB), Int32, (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Cvoid}, Int64), fh[], C_NULL, C_NULL, 0))
            dev = Ref{Float64}(0.0)
            check(ccall((:ihtb_fit_predict, LIB), Int32, (Ptr{Cvoid}, Ptr{UInt8}, Ref{Float64}), fh[], test, dev))
            mses[i] = dev[]
        end
    finally
        ccall((:ihtb_fit_destroy, LIB), Int32, (Ptr{Cvoid},), fh[])
    end
    return MendelIHT.meanloss(mses, q, folds)
end

end # module
