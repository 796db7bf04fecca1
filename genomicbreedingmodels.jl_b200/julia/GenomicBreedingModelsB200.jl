# GenomicBreedingModelsB200.jl -- Julia shim over libgbm_b200.so (include/gbm_b200.h).
#
# Drop-in for the GWAS hot path of GenomicBreedingModels.jl v0.3.0: same function names,
# keyword arguments, return types and exceptions as
#     gwasprep  src/gwas.jl:77-142      gwasols  src/gwas.jl:206-259      gwaslmm  src/gwas.jl:329-399
# and GenomicBreedingCore's grmsimple / grmploidyaware (call sites src/gwas.jl:120, :124).
# Genomes / Phenomes in, Fit out.  One blocking `ccall` per phase from one Julia thread; the
# library never calls back into Julia and never keeps a host pointer after it returns.
#
# NOT EXECUTED IN THE BUILD IMAGE (no Julia there): the Python ctypes harness
# (../gbm_b200) binds the same symbols with the same call sequence and is what the tests run.
module GenomicBreedingModelsB200

using GenomicBreedingCore
using Statistics

export gwasprep, gwasols, gwaslmm, gwasreml, grmsimple_b200, grmploidyaware_b200
export transform1, transform2, epistasisfeatures, square, invoneplus, log10epsdivlog10eps, mult, addnorm, raise

const LIBGBM = get(ENV, "GBM_B200_LIB", joinpath(@__DIR__, "..", "libgbm_b200.so"))

const GBM_OK = Cint(0)
const GBM_ERR_ARGUMENT = Cint(1)
const GBM_ERR_RUNTIME = Cint(2)
const GBM_GRM_SIMPLE = Cint(0)
const GBM_GRM_PLOIDY_AWARE = Cint(1)
const GBM_MODEL_OLS = Cint(0)
const GBM_MODEL_LMM = Cint(1)

function check(code::Cint)
    code == GBM_OK && return nothing
    msg = unsafe_string(ccall((:gbm_last_error, LIBGBM), Cstring, ()))
    code == GBM_ERR_ARGUMENT && throw(ArgumentError(msg))
    throw(ErrorException(msg))
end

const INITIALISED = Ref(false)
function init(device::Integer = parse(Int, get(ENV, "GBM_DEVICE", "0")))
    if !INITIALISED[]
        check(ccall((:gbm_init, LIBGBM), Cint, (Cint,), device))
        INITIALISED[] = true
    end
    nothing
end

# ---- device matrix handle (library-owned HBM, freed by finalizer) --------------------
mutable struct DeviceMatrix
    handle::Ptr{Cvoid}
    n::Int64
    p::Int64
    function DeviceMatrix(h::Ptr{Cvoid}, n, p)
        m = new(h, n, p)
        finalizer(free!, m)
        m
    end
end
function free!(m::DeviceMatrix)
    if m.handle != C_NULL
        ccall((:gbm_matrix_free, LIBGBM), Cint, (Ptr{Cvoid},), m.handle)
        m.handle = C_NULL
    end
    nothing
end

# G = genomes.allele_frequencies[rows, cols]  (src/prediction.jl:129) without the host copy
function upload(A::Matrix{Float64}, rows::Union{Nothing,Vector{Int64}}, cols::Union{Nothing,Vector{Int64}})
    init()
    h = Ref{Ptr{Cvoid}}(C_NULL)
    n0, p0 = size(A)
    if isnothing(rows) && isnothing(cols)
        # the host cores pack dosage data to one byte per genotype on the way (exactness-checked); anything
        # else arrives as Float64, staged through pinned memory by the same cores (a Julia Array is pageable)
        packed = Ref{Cint}(0)
        check(ccall((:gbm_matrix_upload_compact, LIBGBM), Cint,
                    (Ptr{Float64}, Int64, Int64, Int64, Ref{Ptr{Cvoid}}, Ref{Cint}), A, n0, p0, n0, h, packed))
        return DeviceMatrix(h[], n0, p0)
    end
    n = isnothing(rows) ? n0 : length(rows)
    p = isnothing(cols) ? p0 : length(cols)
    check(ccall((:gbm_matrix_upload_indexed, LIBGBM), Cint,
                (Ptr{Float64}, Int64, Int64, Int64, Ptr{Int64}, Int64, Ptr{Int64}, Int64, Ref{Ptr{Cvoid}}),
                A, n0, p0, n0, isnothing(rows) ? C_NULL : rows, n,   # arrays, not pointer(...): ccall roots them
                isnothing(cols) ? C_NULL : cols, p, h))
    DeviceMatrix(h[], n, p)
end

function colstats(m::DeviceMatrix)
    mean = Vector{Float64}(undef, m.p); sd = similar(mean); mnz = similar(mean)
    keep = Vector{UInt8}(undef, m.p); idx = Vector{Int64}(undef, m.p)
    nk = Ref{Int64}(0); mk = Ref{Float64}(0.0)
    check(ccall((:gbm_colstats, LIBGBM), Cint,
                (Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{UInt8}, Ptr{Int64}, Ref{Int64}, Ref{Float64}),
                m.handle, mean, sd, mnz, keep, idx, nk, mk))
    (mean = mean, sd = sd, idx_cols = idx[1:nk[]], min_nonzero_kept = mk[])
end

function grm(m::DeviceMatrix, grm_type::Cint, ploidy::Integer; flags::Integer = 0)
    K = Matrix{Float64}(undef, m.n, m.n)
    tf = Ref{Float64}(0.0)
    check(ccall((:gbm_grm, LIBGBM), Cint, (Ptr{Cvoid}, Cint, Cint, Cint, Ptr{Float64}, Ref{Float64}),
                m.handle, grm_type, ploidy, flags, K, tf))
    K
end

function kstd_pc1(K::Matrix{Float64}; want_kstd::Bool = true, want_pc1::Bool = true)
    n = size(K, 1)
    Ks = want_kstd ? Matrix{Float64}(undef, n, n) : nothing
    pc = want_pc1 ? Vector{Float64}(undef, n) : nothing
    ms = Ref{Float64}(0.0)
    check(ccall((:gbm_kstd_pc1, LIBGBM), Cint, (Ptr{Float64}, Int64, Ptr{Float64}, Ptr{Float64}, Ref{Float64}),
                K, n, want_kstd ? Ks : C_NULL, want_pc1 ? pc : C_NULL, ms))
    (Ks, pc)
end

function scan(m::DeviceMatrix, y::Vector{Float64}, pc::Vector{Float64}, model::Cint)
    stat = Vector{Float64}(undef, m.p); beta = similar(stat); se = similar(stat); nlp = similar(stat)
    check(ccall((:gbm_scan, LIBGBM), Cint,
                (Ptr{Cvoid}, Ptr{Float64}, Int64, Int64, Ptr{Float64}, Int64, Int64, Cint, Cint, Ptr{Float64},
                 Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{UInt8}),
                m.handle, y, 1, m.n, pc, 1, m.n, model, 0, beta, se, stat, nlp, C_NULL, C_NULL, C_NULL))
    (stat = stat, beta = beta, se = se, neglog10p = nlp)
end

# ---- the reference's row filter and validation (src/prediction.jl:67-127), host side ----
function selectrows(genomes::Genomes, phenomes::Phenomes, idx_entries, idx_loci_alleles, idx_trait::Int64)
    if !checkdims(genomes) && !checkdims(phenomes)
        throw(ArgumentError("The Genomes and Phenomes structs are corrupted ☹."))
    end
    !checkdims(genomes) && throw(ArgumentError("The Genomes struct is corrupted ☹."))
    !checkdims(phenomes) && throw(ArgumentError("The Phenomes struct is corrupted ☹."))
    if genomes.entries != phenomes.entries
        throw(ArgumentError("The genomes and phenomes input need to have been merged to have consitent entries."))
    end
    allrows = isnothing(idx_entries)
    idx_entries = allrows ? collect(1:length(genomes.entries)) : idx_entries
    if minimum(idx_entries) < 1 || maximum(idx_entries) > length(genomes.entries)
        throw(ArgumentError("The indexes of the entries, `idx_entries` are out of bounds."))
    end
    if !isnothing(idx_loci_alleles) &&
       (minimum(idx_loci_alleles) < 1 || maximum(idx_loci_alleles) > length(genomes.loci_alleles))
        throw(ArgumentError("The indexes of the loci_alleles, `idx_loci_alleles` are out of bounds."))
    end
    ϕ = phenomes.phenotypes[idx_entries, idx_trait]
    idx = findall(.!ismissing.(ϕ) .&& .!isnan.(ϕ) .&& .!isinf.(ϕ))
    if length(idx) < 2
        throw(ArgumentError("There are less than 2 entries with non-missing phenotype data after merging with the genotype data."))
    end
    y::Vector{Float64} = ϕ[idx]
    if var(y) < 1e-20
        throw(ErrorException("Very low or zero variance in trait: `" * phenomes.traits[idx_trait] * "`."))
    end
    rows = (allrows && length(idx) == length(idx_entries)) ? nothing : idx_entries[idx]
    (rows, idx_loci_alleles, y)
end

struct Prepared
    dm::DeviceMatrix
    y::Vector{Float64}
    K::Union{Nothing,Matrix{Float64}}
    pc1::Union{Nothing,Vector{Float64}}
    stats::NamedTuple
    entries::Vector{String}
    populations::Vector{String}
    loci_alleles::Vector{String}
    trait::String
end

function prepare(genomes, phenomes, idx_entries, idx_loci_alleles, idx_trait, GRM_type, standardise; need_kstd, need_pc1)
    rows, cols, y = selectrows(genomes, phenomes, idx_entries, idx_loci_alleles, idx_trait)   # src/gwas.jl:93-100
    if sum(["simple", "ploidy-aware"] .== GRM_type) == 0                                       # :101-107
        throw(ArgumentError("Unrecognised `GRM_type`. Please select from:\n\t‣ simple\n\t‣ ploidy-aware"))
    end
    var(y) < eps(Float64) && throw(ArgumentError("No variance in the trait: " * phenomes.traits[idx_trait] * "."))  # :109-111
    A = Matrix{Float64}(genomes.allele_frequencies)   # throws on `missing`, as src/prediction.jl:129 does
    dm = upload(A, rows, cols)
    stats = colstats(dm)                               # :112-113
    r = isnothing(rows) ? collect(1:size(A, 1)) : rows
    c = isnothing(cols) ? collect(1:size(A, 2)) : cols
    loci = genomes.loci_alleles[c][stats.idx_cols]     # :115
    full = (isnothing(rows) && isnothing(cols)) ? dm : upload(A, nothing, nothing)   # GRM on the FULL genomes (:120, :124)
    K = if GRM_type == "ploidy-aware"
        ploidy = Int(round(1 / stats.min_nonzero_kept))                              # :119
        grm(full, GBM_GRM_PLOIDY_AWARE, ploidy)
    else
        grm(full, GBM_GRM_SIMPLE, 2)
    end
    full === dm || free!(full)
    pc1 = nothing
    if standardise                                      # :127-131
        y = (y .- mean(y)) ./ std(y)
        Ks, pc1 = kstd_pc1(K; want_kstd = need_kstd, want_pc1 = need_pc1)
        K = Ks
    end
    Prepared(dm, y, K, pc1, stats, genomes.entries[r], genomes.populations[r], loci, phenomes.traits[idx_trait])
end

function newfit(pr::Prepared)::Fit
    n, l = length(pr.entries), length(pr.loci_alleles)
    fit = Fit(n = n, l = l)                              # src/gwas.jl:133-140
    fit.model = ""
    fit.trait = pr.trait
    fit.b_hat_labels = pr.loci_alleles
    fit.entries = pr.entries
    fit.populations = pr.populations
    fit.metrics = Dict("" => 0.0)
    fit
end

function gwasprep(;
    genomes::Genomes, phenomes::Phenomes,
    idx_entries::Union{Nothing,Vector{Int64}} = nothing, idx_loci_alleles::Union{Nothing,Vector{Int64}} = nothing,
    idx_trait::Int64 = 1, GRM_type::String = "simple", standardise::Bool = true, verbose::Bool = false,
)::Tuple{Matrix{Float64},Vector{Float64},Matrix{Float64},Fit}
    pr = prepare(genomes, phenomes, idx_entries, idx_loci_alleles, idx_trait, GRM_type, standardise; need_kstd = true, need_pc1 = false)
    # G = G[:, idx_cols]; G = (G .- mean(G, dims=1)) ./ v[idx_cols]'   (src/gwas.jl:114, :129), on the device
    l = length(pr.stats.idx_cols)
    G = Matrix{Float64}(undef, pr.dm.n, l)
    check(ccall((:gbm_matrix_download_cols, LIBGBM), Cint, (Ptr{Cvoid}, Ptr{Int64}, Int64, Cint, Ptr{Float64}, Int64),
                pr.dm.handle, pr.stats.idx_cols, l, standardise ? 1 : 0, G, pr.dm.n))
    fit = newfit(pr)
    free!(pr.dm)
    (G, pr.y, pr.K, fit)
end

# ---- multi-GPU: GBM_NUM_GPUS > 1 shards the markers over that many GPUs of this box -------------------
# The reference's parallel axis is `Threads.@threads for j = 1:l` (src/gwas.jl:239, :363); here this ONE Julia
# process drives a group of GPUs through the library (gbm_group_create_local: a host thread per GPU inside
# libgbm_b200.so, NCCL for the GRM all-reduce and the PC1 all-reduces, results gathered in locus order).
# Same calls, same Fit; applies when no entries / loci are subset (the reference's own working domain for
# gwasols / gwaslmm, since its GRM is always computed on the full `genomes`, src/gwas.jl:120, :124).
const GROUP = Ref{Ptr{Cvoid}}(C_NULL)
numgpus() = parse(Int, get(ENV, "GBM_NUM_GPUS", "1"))
function group()
    if GROUP[] == C_NULL
        g = Ref{Ptr{Cvoid}}(C_NULL)
        check(ccall((:gbm_group_create_local, LIBGBM), Cint, (Cint, Ptr{Cint}, Ref{Ptr{Cvoid}}), numgpus(), C_NULL, g))
        GROUP[] = g[]
        atexit(() -> ccall((:gbm_group_free, LIBGBM), Cint, (Ptr{Cvoid},), GROUP[]))
    end
    GROUP[]
end

struct GwasTiming   # gbm_gwas_timing of include/gbm_b200.h
    colstats_ms::Float64; grm_ms::Float64; allreduce_ms::Float64; kstd_pc1_ms::Float64; eig_ms::Float64
    scan_ms::Float64; gather_ms::Float64; total_ms::Float64; grm_tflops::Float64; scan_kernel_ms::Float64
    launches::Int64; ploidy::Int32; lanczos_steps::Int32
end

function gwas_multigpu(model_name::String, model::Cint, genomes, phenomes, idx_trait, GRM_type, y)::Fit
    A = Matrix{Float64}(genomes.allele_frequencies)       # throws on `missing`, as src/prediction.jl:129 does
    n, p = size(A)
    sm = Ref{Ptr{Cvoid}}(C_NULL); packed = Ref{Cint}(0)
    check(ccall((:gbm_sharded_upload, LIBGBM), Cint,
                (Ptr{Cvoid}, Ptr{Float64}, Int64, Int64, Int64, Cint, Ref{Ptr{Cvoid}}, Ref{Cint}), group(), A, n, p, n, 1, sm, packed))
    ys = (y .- mean(y)) ./ std(y)                         # src/gwas.jl:128
    stat = Vector{Float64}(undef, p); idx = Vector{Int64}(undef, p); nk = Ref{Int64}(0)
    tm = Ref{GwasTiming}()
    rc = ccall((:gbm_sharded_gwas, LIBGBM), Cint,
               (Ptr{Cvoid}, Ptr{Float64}, Cint, Cint, Cint, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64},
                Ptr{Float64}, Ptr{UInt8}, Ptr{Int64}, Ref{Int64}, Ptr{Float64}, Ref{GwasTiming}),
               sm[], ys, model, GRM_type == "ploidy-aware" ? GBM_GRM_PLOIDY_AWARE : GBM_GRM_SIMPLE, 0, stat, C_NULL, C_NULL,
               C_NULL, C_NULL, C_NULL, C_NULL, idx, nk, C_NULL, tm)
    ccall((:gbm_sharded_free, LIBGBM), Cint, (Ptr{Cvoid},), sm[])
    check(rc)
    idx_cols = idx[1:nk[]]
    fit = Fit(n = n, l = length(idx_cols))                # src/gwas.jl:133-140
    fit.model = model_name
    fit.trait = phenomes.traits[idx_trait]
    fit.b_hat_labels = genomes.loci_alleles[idx_cols]
    fit.entries = genomes.entries
    fit.populations = genomes.populations
    fit.metrics = Dict("" => 0.0)
    b = stat[idx_cols]
    model == GBM_MODEL_LMM && (b[isnan.(b)] .= 0.0)       # failed fits leave 0.0 (src/gwas.jl:367-382)
    fit.b_hat = b
    if !checkdims(fit)
        throw(ErrorException("Error performing GWAS using the " * GRM_type * " GRM."))
    end
    fit
end

function gwas(model_name::String, model::Cint, genomes, phenomes, idx_entries, idx_loci_alleles, idx_trait, GRM_type)::Fit
    if numgpus() > 1
        rows, cols, y = selectrows(genomes, phenomes, idx_entries, idx_loci_alleles, idx_trait)
        if sum(["simple", "ploidy-aware"] .== GRM_type) == 0
            throw(ArgumentError("Unrecognised `GRM_type`. Please select from:\n\t‣ simple\n\t‣ ploidy-aware"))
        end
        var(y) < eps(Float64) && throw(ArgumentError("No variance in the trait: " * phenomes.traits[idx_trait] * "."))
        if isnothing(rows) && isnothing(cols) && size(genomes.allele_frequencies, 2) >= numgpus()
            return gwas_multigpu(model_name, model, genomes, phenomes, idx_trait, GRM_type, y)
        end
    end
    pr = prepare(genomes, phenomes, idx_entries, idx_loci_alleles, idx_trait, GRM_type, true; need_kstd = false, need_pc1 = true)
    if length(pr.entries) != length(pr.pc1)
        free!(pr.dm)
        throw(ArgumentError("The GRM is computed on all entries of `genomes` but some entries were dropped: PC1 and G have different numbers of rows."))
    end
    fit = newfit(pr)
    fit.model = model_name                                # src/gwas.jl:231 / :354
    res = scan(pr.dm, pr.y, pr.pc1, model)                # marker loop, src/gwas.jl:239-249 / :363-389
    b = res.stat[pr.stats.idx_cols]
    if model == GBM_MODEL_LMM
        b[isnan.(b)] .= 0.0                               # failed fits leave 0.0 (src/gwas.jl:367-382)
    end
    fit.b_hat = b
    free!(pr.dm)
    if !checkdims(fit)                                    # src/gwas.jl:255-257 / :395-397
        throw(ErrorException("Error performing GWAS using the " * GRM_type * " GRM."))
    end
    fit
end

gwasols(; genomes::Genomes, phenomes::Phenomes, idx_entries::Union{Nothing,Vector{Int64}} = nothing,
    idx_loci_alleles::Union{Nothing,Vector{Int64}} = nothing, idx_trait::Int64 = 1, GRM_type::String = "simple",
    verbose::Bool = false)::Fit = gwas("GWAS_OLS", GBM_MODEL_OLS, genomes, phenomes, idx_entries, idx_loci_alleles, idx_trait, GRM_type)

gwaslmm(; genomes::Genomes, phenomes::Phenomes, idx_entries::Union{Nothing,Vector{Int64}} = nothing,
    idx_loci_alleles::Union{Nothing,Vector{Int64}} = nothing, idx_trait::Int64 = 1, GRM_type::String = "simple",
    verbose::Bool = false)::Fit = gwas("GWAS_LMM", GBM_MODEL_LMM, genomes, phenomes, idx_entries, idx_loci_alleles, idx_trait, GRM_type)

# gwasreml (src/gwas.jl:549-613): GRM-covariance LMM, variance components re-estimated per marker.
# Engine: K = U S U' (cuSOLVER), U'A by the FP64 DMMA GEMM, per-marker REML delta search on the
# device.  `objective` (an extension; the reference has no such keyword):
#   "reml" (default)  the symmetric un-standardised GRM and the standard REML likelihood, z with the profiled sigma^2;
#   "reference"       the reference's OWN objective, box and statistic (src/gwas.jl:478, :588, :596-599) on the symmetric
#                     part of the column-standardised K that gwasprep hands to loglikreml (:130, :564-573).
# What a rotation-based engine cannot reproduce (the non-symmetric part of that K, the L-BFGS path) is quantified in
# oracle/lmm_oracle.py and DESIGN.md section 2.
const GBM_LMM_REFERENCE_OBJECTIVE = Cint(8)

struct RemlTiming   # gbm_reml_timing of include/gbm_b200.h
    colstats_ms::Float64; grm_ms::Float64; allreduce_ms::Float64; kprep_ms::Float64; eig_ms::Float64
    broadcast_ms::Float64; scan_ms::Float64; gather_ms::Float64; total_ms::Float64; rotation_ms::Float64
    search_ms::Float64; rotation_tflops::Float64; grm_tflops::Float64; launches::Int64; ploidy::Int32; n_gpus::Int32
end

# GBM_NUM_GPUS > 1: the markers sharded over the group, K factored once on the first GPU and U broadcast
# (gbm_sharded_gwasreml); the same Fit as the single-GPU path below.
function gwasreml_multigpu(genomes, phenomes, idx_trait, GRM_type, y, ref::Bool)::Fit
    A = Matrix{Float64}(genomes.allele_frequencies)       # throws on `missing`, as src/prediction.jl:129 does
    n, p = size(A)
    sm = Ref{Ptr{Cvoid}}(C_NULL); packed = Ref{Cint}(0)
    check(ccall((:gbm_sharded_upload, LIBGBM), Cint,
                (Ptr{Cvoid}, Ptr{Float64}, Int64, Int64, Int64, Cint, Ref{Ptr{Cvoid}}, Ref{Cint}), group(), A, n, p, n, 1, sm, packed))
    ys = (y .- mean(y)) ./ std(y)                         # src/gwas.jl:128; gwasreml standardises once more below
    ref && (ys = (ys .- mean(ys)) ./ std(ys))             # (the reference objective's y went through gwasprep first)
    stat = Vector{Float64}(undef, p); idx = Vector{Int64}(undef, p); nk = Ref{Int64}(0); lam0 = Ref{Float64}(0.0)
    tm = Ref{RemlTiming}()
    rc = ccall((:gbm_sharded_gwasreml, LIBGBM), Cint,
               (Ptr{Cvoid}, Ptr{Float64}, Cint, Cint, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64},
                Ptr{Int64}, Ref{Int64}, Ref{Float64}, Ref{RemlTiming}),
               sm[], ys, GRM_type == "ploidy-aware" ? GBM_GRM_PLOIDY_AWARE : GBM_GRM_SIMPLE,
               ref ? GBM_LMM_REFERENCE_OBJECTIVE : Cint(0), stat, C_NULL, C_NULL, C_NULL, C_NULL, idx, nk, lam0, tm)
    ccall((:gbm_sharded_free, LIBGBM), Cint, (Ptr{Cvoid},), sm[])
    check(rc)
    idx_cols = idx[1:nk[]]
    fit = Fit(n = n, l = length(idx_cols))                # src/gwas.jl:133-140
    fit.model = "GWAS_REML"                               # src/gwas.jl:574
    fit.trait = phenomes.traits[idx_trait]
    fit.b_hat_labels = genomes.loci_alleles[idx_cols]
    fit.entries = genomes.entries
    fit.populations = genomes.populations
    fit.metrics = Dict("" => 0.0)
    fit.b_hat = stat[idx_cols]                            # src/gwas.jl:599
    if !checkdims(fit)                                    # src/gwas.jl:609-611
        throw(ErrorException("Error performing GWAS via REML using the " * GRM_type * " GRM."))
    end
    fit
end

function gwasreml(; genomes::Genomes, phenomes::Phenomes, idx_entries::Union{Nothing,Vector{Int64}} = nothing,
    idx_loci_alleles::Union{Nothing,Vector{Int64}} = nothing, idx_trait::Int64 = 1, GRM_type::String = "simple",
    verbose::Bool = false, objective::String = "reml")::Fit
    objective in ("reml", "reference") || throw(ArgumentError("objective must be \"reml\" or \"reference\""))
    ref = objective == "reference"
    if numgpus() > 1
        rows, cols, y = selectrows(genomes, phenomes, idx_entries, idx_loci_alleles, idx_trait)
        if sum(["simple", "ploidy-aware"] .== GRM_type) == 0
            throw(ArgumentError("Unrecognised `GRM_type`. Please select from:\n\t‣ simple\n\t‣ ploidy-aware"))
        end
        var(y) < eps(Float64) && throw(ArgumentError("No variance in the trait: " * phenomes.traits[idx_trait] * "."))
        if isnothing(rows) && isnothing(cols) && size(genomes.allele_frequencies, 2) >= numgpus()
            return gwasreml_multigpu(genomes, phenomes, idx_trait, GRM_type, y, ref)
        end
    end
    pr = prepare(genomes, phenomes, idx_entries, idx_loci_alleles, idx_trait, GRM_type, ref; need_kstd = ref, need_pc1 = false)
    if length(pr.entries) != size(pr.K, 1)
        free!(pr.dm)
        throw(ArgumentError("The GRM is computed on all entries of `genomes` but some entries were dropped: y and the GRM have different sizes."))
    end
    fit = newfit(pr)
    fit.model = "GWAS_REML"                               # src/gwas.jl:574
    y = (pr.y .- mean(pr.y)) ./ std(pr.y)
    plan = Ref{Ptr{Cvoid}}(C_NULL); eig_ms = Ref{Float64}(0.0); lam0 = Ref{Float64}(0.0)
    check(ccall((:gbm_lmm_plan_create, LIBGBM), Cint,
                (Ptr{Float64}, Int64, Ptr{Float64}, Ptr{Float64}, Int64, Int64, Ref{Ptr{Cvoid}}, Ref{Float64}, Ref{Float64}),
                ref ? 0.5 .* (pr.K .+ pr.K') : pr.K, pr.dm.n, y, C_NULL, 0, pr.dm.n, plan, eig_ms, lam0))
    stat = Vector{Float64}(undef, pr.dm.p)
    tf = Ref{Float64}(0.0); sms = Ref{Float64}(0.0)
    rc = ccall((:gbm_lmm_plan_run, LIBGBM), Cint,
               (Ptr{Cvoid}, Ptr{Cvoid}, Cint, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ref{Float64}, Ref{Float64}),
               plan[], pr.dm.handle, ref ? GBM_LMM_REFERENCE_OBJECTIVE : Cint(0), C_NULL, C_NULL, stat, C_NULL, C_NULL, tf, sms)
    ccall((:gbm_lmm_plan_free, LIBGBM), Cint, (Ptr{Cvoid},), plan[])
    free!(pr.dm)
    check(rc)
    fit.b_hat = stat[pr.stats.idx_cols]                   # src/gwas.jl:599
    if !checkdims(fit)                                    # src/gwas.jl:609-611
        throw(ErrorException("Error performing GWAS via REML using the " * GRM_type * " GRM."))
    end
    fit
end

# GRM entry points with the GenomicBreedingCore signatures (returning the bare matrix; wrap in
# GenomicBreedingCore.GRM as needed)
function grmsimple_b200(genomes::Genomes; idx_entries = nothing, idx_loci_alleles = nothing, verbose::Bool = false)
    dm = upload(Matrix{Float64}(genomes.allele_frequencies), idx_entries, idx_loci_alleles)
    K = grm(dm, GBM_GRM_SIMPLE, 2); free!(dm); K
end
function grmploidyaware_b200(genomes::Genomes; ploidy::Int64 = 2, idx_entries = nothing, idx_loci_alleles = nothing, verbose::Bool = false)
    dm = upload(Matrix{Float64}(genomes.allele_frequencies), idx_entries, idx_loci_alleles)
    K = grm(dm, GBM_GRM_PLOIDY_AWARE, ploidy); free!(dm); K
end

# ---- transformation screens (src/transformation.jl:130-239, :319-466, :540-651) -----------------
# The l (transform1) / l^2 (transform2) regressions `ols(genomes = g, phenomes = p).b_hat[2]` run in
# libgbm_b200.so.  `f` must be one of the package's named endofunctions (src/transformation.jl:1-55):
# a closure cannot cross the C ABI and there is no CPU fallback.
square(x) = x^2
invoneplus(x) = 1 / (1 + x)
log10epsdivlog10eps(x) = (log10(x + eps(Float64))) / log10(eps(Float64))
mult(x, y) = x * y
addnorm(x, y) = (x + y) / 2.0
raise(x, y) = x^y
const F1_CODES = IdDict{Any,Cint}(square => 0, invoneplus => 1, log10epsdivlog10eps => 2)
const F2_CODES = IdDict{Any,Cint}(mult => 0, addnorm => 1, raise => 2)
function fcode(f, table, arity)
    haskey(table, f) || throw(ArgumentError("`" * string(f) * "` is not one of the named endofunctions of " * string(arity) *
                                            " argument(s); only those run on the device (no CPU fallback)."))
    table[f]
end

function extractdevice(genomes, phenomes, idx_trait, idx_entries, idx_loci_alleles)
    rows, cols, y = selectrows(genomes, phenomes, idx_entries, idx_loci_alleles, idx_trait)
    A = genomes.allele_frequencies
    any(ismissing, A) && throw(ErrorException("cannot convert a value of type Missing to Float64"))
    dm = upload(Matrix{Float64}(A), rows, cols)
    r = isnothing(rows) ? collect(1:size(A, 1)) : rows
    c = isnothing(cols) ? collect(1:size(A, 2)) : cols
    (dm, y, genomes.entries[r], genomes.populations[r], genomes.loci_alleles[c])
end

function transform1(f::Function, genomes::Genomes, phenomes::Phenomes; idx_trait::Int64 = 1,
                    idx_entries::Union{Nothing,Vector{Int64}} = nothing, idx_loci_alleles::Union{Nothing,Vector{Int64}} = nothing,
                    n_new_features_per_transformation::Int64 = 1_000, ϵ::Float64 = eps(Float64), use_abs::Bool = false,
                    σ²_threshold::Float64 = 0.01, verbose::Bool = false)::Genomes
    code = fcode(f, F1_CODES, 1)
    dm, y, entries, populations, loci_alleles = extractdevice(genomes, phenomes, idx_trait, idx_entries, idx_loci_alleles)
    idx = Vector{Int64}(undef, max(n_new_features_per_transformation, 1))
    count = Ref{Int64}(0)
    check(ccall((:gbm_transform1_screen, LIBGBM), Cint,
                (Ptr{Cvoid}, Ptr{Float64}, Cint, Float64, Cint, Float64, Int64, Ptr{Float64}, Ptr{Int64}, Ref{Int64}),
                dm.handle, y, code, ϵ, use_abs, σ²_threshold, n_new_features_per_transformation, C_NULL, idx, count))
    resize!(idx, count[])
    T = Matrix{Float64}(undef, dm.n, length(idx))
    check(ccall((:gbm_transform1_apply, LIBGBM), Cint,
                (Ptr{Cvoid}, Cint, Float64, Cint, Ptr{Int64}, Int64, Ptr{Float64}, Int64),
                dm.handle, code, ϵ, use_abs, idx, length(idx), T, dm.n))
    free!(dm)
    out = Genomes(n = size(T, 1), p = length(idx))
    out.entries = entries
    out.populations = populations
    out.allele_frequencies = T
    out.loci_alleles = string.(f, "(", loci_alleles[idx], ")")  # src/transformation.jl:235
    checkdims(out) || throw(ErrorException("Error transforming each locus using the function `" * string(f) * "`."))
    out
end

function transform2(f::Function, genomes::Genomes, phenomes::Phenomes; idx_trait::Int64 = 1,
                    idx_entries::Union{Nothing,Vector{Int64}} = nothing, idx_loci_alleles::Union{Nothing,Vector{Int64}} = nothing,
                    n_new_features_per_transformation::Int64 = 1_000, ϵ::Float64 = eps(Float64), use_abs::Bool = false,
                    σ²_threshold::Float64 = 0.01, commutative::Bool = false, verbose::Bool = false)::Genomes
    code = fcode(f, F2_CODES, 2)
    dm, y, entries, populations, loci_alleles = extractdevice(genomes, phenomes, idx_trait, idx_entries, idx_loci_alleles)
    l = dm.p
    counters = Vector{Int64}(undef, max(n_new_features_per_transformation, 1))
    count = Ref{Int64}(0)
    check(ccall((:gbm_transform2_screen, LIBGBM), Cint,
                (Ptr{Cvoid}, Ptr{Float64}, Cint, Float64, Cint, Float64, Cint, Int64, Ptr{Float64}, Ptr{Int64}, Ptr{Float64}, Ref{Int64}),
                dm.handle, y, code, ϵ, use_abs, σ²_threshold, commutative, n_new_features_per_transformation, C_NULL,
                counters, C_NULL, count))
    resize!(counters, count[])
    T = Matrix{Float64}(undef, dm.n, length(counters))
    check(ccall((:gbm_transform2_apply, LIBGBM), Cint,
                (Ptr{Cvoid}, Cint, Float64, Cint, Ptr{Int64}, Int64, Ptr{Float64}, Int64),
                dm.handle, code, ϵ, use_abs, counters, length(counters), T, dm.n))
    free!(dm)
    out = Genomes(n = size(T, 1), p = length(counters))
    out.entries = entries
    out.populations = populations
    out.allele_frequencies = T
    out.loci_alleles = [string(f, "(", loci_alleles[1+div(c - 1, l)], ",", loci_alleles[1+(c-1)%l], ")") for c in counters]  # :445-451
    checkdims(out) || throw(ErrorException("Error transforming each locus using the function `" * string(f) * "`."))
    out
end

function epistasisfeatures(genomes::Genomes, phenomes::Phenomes; idx_trait::Int64 = 1,
                           idx_entries::Union{Nothing,Vector{Int64}} = nothing,
                           idx_loci_alleles::Union{Nothing,Vector{Int64}} = nothing,
                           transformations1 = [square, invoneplus, log10epsdivlog10eps], transformations2 = [mult, addnorm, raise],
                           n_new_features_per_transformation::Int64 = 1_000, n_reps::Int64 = 3, verbose::Bool = false)::Genomes
    selectrows(genomes, phenomes, idx_entries, idx_loci_alleles, idx_trait)  # the argument checks of :552-601
    idx_entries = isnothing(idx_entries) ? collect(1:length(genomes.entries)) : idx_entries
    idx_loci_alleles = isnothing(idx_loci_alleles) ? collect(1:length(genomes.loci_alleles)) : idx_loci_alleles
    genomes = slice(genomes, idx_entries = idx_entries, idx_loci_alleles = idx_loci_alleles)
    phenomes = slice(phenomes, idx_entries = idx_entries, idx_traits = [idx_trait])
    for r = 1:n_reps, f in vcat(transformations1, transformations2)
        g = f ∈ transformations1 ?
            transform1(f, genomes, phenomes, n_new_features_per_transformation = n_new_features_per_transformation) :
            transform2(f, genomes, phenomes, n_new_features_per_transformation = n_new_features_per_transformation)
        idx_new = [findall(g.loci_alleles .== x)[1] for x in setdiff(g.loci_alleles, genomes.loci_alleles)]
        append!(genomes.loci_alleles, g.loci_alleles[idx_new])
        genomes.allele_frequencies = hcat(genomes.allele_frequencies, g.allele_frequencies[:, idx_new])
        genomes.mask = hcat(genomes.mask, g.mask[:, idx_new])
        if (minimum(genomes.allele_frequencies) < 0.0) || (abs(maximum(genomes.allele_frequencies) - 1) > 1e-12)
            throw(ErrorException("The function `" * string(f) * "` generates values outside the expected range of zero to one. Please replace with an appropriate transforamtion function."))
        end
    end
    checkdims(genomes) || throw(ErrorException("Error generating new features."))
    genomes
end

end # module
