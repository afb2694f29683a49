# GenLibCUDA.jl -- the `ccall` shim a GenLib.jl maintainer would add so that
# `gen.phi(ped)` / `gen.phi(ped, probandIDs)` run on libgenlib_cuda.so (B200).
#
# NOT EXECUTED in this repository's CI: Julia is not installed in the build image
# (SURVEY.md F6).  The same C ABI is exercised through Python ctypes by tests/.
#
# It keeps the reference's signature and return type (src/compute.jl:233-304):
#     phi(pedigree::Pedigree, probandIDs::Vector{Int} = pro(pedigree);
#         verbose::Bool = false, compute::Bool = true) -> Matrix{Float32}
# There is no CPU fallback: if the library or a CUDA device is missing, it throws.
module GenLibCUDA

import GenLib
using Libdl

const libgenlib = Ref{String}(get(ENV, "GENLIB_CUDA_LIB", "libgenlib_cuda.so"))

struct LayerInfo            # genlib_layer_info, include/genlib_cuda.h
    n_new::Int32; n_fam::Int32; live_before::Int32; carried::Int32
    ref_founders::Int32; ref_probands::Int32; ref_both::Int32; strip_width::Int32
    alg_elems::Float64; ms_layer::Float64; ms_wait::Float64
    dram_read_bytes::Float64; dram_write_bytes::Float64; l2_bytes::Float64; nvlink_bytes::Float64
end

struct Stats                # genlib_stats
    n_unique::Int32; n_layers::Int32; row_updates::Int64; capacity::Int64; device_bytes::Int64
    alg_bytes::Float64; ms_plan::Float64; ms_upload::Float64; ms_kernels::Float64; ms_fetch::Float64
    h2d_bytes::Int64; d2h_bytes::Int64; kernel_launches::Int32; reserved::Int32
end

function check(status::Cint)
    status == 0 && return
    msg = unsafe_string(ccall((:genlib_last_error, libgenlib[]), Cstring, ()))
    status == 2 && throw(KeyError(msg))            # same exception as pedigree[ID] (src/create.jl:70)
    status == 5 && throw(OutOfMemoryError())
    status == 8 && throw(OverflowError(msg))       # genlib_occ: a count does not fit an Int64
    error("libgenlib_cuda status $status: $msg")
end

"""Flatten a `Pedigree` into 0-based parent ranks (iteration order is rank order,
src/create.jl:234-254)."""
function flatten(pedigree::GenLib.Pedigree)
    n = length(pedigree)
    father = Vector{Int32}(undef, n)
    mother = Vector{Int32}(undef, n)
    for individual in values(pedigree)
        r = individual.rank
        father[r] = isnothing(individual.father) ? Int32(-1) : Int32(individual.father.rank - 1)
        mother[r] = isnothing(individual.mother) ? Int32(-1) : Int32(individual.mother.rank - 1)
    end
    father, mother
end

"""
A `Matrix{Float32}` (or `Float64`) in page-locked host memory (`genlib_pinned_alloc`): the device copies
into it at full PCIe speed.  The memory is given back when the matrix is garbage collected.
"""
function pinned_matrix(::Type{T}, n::Integer) where {T <: Union{Float32, Float64}}
    p = Ref{Ptr{Cvoid}}(C_NULL)
    check(ccall((:genlib_pinned_alloc, libgenlib[]), Cint, (Csize_t, Ptr{Ptr{Cvoid}}), max(1, n * n * sizeof(T)), p))
    A = unsafe_wrap(Array, Ptr{T}(p[]), (Int(n), Int(n)); own = false)
    finalizer(_ -> ccall((:genlib_pinned_free, libgenlib[]), Cint, (Ptr{Cvoid},), p[]), A)
    A
end

"""
    phi(pedigree, probandIDs = pro(pedigree); verbose = false, compute = true,
        numerics = :reference, devices = Int[], pinned = false) -> Matrix{Float32}

`gen.phi` (src/compute.jl:233-304) on the B200 engine.  `devices = [0, 1, ...]` shards the frontier over
several GPUs of the box from this one process (`genlib_phi_multi`: one plan, one host thread per device,
NVLink peer access); the result is bitwise the single-GPU one.  `pinned = true` returns the matrix in
page-locked memory (the 400 MB of a 10 000-proband result then arrive in ~8 ms instead of ~40 ms).
"""
function phi(pedigree::GenLib.Pedigree, probandIDs::Vector{Int} = GenLib.pro(pedigree);
             verbose::Bool = false, compute::Bool = true, numerics::Symbol = :reference,
             device::Integer = -1, devices::Vector{<:Integer} = Int[], pinned::Bool = false)
    father, mother = flatten(pedigree)
    probands = Int32[pedigree[ID].rank - 1 for ID in probandIDs]      # KeyError on unknown ID
    if compute && !verbose
        # The one-call entry points plan on a worker thread and run every generation as soon as it is planned
        # (planning is otherwise the largest host-side part of the call): nothing here needs the plan itself.
        n = length(unique(probands))                                   # duplicates collapse (src/compute.jl:251)
        ϕ = pinned ? pinned_matrix(Float32, n) : Matrix{Float32}(undef, n, n)   # symmetric: layout-free
        n == 0 && return ϕ
        devs = isempty(devices) ? Int32[device] : Int32.(devices)      # one device: genlib_phi; several: sharded rows
        GC.@preserve ϕ check(ccall((:genlib_phi_multi, libgenlib[]), Cint,
            (Int32, Ptr{Int32}, Ptr{Int32}, Int32, Ptr{Int32}, Ptr{Cvoid}, Cint, Cint, Int32, Ptr{Int32}, Ptr{Cvoid}),
            length(father), father, mother, length(probands), probands, ϕ, 0,
            numerics === :fp64 ? 1 : 0, length(devs), devs, C_NULL))
        return ϕ
    end
    plan = Ref{Ptr{Cvoid}}(C_NULL)
    check(ccall((:genlib_plan_create, libgenlib[]), Cint,
                (Int32, Ptr{Int32}, Ptr{Int32}, Int32, Ptr{Int32}, Int32, Ptr{Ptr{Cvoid}}),
                length(father), father, mother, length(probands), probands, 1, plan))
    try
        layers = ccall((:genlib_plan_n_layers, libgenlib[]), Int32, (Ptr{Cvoid},), plan[])
        if verbose || !compute                                         # src/compute.jl:253-262
            for k in 1:layers-1
                info = Ref{LayerInfo}()
                check(ccall((:genlib_plan_layer_info, libgenlib[]), Cint,
                            (Ptr{Cvoid}, Int32, Ref{LayerInfo}), plan[], k, info))
                println("Step $k of $(layers-1): $(info[].ref_founders) founders, " *
                        "$(info[].ref_probands) probands, $(info[].ref_both) both.")
            end
        end
        compute || return nothing                                      # src/compute.jl:264-266
        n = ccall((:genlib_plan_n_unique, libgenlib[]), Int32, (Ptr{Cvoid},), plan[])
        ϕ = pinned ? pinned_matrix(Float32, n) : Matrix{Float32}(undef, n, n)   # symmetric: layout-free
        n == 0 && return ϕ
        if length(devices) > 1                                         # one process, several GPUs
            devs = Int32.(devices)
            GC.@preserve ϕ check(ccall((:genlib_phi_multi, libgenlib[]), Cint,
                (Int32, Ptr{Int32}, Ptr{Int32}, Int32, Ptr{Int32}, Ptr{Cvoid}, Cint, Cint, Int32, Ptr{Int32}, Ptr{Cvoid}),
                length(father), father, mother, length(probands), probands, ϕ, 0,
                numerics === :fp64 ? 1 : 0, length(devs), devs, C_NULL))
            return ϕ
        end
        dev = length(devices) == 1 ? Int(devices[1]) : Int(device)
        engine = Ref{Ptr{Cvoid}}(C_NULL)
        check(ccall((:genlib_engine_create, libgenlib[]), Cint,
                    (Ptr{Cvoid}, Cint, Cint, Ptr{Ptr{Cvoid}}),
                    plan[], numerics === :fp64 ? 1 : 0, dev, engine))
        try
            check(ccall((:genlib_engine_run, libgenlib[]), Cint, (Ptr{Cvoid}, Cint), engine[], 0))
            GC.@preserve ϕ check(ccall((:genlib_engine_fetch, libgenlib[]), Cint,
                                       (Ptr{Cvoid}, Ptr{Cvoid}, Cint), engine[], ϕ, 0))
        finally
            ccall((:genlib_engine_destroy, libgenlib[]), Cvoid, (Ptr{Cvoid},), engine[])
        end
        return ϕ
    finally
        ccall((:genlib_plan_destroy, libgenlib[]), Cvoid, (Ptr{Cvoid},), plan[])
    end
end

"""
    phiMean(pedigree, probandIDs = pro(pedigree)) -> Float64

The mean off-diagonal kinship of `phi(pedigree, probandIDs)` reduced ON THE DEVICE
(`genlib_engine_phi_mean`): the matrix never crosses PCIe.  Binary64 accumulation in a fixed order
(reproducible), where `gen.phiMean(::Matrix{Float32})` (src/compute.jl:454-459) adds Float32 values
pairwise; they agree to Float32 precision.  `gen.phiMean(phi(ped))` itself keeps working: `phi`
returns the `Matrix{Float32}` that method wants.
"""
function phiMean(pedigree::GenLib.Pedigree, probandIDs::Vector{Int} = GenLib.pro(pedigree); device::Integer = -1)
    father, mother = flatten(pedigree)
    probands = Int32[pedigree[ID].rank - 1 for ID in probandIDs]
    plan = Ref{Ptr{Cvoid}}(C_NULL)
    check(ccall((:genlib_plan_create, libgenlib[]), Cint,
                (Int32, Ptr{Int32}, Ptr{Int32}, Int32, Ptr{Int32}, Int32, Ptr{Ptr{Cvoid}}),
                length(father), father, mother, length(probands), probands, 1, plan))
    try
        engine = Ref{Ptr{Cvoid}}(C_NULL)
        check(ccall((:genlib_engine_create, libgenlib[]), Cint, (Ptr{Cvoid}, Cint, Cint, Ptr{Ptr{Cvoid}}),
                    plan[], 0, device, engine))
        try
            check(ccall((:genlib_engine_run, libgenlib[]), Cint, (Ptr{Cvoid}, Cint), engine[], 0))
            mean = Ref{Cdouble}(0)
            check(ccall((:genlib_engine_phi_mean, libgenlib[]), Cint, (Ptr{Cvoid}, Ptr{Cdouble}), engine[], mean))
            return mean[]
        finally
            ccall((:genlib_engine_destroy, libgenlib[]), Cvoid, (Ptr{Cvoid},), engine[])
        end
    finally
        ccall((:genlib_plan_destroy, libgenlib[]), Cvoid, (Ptr{Cvoid},), plan[])
    end
end

"""
    f(pedigree, IDs) -> Vector{Float32}

`gen.f` (src/compute.jl:500-511): inbreeding = kinship of the parents.  The reference runs the
exponential pairwise recursion once per ID; here the parents of all IDs go through ONE sweep of the
engine with Float64 storage (exact while kinships fit 53 bits, i.e. pedigrees up to ~26 generations deep;
beyond that the last bits can differ from the reference's Float64 recursion) and are rounded to Float32.
"""
function f(pedigree::GenLib.Pedigree, IDs::Vector{Int}; device::Integer = -1)
    coefficients = zeros(Float32, length(IDs))
    pairs = [(pedigree[ID].father, pedigree[ID].mother) for ID in IDs]          # KeyError on unknown ID
    parents = sort(unique(Int[p.ID for pr in pairs for p in pr if !isnothing(pr[1]) && !isnothing(pr[2])]))
    isempty(parents) && return coefficients
    k = phi(pedigree, parents; numerics = :fp64, device = device)   # Float32 view of the Float64-storage sweep
    pos = Dict(ID => i for (i, ID) in enumerate(parents))
    for (i, (fa, mo)) in enumerate(pairs)
        (isnothing(fa) || isnothing(mo)) && continue
        coefficients[i] = k[pos[fa.ID], pos[mo.ID]]
    end
    coefficients
end

"""
    sparse_phi(pedigree, probandIDs = pro(pedigree)) -> GenLib.KinshipMatrix

`gen.sparse_phi` (src/compute.jl:321-447) on the GPU: the same engine, planned for sparse_phi's own
floating-point schedule (`GENLIB_SCHEDULE_SPARSE_PHI`), so every look-up `ϕ[ID₁, ID₂]` returns the
reference's bits -- including the 0 the reference returns for a kinship it filed under
`ϕ[earlier][later]` but looks up under `ϕ[lower rank][higher rank]` (src/compute.jl:393 vs :36-40).
`symmetric = true` keeps those kinships (`GENLIB_SCHEDULE_SPARSE_PHI_SYMMETRIC`).  The dense result is
folded back into the reference's `KinshipMatrix` (Dict keyed lower rank -> higher rank, zeros not
stored, src/compute.jl:31-40, 391-394); misfiled and orphaned keys, which no look-up reads, are not
recreated, so `show` may count fewer entries than the reference's.
"""
function sparse_phi(pedigree::GenLib.Pedigree, probandIDs::Vector{Int} = GenLib.pro(pedigree);
                    device::Integer = -1, symmetric::Bool = false)
    father, mother = flatten(pedigree)
    ranks = Int32[pedigree[ID].rank - 1 for ID in probandIDs]           # KeyError on unknown ID
    ids = Int64[individual.ID for individual in values(pedigree)]      # founder() sorts by ID (src/identify.jl:15-19)
    plan = Ref{Ptr{Cvoid}}(C_NULL)
    check(ccall((:genlib_plan_create_ex, libgenlib[]), Cint,
                (Int32, Ptr{Int32}, Ptr{Int32}, Ptr{Int64}, Int32, Ptr{Int32}, Int32, Cint, Ptr{Ptr{Cvoid}}),
                length(father), father, mother, ids, length(ranks), ranks, 1, symmetric ? 2 : 1, plan))
    try
        n = ccall((:genlib_plan_n_unique, libgenlib[]), Int32, (Ptr{Cvoid},), plan[])
        dense = Matrix{Float32}(undef, n, n)
        engine = Ref{Ptr{Cvoid}}(C_NULL)
        check(ccall((:genlib_engine_create, libgenlib[]), Cint, (Ptr{Cvoid}, Cint, Cint, Ptr{Ptr{Cvoid}}),
                    plan[], 0, device, engine))
        try
            check(ccall((:genlib_engine_run, libgenlib[]), Cint, (Ptr{Cvoid}, Cint), engine[], 0))
            GC.@preserve dense check(ccall((:genlib_engine_fetch, libgenlib[]), Cint,
                                           (Ptr{Cvoid}, Ptr{Cvoid}, Cint), engine[], dense, 0))
        finally
            ccall((:genlib_engine_destroy, libgenlib[]), Cvoid, (Ptr{Cvoid},), engine[])
        end
        unique_IDs = unique(probandIDs)                                  # output order = first occurrence
        isolated = GenLib.branching(pedigree, pro = probandIDs)          # sparse_phi's ranks (src/compute.jl:323)
        rank = Dict{Int32, Int}(ID => isolated[ID].rank for ID in unique_IDs)
        dict = Dict{Int32, Dict{Int32, Float32}}(rank[ID] => Dict{Int32, Float32}() for ID in unique_IDs)
        for (a, IDa) in enumerate(unique_IDs), (b, IDb) in enumerate(unique_IDs)
            (ra, rb) = (rank[IDa], rank[IDb])
            (ra == rb || (ra < rb && dense[a, b] != 0)) && (dict[ra][rb] = dense[a, b])
        end
        return GenLib.KinshipMatrix(dict, rank)
    finally
        ccall((:genlib_plan_destroy, libgenlib[]), Cvoid, (Ptr{Cvoid},), plan[])
    end
end

struct GcStats              # genlib_gc_stats
    n_pro::Int32; n_anc::Int32; n_layers::Int32; direction::Int32
    rows::Int64; inputs::Int64; width::Int64; capacity::Int64; device_bytes::Int64
    alg_bytes::Float64; ms_plan::Float64; ms_kernels::Float64; ms_fetch::Float64
    d2h_bytes::Int64; kernel_launches::Int32; n_dev::Int32
end

"""
    gc(pedigree; pro = GenLib.pro(pedigree), ancestors = GenLib.founder(pedigree),
       device = -1, devices = Int[]) -> Matrix{Float64}

`gen.gc` (src/compute.jl:518-595) on the B200 engine: `G[p, a]` = the expected share of proband `p`'s
genome that comes from ancestor `a`, the sum over descent paths of (1/2)^length.  Rows follow `pro`,
columns follow `ancestors`, duplicates kept; an unknown ID throws `KeyError`.  The library writes the
column-major matrix directly (`col_major = 1`), so there is no transpose on the host.  `devices = [0, 1, ...]`
splits the columns over several GPUs of the box; the result is bitwise the one-GPU result.
Like the rest of this shim it is not executed in this repository (no Julia in the build image); the same
call is exercised through Python ctypes by tests/test_gc.py.
"""
function gc(pedigree::GenLib.Pedigree; pro::Vector{Int} = GenLib.pro(pedigree),
            ancestors::Vector{Int} = GenLib.founder(pedigree), device::Integer = -1,
            devices::Vector{<:Integer} = Int[])
    father, mother = flatten(pedigree)
    p = Int32[pedigree[ID].rank - 1 for ID in pro]                   # KeyError on unknown ID
    a = Int32[pedigree[ID].rank - 1 for ID in ancestors]
    devs = isempty(devices) ? Int32[device] : Int32.(devices)
    G = Matrix{Float64}(undef, length(p), length(a))
    stats = Ref{GcStats}()
    GC.@preserve G check(ccall((:genlib_gc, libgenlib[]), Cint,
        (Int32, Ptr{Int32}, Ptr{Int32}, Int32, Ptr{Int32}, Int32, Ptr{Int32}, Ptr{Cvoid}, Cint, Cint, Int32,
         Ptr{Int32}, Ptr{GcStats}),
        length(father), father, mother, length(p), p, length(a), a, pointer(G), 1, 1, length(devs), devs, stats))
    G
end

"""
    occ(pedigree; pro = GenLib.pro(pedigree), ancestors = GenLib.founder(pedigree), typeOcc = "IND",
        device = -1, devices = Int[]) -> Matrix{Int64}

`gen.occ` on the B200 engine: `O[a, p]` = the number of descent paths from ancestor `a` to proband `p`
(1 for `a == p` itself).  ROWS ARE ANCESTORS, columns follow `pro`, duplicates kept; `typeOcc = "TOTAL"`
gives the `length(ancestors) x 1` row sums, reduced on the device.  Another `typeOcc` throws `ArgumentError`
before the library is called; a count or row sum that does not fit an Int64 throws `OverflowError` naming
the first offending (ancestor, proband) pair (0-based list positions and ranks).  The library writes the
column-major matrix directly.  Exercised through Python ctypes by tests/test_occ.py, not executed here.
"""
function occ(pedigree::GenLib.Pedigree; pro::Vector{Int} = GenLib.pro(pedigree),
             ancestors::Vector{Int} = GenLib.founder(pedigree), typeOcc::AbstractString = "IND",
             device::Integer = -1, devices::Vector{<:Integer} = Int[])
    typeOcc in ("IND", "TOTAL") || throw(ArgumentError("typeOcc must be \"IND\" or \"TOTAL\", not \"$typeOcc\""))
    father, mother = flatten(pedigree)
    p = Int32[pedigree[ID].rank - 1 for ID in pro]                   # KeyError on unknown ID
    a = Int32[pedigree[ID].rank - 1 for ID in ancestors]
    devs = isempty(devices) ? Int32[device] : Int32.(devices)
    O = Matrix{Int64}(undef, length(a), typeOcc == "IND" ? length(p) : 1)
    stats = Ref{GcStats}()
    GC.@preserve O check(ccall((:genlib_occ, libgenlib[]), Cint,
        (Int32, Ptr{Int32}, Ptr{Int32}, Int32, Ptr{Int32}, Int32, Ptr{Int32}, Ptr{Int64}, Cint, Cint, Int32,
         Ptr{Int32}, Ptr{GcStats}),
        length(father), father, mother, length(p), p, length(a), a, pointer(O), typeOcc == "IND" ? 0 : 1, 1,
        length(devs), devs, stats))
    O
end

"""
    rec(pedigree; pro = GenLib.pro(pedigree), ancestors = GenLib.founder(pedigree),
        device = -1, devices = Int[]) -> Vector{Int64}

`gen.rec` on the B200 engine: for every ancestor, the number of entries of `pro` that descend from it, the
ancestor itself included, duplicates counted.  Reduced on the device.  Exercised through Python ctypes by
tests/test_occ.py, not executed here.
"""
function rec(pedigree::GenLib.Pedigree; pro::Vector{Int} = GenLib.pro(pedigree),
             ancestors::Vector{Int} = GenLib.founder(pedigree), device::Integer = -1,
             devices::Vector{<:Integer} = Int[])
    father, mother = flatten(pedigree)
    p = Int32[pedigree[ID].rank - 1 for ID in pro]
    a = Int32[pedigree[ID].rank - 1 for ID in ancestors]
    devs = isempty(devices) ? Int32[device] : Int32.(devices)
    r = Vector{Int64}(undef, length(a))
    stats = Ref{GcStats}()
    GC.@preserve r check(ccall((:genlib_rec, libgenlib[]), Cint,
        (Int32, Ptr{Int32}, Ptr{Int32}, Int32, Ptr{Int32}, Int32, Ptr{Int32}, Ptr{Int64}, Int32, Ptr{Int32},
         Ptr{GcStats}),
        length(father), father, mother, length(p), p, length(a), a, pointer(r), length(devs), devs, stats))
    r
end

end # module
