# RANSACB200.jl -- Julia host binding of libransac_b200 (include/rsc.h) for cserteGT3/RANSAC.jl.
#
# UNTESTED IN THIS REPOSITORY'S CI: the build image has no Julia.  The binding mirrors, one to one,
# the ctypes binding that the test-suite exercises (ransac.jl_b200/_lib.py); struct layouts are the
# ones asserted in tests/test_abi_cpu.py.
#
# It keeps RANSAC.jl's public surface: `ransac(pc, params, setenabled)`, `RANSACCloud`, the
# `Fitted*` types and the parameter NamedTuples are RANSAC.jl's own.  What changes is where the work
# happens: for the four built-in shapes `fit` / `scorecandidate` / `refit` / the loop body are
# `ccall`s into the CUDA library.  User-defined shapes keep their Julia methods (docs/src/newprimitive.md).
module RANSACB200

using RANSAC
using RANSAC: FittedShape, FittedPlane, FittedSphere, FittedCylinder, FittedCone, ExtractedShape,
              RANSACCloud, ConfidenceInterval
using StaticArrays
using Libdl

# The library is opened at RUN time (ENV["RANSAC_B200_LIB"] or the loader path) and its entry points are passed to
# `ccall` as `dlsym` pointers: a `(name, library)` tuple must be a compile-time constant on older Julia 1.x, and a
# constant would freeze the path of the machine that precompiled the package.
const LIBHANDLE = Ref{Ptr{Cvoid}}(C_NULL)
const SYMS = Dict{Symbol,Ptr{Cvoid}}()
libpath() = get(ENV, "RANSAC_B200_LIB", "libransac_b200.so")
function fn(name::Symbol)
    get!(SYMS, name) do
        LIBHANDLE[] == C_NULL && (LIBHANDLE[] = Libdl.dlopen(libpath()))
        Libdl.dlsym(LIBHANDLE[], name)
    end
end
__init__() = (LIBHANDLE[] = C_NULL; empty!(SYMS); nothing)   # pointers of a precompile session are never reused

# ---- POD mirrors (include/rsc.h) -------------------------------------------------------------
struct RscCand            # 64 bytes
    type::Int32
    outwards::Int32
    p::NTuple{7,Float64}
end

struct RscParams          # 160 bytes
    drawN::Int32
    minsubsetN::Int32
    prob_det::Float64
    tau::Int64
    itermax::Int32
    extract_s::Int32
    terminate_s::Int32
    n_shape_types::Int32
    shape_types::NTuple{4,Int32}
    collin_threshold::Float64
    parallelthrdeg::Float64
    eps::NTuple{4,Float64}
    alpha::NTuple{4,Float64}
    sphere_par::Float64
    minconeopang::Float64
    compat_flags::UInt32
    lw_period::UInt32         # RSC_SAMPLER_OCTREE: refresh period of the level weights (0/1 = every iteration)
end

struct RscShapeSlot        # 72 bytes: one position of a fit order (a built-in kind or a compiled user type id)
    type::Int32
    nk::Int32
    k::NTuple{8,Float64}
end
RscShapeSlot(type::Integer, k::Vector{Float64}=Float64[]) =
    RscShapeSlot(Int32(type), Int32(length(k)), ntuple(i -> i <= length(k) ? k[i] : 0.0, 8))

const KIND = Dict{Any,Int32}(FittedPlane => 0, FittedSphere => 1, FittedCylinder => 2, FittedCone => 3)
const S_SYM = Dict(:lengthC => Int32(0), :allcand => Int32(1), :nofminset => Int32(2))

tocand(s::FittedPlane) = RscCand(0, 1, (s.point..., s.normal..., 0.0))
tocand(s::FittedSphere) = RscCand(1, s.outwards, (s.center..., s.radius, 0.0, 0.0, 0.0))
tocand(s::FittedCylinder) = RscCand(2, s.outwards, (s.axis..., s.center..., s.radius))
tocand(s::FittedCone) = RscCand(3, s.outwards, (s.apex..., s.axis..., s.opang))

function fromcand(c::RscCand)
    p = c.p
    v(i) = SVector{3,Float64}(p[i], p[i+1], p[i+2])
    c.type == 0 && return FittedPlane(v(1), v(4))
    c.type == 1 && return FittedSphere(v(1), p[4], c.outwards != 0)
    c.type == 2 && return FittedCylinder(v(1), v(4), p[7], c.outwards != 0)
    return FittedCone(v(1), v(4), p[7], c.outwards != 0)
end

"Flatten the nested NamedTuple of `ransacparameters` (utilities.jl:332-433) into the C POD."
function toparams(params)
    it = params.iteration
    types = Int32[KIND[t] for t in it.shape_types if haskey(KIND, t)]   # (user types travel in a fit order)
    st = ntuple(i -> i <= length(types) ? types[i] : Int32(0), 4)
    g(name, f, d) = haskey(params, name) ? Float64(getfield(getfield(params, name), f)) : d
    eps = (g(:plane, :ϵ, 0.3), g(:sphere, :ϵ, 0.3), g(:cylinder, :ϵ, 0.3), g(:cone, :ϵ, 0.3))
    alp = (g(:plane, :α, deg2rad(5)), g(:sphere, :α, deg2rad(5)), g(:cylinder, :α, deg2rad(5)), g(:cone, :α, deg2rad(5)))
    RscParams(it.drawN, it.minsubsetN, it.prob_det, it.τ, it.itermax, S_SYM[it.extract_s], S_SYM[it.terminate_s],
              length(types), st, params.common.collin_threshold, params.common.parallelthrdeg, eps, alp,
              g(:sphere, :sphere_par, 0.02), g(:cone, :minconeopang, deg2rad(2)), UInt32(1), UInt32(0))
end

# ---- context / cloud handles ---------------------------------------------------------------------
const CTX = Ref{Ptr{Cvoid}}(C_NULL)

version() = ccall(fn(:rsc_version), Int32, ())

function check(rc)
    rc == 0 && return
    msg = unsafe_string(ccall(fn(:rsc_last_error), Cstring, (Ptr{Cvoid},), CTX[]))
    error("libransac_b200 error $rc: $msg")
end

function context(device::Integer=0)
    if CTX[] == C_NULL
        h = Ref{Ptr{Cvoid}}(C_NULL)
        rc = ccall(fn(:rsc_ctx_create), Int32, (Int32, Ref{Ptr{Cvoid}}), device, h)
        rc == 0 || error("rsc_ctx_create failed ($rc): an sm_100 (B200) GPU is required, there is no CPU fallback")
        CTX[] = h[]
    end
    CTX[]
end

"""Device twin of a `RANSACCloud`: uploads vertices/normals (float32 SoA on the GPU) and subset 1.
`exact=true` on a Float64 cloud keeps the Float64 coordinates on the device too (`rsc_cloud_create_f64_exact`,
+48 B/point): every decision and fit is then the Float64 one of the points as given."""
mutable struct DeviceCloud
    h::Ptr{Cvoid}
    pc::RANSACCloud
    function DeviceCloud(pc::RANSACCloud; exact::Bool=false)
        ctx = context()
        h = Ref{Ptr{Cvoid}}(C_NULL)
        v, n = pc.vertices, pc.normals            # Vector{SVector{3,T}} is bit-compatible with T[3N]
        if !(eltype(eltype(v)) == eltype(eltype(n)) && eltype(eltype(v)) in (Float32, Float64))
            # mixed or other element types (RANSACCloud keeps the two eltypes apart, octree.jl:102-103): go through Float64
            v = [SVector{3,Float64}(x) for x in v]
            n = [SVector{3,Float64}(x) for x in n]
        end
        GC.@preserve v n begin
            if eltype(eltype(v)) == Float32
                check(ccall(fn(:rsc_cloud_create), Int32, (Ptr{Cvoid}, Ptr{Float32}, Ptr{Float32}, Int64, Ref{Ptr{Cvoid}}),
                            ctx, pointer(v), pointer(n), pc.size, h))
            elseif exact
                check(ccall(fn(:rsc_cloud_create_f64_exact), Int32, (Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}, Int64, Ref{Ptr{Cvoid}}),
                            ctx, pointer(v), pointer(n), pc.size, h))
            else
                check(ccall(fn(:rsc_cloud_create_f64), Int32, (Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}, Int64, Ref{Ptr{Cvoid}}),
                            ctx, pointer(v), pointer(n), pc.size, h))
            end
        end
        idx = Int64.(pc.subsets[1] .- 1)          # 0-based on the C side
        check(ccall(fn(:rsc_cloud_set_subset), Int32, (Ptr{Cvoid}, Int32, Ptr{Int64}, Int64), h[], 0, idx, length(idx)))
        dc = new(h[], pc)
        push_enabled!(dc)
        finalizer(d -> ccall(fn(:rsc_cloud_destroy), Cvoid, (Ptr{Cvoid},), d.h), dc)
    end
end

# pc.isenabled is a BitArray: its `chunks` are exactly the UInt64 words the C ABI expects
push_enabled!(dc) = check(ccall(fn(:rsc_cloud_set_enabled), Int32, (Ptr{Cvoid}, Ptr{UInt64}), dc.h, dc.pc.isenabled.chunks))
pull_enabled!(dc) = check(ccall(fn(:rsc_cloud_get_enabled), Int32, (Ptr{Cvoid}, Ptr{UInt64}), dc.h, dc.pc.isenabled.chunks))

# ---- the operator API for built-in shapes ----------------------------------------------------------
"`scorecandidates!` for a vector of built-in shapes: one launch, returns [(ConfidenceInterval, inpoints)]."
function scorecandidates(dc::DeviceCloud, cands::Vector{<:FittedShape}, subsetID::Integer, params)
    C = length(cands)
    recs = RscCand[tocand(c) for c in cands]
    sub = dc.pc.subsets[subsetID]
    M = length(sub)
    words = cld(M, 32)
    counts = zeros(Int32, C)
    masks = zeros(UInt32, words, C)               # column c = row c of the C layout
    prm = Ref(toparams(params))
    check(ccall(fn(:rsc_score), Int32,
                (Ptr{Cvoid}, Ref{RscParams}, Ptr{RscCand}, Int32, Int32, Ptr{Int32}, Ptr{UInt32}),
                dc.h, prm, recs, C, subsetID - 1, counts, masks))
    map(1:C) do c
        bits = BitVector(undef, words * 32)
        copyto!(reinterpret(UInt32, bits.chunks), 1, view(masks, :, c), 1, words)  # same LSB-first layout
        inpoints = sub[findall(view(bits, 1:M))]
        (RANSAC.estimatescore(M, dc.pc.size, Int(counts[c])), inpoints)
    end
end

"`refit` + `invalidate_indexes!` (plane.jl:137-143 ... fitting.jl:197-202) on the device."
function refit_extract!(dc::DeviceCloud, s::FittedShape, params; disable::Bool=true)
    out = Vector{Int64}(undef, dc.pc.size)
    n = Ref{Int64}(0)
    prm = Ref(toparams(params))
    cand = Ref(tocand(s))
    check(ccall(fn(:rsc_refit_extract), Int32,
                (Ptr{Cvoid}, Ref{RscParams}, Ref{RscCand}, Ptr{Int64}, Ref{Int64}, Int32), dc.h, prm, cand, out, n, disable))
    resize!(out, n[])
    disable && pull_enabled!(dc)
    ExtractedShape(s, out .+ 1)
end

"""
Extension: inlier counts of `cands` -- the counts `scorecandidate` would give on the whole cloud
(`subset = 0`) or on subset `subset` (1-based, like the reference's `subsetID`) -- skipping the
(candidate, 128-point Morton tile) pairs that provably hold no compatible point (`rsc_score_culled`,
`rsc_score_culled_subset`).  The whole-cloud form builds the Morton order on first use; the subset form sorts a
copy of the subset on first use.  Returns `(counts, pairs_total, pairs_survived)`.
"""
function score_culled(dc::DeviceCloud, cands::Vector{<:FittedShape}, params; subset::Integer=0, octree_levels::Integer=11)
    prm = Ref(toparams(params))
    arr = [tocand(c) for c in cands]
    counts = Vector{Int32}(undef, length(arr))
    tot = Ref{Int64}(0); sur = Ref{Int64}(0); ms = Ref{Float64}(0.0)
    if subset > 0
        check(ccall(fn(:rsc_score_culled_subset), Int32,
                    (Ptr{Cvoid}, Ref{RscParams}, Ptr{RscCand}, Int32, Int32, Ptr{Int32}, Ref{Int64}, Ref{Int64}, Ref{Float64}),
                    dc.h, prm, arr, length(arr), subset - 1, counts, tot, sur, ms))
    else
        check(ccall(fn(:rsc_cloud_cells_levels), Int32, (Ptr{Cvoid},), dc.h) > 0 ? Int32(0) :
              ccall(fn(:rsc_cloud_build_cells), Int32, (Ptr{Cvoid}, Int32), dc.h, octree_levels))
        check(ccall(fn(:rsc_score_culled), Int32,
                    (Ptr{Cvoid}, Ref{RscParams}, Ptr{RscCand}, Int32, Ptr{Int32}, Ref{Int64}, Ref{Int64}, Ref{Float64}),
                    dc.h, prm, arr, length(arr), counts, tot, sur, ms))
    end
    Int.(counts), tot[], sur[]
end

"""
Extension: least-squares refit of `s` to the enabled points compatible with it inside `band` * eps (the
paper's refit, which RANSAC.jl leaves out: docs/src/ransac.md:163-169).  Returns
`(refined shape, points used, rms distance)`; follow it with `refit_extract!`.
"""
function refit_lsq(dc::DeviceCloud, s::FittedShape, params; band::Float64=3.0)
    prm = Ref(toparams(params))
    cand = Ref(tocand(s))
    out = Ref(tocand(s))
    n = Ref{Int64}(0)
    rms = Ref{Float64}(NaN)
    check(ccall(fn(:rsc_refit_lsq), Int32,
                (Ptr{Cvoid}, Ref{RscParams}, Ref{RscCand}, Float64, Ref{RscCand}, Ref{Int64}, Ref{Float64}),
                dc.h, prm, cand, band, out, n, rms))
    fromcand(out[]), n[], rms[]
end

"`forcefitshapes!` for S minimal sets given as a 3 x S matrix of (1-based) point indices."
function fit_batch(dc::DeviceCloud, idx::Matrix{Int}, params)
    S = size(idx, 2)
    prm = Ref(toparams(params))
    cap = S * length(params.iteration.shape_types)
    out = Vector{RscCand}(undef, cap)
    out_set = Vector{Int32}(undef, cap)
    n = Ref{Int32}(0)
    check(ccall(fn(:rsc_fit_batch), Int32,
                (Ptr{Cvoid}, Ref{RscParams}, Ptr{Int64}, Int32, Ptr{RscCand}, Ptr{Int32}, Ref{Int32}),
                dc.h, prm, Int64.(idx .- 1), S, out, out_set, n))
    [fromcand(out[i]) for i in 1:n[]], out_set[1:n[]] .+ 1
end

"""
    loop_with_sets(pc, params, sets)

RANSAC.jl's loop (iterations.jl:35-162) with the device doing the work of `forcefitshapes!`,
`scorecandidates!` and `refit` through the per-call ABI, on minimal sets given explicitly (`sets[k][i]` =
0-based index triple of set i of iteration k, or `nothing`): the form in which a run is comparable with
the package itself set for set (julia/make_golden.jl, test/runtests.jl).  Returns
`(extracted, extracted_at, iterations)`.
"""
function loop_with_sets(pc::RANSACCloud, params, sets)
    it = params.iteration
    dc = DeviceCloud(pc)
    shapes = FittedShape[]; scores = ConfidenceInterval[]; inpts = Vector{Int}[]
    extracted = ExtractedShape[]; extracted_at = Int[]
    cc = [0, 0, 0]
    iterations = 0
    for k in 1:it.itermax
        count(pc.isenabled) < it.τ && break
        iterations = k
        trip = [Int.(sets[k][i]) .+ 1 for i in 1:it.minsubsetN if k <= length(sets) && sets[k][i] !== nothing]
        cands = isempty(trip) ? FittedShape[] : fit_batch(dc, hcat(trip...), params)[1]
        cc[2] += length(cands)
        if !isempty(cands)
            for (c, (sc, ip)) in zip(cands, scorecandidates(dc, collect(FittedShape, cands), 1, params))
                push!(shapes, c); push!(scores, sc); push!(inpts, ip)
            end
        end
        cc[3] = k * it.minsubsetN
        cc[1] = length(shapes)
        if !isempty(shapes)
            best = RANSAC.findhighestscore(RANSAC.IterationCandidates(shapes, scores, inpts))
            scr = RANSAC.E(scores[best.index])
            if RANSAC.prob(scr, RANSAC.chooseS(cc, it.extract_s), pc.size, it.drawN) > it.prob_det
                ex = refit_extract!(dc, shapes[best.index], params)       # also clears pc.isenabled
                push!(extracted, ex); push!(extracted_at, k)
                deleteat!(shapes, best.index); deleteat!(scores, best.index); deleteat!(inpts, best.index)
                dead = [j for j in eachindex(inpts) if !all(pc.isenabled[inpts[j]])]
                deleteat!(shapes, dead); deleteat!(scores, dead); deleteat!(inpts, dead)
            end
        end
        RANSAC.prob(it.τ, RANSAC.chooseS(cc, it.terminate_s), pc.size, it.drawN) > it.prob_det && break
    end
    extracted, extracted_at, iterations
end

# ---- normal estimation (rsc_estimate_normals) ------------------------------------------------------------
"""
    estimate_normals(vertices; k=16, viewpoint=nothing) -> Vector{SVector{3,Float32}}

Oriented PCA normals of the `k` (3..32) nearest neighbours of every point, on the device (`rsc_estimate_normals`):
with a `viewpoint` (the sensor of a single scan) every normal faces it, without one the component of largest
magnitude is positive.  Non-finite points and collinear or coincident neighbourhoods get zero normals.  For a raw
scan: `RANSACCloud(V, estimate_normals(V; viewpoint=s), 2)`.
"""
function estimate_normals(vertices::Vector{SVector{3,Float32}}; k::Integer=16, viewpoint=nothing)
    nrm = Vector{SVector{3,Float32}}(undef, length(vertices))
    vp = viewpoint === nothing ? nothing : Float64[viewpoint[1], viewpoint[2], viewpoint[3]]
    GC.@preserve vertices nrm vp begin
        check(ccall(fn(:rsc_estimate_normals), Int32,
                    (Ptr{Cvoid}, Ptr{Float32}, Int64, Int32, Ptr{Float64}, Ptr{Float32}, Ptr{Int64}, Ptr{Int64}),
                    context(), Ptr{Float32}(pointer(vertices)), length(vertices), k,
                    vp === nothing ? Ptr{Float64}(C_NULL) : pointer(vp), Ptr{Float32}(pointer(nrm)),
                    Ptr{Int64}(C_NULL), Ptr{Int64}(C_NULL)))
    end
    nrm
end

"""
    orient_normals(vertices; normals=nothing, k=16) -> Vector{SVector{3,Float32}}

Normals with consistent signs for a cloud without one viewpoint (CAD or mesh samples, merged scans, photogrammetry),
on the device (`rsc_orient_normals`): signs propagate along the minimum spanning forest of the `k`-nearest-neighbour
graph weighted by 1 - |n_i . n_j|, each tree's highest point getting a positive z component.  `normals` are oriented
as given (each row negated or not); `nothing` estimates them first as `estimate_normals(vertices; k)` does.  Points
with a non-finite coordinate or a zero or non-finite normal are returned unchanged.
`RANSACCloud(V, orient_normals(V), 2)`.
"""
function orient_normals(vertices::Vector{SVector{3,Float32}}; normals=nothing, k::Integer=16)
    nrm = Vector{SVector{3,Float32}}(undef, length(vertices))
    nin = normals === nothing ? nothing : convert(Vector{SVector{3,Float32}}, normals)
    nin === nothing || length(nin) == length(vertices) || throw(ArgumentError("normals must match vertices"))
    GC.@preserve vertices nrm nin begin
        check(ccall(fn(:rsc_orient_normals), Int32,
                    (Ptr{Cvoid}, Ptr{Float32}, Int64, Int32, Ptr{Float32}, Ptr{Float32}, Ptr{Int64}, Ptr{Int64}),
                    context(), Ptr{Float32}(pointer(vertices)), length(vertices), k,
                    nin === nothing ? Ptr{Float32}(C_NULL) : Ptr{Float32}(pointer(nin)), Ptr{Float32}(pointer(nrm)),
                    Ptr{Int64}(C_NULL), Ptr{Int64}(C_NULL)))
    end
    nrm
end

# ---- user-defined shapes on the device (include/rsc.h "user-defined shapes") -----------------------------
"""
    compile_user_shape(src::String) -> type id

Compiles a user shape's CUDA source (it defines `rsc_user_compatible`) with NVRTC on the context's device;
the same source returns the same id (>= RSC_USER_TYPE0 = 16).  A compile error raises with NVRTC's log.
"""
function compile_user_shape(src::String)
    id = Ref{Int32}(0)
    check(ccall(fn(:rsc_user_shape_compile), Int32, (Ptr{Cvoid}, Ptr{UInt8}, Int64, Ref{Int32}),
                context(), src, sizeof(src), id))
    id[]
end

"""
    user_score!(counts, masks, dc, recs, k, subsetID)

`scorecandidate` for user-shape records of ONE compiled type (`RscCand(type_id, outwards, p)`): compatible
enabled points of subset `subsetID` (1-based; 0 = the whole cloud) into `counts`, and their bitmasks into
`masks` (`cld(M, 32)` x C `UInt32`, or `nothing`).  `k` = up to 8 constants (e.g. ϵ, cos α).
"""
function user_score!(counts::Vector{Int32}, masks::Union{Nothing,Matrix{UInt32}}, dc::DeviceCloud, recs::Vector{RscCand},
                     k::Vector{Float64}, subsetID::Integer)
    check(ccall(fn(:rsc_user_score), Int32,
                (Ptr{Cvoid}, Ptr{Float64}, Int32, Ptr{RscCand}, Int32, Int32, Ptr{Int32}, Ptr{UInt32}),
                dc.h, k, length(k), recs, length(recs), subsetID - 1, counts,
                masks === nothing ? Ptr{UInt32}(C_NULL) : masks))
    counts
end

"`refit` + `invalidate_indexes!` of a user-shape record on the device: 1-based inlier indices."
function user_refit_extract(dc::DeviceCloud, rec::RscCand, k::Vector{Float64}; disable::Bool=true)
    out = Vector{Int64}(undef, dc.pc.size)
    n = Ref{Int64}(0)
    check(ccall(fn(:rsc_user_refit_extract), Int32,
                (Ptr{Cvoid}, Ptr{Float64}, Int32, Ref{RscCand}, Ptr{Int64}, Ref{Int64}, Int32),
                dc.h, k, length(k), Ref(rec), out, n, disable))
    resize!(out, n[])
    disable && pull_enabled!(dc)
    out .+ 1
end

"""
    sample_fit_user(dc, params, order, seed, set0, S) -> (records, sets, idx)

`samplepointcloud4!` + `forcefitshapes!` for a fit order of built-in kinds and compiled user types that define
`rsc_user_fit` (`order::Vector{RscShapeSlot}`, at most 8, each type once): the sets `rsc_sample_fit` draws, the
candidates as `RscCand` records in (set, position in the order) order, their 1-based sets, and the drawn indices
(drawN x S, 1-based; a column starting with 0 is a failed sample).  An empty order only draws: the sampler of a
Julia plug-in host loop whose shapes still fit in Julia.
"""
function sample_fit_user(dc::DeviceCloud, params, order::Vector{RscShapeSlot}, seed::Integer, set0::Integer, S::Integer)
    prm = Ref(toparams(params))
    cap = max(S * length(order), 1)
    out = Vector{RscCand}(undef, cap)
    out_set = Vector{Int32}(undef, cap)
    idx = Matrix{Int64}(undef, prm[].drawN, S)
    n = Ref{Int32}(0)
    check(ccall(fn(:rsc_sample_fit_user), Int32,
                (Ptr{Cvoid}, Ref{RscParams}, Ptr{Cvoid}, Int32, UInt64, UInt64, Int32, Ptr{RscCand}, Ptr{Int32}, Ptr{Int64}, Ref{Int32}),
                dc.h, prm, order, length(order), seed, set0, S, out, out_set, idx, n))
    out[1:n[]], out_set[1:n[]] .+ 1, idx .+ 1
end

"""
    ransac_user(dc, params, order; seed=1234) -> (records, inlier lists, seconds)

The whole device loop (`rsc_ransac_run_user`) for a fit order of built-in kinds and user types with
`rsc_user_fit`: the extracted shapes as `RscCand` records (user records under their type ids, for the caller to
turn back into its own types) and their 1-based inlier lists.  No extension switch; not for sharded or ranged
clouds.
"""
function ransac_user(dc::DeviceCloud, params, order::Vector{RscShapeSlot}; seed::Integer=1234)
    prm = Ref(toparams(params))
    run = Ref{Ptr{Cvoid}}(C_NULL)
    check(ccall(fn(:rsc_ransac_run_user), Int32, (Ptr{Cvoid}, Ref{RscParams}, Ptr{Cvoid}, Int32, UInt64, Ref{Ptr{Cvoid}}),
                dc.h, prm, order, length(order), seed, run))
    recs = RscCand[]; lists = Vector{Int}[]
    try
        for i in 0:ccall(fn(:rsc_run_nshapes), Int32, (Ptr{Cvoid},), run[])-1
            c = Ref{RscCand}()
            n = Ref{Int64}(0)
            check(ccall(fn(:rsc_run_shape), Int32, (Ptr{Cvoid}, Int32, Ref{RscCand}, Ref{Int64}), run[], i, c, n))
            idx = Vector{Int64}(undef, n[])
            n[] > 0 && check(ccall(fn(:rsc_run_inpoints), Int32, (Ptr{Cvoid}, Int32, Ptr{Int64}), run[], i, idx))
            push!(recs, c[]); push!(lists, idx .+ 1)
        end
        secs = ccall(fn(:rsc_run_seconds), Float64, (Ptr{Cvoid},), run[])
        pull_enabled!(dc)
        return recs, lists, secs
    finally
        ccall(fn(:rsc_run_destroy), Cvoid, (Ptr{Cvoid},), run[])
    end
end

# ---- one process per GPU: sharded storage (include/rsc.h "point-range sharding") ---------------------
"rank 0: the 128-byte NCCL id to hand to the other ranks (MPI.jl bcast, a socket, a file)"
function comm_unique_id()
    id = zeros(UInt8, 128)
    rc = ccall(fn(:rsc_comm_unique_id), Int32, (Ptr{UInt8},), id)
    rc == 0 || error("rsc_comm_unique_id failed ($rc): libnccl.so.2 not loadable?")
    id
end
"every rank: NCCL communicator inside the library (collective)"
comm_init(id::Vector{UInt8}, rank::Integer, nranks::Integer) =
    check(ccall(fn(:rsc_ctx_comm_init), Int32, (Ptr{Cvoid}, Ptr{UInt8}, Int32, Int32), context(), id, rank, nranks))

"""
    ransac(pc, params, setenabled; reset_rand=false, seed=1234, sampler=:root, octree_levels=8,
           progressive=false, lsq=false)

Drop-in for `RANSAC.ransac` when every entry of `params.iteration.shape_types` is a built-in shape:
the whole loop of iterations.jl:35-162 runs inside one `ccall`.  Otherwise falls back to
`RANSAC.ransac` (user-defined shapes run their own Julia methods).

`sampler=:octree` (extension) draws the minimal sets from level-weighted octree cells -- what
samplepointcloud4!/updatelevelweight are written for -- instead of from the root cell, which is what
the shipped package always does (levelweight/levelscore are swapped in the constructor, octree.jl:82-84).
The final weights/scores are written back to `pc.levelweight` / `pc.levelscore` when their length fits.
`progressive=true` (extension) refines overlapping confidence intervals on the subsets 2..r before each
extraction test -- the "TODO: refine if best.overlap" of iterations.jl:110; `lsq=true` (extension) refits
the best candidate by least squares to the compatible points within 3 eps before extracting it
(docs/src/ransac.md:163-169).
"""
function ransac(pc::RANSACCloud, params, setenabled::Bool; reset_rand=false, seed::Integer=1234, sampler::Symbol=:root,
                octree_levels::Integer=8, progressive::Bool=false, lsq::Bool=false)
    all(t -> haskey(KIND, t), params.iteration.shape_types) || return RANSAC.ransac(pc, params, setenabled; reset_rand=reset_rand)
    setenabled && fill!(pc.isenabled, true)
    dc = DeviceCloud(pc)
    run = Ref{Ptr{Cvoid}}(C_NULL)
    p0 = toparams(params)
    if sampler == :octree
        check(ccall(fn(:rsc_cloud_build_cells), Int32, (Ptr{Cvoid}, Int32), dc.h, octree_levels))
        p0 = RscParams((f === :compat_flags ? (p0.compat_flags | UInt32(2)) : getfield(p0, f) for f in fieldnames(RscParams))...)  # RSC_SAMPLER_OCTREE
    end
    withflag(p, bit) = RscParams((f === :compat_flags ? (p.compat_flags | UInt32(bit)) : getfield(p, f) for f in fieldnames(RscParams))...)
    if progressive   # RSC_SCORE_PROGRESSIVE: every subset must be on the device (subset 1 already is)
        for j in 2:length(pc.subsets)
            idx = Int64.(pc.subsets[j] .- 1)
            check(ccall(fn(:rsc_cloud_set_subset), Int32, (Ptr{Cvoid}, Int32, Ptr{Int64}, Int64), dc.h, j - 1, idx, length(idx)))
        end
        p0 = withflag(p0, 16)
    end
    lsq && (p0 = withflag(p0, 8))   # RSC_REFIT_LSQ
    prm = Ref(p0)
    check(ccall(fn(:rsc_ransac_run), Int32, (Ptr{Cvoid}, Ref{RscParams}, UInt64, Ref{Ptr{Cvoid}}),
                dc.h, prm, reset_rand ? 1234 : seed, run))
    extracted = ExtractedShape[]
    try
        for i in 0:ccall(fn(:rsc_run_nshapes), Int32, (Ptr{Cvoid},), run[])-1
            c = Ref{RscCand}()
            n = Ref{Int64}(0)
            check(ccall(fn(:rsc_run_shape), Int32, (Ptr{Cvoid}, Int32, Ref{RscCand}, Ref{Int64}), run[], i, c, n))
            idx = Vector{Int64}(undef, n[])
            n[] > 0 && check(ccall(fn(:rsc_run_inpoints), Int32, (Ptr{Cvoid}, Int32, Ptr{Int64}), run[], i, idx))
            push!(extracted, ExtractedShape(fromcand(c[]), idx .+ 1))
        end
        secs = ccall(fn(:rsc_run_seconds), Float64, (Ptr{Cvoid},), run[])
        lw = zeros(Float64, 11); ls = zeros(Float64, 11)
        nl = ccall(fn(:rsc_run_levelweight), Int32, (Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}), run[], lw, ls)
        if nl > 0 && length(pc.levelweight) == nl
            pc.levelweight .= lw[1:nl]; pc.levelscore .= ls[1:nl]
        end
        pull_enabled!(dc)
        return extracted, trunc(secs, digits=2)
    finally
        ccall(fn(:rsc_run_destroy), Cvoid, (Ptr{Cvoid},), run[])
    end
end

end # module
