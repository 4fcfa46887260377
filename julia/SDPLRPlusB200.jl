# SDPLRPlusB200.jl -- thin `ccall` shim that plugs libsdplrp_b200.so into an UNMODIFIED SDPLRPlus.jl.
#
# NOT EXECUTED IN THIS REPOSITORY'S CI: neither the build container nor the GPU box has a Julia toolchain (DESIGN.md
# section 1), so this file has never been parsed by Julia.  It is written against the reference sources as they are
# (signatures cited per method); the same control flow, through the same C entry points, is exercised by
# sdplrplus.jl_b200/solver.py (ctypes) in tests/ and bench.py.  tests/test_julia_shim.py keeps the ccall signatures in
# step with include/sdplrp_b200.h.
#
# How it works.  `_sdplr` (src/sdplr.jl:140-449) is duck-typed over (data, var, aux): `var.Rt` / `var.Gt` have the type
# parameter TR of `SolverVars{Ti,Tv,TR<:AbstractArray{Tv}}` (src/structs.jl:194-196) and `aux` is untyped.  This module
# supplies
#   * `DevMat <: AbstractMatrix{Float64}`: a name for an r x n matrix that lives on the GPU (R, G, the direction, an L-BFGS
#     slot), used as TR.  The generic calls `_sdplr` makes on such arrays -- `similar`, `zero`, `deepcopy`, `dot`, `norm`,
#     `BLAS.scal!`, `copyto!`, `axpy!`, `.= 0` -- are methods that either do nothing (the fused entry point already did the
#     work) or return the scalar the previous entry point produced;
#   * `B200Auxiliary`: the opaque handle as `aux`;
#   * methods of the seam functions (SURVEY.md 8b) `fg!`, `g!`, `lbfgs_dir!`, `lbfgs_update!`, `linesearch!`,
#     `linesearch_armijo!`, `dual_obj`, `rank_update!`, `DIMACS_errors`, `SDP_S_eigval` for (`SolverVars{..,DevMat}`,
#     `B200Auxiliary`), each a ccall or two.
# The two places where `_sdplr` works on host vectors inline are served by mirrors, so NO patch of the reference is needed:
#   * `norm(var.primal_vio, 2)` (src/sdplr.jl:230-234): `g!` / `fg!` leave a host vector whose 2-norm is the device value;
#   * the dual update loop on `var.λ` / `var.primal_vio_raw` (src/sdplr.jl:358-362): `dual_obj` (which always precedes it,
#     src/sdplr.jl:311-321) downloads both vectors, and the next `fg!` uploads `var.λ` and `var.σ[]`.
#
#     using SDPLRPlus, SDPLRPlusB200
#     res = SDPLRPlusB200.sdplr(C, As, b, r; ptol = 1e-2, objtol = 1e-2, prior_trace_bound = n)
#
# (same signature, keyword handling and result Dict as SDPLRPlus.sdplr, src/sdplr.jl:91-138, 426-448).
module SDPLRPlusB200

using LinearAlgebra, SparseArrays
import SDPLRPlus
import SDPLRPlus: SDPData, SolverVars, SolverStats, BurerMonteiroConfig, SymLowRankMatrix, LBFGSHistory,
    fg!, g!, linesearch!, linesearch_armijo!, lbfgs_dir!, lbfgs_update!, dual_obj, rank_update!, side_dimension,
    barvinok_pataki, set_rank!, _sdplr

const LIB = get(ENV, "SDPLRP_B200_LIB", joinpath(@__DIR__, "..", "sdplrplus.jl_b200", "libsdplrp_b200.so"))

# ids of include/sdplrp_b200.h
const MAT_R, MAT_G, MAT_D = Cint(0), Cint(1), Cint(2)
const MAT_HIST = Cint(-1)      # an L-BFGS slot: owned by the library, never addressed from Julia
const VEC_LAMBDA, VEC_LAMBDA_UB, VEC_B, VEC_PVIO_RAW, VEC_Y, VEC_PVIO_LB, VEC_A_RD, VEC_A_DD = Cint.(0:7)

struct B200Error <: Exception
    code::Int32
    msg::String
end

# One handle per GPU.  The scalars the fused entry points return are kept here until `_sdplr` asks for them through
# `dot` / `norm` (src/sdplr.jl:201, 224-234).
mutable struct Handle
    ptr::Ptr{Cvoid}
    gnorm2::Float64      # ||G||_F^2 of the last g! / fg!
    descent::Float64     # dot(dirt, Gt) of the last lbfgs_dir!
    stepped::Bool        # a line search chose α: the caller's axpy!(α, dirt, Rt) is a no-op, the step runs fused with g!
    pending_alpha::Float64   # that α, until g! issues sdplrp_step_g
    function Handle(device::Integer=0)
        out = Ref{Ptr{Cvoid}}(C_NULL)
        rc = ccall((:sdplrp_create, LIB), Int32, (Int32, Int32, Int32, Ptr{Cvoid}, Ref{Ptr{Cvoid}}), device, 0, 1, C_NULL, out)
        rc == 0 || throw(B200Error(rc, unsafe_string(ccall((:sdplrp_error_string, LIB), Cstring, (Int32,), rc))))
        h = new(out[], 0.0, 0.0, false, NaN)
        finalizer(x -> ccall((:sdplrp_destroy, LIB), Int32, (Ptr{Cvoid},), x.ptr), h)
        return h
    end
end

@inline function check(h::Handle, rc::Int32)
    rc == 0 && return nothing
    throw(B200Error(rc, unsafe_string(ccall((:sdplrp_last_error, LIB), Cstring, (Ptr{Cvoid},), h.ptr))))
end

"""
Device-backed replacement of `SolverAuxiliary` (src/structs.jl:274-361): the aggregated pattern and every
index map of `preprocess_sparsecons` are built on the GPU by `sdplrp_preprocess`.
"""
struct B200Auxiliary
    h::Handle
    n::Int
    m::Int
end
side_dimension(aux::B200Auxiliary) = aux.n   # src/structs.jl:363

"""
Concatenate the sparse matrices in `findnz` order exactly as `SolverAuxiliary` walks them
(src/structs.jl:303-332): sparse / Diagonal `A_i` in order of appearance, then `C` if sparse;
`SymLowRankMatrix` constraints are registered separately.
"""
function B200Auxiliary(data::SDPData; device=0)
    h = Handle(device)
    I, J, V, off, gids = Int64[], Int64[], Float64[], Int64[0], Int64[]
    lowrank = Tuple{Int,Any}[]
    add!(A, gid) = begin
        A isa Diagonal && (A = sparse(A))
        if A isa SymLowRankMatrix
            push!(lowrank, (gid, A))
        else
            i, j, v = findnz(A)      # CSC: column-major; COO: stored order
            append!(I, i); append!(J, j); append!(V, v)
            push!(off, length(I)); push!(gids, gid)
        end
    end
    for (i, A) in enumerate(data.As); add!(A, i); end
    add!(data.C, data.m + 1)
    GC.@preserve off I J V gids check(h, ccall((:sdplrp_preprocess, LIB), Int32,
        (Ptr{Cvoid}, Int64, Int64, Int64, Ptr{Int64}, Ptr{Int64}, Ptr{Int64}, Ptr{Float64}, Ptr{Int64}),
        h.ptr, data.n, data.m, length(gids), off, I, J, V, gids))
    for (gid, A) in lowrank
        B = Matrix{Float64}(A.B); D = Vector{Float64}(A.D.diag)
        GC.@preserve B D check(h, ccall((:sdplrp_add_symlowrank, LIB), Int32,
            (Ptr{Cvoid}, Int64, Int64, Ptr{Float64}, Ptr{Float64}), h.ptr, gid, size(B, 2), B, D))
    end
    bvec = Vector{Float64}(data.b)
    ineq = UInt8.(data.constraint_types)
    GC.@preserve bvec ineq check(h, ccall((:sdplrp_set_problem, LIB), Int32, (Ptr{Cvoid}, Ptr{Float64}, Ptr{UInt8}),
        h.ptr, bvec, data.has_inequalities ? pointer(ineq) : Ptr{UInt8}(C_NULL)))
    return B200Auxiliary(h, data.n, data.m)
end

"""
`DevMat` names an r x n matrix that lives on the device (`id` = SDPLRP_MAT_*, or MAT_HIST for an L-BFGS slot).  It is the
`TR` of `SolverVars{Ti,Tv,TR}` and the array type `lbfgs_init` stores in its `LBFGSVector`s (src/lbfgs.jl:35-47 builds them
with `zero(R)`).  No BLAS-1 call `_sdplr` makes on such arrays moves data.
"""
struct DevMat <: AbstractMatrix{Float64}
    h::Handle
    id::Cint
    r::Int
    n::Int
end
Base.size(A::DevMat) = (A.r, A.n)
Base.getindex(A::DevMat, i::Int, j::Int) = Array(A)[i, j]     # debugging only: downloads the matrix
function Base.Array(A::DevMat)
    A.id == MAT_HIST && error("L-BFGS slots are owned by the library")
    out = Matrix{Float64}(undef, A.r, A.n)
    GC.@preserve out check(A.h, ccall((:sdplrp_download_mat, LIB), Int32, (Ptr{Cvoid}, Cint, Ptr{Float64}), A.h.ptr, A.id, out))
    return out
end
Base.Matrix(A::DevMat) = Array(A)
upload!(A::DevMat, X::Matrix{Float64}) =
    GC.@preserve X check(A.h, ccall((:sdplrp_upload_mat, LIB), Int32, (Ptr{Cvoid}, Cint, Ptr{Float64}), A.h.ptr, A.id, X))

# `dirt = similar(var.Rt)` (src/sdplr.jl:176, 381): the direction array of the library
Base.similar(A::DevMat) = DevMat(A.h, MAT_D, A.r, A.n)
Base.similar(A::DevMat, ::Type{Float64}) = similar(A)
Base.similar(A::DevMat, ::Type{Float64}, dims::Dims{2}) = DevMat(A.h, MAT_D, dims[1], dims[2])
# `zero(R)` inside lbfgs_init (src/lbfgs.jl:41): the history lives in the library (sdplrp_set_rank allocated it)
Base.zero(A::DevMat) = DevMat(A.h, MAT_HIST, A.r, A.n)
# `Rt0 = deepcopy(var.Rt)` (src/sdplr.jl:153-154): the start point as a host matrix, as the reference returns it
Base.deepcopy_internal(A::DevMat, ::IdDict) = Array(A)
# `lbfgshis.vecs[i].s .= 0` of lbfgs_clear! (src/lbfgs.jl:52-59): broadcasting a scalar into an array lowers to fill!
function Base.fill!(A::DevMat, x)
    (A.id == MAT_HIST && iszero(x)) || error("DevMat only supports zero-filling the L-BFGS history")
    check(A.h, ccall((:sdplrp_lbfgs_clear, LIB), Int32, (Ptr{Cvoid},), A.h.ptr))   # idempotent: 2h calls per lbfgs_clear!, microseconds each
    return A
end

# src/sdplr.jl:201  descent = dot(dirt, var.Gt)
LinearAlgebra.dot(dirt::DevMat, Gt::DevMat) = dirt.h.descent
# src/sdplr.jl:224-228  norm(var.Gt, 2)
LinearAlgebra.norm(G::DevMat, p::Real=2) = (p == 2 || error("DevMat: only the Frobenius norm is kept"); sqrt(G.h.gnorm2))
# src/sdplr.jl:202-205  BLAS.scal!(-1, var.Gt); copyto!(dirt, var.Gt)  -- one entry point does both
LinearAlgebra.BLAS.scal!(a::Float64, G::DevMat) = (a == -1.0 || error("DevMat: scal! is only the sign flip of the fallback"); G)
function Base.copyto!(dirt::DevMat, G::DevMat)
    check(G.h, ccall((:sdplrp_use_gradient_direction, LIB), Int32, (Ptr{Cvoid},), G.h.ptr))
    return dirt
end
# src/sdplr.jl:219  axpy!(α, dirt, var.Rt): applied by the fused step + gradient pass that the following g! issues
function LinearAlgebra.axpy!(α, dirt::DevMat, Rt::DevMat)
    (Rt.h.stepped && α == Rt.h.pending_alpha) || error("axpy!(α, dirt, Rt) on device matrices is only valid right after a line search, with its α")
    Rt.h.stepped = false
    return Rt
end

"""
SolverVars whose Rt/Gt are device matrices.  The m-vectors stay host `Vector`s; they mirror device state at the points
where `_sdplr` reads them (see the header of this file).
"""
function device_vars(data::SDPData, aux::B200Auxiliary, r, config::BurerMonteiroConfig)
    host = SolverVars(data, r, config)                       # draws Rt0 / applies init_func exactly as the reference (src/structs.jl:225-240)
    h = aux.h
    check(h, ccall((:sdplrp_set_rank, LIB), Int32, (Ptr{Cvoid}, Int32, Int32), h.ptr, r, config.numlbfgsvecs))
    Rt, Gt = DevMat(h, MAT_R, r, data.n), DevMat(h, MAT_G, r, data.n)
    upload!(Rt, Matrix{Float64}(host.Rt))
    upload_vec(h, VEC_LAMBDA, host.λ)
    check(h, ccall((:sdplrp_set_sigma, LIB), Int32, (Ptr{Cvoid}, Float64), h.ptr, host.σ[]))
    return SolverVars(Rt, Gt, host.λ, host.λ_ub, host.r, host.σ, host.obj, host.y, host.primal_vio_raw,
        host.primal_vio_lb, host.primal_vio, host.A_RD, host.A_DD)
end
upload_vec(h::Handle, id::Cint, v::Vector{Float64}) =
    GC.@preserve v check(h, ccall((:sdplrp_upload_vec, LIB), Int32, (Ptr{Cvoid}, Cint, Ptr{Float64}, Int64), h.ptr, id, v, length(v)))
download_vec!(h::Handle, id::Cint, v::Vector{Float64}) =
    GC.@preserve v check(h, ccall((:sdplrp_download_vec, LIB), Int32, (Ptr{Cvoid}, Cint, Ptr{Float64}, Int64), h.ptr, id, v, length(v)))

# `norm(var.primal_vio, 2)` is evaluated on the host vector (src/sdplr.jl:230-234, src/coreop.jl:339-347): leave one with
# the device's value as its 2-norm
function mirror_pvio_norm!(var, pnorm2)
    fill!(var.primal_vio, 0.0)
    isempty(var.primal_vio) || (var.primal_vio[1] = sqrt(pnorm2))
    return nothing
end

# ---- seam functions (SURVEY.md 8b) for the device types -------------------------------------------------
# Every method below repeats the reference's own parametrisation with Tv = Float64 and the device types filled in, so that
# it is strictly more specific than the generic method it shadows (no dispatch ambiguity).
# src/coreop.jl:323-349  fg!(data, var, aux, normC, normb, config)
function fg!(data, var::SolverVars{Ti,Float64,DevMat}, aux::B200Auxiliary, normC::Float64, normb::Float64, config) where {Ti<:Integer}
    h = aux.h
    # λ and σ may have been changed on the host by the dual / penalty update of the previous major iteration
    # (src/sdplr.jl:358-368): the library's copies are refreshed here, once per major iteration
    upload_vec(h, VEC_LAMBDA, var.λ)
    check(h, ccall((:sdplrp_set_sigma, LIB), Int32, (Ptr{Cvoid}, Float64), h.ptr, var.σ[]))
    out = zeros(4)
    GC.@preserve out check(h, ccall((:sdplrp_fg, LIB), Int32, (Ptr{Cvoid}, Ptr{Float64}), h.ptr, out))
    var.obj[] = out[2]
    h.gnorm2 = out[3]
    mirror_pvio_norm!(var, out[4])
    grad_norm = config.gtol_mode == :relative ? sqrt(out[3]) / normC : sqrt(out[3])
    primal_vio_norm = config.ptol_mode == :relative ? sqrt(out[4]) / normb : sqrt(out[4])
    return out[1], grad_norm, primal_vio_norm
end

# src/coreop.jl:305-317  g!(var, aux).  Right after a line search it is the fused pass sdplrp_step_g: Rt += α dirt, the
# residual recurrence and obj (src/linesearch.jl:118-124), y, G and the two norms `_sdplr` takes next -- one row pass.
function g!(var::SolverVars{Ti,Float64,DevMat}, aux::B200Auxiliary) where {Ti<:Integer}
    h = aux.h
    if !isnan(h.pending_alpha)
        out = zeros(3)
        GC.@preserve out check(h, ccall((:sdplrp_step_g, LIB), Int32, (Ptr{Cvoid}, Float64, Ptr{Float64}), h.ptr, h.pending_alpha, out))
        h.pending_alpha = NaN
        var.obj[] = out[1]; h.gnorm2 = out[2]
        mirror_pvio_norm!(var, out[3])
    else
        gn2, pn2 = Ref(0.0), Ref(0.0)
        check(h, ccall((:sdplrp_g, LIB), Int32, (Ptr{Cvoid}, Ref{Float64}, Ref{Float64}), h.ptr, gn2, pn2))
        h.gnorm2 = gn2[]
        mirror_pvio_norm!(var, pn2[])
    end
    return 0
end

# src/lbfgs.jl:77-124  lbfgs_dir!(dir, lbfgshis, grad; negate=true); the descent dot product comes back with it
function lbfgs_dir!(dirt::DevMat, his::LBFGSHistory{Ti,Float64}, Gt::DevMat; negate::Bool=true) where {Ti<:Integer}
    negate || error("the device two-loop returns the negated direction, as _sdplr asks for")
    d = Ref(0.0)
    check(dirt.h, ccall((:sdplrp_lbfgs_dir, LIB), Int32, (Ptr{Cvoid}, Ref{Float64}), dirt.h.ptr, d))
    dirt.h.descent = d[]
    return nothing
end

# src/lbfgs.jl:129-149  lbfgs_update!(dir, lbfgshis, grad, stepsize)
function lbfgs_update!(dirt::DevMat, his::LBFGSHistory{Ti,Float64}, Gt::DevMat, α::Float64) where {Ti<:Integer}
    check(dirt.h, ccall((:sdplrp_lbfgs_update, LIB), Int32, (Ptr{Cvoid}, Float64), dirt.h.ptr, Float64(α)))
    return nothing
end

# src/linesearch.jl:4-127  linesearch!(var, aux, Dt; α_max): the two 𝒜 passes and the quartic coefficients on the device,
# the root selection of src/linesearch.jl:58-112 by sdplrp_pick_alpha (host code of the library, same candidate rule); the
# commit `primal_vio_raw += α(α A_DD + A_RD)`, obj (src/linesearch.jl:118-124) and `Rt += α Dt` are deferred to the g! that
# `_sdplr` calls next (src/sdplr.jl:219-221), where they run fused with the gradient (sdplrp_step_g)
function linesearch!(var::SolverVars{Ti,Float64,DevMat}, aux::B200Auxiliary, dirt::DevMat; α_max=1.0) where {Ti<:Integer}
    h = aux.h
    biquadratic = zeros(5)
    GC.@preserve biquadratic check(h, ccall((:sdplrp_linesearch_coeffs, LIB), Int32, (Ptr{Cvoid}, Ptr{Float64}), h.ptr, biquadratic))
    α, 𝓛 = Ref(0.0), Ref(0.0)
    rc = GC.@preserve biquadratic ccall((:sdplrp_pick_alpha, LIB), Int32, (Ptr{Float64}, Float64, Ref{Float64}, Ref{Float64}), biquadratic, Float64(α_max), α, 𝓛)
    rc == 0 || error("line search: the slope at 0 is positive (src/linesearch.jl:63-66)")
    h.pending_alpha = α[]; h.stepped = true       # the commit of src/linesearch.jl:118-124 runs fused with the next g!
    return α[], 𝓛[]
end

# src/linesearch.jl:139-191  linesearch_armijo!(var, aux, Dt; α_max): eval_AL and the slope are evaluated on the device for a
# batch of halvings at a time; the acceptance rule is the reference's
function linesearch_armijo!(var::SolverVars{Ti,Float64,DevMat}, aux::B200Auxiliary, dirt::DevMat; α_max=1.0) where {Ti<:Integer}
    h = aux.h
    biquadratic = zeros(5)
    GC.@preserve biquadratic check(h, ccall((:sdplrp_linesearch_coeffs, LIB), Int32, (Ptr{Cvoid}, Ptr{Float64}), h.ptr, biquadratic))
    evalAL(αs) = begin
        L = zeros(length(αs)); slope = Ref(0.0)
        GC.@preserve αs L check(h, ccall((:sdplrp_armijo_eval, LIB), Int32, (Ptr{Cvoid}, Ptr{Float64}, Int32, Ptr{Float64}, Ref{Float64}),
            h.ptr, αs, length(αs), L, slope))
        L, slope[]
    end
    L0v, slope = evalAL([0.0])
    L0, c = L0v[1], 1e-4
    αs = [Float64(α_max) / 2.0^k for k in 0:50]          # α_max and at most 50 halvings
    α, 𝓛 = αs[end], NaN
    found = false
    for s in 1:15:51
        blk = αs[s:min(s + 14, 51)]
        Lb, _ = evalAL(blk)
        k = findfirst(i -> Lb[i] <= L0 + c * blk[i] * slope, 1:length(blk))
        if k !== nothing
            α, 𝓛, found = blk[k], Lb[k], true
            break
        end
        𝓛 = Lb[end]
    end
    h.pending_alpha = α; h.stepped = true
    return α, 𝓛
end

# src/coreop.jl:376-415  dual_obj(data, var, aux, trace_bound, iter; highprecision)
function dual_obj(data, var::SolverVars{Ti,Float64,DevMat}, aux::B200Auxiliary, trace_bound::Float64, iter::Ti; highprecision::Bool=false) where {Ti<:Integer}
    h = aux.h
    v0 = randn(aux.n)                                        # src/coreop.jl:473: the start vector stays Julia's
    dual, lam, steps = Ref(0.0), Ref(0.0), Ref{Int64}(0)
    if highprecision   # SDP_S_eigval (GenericArpack symeigs, src/coreop.jl:386-400) -> thick-restart Lanczos on the device
        GC.@preserve v0 check(h, ccall((:sdplrp_dual_obj_highprecision, LIB), Int32,
            (Ptr{Cvoid}, Float64, Ptr{Float64}, UInt64, Ref{Float64}, Ref{Float64}, Ref{Int64}),
            h.ptr, Float64(trace_bound), v0, 0, dual, lam, steps))
    else
        GC.@preserve v0 check(h, ccall((:sdplrp_dual_obj, LIB), Int32,
            (Ptr{Cvoid}, Float64, Int64, Ptr{Float64}, UInt64, Ref{Float64}, Ref{Float64}, Ref{Int64}),
            h.ptr, Float64(trace_bound), Int64(iter), v0, 0, dual, lam, steps))
    end
    # what _sdplr reads on the host right after this call: var.y for best_λ (src/sdplr.jl:324), var.λ and
    # var.primal_vio_raw for the dual update loop (src/sdplr.jl:358-362)
    download_vec!(h, VEC_Y, var.y)
    download_vec!(h, VEC_PVIO_RAW, var.primal_vio_raw)
    download_vec!(h, VEC_LAMBDA, var.λ)
    return dual[], lam[]
end

# min(bp, 2r) clamped to the ranks sdplrp_set_rank accepts (r <= 256, odd r <= 128): the rule of sdplrp_solve and solver.py
function rank_after_update(bp::Integer, r::Integer)
    t = min(bp, 2r, 256)
    return (isodd(t) && t > 128) ? t - 1 : t
end

# src/coreop.jl:518-526  rank_update!(data, var, config): a fresh point of the new rank on the device
function rank_update!(data, var::SolverVars{Ti,Float64,DevMat}, config::BurerMonteiroConfig{Ti,Float64}) where {Ti<:Integer}
    newr = rank_after_update(barvinok_pataki(data), var.r[])
    set_rank!(data, newr)
    h = var.Rt.h
    return device_vars(data, B200Auxiliary(h, size(var.Rt, 2), length(var.λ)), newr, config)
end

"""
`SDP_S_eigval(var, aux, nevs, preprocessed; which=:SA, ncv, tol, maxiter)` (src/coreop.jl:351-374) on the S last assembled.
"""
function SDPLRPlus.SDP_S_eigval(var::SolverVars{Ti,Float64,DevMat}, aux::B200Auxiliary, nevs::Integer, preprocessed::Bool=false;
                                ncv=min(100, aux.n), tol=0.0, maxiter=1000000, kwargs...) where {Ti<:Integer}
    y = var.y
    preprocessed || GC.@preserve y check(aux.h, ccall((:sdplrp_At_preprocess, LIB), Int32, (Ptr{Cvoid}, Ptr{Float64}), aux.h.ptr, y))
    ev = zeros(nevs); v0 = randn(aux.n)
    dt = @elapsed GC.@preserve ev v0 check(aux.h, ccall((:sdplrp_S_eigval, LIB), Int32,
        (Ptr{Cvoid}, Int64, Int64, Float64, Int64, Ptr{Float64}, UInt64, Ptr{Float64}, Ptr{Float64}, Ptr{Int64}, Ptr{Int64}),
        aux.h.ptr, nevs, ncv, tol, maxiter, v0, 0, ev, C_NULL, C_NULL, C_NULL))
    return ev, dt
end

"""
`DIMACS_errors(data, var, aux)` (src/coreop.jl:426-453) in one call.
"""
function SDPLRPlus.DIMACS_errors(data, var::SolverVars{Ti,Float64,DevMat}, aux::B200Auxiliary) where {Ti<:Integer}
    errs = zeros(6); v0 = randn(aux.n)
    GC.@preserve errs v0 check(aux.h, ccall((:sdplrp_dimacs_errors, LIB), Int32,
        (Ptr{Cvoid}, Float64, Float64, Ptr{Float64}, UInt64, Ptr{Float64}),
        aux.h.ptr, norm(data.b, 2), norm(data.C, 2), v0, 0, errs))
    return errs
end

"""
    round_hyperplane(aux, K; r, G = nothing, seed = 0) -> (obj, sum, best, best_x, G_used)

Goemans-Williamson rounding of the current R (rank `r`) on the device: K candidates x_k = sign(R' g_k) (+1 on ties),
obj[k] = <C, x_k x_k'>, sum[k] = sum(x_k), `best` (1-based) the smallest obj, `best_x` its +-1 vector.  `G` (r x K, one
hyperplane per column) or, `nothing`, seeded standard normals (the same for every K and GPU count).  Reads R only.
"""
function round_hyperplane(aux::B200Auxiliary, K::Integer; r::Integer, G=nothing, seed=0)
    Gin = G === nothing ? Ptr{Float64}(C_NULL) : Matrix{Float64}(G)
    G === nothing || size(Gin) == (r, K) || throw(ArgumentError("G must be r x K"))
    G_used = zeros(r, K); obj = zeros(K); tot = zeros(K); best = Ref{Int64}(0); x = zeros(aux.n)
    GC.@preserve Gin G_used obj tot x check(aux.h, ccall((:sdplrp_round_hyperplane, LIB), Int32,
        (Ptr{Cvoid}, Int64, Ptr{Float64}, UInt64, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ref{Int64}, Ptr{Float64}),
        aux.h.ptr, K, Gin, UInt64(seed), G_used, obj, tot, best, x))
    return obj, tot, Int(best[]), x, G_used
end

"""
    round_local_search(aux, K; r, G = nothing, seed = 0, max_rounds = 1000)
        -> (obj_round, obj, sum, flips, rounds, best, best_x, G_used)

The K candidates of `round_hyperplane`, each refined on the device by parallel one-flip descent until no single vertex
flip lowers <C, xx'> (or `max_rounds` rounds).  `obj_round` are the objectives before the descent, `obj` after,
`rounds[k]` the last round that flipped candidate k (-1: stopped by `max_rounds`), `best` (1-based) the smallest `obj`
and `best_x` its +-1 vector.  Reads R only.
"""
function round_local_search(aux::B200Auxiliary, K::Integer; r::Integer, G=nothing, seed=0, max_rounds=1000)
    Gin = G === nothing ? Ptr{Float64}(C_NULL) : Matrix{Float64}(G)
    G === nothing || size(Gin) == (r, K) || throw(ArgumentError("G must be r x K"))
    G_used = zeros(r, K); obj0 = zeros(K); obj = zeros(K); tot = zeros(K); flips = zeros(Int64, K); rounds = zeros(Int64, K)
    best = Ref{Int64}(0); x = zeros(aux.n)
    GC.@preserve Gin G_used obj0 obj tot flips rounds x check(aux.h, ccall((:sdplrp_round_local_search, LIB), Int32,
        (Ptr{Cvoid}, Int64, Ptr{Float64}, UInt64, Int64, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Int64},
         Ptr{Int64}, Ref{Int64}, Ptr{Float64}),
        aux.h.ptr, K, Gin, UInt64(seed), Int64(max_rounds), G_used, obj0, obj, tot, flips, rounds, best, x))
    return obj0, obj, tot, flips, rounds, Int(best[]), x, G_used
end

function apply_kwargs!(config, kwargs)
    for (k, v) in kwargs
        hasfield(BurerMonteiroConfig, Symbol(k)) ? setfield!(config, Symbol(k), v) : @error "Unrecognized keyword argument $k"
    end
    return config
end
make_data(C, As, b, constraint_types) = constraint_types === nothing ? SDPData(C, As, b) : SDPData(C, As, b, constraint_types)

"""
    sdplr(C, As, b, r; constraint_types = nothing, config = BurerMonteiroConfig{Int,Float64}(), kwargs...)

Same contract as `SDPLRPlus.sdplr` (src/sdplr.jl:91-138); the hot path runs on the B200.
"""
function sdplr(C::AbstractMatrix{Float64}, As::Vector, b::Vector{Float64}, r::Int;
               constraint_types::Union{Nothing,AbstractVector{Bool}}=nothing,
               config::BurerMonteiroConfig{Int,Float64}=BurerMonteiroConfig{Int,Float64}(), device=0, kwargs...)
    apply_kwargs!(config, kwargs)
    local data, aux, var
    preprocess_dt = @elapsed begin
        data = make_data(C, As, b, constraint_types)
        aux = B200Auxiliary(data; device)
        var = device_vars(data, aux, r, config)
    end
    ans = _sdplr(data, var, aux, SolverStats{Float64}(), config)
    ans["Rt"] = Array(ans["Rt"])                 # the reference returns host matrices
    ans["preprocess_time"] = preprocess_dt
    ans["totaltime"] += preprocess_dt
    ans["aux"] = aux                             # R stays on the device: round_hyperplane(ans["aux"], K; r = ans["r"])
    return ans
end

# ---- the whole solve as ONE call (SURVEY.md 8f/f1): the native driver of csrc/driver.cu runs the loop of
# src/sdplr.jl:140-449 inside the library.  Field order = sdplrp_config / sdplrp_result of include/sdplrp_b200.h.
struct NativeConfig
    ptol::Float64; gtol::Float64; objtol::Float64; sigma_0::Float64; sigmafac::Float64; maxtime::Float64; printfreq::Float64
    fprec::Float64; prior_trace_bound::Float64; alpha_max::Float64
    maxmajoriter::Int64; maxiter::Int64; numlbfgsvecs::Int64; rankupd_tol::Int64; printlevel::Int64
    gtol_relative::Int64; ptol_relative::Int64; objtol_relative::Int64; eval_DIMACS_errs::Int64; eigval_highprecision::Int64
    seed::UInt64
end
struct NativeResult
    sigma::Float64; grad_norm::Float64; primal_vio::Float64; obj::Float64; L::Float64; max_dual_value::Float64
    min_duality_gap::Float64; totaltime::Float64; dual_time::Float64; primaltime::Float64; DIMACS_time::Float64
    DIMACS_errs::NTuple{6,Float64}
    iter::Int64; majoriter::Int64; lanczos_steps::Int64; r::Int64; status::Int64
end
# the *_mode fields of BurerMonteiroConfig are Symbols (src/options.jl:21-23)
NativeConfig(c::BurerMonteiroConfig; seed=0) = NativeConfig(c.ptol, c.gtol, c.objtol, c.σ_0, c.σfac, c.maxtime, c.printfreq, c.fprec,
    c.prior_trace_bound, 1.0, c.maxmajoriter, c.maxiter, c.numlbfgsvecs, c.rankupd_tol, c.printlevel,
    Int64(c.gtol_mode == :relative), Int64(c.ptol_mode == :relative), Int64(c.objtol_mode == :relative),
    Int64(c.eval_DIMACS_errs), Int64(c.eigval_highprecision == true), UInt64(seed))

"""
    sdplr_native(C, As, b, r; constraint_types = nothing, kwargs...)

`sdplr` with the outer loop inside the library (`sdplrp_solve`).  Rt0 / λ0 come from `SolverVars(data, r, config)` as
in the reference; the eigenvalue start vectors and the random point of a rank update come from the device generator.
"""
function sdplr_native(C::AbstractMatrix{Float64}, As::Vector, b::Vector{Float64}, r::Int;
                      constraint_types::Union{Nothing,AbstractVector{Bool}}=nothing,
                      config::BurerMonteiroConfig{Int,Float64}=BurerMonteiroConfig{Int,Float64}(), device=0, seed=0, kwargs...)
    apply_kwargs!(config, kwargs)
    data = make_data(C, As, b, constraint_types)
    aux = B200Auxiliary(data; device)
    host = SolverVars(data, r, config)
    Rt0 = Matrix{Float64}(host.Rt); λ0 = Vector{Float64}(host.λ)
    cfg = Ref(NativeConfig(config; seed)); res = Ref{NativeResult}(); best = zeros(data.m + 1)
    GC.@preserve Rt0 λ0 best check(aux.h, ccall((:sdplrp_solve, LIB), Int32,
        (Ptr{Cvoid}, Ref{NativeConfig}, Int64, Ptr{Float64}, Ptr{Float64}, Float64, Float64, Ref{NativeResult}, Ptr{Float64}),
        aux.h.ptr, cfg, r, Rt0, λ0, norm(b, 2), norm(C, 2), res, best))
    R = res[]
    Rt = Array(DevMat(aux.h, MAT_R, Int(R.r), data.n))
    return Dict("Rt" => Rt, "lambda" => best, "Rt0" => Rt0, "lambda0" => λ0, "sigma" => R.sigma, "grad_norm" => R.grad_norm,
        "primal_vio" => R.primal_vio, "obj" => R.obj, "max_dual_value" => R.max_dual_value, "min_duality_gap" => R.min_duality_gap,
        "totaltime" => R.totaltime, "dual_time" => R.dual_time, "primaltime" => R.primaltime, "iter" => R.iter,
        "majoriter" => R.majoriter, "DIMACS_errs" => collect(R.DIMACS_errs), "ptol" => config.ptol, "objtol" => config.objtol,
        "fprec" => config.fprec, "rankupd_tol" => config.rankupd_tol, "r" => Int(R.r), "aux" => aux)
end

end # module
