# LSMB200.jl — ccall glue that puts liblsm_b200.so behind LevelSetMethods.jl's OWN dispatch seam.
#
# NOT EXECUTED IN THIS REPOSITORY'S CI: the build / GPU images have no Julia (SURVEY.md headline 3).  It is written against
# include/lsm_b200.h and mirrors what the Python host mirror (levelsetmethods.jl_b200/api.py) does through ctypes, which IS
# tested on the GPU (tests/test_gpu_parity.py::test_hooks_update_func_and_incremental and the multi-GPU tests).
#
# Usage (the reference's own entry point; nothing in LevelSetMethods changes):
#
#     using LevelSetMethods, LSMB200
#     ϕ  = LSMB200.to_device(MeshField(x -> hypot(x...) - 0.5, grid; bc = NeumannBC()))
#     u  = LSMB200.TimeScaled(MeshField(x -> SVector(-x[2], x[1]), grid), LSMB200.CosScale(3.0))     # stored field × cos(π t / 3)
#     eq = LevelSetEquation(; terms = AdvectionTerm(u, WENO5()), ic = ϕ, integrator = RK3())
#     integrate!(eq, tf)                       # LevelSetMethods.integrate! → _integrate!(…, ϕ::DeviceMeshField, …) below
#     values(current_state(eq))                # lazy download
#
# Seam (SURVEY.md §8b).  `integrate!` (src/levelsetequation.jl:194-203) dispatches on the state type to
#   _integrate!(ls, ϕ::AbstractMeshField, integrator, terms, tc, tf, Δt_max, prehook, posthook)      src/timestepping.jl:101
# whose body calls  _alloc_buffers (:126,141,168), update_term! (levelsetterms.jl:14), compute_cfl (levelsetterms.jl:22),
# _advance! (:128,143,170) and update_band! (meshfield.jl:553).  This module adds a device-backed state type
# `DeviceMeshField <: AbstractMeshField` (meshfield.jl:33) and methods of exactly those functions for it:
#   * no host hooks, device-resident coefficients  → ONE ccall, lsm_integrate runs the whole loop;
#   * prehook / posthook / non-default update_func → the reference's generic loop runs unchanged, each of its calls landing
#     on a method below (compute_cfl → lsm_compute_cfl, _advance! → lsm_stage per stage with update_term! in between, seeing
#     the CURRENT stage field through a lazily downloaded mirror of the library's stage buffer).
module LSMB200

using LevelSetMethods
import LevelSetMethods as LSM
using StaticArrays

const LIB = get(ENV, "LSM_B200_LIB", joinpath(@__DIR__, "..", "liblsm_b200.so"))

# ---- enums of include/lsm_b200.h -------------------------------------------------------------------
const LSM_OK, LSM_ERR_ARG, LSM_ERR_CFL, LSM_ERR_TIME, LSM_ERR_BC = Int32(0), Int32(1), Int32(2), Int32(3), Int32(4)
const F32, F64 = Int32(0), Int32(1)
const BC_PERIODIC, BC_EXTRAP, BC_SYMMETRY = Int32(0), Int32(1), Int32(2)
const TERM_ADVECTION, TERM_NORMAL, TERM_CURVATURE, TERM_EIKONAL = Int32(0), Int32(1), Int32(2), Int32(3)
const COEF_CONST, COEF_FIELD, COEF_SEPARABLE, COEF_NONE, COEF_EXPR = Int32(0), Int32(1), Int32(2), Int32(3), Int32(4)
const TS_NONE, TS_COS, TS_HOST = Int32(0), Int32(1), Int32(2)
const SHAPE_SPHERE, SHAPE_BOX, SHAPE_PLANE, SHAPE_CONST = Int32(0), Int32(1), Int32(2), Int32(3)

struct CBC
    kind::Int32
    P::Int32
end

struct CTerm                      # lsm_term
    kind::Int32
    scheme::Int32
    coef_kind::Int32
    tscale_kind::Int32
    cval::NTuple{3, Float64}
    tparam::Float64
    field::Ptr{Cvoid}
end

last_error() = unsafe_string(ccall((:lsm_last_error, LIB), Cstring, ()))

# status -> the exception the reference throws at the cited line
function check(rc::Int32)
    rc == LSM_OK && return nothing
    msg = last_error()
    rc in (LSM_ERR_CFL, LSM_ERR_TIME, LSM_ERR_BC, LSM_ERR_ARG) && throw(ArgumentError(msg))   # levelsetterms.jl:26, levelsetequation.jl:196, boundaryconditions.jl:184
    error("lsm_b200 (status $rc): $msg")
end

# ---- contexts ------------------------------------------------------------------------------------------
# A context outlives every field created on it: fields keep a reference to their Context, and a Context that is finalised
# first (GC order is unspecified) only marks itself dead — its fields then skip lsm_field_destroy instead of touching freed
# memory (ADVICE r1: use-after-free in the finalizers).
mutable struct Context
    handle::Ptr{Cvoid}
    rank::Int
    nranks::Int
    alive::Bool
end
function _finalize(c::Context)
    c.alive || return
    c.alive = false
    ccall((:lsm_ctx_destroy, LIB), Int32, (Ptr{Cvoid},), c.handle)
    c.handle = C_NULL
    return
end
function Context(device::Integer = 0)
    h = Ref{Ptr{Cvoid}}(C_NULL)
    check(ccall((:lsm_ctx_create, LIB), Int32, (Int32, Ref{Ptr{Cvoid}}), device, h))
    return finalizer(_finalize, Context(h[], 0, 1, true))
end
# one Julia process per GPU (MPI.jl ...): rank 0 creates the id and the host broadcasts its 128 bytes
nccl_unique_id() = (id = zeros(UInt8, 128); check(ccall((:lsm_nccl_unique_id, LIB), Int32, (Ptr{UInt8},), id)); id)
function Context(device::Integer, rank::Integer, nranks::Integer, id::Vector{UInt8})
    h = Ref{Ptr{Cvoid}}(C_NULL)
    check(ccall((:lsm_ctx_create_rank, LIB), Int32, (Int32, Int32, Int32, Ptr{UInt8}, Ref{Ptr{Cvoid}}), device, rank, nranks, id, h))
    return finalizer(_finalize, Context(h[], rank, nranks, true))
end
"All GPUs of the box from ONE Julia task: `lsm_ctx_create_multi` (ncclCommInitAll); `ranks[r]` owns slab r of the last axis."
struct MultiContext
    ranks::Vector{Context}
end
function MultiContext(devices::AbstractVector{<:Integer})
    n = length(devices)
    hs = fill(C_NULL, n)
    check(ccall((:lsm_ctx_create_multi, LIB), Int32, (Int32, Ptr{Int32}, Ptr{Ptr{Cvoid}}), n, Int32.(devices), hs))
    return MultiContext([finalizer(_finalize, Context(hs[r], r - 1, n, true)) for r in 1:n])
end
const DEFAULT = Ref{Union{Nothing, Context}}(nothing)
default_context() = something(DEFAULT[], (DEFAULT[] = Context(parse(Int, get(ENV, "LSM_B200_DEVICE", "0")))))

"(first, count) of the planes of the last dimension rank `ctx.rank` owns (0-based first): `lsm_slab_plan`."
function slab(ctx::Context, n_last::Integer)
    ctx.nranks == 1 && return (0, Int(n_last))
    f, c = Ref{Int32}(0), Ref{Int32}(0)
    check(ccall((:lsm_slab_plan, LIB), Int32, (Int32, Int32, Int32, Ref{Int32}, Ref{Int32}), n_last, ctx.nranks, ctx.rank, f, c))
    return (Int(f[]), Int(c[]))
end

# ---- the device-backed state type -----------------------------------------------------------------------------------
_dtype(::Type{Float32}) = F32
_dtype(::Type{Float64}) = F64
_cbc(::LSM.PeriodicBC) = CBC(BC_PERIODIC, 0)
_cbc(::LSM.ExtrapolationBC{P}) where {P} = CBC(BC_EXTRAP, P)
_cbc(::LSM.SymmetryBC) = CBC(BC_SYMMETRY, 0)

"""
    DeviceMeshField{N,T,V,B} <: LevelSetMethods.AbstractMeshField{N,T,V}

A dense node field whose authoritative copy lives in HBM (`lsm_field`).  `vals` is the host view with the reference's layout
(`Array{V,N}`; `Array{SVector{N,T},N}` for velocities — memory-identical to the AoS layout `lsm_field_upload` expects); the
two copies are kept coherent lazily, like `api.py`'s MeshField: `values(ϕ)` downloads if the device is ahead and marks the
device copy stale (the caller may mutate the array), handing the field to the engine uploads if the host is ahead.
With a multi-rank context the field holds this rank's slab of the last dimension (`vals` has the slab's shape).
"""
mutable struct DeviceMeshField{N, T, V, B} <: LSM.AbstractMeshField{N, T, V}
    vals::Array{V, N}
    mesh::LSM.CartesianGrid{N, T}
    bcs::B
    ctx::Context
    handle::Ptr{Cvoid}
    host_fresh::Bool
    dev_fresh::Bool
    owned::Bool                       # false: a stage buffer owned by the library (lsm_field_stage_buffer)
end

function _destroy(f::DeviceMeshField)
    if f.owned && f.handle != C_NULL && f.ctx.alive
        ccall((:lsm_field_destroy, LIB), Int32, (Ptr{Cvoid},), f.handle)
    end
    f.handle = C_NULL
    return
end

function _create_handle(ctx::Context, g::LSM.CartesianGrid{N}, ::Type{V}, bcs) where {N, V}
    S = V <: Real ? V : eltype(V)
    ncomp = V <: Real ? 1 : N
    n = Int32[size(g)...]
    lc, hc = Float64[g.lc...], Float64[g.hc...]
    h = Ref{Ptr{Cvoid}}(C_NULL)
    check(ccall((:lsm_field_create, LIB), Int32, (Ptr{Cvoid}, Int32, Ptr{Int32}, Int32, Int32, Ptr{Float64}, Ptr{Float64}, Ref{Ptr{Cvoid}}),
                ctx.handle, N, n, _dtype(float(S)), ncomp, lc, hc, h))
    if !isnothing(bcs)
        flat = CBC[_cbc(bcs[d][s]) for d in 1:N for s in 1:2]
        check(ccall((:lsm_field_set_bc, LIB), Int32, (Ptr{Cvoid}, Ptr{CBC}), h[], flat))
    end
    return h[]
end

"""
    to_device(ϕ::MeshField; ctx = default_context())

Device-backed twin of a host `MeshField` (same grid and boundary conditions).  On one rank the host array is ALIASED (like
`_add_boundary_conditions`, meshfield.jl:150-153), on several ranks the rank's slab of the last dimension is copied.
"""
function to_device(ϕ::LSM.MeshField{N, T, V}; ctx::Context = default_context()) where {N, T, V}
    g, bcs = LSM.mesh(ϕ), LSM.boundary_conditions(ϕ)
    vals = values(ϕ)
    if ctx.nranks > 1
        first, count = slab(ctx, size(vals, N))
        vals = copy(selectdim(vals, N, (first + 1):(first + count)))
    end
    d = DeviceMeshField{N, T, V, typeof(bcs)}(vals, g, bcs, ctx, _create_handle(ctx, g, V, bcs), true, false, true)
    return finalizer(_destroy, d)
end
to_device(ϕ::DeviceMeshField; ctx = nothing) = ϕ

"The up-to-date `lsm_field*` of `ϕ` (uploading the host view first when it is the fresh copy)."
function handle!(ϕ::DeviceMeshField)
    if !ϕ.dev_fresh
        v = ϕ.vals
        GC.@preserve v check(ccall((:lsm_field_upload, LIB), Int32, (Ptr{Cvoid}, Ptr{Cvoid}), ϕ.handle, pointer(v)))
        ϕ.dev_fresh = true
    end
    return ϕ.handle
end
function _sync_host!(ϕ::DeviceMeshField)
    if !ϕ.host_fresh
        v = ϕ.vals
        GC.@preserve v check(ccall((:lsm_field_download, LIB), Int32, (Ptr{Cvoid}, Ptr{Cvoid}), ϕ.handle, pointer(v)))
        ϕ.host_fresh = true
    end
    return ϕ.vals
end
_device_advanced!(ϕ::DeviceMeshField) = (ϕ.dev_fresh = true; ϕ.host_fresh = false; ϕ)

# ---- the field interface the rest of the package uses (meshfield.jl:58-61,161-169,213-292) -----------------------------
"`values(ϕ)`: the host array, downloaded if the device is ahead.  The caller may mutate it, so the device copy becomes stale."
Base.values(ϕ::DeviceMeshField) = (v = _sync_host!(ϕ); ϕ.dev_fresh = false; v)
"Read-only look at the current values (does not invalidate the device copy)."
peek(ϕ::DeviceMeshField) = _sync_host!(ϕ)
_hostview(ϕ::DeviceMeshField) = LSM.MeshField(peek(ϕ), ϕ.mesh, ϕ.bcs)                 # ghost cells through the reference's own code
Base.getindex(ϕ::DeviceMeshField{N}, I::CartesianIndex{N}) where {N} = _hostview(ϕ)[I]
Base.getindex(ϕ::DeviceMeshField, I::Integer...) = ϕ[CartesianIndex(I...)]
Base.setindex!(ϕ::DeviceMeshField, v, I...) = (values(ϕ)[I...] = v)
Base.axes(ϕ::DeviceMeshField) = axes(ϕ.vals)
Base.size(ϕ::DeviceMeshField) = size(ϕ.vals)
LSM.update_band!(ϕ::DeviceMeshField; kwargs...) = ϕ                                    # meshfield.jl:553 (full grid: no-op)

"`copy(ϕ)`: an independent device field (device-to-device when the device copy is current: no host round trip)."
function Base.copy(ϕ::DeviceMeshField{N, T, V, B}) where {N, T, V, B}
    d = DeviceMeshField{N, T, V, B}(similar(ϕ.vals), ϕ.mesh, ϕ.bcs, ϕ.ctx, _create_handle(ϕ.ctx, ϕ.mesh, V, ϕ.bcs), false, true, true)
    finalizer(_destroy, d)
    check(ccall((:lsm_field_copy, LIB), Int32, (Ptr{Cvoid}, Ptr{Cvoid}), d.handle, handle!(ϕ)))
    return d
end
function Base.copy!(dest::DeviceMeshField, src::DeviceMeshField)
    check(ccall((:lsm_field_copy, LIB), Int32, (Ptr{Cvoid}, Ptr{Cvoid}), dest.handle, handle!(src)))
    return _device_advanced!(dest)
end
Base.copy!(dest::DeviceMeshField, src::LSM.MeshField) = (copyto!(values(dest), values(src)); dest)
Base.copy!(dest::LSM.MeshField, src::DeviceMeshField) = (copyto!(values(dest), peek(src)); dest)
Base.map(f, ϕ::DeviceMeshField) = to_device(LSM.MeshField(map(f, peek(ϕ)), ϕ.mesh, ϕ.bcs); ctx = ϕ.ctx)
# `LevelSetEquation(; ic, bc)` calls this on a copy of `ic` (levelsetequation.jl:70-76)
function LSM._add_boundary_conditions(ϕ::DeviceMeshField{N, T, V}, bc) where {N, T, V}
    bcs = LSM._normalize_bc(bc, N)
    d = DeviceMeshField{N, T, V, typeof(bcs)}(peek(ϕ), ϕ.mesh, bcs, ϕ.ctx, _create_handle(ϕ.ctx, ϕ.mesh, V, bcs), true, false, true)
    return finalizer(_destroy, d)
end

# ---- analytic fields generated on the device (lsm_field_fill_shape / lsm_field_fill_separable) ---------------------------
function _device_only(g::LSM.CartesianGrid{N, T}, ::Type{V}, bcs, ctx::Context) where {N, T, V}
    first, count = slab(ctx, size(g)[N])
    shape = (size(g)[1:(N - 1)]..., count)
    d = DeviceMeshField{N, T, V, typeof(bcs)}(Array{V, N}(undef, shape), g, bcs, ctx, _create_handle(ctx, g, V, bcs), false, true, true)
    return finalizer(_destroy, d)
end
"`MeshField(x -> norm(x - c) - r, grid)` evaluated on the device (meshfield.jl:208-211): `shape` ∈ (:sphere, :box, :plane, :const)."
function from_shape(g::LSM.CartesianGrid{N, T}, shape::Symbol, params; bc = nothing, V::Type = Float64, ctx::Context = default_context()) where {N, T}
    bcs = isnothing(bc) ? nothing : LSM._normalize_bc(bc, N)
    d = _device_only(g, V, bcs, ctx)
    code = Dict(:sphere => SHAPE_SPHERE, :box => SHAPE_BOX, :plane => SHAPE_PLANE, :const => SHAPE_CONST)[shape]
    p = Float64[params...]
    check(ccall((:lsm_field_fill_shape, LIB), Int32, (Ptr{Cvoid}, Int32, Ptr{Float64}, Int32), d.handle, code, p, length(p)))
    return d
end

# ---- engine coefficient kinds the reference has no type for ---------------------------------------------------------------
"`cos(π t / period)`, evaluated inside the library so that the whole step loop stays on the device."
struct CosScale
    period::Float64
end
"Coefficient `base × g(t)`: `base` a (Device)MeshField or constant, `g` a `CosScale` or a host function `t -> scale`."
struct TimeScaled{B, G}
    base::B
    g::G
end
"Rank-1 separable velocity `u_d = scale[d] · X_d[i] · Y_d[j] · Z_d[k]` from 3·N small tables (no velocity traffic from HBM)."
mutable struct SeparableVelocity{N, T}
    grid::LSM.CartesianGrid{N, T}
    scales::NTuple{N, Float64}
    tabs::NTuple{N, NTuple{N, Vector{Float64}}}       # tabs[d][axis]
    ctx::Context
    handle::Ptr{Cvoid}
end
function SeparableVelocity(g::LSM.CartesianGrid{N, T}, scales, tabs; ctx::Context = default_context()) where {N, T}
    flat = reduce(vcat, [Float64.(tabs[d][a]) for d in 1:N for a in 1:N])
    n = Int32[size(g)...]
    h = Ref{Ptr{Cvoid}}(C_NULL)
    check(ccall((:lsm_field_create_separable, LIB), Int32,
                (Ptr{Cvoid}, Int32, Ptr{Int32}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ref{Ptr{Cvoid}}),
                ctx.handle, N, n, Float64[g.lc...], Float64[g.hc...], Float64[scales...], flat, h))
    s = SeparableVelocity{N, T}(g, Tuple(Float64.(scales)), Tuple(Tuple(Float64.(tabs[d][a]) for a in 1:N) for d in 1:N), ctx, h[])
    return finalizer(x -> (x.ctx.alive && x.handle != C_NULL && ccall((:lsm_field_destroy, LIB), Int32, (Ptr{Cvoid},), x.handle); x.handle = C_NULL), s)
end
"The stored velocity field of a `SeparableVelocity`, materialised on the device (bit-identical to building it on the host)."
function from_separable(s::SeparableVelocity{N, T}; S::Type = Float64) where {N, T}
    d = _device_only(s.grid, SVector{N, S}, nothing, s.ctx)
    check(ccall((:lsm_field_fill_separable, LIB), Int32, (Ptr{Cvoid}, Ptr{Cvoid}), d.handle, s.handle))
    return d
end

"""
    DeviceFunction(exprs...)

A function-valued coefficient `f(x, t)` (`_eval_field`, levelsetterms.jl:42-43) evaluated on the DEVICE: one CUDA C++ expression per
component in `x1 .. xN`, `t`, `pi` and CUDA's double math functions, e.g. `AdvectionTerm(DeviceFunction("-x2", "x1"))` for
`(x, t) -> SVector(-x[2], x[1])`.  Checked and compiled (NVRTC, sm_100a, once per process) by the constructor; the library then
materialises the coefficient in HBM at every time the reference would call `f`, so `integrate!` stays one `lsm_integrate` call.
"""
struct DeviceFunction
    exprs::Vector{String}
    fields::Vector{Any}       # [(ctx, grid, V, DeviceMeshField), ...]: one device field per context, grid and valtype
end
function _cexprs(f, exprs::Vector{String})
    ptrs = Ptr{UInt8}[pointer(e) for e in exprs]
    push!(ptrs, C_NULL)       # the list ends with a NULL pointer
    return GC.@preserve exprs ptrs f(ptrs)
end
function DeviceFunction(exprs::AbstractString...)
    ex = String[exprs...]
    used = [parse(Int, m.captures[1]) for e in ex for m in eachmatch(r"\bx([1-3])\b", e)]
    ndim = length(ex) > 1 ? length(ex) : maximum(used; init = 1)
    _cexprs(ex) do p
        check(ccall((:lsm_expr_check, LIB), Int32, (Int32, Int32, Ptr{Ptr{UInt8}}), ndim, length(ex), p))
    end
    return DeviceFunction(ex, Any[])
end
function _set_expr(d::DeviceMeshField, f::DeviceFunction)
    _cexprs(f.exprs) do p
        check(ccall((:lsm_field_set_expr, LIB), Int32, (Ptr{Cvoid}, Ptr{Ptr{UInt8}}), d.handle, p))
    end
    return d
end
"The device field of `f` for this context, grid and valtype (created on first use; the library fills it when a term needs it)."
function device_field(f::DeviceFunction, ctx::Context, g::LSM.CartesianGrid{N}, ::Type{V}) where {N, V}
    for (c, gg, VV, d) in f.fields
        c === ctx && gg == g && VV === V && return d
    end
    d = _set_expr(_device_only(g, V, nothing, ctx), f)
    push!(f.fields, (ctx, g, V, d))
    return d
end
"`MeshField(f, grid)` (meshfield.jl:208-211) for any `f` written as a `DeviceFunction`, evaluated on the device at `t = 0`."
function from_expr(g::LSM.CartesianGrid{N, T}, expr; bc = nothing, V::Type = Float64, ctx::Context = default_context()) where {N, T}
    f = expr isa DeviceFunction ? expr : DeviceFunction((expr isa AbstractString ? (expr,) : expr)...)
    bcs = isnothing(bc) ? nothing : LSM._normalize_bc(bc, N)
    d = _set_expr(_device_only(g, length(f.exprs) == 1 ? V : SVector{N, V}, bcs, ctx), f)
    check(ccall((:lsm_field_fill_expr, LIB), Int32, (Ptr{Cvoid}, Float64), d.handle, 0.0))
    return d
end

# ---- device mirrors of host coefficient fields, cached per host array -------------------------------------------------------
# A MeshField coefficient (velocity, speed, b, S₀) is uploaded ONCE per (context, host array) and reused by every later
# compute_cfl / stage / integrate! call.  A term with a non-default update_func may rewrite its coefficient: its mirror is
# re-uploaded after every update_term! (`refresh!`).  WeakKeyDict: the mirror dies with the host array.
const MIRRORS = WeakKeyDict{Any, Vector{Any}}()       # host array => [(ctx, DeviceMeshField), ...]
function mirror(ctx::Context, f::LSM.MeshField)
    lst = get!(() -> Any[], MIRRORS, values(f))
    for (c, d) in lst
        c === ctx && return d
    end
    d = to_device(f; ctx)
    push!(lst, (ctx, d))
    return d
end
mirror(ctx::Context, f::DeviceMeshField) = f
refresh!(d::DeviceMeshField) = (d.host_fresh = true; d.dev_fresh = false; d)      # the host array was rewritten by an update_func

# ---- terms -> descriptors -----------------------------------------------------------------------------------------------------
_isdefault(f) = f === nothing || (f isa Function && parentmodule(f) === LSM && occursin("#", string(nameof(f))))   # the no-op closure of the term constructors
_update_func(term) = hasproperty(term, :update_func) ? term.update_func : nothing
_coef(term::LSM.AdvectionTerm) = (TERM_ADVECTION, LSM.scheme(term) isa LSM.WENO5 ? Int32(1) : Int32(0), LSM.velocity(term))
_coef(term::LSM.NormalMotionTerm) = (TERM_NORMAL, Int32(0), LSM.speed(term))
_coef(term::LSM.CurvatureTerm) = (TERM_CURVATURE, Int32(0), LSM.coefficient(term))
_coef(term::LSM.EikonalReinitializationTerm) = (TERM_EIKONAL, Int32(0), term.S₀)

struct Lowered
    terms::Vector{CTerm}
    gscale::Vector{Float64}   # per-term g for TS_HOST terms
    keep::Vector{Any}         # everything the descriptors point at, kept alive for the call
    device_only::Bool         # nothing needs the host between steps
end

function lower(terms, ϕ::DeviceMeshField{N, T, V}, t) where {N, T, V}
    ctx = ϕ.ctx
    out, gs, keep, device_only = CTerm[], Float64[], Any[], true
    for term in terms
        kind, scheme, coef = _coef(term)
        custom = !_isdefault(_update_func(term))
        custom && (device_only = false)
        ts, tp, g = TS_NONE, 1.0, 1.0
        if coef isa TimeScaled
            coef.base isa DeviceFunction && throw(ArgumentError("TimeScaled(DeviceFunction): write the time factor into the expression, which already sees t"))
            if coef.g isa CosScale
                ts, tp = TS_COS, coef.g.period
            else
                ts, g, device_only = TS_HOST, Float64(coef.g(t)), false
            end
            coef = coef.base
        end
        ck, cval, fld = COEF_CONST, (0.0, 0.0, 0.0), C_NULL
        if coef === nothing
            ck = COEF_NONE
        elseif coef isa SeparableVelocity
            ck, fld = COEF_SEPARABLE, coef.handle
            push!(keep, coef)
        elseif coef isa Union{LSM.MeshField, DeviceMeshField}
            d = mirror(ctx, coef)
            custom && coef isa LSM.MeshField && refresh!(d)
            ck, fld = COEF_FIELD, handle!(d)
            push!(keep, d)
        elseif coef isa DeviceFunction
            # f(x, t) on the device: the library materialises it at the CFL and stage times
            nc = kind == TERM_ADVECTION ? N : 1
            length(coef.exprs) == nc || throw(ArgumentError("this coefficient needs $nc expression(s), the DeviceFunction has $(length(coef.exprs))"))
            d = device_field(coef, ctx, LSM.mesh(ϕ), nc == 1 ? V : SVector{N, V})
            ck, fld = COEF_EXPR, d.handle
            push!(keep, d)
        elseif coef isa Function
            # f(x, t) (levelsetterms.jl:43): evaluated on the host at the stage time, like every host callback (slow path)
            device_only = false
            d = to_device(LSM.MeshField(x -> coef(x, t), LSM.mesh(ϕ)); ctx)
            ck, fld = COEF_FIELD, handle!(d)
            push!(keep, d)
        else
            c = Float64[coef...]
            cval = ntuple(i -> i <= length(c) ? c[i] : 0.0, 3)
        end
        push!(out, CTerm(kind, scheme, ck, ts, cval, tp, fld))
        push!(gs, g)
    end
    return Lowered(out, gs, keep, device_only)
end

# ---- the methods on the reference's seam -----------------------------------------------------------------------------------------
const Explicit = Union{LSM.ForwardEuler, LSM.RK2, LSM.RK3}
_code(::LSM.ForwardEuler) = Int32(0)
_code(::LSM.RK2) = Int32(1)
_code(::LSM.RK3) = Int32(2)
_stage_times(::LSM.ForwardEuler, tc, Δt) = (tc,)
_stage_times(::LSM.RK2, tc, Δt) = (tc, tc + Δt)
_stage_times(::LSM.RK3, tc, Δt) = (tc, tc + Δt, tc + 0.5Δt)
# which field a stage differentiates (what the reference hands to update_term!, timestepping.jl:131,146,157,174,186,197):
# 0 = ϕ itself, k = the library's stage buffer k
_stage_inputs(::LSM.ForwardEuler) = (0,)
_stage_inputs(::LSM.RK2) = (0, 1)
_stage_inputs(::LSM.RK3) = (0, 1, 2)

"A lazily downloaded view of the library's stage buffer `which` of `ϕ` (not owned: the library frees it with `ϕ`)."
function stage_buffer(ϕ::DeviceMeshField{N, T, V, B}, which::Integer) where {N, T, V, B}
    h = Ref{Ptr{Cvoid}}(C_NULL)
    check(ccall((:lsm_field_stage_buffer, LIB), Int32, (Ptr{Cvoid}, Int32, Ref{Ptr{Cvoid}}), ϕ.handle, which, h))
    return DeviceMeshField{N, T, V, B}(similar(ϕ.vals), ϕ.mesh, ϕ.bcs, ϕ.ctx, h[], false, true, false)
end

"`compute_cfl(terms, ϕ, t)` — src/levelsetterms.jl:22-38 (min over terms and nodes; ArgumentError unless Δt > 0)."
function LSM.compute_cfl(terms, ϕ::DeviceMeshField, t)
    low = lower(terms, ϕ, t)
    dt = Ref{Float64}(0.0)
    GC.@preserve low check(ccall((:lsm_compute_cfl, LIB), Int32, (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{CTerm}, Int32, Float64, Ptr{Float64}, Ref{Float64}),
                                 ϕ.ctx.handle, handle!(ϕ), low.terms, length(low.terms), t, low.gscale, dt))
    return dt[]
end

"`_alloc_buffers` — src/timestepping.jl:126,141,168: the RK buffers live in the library (allocated once per state field)."
LSM._alloc_buffers(::Explicit, ϕ::DeviceMeshField) = ()

"`_advance!` — src/timestepping.jl:128-202: one `lsm_stage` per RK stage, `update_term!` before each with the stage's input field."
function LSM._advance!(integ::Explicit, ϕ::DeviceMeshField, _buffers, terms, tc, Δt)
    custom = any(term -> !_isdefault(_update_func(term)), terms)
    for (s, (ts, inp)) in enumerate(zip(_stage_times(integ, tc, Δt), _stage_inputs(integ)))
        if custom
            stagefield = inp == 0 ? ϕ : stage_buffer(ϕ, inp)           # downloaded only if the hook reads it
            for term in terms
                LSM.update_term!(term, stagefield, ts)
            end
        end
        low = lower(terms, ϕ, ts)
        GC.@preserve low check(ccall((:lsm_stage, LIB), Int32, (Ptr{Cvoid}, Int32, Int32, Ptr{Cvoid}, Ptr{CTerm}, Int32, Float64, Float64, Ptr{Float64}),
                                     ϕ.ctx.handle, _code(integ), s, handle!(ϕ), low.terms, length(low.terms), tc, Δt, low.gscale))
        _device_advanced!(ϕ)
    end
    return ϕ
end

# ---- InflowImplicit: the engine's semi-implicit advection integrator (LSM_SEMI_IMPLICIT) -------------------------------------------
"""
    InflowImplicit(; cfl = 2.0)

Inflow-implicit / outflow-explicit steps of ONE `AdvectionTerm` on a `DeviceMeshField` (include/lsm_b200.h, "semi-implicit
advection"): the velocity at mid-step, the implicit half solved on the device by a fixed number of Jacobi sweeps.  Stable above
Courant number 1, hence `cfl = 2`.  The idea of `LevelSetMethods.SemiImplicitI2OE`, not its bits: this is a separate type until
the two have been compared where Julia runs.
"""
Base.@kwdef struct InflowImplicit <: LSM.TimeIntegrator
    cfl::Float64 = 2.0
end
LSM.cfl(integ::InflowImplicit) = integ.cfl
_code(::InflowImplicit) = Int32(3)

"`_alloc_buffers`: the right-hand side and the second Jacobi iterate live in the library's stage buffers of `ϕ`."
LSM._alloc_buffers(::InflowImplicit, ϕ::DeviceMeshField) = ()

"`_advance!`: one whole step (`lsm_stage` 1 of 1), `update_term!` first at the mid-step time the velocity is taken at."
function LSM._advance!(integ::InflowImplicit, ϕ::DeviceMeshField, _buffers, terms, tc, Δt)
    ts = tc + 0.5Δt
    if any(term -> !_isdefault(_update_func(term)), terms)
        for term in terms
            LSM.update_term!(term, ϕ, ts)
        end
    end
    low = lower(terms, ϕ, ts)
    GC.@preserve low check(ccall((:lsm_stage, LIB), Int32, (Ptr{Cvoid}, Int32, Int32, Ptr{Cvoid}, Ptr{CTerm}, Int32, Float64, Float64, Ptr{Float64}),
                                 ϕ.ctx.handle, _code(integ), 1, handle!(ϕ), low.terms, length(low.terms), tc, Δt, low.gscale))
    _device_advanced!(ϕ)
    return ϕ
end

"Jacobi sweeps of a semi-implicit step at Courant number `courant` (`lsm_semi_implicit_sweeps`; no GPU needed)."
function semi_implicit_sweeps(courant::Real, ::Type{T} = Float64) where {T}
    k = Ref{Int64}(0)
    check(ccall((:lsm_semi_implicit_sweeps, LIB), Int32, (Float64, Int32, Ref{Int64}), courant, T === Float64 ? Int32(1) : Int32(0), k))
    return k[]
end

"""
`_integrate!` — src/timestepping.jl:101-122.  Default hooks and device-resident coefficients: the whole loop is one
`lsm_integrate` call (Δt = min(Δt_max, cfl·compute_cfl, tf − tc) while tc ≤ tf − eps(tc), landing on tf).  Otherwise the
reference's generic method runs and its calls dispatch to the methods above.
"""
function LSM._integrate!(ls, ϕ::DeviceMeshField, integ::Union{Explicit, InflowImplicit}, terms, tc, tf, Δt_max, prehook, posthook)
    low = lower(terms, ϕ, tc)
    if prehook === identity && posthook === identity && low.device_only
        t_out, steps = Ref{Float64}(tc), Ref{Int64}(0)
        rc = GC.@preserve low ccall((:lsm_integrate, LIB), Int32,
                                    (Ptr{Cvoid}, Int32, Float64, Ptr{Cvoid}, Ptr{CTerm}, Int32, Float64, Float64, Float64, Int64, Ref{Float64}, Ref{Int64}),
                                    ϕ.ctx.handle, _code(integ), LSM.cfl(integ), handle!(ϕ), low.terms, length(low.terms),
                                    Float64(tc), Float64(tf), Float64(Δt_max), -1, t_out, steps)
        _device_advanced!(ϕ)
        ls.t = t_out[]
        check(rc)
        return nothing
    end
    return invoke(LSM._integrate!, Tuple{Any, LSM.AbstractMeshField, LSM.TimeIntegrator, Any, Any, Any, Any, Any, Any},
                  ls, ϕ, integ, terms, tc, tf, Δt_max, prehook, posthook)
end

"`integrate!` of the same equation on every rank's slab from ONE task (`lsm_multi_integrate`; device-resident terms, default hooks)."
function integrate_multi!(mc::MultiContext, eqs::Vector, tf, Δt = Inf)
    n = length(mc.ranks)
    lows = [lower(eqs[r].terms, LSM.current_state(eqs[r]), LSM.current_time(eqs[r])) for r in 1:n]
    all(l -> l.device_only, lows) || throw(ArgumentError("integrate_multi! needs device-resident coefficients and default hooks"))
    integ = LSM.time_integrator(eqs[1])
    t_out, steps = Ref{Float64}(0.0), Ref{Int64}(0)
    GC.@preserve lows check(ccall((:lsm_multi_integrate, LIB), Int32,
                                  (Int32, Ptr{Ptr{Cvoid}}, Int32, Float64, Ptr{Ptr{Cvoid}}, Ptr{Ptr{CTerm}}, Int32, Float64, Float64, Float64, Int64, Ref{Float64}, Ref{Int64}),
                                  n, [c.handle for c in mc.ranks], _code(integ), LSM.cfl(integ), [handle!(LSM.current_state(e)) for e in eqs],
                                  [pointer(l.terms) for l in lows], length(lows[1].terms), Float64(LSM.current_time(eqs[1])), Float64(tf), Float64(Δt), -1, t_out, steps))
    for e in eqs
        _device_advanced!(LSM.current_state(e)); e.t = t_out[]
    end
    return eqs
end

# ---- "next" rows: reductions, velocity extension, set operations on device fields ---------------------------------------------------
"`volume(ϕ)` / `perimeter(ϕ)` — src/levelsetops.jl:27-33,139-149, reduced on the device (8 bytes of D2H: a cheap posthook)."
function LSM.volume(ϕ::DeviceMeshField)
    out = Ref{Float64}(0)
    check(ccall((:lsm_volume, LIB), Int32, (Ptr{Cvoid}, Ptr{Cvoid}, Ref{Float64}), ϕ.ctx.handle, handle!(ϕ), out))
    return out[]
end
function LSM.perimeter(ϕ::DeviceMeshField)
    out = Ref{Float64}(0)
    check(ccall((:lsm_perimeter, LIB), Int32, (Ptr{Cvoid}, Ptr{Cvoid}, Ref{Float64}), ϕ.ctx.handle, handle!(ϕ), out))
    return out[]
end

"""
    interface_mesh(ϕ::DeviceMeshField{N}; level = 0) -> (vertices, faces, keys)

The interface {ϕ = level} extracted on the device (`lsm_interface_extract`: marching simplices on the Freudenthal–Kuhn
triangulation, watertight, triangles oriented toward ϕ > level, segments with ϕ <= level on their left); only the mesh is copied
back, not `values(ϕ)`.  `vertices::Vector{SVector{N,Float64}}`, `faces::Vector{NTuple{N,Int32}}` (1-based): the arrays
`Makie.mesh` (3-D) and `linesegments` (2-D) take.  `keys` are the global lattice-edge ids of the vertices (sorted).
"""
function interface_mesh(ϕ::DeviceMeshField{N}; level::Real = 0) where {N}
    nv, np = Ref{Int64}(0), Ref{Int64}(0)
    check(ccall((:lsm_interface_extract, LIB), Int32, (Ptr{Cvoid}, Ptr{Cvoid}, Float64, Ref{Int64}, Ref{Int64}),
                ϕ.ctx.handle, handle!(ϕ), Float64(level), nv, np))
    return _fetch_interface(ϕ.ctx, Val(N), nv[], np[])
end

function _fetch_interface(ctx::Context, ::Val{N}, nv::Integer, np::Integer) where {N}
    V = Matrix{Float64}(undef, N, nv)          # AoS: vertex-major, N coordinates each
    K = Vector{Int64}(undef, nv)
    P = Matrix{Int32}(undef, N, np)
    check(ccall((:lsm_interface_fetch, LIB), Int32, (Ptr{Cvoid}, Ptr{Float64}, Ptr{Int64}, Ptr{Int32}),
                ctx.handle, nv == 0 ? C_NULL : pointer(V), nv == 0 ? C_NULL : pointer(K), np == 0 ? C_NULL : pointer(P)))
    verts = [SVector{N, Float64}(ntuple(d -> V[d, j], N)) for j in 1:nv]
    faces = [ntuple(d -> P[d, j] + Int32(1), N) for j in 1:np]
    return verts, faces, K
end

"`interface_mesh` of a field slab-decomposed over `mc` (collective, `lsm_multi_interface_extract`): the per-rank pieces welded by key."
function interface_mesh(mc::MultiContext, ϕs::Vector{<:DeviceMeshField{N}}; level::Real = 0) where {N}
    n = length(mc.ranks)
    nv, np = zeros(Int64, n), zeros(Int64, n)
    check(ccall((:lsm_multi_interface_extract, LIB), Int32, (Int32, Ptr{Ptr{Cvoid}}, Ptr{Ptr{Cvoid}}, Float64, Ptr{Int64}, Ptr{Int64}),
                n, [c.handle for c in mc.ranks], [handle!(ϕ) for ϕ in ϕs], Float64(level), nv, np))
    pieces = [_fetch_interface(mc.ranks[r], Val(N), nv[r], np[r]) for r in 1:n]
    keys = reduce(vcat, [p[3] for p in pieces])
    verts_all = reduce(vcat, [p[1] for p in pieces])
    perm = sortperm(keys; alg = MergeSort)
    newidx = Vector{Int32}(undef, length(keys))
    verts, ukeys = SVector{N, Float64}[], Int64[]
    for j in perm
        if isempty(ukeys) || keys[j] != ukeys[end]
            push!(verts, verts_all[j]); push!(ukeys, keys[j])
        end
        newidx[j] = length(ukeys)
    end
    faces = NTuple{N, Int32}[]
    off = 0
    for p in pieces
        append!(faces, [ntuple(d -> newidx[f[d] + off], N) for f in p[2]])
        off += length(p[3])
    end
    return verts, faces, ukeys
end

"""
    redistance!(ϕ::DeviceMeshField; band = 3, order = 1) -> ϕ

Replace ϕ, in place on the device, by the signed distance to its zero level set (`lsm_redistance`): the piecewise-linear mesh
`interface_mesh(ϕ)` returns, which is never built.  Nodes within `band` cells of it get their exact closest point, jump flooding
carries closest points to the rest of the grid; every node keeps its sign, NaN nodes stay NaN.  No boundary conditions needed, no
copy to the host and no synchronisation, so it fits a prehook: `integrate!(eq, tf; prehook = ls -> redistance!(current_state(ls)))`.
`order = 3` (`lsm_redistance_cubic`) refines every closest point by Newton's method on the zero set of the cubic interpolant of ϕ
(`interpolate_cubic`), third-order accurate; a node where Newton fails keeps its linear closest point.
The same idea as `LevelSetMethods.reinitialize!` (reinitializer.jl:12-42, Newton on Bernstein patches from KD-tree seeds, host),
but the seeds (the linear mesh) and the one-sided stencils at the box faces are not verified against it, so the two are not
bit-compatible; that is why this is not a method of `reinitialize!`.
"""
function redistance!(ϕ::DeviceMeshField; band::Integer = 3, order::Integer = 1)
    if order == 1
        check(ccall((:lsm_redistance, LIB), Int32, (Ptr{Cvoid}, Ptr{Cvoid}, Int32, Ptr{Int64}), ϕ.ctx.handle, handle!(ϕ), band, C_NULL))
    elseif order == 3
        check(ccall((:lsm_redistance_cubic, LIB), Int32, (Ptr{Cvoid}, Ptr{Cvoid}, Int32, Ptr{Int64}, Ptr{Int64}),
                    ϕ.ctx.handle, handle!(ϕ), band, C_NULL, C_NULL))
    else
        throw(ArgumentError("redistance!: order must be 1 or 3 (got $order)"))
    end
    return _device_advanced!(ϕ)
end

"""
    narrow_band!(ϕ::DeviceMeshField; halfwidth = 3) -> ϕ

Make the explicit steps of ϕ update only the bricks near its zero level set (`lsm_field_set_band`), the idea of the reference's
`NarrowBandMeshField` and `update_band!` (meshfield.jl:314-588) with dense storage: nodes off the band keep their values, and every
other operation sees the whole field.  `halfwidth` is in cells of the smallest mesh size; `halfwidth = 0` turns the band off.
Bricks are 32 × 16 (× 16) nodes; see include/lsm_b200.h for the band's rules.
"""
function narrow_band!(ϕ::DeviceMeshField; halfwidth::Real = 3)
    check(ccall((:lsm_field_set_band, LIB), Int32, (Ptr{Cvoid}, Float64), handle!(ϕ), Float64(halfwidth)))
    return ϕ
end

"""
    band_info(ϕ::DeviceMeshField) -> (core, active, shell, states)

The band of ϕ's current values (`lsm_field_band`): brick counts and one state per brick in an array of brick coordinates
(0 frozen, 1 shell, 2 active, 3 active and core).
"""
function band_info(ϕ::DeviceMeshField{N}) where {N}
    n = size(ϕ.vals)
    nb = ntuple(d -> cld(n[d], (32, 16, 16)[d]), N)
    states = Array{UInt8, N}(undef, nb)
    counts = zeros(Int64, 3)
    check(ccall((:lsm_field_band, LIB), Int32, (Ptr{Cvoid}, Ptr{Int64}, Ptr{UInt8}), handle!(ϕ), counts, states))
    return (core = counts[1], active = counts[2], shell = counts[3], states = states)
end

"""
    interpolate_cubic(ϕ::DeviceMeshField, X::AbstractMatrix) -> (values, gradients, hessians)

The tensor-product cubic interpolant of ϕ (`lsm_interpolate_cubic`) at the columns of X (N × npts): `values` (npts),
`gradients` (N × npts) and `hessians` (N × N × npts), evaluated on the device; NaN at points outside the grid.  The same
polynomial per cell as the reference's Bernstein patch of an `InterpolatedField` (interpolation.jl, bernstein.jl), not the same
bits; one-sided stencils at the box faces, no boundary conditions.
"""
function interpolate_cubic(ϕ::DeviceMeshField{N}, X::AbstractMatrix) where {N}
    size(X, 1) == N || throw(DimensionMismatch("interpolate_cubic: X must have $N rows (one column per point), got $(size(X, 1))"))
    pts = Matrix{Float64}(X)
    npts = size(pts, 2)
    val = Vector{Float64}(undef, npts)
    grad = Matrix{Float64}(undef, N, npts)
    hess = Array{Float64, 3}(undef, N, N, npts)
    check(ccall((:lsm_interpolate_cubic, LIB), Int32, (Ptr{Cvoid}, Ptr{Cvoid}, Int64, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}),
                ϕ.ctx.handle, handle!(ϕ), npts, pts, val, grad, hess))
    return val, grad, hess
end

"""
    extend_closest_point!(F::DeviceMeshField, ϕ::DeviceMeshField; band = 3, redistance = false) -> F

Give every node of F, in place on the device, the value of F at its closest point on the zero level set of ϕ
(`lsm_extend_closest_point`): the closest points `redistance!(ϕ)` finds, with F interpolated linearly on the mesh, so a speed known
near the interface becomes constant along the normals and a constant F comes back unchanged.  NaN nodes of ϕ keep their F.  With
`redistance = true` the same call also makes ϕ its signed distance, bit for bit what `redistance!` writes:
`integrate!(eq, tf; prehook = ls -> extend_closest_point!(v, current_state(ls); redistance = true))`.  No boundary conditions, no
copy to the host, no synchronisation.  Deliberately not a method of `LevelSetMethods.extend_along_normals!`, which solves the
upwind extension PDE for a number of pseudo-time iterations.
"""
function extend_closest_point!(F::DeviceMeshField, ϕ::DeviceMeshField; band::Integer = 3, redistance::Bool = false)
    check(ccall((:lsm_extend_closest_point, LIB), Int32, (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Cvoid}, Int32, Int32, Ptr{Int64}),
                ϕ.ctx.handle, handle!(F), handle!(ϕ), band, redistance ? 1 : 0, C_NULL))
    redistance && _device_advanced!(ϕ)
    return _device_advanced!(F)
end

"""
    level_set_integrals(ϕ::DeviceMeshField; F = nothing, level = 0) -> (inside, interface, F_inside, F_interface)

The measures of {ϕ ≤ level} and {ϕ = level} and the integrals of F over both, on the device (`lsm_level_set_integrals`; 32 bytes
reach the host).  The geometry is the sharp piecewise-linear interface of `interface_mesh` and the region it bounds, with F
interpolated linearly (exact for a linear F); `F_inside` / `F_interface` are `nothing` without F.  Moments come from an F such as
the device field of `x1`.  Deliberately not methods of `LevelSetMethods.volume` / `perimeter`, which keep the reference's smoothed
Heaviside and delta sums (levelsetops.jl:27-33,139-149).
"""
function level_set_integrals(ϕ::DeviceMeshField; F::Union{DeviceMeshField, Nothing} = nothing, level::Real = 0)
    out = zeros(Float64, 4)
    check(ccall((:lsm_level_set_integrals, LIB), Int32, (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Cvoid}, Float64, Ptr{Float64}),
                ϕ.ctx.handle, handle!(ϕ), F === nothing ? C_NULL : handle!(F), Float64(level), out))
    return (inside = out[1], interface = out[2], F_inside = F === nothing ? nothing : out[3],
            F_interface = F === nothing ? nothing : out[4])
end

"`level_set_integrals` of a field slab-decomposed over `mc` (collective, `lsm_multi_level_set_integrals`): the single-GPU value bit for bit."
function level_set_integrals(mc::MultiContext, ϕs::Vector{<:DeviceMeshField}; Fs = nothing, level::Real = 0)
    n = length(mc.ranks)
    out = zeros(Float64, 4)
    check(ccall((:lsm_multi_level_set_integrals, LIB), Int32, (Int32, Ptr{Ptr{Cvoid}}, Ptr{Ptr{Cvoid}}, Ptr{Ptr{Cvoid}}, Float64, Ptr{Float64}),
                n, [c.handle for c in mc.ranks], [handle!(ϕ) for ϕ in ϕs], Fs === nothing ? C_NULL : [handle!(F) for F in Fs],
                Float64(level), out))
    return (inside = out[1], interface = out[2], F_inside = Fs === nothing ? nothing : out[3],
            F_interface = Fs === nothing ? nothing : out[4])
end

"`extend_along_normals!(F, ϕ; …)` — src/velocityextension.jl:20-78 on device fields."
function LSM.extend_along_normals!(F::DeviceMeshField, ϕ::DeviceMeshField; nb_iters::Integer = 50, cfl::Real = 0.45, frozen = nothing,
                                   interface_band::Real = 1.5, min_norm::Real = 1.0e-14)
    size(F) == size(ϕ) || throw(ArgumentError("F must have the same size as ϕ"))
    frozen === nothing || size(frozen) == size(ϕ) || throw(ArgumentError("frozen mask must have the same size as ϕ"))
    mask = frozen === nothing ? UInt8[] : UInt8.(frozen)
    GC.@preserve mask check(ccall((:lsm_extend_along_normals, LIB), Int32,
                                  (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Cvoid}, Int32, Float64, Ptr{UInt8}, Float64, Float64),
                                  ϕ.ctx.handle, handle!(F), handle!(ϕ), nb_iters, cfl, frozen === nothing ? C_NULL : pointer(mask),
                                  interface_band, min_norm))
    return _device_advanced!(F)
end

# set operations (src/levelsetops.jl:253-325): 0 union!, 1 intersect!, 2 setdiff!, 3 complement!
function _csg!(a::DeviceMeshField, b::Union{DeviceMeshField, Nothing}, op::Integer)
    check(ccall((:lsm_field_csg, LIB), Int32, (Ptr{Cvoid}, Ptr{Cvoid}, Ptr{Cvoid}, Int32),
                a.ctx.handle, handle!(a), b === nothing ? C_NULL : handle!(b), op))
    return _device_advanced!(a)
end
Base.union!(a::DeviceMeshField, b::DeviceMeshField) = _csg!(a, b, 0)
Base.intersect!(a::DeviceMeshField, b::DeviceMeshField) = _csg!(a, b, 1)
Base.setdiff!(a::DeviceMeshField, b::DeviceMeshField) = _csg!(a, b, 2)
LSM.complement!(a::DeviceMeshField) = _csg!(a, nothing, 3)
Base.union(a::DeviceMeshField, b::DeviceMeshField) = union!(copy(a), b)
Base.intersect(a::DeviceMeshField, b::DeviceMeshField) = intersect!(copy(a), b)
Base.setdiff(a::DeviceMeshField, b::DeviceMeshField) = setdiff!(copy(a), b)
LSM.complement(a::DeviceMeshField) = LSM.complement!(copy(a))

end # module
