# DZOptimizationB200.jl -- the reference-side binding: DZOptimization.jl's optimizer API over
# libdzopt_b200.so (C ABI: include/dzopt.h).  Julia host code `ccall`s the library; step! runs as
# hand-written sm_100a CUDA kernels in Float64.
#
# Drop-in for the README loop (README.md:33-41 of the reference):
#
#     using DZOptimizationB200
#     using DZOptimizationB200.ExampleFunctions: rosenbrock_function, rosenbrock_gradient!
#     opt = BFGSOptimizer(rosenbrock_function, rosenbrock_gradient!, rand(2), 1.0)
#     while !opt.has_converged[]
#         step!(opt)
#         println(opt.current_objective_value[], " ", opt.current_point)
#     end
#
# NOTE: there is no Julia in the build/test environment of this repository, so this file is
# reviewed against the header but has not been executed; tests/ drive the very same C symbols
# through ctypes (dzoptimization.jl_b200/__init__.py is the executed twin of this file).
#
# Julia closures cannot run inside a CUDA kernel, so `f`, `g!` and `c!` must be the device
# versions of legacy/ExampleFunctions.jl exported below; anything else raises ArgumentError.
module DZOptimizationB200

export BFGSOptimizer, GradientDescentOptimizer, LBFGSOptimizer, AdGDOptimizer, LegacyLBFGSOptimizer, LineSearchEvaluator,
    L2RegularizationWrapper,
    L2GradientWrapper, UniformBoxConstraint, UniformBoxGradientWrapper, QuadraticLineSearch, step!, StepType, NullStep,
    GradientDescentStep, BFGSStep, NULL_CONSTRAINT, SPHERE_CONSTRAINT,
    accelerated_pairwise_radial_energy, accelerated_pairwise_radial_gradient!, accelerated_pairwise_radial_hvp!

const libdzopt = get(ENV, "DZOPT_B200_LIB", joinpath(@__DIR__, "..", "csrc", "libdzopt_b200.so"))

# ------------------------------------------------------------------ device callbacks (ids of include/dzopt.h)
struct DeviceFunction
    objective::Cint      # DZO_OBJ_*
    role::Symbol         # :objective | :gradient
end
struct DeviceConstraint
    id::Cint             # DZO_CONSTRAINT_*
end
const NULL_CONSTRAINT = DeviceConstraint(0)      # x -> true        (legacy/DZOptimization.jl:384,759)
const SPHERE_CONSTRAINT = DeviceConstraint(1)    # normalise columns + tangent-projected gradient

struct RadialFunction
    potential::Cint      # DZO_POT_*
    derivative::Int      # 0 energy, 1 first, 2 second derivative
end

module ExampleFunctions
import ..DeviceFunction, ..RadialFunction
export rosenbrock_function, rosenbrock_gradient!, riesz_energy, riesz_gradient!,
    lj_energy, lj_first_derivative, lj_second_derivative
const rosenbrock_function = DeviceFunction(1, :objective)     # legacy/ExampleFunctions.jl:10-15
const rosenbrock_gradient! = DeviceFunction(1, :gradient)     # :17-24
const riesz_energy = DeviceFunction(2, :objective)            # :30-45
const riesz_gradient! = DeviceFunction(2, :gradient)          # :47-83
const lj_energy = RadialFunction(1, 0)                        # src/ExampleFunctions.jl:16-27
const lj_first_derivative = RadialFunction(1, 1)              # :30-47
const lj_second_derivative = RadialFunction(1, 2)             # :50-72
end

@enum StepType NullStep GradientDescentStep BFGSStep           # legacy/DZOptimization.jl:727-731

struct QuadraticLineSearch                                      # :181-188
    max_increases::Int
end
QuadraticLineSearch() = QuadraticLineSearch(0)

struct DZOptError <: Exception
    code::Cint
    msg::String
end
function check(rc::Cint)
    rc == 0 && return nothing
    msg = unsafe_string(ccall((:dzo_last_error, libdzopt), Cstring, ()))
    # the reference raises AssertionError for these two (:771, :773)
    (rc == -2 || rc == -3) && throw(AssertionError(msg))
    throw(DZOptError(rc, msg))
end

function resolve(f, g!, c!)
    (f isa DeviceFunction && f.role == :objective) ||
        throw(ArgumentError("objective_function must be a device objective from DZOptimizationB200.ExampleFunctions"))
    (g! isa DeviceFunction && g!.role == :gradient && g!.objective == f.objective) ||
        throw(ArgumentError("gradient_function! must be the device gradient of the same example function"))
    c! isa DeviceConstraint || throw(ArgumentError("constraint_function! must be NULL_CONSTRAINT or SPHERE_CONSTRAINT"))
    return f.objective, c!.id
end

# ================================================================== BFGSOptimizer (legacy :733-751)
mutable struct BFGSOptimizer{N}
    handle::Ptr{Cvoid}
    dims::NTuple{N,Int}
    n::Int
    function BFGSOptimizer(handle, dims::NTuple{N,Int}) where {N}
        opt = new{N}(handle, dims, prod(dims))
        finalizer(o -> ccall((:dzo_bfgs_destroy, libdzopt), Cvoid, (Ptr{Cvoid},), o.handle), opt)
        return opt
    end
end

# BFGSOptimizer(f, g!, x0, step)  :753-760    /    BFGSOptimizer(f, g!, c!, x0, step)  :762-810
BFGSOptimizer(f, g!, x0::Array{Float64}, step::Float64; device::Integer=0) =
    BFGSOptimizer(f, g!, NULL_CONSTRAINT, x0, step; device=device)
function BFGSOptimizer(f, g!, c!, x0::Array{Float64,N}, step::Float64; device::Integer=0) where {N}
    obj, cid = resolve(f, g!, c!)
    dim = obj == 2 ? size(x0, 1) : 0
    h = Ref{Ptr{Cvoid}}(C_NULL)
    check(ccall((:dzo_bfgs_create, libdzopt), Cint,
        (Ref{Ptr{Cvoid}}, Cint, Cint, Int64, Int64, Int64, Ptr{Float64}, Float64, Cint),
        h, obj, cid, dim, length(x0), 1, x0, step, device))
    return BFGSOptimizer(h[], size(x0))
end

# step!(opt)  :891-994 -- returns opt (:993)
function step!(opt::BFGSOptimizer)
    check(ccall((:dzo_bfgs_step, libdzopt), Cint, (Ptr{Cvoid}, Cint), opt.handle, 1))
    return opt
end

vecfield(opt, sym) = (out = Array{Float64}(undef, opt.dims);
    check(ccall((sym, libdzopt), Cint, (Ptr{Cvoid}, Ptr{Float64}), opt.handle, out)); out)
function scalarfield(opt, sym, ::Type{T}) where {T}
    out = Array{T,0}(undef)                      # 0-dim Array, read with [] like the reference's fields
    check(ccall((sym, libdzopt), Cint, (Ptr{Cvoid}, Ptr{T}), opt.handle, out))
    return out
end

function Base.getproperty(opt::BFGSOptimizer, s::Symbol)
    s === :current_point && return vecfield(opt, :dzo_bfgs_get_point)                     # :739
    s === :current_gradient && return vecfield(opt, :dzo_bfgs_get_gradient)               # :741
    s === :delta_point && return vecfield(opt, :dzo_bfgs_get_delta_point)                 # :742
    s === :delta_gradient && return vecfield(opt, :dzo_bfgs_get_delta_gradient)           # :743
    s === :next_step_direction && return vecfield(opt, :dzo_bfgs_get_direction)           # :747
    s === :current_objective_value && return scalarfield(opt, :dzo_bfgs_get_objective, Float64)   # :740
    s === :last_step_length && return scalarfield(opt, :dzo_bfgs_get_step_length, Float64)        # :744
    s === :iteration_count && return scalarfield(opt, :dzo_bfgs_get_iteration_count, Int64)       # :737
    if s === :last_step_type                                                                      # :745
        t = scalarfield(opt, :dzo_bfgs_get_step_type, Int32)
        return fill(StepType(t[]))
    end
    if s === :has_terminated || s === :has_converged                                # :738 / README.md:38
        t = scalarfield(opt, :dzo_bfgs_get_terminated, UInt8)
        return fill(t[] != 0)
    end
    if s === :approximate_inverse_hessian                                           # :746
        n = getfield(opt, :n)
        H = Matrix{Float64}(undef, n, n)
        check(ccall((:dzo_bfgs_get_inverse_hessian, libdzopt), Cint, (Ptr{Cvoid}, Int64, Ptr{Float64}),
            getfield(opt, :handle), 0, H))
        return H
    end
    return getfield(opt, s)
end

# ================================================================== GradientDescentOptimizer (legacy :305-327)
mutable struct GradientDescentOptimizer{N}
    handle::Ptr{Cvoid}
    dims::NTuple{N,Int}
    n::Int
    function GradientDescentOptimizer(handle, dims::NTuple{N,Int}) where {N}
        opt = new{N}(handle, dims, prod(dims))
        finalizer(o -> ccall((:dzo_gd_destroy, libdzopt), Cvoid, (Ptr{Cvoid},), o.handle), opt)
        return opt
    end
end

# GradientDescentOptimizer(f, g!, ls, x0, step) :377-390 / (c!, f, g!, ls, x0, step) :330-337
GradientDescentOptimizer(f, g!, ls::QuadraticLineSearch, x0::Array{Float64}, step::Float64; device::Integer=0) =
    GradientDescentOptimizer(NULL_CONSTRAINT, f, g!, ls, x0, step; device=device)
function GradientDescentOptimizer(c!, f, g!, ls::QuadraticLineSearch, x0::Array{Float64,N}, step::Float64;
    device::Integer=0) where {N}
    obj, cid = resolve(f, g!, c!)
    dim = obj == 2 ? size(x0, 1) : 0
    h = Ref{Ptr{Cvoid}}(C_NULL)
    check(ccall((:dzo_gd_create, libdzopt), Cint,
        (Ref{Ptr{Cvoid}}, Cint, Cint, Int64, Int64, Int64, Ptr{Float64}, Float64, Cint, Cint),
        h, obj, cid, dim, length(x0), 1, x0, step, ls.max_increases, device))
    return GradientDescentOptimizer(h[], size(x0))
end

# objective evaluations so far (constructor + line-search probes, :36-44) of a one-problem optimizer
function evaluation_count(opt::GradientDescentOptimizer)
    c = Ref{Int64}(0)
    check(ccall((:dzo_gd_get_evaluation_count, libdzopt), Cint, (Ptr{Cvoid}, Ref{Int64}), opt.handle, c))
    return c[]
end

function step!(opt::GradientDescentOptimizer)                                       # :393-449
    check(ccall((:dzo_gd_step, libdzopt), Cint, (Ptr{Cvoid}, Cint), opt.handle, 1))
    return opt
end

function Base.getproperty(opt::GradientDescentOptimizer, s::Symbol)
    s === :current_point && return vecfield(opt, :dzo_gd_get_point)                       # :308
    s === :delta_point && return vecfield(opt, :dzo_gd_get_delta_point)                   # :309
    s === :current_gradient && return vecfield(opt, :dzo_gd_get_gradient)                 # :316
    s === :delta_gradient && return vecfield(opt, :dzo_gd_get_delta_gradient)             # :317
    s === :next_step_direction && return vecfield(opt, :dzo_gd_get_direction)             # :320
    s === :current_objective_value && return scalarfield(opt, :dzo_gd_get_objective, Float64)       # :312
    s === :delta_objective_value && return scalarfield(opt, :dzo_gd_get_delta_objective, Float64)   # :313
    s === :last_step_length && return scalarfield(opt, :dzo_gd_get_step_length, Float64)            # :321
    s === :iteration_count && return scalarfield(opt, :dzo_gd_get_iteration_count, Int64)           # :324
    if s === :has_terminated || s === :has_converged                                                # :325
        t = scalarfield(opt, :dzo_gd_get_terminated, UInt8)
        return fill(t[] != 0)
    end
    return getfield(opt, s)
end

# ================================================================== batched mode (README.md:12)
# "run multiple optimizers in parallel": one handle holds `batch` independent optimizers whose
# states live in adjacent device arrays; x0 is n x batch.  Scalar fields come back as Vectors.
mutable struct BatchedBFGSOptimizer
    handle::Ptr{Cvoid}
    n::Int
    batch::Int
end
function BatchedBFGSOptimizer(f, g!, x0::Matrix{Float64}, step::Float64; device::Integer=0)
    obj, cid = resolve(f, g!, NULL_CONSTRAINT)
    h = Ref{Ptr{Cvoid}}(C_NULL)
    check(ccall((:dzo_bfgs_create, libdzopt), Cint,
        (Ref{Ptr{Cvoid}}, Cint, Cint, Int64, Int64, Int64, Ptr{Float64}, Float64, Cint),
        h, obj, cid, 0, size(x0, 1), size(x0, 2), x0, step, device))
    opt = BatchedBFGSOptimizer(h[], size(x0, 1), size(x0, 2))
    finalizer(o -> ccall((:dzo_bfgs_destroy, libdzopt), Cvoid, (Ptr{Cvoid},), o.handle), opt)
    return opt
end
function step!(opt::BatchedBFGSOptimizer, k::Integer=1)      # k consecutive step! calls in ONE kernel launch
    check(ccall((:dzo_bfgs_step, libdzopt), Cint, (Ptr{Cvoid}, Cint), opt.handle, k))
    return opt
end
function current_points(opt::BatchedBFGSOptimizer)
    out = Matrix{Float64}(undef, opt.n, opt.batch)
    check(ccall((:dzo_bfgs_get_point, libdzopt), Cint, (Ptr{Cvoid}, Ptr{Float64}), opt.handle, out))
    return out
end
function current_objective_values(opt::BatchedBFGSOptimizer)
    out = Vector{Float64}(undef, opt.batch)
    check(ccall((:dzo_bfgs_get_objective, libdzopt), Cint, (Ptr{Cvoid}, Ptr{Float64}), opt.handle, out))
    return out
end
# Zero-copy mirrors of the two fields the README loop reads every iteration: the step kernels store
# current_objective_value / has_terminated of every problem into page-locked host Vectors while they run, and the two
# accessors below only synchronise (dzo_bfgs_mirror_fields, include/dzopt.h).  The Vectors wrap dzo_host_alloc memory
# and stay valid until `unmirror_fields!` or finalisation.
function mirror_fields!(opt::BatchedBFGSOptimizer)
    pf, pt = Ref{Ptr{Cvoid}}(C_NULL), Ref{Ptr{Cvoid}}(C_NULL)
    check(ccall((:dzo_host_alloc, libdzopt), Cint, (Ref{Ptr{Cvoid}}, UInt64), pf, 8 * opt.batch))
    check(ccall((:dzo_host_alloc, libdzopt), Cint, (Ref{Ptr{Cvoid}}, UInt64), pt, opt.batch))
    f = unsafe_wrap(Array, Ptr{Float64}(pf[]), opt.batch)
    t = unsafe_wrap(Array, Ptr{UInt8}(pt[]), opt.batch)
    check(ccall((:dzo_bfgs_mirror_fields, libdzopt), Cint, (Ptr{Cvoid}, Ptr{Float64}, Ptr{UInt8}), opt.handle, f, t))
    return f, t
end
function unmirror_fields!(opt::BatchedBFGSOptimizer, f::Vector{Float64}, t::Vector{UInt8})
    check(ccall((:dzo_bfgs_mirror_fields, libdzopt), Cint, (Ptr{Cvoid}, Ptr{Float64}, Ptr{UInt8}), opt.handle, C_NULL, C_NULL))
    ccall((:dzo_host_free, libdzopt), Cint, (Ptr{Cvoid},), pointer(f))
    ccall((:dzo_host_free, libdzopt), Cint, (Ptr{Cvoid},), pointer(t))
    return nothing
end
# after step!(opt): the mirrors are current once these return
mirrored_objective_values!(opt::BatchedBFGSOptimizer, f::Vector{Float64}) =
    (check(ccall((:dzo_bfgs_get_objective, libdzopt), Cint, (Ptr{Cvoid}, Ptr{Float64}), opt.handle, f)); f)
mirrored_terminated!(opt::BatchedBFGSOptimizer, t::Vector{UInt8}) =
    (check(ccall((:dzo_bfgs_get_terminated, libdzopt), Cint, (Ptr{Cvoid}, Ptr{UInt8}), opt.handle, t)); t)

function count_active(opt::BatchedBFGSOptimizer)
    c = Ref{Int64}(0)
    check(ccall((:dzo_bfgs_count_active, libdzopt), Cint, (Ptr{Cvoid}, Ref{Int64}), opt.handle, c))
    return c[]
end

# What the step! calls did, counted on the device (dzo_bfgs_get_step_kind_counts): BFGS-type steps that read H / whose H
# was the implicit identity, gradient-descent steps, terminations, step! calls on terminated problems.
function step_kind_counts(opt::BatchedBFGSOptimizer; reset::Bool=false)
    c = zeros(Int64, 8)
    check(ccall((:dzo_bfgs_get_step_kind_counts, libdzopt), Cint, (Ptr{Cvoid}, Ptr{Int64}, Cint), opt.handle, c, reset ? 1 : 0))
    return (bfgs_read_h=c[1], bfgs_identity_h=c[2], gradient_descent=c[3], terminate=c[4], idle=c[5] + c[6])
end

# ================================================================== LBFGSOptimizer (live src/DZOptimization.jl:321-509)
mutable struct LBFGSOptimizer
    handle::Ptr{Cvoid}
    n::Int
    history_length::Int
end
# LBFGSOptimizer(c!, f, g!, x0, initial_step_length, history_length)  :400-427 ; c! may be `nothing`
function LBFGSOptimizer(c!, f, g!, x0::Vector{Float64}, step::Float64, history_length::Int; device::Integer=0)
    obj, cid = resolve(f, g!, c! === nothing ? NULL_CONSTRAINT : c!)
    @assert step > 0                                                                 # :375
    h = Ref{Ptr{Cvoid}}(C_NULL)
    check(ccall((:dzo_lbfgs_create, libdzopt), Cint,
        (Ref{Ptr{Cvoid}}, Cint, Cint, Int64, Int64, Ptr{Float64}, Float64, Cint, Cint),
        h, obj, cid, 0, length(x0), x0, step, history_length, device))
    opt = LBFGSOptimizer(h[], length(x0), history_length)
    finalizer(o -> ccall((:dzo_lbfgs_destroy, libdzopt), Cvoid, (Ptr{Cvoid},), o.handle), opt)
    return opt
end
function step!(opt::LBFGSOptimizer)                                                 # :454-509
    check(ccall((:dzo_lbfgs_step, libdzopt), Cint, (Ptr{Cvoid}, Cint), getfield(opt, :handle), 1))
    return opt
end
function Base.getproperty(opt::LBFGSOptimizer, s::Symbol)
    h, n = getfield(opt, :handle), getfield(opt, :n)
    vec(sym) = (out = Vector{Float64}(undef, n); check(ccall((sym, libdzopt), Cint, (Ptr{Cvoid}, Ptr{Float64}), h, out)); out)
    sc(sym, T) = (out = Array{T,0}(undef); check(ccall((sym, libdzopt), Cint, (Ptr{Cvoid}, Ptr{T}), h, out)); out)
    s === :current_point && return vec(:dzo_lbfgs_get_point)                        # :330
    s === :delta_point && return vec(:dzo_lbfgs_get_delta_point)                    # :331
    s === :current_gradient && return vec(:dzo_lbfgs_get_gradient)                  # :334
    s === :delta_gradient && return vec(:dzo_lbfgs_get_delta_gradient)              # :335
    s === :step_direction && return vec(:dzo_lbfgs_get_direction)                   # :337
    s === :current_objective_value && return sc(:dzo_lbfgs_get_objective, Float64)  # :332
    s === :delta_objective_value && return sc(:dzo_lbfgs_get_delta_objective, Float64)  # :333
    s === :iteration_count && return sc(:dzo_lbfgs_get_iteration_count, Int64)      # :328
    if s === :is_stuck || s === :has_converged                                      # :327
        t = sc(:dzo_lbfgs_get_stuck, UInt8)
        return fill(t[] != 0)
    end
    return getfield(opt, s)
end

# `batch` independent live LBFGSOptimizers in one handle (dzo_lbfgs_create_batched, one device thread per problem, every
# sum in the reference's sequential order); x0 is n x batch, scalar fields come back as Vectors.  (c! = NULL_CONSTRAINT)
mutable struct BatchedLBFGSOptimizer
    handle::Ptr{Cvoid}
    n::Int
    batch::Int
    history_length::Int
end
function BatchedLBFGSOptimizer(c!, f, g!, x0::Matrix{Float64}, step::Float64, history_length::Int; device::Integer=0)
    obj, cid = resolve(f, g!, c! === nothing ? NULL_CONSTRAINT : c!)
    @assert step > 0                                                                 # :375
    h = Ref{Ptr{Cvoid}}(C_NULL)
    check(ccall((:dzo_lbfgs_create_batched, libdzopt), Cint,
        (Ref{Ptr{Cvoid}}, Cint, Cint, Int64, Int64, Int64, Ptr{Float64}, Float64, Cint, Cint),
        h, obj, cid, 0, size(x0, 1), size(x0, 2), x0, step, history_length, device))
    opt = BatchedLBFGSOptimizer(h[], size(x0, 1), size(x0, 2), history_length)
    finalizer(o -> ccall((:dzo_lbfgs_destroy, libdzopt), Cvoid, (Ptr{Cvoid},), o.handle), opt)
    return opt
end
function step!(opt::BatchedLBFGSOptimizer, k::Integer=1)     # k consecutive step! calls in ONE kernel launch
    check(ccall((:dzo_lbfgs_step, libdzopt), Cint, (Ptr{Cvoid}, Cint), opt.handle, k))
    return opt
end
function current_points(opt::BatchedLBFGSOptimizer)
    out = Matrix{Float64}(undef, opt.n, opt.batch)
    check(ccall((:dzo_lbfgs_get_point, libdzopt), Cint, (Ptr{Cvoid}, Ptr{Float64}), opt.handle, out))
    return out
end
function current_objective_values(opt::BatchedLBFGSOptimizer)
    out = Vector{Float64}(undef, opt.batch)
    check(ccall((:dzo_lbfgs_get_objective, libdzopt), Cint, (Ptr{Cvoid}, Ptr{Float64}), opt.handle, out))
    return out
end
function is_stuck_values(opt::BatchedLBFGSOptimizer)
    out = Vector{UInt8}(undef, opt.batch)
    check(ccall((:dzo_lbfgs_get_stuck, libdzopt), Cint, (Ptr{Cvoid}, Ptr{UInt8}), opt.handle, out))
    return out .!= 0
end

# ================================================================== AdGDOptimizer (live src/DZOptimization.jl:179-312)
mutable struct AdGDOptimizer
    handle::Ptr{Cvoid}
    n::Int
end
function AdGDOptimizer(c!, f, g!, x0::Vector{Float64}, step::Float64; device::Integer=0)      # :252-271
    obj, cid = resolve(f, g!, c! === nothing ? NULL_CONSTRAINT : c!)
    @assert step > 0                                                                 # :232
    h = Ref{Ptr{Cvoid}}(C_NULL)
    check(ccall((:dzo_adgd_create, libdzopt), Cint,
        (Ref{Ptr{Cvoid}}, Cint, Cint, Int64, Int64, Ptr{Float64}, Float64, Cint),
        h, obj, cid, 0, length(x0), x0, step, device))
    opt = AdGDOptimizer(h[], length(x0))
    finalizer(o -> ccall((:dzo_adgd_destroy, libdzopt), Cvoid, (Ptr{Cvoid},), getfield(o, :handle)), opt)
    return opt
end
function step!(opt::AdGDOptimizer)                                                  # :274-312
    check(ccall((:dzo_adgd_step, libdzopt), Cint, (Ptr{Cvoid}, Cint), getfield(opt, :handle), 1))
    return opt
end
function Base.getproperty(opt::AdGDOptimizer, s::Symbol)
    h, n = getfield(opt, :handle), getfield(opt, :n)
    vec(sym) = (out = Vector{Float64}(undef, n); check(ccall((sym, libdzopt), Cint, (Ptr{Cvoid}, Ptr{Float64}), h, out)); out)
    s === :current_point && return vec(:dzo_adgd_get_point)                         # :188
    s === :delta_point && return vec(:dzo_adgd_get_delta_point)                     # :189
    s === :current_gradient && return vec(:dzo_adgd_get_gradient)                   # :192
    s === :delta_gradient && return vec(:dzo_adgd_get_delta_gradient)               # :193
    sc = Vector{Float64}(undef, 6)
    check(ccall((:dzo_adgd_get_scalars, libdzopt), Cint, (Ptr{Cvoid}, Ptr{Float64}), h, sc))
    s === :current_objective_value && return fill(sc[1])                            # :190
    s === :delta_objective_value && return fill(sc[2])                              # :191
    s === :current_step_size && return fill(sc[3])                                  # :195
    s === :previous_step_size && return fill(sc[4])                                 # :196
    s === :iteration_count && return fill(Int(sc[5]))                               # :186
    (s === :is_stuck || s === :has_converged) && return fill(sc[6] != 0)            # :185
    return getfield(opt, s)
end

# ================================================================== legacy decorators (legacy/DZOptimization.jl:222-296)
# The reference wraps callables; here the wrappers are peeled into decorator bits for the device objective.
struct L2RegularizationWrapper{F}; objective_function::F; lambda::Float64; end           # :228-234
struct L2GradientWrapper{G}; gradient_function!::G; lambda::Float64; end                 # :237-251
struct UniformBoxConstraint; lower_bound::Float64; upper_bound::Float64; end            # :257-272
struct UniformBoxGradientWrapper{G}; gradient_function!::G; lower_bound::Float64; upper_bound::Float64; end   # :275-296

function resolve_decorated(c!, f, g!)
    lam_f = lam_g = nothing
    box_c = box_g = nothing
    if f isa L2RegularizationWrapper; lam_f = f.lambda; f = f.objective_function; end
    if g! isa UniformBoxGradientWrapper; box_g = (g!.lower_bound, g!.upper_bound); g! = g!.gradient_function!; end
    if g! isa L2GradientWrapper; lam_g = g!.lambda; g! = g!.gradient_function!; end
    g! isa UniformBoxGradientWrapper && throw(ArgumentError("device order is UniformBoxGradientWrapper(L2GradientWrapper(g!, lambda), lo, hi)"))
    if c! isa UniformBoxConstraint; box_c = (c!.lower_bound, c!.upper_bound); c! = NULL_CONSTRAINT; end
    c! === nothing && (c! = NULL_CONSTRAINT)
    lam_f == lam_g || throw(ArgumentError("L2RegularizationWrapper and L2GradientWrapper must share one lambda"))
    box_c == box_g || throw(ArgumentError("UniformBoxConstraint and UniformBoxGradientWrapper must share their bounds"))
    obj, cid = resolve(f, g!, c!)
    return obj, cid, lam_f, box_c
end

# ================================================================== legacy LBFGSOptimizer (legacy/DZOptimization.jl:458-695)
# (the live package's optimizer of the same name is LBFGSOptimizer above)
mutable struct LegacyLBFGSOptimizer
    handle::Ptr{Cvoid}
    n::Int
    m::Int
end
function LegacyLBFGSOptimizer(c!, f, g!, ls::QuadraticLineSearch, x0::Vector{Float64}, step::Float64,
    history_length::Int; device::Integer=0)                                         # :489-548
    obj, cid, lam, box = resolve_decorated(c!, f, g!)
    @assert history_length > 0                                                       # :528
    decor = (lam === nothing ? 0 : 1) | (box === nothing ? 0 : 2)
    lo, hi = box === nothing ? (0.0, 0.0) : box
    h = Ref{Ptr{Cvoid}}(C_NULL)
    check(ccall((:dzo_legacy_lbfgs_create, libdzopt), Cint,
        (Ref{Ptr{Cvoid}}, Cint, Cint, Int64, Int64, Ptr{Float64}, Float64, Cint, Cint, Cint, Float64, Float64, Float64, Cint),
        h, obj, cid, 0, length(x0), x0, step, history_length, ls.max_increases, decor,
        lam === nothing ? 0.0 : lam, lo, hi, device))
    opt = LegacyLBFGSOptimizer(h[], length(x0), history_length)
    finalizer(o -> ccall((:dzo_legacy_lbfgs_destroy, libdzopt), Cvoid, (Ptr{Cvoid},), getfield(o, :handle)), opt)
    return opt
end
LegacyLBFGSOptimizer(f, g!, ls::QuadraticLineSearch, x0::Vector{Float64}, step::Float64, history_length::Int; kw...) =
    LegacyLBFGSOptimizer(NULL_CONSTRAINT, f, g!, ls, x0, step, history_length; kw...)   # :551-562
function step!(opt::LegacyLBFGSOptimizer)                                           # :565-695
    check(ccall((:dzo_legacy_lbfgs_step, libdzopt), Cint, (Ptr{Cvoid}, Cint), getfield(opt, :handle), 1))
    return opt
end
function Base.getproperty(opt::LegacyLBFGSOptimizer, s::Symbol)
    h, n, m = getfield(opt, :handle), getfield(opt, :n), getfield(opt, :m)
    vec(sym) = (out = Vector{Float64}(undef, n); check(ccall((sym, libdzopt), Cint, (Ptr{Cvoid}, Ptr{Float64}), h, out)); out)
    s === :current_point && return vec(:dzo_legacy_lbfgs_get_point)                 # :461
    s === :delta_point && return vec(:dzo_legacy_lbfgs_get_delta_point)             # :462
    s === :current_gradient && return vec(:dzo_legacy_lbfgs_get_gradient)           # :469
    s === :delta_gradient && return vec(:dzo_legacy_lbfgs_get_delta_gradient)       # :470
    s === :next_step_direction && return vec(:dzo_legacy_lbfgs_get_direction)       # :473
    if s === :_rho || s === :_alpha                                                 # :480-481
        rho, alpha = Vector{Float64}(undef, m), Vector{Float64}(undef, m)
        check(ccall((:dzo_legacy_lbfgs_get_history, libdzopt), Cint, (Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}), h, rho, alpha))
        return s === :_rho ? rho : alpha
    end
    sc = Vector{Float64}(undef, 6)
    check(ccall((:dzo_legacy_lbfgs_get_scalars, libdzopt), Cint, (Ptr{Cvoid}, Ptr{Float64}), h, sc))
    s === :current_objective_value && return fill(sc[1])                            # :465
    s === :delta_objective_value && return fill(sc[2])                              # :466
    s === :last_step_length && return fill(sc[3])                                   # :474
    s === :iteration_count && return fill(Int(sc[4]))                               # :477
    (s === :has_terminated || s === :has_converged) && return fill(sc[5] != 0)      # :478
    s === :_history_count && return fill(Int(sc[6]))                                # :484
    return getfield(opt, s)
end

# ================================================================== LineSearchEvaluator (live src/DZOptimization.jl:12-92)
struct LineSearchEvaluator
    objective::Cint
    constraint::Cint
    current_point::Vector{Float64}
    current_objective_value::Array{Float64,0}
    current_gradient::Vector{Float64}
    step_direction::Vector{Float64}
    overlap::Array{Float64,0}
    trial_point::Vector{Float64}
    trial_objective_value::Array{Float64,0}
    trial_gradient::Vector{Float64}
    improvement_ratio::Array{Float64,0}
    slope_ratio::Array{Float64,0}
end
function LineSearchEvaluator(c!, f, g!, x::Vector{Float64}, fx::Float64, gx::Vector{Float64}, dir::Vector{Float64},
    overlap::Float64)                                                                # :29-63
    obj, cid = resolve(f, g!, c! === nothing ? NULL_CONSTRAINT : c!)
    @assert axes(x) == axes(gx) == axes(dir)                                         # :41-43
    return LineSearchEvaluator(obj, cid, x, fill(fx), gx, dir, fill(overlap), similar(x), Array{Float64,0}(undef),
        similar(gx), Array{Float64,0}(undef), Array{Float64,0}(undef))
end
function (lse::LineSearchEvaluator)(step_size::Float64, compute_gradient::Bool)      # :66-92
    res = Vector{Float64}(undef, 3)
    check(ccall((:dzo_dev_line_search_evaluate, libdzopt), Cint,
        (Cint, Cint, Int64, Cint, Int64, Ptr{Float64}, Float64, Ptr{Float64}, Float64, Float64, Cint, Ptr{Float64},
            Ptr{Float64}, Ptr{Float64}, Cint),
        lse.objective, lse.constraint, 0, 1, length(lse.current_point), lse.current_point, lse.current_objective_value[],
        lse.step_direction, lse.overlap[], step_size, compute_gradient ? 1 : 0, lse.trial_point, lse.trial_gradient, res, 0))
    lse.trial_objective_value[] = res[1]
    lse.improvement_ratio[] = res[2]
    compute_gradient && (lse.slope_ratio[] = res[3])
    return res[1]
end

# ================================================================== pairwise radial kernels (live src/ExampleFunctions.jl)
# Host Vectors here; a CUDA.jl user passes `pointer(cu_x)` to the dzo_pairwise_*_device entry points instead and
# gets the reference's asynchronous launch semantics (src/ExampleFunctions.jl:171, :292, :463-466).
function accelerated_pairwise_radial_energy(f::RadialFunction, x::Vector{Float64}, y::Vector{Float64},
    z::Vector{Float64}; order::Integer=0, workgroupsize::Int=256)                   # :152-173
    @assert f.derivative == 0 && axes(x) == axes(y) == axes(z)
    e = Ref{Float64}(0.0)
    check(ccall((:dzo_dev_pairwise_energy, libdzopt), Cint,
        (Cint, Cint, Int64, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ref{Float64}, Cint),
        f.potential, order, length(x), x, y, z, C_NULL, e, 0))
    return e[]
end
function accelerated_pairwise_radial_gradient!(gx, gy, gz, f::RadialFunction, x::Vector{Float64},
    y::Vector{Float64}, z::Vector{Float64}; order::Integer=0, workgroupsize::Int=256)   # :265-294
    @assert f.derivative == 1 && axes(gx) == axes(gy) == axes(gz) == axes(x) == axes(y) == axes(z)
    check(ccall((:dzo_dev_pairwise_gradient, libdzopt), Cint,
        (Cint, Cint, Int64, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Cint),
        f.potential, order, length(x), x, y, z, gx, gy, gz, 0))
    return nothing
end
function accelerated_pairwise_radial_hvp!(px, py, pz, f1::RadialFunction, f2::RadialFunction, x, y, z, u, v, w;
    order::Integer=0, workgroupsize::Int=256)                                       # :427-468
    @assert f1.derivative == 1 && f2.derivative == 2 && f1.potential == f2.potential
    check(ccall((:dzo_dev_pairwise_hvp, libdzopt), Cint,
        (Cint, Cint, Int64, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64},
            Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Cint),
        f1.potential, order, length(x), x, y, z, u, v, w, px, py, pz, 0))
    return nothing
end

end # module
