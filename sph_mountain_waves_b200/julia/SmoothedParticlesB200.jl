# SmoothedParticlesB200.jl — the reference's `structs.jl`, `core.jl` and `IO.jl` re-implemented as a
# thin `ccall` layer over libsphmw.so (include/sphmw.h).
#
# How it is wired into moschehaus/sph-mountain-waves (INTEGRATION.md §3): in
# `src/SmoothedParticles.jl` the three lines
#       include("structs.jl")   include("core.jl")   include("IO.jl")
# become one `include("b200/SmoothedParticlesB200.jl")`.  Everything else of the package —
# `algebra.jl` (RealVector), `kernels.jl`, `grids.jl` (Grid, covering, generate_particles!),
# `geometry.jl` (Shape, boundarybox, is_inside) and the export lists — stays the reference's own
# code, so `make_system()` of a driver (src/current/wcsph_perturbed_witch.jl:152-170) runs
# unchanged.  The signatures below are the reference's, verbatim:
#       ParticleSystem(T::DataType, domain::Shape, h::Float64)              structs.jl:57
#       create_cell_list!(sys)                                              core.jl:51
#       apply!(sys, action!; self=false, parameters...)                     core.jl:151
#       apply_unary!(sys, action!) / apply_binary!(sys, action!)            core.jl:125,138
#       ParticleField(sys, var)                                             structs.jl:118
#       new_pvd_file(path) / save_frame!(data, sys, vars...) / save_pvd_file(data)   IO.jl:20-75
#       import_particles!(sys, path, particle_constructor)                  IO.jl:83
# A driver keeps its `mutable struct Particle <: AbstractParticle` and its closures.  Closures
# cannot cross a C ABI (and nothing is compiled at run time): a closure is used as a NAME and must
# belong to the device operator menu (`sphmw_op_list`); the one line a driver adds is
#       use_device_operators!("wcsph"; dt=dt, g=g, c=c, gamma=γ, ...)     # scheme + its constants
# after which `compute_density!` resolves to "wcsph.compute_density", and so on.  Anything outside
# the menu throws (no CPU fallback).
#
# Host/device coherence.  `sys.particles` stays a `Vector{T}` of the driver's mutable structs.
# Device state is authoritative between operators; touching `sys.particles` (diagnostics,
# generate_particles!, plots) first brings the host objects up to date and makes the next device
# call upload them again — correct for arbitrary host code, and cheap for the drivers, which read
# particles only at frame output (every 8-55 steps, wcsph_perturbed_witch.jl:375).
#
# NOT EXECUTED in the build image (no `julia` binary there); the Python ctypes binding
# (sph_mountain_waves_b200/_capi.py) and the C test (tests/c/test_capi.c) call the very same
# symbols with the same struct layout (checked by tests/test_capi_layout.py).

const libsphmw = get(ENV, "LIBSPHMW", joinpath(@__DIR__, "libsphmw.so"))

abstract type AbstractParticle end
abstract type Shape end          # geometry.jl adds the shapes and boundarybox (structs.jl:19)

struct SphmwConfig               # == `struct sphmw_config` (include/sphmw.h), 88 bytes
    box_min::NTuple{3,Cdouble}
    box_max::NTuple{3,Cdouble}
    h::Cdouble
    capacity::Int64
    device::Int32
    flags::Int32
    slab_lo::Int64
    slab_hi::Int64
end

struct SphmwError <: Exception
    code::Int
    msg::String
end
Base.showerror(io::IO, e::SphmwError) = print(io, "libsphmw error ", e.code, ": ", e.msg)
function check(rc::Integer)
    rc < 0 && throw(SphmwError(rc, unsafe_string(ccall((:sphmw_last_error, libsphmw), Cstring, ()))))
    return rc
end

function attribute_type(type::DataType, var::Symbol)
    ind = findfirst(s -> s == var, fieldnames(type))
    ind === nothing && throw("Variable " * string(var) * " does not exist!")   # structs.jl:128-133
    return fieldtypes(type)[ind]
end

"""
    ParticleSystem(T::Type, domain::Shape, h::Float64)

Same contract as structs.jl:43-92: particles of type `T`, removed once outside the bounding box of
`domain`, neighbours within `h`.  Keywords (all optional, none exists in the reference):
`capacity` (device slots; default: grown on demand at the first upload), `device`, `flags`
(SPHMW_FLAG_*), and for x-slabs over several GPUs `rank`, `world`, `nccl_id` (128 bytes from
`comm_unique_id()`, the same on every rank), `halo_capacity`, `open_box` (particles may leave the
bounding box: the library then replays the swap-from-end renumbering of core.jl:72-81 across ranks
after every halo exchange, `sphmw_comm_open_box`).  The adiabatic flow driver ("aflow") runs on slabs
with `open_box=true`; hopkins_total needs `flags=SPHMW_FLAG_GHOST3` (three ghost columns), like the
other Hopkins drivers.
"""
mutable struct ParticleSystem{T<:AbstractParticle}
    h::Float64
    domain::Shape
    key_phase::NTuple{3,Int64}
    key_lim::NTuple{3,Int64}
    key_max::Int64
    key_diff::Vector{Int64}
    _particles::Vector{T}
    ctx::Ptr{Cvoid}
    capacity::Int64
    device::Int
    flags::Int
    slab::NTuple{2,Int64}
    comm::Any                 # (rank, world, id, halo_capacity, open_box) or nothing
    host_touched::Bool        # host objects may differ from the device: upload before the next device call
    device_ahead::Bool        # device state is newer than the host objects
    function ParticleSystem(T::DataType, domain::Shape, h::Float64; capacity::Integer=0, device::Integer=0,
                            flags::Integer=0, rank::Integer=0, world::Integer=1, nccl_id=nothing,
                            halo_capacity::Integer=0, open_box::Bool=false)
        @assert(h > 0.0, "invalid ParticleSystem declaration! (h must be a positive float)")
        @assert(T <: AbstractParticle, "invalid ParticleSystem declaration! (" * string(T) * " is not an AbstractParticle subtype)")
        @assert(hasfield(T, :x) && (attribute_type(T, :x) == RealVector), "invalid ParticleSystem declaration! (particles must have a field `x::RealVector`)")
        box = boundarybox(domain)                                   # structs.jl:63-68
        x_min = (box.x1_min, box.x2_min, box.x3_min)
        x_max = (box.x1_max, box.x2_max, box.x3_max)
        key_phase = Int64.(floor.(x_min ./ h))
        key_lim = Int64.(floor.(x_max ./ h)) .- key_phase .+ 1
        key_diff = Int64[]
        if key_lim[3] == 1
            for di in -1:1, dj in -1:1
                push!(key_diff, di + key_lim[1] * dj)
            end
        else
            for di in -1:1, dj in -1:1, dk in -1:1
                push!(key_diff, di + key_lim[1] * (dj + key_lim[2] * dk))
            end
        end
        slab = (Int64(-1), Int64(-1))
        comm = nothing
        if world > 1
            # equal shares of cell columns, rank r the r-th from the left (slabs.plan_slab)
            lo = div(key_lim[1] * rank, world)
            hi = div(key_lim[1] * (rank + 1), world)
            slab = (Int64(lo), Int64(hi))
            comm = (Int(rank), Int(world), nccl_id, Int64(halo_capacity), open_box)
        end
        sys = new{T}(h, box, key_phase, key_lim, prod(key_lim), key_diff, T[], C_NULL, Int64(capacity), Int(device),
                     Int(flags), slab, comm, true, false)
        finalizer(s -> (s.ctx != C_NULL && ccall((:sphmw_destroy, libsphmw), Cint, (Ptr{Cvoid},), s.ctx); nothing), sys)
        return sys
    end
end

get_particle_type(::ParticleSystem{T}) where T = T

# `sys.particles`: the host objects, brought up to date first; whoever holds them may change them
function Base.getproperty(sys::ParticleSystem, name::Symbol)
    if name === :particles
        getfield(sys, :device_ahead) && download!(sys)
        setfield!(sys, :host_touched, true)
        return getfield(sys, :_particles)
    end
    return getfield(sys, name)
end

# ---- driver constants and the closure -> operator map ---------------------------------------
const PARAMS = Dict{String,Float64}()
const SCHEME = Ref("wcsph")
const OPERATORS = IdDict{Function,String}()
const MENU = Set{String}()

function menu()
    if isempty(MENU)
        n = ccall((:sphmw_op_list, libsphmw), Int64, (Ptr{UInt8}, Int64), C_NULL, 0)
        buf = Vector{UInt8}(undef, n)
        GC.@preserve buf ccall((:sphmw_op_list, libsphmw), Int64, (Ptr{UInt8}, Int64), buf, n)
        for line in split(unsafe_string(pointer(buf)), '\n'; keepempty=false)
            push!(MENU, String(first(split(line, ' '))))
        end
    end
    return MENU
end

"""
    use_device_operators!(scheme; constants...)

The one line a driver adds: which family of device operators its closures name ("wcsph",
"hopkins", "hopkins_full", "hopkins_total", "dambreak", "collision", "flow", "aflow", "packing") and the
values of the module-level constants those closures capture, under libsphmw's names
(`sphmw_set_param`: dt, g, c, gamma, alpha, beta, eps, eta, rho0, R_mass, R_gas, T_bg, rho_floor,
P_floor, z_t, z_b, gamma_r, fluid, ...).
"""
function use_device_operators!(scheme::String; constants...)
    SCHEME[] = scheme
    for (k, v) in constants
        PARAMS[String(k)] = Float64(v)
    end
    return nothing
end
"explicit name for one closure (overrides the scheme rule)"
register_operator!(f::Function, name::String) = (OPERATORS[f] = name; f)

function operator_name(f::Function)
    haskey(OPERATORS, f) && return OPERATORS[f]
    base = replace(String(nameof(f)), "!" => "")
    # closures a driver shares character for character with another one live under that one's name:
    # the Hopkins drivers reuse the WCSPH unary operators, the adiabatic flow driver the isothermal
    # one's accelerate! and internal_force!
    shared = startswith(SCHEME[], "hopkins") ? ("hopkins", "wcsph") : SCHEME[] == "aflow" ? ("flow",) : ()
    for prefix in (SCHEME[], shared...)
        name = prefix * "." * base
        name in menu() && return (OPERATORS[f] = name)
    end
    throw(SphmwError(-3, "closure $(nameof(f)) is not in the device operator menu of scheme '$(SCHEME[])' (no CPU fallback)"))
end

# ---- host <-> device -----------------------------------------------------------------------
function ensure_context!(sys::ParticleSystem{T}) where T
    sys.ctx != C_NULL && return
    N = length(getfield(sys, :_particles))
    cap = max(sys.capacity, N + div(N, 4) + 1024)
    box = sys.domain
    cfg = Ref(SphmwConfig((box.x1_min, box.x2_min, box.x3_min), (box.x1_max, box.x2_max, box.x3_max), sys.h, cap,
                          Int32(sys.device), Int32(sys.flags), sys.slab[1], sys.slab[2]))
    out = Ref{Ptr{Cvoid}}(C_NULL)
    check(ccall((:sphmw_create, libsphmw), Cint, (Ref{SphmwConfig}, Ref{Ptr{Cvoid}}), cfg, out))
    setfield!(sys, :ctx, out[])
    setfield!(sys, :capacity, Int64(cap))
    if sys.comm !== nothing
        rank, world, id, hc, open_box = sys.comm
        id === nothing && throw(SphmwError(-1, "world > 1 needs nccl_id = comm_unique_id() of rank 0"))
        GC.@preserve id check(ccall((:sphmw_comm_init, libsphmw), Cint, (Ptr{Cvoid}, Int32, Int32, Ptr{UInt8}, Int64),
                                    sys.ctx, rank, world, id, hc > 0 ? hc : max(4096, div(cap, 8))))
        open_box && check(ccall((:sphmw_comm_open_box, libsphmw), Cint, (Ptr{Cvoid}, Int32), sys.ctx, 1))
    end
end
"128 bytes identifying an NCCL communicator: made by ONE rank, handed to the others (MPI.bcast, a file ...)"
function comm_unique_id()
    id = zeros(UInt8, 128)
    GC.@preserve id check(ccall((:sphmw_comm_unique_id, libsphmw), Cint, (Ptr{UInt8},), id))
    return id
end

"AoS (vector of heap objects, structs.jl:53) -> SoA staging buffers -> device"
function upload!(sys::ParticleSystem{T}) where T
    ensure_context!(sys)
    ps = getfield(sys, :_particles)
    N = length(ps)
    N > sys.capacity && throw(SphmwError(-4, "$(N) particles exceed the device capacity $(sys.capacity); pass capacity= to ParticleSystem"))
    for (k, v) in PARAMS
        check(ccall((:sphmw_set_param, libsphmw), Cint, (Ptr{Cvoid}, Cstring, Cdouble), sys.ctx, k, v))
    end
    check(ccall((:sphmw_resize, libsphmw), Cint, (Ptr{Cvoid}, Int64), sys.ctx, 0))
    check(ccall((:sphmw_resize, libsphmw), Cint, (Ptr{Cvoid}, Int64), sys.ctx, N))
    for f in fieldnames(T)
        FT = fieldtype(T, f)
        if FT == Float64
            buf = Float64[getfield(p, f) for p in ps]
            GC.@preserve buf check(ccall((:sphmw_upload, libsphmw), Cint, (Ptr{Cvoid}, Cstring, Ptr{Cdouble}, Int64, Int32),
                                         sys.ctx, String(f), buf, N, 1))
        elseif FT == RealVector
            buf = Matrix{Float64}(undef, N, 3)            # component-major: buf[i, c]
            for (i, p) in enumerate(ps), c in 1:3
                buf[i, c] = getfield(p, f)[c]
            end
            GC.@preserve buf check(ccall((:sphmw_upload, libsphmw), Cint, (Ptr{Cvoid}, Cstring, Ptr{Cdouble}, Int64, Int32),
                                         sys.ctx, String(f), buf, N, 3))
        end                                               # other field types stay on the host
    end
    setfield!(sys, :host_touched, false)
    setfield!(sys, :device_ahead, false)
end

"device -> host objects; removal keeps the reference's swap-from-end order (core.jl:72-81)"
function download!(sys::ParticleSystem{T}) where T
    n = Ref{Int64}(0)
    check(ccall((:sphmw_count, libsphmw), Cint, (Ptr{Cvoid}, Ref{Int64}), sys.ctx, n))
    N = n[]
    ps = getfield(sys, :_particles)
    resize!(ps, N)
    for f in fieldnames(T)
        FT = fieldtype(T, f)
        if FT == Float64
            buf = Vector{Float64}(undef, N)
            GC.@preserve buf check(ccall((:sphmw_download, libsphmw), Cint, (Ptr{Cvoid}, Cstring, Ptr{Cdouble}, Int64, Int32),
                                         sys.ctx, String(f), buf, N, 1))
            for i in 1:N; setfield!(ps[i], f, buf[i]); end
        elseif FT == RealVector
            buf = Matrix{Float64}(undef, N, 3)
            GC.@preserve buf check(ccall((:sphmw_download, libsphmw), Cint, (Ptr{Cvoid}, Cstring, Ptr{Cdouble}, Int64, Int32),
                                         sys.ctx, String(f), buf, N, 3))
            for i in 1:N; setfield!(ps[i], f, RealVector(buf[i, 1], buf[i, 2], buf[i, 3])); end
        end
    end
    setfield!(sys, :device_ahead, false)
end
before_device_call!(sys::ParticleSystem) = (getfield(sys, :host_touched) || sys.ctx == C_NULL) && upload!(sys)

# ---- core.jl ---------------------------------------------------------------------------------
dist(p::AbstractParticle, q::AbstractParticle)::Float64 = norm(p.x - q.x)   # core.jl:8-10

"create_cell_list!(sys) — core.jl:51-90 (on a slab context: halo exchange, then the sort)"
function create_cell_list!(sys::ParticleSystem)
    before_device_call!(sys)
    n = Ref{Int64}(0)
    check(ccall((:sphmw_create_cell_list, libsphmw), Cint, (Ptr{Cvoid}, Ref{Int64}), sys.ctx, n))
    setfield!(sys, :device_ahead, true)
    return nothing
end

"apply!(sys, action!; self, parameters...) — core.jl:151-161.  Arity is a property of the device operator; `parameters` (numbers only) are set as driver constants before the call"
function apply!(sys::ParticleSystem, action!::Function; self::Bool=false, parameters...)
    name = operator_name(action!)
    before_device_call!(sys)
    for (k, v) in parameters
        v isa Real || throw(SphmwError(-3, "apply!: parameter $(k) is not a number; closures with such parameters have no device operator"))
        check(ccall((:sphmw_set_param, libsphmw), Cint, (Ptr{Cvoid}, Cstring, Cdouble), sys.ctx, String(k), Float64(v)))
    end
    check(ccall((:sphmw_apply, libsphmw), Cint, (Ptr{Cvoid}, Cstring, Int32), sys.ctx, name, self ? 1 : 0))
    setfield!(sys, :device_ahead, true)
    return nothing
end
apply_unary!(sys::ParticleSystem, action!::Function) = apply!(sys, action!)
apply_binary!(sys::ParticleSystem, action!::Function) = apply!(sys, action!)

"fused fast path ≙ `for k in 1:n verlet_step!(sys) end` (wcsph_perturbed_witch.jl:309-332); optional"
function verlet_steps!(sys::ParticleSystem, n::Integer; scheme::String=SCHEME[])
    before_device_call!(sys)
    check(ccall((:sphmw_step, libsphmw), Cint, (Ptr{Cvoid}, Cstring, Int32), sys.ctx, scheme, n))
    setfield!(sys, :device_ahead, true)
    return nothing
end

"""
    add_new_particles!(sys)

≙ add_new_particles!(sys) of the constant-U flow drivers (isothermal_flow_witch.jl:175-186 under scheme
"flow", adiabatic_flow_witch.jl:197-208 under "aflow"): INFLOW particles that entered the domain turn
FLUID and a successor is created bc_width upstream with the driver's Particle constructor — on the
device.  Returns the number of particles added.  On x-slabs (`open_box=true`) the call is collective:
every rank makes the successors of its own particles with the reference's global indices, and the
number returned is the total over all ranks, as on one GPU.
"""
function add_new_particles!(sys::ParticleSystem)
    before_device_call!(sys)
    n = Ref{Int64}(0)
    if SCHEME[] == "aflow"
        check(ccall((:sphmw_aflow_add_new_particles, libsphmw), Cint, (Ptr{Cvoid}, Ref{Int64}), sys.ctx, n))
    else
        check(ccall((:sphmw_flow_add_new_particles, libsphmw), Cint, (Ptr{Cvoid}, Ref{Int64}), sys.ctx, n))
    end
    setfield!(sys, :device_ahead, true)
    return n[]
end

"""
    point_sums(sys, ops::Vector{String}, X::AbstractMatrix) -> Matrix{Float64}

≙ `sum(sys, f, x)` (core.jl:240-291) at every column of the 3 x n matrix `X`, on the device
(sphmw_point_sum): row o of the result is op o summed over the particles within sys.h of each point, in
the reference's traversal order, with no self-exclusion.  Ops: "count", "mW", "VW", "mW*<f>",
"VW*<f>" (term m W, (m f) W, (m/ρ) W, ((m/ρ) f) W; W = wendland2 in 2D, wendland3 in 3D); <f> is a
field name ("ρ′", "θ", ...) or a vector component "v[0]" (0-based).  Points outside the domain's
bounding box give NaN.  Needs a current cell list (create_cell_list! after the last move!).
"""
function point_sums(sys::ParticleSystem, ops::Vector{String}, X::AbstractMatrix)
    size(X, 1) == 3 || throw(SphmwError(-1, "point_sums: X must be 3 x n"))
    before_device_call!(sys)
    n = size(X, 2)
    soa = Vector{Float64}(undef, 3n)
    for i in 1:n, c in 1:3
        soa[(c - 1) * n + i] = X[c, i]
    end
    out = Vector{Float64}(undef, length(ops) * n)
    GC.@preserve ops begin
        ptrs = [Base.unsafe_convert(Cstring, Base.cconvert(Cstring, o)) for o in ops]
        check(ccall((:sphmw_point_sum, libsphmw), Cint, (Ptr{Cvoid}, Ptr{Cstring}, Int32, Ptr{Float64}, Int64, Ptr{Float64}),
                    sys.ctx, ptrs, length(ptrs), soa, n, out))
    end
    return permutedims(reshape(out, n, length(ops)))
end
"≙ `sum(sys, f, x)` of core.jl:240-291 for a device op string (see point_sums)"
Base.sum(sys::ParticleSystem, op::String, x::RealVector)::Float64 =
    point_sums(sys, [op], reshape([x[1], x[2], x[3]], 3, 1))[1, 1]
Base.sum(sys::ParticleSystem, f::Function, x) =
    throw(SphmwError(-3, "sum: the closure $(nameof(f)) cannot run on the device; a point sum takes a device op string (\"mW\", \"VW*<field>\", ...: see point_sums)"))

assemble_matrix(args...) = throw(SphmwError(-3, "assemble_matrix (ISPH, core.jl:175-246) is outside the device path"))
assemble_vector(args...) = throw(SphmwError(-3, "assemble_vector (ISPH, core.jl:248-291) is outside the device path"))

# ---- structs.jl:118-125 ------------------------------------------------------------------------
struct ParticleField <: AbstractArray{Float64,1}
    sys::ParticleSystem
    varS::Symbol
end
const DataField = ParticleField
Base.size(f::ParticleField) = (length(f.sys.particles),)
Base.getindex(f::ParticleField, i::Int64) = getproperty(f.sys.particles[i], f.varS)
Base.setindex!(f::ParticleField, val::Any, k::Int64) = setproperty!(f.sys.particles[k], f.varS, val)

# ---- IO.jl ---------------------------------------------------------------------------------------
mutable struct DataStorage
    path::String
    frame::Int64
    sys::Union{Nothing,ParticleSystem}
end

"new_pvd_file(path)::DataStorage — IO.jl:20-26"
function new_pvd_file(path::String)::DataStorage
    if !ispath(path)
        mkpath(path)
        @info("created new path: " * path)
    end
    return DataStorage(path, 0, nothing)
end

"save_frame!(data, sys, vars...) — IO.jl:53-75: written straight from the device arrays (frame<k>.vtp, zlib, appended raw)"
function save_frame!(data::DataStorage, sys::ParticleSystem, vars::Symbol...)
    before_device_call!(sys)
    if data.sys === nothing
        check(ccall((:sphmw_pvd_open, libsphmw), Cint, (Ptr{Cvoid}, Cstring), sys.ctx, data.path))
        data.sys = sys
    end
    for var in vars
        attribute_type(get_particle_type(sys), var)           # unknown variable: the reference's exception
    end
    names = [String(v) for v in vars]
    GC.@preserve names begin
        ptrs = [Base.unsafe_convert(Cstring, Base.cconvert(Cstring, n)) for n in names]
        check(ccall((:sphmw_pvd_save_frame, libsphmw), Cint, (Ptr{Cvoid}, Ptr{Cstring}, Int32), sys.ctx, ptrs, length(ptrs)))
    end
    data.frame += 1
end

"save_pvd_file(data) — IO.jl:33-35"
function save_pvd_file(data::DataStorage)
    data.sys === nothing && return
    check(ccall((:sphmw_pvd_close, libsphmw), Cint, (Ptr{Cvoid},), data.sys.ctx))
end

"import_particles!(sys, path, particle_constructor) — IO.jl:83-122, on libsphmw's .vtp reader"
function import_particles!(sys::ParticleSystem, path::String, particle_constructor::Function)
    vtp = Ref{Ptr{Cvoid}}(C_NULL)
    check(ccall((:sphmw_vtp_open, libsphmw), Cint, (Cstring, Ref{Ptr{Cvoid}}), path, vtp))
    try
        np = Ref{Int64}(0); na = Ref{Int32}(0)
        check(ccall((:sphmw_vtp_info, libsphmw), Cint, (Ptr{Cvoid}, Ref{Int64}, Ref{Int32}), vtp[], np, na))
        N = np[]
        read_array(name, ncomp) = begin
            buf = Vector{Float64}(undef, N * ncomp)
            GC.@preserve buf check(ccall((:sphmw_vtp_read, libsphmw), Cint, (Ptr{Cvoid}, Cstring, Ptr{Cdouble}, Int64),
                                         vtp[], name, buf, N * ncomp))
            buf
        end
        arrays = Dict{String,Int}()
        for i in 0:(na[] - 1)
            nm = Vector{UInt8}(undef, 256); nc = Ref{Int32}(0)
            GC.@preserve nm check(ccall((:sphmw_vtp_array, libsphmw), Cint, (Ptr{Cvoid}, Int32, Ptr{UInt8}, Int64, Ref{Int32}),
                                        vtp[], i, nm, 256, nc))
            arrays[unsafe_string(pointer(nm))] = nc[]
        end
        pts = read_array("Points", 3)
        ps = sys.particles                      # (syncs and marks the host as touched)
        N0 = length(ps)
        resize!(ps, N0 + N)
        PType = get_particle_type(sys)
        for i in 1:N
            ps[N0 + i] = particle_constructor(RealVector(pts[3i - 2], pts[3i - 1], pts[3i]))
        end
        for fieldname in fieldnames(PType)
            haskey(arrays, string(fieldname)) || continue
            Type = attribute_type(PType, fieldname)
            vals = read_array(string(fieldname), arrays[string(fieldname)])
            if Type <: Number
                for i in 1:N; setproperty!(ps[N0 + i], fieldname, vals[i]); end
            elseif Type <: RealVector
                for i in 1:N; setproperty!(ps[N0 + i], fieldname, RealVector(vals[3i - 2], vals[3i - 1], vals[3i])); end
            else
                error("Cannot import data field with type:" * string(Type))
            end
        end
    finally
        ccall((:sphmw_vtp_close, libsphmw), Cint, (Ptr{Cvoid},), vtp[])
    end
end
