# PixellB200.jl -- Julia host side of the B200 SHT engine: Pixell.jl's map2alm / alm2map method table
# (src/transforms.jl:88-265 of simonsobs/Pixell.jl v0.2.9) on top of the C ABI of libpixsht.so (include/pixsht.h).
#
# NOT EXECUTED IN THE BUILD IMAGE (no Julia there, SURVEY.md F12); kept thin enough to be checked by inspection: every
# method only (1) derives the ring geometry from the WCS exactly as the reference does, (2) `ccall`s one C function
# with the caller's own arrays, (3) wraps the result in the reference's return type.  The Python mirror
# pixell.jl_b200/pixsht/transforms.py is the same logic, and that one is exercised by the test-suite.
#
# Usage inside Pixell (see INTEGRATION.md): `include("PixellB200.jl"); using .PixellB200` after `using Pixell`; the
# methods below are more specific than nothing in Pixell -- they REPLACE the libsharp-backed ones, so load this file
# instead of src/transforms.jl, or call `PixellB200.map2alm` / `PixellB200.alm2map` explicitly.
module PixellB200

using Pixell: Enmap, getwcs, pix2sky, slice_geometry
import Healpix: Alm

const libpixsht = get(ENV, "PIXSHT_LIB", joinpath(@__DIR__, "..", "lib", "libpixsht.so"))

const PIXSHT_F64, PIXSHT_F32 = Cint(0), Cint(1)
const PIXSHT_MAP2ALM, PIXSHT_ALM2MAP = Cint(0), Cint(1)
const PIXSHT_HOST = Cint(0)
const PIXSHT_POLCONV_COSMO, PIXSHT_POLCONV_IAU = Cint(0), Cint(1)

# mirrors `struct pixsht_geom` of include/pixsht.h (field order and widths matter)
struct PixshtGeom
    nphi::Int32
    nrings_total::Int32
    ring_first::Int32
    nrings::Int32
    nx::Int32
    flipx::Int32
    flipy::Int32
    ring_scheme::Int32     # 0: Clenshaw-Curtis rings (the reference's SHT grid), 1: Fejer-1
    phi0::Float64
end

struct PixshtError <: Exception
    code::Int
    msg::String
end
Base.showerror(io::IO, e::PixshtError) = print(io, "pixsht error ", e.code, ": ", e.msg)

last_error() = unsafe_string(ccall((:pixsht_last_error, libpixsht), Cstring, ()))
check(rc::Integer) = rc == 0 ? nothing : throw(PixshtError(rc, last_error()))

# ---- ring bookkeeping: the reference's own helpers (src/transforms.jl:3-30,85) do the work -----------------------
import Pixell: fullringsize, fullringnum, getlmax, first_last_rings_in_fullsky, get_flip_slices

"""Describe how an (nx, ny) map with `wcs` sits on the full-sky CC ring grid (pixsht_geom).  Same derivation as
make_cc_geom_info (src/transforms.jl:33-46): flip slices -> sliced WCS -> ring sub-range and phi0.  The reference then
flips/pads the map on the host (create_sht_band, :66-82); here the flips/padding are two flags and `nx`, applied inside
the FFT kernels, so the caller's array is passed untouched."""
function sht_geom(shape, wcs0)
    fx, fy = get_flip_slices(shape, wcs0)
    _, wcs = slice_geometry(shape, wcs0, fx, fy, shape[3:end])
    subinds = first_last_rings_in_fullsky(shape, wcs)
    @assert first(subinds) ≤ last(subinds)                 # vertical angle must be increasing (:38)
    @assert length(subinds) == shape[2]
    phi0 = pix2sky(shape, wcs, 1, 2)[1]                    # (:41)
    PixshtGeom(fullringsize(wcs), fullringnum(wcs), first(subinds) - 1, shape[2], shape[1],
               step(fx) < 0, step(fy) < 0, 0, phi0)
end

# ---- plans: one per (geometry, lmax, mmax, eltype); finalizer frees the device tables -------------------------------
mutable struct Plan
    ptr::Ptr{Cvoid}
    nalm::Int
end

const PLANS = Dict{Any,Plan}()
const PLAN_LOCK = ReentrantLock()

"GPUs of the plans: ENV[\"PIXSHT_DEVICES\"] = \"0,1,2,3\" -> one process drives all of them (pixsht_plan_create_multi); default: GPU 0."
function devices()
    v = strip(get(ENV, "PIXSHT_DEVICES", ""))
    isempty(v) ? Cint[0] : Cint[parse(Cint, x) for x in split(v, ',') if !isempty(strip(x))]
end

function plan_for(shape, wcs, lmax::Int, mmax::Int, ::Type{T}) where {T<:Union{Float32,Float64}}
    g = sht_geom(shape, wcs)
    devs = devices()
    key = (g, lmax, mmax, T, Tuple(devs))
    lock(PLAN_LOCK) do
        get!(PLANS, key) do
            out = Ref{Ptr{Cvoid}}(C_NULL)
            dt = T === Float64 ? PIXSHT_F64 : PIXSHT_F32
            if length(devs) == 1
                check(ccall((:pixsht_plan_create, libpixsht), Cint,
                            (Ref{Ptr{Cvoid}}, Ref{PixshtGeom}, Cint, Cint, Cint, Cint),
                            out, g, lmax, mmax, dt, devs[1]))
            else
                # one blocking call, N GPUs: m-sharded Legendre stage, ring-sharded FFT stage, phase rows exchanged over NVLink
                check(ccall((:pixsht_plan_create_multi, libpixsht), Cint,
                            (Ref{Ptr{Cvoid}}, Ref{PixshtGeom}, Cint, Cint, Cint, Cint, Ptr{Cint}),
                            out, g, lmax, mmax, dt, length(devs), devs))
            end
            p = Plan(out[], Int(ccall((:pixsht_nalm, libpixsht), Int64, (Cint, Cint), lmax, mmax)))
            finalizer(p) do q   # thread-safe in the library; tolerates a torn-down CUDA context
                ccall((:pixsht_plan_destroy, libpixsht), Cvoid, (Ptr{Cvoid},), q.ptr)
            end
            p
        end
    end
end

# Stokes-U sign convention of the maps handed to the next calls on this plan (pixsht_plan_set_polconv).  Pixell's read_map
# negates U of a POLCCONV = "IAU" file on the host (resolve_polcconv!, src/enmap.jl:178-196); `read_map(...)` followed by
# `map2alm(m)` therefore keeps working unchanged.  To skip that host pass over the map, keep the file's values
# (`read_map(path; wcs=...)` or FITSIO directly) and call `map2alm(m; polcconv="IAU")`: the sign is applied inside the FFT kernels.
function set_polconv!(p::Plan, polcconv::AbstractString)
    c = polcconv == "IAU" ? PIXSHT_POLCONV_IAU : polcconv == "COSMO" ? PIXSHT_POLCONV_COSMO :
        throw(ArgumentError("polcconv must be \"COSMO\" or \"IAU\""))
    check(ccall((:pixsht_plan_set_polconv, libpixsht), Cint, (Ptr{Cvoid}, Cint), p.ptr, c))
end

function execute!(p::Plan, dir::Cint, alms::Vector{<:AbstractVector}, maps::Vector{<:AbstractArray})
    ncomp = length(alms)
    GC.@preserve alms maps begin
        aptr = Ptr{Cvoid}[pointer(a) for a in alms]
        mptr = Ptr{Cvoid}[pointer(m) for m in maps]
        check(ccall((:pixsht_execute, libpixsht), Cint,
                    (Ptr{Cvoid}, Cint, Cint, Ptr{Ptr{Cvoid}}, Ptr{Ptr{Cvoid}}, Cint),
                    p.ptr, dir, ncomp, aptr, mptr, PIXSHT_HOST))
    end
end

# map2alm refined by `niter` Jacobi iterations, a <- a + A(m - Y a), with the maps, residual and alm kept on the GPU between
# iterations (pixsht_map2alm_iter; niter = 0 is exactly execute!(p, PIXSHT_MAP2ALM, ...)).  Single-GPU plans only.
function map2alm_iter!(p::Plan, alms::Vector{<:AbstractVector}, maps::Vector{<:AbstractArray}, niter::Integer)
    ncomp = length(alms)
    GC.@preserve alms maps begin
        aptr = Ptr{Cvoid}[pointer(a) for a in alms]
        mptr = Ptr{Cvoid}[pointer(m) for m in maps]
        check(ccall((:pixsht_map2alm_iter, libpixsht), Cint,
                    (Ptr{Cvoid}, Cint, Ptr{Ptr{Cvoid}}, Ptr{Ptr{Cvoid}}, Cint, Cint),
                    p.ptr, ncomp, aptr, mptr, niter, PIXSHT_HOST))
    end
end

# The reference promotes every map to Float64 before the transform (create_sht_band, src/transforms.jl:71) and returns
# ComplexF64 alm; so does this binding.  ENV["PIXSHT_F32_BOUNDARY"] = "1" opts in to the Float32-boundary plan for Float32
# maps (half the PCIe volume, ring FFTs in Float32: ~1e-7 relative, NOT the reference's numerics).
f32_boundary() = get(ENV, "PIXSHT_F32_BOUNDARY", "0") == "1"
compute_type(::Type{Float32}) = f32_boundary() ? Float32 : Float64
compute_type(::Type) = Float64

# Page-locked host arrays for the library's outputs (pixsht_host_alloc): the host-pointer call overlaps its copies with the
# kernels only from / to page-locked memory.  The finalizer returns the memory to the library.
function pinned_zeros(::Type{T}, dims::Int...) where {T}
    n = prod(dims)
    ptr = Ref{Ptr{Cvoid}}(C_NULL)
    check(ccall((:pixsht_host_alloc, libpixsht), Cint, (Ref{Ptr{Cvoid}}, Csize_t), ptr, max(n, 1) * sizeof(T)))
    a = unsafe_wrap(Array, Ptr{T}(ptr[]), dims; own=false)
    fill!(a, zero(T))
    finalizer(a) do x
        ccall((:pixsht_host_free, libpixsht), Cint, (Ptr{Cvoid},), pointer(x))
    end
    a
end
"Page-lock an array the caller owns for the duration of `f` (pixsht_host_register / pixsht_host_unregister)."
function with_registered(f, arrays...)
    regs = Ptr{Cvoid}[]
    try
        for a in arrays
            check(ccall((:pixsht_host_register, libpixsht), Cint, (Ptr{Cvoid}, Csize_t), pointer(a), sizeof(a)))
            push!(regs, pointer(a))
        end
        GC.@preserve arrays f()
    finally
        for p in regs
            ccall((:pixsht_host_unregister, libpixsht), Cint, (Ptr{Cvoid},), p)
        end
    end
end
as_complex(a::AbstractVector{ComplexF64}) = a                 # already the library's element type: no copy
as_complex(a::AbstractVector) = ComplexF64.(a)

# a contiguous column-major plane of eltype T is passed as it is (Array, or a contiguous view such as m[:, :, c]);
# anything else is copied / converted once
is_dense(m::Array) = true
is_dense(m::SubArray) = Base.iscontiguous(m)
is_dense(m) = false
dense(m::AbstractArray{T}, ::Type{T}) where {T} = is_dense(m) ? m : Array(m)
dense(m::AbstractArray, ::Type{T}) where {T} = Array{T}(m)

# ---- map2alm: src/transforms.jl:88-165 -------------------------------------------------------------------------
function _map2alm(maps::Vector, wcs, shape; lmax=nothing, mmax=lmax, polcconv="COSMO", niter=0)
    if isnothing(lmax)
        lmax = getlmax(wcs); mmax = lmax
    end
    T = compute_type(eltype(maps[1]))
    p = plan_for(shape, wcs, lmax, mmax, T)
    set_polconv!(p, polcconv)
    planes = [dense(m, T) for m in maps]
    alms = [pinned_zeros(Complex{T}, p.nalm) for _ in planes]
    niter == 0 ? execute!(p, PIXSHT_MAP2ALM, alms, planes) : map2alm_iter!(p, alms, planes, niter)
    [Alm(lmax, mmax, as_complex(a)) for a in alms]
end

map2alm(m::Enmap{T,2}; lmax=nothing, mmax=lmax, niter=0) where {T} =
    _map2alm([parent(m)], getwcs(m), size(m); lmax=lmax, mmax=mmax, niter=niter)[1]

function map2alm(ms::NTuple{2,Enmap{T,2}}; lmax=nothing, mmax=lmax, polcconv="COSMO", niter=0) where {T}
    e, b = _map2alm([parent(ms[1]), parent(ms[2])], getwcs(ms[1]), size(ms[1]); lmax=lmax, mmax=mmax, polcconv=polcconv, niter=niter)
    (e, b)
end

function map2alm(ms::NTuple{3,Enmap{T,2}}; lmax=nothing, mmax=lmax, polcconv="COSMO", niter=0) where {T}
    t, e, b = _map2alm([parent(m) for m in ms], getwcs(ms[1]), size(ms[1]); lmax=lmax, mmax=mmax, polcconv=polcconv, niter=niter)
    (t, e, b)
end

function map2alm(m::Enmap{T,3}; lmax=nothing, mmax=lmax, polcconv="COSMO", niter=0) where {T}
    ncomp = size(m, 3)
    1 <= ncomp <= 3 || throw(ArgumentError("SHTs require shape (nx,ny,ncomp) with 1 ≤ ncomp ≤ 3, for I, QU, and IQU."))
    planes = [view(parent(m), :, :, c) for c in 1:ncomp]   # contiguous column-major planes: no copy for Array storage
    out = _map2alm(planes, getwcs(m), size(m)[1:2]; lmax=lmax, mmax=mmax, polcconv=polcconv, niter=niter)
    ncomp == 1 ? out[1] : Tuple(out)
end

# ---- alm2map: src/transforms.jl:206-265 (return types of SURVEY.md F11 preserved) -------------------------------------
function _alm2map(alms::Vector{<:Alm}, shape, wcs; polcconv="COSMO")
    lmax, mmax = alms[1].lmax, alms[1].mmax
    p = plan_for(shape[1:2], wcs, lmax, mmax, Float64)
    set_polconv!(p, polcconv)
    vecs = [as_complex(a.alm) for a in alms]
    maps = [pinned_zeros(Float64, shape[1], shape[2]) for _ in alms]
    execute!(p, PIXSHT_ALM2MAP, vecs, maps)
    [Enmap(m, wcs) for m in maps]
end

alm2map(alm::Alm, shape, wcs) = _alm2map([alm], shape, wcs)[1]
alm2map(alms::NTuple{2,<:Alm}, shape, wcs; polcconv="COSMO") = _alm2map(collect(alms), shape, wcs; polcconv=polcconv)          # Vector of 2 Enmaps (:251)
alm2map(alms::NTuple{3,<:Alm}, shape, wcs; polcconv="COSMO") = Tuple(_alm2map(collect(alms), shape, wcs; polcconv=polcconv))   # Tuple (:254-255)
function alm2map(alms::Vector{<:Alm}, shape, wcs; polcconv="COSMO")
    n = length(alms)
    n == 1 && return alm2map(alms[1], shape, wcs)
    n == 2 && return alm2map((alms[1], alms[2]), shape, wcs; polcconv=polcconv)
    n == 3 && return alm2map((alms[1], alms[2], alms[3]), shape, wcs; polcconv=polcconv)
    throw(ArgumentError("1, 2 or 3 Alm are supported"))
end

# ---- pixel areas: pixareamap / pixareamap! (src/projections/car_proj.jl:265-273, src/enmap_ops.jl:124-138) -----------------
"Pixel area (steradians) of every map row, in the map's row order (pixsht_ring_pixarea); CAR areas do not depend on RA."
function ring_pixarea(shape, wcs)
    g = sht_geom(shape, wcs)
    area = Vector{Float64}(undef, shape[2])
    check(ccall((:pixsht_ring_pixarea, libpixsht), Cint, (Ref{PixshtGeom}, Ptr{Float64}), g, area))
    area
end
function pixareamap!(pixareas::Enmap)
    area = ring_pixarea(size(pixareas), getwcs(pixareas))
    parent(pixareas) .= reshape(area, 1, :)
    pixareas
end
pixareamap(shape, wcs) = pixareamap!(Enmap(Array{Float64}(undef, shape[1], shape[2]), wcs))
pixareamap(m::Enmap) = pixareamap!(similar(m))

# ---- simulation sweeps: many spin-0 maps on one geometry (no counterpart upstream, where this is a loop over map2alm) ----
# Up to four maps share one Legendre recurrence inside the library (pixsht_execute_batch).
function execute_batch!(p::Plan, dir::Cint, alms::Vector{<:AbstractVector}, maps::Vector{<:AbstractArray})
    GC.@preserve alms maps begin
        aptr = Ptr{Cvoid}[pointer(a) for a in alms]
        mptr = Ptr{Cvoid}[pointer(m) for m in maps]
        check(ccall((:pixsht_execute_batch, libpixsht), Cint,
                    (Ptr{Cvoid}, Cint, Cint, Ptr{Ptr{Cvoid}}, Ptr{Ptr{Cvoid}}, Cint),
                    p.ptr, dir, length(alms), aptr, mptr, PIXSHT_HOST))
    end
end

"map2alm of every map of `ms` (same shape and WCS, spin 0); equals `[map2alm(m; lmax, mmax) for m in ms]`."
function map2alm_batch(ms::Vector{<:Enmap{T,2}}; lmax=nothing, mmax=lmax) where {T}
    wcs, shape = getwcs(ms[1]), size(ms[1])
    if isnothing(lmax)
        lmax = getlmax(wcs); mmax = lmax
    end
    C = compute_type(T)
    p = plan_for(shape, wcs, lmax, mmax, C)
    planes = [dense(parent(m), C) for m in ms]
    alms = [pinned_zeros(Complex{C}, p.nalm) for _ in planes]
    execute_batch!(p, PIXSHT_MAP2ALM, alms, planes)
    [Alm(lmax, mmax, as_complex(a)) for a in alms]
end

"alm2map of every Alm of `alms` (same lmax, mmax) onto the same geometry; equals `[alm2map(a, shape, wcs) for a in alms]`."
function alm2map_batch(alms::Vector{<:Alm}, shape, wcs)
    lmax, mmax = alms[1].lmax, alms[1].mmax
    p = plan_for(shape[1:2], wcs, lmax, mmax, Float64)
    vecs = [as_complex(a.alm) for a in alms]
    maps = [pinned_zeros(Float64, shape[1], shape[2]) for _ in alms]
    execute_batch!(p, PIXSHT_ALM2MAP, vecs, maps)
    [Enmap(m, wcs) for m in maps]
end

export map2alm, alm2map, map2alm_batch, alm2map_batch, with_registered, pixareamap, pixareamap!, ring_pixarea

end # module
