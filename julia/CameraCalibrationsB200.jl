# CameraCalibrationsB200.jl -- the `ccall` shim a maintainer of CameraCalibrations.jl adds to
# evaluate a fitted `Calibration` on a B200 through libcamcal_b200.so (include/camcal_b200.h).
#
# NOT RUN IN THIS REPOSITORY'S CI: the build image has no Julia (SURVEY.md F1).  The Python
# package `cameracalibrations_b200` binds the very same symbols with ctypes and is what the tests
# and bench.py exercise; this file is the reference-side binding shown in INTEGRATION.md.
#
# Nothing of the reference's API changes: `fit`, `Calibration`, `save`/`load`, the scalar
# callables `c(::RowCol, i)` / `c(::XYZ, i)` and `rectification` stay as they are
# (src/meta.jl:82-103).  This module ADDS batch methods that take whole arrays and run on the GPU.
module CameraCalibrationsB200

using CameraCalibrations: Calibration, RowCol, XYZ
import CameraCalibrations
using StaticArrays

const libcamcal = get(ENV, "LIBCAMCAL_B200", "libcamcal_b200.so")

# ---- PODs of include/camcal_b200.h ------------------------------------------------------------
struct CcIntr            # cc_intr
    frow::Cdouble; fcol::Cdouble; crow::Cdouble; ccol::Cdouble; k::Cdouble; checker_size::Cdouble
end
struct CcView            # cc_view
    rvec::NTuple{3,Cdouble}; tvec::NTuple{3,Cdouble}
end

# Calibration fields -> PODs (src/meta.jl:17-25, src/buildcalibrations.jl:1-6)
function CcIntr(c::Calibration)
    d = c.intrinsic.linear.diag
    t = c.intrinsic.translation
    CcIntr(d[1], d[2], t[1], t[2], c.k, 1 / c.scale.linear.diag[1])
end
function CcView(c::Calibration, i::Int)
    e = c.extrinsics[i]                      # AffineMap{RotationVec, SVector{3}}
    r = e.linear
    CcView((r.sx, r.sy, r.sz), Tuple(e.translation))
end

struct CamcalError <: Exception
    status::Cint
    msg::String
end
function check(rc::Cint)
    rc == 0 && return nothing
    throw(CamcalError(rc, unsafe_string(ccall((:cc_last_error_string, libcamcal), Cstring, ()))))
end

# ---- context ------------------------------------------------------------------------------------
mutable struct Context
    handle::Ptr{Cvoid}
    function Context(device::Integer = 0)
        h = Ref{Ptr{Cvoid}}(C_NULL)
        check(ccall((:cc_ctx_create, libcamcal), Cint, (Cint, Ptr{Ptr{Cvoid}}), device, h))
        ctx = new(h[])
        finalizer(x -> ccall((:cc_ctx_destroy, libcamcal), Cint, (Ptr{Cvoid},), x.handle), ctx)
        ctx
    end
end
const CTX = Ref{Union{Nothing,Context}}(nothing)
# one context per process, created on first use (`something(a, b)` would evaluate b -- a NEW
# context -- on every call, leaking device buffers and discarding the cached rectification plans)
function context()
    ctx = CTX[]
    if ctx === nothing
        ctx = Context(0)
        CTX[] = ctx
    end
    ctx
end

# ---- load hook (src/io.jl:19-26) ------------------------------------------------------------------
# `CameraCalibrations.load` rebuilds the closure chains of the object; this wrapper also derives, once,
# the parameter blocks every batch call passes to the library (by value: no device upload is needed,
# kernel parameters travel in the launch).  What IS device-resident per calibration is the
# rectification tile plan, cached inside the context keyed by (parameters, ratio, axes, frame size).
# The JSON file format is untouched.
struct DeviceCalibration
    c::Calibration
    intr::CcIntr
    views::Vector{CcView}
end
DeviceCalibration(c::Calibration) = DeviceCalibration(c, CcIntr(c), [CcView(c, i) for i in eachindex(c.extrinsics)])
"`load_b200(file)`: `CameraCalibrations.load(file)` plus the cached parameter blocks."
load_b200(file) = DeviceCalibration(CameraCalibrations.load(file))
(d::DeviceCalibration)(args...) = d.c(args...)                       # everything the object can do still works

# ---- batch pixel -> world: bulk form of c.(imgpoints, i), src/buildcalibrations.jl:46 --------
"""
    c(rows::Vector{Float64}, cols::Vector{Float64}, i) -> (x, y, z)

SoA batch of `(c::Calibration)(::RowCol, i)` (src/meta.jl:82) on the GPU (host arrays in and out).
"""
function (c::Calibration)(rows::Vector{Float64}, cols::Vector{Float64}, i::Int)
    n = length(rows); @assert length(cols) == n
    checkbounds(c.extrinsics, i)             # BoundsError like the reference
    x, y, z = similar(rows), similar(rows), similar(rows)
    intr, view = Ref(CcIntr(c)), Ref(CcView(c, i))
    check(ccall((:cc_img2world_f64_host, libcamcal), Cint,
                (Ptr{Cvoid}, Ref{CcIntr}, Ref{CcView}, Ptr{Cdouble}, Ptr{Cdouble}, Ptr{Cdouble},
                 Ptr{Cdouble}, Ptr{Cdouble}, Csize_t),
                context().handle, intr, view, rows, cols, x, y, z, n))
    x, y, z
end

"Batch of `rectification(c, i)` (src/meta.jl:99): z is not computed."
function rectification_batch(c::Calibration, i::Int, rows::Vector{Float64}, cols::Vector{Float64})
    n = length(rows)
    x, y = similar(rows), similar(rows)
    check(ccall((:cc_img2world_f64_host, libcamcal), Cint,
                (Ptr{Cvoid}, Ref{CcIntr}, Ref{CcView}, Ptr{Cdouble}, Ptr{Cdouble}, Ptr{Cdouble},
                 Ptr{Cdouble}, Ptr{Cdouble}, Csize_t),
                context().handle, Ref(CcIntr(c)), Ref(CcView(c, i)), rows, cols, x, y, C_NULL, n))
    x, y
end

# ---- batch world -> pixel: bulk form of c.(objpoints, i), src/buildcalibrations.jl:29 --------
function (c::Calibration)(x::Vector{Float64}, y::Vector{Float64}, z::Vector{Float64}, i::Int)
    n = length(x)
    checkbounds(c.extrinsics, i)
    rows, cols = similar(x), similar(x)
    check(ccall((:cc_world2img_f64_host, libcamcal), Cint,
                (Ptr{Cvoid}, Ref{CcIntr}, Ref{CcView}, Ptr{Cdouble}, Ptr{Cdouble}, Ptr{Cdouble},
                 Ptr{Cdouble}, Ptr{Cdouble}, Csize_t),
                context().handle, Ref(CcIntr(c)), Ref(CcView(c, i)), x, y, z, rows, cols, n))
    rows, cols
end

# ---- many views in one call: the broadcasts c.(pts_v, v) over the views, src/buildcalibrations.jl:29,46 ----
# Points [sum(counts[1:s-1]) + 1, sum(counts[1:s])] use view idxs[s]; one library call (one table upload, one
# pipeline, one wait) for all of them.  Every point's result equals the single-view method's bit for bit.
function _offsets(c::Calibration, n::Integer, idxs::AbstractVector{Int}, counts::AbstractVector{<:Integer})
    @assert length(idxs) == length(counts) >= 1 && all(>=(0), counts) && sum(counts) == n
    foreach(i -> checkbounds(c.extrinsics, i), idxs)        # BoundsError like the reference
    Csize_t[0; cumsum(counts)]
end

"""
    c(rows, cols, idxs::AbstractVector{Int}, counts) -> (x, y, z)

Pixel -> world for consecutive segments of points, segment s with view `idxs[s]` (host arrays).
"""
function (c::Calibration)(rows::Vector{Float64}, cols::Vector{Float64}, idxs::AbstractVector{Int},
                          counts::AbstractVector{<:Integer})
    n = length(rows); @assert length(cols) == n
    offsets = _offsets(c, n, idxs, counts)
    views = [CcView(c, i) for i in idxs]
    x, y, z = similar(rows), similar(rows), similar(rows)
    check(ccall((:cc_img2world_f64_views_host, libcamcal), Cint,
                (Ptr{Cvoid}, Ref{CcIntr}, Ptr{CcView}, Cint, Ptr{Csize_t}, Ptr{Cdouble}, Ptr{Cdouble},
                 Ptr{Cdouble}, Ptr{Cdouble}, Ptr{Cdouble}),
                context().handle, Ref(CcIntr(c)), views, length(views), offsets, rows, cols, x, y, z))
    x, y, z
end

"World -> pixel for consecutive segments of points, segment s with view `idxs[s]` (host arrays)."
function (c::Calibration)(x::Vector{Float64}, y::Vector{Float64}, z::Vector{Float64}, idxs::AbstractVector{Int},
                          counts::AbstractVector{<:Integer})
    n = length(x); @assert length(y) == n && length(z) == n
    offsets = _offsets(c, n, idxs, counts)
    views = [CcView(c, i) for i in idxs]
    rows, cols = similar(x), similar(x)
    check(ccall((:cc_world2img_f64_views_host, libcamcal), Cint,
                (Ptr{Cvoid}, Ref{CcIntr}, Ptr{CcView}, Cint, Ptr{Csize_t}, Ptr{Cdouble}, Ptr{Cdouble},
                 Ptr{Cdouble}, Ptr{Cdouble}, Ptr{Cdouble}),
                context().handle, Ref(CcIntr(c)), views, length(views), offsets, x, y, z, rows, cols))
    rows, cols
end

# ---- the reference's own point types: c(pts, i) on Array{RowCol} / Array{XYZ}, src/meta.jl:82,88 --------
# A RowCol is an SVector{2,Float64} and an XYZ an SVector{3,Float64}, so an Array of them is the packed
# n × 2 / n × 3 layout of cc_*_aos: its memory goes to the library as is, and the result comes back in the
# caller's shape.  These are methods on whole arrays; the scalar callables and `c.(pts, i)` are untouched.
function _map_aos(sym::Symbol, c::Calibration, i::Int, pts::Array, out::Array, dim::Integer)
    checkbounds(c.extrinsics, i)             # BoundsError like the reference
    if sym === :img2world
        check(ccall((:cc_img2world_f64_aos_host, libcamcal), Cint,
                    (Ptr{Cvoid}, Ref{CcIntr}, Ref{CcView}, Cint, Ptr{Csize_t}, Ptr{Cdouble}, Ptr{Cdouble}, Cint, Csize_t),
                    context().handle, Ref(CcIntr(c)), Ref(CcView(c, i)), 1, C_NULL, pts, out, dim, length(pts)))
    else
        check(ccall((:cc_world2img_f64_aos_host, libcamcal), Cint,
                    (Ptr{Cvoid}, Ref{CcIntr}, Ref{CcView}, Cint, Ptr{Csize_t}, Ptr{Cdouble}, Cint, Ptr{Cdouble}, Csize_t),
                    context().handle, Ref(CcIntr(c)), Ref(CcView(c, i)), 1, C_NULL, pts, dim, out, length(pts)))
    end
    out
end

"`c(pts::Array{RowCol}, i)`: `c.(pts, i)` in one call, an Array{XYZ} of the same shape."
(c::Calibration)(pts::Array{RowCol,N}, i::Int) where {N} =
    _map_aos(:img2world, c, i, pts, Array{XYZ,N}(undef, size(pts)), 3)

"`c(pts::Array{XYZ}, i)`: `c.(pts, i)` in one call, an Array{RowCol} of the same shape."
(c::Calibration)(pts::Array{XYZ,N}, i::Int) where {N} =
    _map_aos(:world2img, c, i, pts, Array{RowCol,N}(undef, size(pts)), 3)

"`rectification(c, i).(pts)` in one call (src/meta.jl:99): z is not computed."
rectification_batch(c::Calibration, i::Int, pts::Array{RowCol,N}) where {N} =
    _map_aos(:img2world, c, i, pts, Array{SVector{2,Float64},N}(undef, size(pts)), 2)

# Many views: the loop `c.(pts_v, v)` over views as one concatenation, one call and one array back per view.
function _map_aos_views(sym::Symbol, c::Calibration, ptss::AbstractVector, idxs::AbstractVector{Int}, ::Type{O},
                        dim::Integer) where {O}
    @assert length(ptss) == length(idxs) >= 1
    counts = length.(ptss)
    offsets = _offsets(c, sum(counts), idxs, counts)
    views = [CcView(c, i) for i in idxs]
    pts = reduce(vcat, vec.(ptss))
    out = Vector{O}(undef, length(pts))
    if sym === :img2world
        check(ccall((:cc_img2world_f64_aos_host, libcamcal), Cint,
                    (Ptr{Cvoid}, Ref{CcIntr}, Ptr{CcView}, Cint, Ptr{Csize_t}, Ptr{Cdouble}, Ptr{Cdouble}, Cint, Csize_t),
                    context().handle, Ref(CcIntr(c)), views, length(views), offsets, pts, out, dim, length(pts)))
    else
        check(ccall((:cc_world2img_f64_aos_host, libcamcal), Cint,
                    (Ptr{Cvoid}, Ref{CcIntr}, Ptr{CcView}, Cint, Ptr{Csize_t}, Ptr{Cdouble}, Cint, Ptr{Cdouble}, Csize_t),
                    context().handle, Ref(CcIntr(c)), views, length(views), offsets, pts, dim, out, length(pts)))
    end
    [reshape(out[offsets[s]+1:offsets[s+1]], size(ptss[s])) for s in eachindex(ptss)]
end

"`c(ptss, idxs)`: `[c.(ptss[s], idxs[s]) for s in eachindex(ptss)]` in one call."
(c::Calibration)(ptss::AbstractVector{<:Array{RowCol}}, idxs::AbstractVector{Int}) =
    _map_aos_views(:img2world, c, ptss, idxs, XYZ, 3)
(c::Calibration)(ptss::AbstractVector{<:Array{XYZ}}, idxs::AbstractVector{Int}) =
    _map_aos_views(:world2img, c, ptss, idxs, RowCol, 3)

# ---- full-frame rectification: warp(img, tform, axs), src/plot_calibration.jl:40 -------------
# `imgs` is a stack of frames of size (sz1, sz2, nframes): the memory is passed as is (first
# RowCol axis contiguous).  `ratio` from get_ratio (:8-13), `axs` from get_axes (:1-6).
function warp_batch(c::Calibration, i::Int, imgs::Array{Float32,3}, ratio::Float64,
                    axs::NTuple{2,<:AbstractUnitRange}; fill::Float32 = NaN32, fast::Bool = false)
    sz1, sz2, nf = size(imgs)
    out = similar(imgs)
    axs_min = Int64[first(axs[1]), first(axs[2])]
    check(ccall((:cc_rectify_f32c1_host, libcamcal), Cint,
                (Ptr{Cvoid}, Ref{CcIntr}, Ref{CcView}, Cdouble, Ptr{Int64}, Ptr{Cfloat}, Ptr{Cfloat},
                 Cint, Cint, Csize_t, Csize_t, Cint, Cfloat, Cuint),
                context().handle, Ref(CcIntr(c)), Ref(CcView(c, i)), ratio, axs_min, imgs, out,
                sz1, sz2, sz1, sz1 * sz2, nf, fill, fast ? 1 : 0))
    out
end

# RGB{N0f8} frames: reinterpret(UInt8, imgs) has size (3, sz1, sz2, nframes) = u8c3 layout
function warp_batch(c::Calibration, i::Int, imgs::Array{UInt8,4}, ratio::Float64,
                    axs::NTuple{2,<:AbstractUnitRange}; fill::NTuple{3,UInt8} = (0x00, 0x00, 0x00),
                    fast::Bool = false)
    @assert size(imgs, 1) == 3
    _, sz1, sz2, nf = size(imgs)
    out = similar(imgs)
    axs_min = Int64[first(axs[1]), first(axs[2])]
    check(ccall((:cc_rectify_u8c3_host, libcamcal), Cint,
                (Ptr{Cvoid}, Ref{CcIntr}, Ref{CcView}, Cdouble, Ptr{Int64}, Ptr{UInt8}, Ptr{UInt8},
                 Cint, Cint, Csize_t, Csize_t, Cint, Ptr{UInt8}, Cuint),
                context().handle, Ref(CcIntr(c)), Ref(CcView(c, i)), ratio, axs_min, imgs, out,
                sz1, sz2, sz1, sz1 * sz2, nf, UInt8[fill...], fast ? 1 : 0))
    out
end

# The reference's plot loop (src/plot_calibration.jl:36-42) in ONE call: frames of `imgs` belong to the
# views in order, nframes ÷ length(views) each (frames [(v-1)k+1, vk] use view v, ratios[v] and axs[v]).
# Host arrays go through cc_rectify_views_*_host: one chunk pipeline over all views, with the views' tile
# plans built while the frames stream.
function warp_views(d::DeviceCalibration, imgs::Array{Float32,3}, ratios::Vector{Float64},
                    axss::Vector{<:NTuple{2,<:AbstractUnitRange}}; fill::Float32 = NaN32, fast::Bool = false)
    sz1, sz2, nf = size(imgs)
    nv = length(d.views)
    @assert nv > 0 && nf % nv == 0 && nv == length(ratios) == length(axss)
    out = similar(imgs)
    axs_mins = Int64[first(a[j]) for a in axss for j in 1:2]
    check(ccall((:cc_rectify_views_f32c1_host, libcamcal), Cint,
                (Ptr{Cvoid}, Ref{CcIntr}, Ptr{CcView}, Cint, Ptr{Cdouble}, Ptr{Int64}, Ptr{Cfloat}, Ptr{Cfloat},
                 Cint, Cint, Csize_t, Csize_t, Cint, Cfloat, Cuint),
                context().handle, Ref(d.intr), d.views, nv, ratios, axs_mins, imgs, out,
                sz1, sz2, sz1, sz1 * sz2, nf ÷ nv, fill, fast ? 1 : 0))
    out
end

# RGB{N0f8} frames -- what the reference's plot warps (RGB.(load(file))): reinterpret(UInt8, imgs) has
# size (3, sz1, sz2, nframes) = u8c3 layout
function warp_views(d::DeviceCalibration, imgs::Array{UInt8,4}, ratios::Vector{Float64},
                    axss::Vector{<:NTuple{2,<:AbstractUnitRange}}; fill::NTuple{3,UInt8} = (0x00, 0x00, 0x00),
                    fast::Bool = false)
    @assert size(imgs, 1) == 3
    _, sz1, sz2, nf = size(imgs)
    nv = length(d.views)
    @assert nv > 0 && nf % nv == 0 && nv == length(ratios) == length(axss)
    out = similar(imgs)
    axs_mins = Int64[first(a[j]) for a in axss for j in 1:2]
    check(ccall((:cc_rectify_views_u8c3_host, libcamcal), Cint,
                (Ptr{Cvoid}, Ref{CcIntr}, Ptr{CcView}, Cint, Ptr{Cdouble}, Ptr{Int64}, Ptr{UInt8}, Ptr{UInt8},
                 Cint, Cint, Csize_t, Csize_t, Cint, Ptr{UInt8}, Cuint),
                context().handle, Ref(d.intr), d.views, nv, ratios, axs_mins, imgs, out,
                sz1, sz2, sz1, sz1 * sz2, nf ÷ nv, UInt8[fill...], fast ? 1 : 0))
    out
end

# ---- image ingest on the device: RGB.(FileIO.load(file)) for JPEG files, src/plot_calibration.jl:37 --
# The compressed bytes go to the GPU (nvJPEG + a transposition kernel inside the library); the result is a
# DEVICE pointer to (3, sz1, sz2, n) bytes -- the u8c3 layout cc_rectify_u8c3[_views] take -- so a plot loop
# over JPEG files never holds decoded pixels on the host.  `dst` comes from the caller's device allocator
# (CUDA.jl's CuArray{UInt8,4}(undef, 3, sz1, sz2, n) works: pass pointer(dst)).
function jpeg_info(bytes::Vector{UInt8})
    sz1 = Ref{Cint}(0); sz2 = Ref{Cint}(0); ch = Ref{Cint}(0)
    check(ccall((:cc_jpeg_info, libcamcal), Cint, (Ptr{UInt8}, Csize_t, Ref{Cint}, Ref{Cint}, Ref{Cint}),
                bytes, length(bytes), sz1, sz2, ch))
    (Int(sz1[]), Int(sz2[]), Int(ch[]))
end
function load_jpegs!(dst::Ptr{UInt8}, files::Vector{String}; stream::Ptr{Cvoid} = C_NULL)
    blobs = [read(f) for f in files]
    sz1, sz2, _ = jpeg_info(blobs[1])
    GC.@preserve blobs begin
        ptrs = [pointer(b) for b in blobs]
        lens = Csize_t[length(b) for b in blobs]
        check(ccall((:cc_jpeg_decode_u8c3, libcamcal), Cint,
                    (Ptr{Cvoid}, Ptr{Ptr{UInt8}}, Ptr{Csize_t}, Cint, Ptr{UInt8}, Cint, Cint, Csize_t, Csize_t, Ptr{Cvoid}),
                    context().handle, ptrs, lens, length(blobs), dst, sz1, sz2, sz1, sz1 * sz2, stream))
        check(ccall((:cc_ctx_synchronize, libcamcal), Cint, (Ptr{Cvoid},), context().handle))   # blobs may be freed after this
    end
    (sz1, sz2, length(blobs))
end

# ---- multi-GPU: one Julia process per GPU (Distributed / MPI), NCCL inside the library ------------
# rank 0:  id = comm_unique_id();  ship the 128 bytes to the other ranks (MPI.Bcast!, a file, ...)
# all:     comm_init_rank(nranks, rank, id)
# then cc_reproj_jtj_f64 + allreduce_shared!, or the whole fit with lm_fit_device!, run over the ranks.
function comm_unique_id()
    id = Vector{UInt8}(undef, 128)
    check(ccall((:cc_comm_unique_id, libcamcal), Cint, (Ptr{UInt8},), id))
    id
end
comm_init_rank(nranks::Integer, rank::Integer, id::Vector{UInt8}) =
    check(ccall((:cc_comm_init_rank, libcamcal), Cint, (Ptr{Cvoid}, Cint, Cint, Ptr{UInt8}), context().handle, nranks, rank, id))
"in-place sum over the ranks of `count` doubles at DEVICE pointer `buf`"
allreduce_shared!(buf::Ptr{Cdouble}, count::Integer; stream::Ptr{Cvoid} = C_NULL) =
    check(ccall((:cc_allreduce_shared, libcamcal), Cint, (Ptr{Cvoid}, Ptr{Cdouble}, Csize_t, Ptr{Cvoid}),
                context().handle, buf, count, stream))

# One Julia session driving several GPUs: one context per device, joined in one communicator.
struct ContextGroup
    handles::Vector{Ptr{Cvoid}}
end
function ContextGroup(devs::Vector{<:Integer})
    h = Vector{Ptr{Cvoid}}(undef, length(devs))
    check(ccall((:cc_ctx_create_group, libcamcal), Cint, (Cint, Ptr{Cint}, Ptr{Ptr{Cvoid}}), length(devs), Cint.(devs), h))
    g = ContextGroup(h)
    finalizer(x -> ccall((:cc_ctx_destroy_group, libcamcal), Cint, (Cint, Ptr{Ptr{Cvoid}}), length(x), x), g.handles)   # x is the handle vector
    g
end
"in-place sum over the group of `count` doubles at the device pointers `bufs[i]` (one per context)"
allreduce_shared!(g::ContextGroup, bufs::Vector{Ptr{Cdouble}}, count::Integer) =
    check(ccall((:cc_allreduce_shared_group, libcamcal), Cint, (Ptr{Ptr{Cvoid}}, Cint, Ptr{Ptr{Cdouble}}, Csize_t, Ptr{Ptr{Cvoid}}),
                g.handles, length(g.handles), bufs, count, C_NULL))

# ---- residual + normal-equation blocks (what calibrateCamera reduces, src/detect_fit.jl:47) ---
function reproj_jtj(c::Calibration, aspect::Float64, objpoints::Matrix{Float64},   # 3 x ncorners
                    imgpoints::Array{Float64,3})                                    # 2 x ncorners x nviews
    nc, nv = size(imgpoints, 2), size(imgpoints, 3)
    views = [CcView(c, i) for i in 1:nv]
    per_view = Matrix{Float64}(undef, 66, nv)
    shared = Vector{Float64}(undef, 21)
    check(ccall((:cc_reproj_jtj_f64_host, libcamcal), Cint,
                (Ptr{Cvoid}, Ref{CcIntr}, Cdouble, Ptr{CcView}, Cint, Ptr{Cdouble}, Ptr{Cdouble}, Cint,
                 Ptr{Cdouble}, Ptr{Cdouble}),
                context().handle, Ref(CcIntr(c)), aspect, views, nv, objpoints, imgpoints, nc,
                per_view, shared))
    per_view, shared
end

# ---- the fit itself: replaces the OpenCV.calibrateCamera call of src/detect_fit.jl:47 --------
# Starting values as calibrateCamera derives them (principal point at the image centre, focal
# length from the homographies: OpenCV.initCameraMatrix2D; per-view pose: OpenCV.solvePnP), then ONE
# ccall runs the whole Levenberg-Marquardt loop on the device (same flags :40, same CRITERIA).
# `k`, `Rs`, `ts`, `frow`, ... come back in the NamedTuple fit_model returns today (:60).
function lm_fit!(intr::Base.RefValue{CcIntr}, views::Vector{CcView}, aspect::Float64, with_distortion::Bool,
                 objpoints::Matrix{Float64},           # 3 x ncorners, board units
                 imgpoints::Array{Float64,3};          # 2 x ncorners x nviews, (row, col)
                 max_iter::Int = 30, eps::Float64 = 1e-3)
    nc, nv = size(imgpoints, 2), size(imgpoints, 3)
    rms, its = Ref{Cdouble}(0), Ref{Cint}(0)
    check(ccall((:cc_lm_fit_f64_host, libcamcal), Cint,
                (Ptr{Cvoid}, Ref{CcIntr}, Cdouble, Cuint, Ptr{CcView}, Cint, Ptr{Cdouble}, Ptr{Cdouble}, Cint,
                 Cint, Cdouble, Ref{Cdouble}, Ref{Cint}),
                context().handle, intr, aspect, with_distortion ? 0x0f : 0x07, views, nv, objpoints, imgpoints,
                nc, max_iter, eps, rms, its))
    (; k = intr[].k, Rs = [collect(v.rvec) for v in views], ts = [collect(v.tvec) for v in views],
       frow = intr[].frow, fcol = intr[].fcol, crow = intr[].crow, ccol = intr[].ccol, rms = rms[], iterations = its[])
end

# The same fit on DEVICE arrays (e.g. CUDA.jl CuArrays passed as pointers), over this rank's shard of
# the views when the context has a communicator: cc_lm_initial_guess_f64 + cc_lm_fit_f64.  The loop
# state lives on the device; an iteration costs two NCCL all-reduces and no host synchronisation.
function lm_fit_device!(intr::Base.RefValue{CcIntr}, views::Ptr{CcView}, nviews::Integer, obj::Ptr{Cdouble},
                        img::Ptr{Cdouble}, ncorners::Integer, sz::NTuple{2,Int}, aspect::Float64,
                        with_distortion::Bool; max_iter::Int = 30, eps::Float64 = 1e-3, init::Bool = true,
                        stream::Ptr{Cvoid} = C_NULL)
    if init
        check(ccall((:cc_lm_initial_guess_f64, libcamcal), Cint,
                    (Ptr{Cvoid}, Ptr{Cdouble}, Ptr{Cdouble}, Cint, Cint, Cint, Cint, Cdouble, Ref{CcIntr}, Ptr{CcView}, Ptr{Cvoid}),
                    context().handle, obj, img, nviews, ncorners, sz[1], sz[2], aspect, intr, views, stream))
    end
    rms, its = Ref{Cdouble}(0), Ref{Cint}(0)
    check(ccall((:cc_lm_fit_f64, libcamcal), Cint,
                (Ptr{Cvoid}, Ref{CcIntr}, Cdouble, Cuint, Ptr{CcView}, Cint, Ptr{Cdouble}, Ptr{Cdouble}, Cint, Cint,
                 Cdouble, Ref{Cdouble}, Ref{Cint}, Ptr{Cvoid}),
                context().handle, intr, aspect, with_distortion ? 0x0f : 0x07, views, nviews, obj, img, ncorners,
                max_iter, eps, rms, its, stream))
    (; rms = rms[], iterations = its[])
end

end # module
