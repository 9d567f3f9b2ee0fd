# RayTracingB200.jl -- the `ccall` glue a RayTracing.jl maintainer adds to route `trace!` / `segmentize!`
# through librt_b200.so (C ABI: include/rt_b200.h).  `include` it at the end of src/RayTracing.jl (after
# "trackgenerator.jl"); see INTEGRATION.md for the 6-line dispatch patch.  It fills the reference's OWN structs
# (Track{BCFwd,BCBwd,DFwd,DBwd}, Segment, TrackGenerator fields), so accessors, tests and plot recipes keep working.
#
# NOT EXERCISED IN THIS REPOSITORY'S CI: Julia is absent from the build image.  The same ABI calls, in the same
# order and with the same arguments, are exercised through ctypes by raytracing.jl_b200/api.py (tests/ -m gpu).

const LIBRT_B200 = get(ENV, "RT_B200_LIB", "librt_b200.so")

# device context per TrackGenerator, keyed by its (mutable) tracks_by_uid vector
const _B200_CTX = IdDict{Any,Ptr{Cvoid}}()

function _b200_check(ctx::Ptr{Cvoid}, rc::Cint)
    rc == 0 && return nothing
    msg = unsafe_string(ccall((:rt_last_error, LIBRT_B200), Cstring, (Ptr{Cvoid},), ctx))
    rc == -4 && throw(DomainError("could not found track exit point."))     # trackgenerator.jl:219
    error(msg)                                                               # carries the reference's own message
end

function _b200_context(t::TrackGenerator)
    haskey(_B200_CTX, t.tracks_by_uid) && return _B200_CTX[t.tracks_by_uid]
    ref = Ref{Ptr{Cvoid}}(C_NULL)
    dev = parse(Cint, get(ENV, "RT_B200_DEVICE", "0"))
    rc = ccall((:rt_create, LIBRT_B200), Cint, (Ptr{Ptr{Cvoid}}, Cint), ref, dev)
    rc == 0 || error("rt_create failed: no usable CUDA device (there is no CPU fallback)")
    ctx = ref[]
    # ---- flatten the Gridap model: Mesh(model) already holds the two Tables and the bounding box (mesh.jl:24-31)
    mesh = t.mesh
    coords = get_node_coordinates(get_grid(mesh.model))          # Vector{VectorValue{2,Float64}} = contiguous x,y pairs
    xy = reinterpret(Float64, coords)
    cn, nc = mesh.cell_nodes, mesh.node_cells                    # Gridap Table{Int32}: .data / .ptrs, 1-based
    bbmin = Float64[mesh.bb_min[1], mesh.bb_min[2]]
    bbmax = Float64[mesh.bb_max[1], mesh.bb_max[2]]
    rc = ccall((:rt_mesh_upload, LIBRT_B200), Cint,
        (Ptr{Cvoid}, Int32, Ptr{Float64}, Int32, Ptr{Int32}, Ptr{Int32}, Ptr{Int32}, Ptr{Int32}, Ptr{Float64}, Ptr{Float64}),
        ctx, Int32(length(coords)), xy, Int32(length(cn)), Vector{Int32}(cn.ptrs), Vector{Int32}(cn.data),
        Vector{Int32}(nc.ptrs), Vector{Int32}(nc.data), bbmin, bbmax)
    _b200_check(ctx, rc)
    _B200_CTX[t.tracks_by_uid] = ctx
    finalizer(t.tracks_by_uid) do v
        c = pop!(_B200_CTX, v, C_NULL)
        c == C_NULL || ccall((:rt_destroy, LIBRT_B200), Cvoid, (Ptr{Cvoid},), c)
    end
    return ctx
end

_bc_code(bc::BoundaryType) = Int32(Int(bc))   # Vacuum=0, Reflective=1, Periodic=2 (boundary.jl:12-16)

"""
    b200_trace!(t::TrackGenerator)

Device version of `trace!` (trackgenerator.jl:134-280).  The per-angle effective quadrature (the only libm
work of the path) is computed here exactly like lines :150-166, so ϕs/δs/ωₐ are Julia's own values.
"""
function b200_trace!(t::TrackGenerator{T}) where {T}
    @unpack mesh, bcs, azimuthal_quadrature, n_tracks_x, n_tracks_y, n_tracks, tracks, tracks_by_uid = t
    @unpack δs, ϕs = azimuthal_quadrature
    n2 = nazim2(azimuthal_quadrature)
    δx = Vector{T}(undef, n2); δy = Vector{T}(undef, n2)
    Δx, Δy = width(mesh), height(mesh)
    for i in right_dir(azimuthal_quadrature)
        ϕ = ϕs[i] = atan((Δy * n_tracks_x[i]) / (Δx * n_tracks_y[i]))
        δx[i] = Δx / n_tracks_x[i]; δy[i] = Δy / n_tracks_y[i]; δs[i] = δx[i] * sin(ϕ)
        j = suplementary_idx(azimuthal_quadrature, i)
        ϕs[j] = π - ϕ; δx[j] = δx[i]; δy[j] = δy[i]; δs[j] = δs[i]
    end
    init_weights!(azimuthal_quadrature)

    ctx = _b200_context(t)
    codes = Int32[_bc_code(bcs.top), _bc_code(bcs.bottom), _bc_code(bcs.right), _bc_code(bcs.left)]
    n = t.n_total_tracks
    rc = ccall((:rt_trace, LIBRT_B200), Cint,
        (Ptr{Cvoid}, Int32, Ptr{Int64}, Ptr{Int64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64},
         Ptr{Float64}, Ptr{Float64}, Ptr{Int32}, Int64, Int64),
        ctx, Int32(n2), Vector{Int64}(n_tracks_x), Vector{Int64}(n_tracks_y), ϕs, sin.(ϕs), cos.(ϕs), tan.(ϕs),
        δx, δy, codes, 1, n + 1)
    _b200_check(ctx, rc)

    azim = Vector{Int64}(undef, n); tidx = Vector{Int64}(undef, n)
    p = Matrix{Float64}(undef, 2, n); q = Matrix{Float64}(undef, 2, n)
    ϕ = Vector{Float64}(undef, n); ℓ = Vector{Float64}(undef, n); abc = Matrix{Float64}(undef, 3, n)
    bcf = Vector{Int8}(undef, n); bcb = similar(bcf); df = similar(bcf); db = similar(bcf)
    nf = Vector{Int64}(undef, n); nb = Vector{Int64}(undef, n)
    rc = ccall((:rt_tracks_download, LIBRT_B200), Cint,
        (Ptr{Cvoid}, Ptr{Int64}, Ptr{Int64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64},
         Ptr{Int8}, Ptr{Int8}, Ptr{Int8}, Ptr{Int8}, Ptr{Int64}, Ptr{Int64}),
        ctx, azim, tidx, p, q, ϕ, ℓ, abc, bcf, bcb, df, db, nf, nb)
    _b200_check(ctx, rc)
    for uid in 1:n
        track = Track{BoundaryType(bcf[uid]),BoundaryType(bcb[uid]),DirectionType(df[uid]),DirectionType(db[uid])}(
            uid, Int(azim[uid]), Int(tidx[uid]), Point2D(p[1, uid], p[2, uid]), Point2D(q[1, uid], q[2, uid]),
            ϕ[uid], ℓ[uid], SVector(abc[1, uid], abc[2, uid], abc[3, uid]), Vector{Segment{T}}())
        tracks_by_uid[uid] = track
        tracks[azim[uid]][tidx[uid]] = track
    end
    for uid in 1:n                                           # next_tracks (trackgenerator.jl:282-348)
        tracks_by_uid[uid].next_track_fwd = tracks_by_uid[nf[uid]]
        tracks_by_uid[uid].next_track_bwd = tracks_by_uid[nb[uid]]
    end
    return t
end

"""
    B200Segments{T} <: AbstractVector{Segment{T}}

Lazy view of one track's segments over the SoA columns the device produced: a `Segment` (src/segment.jl:23-29) is only built when
it is indexed, so a `segmentize!` of 5e7 segments does not allocate 5e7 `Segment`s with 5e7 empty `τ` vectors up front.  The
columns are the COMPACT download (include/rt_b200.h: rt_segments_download_compact): `q`, `ℓ`, `element` crossed the bus, the entry
point is the exit point of the segment before it (`p[i] = q[i-1]`) except at the positions of the exception list, which the
constructor of the columns has already patched into `px`, `py` lazily per track (see `_b200_track_p`).
"""
struct B200Segments{T} <: AbstractVector{Segment{T}}
    cols::Any          # B200Columns
    lo::Int            # 1-based position of the track's first segment in the columns
    n::Int
end
Base.size(v::B200Segments) = (v.n,)
function Base.getindex(v::B200Segments{T}, i::Int) where {T}
    @boundscheck checkbounds(v, i)
    c = v.cols
    s = v.lo + i - 1
    px, py = _b200_p(c, s)
    return Segment(Point2D(px, py), Point2D(c.qx[s], c.qy[s]), c.len[s], Vector{T}(), c.element[s])
end

"the columns of one `segmentize!`: what crossed the bus plus the (sorted) exception list"
struct B200Columns
    qx::Vector{Float64}
    qy::Vector{Float64}
    len::Vector{Float64}
    element::Vector{Int32}
    exc_index::Vector{Int64}   # sorted, 1-based positions whose p is NOT the preceding q (first segment of a track, ...)
    exc_px::Vector{Float64}
    exc_py::Vector{Float64}
end
function _b200_p(c::B200Columns, s::Int)
    k = searchsortedfirst(c.exc_index, s)
    (k <= length(c.exc_index) && c.exc_index[k] == s) && return c.exc_px[k], c.exc_py[k]
    return c.qx[s-1], c.qy[s-1]
end

const _B200_COLS = IdDict{Any,Tuple{B200Columns,Vector{Int64}}}()   # per TrackGenerator: columns + offsets

"""
    b200_segments(t::TrackGenerator, uid) -> B200Segments

Lazy `Vector{Segment}`-like view of track `uid` after `b200_segmentize!(t; materialize=false)`.
"""
function b200_segments(t::TrackGenerator{T}, uid::Integer) where {T}
    cols, off = _B200_COLS[t.tracks_by_uid]
    return B200Segments{T}(cols, off[uid] + 1, off[uid+1] - off[uid])
end

"""
    b200_segmentize!(t::TrackGenerator; k=5, rtol=√eps, materialize=true)

Device version of `segmentize!` (trackgenerator.jl:357-369): walk (count + record) → scan → evaluation (+ fused `fill_volumes`).
The records come back over the thin wire (28 bytes per segment).  With `materialize=true` every `track.segments` is refilled with
the reference's own `Segment` objects, exactly as `_segmentize_track!` leaves them (one `Segment` + one empty `τ` per segment:
fine for the reference's own problem sizes, seconds for 5e7 segments); with `materialize=false` they stay empty and
`b200_segments(t, uid)` gives a lazy view instead.  For meshes whose segments do not fit host memory use `rt_segments_device` /
the batch callback.
"""
function b200_segmentize!(t::TrackGenerator{T}; k::Int=5, rtol::Real=Base.rtoldefault(T), materialize::Bool=true) where {T}
    @unpack tracks_by_uid, azimuthal_quadrature, volumes = t
    !isassigned(tracks_by_uid, 1) && error("Segmentation is intended after tracing. Please, " *
                                           "call `trace!` first!")
    ctx = _b200_context(t)
    nseg = Ref{Int64}(0); bad = Ref{Int64}(0); st = Ref{Int32}(0)
    rc = ccall((:rt_segmentize, LIBRT_B200), Cint,
        (Ptr{Cvoid}, Float64, Int32, Float64, Int32, Ptr{Float64}, UInt32, Ptr{Cvoid}, Ptr{Cvoid},
         Ptr{Int64}, Ptr{Int64}, Ptr{Int32}),
        ctx, Float64(t.tiny_step), Int32(k), Float64(rtol), Int32(MAX_ITER), azimuthal_quadrature.δs, UInt32(0),
        C_NULL, C_NULL, nseg, bad, st)
    if rc != 0
        # every rank of a communicator enters the all-reduce once per segmentize!, also the one that is about to throw
        # (include/rt_b200.h, rt_volumes): keep the message of rt_segmentize, join, then raise it
        msg = unsafe_string(ccall((:rt_last_error, LIBRT_B200), Cstring, (Ptr{Cvoid},), ctx))
        ccall((:rt_volumes, LIBRT_B200), Cint, (Ptr{Cvoid}, Ptr{Float64}), ctx, C_NULL)
        error(msg)                                            # RT_ERR_TRACK carries the reference's error text + uid
    end
    n = t.n_total_tracks; S = nseg[]
    off = Vector{Int64}(undef, n + 1)
    _b200_check(ctx, ccall((:rt_segment_offsets, LIBRT_B200), Cint, (Ptr{Cvoid}, Ptr{Int64}, Ptr{Int32}), ctx, off, C_NULL))
    qx = Vector{Float64}(undef, S); qy = similar(qx); len = similar(qx); el = Vector{Int32}(undef, S)
    cap = 4n + S ÷ 64 + 1024
    ei = Vector{Int64}(undef, cap); ex = Vector{Float64}(undef, cap); ey = similar(ex); ne = Ref{Int64}(0)
    rc = ccall((:rt_segments_download_compact, LIBRT_B200), Cint,
        (Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Int32}, Int64, Ptr{Int64}, Ptr{Float64}, Ptr{Float64}, Ptr{Int64}),
        ctx, qx, qy, len, el, cap, ei, ex, ey, ne)
    if rc == -10                                              # RT_ERR_NOMEM: more exceptions than room; the call reported how many
        cap = ne[] + 1024; resize!(ei, cap); resize!(ex, cap); resize!(ey, cap)
        rc = ccall((:rt_segments_download_compact, LIBRT_B200), Cint,
            (Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}, Ptr{Float64}, Ptr{Int32}, Int64, Ptr{Int64}, Ptr{Float64}, Ptr{Float64}, Ptr{Int64}),
            ctx, C_NULL, C_NULL, C_NULL, C_NULL, cap, ei, ex, ey, ne)
    end
    _b200_check(ctx, rc)
    resize!(ei, ne[]); resize!(ex, ne[]); resize!(ey, ne[])
    o = sortperm(ei)
    cols = B200Columns(qx, qy, len, el, ei[o] .+ 1, ex[o], ey[o])   # (the ABI's indices are 0-based positions)
    _B200_COLS[tracks_by_uid] = (cols, off)
    for uid in 1:n
        segs = tracks_by_uid[uid].segments
        empty!(segs)
        materialize || continue
        sizehint!(segs, off[uid+1] - off[uid])
        for s in off[uid]+1:off[uid+1]
            px, py = _b200_p(cols, s)
            push!(segs, Segment(Point2D(px, py), Point2D(qx[s], qy[s]), len[s], Vector{T}(), el[s]))
        end
    end
    _b200_check(ctx, ccall((:rt_volumes, LIBRT_B200), Cint, (Ptr{Cvoid}, Ptr{Float64}), ctx, volumes))
    return t
end

# ---- what a transport sweep consumes, kept on the device (include/rt_b200.h: rt_tracks_device, rt_quadrature_device,
# ---- rt_optical_lengths) -------------------------------------------------------------------------------------------

"""
    b200_optical_lengths!(t::TrackGenerator, Σt::Matrix{Float64}) -> Matrix{Float64}

`τ[g, s] = Σt[g, element(s)] * ℓ(s)` for every segment, evaluated on the device (`Σt` is n_groups × n_cells, so its memory is
the element-major n_cells × n_groups array the ABI asks for) and copied into each `segment.τ` (src/segment.jl:27), which the
reference leaves empty.  The device buffer stays resident for an on-GPU sweep.
"""
function b200_optical_lengths!(t::TrackGenerator{T}, Σt::Matrix{Float64}) where {T}
    ctx = _b200_context(t)
    G = size(Σt, 1)
    S = sum(length(track.segments) for track in t.tracks_by_uid)
    τ = Matrix{Float64}(undef, G, S)                          # layout 0: per-segment vectors, concatenated
    dτ = Ref{Ptr{Float64}}(C_NULL)
    _b200_check(ctx, ccall((:rt_optical_lengths, LIBRT_B200), Cint,
        (Ptr{Cvoid}, Int32, Ptr{Float64}, Int32, Ptr{Ptr{Float64}}, Ptr{Float64}), ctx, Int32(G), Σt, Int32(0), dτ, τ))
    s = 0
    for track in t.tracks_by_uid, segment in track.segments
        s += 1
        resize!(segment.τ, G); copyto!(segment.τ, view(τ, :, s))
    end
    return τ
end

"""
    b200_correct_volumes!(t::TrackGenerator) -> Vector{Float64}

What `fill_volumes` announces but leaves as a TODO (src/trackgenerator.jl:388-397): every `segment.ℓ` of element `e` is scaled by
`element_volume(e) / t.volumes[e]` on the device (include/rt_b200.h: rt_correct_volumes), so that the traced volumes of the
corrected lengths equal the exact cell areas.  Returns the per-element factors; call it after `segmentize!` when
`t.volume_correction` is set.  (`Segment` is immutable: the corrected lengths are read back into fresh `Segment`s.)
"""
function b200_correct_volumes!(t::TrackGenerator{T}) where {T}
    ctx = _b200_context(t)
    factors = Vector{Float64}(undef, num_cells(t.mesh.model))
    _b200_check(ctx, ccall((:rt_correct_volumes, LIBRT_B200), Cint, (Ptr{Cvoid}, Ptr{Float64}, Ptr{Ptr{Float64}}), ctx, factors, C_NULL))
    for track in t.tracks_by_uid, (i, s) in enumerate(track.segments)
        track.segments[i] = Segment{T}(s.p, s.q, s.ℓ * factors[s.element], s.τ, s.element)
    end
    return factors
end

"""
    b200_mesh_upload_device_ingest(ctx, model)

Mesh ingestion at scale: only node coordinates and the cell→node table cross the ABI; the vertex→cells table
(`get_faces(topology, 0, 2)`, src/mesh.jl:27) and the bounding box (src/mesh.jl:53-69, whose `min(xs...)` splat does not
scale) are built on the device.  Returns `(bb_min, bb_max)`.
"""
function b200_mesh_upload_device_ingest(ctx::Ptr{Cvoid}, model)
    grid = get_grid(model)
    coords = get_node_coordinates(grid)
    cn = get_cell_node_ids(grid)
    rc = ccall((:rt_mesh_upload, LIBRT_B200), Cint,
        (Ptr{Cvoid}, Int32, Ptr{Float64}, Int32, Ptr{Int32}, Ptr{Int32}, Ptr{Int32}, Ptr{Int32}, Ptr{Float64}, Ptr{Float64}),
        ctx, Int32(length(coords)), reinterpret(Float64, coords), Int32(length(cn)), Vector{Int32}(cn.ptrs),
        Vector{Int32}(cn.data), C_NULL, C_NULL, C_NULL, C_NULL)
    _b200_check(ctx, rc)
    lo = zeros(2); hi = zeros(2)
    _b200_check(ctx, ccall((:rt_mesh_bbox, LIBRT_B200), Cint, (Ptr{Cvoid}, Ptr{Float64}, Ptr{Float64}), ctx, lo, hi))
    return Point2D(lo[1], lo[2]), Point2D(hi[1], hi[2])
end

# ---- point location outside the walk (include/rt_b200.h: rt_find_elements) ------------------------------------------------

"""
    b200_find_elements(t::TrackGenerator, xs::AbstractVector; k=2) -> Vector{Int32}

`find_element(t.mesh, x, k)` (src/mesh.jl:103-146) for every point `x` of `xs` (anything indexable as `x[1]`, `x[2]`: `Point2D`,
`VectorValue`, a 2-vector) in one device call, instead of one KD-tree query per point: the cell of each point, or -1 like the
reference when no cell passes.  Nearest-node distance ties go to the lowest node id.  Needs only the uploaded mesh (no `trace!`).
"""
function b200_find_elements(t::TrackGenerator, xs::AbstractVector; k::Integer=2)
    ctx = _b200_context(t)
    n = length(xs)
    xy = Vector{Float64}(undef, 2n)
    for (i, x) in enumerate(xs)
        xy[2i-1] = x[1]; xy[2i] = x[2]
    end
    element = Vector{Int32}(undef, n)
    _b200_check(ctx, ccall((:rt_find_elements, LIBRT_B200), Cint,
        (Ptr{Cvoid}, Int64, Ptr{Float64}, Int32, Ptr{Int32}, Ptr{Ptr{Int32}}), ctx, Int64(n), xy, Int32(k), element, C_NULL))
    return element
end

"""
    b200_find_element(t::TrackGenerator, x; k=2) -> Int32

`find_element(t.mesh, x, k)` (src/mesh.jl:103-146) for one point, with the reference's return value.
"""
b200_find_element(t::TrackGenerator, x; k::Integer=2) = b200_find_elements(t, [x]; k=k)[1]
