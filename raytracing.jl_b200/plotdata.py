"""Plot-friendly views of the results: the arrays the reference's Plots.jl recipes assemble (src/plot_recipes.jl), built from the
SoA columns in one vectorised step instead of a loop over boxed Segment objects (the recipe for ``Vector{Track}`` grows three
matrices with ``hcat`` once per segment, :50-74), plus flat NaN-separated polylines for plotting libraries that take one long
path (SURVEY 8f-4), and a per-cell field sampled on a pixel raster for a heatmap (the recipe for ``Mesh`` draws one polygon per
cell, which does not scale to a million cells).  Presentation only: nothing here touches the device except ``cell_raster``, which
locates its pixels with one ``TrackGenerator.find_elements`` call."""
from __future__ import annotations

import numpy as np


def track_lines(tg):
    """``plot(t::TrackGenerator)`` (src/plot_recipes.jl:3-24): x and y of shape (2, n_tracks) -- entry and exit point of every track
    of this shard."""
    t = tg.track_data
    return np.stack([t["p"][:, 0], t["q"][:, 0]]), np.stack([t["p"][:, 1], t["q"][:, 1]])


def segment_lines(source, uid=None):
    """``plot(segments::Vector{Segment})`` / ``plot(tracks::Vector{Track})`` (src/plot_recipes.jl:26-74): x, y, z of shape
    (2, n_segments) with z = the element of the segment (``line_z``).  ``source`` is a TrackGenerator (every resident segment, or
    the tracks ``uid`` = one uid / a list of uids) or the dict ``track.segments.arrays()``."""
    if isinstance(source, dict):
        cols = source
    elif uid is None:
        s = source.segments
        cols = {k: s[k] for k in ("px", "py", "qx", "qy", "element")}
    else:
        uids = [uid] if np.isscalar(uid) else list(uid)
        parts = [source.tracks_by_uid[int(u)].segments.arrays() for u in uids]
        cols = {k: np.concatenate([p[k] for p in parts]) for k in ("px", "py", "qx", "qy", "element")}
    z = cols["element"].astype(np.float64)
    return np.stack([cols["px"], cols["qx"]]), np.stack([cols["py"], cols["qy"]]), np.stack([z, z])


def mesh_lines(mesh):
    """``plot(mesh::Mesh)`` (src/plot_recipes.jl:76-107): x, y of shape (nn + 1, n_cells), every cell's node cycle closed with its
    first node; like the reference, it refuses meshes whose cells do not all have the same number of nodes."""
    ptrs, data = mesh.cell_nodes
    sizes = np.diff(ptrs.astype(np.int64))
    if not np.all(sizes == sizes[0]):
        raise ValueError("error")  # src/plot_recipes.jl:85
    nn = int(sizes[0])
    ids = data.astype(np.int64).reshape(-1, nn) - 1
    ids = np.concatenate([ids, ids[:, :1]], axis=1)
    xy = mesh.model.node_coordinates
    return xy[ids, 0].T.copy(), xy[ids, 1].T.copy()


def flat_polyline(x, y, z=None):
    """(k, n) line matrices -> flat arrays in which consecutive lines are separated by a NaN: one path for the whole plot."""
    k, n = x.shape
    out = []
    for a in (x, y) + ((z,) if z is not None else ()):
        f = np.full((k + 1, n), np.nan)
        f[:k] = a
        out.append(f.T.reshape(-1)[:-1] if n else f.T.reshape(-1))
    return tuple(out)


def flat_mesh_edges(mesh):
    """NaN-separated closed polygons of every cell, also for meshes that mix triangles and quadrilaterals."""
    ptrs, data = mesh.cell_nodes
    p = ptrs.astype(np.int64) - 1
    ids = data.astype(np.int64) - 1
    sizes = np.diff(p)
    n_cells = sizes.size
    total = int(sizes.sum()) + 2 * n_cells  # nodes + closing node + NaN per cell
    starts = p[:-1] + 2 * np.arange(n_cells)
    x = np.full(total, np.nan)
    y = np.full(total, np.nan)
    xy = mesh.model.node_coordinates
    pos = np.arange(ids.size) + 2 * np.repeat(np.arange(n_cells), sizes)
    x[pos], y[pos] = xy[ids, 0], xy[ids, 1]
    close = starts + sizes
    x[close], y[close] = xy[ids[p[:-1]], 0], xy[ids[p[:-1]], 1]
    return x[:-1], y[:-1]


def cell_raster(tg, nx, ny, values=None):
    """A per-cell field as an ``ny`` x ``nx`` heatmap over the bounding box: every pixel centre is located with find_element
    (src/mesh.jl:103-146, k = 2) in one ``tg.find_elements`` call.  Returns matrices (x, y, z) of shape (ny, nx): pixel centres
    (row j = the j-th row from the bottom) and z = ``values[e - 1]`` of the pixel's cell e, or e itself when ``values`` is None;
    NaN where find_element returns -1."""
    lo, hi = np.asarray(tg.mesh.bb_min, np.float64), np.asarray(tg.mesh.bb_max, np.float64)
    xs = lo[0] + (np.arange(nx) + 0.5) * ((hi[0] - lo[0]) / nx)
    ys = lo[1] + (np.arange(ny) + 0.5) * ((hi[1] - lo[1]) / ny)
    x, y = np.meshgrid(xs, ys, indexing="xy")
    ids, _ = tg.find_elements(np.stack([x.reshape(-1), y.reshape(-1)], axis=1))
    found = ids > 0
    z = np.full(ids.shape, np.nan)
    z[found] = ids[found] if values is None else np.asarray(values, np.float64)[ids[found] - 1]
    return x, y, z.reshape(ny, nx)
