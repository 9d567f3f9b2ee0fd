"""Host-side mesh model: the flattening source for the device arrays.

Mirrors what the reference reads from a Gridap ``UnstructuredDiscreteModel`` in ``Mesh(model)``
(reference ``src/mesh.jl:24-31``): node coordinates, the cell->nodes table and the vertex->cells
table, both as 1-based CSR tables exactly like Gridap's ``Table{Int32}`` (``.data`` / ``.ptrs``), and
the bounding box (``src/mesh.jl:53-69``).  Readers for the two fixture formats the reference ships
(``demo/pincell.json`` Gridap JSON v0.15, ``demo/pincell.msh`` MSH 4.1 ASCII) are included.
"""
from __future__ import annotations

import json
from dataclasses import dataclass, field

import numpy as np


@dataclass
class UnstructuredDiscreteModel:
    """Mesh in Gridap's layout: ``cell_ptrs``/``cell_data`` are the 1-based CSR ``Table`` of cell -> nodes.  Triangles (what the
    reference walks, src/mesh.jl:149-150) and, as SURVEY 8(f)-4 asks, 4-node quadrilaterals whose stored nodes form a CYCLE
    (consecutive nodes are edges: the assumption of ``intersections``, src/intersection.jl:46-51)."""

    node_coordinates: np.ndarray  # (n_nodes, 2) float64, contiguous x,y pairs
    cell_ptrs: np.ndarray  # (n_cells + 1,) int32, 1-based
    cell_data: np.ndarray  # int32, 1-based node ids, 3 or 4 per cell
    labels: dict = field(default_factory=dict)

    def __post_init__(self):
        self.node_coordinates = np.ascontiguousarray(self.node_coordinates, dtype=np.float64).reshape(-1, 2)
        self.cell_ptrs = np.ascontiguousarray(self.cell_ptrs, dtype=np.int32)
        self.cell_data = np.ascontiguousarray(self.cell_data, dtype=np.int32)

    @property
    def num_nodes(self) -> int:
        return self.node_coordinates.shape[0]

    @property
    def num_cells(self) -> int:
        return self.cell_ptrs.shape[0] - 1

    @classmethod
    def from_triangles(cls, xy: np.ndarray, tri0: np.ndarray, sort_nodes: bool = True, **kw):
        """Build from 0-based (n_cells, 3) triangles. Gridap models loaded with ``orientation=true``
        store ascending node ids per cell, which ``sort_nodes`` reproduces."""
        tri = np.asarray(tri0, dtype=np.int64)
        if sort_nodes:
            tri = np.sort(tri, axis=1)
        n = tri.shape[0]
        ptrs = (np.arange(n + 1, dtype=np.int64) * 3 + 1).astype(np.int32)
        return cls(np.asarray(xy, dtype=np.float64), ptrs, (tri.reshape(-1) + 1).astype(np.int32), **kw)

    @classmethod
    def from_cells(cls, xy: np.ndarray, cells0, **kw):
        """Build from a list of 0-based node tuples of length 3 or 4, node order kept as given (quadrilaterals: a cycle)."""
        counts = np.fromiter((len(c) for c in cells0), dtype=np.int64, count=len(cells0))
        ptrs = np.concatenate([[1], 1 + np.cumsum(counts)]).astype(np.int32)
        data = (np.fromiter((n for c in cells0 for n in c), dtype=np.int64, count=int(counts.sum())) + 1).astype(np.int32)
        return cls(np.asarray(xy, dtype=np.float64), ptrs, data, **kw)

    @property
    def cell_sizes(self) -> np.ndarray:
        return np.diff(self.cell_ptrs.astype(np.int64))

    @property
    def has_quads(self) -> bool:
        return bool(np.any(self.cell_sizes == 4))

    def cell_regions(self, names) -> np.ndarray:
        """The region (material) of every cell as int32 values in [1, len(names)]: the 1-based position in ``names`` of the first
        name whose tag contains the cell's entity (``labels``: Gridap's face labeling ``names`` / ``tags`` / ``entities_2``, or
        the physical groups of a .msh file).  Overlapping tags go to the name listed first.  An unknown name, or a cell in none of
        the named tags, raises ValueError.  What ``TrackGenerator.set_regions`` takes."""
        lab = self.labels or {}
        known, tags, ent = list(lab.get("names") or []), lab.get("tags"), lab.get("entities_2")
        if ent is None or tags is None:
            raise ValueError("the model carries no cell labeling (names / tags / entities_2)")
        ent = np.asarray(ent, dtype=np.int64).reshape(-1)
        if ent.shape[0] != self.num_cells:
            raise ValueError(f"the labeling has {ent.shape[0]} cell entities for {self.num_cells} cells")
        region = np.zeros(self.num_cells, dtype=np.int32)
        for r, name in enumerate(names, start=1):
            if name not in known:
                raise ValueError(f"unknown label {name!r}: the model has {known}")
            hit = (region == 0) & np.isin(ent, np.asarray(tags[known.index(name)], dtype=np.int64))
            region[hit] = r
        missing = np.flatnonzero(region == 0)
        if missing.size:
            raise ValueError(f"{missing.size} cells are in none of the tags {list(names)}; the first is cell {missing[0] + 1} "
                             f"(entity {ent[missing[0]]})")
        return region

    def triangles0(self) -> np.ndarray:
        """0-based (n_cells, 3) view of the cell table (triangles only)."""
        if self.has_quads:
            raise ValueError("triangles0: the mesh holds quadrilaterals")
        return self.cell_data.reshape(-1, 3).astype(np.int64) - 1


def DiscreteModelFromFile(path: str) -> UnstructuredDiscreteModel:
    """Reader for Gridap's ``DiscreteModel`` JSON (the format of ``demo/pincell.json``,
    used by reference ``test/runtests.jl:5-6``)."""
    with open(path) as fh:
        d = json.load(fh)
    g = d["grid"]
    xy = np.asarray(g["node_coordinates"], dtype=np.float64).reshape(-1, int(g.get("Dp", 2)))[:, :2]
    ptrs = np.asarray(g["cell_node_ids"]["ptrs"], dtype=np.int32)
    data = np.asarray(g["cell_node_ids"]["data"], dtype=np.int32)
    if not np.all(np.isin(np.diff(ptrs), (3, 4))):
        raise ValueError("only linear triangles and quadrilaterals are supported")
    lab = d.get("labeling", {})
    labels = {"names": lab.get("names"), "tags": lab.get("tags"), "entities_2": lab.get("entities_2")}
    return UnstructuredDiscreteModel(xy, ptrs, data, labels)


def GmshDiscreteModel(path: str, renumber: bool = True) -> UnstructuredDiscreteModel:
    """Reader for MSH 4.1 ASCII (``demo/pincell.msh``; reference README quick start). Keeps the 3-node
    triangles (element type 2), nodes in tag order, node ids ascending within each cell like the
    Gridap model the reference builds from the same file.  The physical groups become ``labels`` as Gridap names them: one
    name per ``$PhysicalNames`` entry, its tag the surface entities of ``$Entities`` that carry the group, and ``entities_2`` the
    surface entity of every triangle (cells stay in file order, whatever the node renumbering): see ``cell_regions``."""
    with open(path) as fh:
        lines = fh.read().split("\n")
    idx = {ln.strip(): i for i, ln in enumerate(lines) if ln.startswith("$")}
    ver = lines[idx["$MeshFormat"] + 1].split()
    if not ver[0].startswith("4"):
        raise ValueError("only MSH 4.x ASCII is supported")
    # $Nodes: numEntityBlocks numNodes minTag maxTag ; per block: dim tag parametric n ; n tags ; n coords
    i = idx["$Nodes"] + 1
    nblocks, nnodes = (int(v) for v in lines[i].split()[:2])
    i += 1
    tags = np.empty(nnodes, dtype=np.int64)
    xyz = np.empty((nnodes, 3), dtype=np.float64)
    k = 0
    for _ in range(nblocks):
        _, _, _, nb = (int(v) for v in lines[i].split())
        i += 1
        for j in range(nb):
            tags[k + j] = int(lines[i + j])
        i += nb
        for j in range(nb):
            xyz[k + j] = [float(v) for v in lines[i + j].split()[:3]]
        i += nb
        k += nb
    order = np.argsort(tags, kind="stable")
    tags, xyz = tags[order], xyz[order]
    i = idx["$Elements"] + 1
    nblocks = int(lines[i].split()[0])
    i += 1
    tris, tri_ent = [], []
    for _ in range(nblocks):
        _, etag, etype, nb = (int(v) for v in lines[i].split())
        i += 1
        if etype == 2:
            for j in range(nb):
                tris.append([int(v) for v in lines[i + j].split()[1:4]])
            tri_ent += [etag] * nb
        i += nb
    labels = _msh_labels(lines, idx)
    if labels:
        labels["entities_2"] = tri_ent
    tri_tags = np.asarray(tris, dtype=np.int64)
    tri0 = np.searchsorted(tags, tri_tags)
    if renumber:  # keep only nodes referenced by triangles, in tag order
        used = np.unique(tri0)
        remap = -np.ones(nnodes, dtype=np.int64)
        remap[used] = np.arange(used.size)
        tri0 = remap[tri0]
        xyz = xyz[used]
    return UnstructuredDiscreteModel.from_triangles(xyz[:, :2], tri0, sort_nodes=True, labels=labels)


def _msh_labels(lines, idx) -> dict:
    """{names, tags} of the physical groups of an MSH 4.1 file: ``$PhysicalNames`` (dim tag "name") and, from ``$Entities``, the
    surfaces that carry each group (a group of points or curves tags no surface).  Empty without ``$PhysicalNames``."""
    if "$PhysicalNames" not in idx or "$Entities" not in idx:
        return {}
    i = idx["$PhysicalNames"] + 1
    groups = []  # (dim, physical tag, name) in file order
    for ln in lines[i + 1:i + 1 + int(lines[i].split()[0])]:
        dim, tag, name = ln.split(maxsplit=2)
        groups.append((int(dim), int(tag), name.strip().strip('"')))
    i = idx["$Entities"] + 1
    n_pts, n_crv, n_srf = (int(v) for v in lines[i].split()[:3])
    surfaces = {}  # physical tag -> surface entity tags
    # points: tag x y z nPhys phys... ; curves and surfaces: tag minX minY minZ maxX maxY maxZ nPhys phys... nBound bound...
    for ln in lines[i + 1 + n_pts + n_crv:i + 1 + n_pts + n_crv + n_srf]:
        v = ln.split()
        for ph in v[8:8 + int(v[7])]:
            surfaces.setdefault(int(ph), []).append(int(v[0]))
    names, tags = [], []
    for dim, tag, name in groups:
        if name in names:  # (a name given to groups of several dimensions: one label)
            tags[names.index(name)] += surfaces.get(tag, []) if dim == 2 else []
            continue
        names.append(name)
        tags.append(list(surfaces.get(tag, [])) if dim == 2 else [])
    return {"names": names, "tags": tags}


def vertex_to_cells(n_nodes: int, cell_ptrs: np.ndarray, cell_data: np.ndarray):
    """vertex->cells CSR (1-based), cells around each node in ascending cell id -- the table the
    reference gets from ``get_faces(get_grid_topology(model), 0, 2)`` (``src/mesh.jl:27``)."""
    n_cells = cell_ptrs.shape[0] - 1
    counts = np.diff(cell_ptrs.astype(np.int64))
    cell_of_entry = np.repeat(np.arange(1, n_cells + 1, dtype=np.int32), counts)
    order = np.argsort(cell_data, kind="stable")
    data = cell_of_entry[order]
    deg = np.bincount(cell_data.astype(np.int64) - 1, minlength=n_nodes)
    ptrs = np.empty(n_nodes + 1, dtype=np.int64)
    ptrs[0] = 1
    np.cumsum(deg, out=ptrs[1:])
    ptrs[1:] += 1
    return ptrs.astype(np.int32), np.ascontiguousarray(data, dtype=np.int32)


class Mesh:
    """Counterpart of the reference ``Mesh`` struct (``src/mesh.jl:10-31``): ``model``, ``node_cells``,
    ``cell_nodes`` (both as (ptrs, data) 1-based CSR pairs), ``bb_min``, ``bb_max``.  The KD-tree of the
    reference is replaced by a uniform node grid built on the device at upload time."""

    def __init__(self, model: UnstructuredDiscreteModel, device_ingest: bool = False):
        """``device_ingest=True`` leaves the vertex->cells table and the bounding box to the device (``rt_mesh_upload`` with
        NULL tables): nothing of size O(mesh) is computed on the host.  ``bb_min``/``bb_max`` are then filled in by the first
        ``TrackGenerator`` built on this mesh, and ``node_cells`` is computed on first use (the oracle needs it)."""
        self.model = model
        self.cell_nodes = (model.cell_ptrs, model.cell_data)
        self.device_ingest = bool(device_ingest)
        self._node_cells = None
        self.bb_min = self.bb_max = None
        if not device_ingest:
            self._node_cells = vertex_to_cells(model.num_nodes, model.cell_ptrs, model.cell_data)
            xy = model.node_coordinates
            # src/mesh.jl:53-69: min / max over all node coordinates
            self.bb_min = np.array([xy[:, 0].min(), xy[:, 1].min()], dtype=np.float64)
            self.bb_max = np.array([xy[:, 0].max(), xy[:, 1].max()], dtype=np.float64)

    @property
    def node_cells(self):
        if self._node_cells is None:
            self._node_cells = vertex_to_cells(self.model.num_nodes, self.model.cell_ptrs, self.model.cell_data)
        return self._node_cells

    @property
    def width(self) -> float:  # src/mesh.jl:76
        return float(self.bb_max[0] - self.bb_min[0])

    @property
    def height(self) -> float:  # src/mesh.jl:83
        return float(self.bb_max[1] - self.bb_min[1])

    @property
    def num_cells(self) -> int:
        return self.model.num_cells

    @property
    def num_nodes(self) -> int:
        return self.model.num_nodes
