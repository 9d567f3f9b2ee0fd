"""Host-side mirror of RayTracing.jl's public API for the trace! -> segmentize! path.

    tg = TrackGenerator(model, n_azim, delta, bcs=BoundaryConditions(...))   # src/trackgenerator.jl:80-125
    trace_(tg)                                                                # trace!      (:134-280)
    segmentize_(tg)                                                           # segmentize! (:357-369)
    tg.tracks_by_uid[i].segments                                              # same layout as the reference

Julia's ``!`` suffix becomes a trailing underscore.  Field and accessor names follow the reference
(``phis`` = ϕs, ``deltas`` = δs, ``weights`` = ωₐ, ``ell`` = ℓ, ``tau`` = τ).  All geometry runs in the CUDA
library behind the C ABI (include/rt_b200.h); this module only computes the <=128 per-angle libm values the
ABI asks the caller for, and wraps device results in numpy arrays.  Indices are 1-based like the reference.
"""
from __future__ import annotations

import ctypes as C
import math
from collections.abc import Mapping
from dataclasses import dataclass
from enum import IntEnum

import numpy as np

from . import _lib
from .mesh import Mesh, UnstructuredDiscreteModel

RTOL_DEFAULT = math.sqrt(2.0 ** -52)  # Base.rtoldefault(Float64)
MAX_ITER = 10_000  # src/track.jl:104


class DomainError(ValueError):
    """Julia's DomainError (src/azimuthal_quad.jl:22-25, src/trackgenerator.jl:219)."""


class BoundaryType(IntEnum):  # src/boundary.jl:12-16
    Vacuum = 0
    Reflective = 1
    Periodic = 2


Vacuum, Reflective, Periodic = BoundaryType.Vacuum, BoundaryType.Reflective, BoundaryType.Periodic


class DirectionType(IntEnum):  # src/track.jl:11-14
    Forward = 0
    Backward = 1


Forward, Backward = DirectionType.Forward, DirectionType.Backward


@dataclass(frozen=True)
class BoundaryConditions:  # src/boundary.jl:38-46 (keyword constructor, all Vacuum by default)
    top: BoundaryType = Vacuum
    bottom: BoundaryType = Vacuum
    right: BoundaryType = Vacuum
    left: BoundaryType = Vacuum

    def codes(self) -> np.ndarray:
        return np.array([int(self.top), int(self.bottom), int(self.right), int(self.left)], dtype=np.int32)


class AzimuthalQuadrature:  # src/azimuthal_quad.jl:8-34
    def __init__(self, n_azim: int, delta: float):
        if not n_azim > 0:
            raise DomainError(f"{n_azim}: number of azimuthal angles must be positive.")
        if n_azim % 4 != 0:
            raise DomainError(f"{n_azim}: number of azimuthal angles must be a multiple of 4.")
        if not delta > 0:
            raise DomainError(f"{delta}: azimuthal spacing must be positive.")
        self.n_azim = n_azim
        self.delta = float(delta)
        n2 = n_azim // 2
        self.deltas = np.zeros(n2)
        self.phis = np.zeros(n2)
        self.weights = np.zeros(n2)


def nazim(aq: AzimuthalQuadrature) -> int:
    return aq.n_azim


def nazim2(aq: AzimuthalQuadrature) -> int:
    return aq.n_azim // 2


def nazim4(aq: AzimuthalQuadrature) -> int:
    return aq.n_azim // 4


def init_weights_(aq: AzimuthalQuadrature) -> None:  # src/azimuthal_quad.jl:35-53
    n2, n4 = nazim2(aq), nazim4(aq)
    ph, w = aq.phis, aq.weights
    for i in range(1, n4 + 1):
        if i == 1:
            v = ph[i] - ph[i - 1]
        elif i == n4:
            v = math.pi - ph[i - 1] - ph[i - 2]
        else:
            v = ph[i] - ph[i - 2]
        v /= 4 * math.pi
        w[i - 1] = v
        w[n2 - i] = v


class Segment:  # src/segment.jl:23-29
    __slots__ = ("p", "q", "ell", "tau", "element")

    def __init__(self, p, q, ell, element):
        self.p, self.q, self.ell, self.tau, self.element = p, q, ell, [], element

    def __repr__(self):
        return f"Segment(p={self.p}, q={self.q}, ell={self.ell}, element={self.element})"


LENGTHS_ONLY_MSG = ("the segments were produced with RT_SEG_LENGTHS_ONLY (segmentize_(..., lengths_only=True)), which writes only "
                    "len and element: there are no end points p / q")


class SegmentColumns(Mapping):
    """The SoA columns px, py, qx, qy, len, element of the resident Segment batch.  After a COMPACT download
    (``fetch_segments(compact=True)``, rt_segments_download_compact) only qx, qy, len, element crossed the bus; ``px`` / ``py``
    are rebuilt on first use from p[i] = q[i-1] plus the exception list -- whole columns through ``cols["px"]``, or just the
    range of one track through ``p_range`` (what ``track.segments`` uses).  Both are bit-identical to a full download.
    With ``lengths_only`` (the batch of a ``segmentize_(..., lengths_only=True)``) there are only len and element."""

    KEYS = ("px", "py", "qx", "qy", "len", "element")

    def __init__(self, cols, exceptions=None, lengths_only=False):
        self._cols = dict(cols)
        self.lengths_only = lengths_only
        self._keys = ("len", "element") if lengths_only else self.KEYS
        self._exc = None
        if exceptions is not None:
            idx, ex, ey = exceptions
            o = np.argsort(idx, kind="stable")
            self._exc = (idx[o], ex[o], ey[o])

    @property
    def compact(self):
        return self._exc is not None

    def __getitem__(self, key):
        if self.lengths_only and key in self.KEYS and key not in self._keys:
            raise KeyError(f"{key!r}: {LENGTHS_ONLY_MSG}")
        if key not in self._cols:
            if key == "len" and self._exc is not None:
                # Segment(p, q): norm(p - q) (src/segment.jl:32) with the operations of the device code, in the same order:
                # IEEE subtract, multiply, add and square root, none of them fused -- the same bits
                dx, dy = self["px"] - self._cols["qx"], self["py"] - self._cols["qy"]
                self._cols["len"] = np.sqrt(dx * dx + dy * dy)
            elif key in ("px", "py") and self._exc is not None:
                idx, ex, ey = self._exc
                for name, q, e in (("px", self._cols["qx"], ex), ("py", self._cols["qy"], ey)):
                    p = np.empty_like(q)
                    p[1:] = q[:-1]
                    p[idx] = e
                    self._cols[name] = p
            else:
                raise KeyError(key)
        return self._cols[key]

    def __iter__(self):
        return iter(self._keys)

    def __len__(self):
        return len(self._keys)

    def p_range(self, lo, hi):
        """(px, py) of the segments [lo, hi) of the resident batch without rebuilding the whole columns"""
        if self.lengths_only:
            raise KeyError(LENGTHS_ONLY_MSG)
        if "px" in self._cols:
            return self._cols["px"][lo:hi], self._cols["py"][lo:hi]
        idx, ex, ey = self._exc
        out = []
        a, b = np.searchsorted(idx, lo), np.searchsorted(idx, hi)
        for q, e in ((self._cols["qx"], ex), (self._cols["qy"], ey)):
            p = np.empty(hi - lo, q.dtype)
            if hi - lo > 1:
                p[1:] = q[lo:hi - 1]
            if lo > 0 and hi > lo:
                p[0] = q[lo - 1]
            p[idx[a:b] - lo] = e[a:b]
            out.append(p)
        return out[0], out[1]


class SegmentList:
    """``track.segments``: a read-only sequence of Segment records backed by the SoA buffers."""

    def __init__(self, tg, lo, hi):
        self._tg, self._lo, self._hi = tg, lo, hi
        self._p = None

    def __len__(self):
        return self._hi - self._lo

    def __getitem__(self, i):
        n = len(self)
        if isinstance(i, slice):
            return [self[j] for j in range(*i.indices(n))]
        if i < 0:
            i += n
        if not 0 <= i < n:
            raise IndexError(i)
        if self._tg._lengths_only:
            raise RuntimeError(f"a Segment needs p and q: {LENGTHS_ONLY_MSG} (read tg.segments['len'] / ['element'])")
        s, o = self._tg.segments, self._lo + i
        if self._p is None:
            self._p = s.p_range(self._lo, self._hi)
        return Segment(np.array([self._p[0][i], self._p[1][i]]), np.array([s["qx"][o], s["qy"][o]]), float(s["len"][o]),
                       int(s["element"][o]))

    def __iter__(self):
        return (self[i] for i in range(len(self)))

    def arrays(self):
        """SoA slices (px, py, qx, qy, len, element) of this track."""
        s = self._tg.segments
        px, py = s.p_range(self._lo, self._hi)
        return {"px": px, "py": py, **{k: s[k][self._lo:self._hi] for k in ("qx", "qy", "len", "element")}}


class Track:  # src/track.jl:42-57 ; a view over the track SoA
    def __init__(self, tg, idx):
        self._tg, self._i = tg, idx

    def _col(self, name):
        return self._tg.track_data[name][self._i]

    uid = property(lambda s: int(s._tg.uid_begin + s._i))
    azim_idx = property(lambda s: int(s._col("azim_idx")))
    track_idx = property(lambda s: int(s._col("track_idx")))
    p = property(lambda s: s._col("p").copy())
    q = property(lambda s: s._col("q").copy())
    phi = property(lambda s: float(s._col("phi")))
    ell = property(lambda s: float(s._col("len")))
    ABC = property(lambda s: s._col("abc").copy())
    next_track_fwd = property(lambda s: s._tg.tracks_by_uid[int(s._col("next_fwd"))])
    next_track_bwd = property(lambda s: s._tg.tracks_by_uid[int(s._col("next_bwd"))])

    @property
    def segments(self):
        tg = self._tg
        off = tg.segment_offsets
        u0, u1, base, n = tg.resident_batch()
        if not u0 <= self.uid < u1:  # batched fill (rt_set_segment_capacity / a shard larger than memory): only one batch is resident
            raise LookupError(f"segments of track uid {self.uid} are not resident: the device holds the batch of uids [{u0}, {u1}) "
                              "(consume earlier batches through segmentize_(..., on_batch=...))")
        lo, hi = int(off[self._i] - base), int(off[self._i + 1] - base)
        if not 0 <= lo <= hi <= n:
            raise IndexError(f"segment range [{lo}, {hi}) of track uid {self.uid} outside the resident batch of {n} segments")
        return SegmentList(tg, lo, hi)

    def __repr__(self):
        return f"Track(uid={self.uid}, azim_idx={self.azim_idx}, track_idx={self.track_idx}, p={self.p}, q={self.q})"


def bc_fwd(track: Track) -> BoundaryType:  # src/track.jl:82
    return BoundaryType(int(track._col("bc_fwd")))


def bc_bwd(track: Track) -> BoundaryType:
    return BoundaryType(int(track._col("bc_bwd")))


def dir_next_track_fwd(track: Track) -> DirectionType:
    return DirectionType(int(track._col("dir_fwd")))


def dir_next_track_bwd(track: Track) -> DirectionType:
    return DirectionType(int(track._col("dir_bwd")))


def ell(x):  # RayTracing.ℓ (src/segment.jl:35)
    return x.ell


class _TracksByUid:
    """``tg.tracks_by_uid[uid]`` with the reference's 1-based uid; only this rank's shard is resident."""

    def __init__(self, tg):
        self._tg = tg

    def __len__(self):
        return self._tg.n_total_tracks

    def __getitem__(self, uid):
        tg = self._tg
        if not tg._traced:
            raise RuntimeError("UndefRefError: access to undefined reference (call trace_ first)")
        if isinstance(uid, slice):
            return [self[u] for u in range(*uid.indices(len(self) + 1)) if u >= 1]
        if not tg.uid_begin <= uid < tg.uid_end:
            raise IndexError(f"uid {uid} outside this shard [{tg.uid_begin}, {tg.uid_end})")
        return Track(tg, uid - tg.uid_begin)

    def __iter__(self):
        return (self[u] for u in range(self._tg.uid_begin, self._tg.uid_end))


class _TracksByAngle:
    """``tg.tracks[i][j]`` (1-based azimuthal index, then 1-based track index)."""

    def __init__(self, tg, i=None):
        self._tg, self._i = tg, i

    def __getitem__(self, k):
        tg = self._tg
        if self._i is None:
            if not 1 <= k <= nazim2(tg.azimuthal_quadrature):
                raise IndexError(k)
            return _TracksByAngle(tg, k)
        if not 1 <= k <= tg.n_tracks[self._i - 1]:
            raise IndexError(k)
        return tg.tracks_by_uid[int(tg._base[self._i - 1] + k)]

    def __len__(self):
        tg = self._tg
        return nazim2(tg.azimuthal_quadrature) if self._i is None else int(tg.n_tracks[self._i - 1])


class TrackLayout:
    """The pure-host part of the TrackGenerator constructor (src/trackgenerator.jl:84-108): quadrature object and
    track counts per angle.  No device is touched; shard planning and the per-angle tables only need this."""

    def __init__(self, mesh: Mesh, n_azim: int, delta: float):
        self.mesh = mesh
        aq = AzimuthalQuadrature(n_azim, delta)
        self.azimuthal_quadrature = aq
        n2, n4 = nazim2(aq), nazim4(aq)
        dx, dy = mesh.width, mesh.height
        self.n_tracks_x = np.zeros(n2, dtype=np.int64)
        self.n_tracks_y = np.zeros(n2, dtype=np.int64)
        self.n_tracks = np.zeros(n2, dtype=np.int64)
        for i in range(1, n4 + 1):  # src/trackgenerator.jl:96-108
            phi = math.pi / n2 * (i - 1 / 2)
            nx = int(math.floor(dx / delta * abs(math.sin(phi))) + 1)
            ny = int(math.floor(dy / delta * abs(math.cos(phi))) + 1)
            j = n2 - i + 1
            self.n_tracks_x[i - 1] = self.n_tracks_x[j - 1] = nx
            self.n_tracks_y[i - 1] = self.n_tracks_y[j - 1] = ny
            self.n_tracks[i - 1] = self.n_tracks[j - 1] = nx + ny
        self.n_total_tracks = int(self.n_tracks.sum())
        self._base = np.concatenate([[0], np.cumsum(self.n_tracks)]).astype(np.int64)


class TrackGenerator(TrackLayout):
    """TrackGenerator(model, n_azim, delta; bcs, tiny_step=1e-8, volume_correction=false)
    (src/trackgenerator.jl:80-125).  Extra keywords select the GPU and the uid shard:
    ``device`` (CUDA ordinal) and ``shard=(rank, n_ranks)`` -- tracks are split into ``n_ranks`` contiguous uid
    ranges of equal total track length, the mesh is replicated."""

    def __init__(self, model, n_azim: int, delta: float, bcs: BoundaryConditions | None = None, tiny_step: float = 1e-8,
                 volume_correction: bool = False, device: int = 0, shard: tuple[int, int] = (0, 1)):
        if isinstance(model, Mesh):
            mesh = model
        elif isinstance(model, UnstructuredDiscreteModel):
            mesh = Mesh(model)
        else:
            raise TypeError("model must be an UnstructuredDiscreteModel")
        AzimuthalQuadrature(n_azim, delta)  # argument errors (src/azimuthal_quad.jl:22-25) come before any device work
        self.mesh = mesh
        self._pinned, self._pinned_mesh, self._ctx = {}, None, None
        # device context + mesh upload (Mesh(model), src/mesh.jl:24-31) -- before the layout: with device-side ingestion the
        # bounding box the layout needs comes back from the device
        L = _lib.lib()
        h = C.c_void_p()
        rc = L.rt_create(C.byref(h), int(device))
        if rc:
            raise _lib.RTError(rc, f"rt_create(device={device}) failed: no usable CUDA device (there is no CPU fallback)")
        self._ctx = h
        self._traced = self._segmented = False
        self._track_data = self._segments = self._offsets = None
        self.upload_mesh()
        super().__init__(mesh, n_azim, delta)
        self.bcs = bcs if bcs is not None else BoundaryConditions()
        self.tiny_step = float(tiny_step)
        self.volume_correction = bool(volume_correction)
        self._pinned_volumes = _lib.PinnedArray((max(mesh.num_cells, 1),), np.float64)  # (rt_volumes copies straight into it)
        self.volumes = self._pinned_volumes.array[:mesh.num_cells]
        self.volumes[:] = 0.0
        self.tracks = _TracksByAngle(self)
        self.tracks_by_uid = _TracksByUid(self)
        self.shard = (int(shard[0]), int(shard[1]))
        self.uid_begin, self.uid_end = 1, self.n_total_tracks + 1
        self._traced = False
        self._segmented = False
        self._track_data = None
        self._segments = None
        self._offsets = None
        self._resident = None
        self._in_batch = False  # inside the on_batch of segmentize_: the batch it received is resident
        self._lengths_only = False  # the last segmentize_ wrote only len and element (RT_SEG_LENGTHS_ONLY)
        self.volume_factors = None
        self.n_segments = 0

    def _mesh_arrays(self):
        """The arrays rt_mesh_upload reads: xy, cell ptrs/data and -- unless the mesh leaves them to the device -- the
        vertex->cells ptrs/data."""
        mesh, m = self.mesh, self.mesh.model
        a = [m.node_coordinates.reshape(-1), mesh.cell_nodes[0], mesh.cell_nodes[1]]
        if not mesh.device_ingest:
            a += [mesh.node_cells[0], mesh.node_cells[1]]
        return a

    def pin_mesh(self):
        """Keep the flattened mesh arrays in page-locked host memory, so that upload_mesh() is one asynchronous DMA per
        array at full PCIe rate (a Julia caller would register its Gridap arrays with cudaHostRegister instead)."""
        self._pinned_mesh = []
        for a in self._mesh_arrays():
            buf = _lib.PinnedArray(a.shape, a.dtype)
            buf.array[...] = a
            self._pinned_mesh.append(buf)

    def upload_mesh(self):
        """Host -> device copy of the flattened mesh + device-side preparation (rt_mesh_upload)."""
        mesh, m = self.mesh, self.mesh.model
        arrs = [b.array for b in self._pinned_mesh] if self._pinned_mesh else self._mesh_arrays()
        xy, cp, cd = arrs[:3]
        np_, nd = (arrs[3], arrs[4]) if len(arrs) == 5 else (None, None)
        L = _lib.lib()
        _lib.check(self._ctx, L.rt_mesh_upload(self._ctx, m.num_nodes, xy, m.num_cells, cp, cd, _lib.ptr(np_), _lib.ptr(nd),
                                               _lib.ptr(mesh.bb_min), _lib.ptr(mesh.bb_max)))
        if mesh.bb_min is None:  # reduced on the device (src/mesh.jl:53-69)
            lo, hi = np.zeros(2), np.zeros(2)
            _lib.check(self._ctx, L.rt_mesh_bbox(self._ctx, lo, hi))
            mesh.bb_min, mesh.bb_max = lo, hi
        self._traced = self._segmented = False
        self._track_data = self._segments = self._offsets = self._resident = None
        self._n_regions = 0  # (rt_mesh_upload clears the region map)

    def device_node_cells(self):
        """The vertex->cells table as the device holds it (1-based CSR like Gridap's Table)."""
        m = self.mesh.model
        ptrs, data = np.zeros(m.num_nodes + 1, np.int32), np.zeros(3 * m.num_cells, np.int32)
        _lib.check(self._ctx, _lib.lib().rt_mesh_node_cells(self._ctx, _lib.ptr(ptrs), _lib.ptr(data)))
        return ptrs, data

    def mesh_h2d_bytes(self) -> int:
        mesh, m = self.mesh, self.mesh.model
        return int(sum(a.nbytes for a in self._mesh_arrays()))

    def set_option(self, name: str, value: float):
        """Tuning knob of the library (``rt_set_option``, include/rt_b200.h): "chunk_segments", "band_min", "band_div",
        "target_walkers", "order_grid", "order_classes", "pipeline", ...  None of them changes a result."""
        _lib.check(self._ctx, _lib.lib().rt_set_option(self._ctx, name.encode(), float(value)))

    def timer_start(self):
        _lib.check(self._ctx, _lib.lib().rt_timer_start(self._ctx))

    def timer_stop(self) -> float:
        ms = C.c_double(0.0)
        _lib.check(self._ctx, _lib.lib().rt_timer_stop(self._ctx, C.byref(ms)))
        return ms.value

    # ---- lazily fetched device results -------------------------------------------------------------
    def _resident_valid(self):
        """a Segment batch is resident: after segmentize_, or inside its on_batch"""
        return self._segmented or self._in_batch

    @property
    def track_data(self):
        if self._track_data is None:
            if not self._traced:
                raise RuntimeError("call trace_ first")
            n = self.uid_end - self.uid_begin
            t = dict(azim_idx=np.zeros(n, np.int64), track_idx=np.zeros(n, np.int64), p=np.zeros((n, 2)), q=np.zeros((n, 2)),
                     phi=np.zeros(n), len=np.zeros(n), abc=np.zeros((n, 3)), bc_fwd=np.zeros(n, np.int8),
                     bc_bwd=np.zeros(n, np.int8), dir_fwd=np.zeros(n, np.int8), dir_bwd=np.zeros(n, np.int8),
                     next_fwd=np.zeros(n, np.int64), next_bwd=np.zeros(n, np.int64))
            _lib.check(self._ctx, _lib.lib().rt_tracks_download(self._ctx, *[_lib.ptr(v) for v in t.values()]))
            self._track_data = t
        return self._track_data

    @property
    def segment_offsets(self):
        if self._offsets is None:
            if not self._segmented:
                raise RuntimeError("call segmentize_ first")
            n = self.uid_end - self.uid_begin
            self._offsets = np.zeros(n + 1, np.int64)
            self._status = np.zeros(n, np.int32)
            _lib.check(self._ctx, _lib.lib().rt_segment_offsets(self._ctx, _lib.ptr(self._offsets), _lib.ptr(self._status)))
        return self._offsets

    @property
    def segment_status(self):
        """per-track status of the last segmentize_ (RT_TRACK_*: 0 ok, 1 "Try increasing k", 2 length check, 4 undefined x_int)"""
        self.segment_offsets
        return self._status

    @property
    def segments(self):
        """SoA dict px, py, qx, qy, len, element of the resident batch (the whole shard when it fitted); len and element only
        after ``segmentize_(..., lengths_only=True)``."""
        if self._segments is None:
            self.fetch_segments()
        return self._segments

    def resident_batch(self):
        """(uid_begin, uid_end, offset_base, n_segments) of the Segment batch the device holds (``rt_segments_device``), read
        when first needed after a segmentize_ and dropped whenever the segments are invalidated."""
        if self._resident is None:
            if not self._resident_valid():
                raise RuntimeError("call segmentize_ first")
            view = _lib.rt_batch()
            _lib.check(self._ctx, _lib.lib().rt_segments_device(self._ctx, C.byref(view)))
            self._resident = (int(view.uid_begin), int(view.uid_end), int(view.offset_base), int(view.n_segments))
        return self._resident

    def fetch_segments(self, pinned: bool = False, compact: bool = False, max_exceptions: int | None = None):
        """Device -> host copy of the Segment records of the resident batch.  By default into fresh numpy arrays the caller owns.
        ``pinned=True`` stages into page-locked buffers that are REUSED by the next pinned fetch of this TrackGenerator (full PCIe
        rate, no allocation per call): the arrays returned by an earlier pinned fetch then show the new data.  A buffer that has
        to grow is never freed under a view that is still alive (its memory is released when the last view dies).
        ``compact=True`` moves 28 instead of 44 bytes per segment (rt_segments_download_compact): q, len, element plus the list of
        positions where p is not the preceding q; ``px`` / ``py`` are rebuilt on the host on first use (SegmentColumns).
        ``compact="q"`` leaves ``len`` on the device as well (20 bytes per segment): it is rebuilt as norm(p - q) with the same
        IEEE operations (not after ``correct_volumes``, which rescales the resident lengths).
        Inside ``on_batch`` of segmentize_ it copies the batch the callback received.  After ``segmentize_(..., lengths_only=True)``
        it copies len and element (12 bytes per segment); ``compact`` is then an error."""
        if not self._resident_valid():
            raise RuntimeError("call segmentize_ first")
        if compact and self._lengths_only:
            raise RuntimeError(f"fetch_segments(compact=...) sends q and rebuilds p: {LENGTHS_ONLY_MSG}")
        L = _lib.lib()
        n = self.resident_batch()[3]
        names = [("px", np.float64), ("py", np.float64), ("qx", np.float64), ("qy", np.float64), ("len", np.float64),
                 ("element", np.int32)]
        if self._lengths_only:
            names = names[4:]
        if compact:
            names = names[2:]
            if compact == "q":
                names = [nd for nd in names if nd[0] != "len"]

        def buffer(name, dt, count):
            if not pinned:
                return np.zeros(count, dt)
            buf = self._pinned.get(name)
            if buf is None or buf.array.shape[0] < count:
                buf = _lib.PinnedArray((max(count, 1),), dt)  # (the old buffer lives on for as long as views of it do)
                self._pinned[name] = buf
            return buf.array[:count]

        out = {name: buffer(name, dt, n) for name, dt in names}
        if not compact:
            _lib.check(self._ctx, L.rt_segments_download(self._ctx, *[_lib.ptr(out.get(k)) for k in SegmentColumns.KEYS]))
            self._segments = SegmentColumns(out, lengths_only=self._lengths_only)
            return self._segments
        cap = max(getattr(self, "_exc_cap", 0), 4 * (self.uid_end - self.uid_begin) + n // 64 + 1024) if max_exceptions is None else int(max_exceptions)
        for _ in range(2):
            ei, ex, ey = buffer("exc_index", np.int64, cap), buffer("exc_px", np.float64, cap), buffer("exc_py", np.float64, cap)
            k = C.c_int64(0)
            rc = L.rt_segments_download_compact(self._ctx, *[_lib.ptr(out.get(kk)) for kk in ("qx", "qy", "len", "element")], cap,
                                                _lib.ptr(ei), _lib.ptr(ex), _lib.ptr(ey), C.byref(k))
            if rc != -10:  # RT_ERR_NOMEM: more exceptions than room -- once more with the count the call reported
                break
            cap = int(k.value) + 1024
        _lib.check(self._ctx, rc)
        self._exc_cap = cap if max_exceptions is None else getattr(self, "_exc_cap", 0)
        self.n_exceptions = int(k.value)
        self._segments = SegmentColumns(out, (ei[:k.value], ex[:k.value], ey[:k.value]))
        return self._segments

    # ---- sweep-facing device views (SURVEY 8f-1) ----------------------------------------------------
    def track_view(self):
        """Device-resident Track records of this shard (``rt_tracks_device``) as ``DeviceColumn``s: p, q, len, ABC, azim,
        next-track uids, boundary conditions and link directions -- what a transport sweep follows between tracks."""
        v = _lib.rt_track_view()
        _lib.check(self._ctx, _lib.lib().rt_tracks_device(self._ctx, C.byref(v)))
        n = int(v.n_tracks)
        kinds = {"d_azim": "<i4", "d_track_idx": "<i8", "d_next_fwd": "<i8", "d_next_bwd": "<i8", "d_bc_fwd": "|i1",
                 "d_bc_bwd": "|i1", "d_dir_fwd": "|i1", "d_dir_bwd": "|i1"}
        out = {"uid_begin": int(v.uid_begin), "n_tracks": n}
        for name, _ in v._fields_[2:-1]:
            out[name[2:]] = DeviceColumn(getattr(v, name), n, kinds.get(name, "<f8"))
        return out

    def quadrature_device(self):
        """(omega, view): the azimuthal weights of init_weights! computed on the device, and DeviceColumns of the per-angle
        tables phi / sin / cos / delta_eff / omega."""
        v = _lib.rt_quad_view()
        n2 = nazim2(self.azimuthal_quadrature)
        omega = np.zeros(n2)
        _lib.check(self._ctx, _lib.lib().rt_quadrature_device(self._ctx, C.byref(v), _lib.ptr(omega)))
        view = {k[2:]: DeviceColumn(getattr(v, k), n2, "<f8") for k in ("d_phi", "d_sin", "d_cos", "d_delta_eff", "d_omega")
                if getattr(v, k)}
        return omega, view

    def optical_lengths(self, sigma_t, layout: int = 0, fetch: bool = True):
        """tau[s][g] = sigma_t[element(s)][g] * len(s) on the device for the resident segments (Segment.tau, src/segment.jl:27).
        ``sigma_t``: (n_cells, n_groups).  Returns (numpy copy or None, DeviceColumn); the device buffer is reused by the next call.
        Inside ``on_batch`` of segmentize_: tau of the batch the callback received."""
        sig = np.ascontiguousarray(sigma_t, dtype=np.float64)
        if sig.ndim != 2 or sig.shape[0] != self.mesh.num_cells:
            raise ValueError("sigma_t must have shape (n_cells, n_groups)")
        G = sig.shape[1]
        view = _lib.rt_batch()
        _lib.check(self._ctx, _lib.lib().rt_segments_device(self._ctx, C.byref(view)))
        n = int(view.n_segments)
        host = np.zeros((n, G) if layout == 0 else (G, n)) if fetch else None
        d = C.c_void_p()
        _lib.check(self._ctx, _lib.lib().rt_optical_lengths(self._ctx, G, sig.reshape(-1), int(layout), C.byref(d), _lib.ptr(host)))
        return host, DeviceColumn(d.value, n * G, "<f8")

    # ---- material regions (a transport code's cross sections are per material) ----------------------------------------------
    def set_regions(self, cell_region, n_regions: int | None = None):
        """The region (material) of every cell, 1-based (``UnstructuredDiscreteModel.cell_regions``), checked and ordered on the
        device (rt_set_regions).  ``n_regions`` defaults to the largest value.  A value outside [1, n_regions] raises and keeps the
        previous map; ``None`` clears the map.  ``upload_mesh`` clears it too."""
        L = _lib.lib()
        if cell_region is None:
            _lib.check(self._ctx, L.rt_set_regions(self._ctx, 0, None))
            self._n_regions = 0
            return
        reg = np.ascontiguousarray(cell_region, dtype=np.int32).reshape(-1)
        if reg.shape[0] != self.mesh.num_cells:
            raise ValueError(f"cell_region has {reg.shape[0]} values for {self.mesh.num_cells} cells")
        n = int(reg.max()) if n_regions is None else int(n_regions)
        _lib.check(self._ctx, L.rt_set_regions(self._ctx, n, _lib.ptr(reg)))
        self._n_regions = n

    @property
    def n_regions(self) -> int:
        """regions of the map set with ``set_regions`` (0: none)"""
        return getattr(self, "_n_regions", 0)

    def optical_lengths_by_region(self, sigma_t, layout: int = 0, fetch: bool = True):
        """``optical_lengths`` with the cross sections per region: tau[s][g] = sigma_t[region(element(s))][g] * len(s), ``sigma_t``
        of shape (n_regions, n_groups).  Bit-equal to ``optical_lengths`` with the table expanded cell by cell, and the same return
        value: (numpy copy or None, DeviceColumn).  Needs ``set_regions``; inside ``on_batch`` of segmentize_ it acts on the batch
        the callback received."""
        sig = np.ascontiguousarray(sigma_t, dtype=np.float64)
        if sig.ndim != 2 or sig.shape[0] != self.n_regions:
            raise ValueError(f"sigma_t must have shape (n_regions = {self.n_regions}, n_groups)")
        G = sig.shape[1]
        view = _lib.rt_batch()
        _lib.check(self._ctx, _lib.lib().rt_segments_device(self._ctx, C.byref(view)))
        n = int(view.n_segments)
        host = np.zeros((n, G) if layout == 0 else (G, n)) if fetch else None
        d = C.c_void_p()
        _lib.check(self._ctx, _lib.lib().rt_optical_lengths_by_region(self._ctx, G, sig.reshape(-1), int(layout), C.byref(d),
                                                                        _lib.ptr(host)))
        return host, DeviceColumn(d.value, n * G, "<f8")

    def region_volumes(self, traced: bool = True, exact: bool = True):
        """(traced, exact): per-region sums of ``tg.volumes`` (the traced volumes of the last segmentize_, all-reduced or chained
        with a communicator) and of ``element_volumes()`` (triangle meshes only), summed on the device over the cells of each
        region in ascending id (rt_region_volumes) -- what δ and n_azim are chosen by.  Either may be skipped (None)."""
        t = np.zeros(self.n_regions) if traced else None
        e = np.zeros(self.n_regions) if exact else None
        _lib.check(self._ctx, _lib.lib().rt_region_volumes(self._ctx, _lib.ptr(t), _lib.ptr(e)))
        return t, e

    def find_elements(self, xy, k: int = 2, fetch: bool = True):
        """find_element(mesh, x, k) (src/mesh.jl:103-146) for every row of ``xy`` (n, 2) in one device call (rt_find_elements): the
        1-based cell of each point, -1 where no cell passes.  Returns (int32 ids or None, DeviceColumn); the device buffer is reused
        by the next call.  Needs only the uploaded mesh; it leaves the segments, volumes and stats of segmentize_ as they are and may
        be called inside its ``on_batch``."""
        pts = np.ascontiguousarray(xy, dtype=np.float64)
        if pts.ndim != 2 or pts.shape[1] != 2:
            raise ValueError("xy must have shape (n, 2)")
        n = pts.shape[0]
        ids = np.empty(n, np.int32) if fetch else None
        d = C.c_void_p()
        _lib.check(self._ctx, _lib.lib().rt_find_elements(self._ctx, n, pts.reshape(-1), int(k), _lib.ptr(ids), C.byref(d)))
        return ids, DeviceColumn(d.value, n, "<i4")

    def element_volumes(self):
        """element_volume of every cell (src/trackgenerator.jl:402-411: the `volumes2` the reference computes and discards)."""
        a = np.zeros(self.mesh.num_cells)
        _lib.check(self._ctx, _lib.lib().rt_element_volumes(self._ctx, _lib.ptr(a), None))
        return a

    def correct_volumes(self):
        """The reference's announced volume correction (src/trackgenerator.jl:388): resident segment lengths are scaled by
        area[element] / volumes[element].  Returns the per-element factors; ``tg.segments`` is re-read afterwards.
        Inside ``on_batch`` of segmentize_ it corrects the batch the callback received with the volumes of the segmentize_ before
        the running one (see segmentize_)."""
        f = np.zeros(self.mesh.num_cells)
        _lib.check(self._ctx, _lib.lib().rt_correct_volumes(self._ctx, _lib.ptr(f), None))
        self._segments = None
        return f

    def chunk_stats(self):
        s = np.zeros(8)
        _lib.check(self._ctx, _lib.lib().rt_debug_chunk_stats(self._ctx, s))
        return dict(zip(["working_chunks", "void_seeds", "mean_segments", "max_segments", "sum_unit_max", "sum_unit_mean", "slots", "units"], s.tolist()))

    def phase_ms(self):
        ms = np.zeros(6)
        _lib.lib().rt_phase_ms(self._ctx, ms)
        return dict(zip(["upload", "trace", "count", "scan", "fill", "volumes"], ms.tolist()))

    def stats(self):
        s = np.zeros(8)
        _lib.lib().rt_stats(self._ctx, s)
        return dict(zip(["launches", "fast_transitions", "literal_iterations", "nn_queries", "knn_queries", "count_ms",
                         "fill_ms", "scan_ms"], s.tolist()))

    def info(self, key: str) -> float:
        v = C.c_double(0.0)
        _lib.check(self._ctx, _lib.lib().rt_info(self._ctx, key.encode(), C.byref(v)))
        return v.value

    def neighbours(self):
        nb = np.zeros(3 * self.mesh.num_cells, np.int32)
        _lib.check(self._ctx, _lib.lib().rt_mesh_neighbours(self._ctx, nb))
        return nb.reshape(-1, 3)

    def close(self):
        if getattr(self, "_ctx", None):
            for b in list(getattr(self, "_pinned_mesh", None) or []):
                b.free()
            self._pinned = {}  # (result buffers are released when the last numpy view of them dies)
            self._pinned_mesh = None
            self._segments = None
            _lib.lib().rt_destroy(self._ctx)
            self._ctx = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __repr__(self):  # src/trackgenerator.jl:52-63
        aq = self.azimuthal_quadrature
        return ("  Number of azimuthal angles in (0, π): %d\n  Azimuthal angles in (0, π): %s\n"
                "  Effective azimuthal spacings: %s\n  Total tracks: %d\n  Correct volumes: %s" %
                (nazim2(aq), np.round(np.degrees(aq.phis), 2), np.round(aq.deltas, 3), self.n_total_tracks,
                 str(self.volume_correction).lower()))


def find_element(tg: TrackGenerator, x, k: int = 2) -> int:
    """find_element(mesh, x, k=2) (src/mesh.jl:103-146) for one point ``x`` = (x, y) on the mesh of ``tg``: the 1-based cell, or -1
    like the reference when no cell passes.  For many points use ``tg.find_elements``."""
    ids, _ = tg.find_elements(np.asarray(x, dtype=np.float64).reshape(1, 2), k)
    return int(ids[0])


def _angle_tables(tg: TrackLayout):
    """Effective angles/spacings of trace! (src/trackgenerator.jl:150-166) with the host libm, plus the sin/cos/tan
    tables the device needs (no device trigonometry, see include/rt_b200.h)."""
    aq = tg.azimuthal_quadrature
    n2, n4 = nazim2(aq), nazim4(aq)
    dx, dy = tg.mesh.width, tg.mesh.height
    dxe, dye = np.zeros(n2), np.zeros(n2)
    for i in range(1, n4 + 1):
        phi = math.atan((dy * float(tg.n_tracks_x[i - 1])) / (dx * float(tg.n_tracks_y[i - 1])))
        aq.phis[i - 1] = phi
        dxe[i - 1] = dx / float(tg.n_tracks_x[i - 1])
        dye[i - 1] = dy / float(tg.n_tracks_y[i - 1])
        aq.deltas[i - 1] = dxe[i - 1] * math.sin(phi)
        j = n2 - i + 1
        aq.phis[j - 1] = math.pi - phi
        dxe[j - 1], dye[j - 1], aq.deltas[j - 1] = dxe[i - 1], dye[i - 1], aq.deltas[i - 1]
    init_weights_(aq)
    sin_t = np.array([math.sin(p) for p in aq.phis])
    cos_t = np.array([math.cos(p) for p in aq.phis])
    tan_t = np.array([math.tan(p) for p in aq.phis])
    return sin_t, cos_t, tan_t, dxe, dye


def trace_(tg: TrackGenerator) -> TrackGenerator:
    """trace!(tg): effective quadrature on the host, then ONE kernel over (phi, track) pairs."""
    L = _lib.lib()
    sin_t, cos_t, tan_t, dxe, dye = _angle_tables(tg)
    aq = tg.azimuthal_quadrature
    n2 = nazim2(aq)
    rank, n_ranks = tg.shard
    if n_ranks > 1:
        from .distributed import plan_shards

        bounds = plan_shards(tg, n_ranks)  # host planner (rt_plan_shards is the same split computed on the device)
        tg.shard_bounds = bounds
        tg.uid_begin, tg.uid_end = int(bounds[rank]), int(bounds[rank + 1])
    else:
        tg.uid_begin, tg.uid_end = 1, tg.n_total_tracks + 1
    tg._traced = False
    tg._segmented = False
    tg._track_data = tg._segments = tg._offsets = tg._resident = None
    rc = L.rt_trace(tg._ctx, n2, tg.n_tracks_x, tg.n_tracks_y, aq.phis, sin_t, cos_t, tan_t, dxe, dye, tg.bcs.codes(),
                    tg.uid_begin, tg.uid_end)
    if rc == -4:
        raise DomainError("could not found track exit point.")
    _lib.check(tg._ctx, rc)
    tg._traced = True
    return tg


class DeviceColumn:
    """A device-resident column of a segment batch, consumable by torch / cupy through ``__cuda_array_interface__``."""

    def __init__(self, ptr, n, typestr):
        self.__cuda_array_interface__ = {"shape": (int(n),), "typestr": typestr, "data": (int(ptr or 0), False), "version": 2}


class SegmentBatch:
    """One uid batch of Segment records as produced on the device (``rt_batch`` of include/rt_b200.h): what an on-GPU consumer
    (a transport sweep) sees when the shard's segments do not fit in memory at once.  ``px``, ``py``, ``qx``, ``qy`` are None
    after ``segmentize_(..., lengths_only=True)``."""

    def __init__(self, b):
        self.uid_begin, self.uid_end, self.n_segments = int(b.uid_begin), int(b.uid_end), int(b.n_segments)
        self.offset_base, self.attempt, self.stream = int(b.offset_base), int(b.attempt), b.stream
        self.d_offsets = b.d_offsets  # device pointer: int64 offsets of the shard's tracks (n_shard + 1)
        n = self.n_segments
        self.px, self.py, self.qx, self.qy = (DeviceColumn(p, n, "<f8") if p else None for p in (b.d_px, b.d_py, b.d_qx, b.d_qy))
        self.len = DeviceColumn(b.d_len, n, "<f8")
        self.element = DeviceColumn(b.d_element, n, "<i4")


def segmentize_(tg: TrackGenerator, k: int = 5, rtol: float = RTOL_DEFAULT, flags: int = 0, max_iter: int = MAX_ITER,
                check: bool = True, fetch_volumes: bool = True, on_batch=None, exact_volumes: bool = False,
                lengths_only: bool = False) -> TrackGenerator:
    """segmentize!(tg; k, rtol): count pass -> scan -> fill pass (+ fused fill_volumes) on the device.
    ``on_batch(SegmentBatch)`` is called after every uid batch of the fill pass (one batch when everything fits).  Inside it
    ``tg.resident_batch()``, ``tg.fetch_segments()`` / ``tg.segments``, ``tg.optical_lengths()``, ``tg.optical_lengths_by_region()``
    and ``tg.correct_volumes()`` act on that batch.  An exception raised by ``on_batch`` stops the call and is re-raised here -- on a TrackGenerator with a
    communicator only after this rank has joined the call's all-reduce of the volumes (as after any other failure), so that its
    peers are not left waiting inside it.

    ``tg.volume_correction`` corrects the segments (``tg.volume_factors``) only when they all stay resident; otherwise, and with
    ``on_batch`` or RT_SEG_COUNT_ONLY, ``tg.volume_factors`` is None.  Batched segments are corrected by a second segmentize_
    whose ``on_batch`` calls ``tg.correct_volumes()`` for every batch: the factors come from the volumes of the call before it,
    which must have run with volumes, and the correcting call may use RT_SEG_NO_VOLUMES (its own volumes would be those of the
    lengths before correction).

    ``exact_volumes=True`` (RT_SEG_EXACT_VOLUMES) sums the volumes in the reference's order -- tracks in uid order, segments in
    walk order -- so that they are bit-equal to fill_volumes and the same whatever the run, pipeline, knobs, segment capacity or
    number of ranks; the default sums them with atomics, whose last bits vary.  It cannot be combined with RT_SEG_COUNT_ONLY or
    RT_SEG_NO_VOLUMES, and with a communicator of several ranks each shard must fit in one batch and the shards must be in
    ascending uid order by rank.

    ``lengths_only=True`` (RT_SEG_LENGTHS_ONLY) writes only the len and element columns, 12 instead of 44 bytes per segment, for
    consumers that never read the end points (``optical_lengths``, ``correct_volumes``, an on-device sweep): everything else is
    computed as without it, and len / element are the same bits.  ``tg.segments`` then has only ``len`` and ``element``,
    ``SegmentBatch`` gives None for the end-point columns, and ``track.segments[i]`` and ``fetch_segments(compact=...)`` raise."""
    L = _lib.lib()
    if exact_volumes:
        flags |= _lib.RT_SEG_EXACT_VOLUMES
    if lengths_only:
        flags |= _lib.RT_SEG_LENGTHS_ONLY
    cb = None
    if on_batch is not None:
        def _cb(bptr, _user):
            tg._in_batch = True
            try:
                on_batch(SegmentBatch(bptr.contents))
                return 0
            except Exception as e:  # noqa: BLE001 -- reported through the return code
                tg._batch_error = e
                return 1
            finally:
                tg._in_batch = False
                tg._segments = tg._resident = None  # (read again from the device if needed: a later batch replaces this one)

        cb = _lib.BATCH_CB(_cb)
    if not tg._traced:
        raise RuntimeError("Segmentation is intended after tracing. Please, call `trace!` first!")
    tg._segmented = False
    tg._segments = tg._offsets = tg._resident = None
    tg._lengths_only = bool(flags & _lib.RT_SEG_LENGTHS_ONLY) and not flags & _lib.RT_SEG_COUNT_ONLY
    tg.volume_factors = None
    nseg, bad_uid, bad_status = C.c_int64(0), C.c_int64(0), C.c_int32(0)
    delta = tg.azimuthal_quadrature.deltas
    rc = L.rt_segmentize(tg._ctx, tg.tiny_step, int(k), float(rtol), int(max_iter), _lib.ptr(delta), int(flags),
                         C.cast(cb, C.c_void_p) if cb is not None else None, None,
                         C.byref(nseg), C.byref(bad_uid), C.byref(bad_status))
    batch_error, tg._batch_error = getattr(tg, "_batch_error", None), None
    tg.n_segments = int(nseg.value)
    tg.first_bad_uid, tg.bad_status = int(bad_uid.value), int(bad_status.value)
    want_vol = not (flags & _lib.RT_SEG_NO_VOLUMES)
    if rc not in (0, -8):
        # every rank of a communicator has to enter the all-reduce once per segmentize! -- a rank that failed (also because its
        # on_batch raised: the call then stops with RT_ERR_ARG) joins it with a zero contribution and the failed-rank flag
        # (rt_volumes), so that its peers are not left waiting; then the error is raised, the exception of on_batch if there is one
        msg = L.rt_last_error(tg._ctx)
        if want_vol and getattr(tg, "_has_comm", False):
            L.rt_volumes(tg._ctx, None)
        if batch_error is not None:
            raise batch_error
        raise _lib.RTError(rc, msg.decode() if msg else "")
    tg._segmented = True
    err = None
    if rc == -8 and check:  # a track failed like it does in the reference (src/track.jl:141,172); the other tracks are segmentized
        msg = L.rt_last_error(tg._ctx)
        err = _lib.RTError(rc, msg.decode() if msg else "")
    if want_vol:
        rcv = L.rt_volumes(tg._ctx, _lib.ptr(tg.volumes) if fetch_volumes else None)
        if err is not None:
            raise err  # (after the collective: the peers of this rank are not left inside ncclAllReduce)
        _lib.check(tg._ctx, rcv)
        # volume_correction = true: the reference's TODO (src/trackgenerator.jl:388), applied when every segment is resident
        # (the resident batch, not the allocated capacity: columns sized by an earlier call can be larger than the batches)
        if tg.volume_correction and on_batch is None and not (flags & _lib.RT_SEG_COUNT_ONLY) and tg.resident_batch()[3] == tg.n_segments:
            tg.volume_factors = tg.correct_volumes()
    elif err is not None:
        raise err
    return tg
