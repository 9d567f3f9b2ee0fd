"""B200-native drop-in for the trace! -> segmentize! hot path of RayTracing.jl (see DESIGN.md)."""
from .mesh import DiscreteModelFromFile, GmshDiscreteModel, Mesh, UnstructuredDiscreteModel  # noqa: F401
from . import plotdata, synth  # noqa: F401
from .api import (  # noqa: F401
    AzimuthalQuadrature, Backward, BoundaryConditions, BoundaryType, DirectionType, DomainError, Forward, Periodic,
    Reflective, Segment, SegmentColumns, Track, TrackGenerator, TrackLayout, Vacuum, bc_bwd, bc_fwd, dir_next_track_bwd, dir_next_track_fwd, ell,
    find_element, nazim, nazim2, nazim4, segmentize_, trace_, RTOL_DEFAULT, MAX_ITER,
)
from ._lib import RTError, RT_SEG_COUNT_ONLY, RT_SEG_LITERAL, RT_SEG_NO_CHUNKS, RT_SEG_NO_VOLUMES, RT_SEG_SEQUENTIAL, build  # noqa: F401
