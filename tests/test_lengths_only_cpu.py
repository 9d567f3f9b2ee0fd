"""RT_SEG_LENGTHS_ONLY without a device: the flag's value agrees in the header, the ctypes binding and the Julia glue, the glue's
lengths-only download passes NULL for the four end-point columns with the header's argument kinds, and the host containers of a
lengths-only batch (SegmentColumns, SegmentBatch, track.segments, fetch_segments(compact=...)) behave as documented."""
import os
import re

import numpy as np
import pytest

import raytracing_jl_b200 as rt
from raytracing_jl_b200 import _lib
from raytracing_jl_b200.api import SegmentBatch, SegmentColumns, SegmentList, TrackGenerator
from tests.test_abi_cpu import _c_prototypes

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_flag_value_agrees():
    hdr = open(os.path.join(ROOT, "include", "rt_b200.h")).read()
    assert re.search(r"RT_SEG_LENGTHS_ONLY\s*=\s*64\b", hdr)
    assert _lib.RT_SEG_LENGTHS_ONLY == rt.RT_SEG_LENGTHS_ONLY == 64
    jl = open(os.path.join(ROOT, "julia", "RayTracingB200.jl")).read()
    assert "(lengths_only ? 64 : 0)" in jl and "RT_SEG_LENGTHS_ONLY" in jl


def test_julia_lengths_only_download():
    """the glue's rt_segments_download of len / element: the header's argument kinds, NULL for px, py, qx, qy"""
    src = open(os.path.join(ROOT, "julia", "RayTracingB200.jl")).read()
    body = src[src.index("if lengths_only\n"):]
    m = re.search(r"ccall\(\(:rt_segments_download, LIBRT_B200\), Cint,\s*\(([^)]*)\),\s*([^)]*)\)", body)
    assert m, "no rt_segments_download in the lengths-only branch"
    kinds = ["ptr" if t.strip().startswith("Ptr{") else t.strip() for t in m.group(1).split(",")]
    assert kinds == _c_prototypes()["rt_segments_download"]
    args = [a.strip() for a in m.group(2).split(",")]
    assert args == ["ctx", "C_NULL", "C_NULL", "C_NULL", "C_NULL", "len", "el"]
    # materialize=true is refused before the device is asked for anything
    fn = src[src.index("function b200_segmentize!"):]
    assert fn.index("lengths_only && materialize && error(") < fn.index("_b200_context(t)")


def two_columns(n=5):
    return SegmentColumns({"len": np.arange(n, dtype=np.float64), "element": np.arange(1, n + 1, dtype=np.int32)}, lengths_only=True)


def test_segment_columns_with_two_columns():
    s = two_columns()
    assert list(s) == ["len", "element"] and len(s) == 2 and sorted(dict(s)) == ["element", "len"]
    assert s["len"][3] == 3.0 and s["element"][0] == 1
    for key in ("px", "py", "qx", "qy"):
        assert key not in s
        with pytest.raises(KeyError, match="RT_SEG_LENGTHS_ONLY"):
            s[key]
    with pytest.raises(KeyError, match="RT_SEG_LENGTHS_ONLY"):
        s.p_range(0, 2)
    with pytest.raises(KeyError):
        s["tau"]
    full = SegmentColumns({k: np.zeros(2) for k in SegmentColumns.KEYS})
    assert list(full) == list(SegmentColumns.KEYS) and not full.lengths_only


class _FakeTG:
    _lengths_only = True
    segments = two_columns()

    def _resident_valid(self):
        return True


def test_track_segments_and_compact_fetch_raise():
    segs = SegmentList(_FakeTG(), 1, 4)
    assert len(segs) == 3
    with pytest.raises(RuntimeError, match="RT_SEG_LENGTHS_ONLY"):
        segs[0]
    with pytest.raises(RuntimeError, match="RT_SEG_LENGTHS_ONLY"):
        TrackGenerator.fetch_segments(_FakeTG(), compact=True)


def test_segment_batch_without_end_points():
    b = _lib.rt_batch(uid_begin=3, uid_end=9, n_segments=40, d_offsets=0x1000, offset_base=7, d_px=None, d_py=None, d_qx=None,
                      d_qy=None, d_len=0x2000, d_element=0x3000, stream=None, attempt=0)
    sb = SegmentBatch(b)
    assert (sb.px, sb.py, sb.qx, sb.qy) == (None, None, None, None)
    assert sb.len.__cuda_array_interface__["data"][0] == 0x2000 and sb.len.__cuda_array_interface__["shape"] == (40,)
    assert sb.element.__cuda_array_interface__["typestr"] == "<i4"
