"""ctypes binding of librt_b200.so (the C ABI declared in include/rt_b200.h).

There is NO CPU fallback: if the CUDA library is missing, or no CUDA device can be opened, every entry
point raises.  ``build()`` compiles the library in-tree with nvcc for sm_100a.
"""
from __future__ import annotations

import ctypes as C
import glob
import os
import subprocess

import numpy as np

_PKG = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(_PKG)
SO_PATH = os.environ.get("RT_B200_LIB") or os.path.join(_PKG, "librt_b200.so")  # RT_B200_LIB: an alternative build
_CSRC = os.path.join(_PKG, "csrc")

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-fmad=false", "-std=c++17",
              "-shared", "-Xcompiler", "-fPIC"]


class RTError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"[rt_b200 {code}] {msg}")
        self.code = code
        self.msg = msg


def build(force: bool = False, verbose: bool = False) -> str:
    """nvcc -gencode arch=compute_100a,code=sm_100a ... -> raytracing.jl_b200/librt_b200.so"""
    # every file under csrc/ is a dependency (rt_b200.cu includes all the .cuh files), plus the public header
    main = os.path.join(_CSRC, "rt_b200.cu")
    deps = sorted(glob.glob(os.path.join(_CSRC, "*.cu")) + glob.glob(os.path.join(_CSRC, "*.cuh"))) + [os.path.join(_ROOT, "include", "rt_b200.h")]
    if (not force) and os.path.exists(SO_PATH) and all(os.path.getmtime(SO_PATH) >= os.path.getmtime(s) for s in deps):
        return SO_PATH
    nvcc = os.environ.get("NVCC", "nvcc")
    cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-o", SO_PATH, main, "-ldl"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + r.stdout + r.stderr)
    if verbose:
        print(r.stderr)
    return SO_PATH


_f64 = np.ctypeslib.ndpointer(dtype=np.float64, flags="C_CONTIGUOUS")
_i32 = np.ctypeslib.ndpointer(dtype=np.int32, flags="C_CONTIGUOUS")
_i64 = np.ctypeslib.ndpointer(dtype=np.int64, flags="C_CONTIGUOUS")
_vp = C.c_void_p


class rt_batch(C.Structure):
    _fields_ = [("uid_begin", C.c_int64), ("uid_end", C.c_int64), ("n_segments", C.c_int64), ("d_offsets", _vp),
                ("offset_base", C.c_int64), ("d_px", _vp), ("d_py", _vp), ("d_qx", _vp), ("d_qy", _vp), ("d_len", _vp),
                ("d_element", _vp), ("stream", _vp), ("attempt", C.c_int32)]


BATCH_CB = C.CFUNCTYPE(C.c_int, C.POINTER(rt_batch), _vp)


class rt_track_view(C.Structure):
    _fields_ = [("uid_begin", C.c_int64), ("n_tracks", C.c_int64)] + [(n, _vp) for n in (
        "d_px", "d_py", "d_qx", "d_qy", "d_len", "d_a", "d_b", "d_c", "d_azim", "d_track_idx", "d_next_fwd", "d_next_bwd",
        "d_bc_fwd", "d_bc_bwd", "d_dir_fwd", "d_dir_bwd", "stream")]


class rt_quad_view(C.Structure):
    _fields_ = [("n_azim_2", C.c_int32)] + [(n, _vp) for n in ("d_phi", "d_sin", "d_cos", "d_delta_eff", "d_omega")]

# name -> (restype, argtypes); every symbol include/rt_b200.h declares
SYMBOLS = {
    "rt_create": (C.c_int, [C.POINTER(_vp), C.c_int]),
    "rt_destroy": (None, [_vp]),
    "rt_last_error": (C.c_char_p, [_vp]),
    "rt_version": (C.c_char_p, []),
    "rt_host_alloc": (C.c_int, [C.POINTER(_vp), C.c_size_t]),
    "rt_host_free": (C.c_int, [_vp]),
    "rt_mesh_upload": (C.c_int, [_vp, C.c_int32, _f64, C.c_int32, _i32, _i32, _vp, _vp, _vp, _vp]),
    "rt_mesh_bbox": (C.c_int, [_vp, _f64, _f64]),
    "rt_mesh_node_cells": (C.c_int, [_vp, _vp, _vp]),
    "rt_mesh_neighbours": (C.c_int, [_vp, _i32]),
    "rt_trace": (C.c_int, [_vp, C.c_int32, _i64, _i64, _f64, _f64, _f64, _f64, _f64, _f64, _i32, C.c_int64, C.c_int64]),
    "rt_tracks_download": (C.c_int, [_vp] + [_vp] * 13),
    "rt_plan_shards": (C.c_int, [_vp, C.c_int32, _i64, _i64, _f64, _f64, _f64, _f64, C.c_int32, _i64]),
    "rt_set_segment_capacity": (C.c_int, [_vp, C.c_int64]),
    "rt_segmentize": (C.c_int, [_vp, C.c_double, C.c_int32, C.c_double, C.c_int32, _vp, C.c_uint32, _vp, _vp,
                                C.POINTER(C.c_int64), C.POINTER(C.c_int64), C.POINTER(C.c_int32)]),
    "rt_segment_offsets": (C.c_int, [_vp, _vp, _vp]),
    "rt_segments_download": (C.c_int, [_vp] + [_vp] * 6),
    "rt_segments_download_compact": (C.c_int, [_vp, _vp, _vp, _vp, _vp, C.c_int64, _vp, _vp, _vp, C.POINTER(C.c_int64)]),
    "rt_segments_device": (C.c_int, [_vp, C.POINTER(rt_batch)]),
    "rt_volumes": (C.c_int, [_vp, _vp]),
    "rt_tracks_device": (C.c_int, [_vp, C.POINTER(rt_track_view)]),
    "rt_quadrature_device": (C.c_int, [_vp, C.POINTER(rt_quad_view), _vp]),
    "rt_optical_lengths": (C.c_int, [_vp, C.c_int32, _f64, C.c_int32, C.POINTER(_vp), _vp]),
    "rt_set_regions": (C.c_int, [_vp, C.c_int32, _vp]),
    "rt_optical_lengths_by_region": (C.c_int, [_vp, C.c_int32, _f64, C.c_int32, C.POINTER(_vp), _vp]),
    "rt_region_volumes": (C.c_int, [_vp, _vp, _vp]),
    "rt_element_volumes": (C.c_int, [_vp, _vp, C.POINTER(_vp)]),
    "rt_correct_volumes": (C.c_int, [_vp, _vp, C.POINTER(_vp)]),
    "rt_find_elements": (C.c_int, [_vp, C.c_int64, _f64, C.c_int32, _vp, C.POINTER(_vp)]),
    "rt_comm_unique_id": (C.c_int, [_vp, C.c_char_p]),
    "rt_comm_init": (C.c_int, [_vp, C.c_int32, C.c_int32, C.c_char_p]),
    "rt_stats": (C.c_int, [_vp, _f64]),
    "rt_phase_ms": (C.c_int, [_vp, _f64]),
    "rt_debug_chunk_stats": (C.c_int, [_vp, _f64]),
    "rt_info": (C.c_int, [_vp, C.c_char_p, C.POINTER(C.c_double)]),
    "rt_set_option": (C.c_int, [_vp, C.c_char_p, C.c_double]),
    "rt_selftest_division": (C.c_int, [_vp, C.c_int64, C.c_uint64, C.c_int32, C.POINTER(C.c_int64)]),
    "rt_timer_start": (C.c_int, [_vp]),
    "rt_timer_stop": (C.c_int, [_vp, C.POINTER(C.c_double)]),
}

RT_SEG_LITERAL, RT_SEG_NO_VOLUMES, RT_SEG_COUNT_ONLY, RT_SEG_NO_CHUNKS, RT_SEG_SEQUENTIAL = 1, 2, 4, 8, 16
RT_SEG_EXACT_VOLUMES = 32
RT_SEG_LENGTHS_ONLY = 64

_lib = None


def lib():
    """Load librt_b200.so; raises (loudly) if it has not been built -- there is no fallback path."""
    global _lib
    if _lib is None:
        if not os.path.exists(SO_PATH):
            raise RTError(-1, f"{SO_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                              "(nvcc, sm_100a). There is no CPU fallback.")
        L = C.CDLL(SO_PATH)
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(L, name)  # AttributeError if the library does not export a declared symbol
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def check(ctx, rc):
    if rc != 0:
        msg = lib().rt_last_error(ctx)
        raise RTError(rc, msg.decode() if msg else "")


def ptr(a):
    return None if a is None else a.ctypes.data_as(_vp)


class _PinnedBlock:
    """Owns one cudaHostAlloc allocation; freed when the last numpy view of it is gone (or explicitly)."""

    def __init__(self, nbytes):
        self.p = _vp()
        rc = lib().rt_host_alloc(C.byref(self.p), max(1, nbytes))
        if rc:
            raise RTError(rc, "rt_host_alloc failed")

    def free(self):
        if self.p:
            lib().rt_host_free(self.p)
            self.p = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class PinnedArray:
    """numpy view over cudaHostAlloc'ed memory (rt_host_alloc).  The allocation is owned by the buffer object every view of
    ``array`` keeps alive through its ``base`` chain: dropping the PinnedArray never frees memory a view still points into.
    ``free()`` releases it at once -- only for buffers whose views the caller controls (the staged mesh arrays)."""

    def __init__(self, shape, dtype):
        self.dtype = np.dtype(dtype)
        n = int(np.prod(shape))
        self._block = _PinnedBlock(n * self.dtype.itemsize)
        buf = (C.c_char * (n * self.dtype.itemsize)).from_address(self._block.p.value)
        buf._owner = self._block  # numpy view -> memoryview -> buf -> block
        self.array = np.frombuffer(buf, dtype=self.dtype, count=n).reshape(shape)

    def free(self):
        self.array = None
        self._block.free()
