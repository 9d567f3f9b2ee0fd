"""find_elements(om, mesh, xy, k): the CPU oracle's find_element (src/mesh.jl:103-146) for every row of xy (n, 2) in one call, and
how many points entered the k-nearest-node branch -- the reference the device's rt_find_elements is compared with.  The loop is
tests/locate_oracle.c, compiled against the oracle's library into a temporary directory on first use."""
import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

from oracle import oracle

_SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "locate_oracle.c")
_i32p = np.ctypeslib.ndpointer(dtype=np.int32, flags="C_CONTIGUOUS")
_f64p = np.ctypeslib.ndpointer(dtype=np.float64, flags="C_CONTIGUOUS")
_lib = None


def lib():
    global _lib
    if _lib is None:
        so_oracle = oracle.build()
        d = tempfile.mkdtemp(prefix="locate_oracle_")
        atexit.register(shutil.rmtree, d, True)
        so = os.path.join(d, "liblocate_oracle.so")
        subprocess.run(["gcc", "-O2", "-fPIC", "-std=gnu11", "-shared", "-o", so, _SRC, so_oracle], check=True, capture_output=True)
        oracle.lib()
        L = C.CDLL(so)
        L.loc_find_elements.argtypes = [C.c_void_p, _i32p, _i32p, C.c_int64, _f64p, C.c_int, _i32p]
        L.loc_find_elements.restype = C.c_int64
        _lib = L
    return _lib


def find_elements(om, mesh, xy, k=2):
    """(int32 ids, 1-based or -1; points that entered the knn branch) on the oracle mesh ``om`` built from ``mesh``"""
    pts = np.ascontiguousarray(xy, dtype=np.float64).reshape(-1, 2)
    ptrs, data = (np.ascontiguousarray(a, np.int32) for a in mesh.node_cells)
    ids = np.zeros(pts.shape[0], np.int32)
    n_knn = lib().loc_find_elements(om._h, ptrs, data, pts.shape[0], pts.reshape(-1), int(k), ids)
    return ids, int(n_knn)
