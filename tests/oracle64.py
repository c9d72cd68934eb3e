"""The CPU oracle for int64 and uint64 volumes (tests/oracle64.cpp), with the interface of oracle/oracle_py.py.

TEST INFRASTRUCTURE.  The library is compiled once per process into a temporary directory, with the flags of
oracle/Makefile (no contraction or reassociation of the projection arithmetic).  Volumes of the other pixel types go to
oracle_py itself."""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

from util import ROOT, oracle

CODES = {np.dtype(np.int64): 8, np.dtype(np.uint64): 9}
_lib = None


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        out = os.path.join(tempfile.mkdtemp(prefix="oracle64_"), "liboracle64.so")
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-ffp-contract=off", "-fno-fast-math", "-shared", "-o", out,
                               os.path.join(ROOT, "tests", "oracle64.cpp")])
        L = C.CDLL(out)
        O = oracle()
        pd, pu64, vp = C.POINTER(C.c_double), C.POINTER(C.c_uint64), C.c_void_p
        L.orc64_cuberille.restype = vp
        L.orc64_cuberille.argtypes = [vp, C.c_int, pu64, pd, pd, C.POINTER(O._Params)]
        L.orc64_classify.argtypes = [vp, C.c_int, pu64, C.c_double, vp, C.c_uint64]
        L.orc64_project_points.argtypes = [vp, C.c_int, pu64, pd, pd, C.POINTER(O._Params), vp, C.c_uint64]
        L.orc64_sample.argtypes = [vp, C.c_int, pu64, pd, pd, vp, C.c_uint64, vp, vp]
        for name, rt in [("orc_num_points", C.c_uint64), ("orc_num_cells", C.c_uint64), ("orc_verts_per_cell", C.c_int),
                         ("orc_points", vp), ("orc_cells", vp), ("orc_cell_data", vp), ("orc_cell_data_bytes", C.c_uint64),
                         ("orc_step_length_used", C.c_double)]:
            getattr(L, name).restype = rt
            getattr(L, name).argtypes = [vp]
        L.orc_free.restype = None
        L.orc_free.argtypes = [vp]
        _lib = L
    return _lib


def cuberille(vol: np.ndarray, iso, *, triangles=True, project=True, cell_data=False, mode=0, thr=0.5, step=-1.0,
              relax=0.95, max_steps=50, spacing=None, origin=None, border_faces=False, region_index=(0, 0, 0),
              direction=None, method=0):
    """oracle_py.cuberille for any pixel type (no per-slice counts for the 64-bit ones)"""
    O = oracle()
    if vol.dtype not in CODES:
        return O.cuberille(vol, iso, triangles=triangles, project=project, cell_data=cell_data, mode=mode, thr=thr,
                           step=step, relax=relax, max_steps=max_steps, spacing=spacing, origin=origin,
                           border_faces=border_faces, region_index=region_index, direction=direction, method=method)
    L = lib()
    dims, sp, og = O._geom(vol, spacing, origin)
    P = O._params(iso, triangles, project, cell_data, mode, thr, step, relax, max_steps, border_faces, region_index,
                  direction, method)
    h = L.orc64_cuberille(vol.ctypes.data, CODES[vol.dtype], dims, sp, og, C.byref(P))
    assert h
    try:
        n, m, k = L.orc_num_points(h), L.orc_num_cells(h), L.orc_verts_per_cell(h)
        pts = np.empty((n, 3), np.float32)
        if n:
            C.memmove(pts.ctypes.data, L.orc_points(h), pts.nbytes)
        cells = np.empty((m, k), np.uint64)
        if m:
            C.memmove(cells.ctypes.data, L.orc_cells(h), cells.nbytes)
        cd = None
        if cell_data:
            cd = np.empty(m, vol.dtype)
            if m:
                assert L.orc_cell_data_bytes(h) == cd.nbytes
                C.memmove(cd.ctypes.data, L.orc_cell_data(h), cd.nbytes)
        return O.Mesh(pts, cells, cd, L.orc_step_length_used(h))
    finally:
        L.orc_free(h)


def classify(vol: np.ndarray, iso, words_per_row: int | None = None) -> np.ndarray:
    O = oracle()
    if vol.dtype not in CODES:
        return O.classify(vol, iso, words_per_row)
    dims, _, _ = O._geom(vol, None, None)
    wpr = words_per_row or (vol.shape[2] + 31) // 32
    out = np.zeros((vol.shape[0], vol.shape[1], wpr), np.uint32)
    assert lib().orc64_classify(vol.ctypes.data, CODES[vol.dtype], dims, float(iso), out.ctypes.data, wpr) == 0
    return out


def project_points(vol: np.ndarray, iso, pts: np.ndarray, *, thr=0.5, step=-1.0, relax=0.95, max_steps=50,
                   spacing=None, origin=None, direction=None, method=0) -> np.ndarray:
    O = oracle()
    if vol.dtype not in CODES:
        return O.project_points(vol, iso, pts, thr=thr, step=step, relax=relax, max_steps=max_steps, spacing=spacing,
                                origin=origin, direction=direction, method=method)
    dims, sp, og = O._geom(vol, spacing, origin)
    P = O._params(iso, True, True, False, O.LITERAL, thr, step, relax, max_steps, direction=direction, method=method)
    out = np.ascontiguousarray(pts, np.float32).copy()
    assert lib().orc64_project_points(vol.ctypes.data, CODES[vol.dtype], dims, sp, og, C.byref(P), out.ctypes.data,
                                      out.shape[0]) == 0
    return out


def sample(vol: np.ndarray, pts: np.ndarray, spacing=None, origin=None):
    O = oracle()
    if vol.dtype not in CODES:
        return O.sample(vol, pts, spacing, origin)
    dims, sp, og = O._geom(vol, spacing, origin)
    p = np.ascontiguousarray(pts, np.float64)
    val = np.empty(p.shape[0], np.float64)
    grad = np.empty((p.shape[0], 3), np.float64)
    assert lib().orc64_sample(vol.ctypes.data, CODES[vol.dtype], dims, sp, og, p.ctypes.data, p.shape[0],
                              val.ctypes.data, grad.ctypes.data) == 0
    return val, grad
