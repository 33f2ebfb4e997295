"""ORACLE (test infrastructure): ctypes front-end of ``mc_oracle.c`` plus the
reference's vertex rescale (surface_extractors.py:38-45, 74-75).  PARITY UNPINNED
for the marching-cubes arithmetic itself (see mc_oracle.c header)."""
from __future__ import annotations

import ctypes
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "_build", "libhy3d_mc_oracle.so")
_lib = None


def build(force: bool = False) -> str:
    src = os.path.join(_HERE, "mc_oracle.c")
    if force or not os.path.exists(_SO) or os.path.getmtime(_SO) < os.path.getmtime(src):
        subprocess.check_call(["make", "-s", "-C", _HERE, "_build/libhy3d_mc_oracle.so"])
    return _SO


def _load():
    global _lib
    if _lib is None:
        build()
        lib = ctypes.CDLL(_SO)
        lib.hy3d_oracle_mc.restype = ctypes.c_int
        lib.hy3d_oracle_mc.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_float,
                                       ctypes.POINTER(ctypes.c_void_p), ctypes.POINTER(ctypes.c_int64),
                                       ctypes.POINTER(ctypes.c_void_p), ctypes.POINTER(ctypes.c_int64)]
        lib.hy3d_oracle_free.argtypes = [ctypes.c_void_p]
        lib.hy3d_oracle_mc_cases.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                             ctypes.c_float, ctypes.c_void_p]
        _lib = lib
    return _lib


def marching_cubes(vol: np.ndarray, level: float = 0.0, method: str = "lewiner"):
    """Same call shape as ``skimage.measure.marching_cubes``: returns
    ``(verts[V,3] float32 in index units, faces[F,3] int32, normals=None, values=None)``.
    Raises like skimage does: ValueError when ``level`` is outside the data range
    (NaN in the volume disables the check), RuntimeError when no surface results."""
    vol = np.ascontiguousarray(vol, dtype=np.float32)
    if vol.ndim != 3:
        raise ValueError("Input volume should be a 3D numpy array.")
    if level < vol.min() or level > vol.max():
        raise ValueError("Surface level must be within volume data range.")
    verts, faces = marching_cubes_raw(vol, level)
    if len(faces) == 0:
        raise RuntimeError("No surface found at the given iso value.")
    return verts, faces, None, None


def marching_cubes_raw(vol: np.ndarray, level: float = 0.0):
    """``marching_cubes`` without skimage's argument checks: ``(verts[V,3] float32 in index units, faces[F,3] int32)``,
    empty arrays when nothing crosses ``level`` — the form ``hy3d_mc_count`` / ``hy3d_mc_emit`` return with a unit
    transform."""
    lib = _load()
    pv, pf, nv, nf = ctypes.c_void_p(), ctypes.c_void_p(), ctypes.c_int64(), ctypes.c_int64()
    vol = np.ascontiguousarray(vol, np.float32)
    rc = lib.hy3d_oracle_mc(vol.ctypes.data, *vol.shape, float(level), ctypes.byref(pv), ctypes.byref(nv), ctypes.byref(pf),
                            ctypes.byref(nf))
    if rc != 0:
        raise MemoryError("oracle marching cubes")
    V, Fc = nv.value, nf.value
    verts = np.ctypeslib.as_array(ctypes.cast(pv, ctypes.POINTER(ctypes.c_float)), shape=(max(V, 1), 3))[:V].copy()
    faces = np.ctypeslib.as_array(ctypes.cast(pf, ctypes.POINTER(ctypes.c_int32)), shape=(max(Fc, 1), 3))[:Fc].copy()
    lib.hy3d_oracle_free(pv)
    lib.hy3d_oracle_free(pf)
    return verts, faces


def cube_cases(vol: np.ndarray, level: float = 0.0) -> np.ndarray:
    vol = np.ascontiguousarray(vol, dtype=np.float32)
    out = np.empty(tuple(s - 1 for s in vol.shape), dtype=np.uint8)
    _load().hy3d_oracle_mc_cases(vol.ctypes.data, vol.shape[0], vol.shape[1], vol.shape[2], float(level),
                                 out.ctypes.data)
    return out


def mc_surface_extract(grid_logit: np.ndarray, *, mc_level, bounds, octree_resolution):
    """``MCSurfaceExtractor.run`` (surface_extractors.py:68-76): marching cubes then
    ``v / (res+1) * bbox_size + bbox_min`` in float64 (numpy promotion: float32
    verts / int list -> float64), cast to float32 by the caller (:55)."""
    verts, faces, _, _ = marching_cubes(grid_logit, mc_level, method="lewiner")
    if isinstance(bounds, float):
        bounds = [-bounds, -bounds, -bounds, bounds, bounds, bounds]
    bbox_min, bbox_max = np.array(bounds[0:3]), np.array(bounds[3:6])
    bbox_size = bbox_max - bbox_min
    grid_size = [int(octree_resolution) + 1] * 3
    verts = verts / grid_size * bbox_size + bbox_min
    return verts.astype(np.float32), np.ascontiguousarray(faces)
