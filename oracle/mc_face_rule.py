"""ORACLE (test infrastructure): ctypes front-end of ``mc_face_rule.c`` -- marching cubes with ``face_rule`` "sign"
(exactly ``oracle.mc``) or "asymptotic" (Lewiner's face test on ambiguous faces), plus the reference's vertex rescale.
Same call shapes as ``oracle.mc``."""
from __future__ import annotations

import ctypes
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "_build", "libhy3d_mc_face_rule_oracle.so")
_SRCS = [os.path.join(_HERE, "mc_face_rule.c"), os.path.join(_HERE, "mc_oracle.c")]
FACE_RULES = {"sign": 0, "asymptotic": 1}
_lib = None


def build(force: bool = False) -> str:
    """Compiles the library into oracle/_build (flags of oracle/Makefile) when it is missing or older than its sources."""
    if force or not os.path.exists(_SO) or os.path.getmtime(_SO) < max(os.path.getmtime(s) for s in _SRCS):
        os.makedirs(os.path.dirname(_SO), exist_ok=True)
        subprocess.check_call([os.environ.get("CC", "gcc"), "-O2", "-fPIC", "-shared", "-ffp-contract=off", "-std=c11",
                               "-Wall", "-o", _SO, _SRCS[0], "-lm"])
    return _SO


def _load():
    global _lib
    if _lib is None:
        build()
        lib = ctypes.CDLL(_SO)
        lib.hy3d_oracle_mc_rule.restype = ctypes.c_int
        lib.hy3d_oracle_mc_rule.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_float,
                                            ctypes.c_int, ctypes.POINTER(ctypes.c_void_p), ctypes.POINTER(ctypes.c_int64),
                                            ctypes.POINTER(ctypes.c_void_p), ctypes.POINTER(ctypes.c_int64)]
        lib.hy3d_oracle_cube_triangles.restype = ctypes.c_int
        lib.hy3d_oracle_cube_triangles.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.c_void_p]
        lib.hy3d_oracle_free.argtypes = [ctypes.c_void_p]
        _lib = lib
    return _lib


def marching_cubes_raw(vol: np.ndarray, level: float = 0.0, face_rule: str = "sign"):
    """``oracle.mc.marching_cubes_raw`` under ``face_rule``: ``(verts[V,3] float32 in index units, faces[F,3] int32)``."""
    lib = _load()
    pv, pf, nv, nf = ctypes.c_void_p(), ctypes.c_void_p(), ctypes.c_int64(), ctypes.c_int64()
    vol = np.ascontiguousarray(vol, np.float32)
    if vol.ndim != 3:
        raise ValueError("Input volume should be a 3D numpy array.")
    rc = lib.hy3d_oracle_mc_rule(vol.ctypes.data, *vol.shape, float(level), FACE_RULES[face_rule], ctypes.byref(pv),
                                 ctypes.byref(nv), ctypes.byref(pf), ctypes.byref(nf))
    if rc != 0:
        raise MemoryError("oracle marching cubes")
    V, Fc = nv.value, nf.value
    verts = np.ctypeslib.as_array(ctypes.cast(pv, ctypes.POINTER(ctypes.c_float)), shape=(max(V, 1), 3))[:V].copy()
    faces = np.ctypeslib.as_array(ctypes.cast(pf, ctypes.POINTER(ctypes.c_int32)), shape=(max(Fc, 1), 3))[:Fc].copy()
    lib.hy3d_oracle_free(pv)
    lib.hy3d_oracle_free(pf)
    return verts, faces


def marching_cubes(vol: np.ndarray, level: float = 0.0, method: str = "lewiner", face_rule: str = "sign"):
    """``oracle.mc.marching_cubes`` (skimage's call shape and errors) under ``face_rule``."""
    vol = np.ascontiguousarray(vol, dtype=np.float32)
    if vol.ndim != 3:
        raise ValueError("Input volume should be a 3D numpy array.")
    if level < vol.min() or level > vol.max():
        raise ValueError("Surface level must be within volume data range.")
    verts, faces = marching_cubes_raw(vol, level, face_rule)
    if len(faces) == 0:
        raise RuntimeError("No surface found at the given iso value.")
    return verts, faces, None, None


def mc_surface_extract(grid_logit: np.ndarray, *, mc_level, bounds, octree_resolution, face_rule: str = "sign"):
    """``oracle.mc.mc_surface_extract`` under ``face_rule``: marching cubes, then ``v / (res+1) * bbox_size + bbox_min``
    in float64, cast to float32."""
    verts, faces, _, _ = marching_cubes(grid_logit, mc_level, face_rule=face_rule)
    if isinstance(bounds, float):
        bounds = [-bounds, -bounds, -bounds, bounds, bounds, bounds]
    bbox_min, bbox_max = np.array(bounds[0:3]), np.array(bounds[3:6])
    grid_size = [int(octree_resolution) + 1] * 3
    verts = verts / grid_size * (bbox_max - bbox_min) + bbox_min
    return verts.astype(np.float32), np.ascontiguousarray(faces)


def cube_triangles(case: int, connect: int) -> np.ndarray:
    """Triangles (edge ids, [n,3] int32) the oracle traces for one cube case; bit f of ``connect``: ambiguous face f
    (``FACE`` order of mc_oracle.c) connects its inside corners."""
    tri = np.empty((10, 3), np.int32)
    n = _load().hy3d_oracle_cube_triangles(int(case), int(connect), tri.ctypes.data)
    return tri[:n].copy()

