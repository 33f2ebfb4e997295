"""ORACLE (test infrastructure, never shipped): numpy restatement of what the step right after the hot path does to the
mesh — ``export_to_trimesh`` (reference hy3dgen/shapegen/pipelines.py:95-110):

    mesh.mesh_f = mesh.mesh_f[:, ::-1]
    trimesh.Trimesh(mesh.mesh_v, mesh.mesh_f)            # process=True

PARITY UNPINNED: ``trimesh`` is an un-vendored, un-pinned dependency (requirements.txt lists it without a version; it is
absent from /root/reference, this image and the wheelhouse) and the reference holds no vector at this boundary.  What is
restated is the published behaviour of ``Trimesh.process`` relevant to a marching-cubes mesh with NaN vertices:
``remove_infinite_values`` drops every face that references a non-finite vertex and then those vertices, and
``merge_vertices`` keeps only referenced vertices; both preserve the order of the survivors and re-index the faces.
(``merge_vertices`` also merges vertices closer than 1e-8: not restated — a welded marching-cubes mesh has none except
where a grid value equals the iso level exactly.)
"""
from __future__ import annotations

import numpy as np


def bits_equal(a: np.ndarray, b: np.ndarray) -> bool:
    """Same shape and the same float32 bit patterns (NaN payloads included)."""
    return a.shape == b.shape and np.array_equal(a.view(np.uint32), b.view(np.uint32))


def assert_same_mesh(got, ref):
    """(verts, faces) pairs: identical faces; vertices NaN at the same places and bit-identical elsewhere (the NaN payload
    of a vertex interpolated from a NaN sample is not part of the contract)."""
    (v, f), (vo, fo) = got, ref
    assert v.shape == vo.shape and np.array_equal(f, fo)
    nan = np.isnan(v)
    assert np.array_equal(nan, np.isnan(vo))
    assert np.array_equal(v[~nan].view(np.uint32), vo[~nan].view(np.uint32))


def export_clean(mesh_v: np.ndarray, mesh_f: np.ndarray, flip_winding: bool = True):
    v = np.asarray(mesh_v)
    f = np.asarray(mesh_f)
    if flip_winding:
        f = f[:, ::-1]                                                   # pipelines.py:103
    finite_v = np.isfinite(v).all(axis=1)
    keep_f = finite_v[f].all(axis=1)                                     # remove_infinite_values: faces first
    f = f[keep_f]
    ref = np.zeros(len(v), dtype=bool)
    ref[f.reshape(-1)] = True                                            # merge_vertices: referenced vertices only
    remap = np.cumsum(ref) - 1
    return np.ascontiguousarray(v[ref]), np.ascontiguousarray(remap[f].astype(f.dtype))
