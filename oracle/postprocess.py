"""ORACLE (test infrastructure, never shipped): numpy statement of the two mesh filters of the reference's
``hy3dgen/shapegen/postprocessors.py`` that ``hy3dgeo.FloaterRemover`` / ``hy3dgeo.DegenerateFaceRemover`` and
``hy3d_mesh_remove_floaters`` / ``hy3d_mesh_weld`` implement on the GPU.

PARITY UNPINNED: the reference builds both on pymeshlab (and ``DegenerateFaceRemover`` on a save / load round trip
through pymeshlab and trimesh), none of which is available here, and the reference holds no vector at this boundary.  What
follows is the project's own restatement of the filters' intent, and this module is the contract the kernels are tested
against bit for bit.

Floater removal (pymeshlab ``compute_selection_by_small_disconnected_components_per_face(nbfaceratio=0.005)``, then
``compute_selection_transfer_face_to_vertex(inclusive=False)``, then ``meshing_remove_selected_vertices_and_faces``):
  * two faces are adjacent iff they share an undirected edge {a, b} with a != b; an edge may have any number of faces
    (VCG's face-face adjacency); components are the connected classes of that relation;
  * ``min_faces = int(0.005 * F)`` (float64 product, truncated); a component is small iff it has fewer than min_faces faces;
  * a vertex is selected iff a face of a small component uses it; a face is removed iff any of its vertices is selected
    (so faces of a large component touching a floater at a shared vertex go too).

Degenerate-face removal (the intent of the reference's round trip on a marching-cubes mesh: weld coincident vertices and
drop the faces that collapse):
  * weld key = the three float32 bit patterns, -0.0 taken as +0.0; a vertex with a non-finite coordinate is never merged;
  * every vertex is replaced by the smallest vertex id with the same key; a face with two equal ids is then removed;
  * not done: faces with three distinct collinear vertices and duplicate faces are kept; trimesh's 1e-8 rounding merge is
    not reproduced (only bit-equal positions merge).

Both end in the compaction of ``oracle/mesh.py``: surviving faces keep their order and winding and are re-indexed,
vertices are kept iff a surviving face references them, in their original order.
"""
from __future__ import annotations

import numpy as np
from scipy.sparse import coo_matrix
from scipy.sparse.csgraph import connected_components

NBFACERATIO = 0.005


def min_faces_for(num_faces: int, ratio: float = NBFACERATIO) -> int:
    return int(float(ratio) * int(num_faces))


def _compact(v: np.ndarray, f: np.ndarray, keep_f: np.ndarray):
    f = f[keep_f]
    ref = np.zeros(len(v), dtype=bool)
    ref[f.reshape(-1)] = True
    remap = np.cumsum(ref) - 1
    return np.ascontiguousarray(v[ref]), np.ascontiguousarray(remap[f].astype(np.int32).reshape(-1, 3))


def edge_components(f: np.ndarray) -> np.ndarray:
    """Component label of every face, faces joined iff they share an undirected edge {a, b}, a != b."""
    f = np.asarray(f, dtype=np.int64).reshape(-1, 3)
    F = len(f)
    if F == 0:
        return np.zeros(0, dtype=np.int64)
    a = f[:, [0, 1, 2]].reshape(-1)
    b = f[:, [1, 2, 0]].reshape(-1)
    face = np.repeat(np.arange(F), 3)
    ok = a != b
    lo, hi, face = np.minimum(a, b)[ok], np.maximum(a, b)[ok], face[ok]
    _, edge = np.unique(lo * (int(f.max()) + 1) + hi, return_inverse=True)
    # bipartite graph: face nodes [0, F), edge nodes [F, F + E)
    n = F + (int(edge.max()) + 1 if len(edge) else 0)
    g = coo_matrix((np.ones(len(face), dtype=np.int8), (face, F + edge.reshape(-1))), shape=(n, n))
    _, labels = connected_components(g, directed=False)
    return labels[:F]


def vertex_components(f: np.ndarray, num_verts: int) -> int:
    """Number of components when faces are joined by a shared vertex (the relation the floater filter does NOT use)."""
    f = np.asarray(f, dtype=np.int64).reshape(-1, 3)
    F = len(f)
    g = coo_matrix((np.ones(3 * F, dtype=np.int8), (np.repeat(np.arange(F), 3), F + f.reshape(-1))),
                   shape=(F + num_verts, F + num_verts))
    _, labels = connected_components(g, directed=False)
    return len(np.unique(labels[:F]))


def remove_floaters(v: np.ndarray, f: np.ndarray, min_faces: int | None = None):
    """FloaterRemover: -> (vertices, faces) without the small edge-connected components and the faces touching them."""
    v, f = np.asarray(v), np.asarray(f).reshape(-1, 3)
    if min_faces is None:
        min_faces = min_faces_for(len(f))
    labels = edge_components(f)
    size = np.bincount(labels, minlength=1) if len(labels) else np.zeros(0, np.int64)
    small = size[labels] < min_faces
    sel = np.zeros(len(v), dtype=bool)
    sel[f[small].reshape(-1)] = True
    return _compact(v, f, ~sel[f].any(axis=1))


def weld_representatives(v: np.ndarray) -> np.ndarray:
    """Smallest vertex id with the same weld key, per vertex (non-finite vertices: themselves)."""
    v = np.ascontiguousarray(v, dtype=np.float32).reshape(-1, 3)
    bits = v.view(np.uint32).copy()
    bits[bits == 0x80000000] = 0
    finite = np.isfinite(v).all(axis=1)
    rep = np.arange(len(v), dtype=np.int64)
    idx = np.nonzero(finite)[0]
    if len(idx):
        _, first, inv = np.unique(bits[idx], axis=0, return_index=True, return_inverse=True)
        rep[idx] = idx[first][inv.reshape(-1)]                  # np.unique's first occurrence = smallest id of the key
    return rep


def weld(v: np.ndarray, f: np.ndarray):
    """DegenerateFaceRemover: -> (vertices, faces) with bit-equal vertices merged and collapsed faces removed."""
    v, f = np.asarray(v), np.asarray(f).reshape(-1, 3)
    g = weld_representatives(v)[f]
    keep = (g[:, 0] != g[:, 1]) & (g[:, 1] != g[:, 2]) & (g[:, 0] != g[:, 2])
    return _compact(v, g, keep)
