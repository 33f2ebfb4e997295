"""Mesh post-processing on the GPU — ``FloaterRemover``, ``DegenerateFaceRemover`` and ``FaceReducer`` of the reference's
``hy3dgen/shapegen/postprocessors.py``, which every Hunyuan3D-2 front end runs on the mesh ``latents2mesh`` returns::

    mesh = FloaterRemover()(mesh)
    mesh = DegenerateFaceRemover()(mesh)
    mesh = FaceReducer()(mesh)          # max_facenum=40000

The reference builds all three on pymeshlab (CPU).  Here they are ``hy3d_mesh_remove_floaters`` / ``hy3d_mesh_weld`` /
``hy3d_mesh_decimate`` of ``libhy3dgeo.so``; the contracts they meet bit for bit are ``oracle/postprocess.py`` and
``oracle/decimate.py`` (DESIGN.md §2: parity with pymeshlab is unpinned).  ``FaceReducer`` keeps boundaries exactly,
never lets a face flip, and collapses edges in rounds of independent collapses instead of one heap.

Each class takes a ``Latent2MeshOutput`` (returns a new one holding float32 / int32 numpy arrays) or a ``trimesh.Trimesh``
(returns ``trimesh.Trimesh(..., process=False)``); the input is never modified.  Positions are processed in float32.
Anything else — a path, a pymeshlab ``MeshSet`` — raises ``TypeError``.  There is no CPU path: without a CUDA device the
call raises ``RuntimeError``.  ``run_device(verts, faces)`` works on CUDA tensors, so the three filters chain without the
mesh crossing PCIe in between.
"""
from __future__ import annotations

import numpy as np
import torch

from . import utils
from ._lib import get_context
from .surface_extractors import Latent2MeshOutput, _to_host

NBFACERATIO = 0.005          # compute_selection_by_small_disconnected_components_per_face(nbfaceratio=0.005)


def _check_device_mesh(verts, faces):
    if not (isinstance(verts, torch.Tensor) and isinstance(faces, torch.Tensor) and verts.is_cuda and faces.is_cuda):
        raise TypeError("run_device takes CUDA tensors verts [V, 3] and faces [F, 3] (hy3dgeo has no CPU path)")


def _apply(mesh, run_device):
    """Host mesh -> device -> ``run_device`` -> host mesh of the same kind."""
    try:
        import trimesh
    except ImportError:
        trimesh = None
    if isinstance(mesh, Latent2MeshOutput):
        v, f = mesh.mesh_v, mesh.mesh_f
    elif trimesh is not None and isinstance(mesh, trimesh.Trimesh):
        v, f = mesh.vertices, mesh.faces
    else:
        raise TypeError(f"expected a Latent2MeshOutput or a trimesh.Trimesh, got {type(mesh).__name__}")
    if not torch.cuda.is_available():
        raise RuntimeError("hy3dgeo runs on CUDA devices only (no CPU fallback)")
    dev = torch.device("cuda", torch.cuda.current_device())
    vd = torch.from_numpy(np.ascontiguousarray(v, dtype=np.float32)).to(dev, non_blocking=True)
    fd = torch.from_numpy(np.ascontiguousarray(f, dtype=np.int32)).to(dev, non_blocking=True)
    vo, fo = _to_host(*run_device(vd, fd))
    if isinstance(mesh, Latent2MeshOutput):
        return Latent2MeshOutput(mesh_v=vo, mesh_f=fo)
    return trimesh.Trimesh(vo, fo, process=False)


class FloaterRemover:
    """Removes the connected components of fewer than ``int(0.005 * F)`` faces (faces connected through shared edges), and
    every face that touches one of their vertices; unreferenced vertices are dropped, the order of the survivors is kept."""

    @utils.synchronize_timer('FloaterRemover')
    def __call__(self, mesh):
        return _apply(mesh, self.run_device)

    def run_device(self, verts: torch.Tensor, faces: torch.Tensor):
        """CUDA tensors (verts float32 [V, 3], faces int32 [F, 3]) -> the filtered mesh as device tensors."""
        _check_device_mesh(verts, faces)
        min_faces = int(NBFACERATIO * int(faces.shape[0]))
        return get_context(verts.device).mesh_remove_floaters(verts, faces, min_faces)


class DegenerateFaceRemover:
    """Welds vertices at bit-equal positions (``-0.0 == +0.0``; NaN / inf vertices are never merged) into the smallest vertex
    id and removes the faces that collapse; unreferenced vertices are dropped, the order of the survivors is kept.  Faces
    with three distinct collinear vertices and duplicate faces are kept, and there is no distance tolerance."""

    @utils.synchronize_timer('DegenerateFaceRemover')
    def __call__(self, mesh):
        return _apply(mesh, self.run_device)

    def run_device(self, verts: torch.Tensor, faces: torch.Tensor):
        """CUDA tensors (verts float32 [V, 3], faces int32 [F, 3]) -> the welded mesh as device tensors."""
        _check_device_mesh(verts, faces)
        return get_context(verts.device).mesh_weld(verts, faces)


class FaceReducer:
    """Quadric edge-collapse decimation to ``max_facenum`` faces (the result has ``max_facenum - 1`` or ``max_facenum``
    faces, more only when no valid collapse is left); a mesh with no more than ``max_facenum`` faces is returned as given.
    Boundary and non-manifold vertices never move, collapses that would flip a face or change the topology are refused,
    and the order of the surviving vertices and faces is kept (hy3dgeo.h: hy3d_mesh_decimate)."""

    @utils.synchronize_timer('FaceReducer')
    def __call__(self, mesh, max_facenum: int = 40000):
        _check_max_facenum(max_facenum)
        return _apply(mesh, lambda v, f: self.run_device(v, f, max_facenum))

    def run_device(self, verts: torch.Tensor, faces: torch.Tensor, max_facenum: int = 40000):
        """CUDA tensors (verts float32 [V, 3], faces int32 [F, 3]) -> the decimated mesh as device tensors."""
        _check_device_mesh(verts, faces)
        _check_max_facenum(max_facenum)
        return get_context(verts.device).mesh_decimate(verts, faces, int(max_facenum))[:2]


def _check_max_facenum(max_facenum):
    if int(max_facenum) < 1:
        raise ValueError(f"max_facenum must be >= 1, got {max_facenum}")
