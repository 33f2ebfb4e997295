"""Mesh post-processing on the GPU — ``FloaterRemover`` and ``DegenerateFaceRemover`` of the reference's
``hy3dgen/shapegen/postprocessors.py``, which every Hunyuan3D-2 front end runs on the mesh ``latents2mesh`` returns::

    mesh = FloaterRemover()(mesh)
    mesh = DegenerateFaceRemover()(mesh)

The reference builds both on pymeshlab (CPU).  Here they are ``hy3d_mesh_remove_floaters`` / ``hy3d_mesh_weld`` of
``libhy3dgeo.so``; the contract they meet bit for bit is ``oracle/postprocess.py`` (DESIGN.md §2: parity with pymeshlab is
unpinned).  ``FaceReducer`` (quadric edge-collapse decimation) is not provided: keep pymeshlab's.

Each class takes a ``Latent2MeshOutput`` (returns a new one holding float32 / int32 numpy arrays) or a ``trimesh.Trimesh``
(returns ``trimesh.Trimesh(..., process=False)``); the input is never modified.  Positions are processed in float32.
Anything else — a path, a pymeshlab ``MeshSet`` — raises ``TypeError``.  There is no CPU path: without a CUDA device the
call raises ``RuntimeError``.  ``run_device(verts, faces)`` works on CUDA tensors, so the two filters chain without the mesh
crossing PCIe in between.
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
