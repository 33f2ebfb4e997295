"""hy3dgeo — B200-native (sm_100a) geometry decoding for Hunyuan3D-2.

Drop-in replacements for the reference's ``volume_decoder`` / ``surface_extractor``
plugin slots (reference hy3dgen/shapegen/models/autoencoders/model.py:92-110)
and for the ``FloaterRemover`` / ``DegenerateFaceRemover`` mesh filters
(reference hy3dgen/shapegen/postprocessors.py; ``FaceReducer`` is ``hy3dgeo.postprocessors.FaceReducer``), backed by hand-written CUDA kernels behind the C-ABI declared in
``include/hy3dgeo.h``.  There is no CPU fallback: every compute entry point
raises if ``libhy3dgeo.so`` is missing.
"""
from . import weights, utils, _lib, volume_decoders, surface_extractors, model, postprocessors  # noqa: F401
from .model import B200ShapeVAE, GeoDecoder, install, enable_flashvdm_decoder  # noqa: F401
from .postprocessors import DegenerateFaceRemover, FloaterRemover  # noqa: F401
from .surface_extractors import (DMCSurfaceExtractor, Latent2MeshOutput, MCSurfaceExtractor,  # noqa: F401
                                 SurfaceExtractor, SurfaceExtractors, export_to_trimesh)
from .volume_decoders import (FlashVDMVolumeDecoding, HierarchicalVolumeDecoding,  # noqa: F401
                              VanillaVolumeDecoder)

__all__ = ["B200ShapeVAE", "GeoDecoder", "install", "enable_flashvdm_decoder", "VanillaVolumeDecoder",
           "HierarchicalVolumeDecoding", "FlashVDMVolumeDecoding", "MCSurfaceExtractor", "DMCSurfaceExtractor",
           "SurfaceExtractor", "SurfaceExtractors", "Latent2MeshOutput", "export_to_trimesh", "FloaterRemover",
           "DegenerateFaceRemover"]
