"""ctypes binding of ``libhy3dgeo.so`` (C-ABI in ``include/hy3dgeo.h``).

There is no fallback: if the shared library is missing or cannot be loaded, any
attempt to compute raises ``RuntimeError`` (build it with
``python -c "import __graft_entry__ as g; g.build()"`` or ``make -C hunyuan3d-2_b200/csrc``).
"""
from __future__ import annotations

import ctypes as C
import weakref
import os
import threading
from typing import Optional

import numpy as np
import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libhy3dgeo.so")

PRECISION_FP32_SIMT = 0
PRECISION_FP16_TC = 1

_lib = None
_lib_lock = threading.Lock()

c_f32p = C.c_void_p
c_i32p = C.c_void_p


class DecoderDesc(C.Structure):
    _fields_ = [(n, C.c_int32) for n in
                ("width", "heads", "mlp_ratio", "latent_width", "num_freqs", "include_pi", "ln_post", "qk_norm")] + \
               [(n, C.c_void_p) for n in
                ("query_proj_w", "query_proj_b", "latents_proj_w", "latents_proj_b",
                 "ln1_w", "ln1_b", "ln2_w", "ln2_b", "ln3_w", "ln3_b",
                 "c_q_w", "c_q_b", "c_kv_w", "c_kv_b", "c_proj_w", "c_proj_b",
                 "q_norm_w", "q_norm_b", "k_norm_w", "k_norm_b",
                 "c_fc_w", "c_fc_b", "mlp_proj_w", "mlp_proj_b",
                 "ln_post_w", "ln_post_b", "out_w", "out_b")]


class TransformerLayer(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in
                ("ln1_w", "ln1_b", "c_qkv_w", "c_qkv_b", "c_proj_w", "c_proj_b", "q_norm_w", "q_norm_b", "k_norm_w", "k_norm_b",
                 "ln2_w", "ln2_b", "c_fc_w", "c_fc_b", "mlp_proj_w", "mlp_proj_b")]


class TransformerDesc(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("width", "heads", "layers", "embed_dim", "qk_norm")] + \
               [("post_kl_w", C.c_void_p), ("post_kl_b", C.c_void_p), ("layer", C.POINTER(TransformerLayer))]


class Coords(C.Structure):
    _fields_ = [("mode", C.c_int32), ("cell", C.c_float * 3), ("bmin", C.c_float * 3),
                ("axis0", C.c_void_p), ("axis1", C.c_void_p), ("axis2", C.c_void_p)]


# name -> (restype, argtypes): every symbol declared in include/hy3dgeo.h
SYMBOLS = {
    "hy3d_create": (C.c_int, [C.c_int, C.c_void_p, C.POINTER(C.c_void_p)]),
    "hy3d_destroy": (None, [C.c_void_p]),
    "hy3d_set_stream": (C.c_int, [C.c_void_p, C.c_void_p]),
    "hy3d_last_error": (C.c_char_p, [C.c_void_p]),
    "hy3d_set_precision": (C.c_int, [C.c_void_p, C.c_int]),
    "hy3d_set_mc_face_rule": (C.c_int, [C.c_void_p, C.c_int]),
    "hy3d_launch_count": (C.c_int64, [C.c_void_p]),
    "hy3d_attention_info": (C.c_int, [C.c_void_p, C.POINTER(C.c_float), C.POINTER(C.c_int32), C.POINTER(C.c_float)]),
    "hy3d_set_decoder_weights": (C.c_int, [C.c_void_p, C.POINTER(DecoderDesc)]),
    "hy3d_set_transformer_weights": (C.c_int, [C.c_void_p, C.POINTER(TransformerDesc)]),
    "hy3d_transformer_forward": (C.c_int, [C.c_void_p, c_f32p, C.c_int32, c_f32p]),
    "hy3d_transformer_begin": (C.c_int, [C.c_void_p, c_f32p, C.c_int32, C.c_int32, C.c_int32]),
    "hy3d_transformer_layer_kv": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p]),
    "hy3d_transformer_layer_rest": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p]),
    "hy3d_transformer_end": (C.c_int, [C.c_void_p, c_f32p]),
    "hy3d_prepare_kv": (C.c_int, [C.c_void_p, c_f32p, C.c_int32]),
    "hy3d_decode_points": (C.c_int, [C.c_void_p, c_f32p, C.c_int64, c_f32p]),
    "hy3d_decode_dense": (C.c_int, [C.c_void_p, c_f32p, c_f32p, c_f32p, C.c_int32, C.c_int32, C.c_int32,
                                    C.c_int64, C.c_int64, c_f32p]),
    "hy3d_decode_list": (C.c_int, [C.c_void_p, c_i32p, C.c_int64, C.c_int32, C.c_int32, C.c_int32,
                                   C.POINTER(C.c_float), C.POINTER(C.c_float), c_f32p]),
    "hy3d_decode_list_values": (C.c_int, [C.c_void_p, c_i32p, C.c_int64, C.c_int32, C.c_int32, C.c_int32,
                                          C.POINTER(C.c_float), C.POINTER(C.c_float), c_f32p]),
    "hy3d_scatter": (C.c_int, [C.c_void_p, c_i32p, c_f32p, C.c_int64, C.c_int64, c_f32p]),
    "hy3d_scatter_window": (C.c_int, [C.c_void_p, c_i32p, c_f32p, C.c_int64, C.c_int64, C.c_int64, c_f32p]),
    "hy3d_flash_select": (C.c_int, [C.c_void_p, c_i32p, C.c_int64, C.c_int32, C.c_int32, C.c_int32, C.POINTER(Coords),
                                    c_i32p, C.c_int32, C.c_int32, C.c_int32]),
    "hy3d_decode_flash": (C.c_int, [C.c_void_p, c_i32p, C.c_int64, C.c_int32, C.c_int32, C.c_int32, C.POINTER(Coords),
                                    c_i32p, c_f32p]),
    "hy3d_flash_select_range": (C.c_int, [C.c_void_p, c_i32p, C.c_int64, C.c_int32, C.c_int32, C.c_int32, C.POINTER(Coords),
                                          c_i32p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32]),
    "hy3d_decode_flash_values": (C.c_int, [C.c_void_p, c_i32p, C.c_int64, C.c_int32, C.c_int32, C.c_int32, C.POINTER(Coords),
                                           c_i32p, c_f32p]),
    "hy3d_flash_layout_bins": (C.c_int, [C.c_void_p, c_i32p, C.c_int64, C.c_int32, C.c_int32, C.c_int32, C.POINTER(Coords),
                                         C.c_int32, c_i32p, C.c_int64, c_i32p, c_i32p, C.c_int64, c_i32p, c_i32p]),
    "hy3d_flash_layout_minigrids": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, c_i32p, C.c_int64, c_i32p, c_i32p,
                                              C.c_int64, c_i32p]),
    "hy3d_flash_selection": (C.c_int, [C.c_void_p, c_i32p, C.c_int64]),
    "hy3d_flash_group_tokens": (C.c_int, [C.c_void_p, c_i32p, C.c_int32]),
    "hy3d_refine_level": (C.c_int, [C.c_void_p, c_f32p, C.c_int32, C.c_int32, C.c_float, C.c_int32, c_i32p, C.c_int64,
                                    C.POINTER(C.c_int64)]),
    "hy3d_fill": (C.c_int, [C.c_void_p, c_f32p, C.c_int64, C.c_float]),
    "hy3d_sentinel_to_nan": (C.c_int, [C.c_void_p, c_f32p, C.c_int64, C.c_float]),
    "hy3d_mc_count": (C.c_int, [C.c_void_p, c_f32p, C.c_int32, C.c_int32, C.c_int32, C.c_float,
                                C.POINTER(C.c_int64), C.POINTER(C.c_int64), C.POINTER(C.c_float)]),
    "hy3d_mc_emit": (C.c_int, [C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_double),
                               c_f32p, c_i32p]),
    "hy3d_mc_count_slab": (C.c_int, [C.c_void_p, c_f32p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_float,
                                     C.POINTER(C.c_int64), C.POINTER(C.c_int64), C.POINTER(C.c_float)]),
    "hy3d_mc_emit_slab": (C.c_int, [C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_double),
                                    C.c_int32, C.c_int64, c_f32p, c_i32p]),
    "hy3d_dmc_count": (C.c_int, [C.c_void_p, c_f32p, C.c_int32, C.c_int32, C.c_int32,
                                 C.POINTER(C.c_int64), C.POINTER(C.c_int64), C.POINTER(C.c_float)]),
    "hy3d_dmc_emit": (C.c_int, [C.c_void_p, c_f32p, c_i32p]),
    "hy3d_dmc_count_slab": (C.c_int, [C.c_void_p, c_f32p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                      C.POINTER(C.c_int64), C.POINTER(C.c_int64), C.POINTER(C.c_float)]),
    "hy3d_dmc_emit_slab": (C.c_int, [C.c_void_p, C.c_int64, c_f32p, c_i32p, c_i32p]),
    "hy3d_dmc_center": (C.c_int, [C.c_void_p, c_f32p, C.c_int64, C.POINTER(C.c_int32)]),
    "hy3d_mesh_clean": (C.c_int, [C.c_void_p, c_f32p, C.c_int64, c_i32p, C.c_int64, C.c_int32, c_f32p, c_i32p,
                                  C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "hy3d_mesh_remove_floaters": (C.c_int, [C.c_void_p, c_f32p, C.c_int64, c_i32p, C.c_int64, C.c_int64, c_f32p, c_i32p,
                                            C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "hy3d_mesh_weld": (C.c_int, [C.c_void_p, c_f32p, C.c_int64, c_i32p, C.c_int64, c_f32p, c_i32p,
                                 C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "hy3d_mesh_decimate": (C.c_int, [C.c_void_p, c_f32p, C.c_int64, c_i32p, C.c_int64, C.c_int64, c_f32p, c_i32p,
                                     C.POINTER(C.c_int64), C.POINTER(C.c_int64), C.POINTER(C.c_int32)]),
    "hy3d_profile": (C.c_int, [C.c_void_p, C.c_int]),
    "hy3d_profile_read": (C.c_int, [C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_int64)]),
    "hy3d_debug_watchdog": (C.c_int, [C.c_void_p, C.POINTER(C.c_int32)]),
    "hy3d_debug_force_online_softmax": (C.c_int, [C.c_void_p, C.c_int]),
    "hy3d_debug_attn_redo": (C.c_int, [C.c_void_p, C.POINTER(C.c_int32)]),
    "hy3d_mc_cases": (C.c_int, [C.c_void_p, c_f32p, C.c_int32, C.c_int32, C.c_int32, C.c_float, C.c_void_p]),
}


def load_library():
    """dlopen libhy3dgeo.so and type every exported symbol.  Loud on failure."""
    global _lib
    with _lib_lock:
        if _lib is None:
            if not os.path.exists(LIB_PATH):
                raise RuntimeError(
                    f"{LIB_PATH} not found: the CUDA extension is not built and there is no fallback. "
                    "Run `python -c 'import __graft_entry__ as g; g.build()'`.")
            lib = C.CDLL(LIB_PATH)
            for name, (res, args) in SYMBOLS.items():
                fn = getattr(lib, name)          # AttributeError if the .so lacks a declared symbol
                fn.restype = res
                fn.argtypes = args
            _lib = lib
    return _lib


# marching cubes, ambiguous faces (hy3dgeo.h hy3d_set_mc_face_rule): "sign" separates the inside corners, "asymptotic"
# decides from the four values as scikit-image's Lewiner face test does
MC_FACE_RULES = {"sign": 0, "asymptotic": 1}


class Hy3dError(RuntimeError):
    pass


def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else C.c_void_p(t.data_ptr())


class GeoContext:
    """One ``hy3d_ctx`` for one CUDA device.  Not thread-safe (one per thread and
    device, see ``get_context``).  All launches go to torch's current stream."""

    def __init__(self, device: torch.device):
        if device.type != "cuda":
            raise RuntimeError("hy3dgeo runs on CUDA devices only (no CPU fallback)")
        self.lib = load_library()
        self.device = torch.device("cuda", device.index if device.index is not None else torch.cuda.current_device())
        h = C.c_void_p()
        rc = self.lib.hy3d_create(self.device.index, self._stream(), C.byref(h))
        if rc != 0:
            raise Hy3dError(f"hy3d_create failed ({rc}): needs an sm_100 (B200) device")
        self.h = h
        self._weights_key = None
        self._kv_key = None
        self._keep = []        # tensors that must outlive async copies

    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def _check(self, rc: int, what: str):
        if rc != 0:
            msg = self.lib.hy3d_last_error(self.h)
            raise Hy3dError(f"{what} failed ({rc}): {msg.decode() if msg else ''}")

    def sync_stream(self):
        self._check(self.lib.hy3d_set_stream(self.h, self._stream()), "hy3d_set_stream")

    def close(self):
        if getattr(self, "h", None):
            self.lib.hy3d_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- decoder -----------------------------------------------------------------------------
    def set_precision(self, precision: int):
        self._check(self.lib.hy3d_set_precision(self.h, precision), "hy3d_set_precision")

    @property
    def launches(self) -> int:
        return int(self.lib.hy3d_launch_count(self.h))

    def attention_info(self):
        """(weight-only score bound, kernel name, measured score bound of the current K/V) of the decoder currently loaded."""
        b, f, m = C.c_float(), C.c_int32(), C.c_float()
        self._check(self.lib.hy3d_attention_info(self.h, C.byref(b), C.byref(f), C.byref(m)), "hy3d_attention_info")
        return float(b.value), ["online-softmax", "bounded-score", "bounded-score + per-head shift + exact redo"][f.value], float(m.value)

    @staticmethod
    def _same_owner(ref, owner) -> bool:
        """The cached weights belong to `owner` iff the weak reference taken when they were loaded is still alive
        and points at it.  id() / data_ptr() values alone are not identities: CPython and the caching allocator
        hand the same values to new objects once the old ones are freed."""
        return owner is not None and ref is not None and ref() is owner

    def has_decoder(self, key, owner) -> bool:
        """True when the decoder weights cached in this context were loaded from `owner` under the same `key`."""
        return key is not None and key == self._weights_key and self._same_owner(getattr(self, "_weights_owner", None), owner)

    def invalidate_weights(self):
        """Forget the cached decoder / transformer weights (after an edit through ``param.data``, which no key can see)."""
        self._weights_key = None
        self._tf_key = None

    def set_decoder(self, sd, cfg, key=None, owner=None):
        """sd: decoder state dict (keys without ``geo_decoder.``), cfg: ShapeVAEConfig.  `key` (+ the live `owner`
        object it was computed from) lets repeated calls with unchanged weights skip the upload."""
        if key is not None and key == self._weights_key and self._same_owner(getattr(self, "_weights_owner", None), owner):
            return
        self.sync_stream()
        dev = self.device

        def g(name):
            t = sd.get(name)
            if t is None:
                return None
            t = t.detach().to(device=dev, dtype=torch.float32).contiguous()
            self._keep.append(t)
            return t
        self._keep = []
        c = "cross_attn_decoder."
        d = DecoderDesc()
        d.width, d.heads = cfg.dec_width, cfg.dec_heads
        d.mlp_ratio, d.latent_width = cfg.geo_decoder_mlp_expand_ratio, cfg.width
        d.num_freqs, d.include_pi = cfg.num_freqs, int(cfg.include_pi)
        d.ln_post, d.qk_norm = int(cfg.geo_decoder_ln_post), int(cfg.dec_qk_norm)
        names = {
            "query_proj_w": "query_proj.weight", "query_proj_b": "query_proj.bias",
            "latents_proj_w": "latents_proj.weight", "latents_proj_b": "latents_proj.bias",
            "ln1_w": c + "ln_1.weight", "ln1_b": c + "ln_1.bias", "ln2_w": c + "ln_2.weight", "ln2_b": c + "ln_2.bias",
            "ln3_w": c + "ln_3.weight", "ln3_b": c + "ln_3.bias",
            "c_q_w": c + "attn.c_q.weight", "c_q_b": c + "attn.c_q.bias",
            "c_kv_w": c + "attn.c_kv.weight", "c_kv_b": c + "attn.c_kv.bias",
            "c_proj_w": c + "attn.c_proj.weight", "c_proj_b": c + "attn.c_proj.bias",
            "q_norm_w": c + "attn.attention.q_norm.weight", "q_norm_b": c + "attn.attention.q_norm.bias",
            "k_norm_w": c + "attn.attention.k_norm.weight", "k_norm_b": c + "attn.attention.k_norm.bias",
            "c_fc_w": c + "mlp.c_fc.weight", "c_fc_b": c + "mlp.c_fc.bias",
            "mlp_proj_w": c + "mlp.c_proj.weight", "mlp_proj_b": c + "mlp.c_proj.bias",
            "ln_post_w": "ln_post.weight", "ln_post_b": "ln_post.bias",
            "out_w": "output_proj.weight", "out_b": "output_proj.bias",
        }
        for field, name in names.items():
            t = g(name)
            setattr(d, field, None if t is None else t.data_ptr())
        self._check(self.lib.hy3d_set_decoder_weights(self.h, C.byref(d)), "hy3d_set_decoder_weights")
        torch.cuda.current_stream(self.device).synchronize()     # device->device copies done; staging may go
        self._keep = []
        self._weights_key = key
        self._weights_owner = weakref.ref(owner) if owner is not None else None
        self._kv_key = None

    def set_transformer(self, sd, cfg, key=None, owner=None):
        """sd: full ShapeVAE state dict (post_kl.*, transformer.resblocks.*), cfg: ShapeVAEConfig."""
        if key is not None and key == getattr(self, "_tf_key", None) and self._same_owner(getattr(self, "_tf_owner", None), owner):
            return
        self.sync_stream()
        keep = []

        def g(name):
            t = sd.get(name)
            if t is None:
                return None
            t = t.detach().to(device=self.device, dtype=torch.float32).contiguous()
            keep.append(t)
            return t.data_ptr()
        L = cfg.num_decoder_layers
        layers = (TransformerLayer * L)()
        names = {"ln1_w": "ln_1.weight", "ln1_b": "ln_1.bias", "c_qkv_w": "attn.c_qkv.weight", "c_qkv_b": "attn.c_qkv.bias",
                 "c_proj_w": "attn.c_proj.weight", "c_proj_b": "attn.c_proj.bias",
                 "q_norm_w": "attn.attention.q_norm.weight", "q_norm_b": "attn.attention.q_norm.bias",
                 "k_norm_w": "attn.attention.k_norm.weight", "k_norm_b": "attn.attention.k_norm.bias",
                 "ln2_w": "ln_2.weight", "ln2_b": "ln_2.bias", "c_fc_w": "mlp.c_fc.weight", "c_fc_b": "mlp.c_fc.bias",
                 "mlp_proj_w": "mlp.c_proj.weight", "mlp_proj_b": "mlp.c_proj.bias"}
        for l in range(L):
            for field, nm in names.items():
                setattr(layers[l], field, g(f"transformer.resblocks.{l}.{nm}"))
        d = TransformerDesc()
        d.width, d.heads, d.layers, d.embed_dim, d.qk_norm = cfg.width, cfg.heads, L, cfg.embed_dim, int(cfg.qk_norm)
        d.post_kl_w, d.post_kl_b = g("post_kl.weight"), g("post_kl.bias")
        d.layer = layers
        self._check(self.lib.hy3d_set_transformer_weights(self.h, C.byref(d)), "hy3d_set_transformer_weights")
        torch.cuda.current_stream(self.device).synchronize()
        self._tf_key = key
        self._tf_owner = weakref.ref(owner) if owner is not None else None
        self._tf_width = cfg.width

    def transformer_forward(self, z: torch.Tensor) -> torch.Tensor:
        """z: [M, embed_dim] -> latents [M, width] float32 (ShapeVAE.forward for one item)."""
        self.sync_stream()
        z = z.detach().to(device=self.device, dtype=torch.float32).contiguous()
        out = torch.empty((z.shape[0], self._tf_width), dtype=torch.float32, device=self.device)
        self._check(self.lib.hy3d_transformer_forward(self.h, _ptr(z), z.shape[0], _ptr(out)), "hy3d_transformer_forward")
        return out

    def transformer_forward_parallel(self, z: torch.Tensor, heads: int, layers: int, group=None) -> torch.Tensor:
        """Sequence-parallel ShapeVAE.forward for one item over a process group (see hy3dgeo.h): z [M, embed_dim] is known
        on every rank, rank r runs the rows [r M / world, (r+1) M / world); per layer the K / V tile images are all-gathered
        (NCCL), at the end the latent rows.  Returns the full latents [M, width] float32 on every rank."""
        import torch.distributed as dist
        self.sync_stream()
        world, rank = dist.get_world_size(group), dist.get_rank(group)
        M = z.shape[0]
        Ml = M // world
        if M % world or Ml % 128:
            raise ValueError(f"{M} tokens cannot be split into {world} parts that are multiples of 128")
        zl = z[rank * Ml:(rank + 1) * Ml].detach().to(device=self.device, dtype=torch.float32).contiguous()
        chunk = 2 * heads * (Ml // 128) * 16384
        kv = torch.empty(world * chunk, dtype=torch.uint8, device=self.device)
        staged = dist.get_backend(group) == "gloo"        # 2-process tests sharing one GPU: gloo moves host tensors only

        def gather_inplace(full, part):
            if not staged:
                dist.all_gather_into_tensor(full, part, group=group)
                return
            host = torch.empty(full.shape, dtype=full.dtype)
            dist.all_gather(list(host.view(world, -1).unbind(0)), part.reshape(-1).cpu(), group=group)
            full.copy_(host)
        self._check(self.lib.hy3d_transformer_begin(self.h, _ptr(zl), Ml, world, rank), "hy3d_transformer_begin")
        for l in range(layers):
            self._check(self.lib.hy3d_transformer_layer_kv(self.h, l, _ptr(kv)), "hy3d_transformer_layer_kv")
            gather_inplace(kv, kv[rank * chunk:(rank + 1) * chunk])
            self._check(self.lib.hy3d_transformer_layer_rest(self.h, l, _ptr(kv)), "hy3d_transformer_layer_rest")
        out = torch.empty((M, self._tf_width), dtype=torch.float32, device=self.device)
        mine = out[rank * Ml:(rank + 1) * Ml]
        self._check(self.lib.hy3d_transformer_end(self.h, _ptr(mine)), "hy3d_transformer_end")
        gather_inplace(out, mine)
        return out

    def prepare_kv(self, latents: torch.Tensor):
        """latents: [M, latent_width] on this device (any float dtype)."""
        self.sync_stream()
        lat = latents.detach().to(device=self.device, dtype=torch.float32).contiguous()
        self._check(self.lib.hy3d_prepare_kv(self.h, _ptr(lat), lat.shape[0]), "hy3d_prepare_kv")
        self._lat_keep = lat

    def decode_points(self, xyz: torch.Tensor) -> torch.Tensor:
        self.sync_stream()
        xyz = xyz.detach().to(device=self.device, dtype=torch.float32).contiguous().view(-1, 3)
        out = torch.empty(xyz.shape[0], dtype=torch.float32, device=self.device)
        self._check(self.lib.hy3d_decode_points(self.h, _ptr(xyz), xyz.shape[0], _ptr(out)), "hy3d_decode_points")
        return out

    def decode_dense(self, axes, first: int, count: int, out: torch.Tensor):
        """axes: three float32 numpy tables; out: float32 cuda tensor with >= count elements."""
        self.sync_stream()
        a = [np.ascontiguousarray(x, dtype=np.float32) for x in axes]
        self._check(self.lib.hy3d_decode_dense(self.h, a[0].ctypes.data, a[1].ctypes.data, a[2].ctypes.data,
                                               len(a[0]), len(a[1]), len(a[2]), first, count, _ptr(out)),
                    "hy3d_decode_dense")

    def decode_list(self, index: torch.Tensor, n: int, dims, cell, bmin, grid: torch.Tensor):
        self.sync_stream()
        cc = (C.c_float * 3)(*[float(v) for v in cell])
        bb = (C.c_float * 3)(*[float(v) for v in bmin])
        self._check(self.lib.hy3d_decode_list(self.h, _ptr(index), n, dims[0], dims[1], dims[2], cc, bb, _ptr(grid)),
                    "hy3d_decode_list")

    def watchdog(self):
        """Sync and return the tensor-path watchdog record (all zeros = healthy)."""
        out = (C.c_int32 * 8)()
        self._check(self.lib.hy3d_debug_watchdog(self.h, out), "hy3d_debug_watchdog")
        return list(out)

    FAMILIES = ["embed", "gemm_query_proj", "layernorm", "gemm_c_q", "attention", "gemm_c_proj", "gemm_c_fc",
                "gemm_mlp_proj", "head", "mc_bits", "mc_rowcount", "mc_scan", "mc_emit", "octree", "kv_prepare", "kv_select"]

    def profile(self, enable: bool):
        self._check(self.lib.hy3d_profile(self.h, int(enable)), "hy3d_profile")

    def profile_read(self):
        """{family: (total_ms, launches)} since the last read (device time, CUDA events)."""
        ms = (C.c_double * 16)()
        cnt = (C.c_int64 * 16)()
        self._check(self.lib.hy3d_profile_read(self.h, ms, cnt), "hy3d_profile_read")
        return {f: (ms[i], cnt[i]) for i, f in enumerate(self.FAMILIES)}

    def debug_force_online_softmax(self, enable: bool):
        """Run every attention launch of this context on the online-softmax kernel (tests use it as a reference)."""
        self._check(self.lib.hy3d_debug_force_online_softmax(self.h, int(enable)), "hy3d_debug_force_online_softmax")

    def debug_attn_redo(self) -> int:
        n = C.c_int32()
        self._check(self.lib.hy3d_debug_attn_redo(self.h, C.byref(n)), "hy3d_debug_attn_redo")
        return int(n.value)

    def check_watchdog(self):
        rec = self.watchdog()
        if rec[0]:
            raise Hy3dError(f"tcgen05 kernel barrier timeout: block {rec[1]} thread {rec[2]} bar 0x{rec[3]:x} parity {rec[4]}")

    def decode_list_values(self, index: torch.Tensor, dims, cell, bmin) -> torch.Tensor:
        self.sync_stream()
        index = index.contiguous()
        out = torch.empty(index.numel(), dtype=torch.float32, device=self.device)
        cc = (C.c_float * 3)(*[float(v) for v in cell])
        bb = (C.c_float * 3)(*[float(v) for v in bmin])
        self._check(self.lib.hy3d_decode_list_values(self.h, _ptr(index), index.numel(), dims[0], dims[1], dims[2], cc, bb,
                                                     _ptr(out)), "hy3d_decode_list_values")
        return out

    def scatter(self, index: torch.Tensor, values: torch.Tensor, grid: torch.Tensor, base: int = 0):
        """grid.flat[index[q] - base] = values[q] (``base`` = flat offset of a slab's first plane in the whole grid)."""
        self.sync_stream()
        self._check(self.lib.hy3d_scatter(self.h, _ptr(index.contiguous()), _ptr(values.contiguous()), index.numel(), int(base),
                                          _ptr(grid)), "hy3d_scatter")

    def scatter_window(self, index: torch.Tensor, values: torch.Tensor, grid: torch.Tensor, base: int):
        """grid.flat[index[q] - base] = values[q] for the entries with base <= index[q] < base + grid.numel(), the others
        skipped (a slab of a grid partitioned across GPUs, halo planes included)."""
        self.sync_stream()
        self._check(self.lib.hy3d_scatter_window(self.h, _ptr(index.contiguous()), _ptr(values.contiguous()), index.numel(),
                                                 int(base), grid.numel(), _ptr(grid)), "hy3d_scatter_window")

    # ---- FlashVDM ---------------------------------------------------------------------------
    @staticmethod
    def _coords(cell=None, bmin=None, axes=None):
        c = Coords()
        keep = []
        if axes is not None:
            c.mode = 3
            keep = [np.ascontiguousarray(a, dtype=np.float32) for a in axes]
            c.axis0, c.axis1, c.axis2 = (a.ctypes.data for a in keep)
        else:
            c.mode = 2
            c.cell = (C.c_float * 3)(*[float(v) for v in cell])
            c.bmin = (C.c_float * 3)(*[float(v) for v in bmin])
        return c, keep

    def flash_select(self, sample_index: torch.Tensor, dims, sample_off: torch.Tensor, n_groups: int, topk: int,
                     merge: bool, cell=None, bmin=None, axes=None):
        self.sync_stream()
        c, keep = self._coords(cell, bmin, axes)
        self._check(self.lib.hy3d_flash_select(self.h, _ptr(sample_index), sample_index.numel(), dims[0], dims[1], dims[2],
                                               C.byref(c), _ptr(sample_off), n_groups, topk, int(merge)), "hy3d_flash_select")

    def flash_select_range(self, sample_index: torch.Tensor, n_samples: int, dims, sample_off: torch.Tensor, n_groups: int,
                           g0: int, g1: int, topk: int, merge: bool, cell=None, bmin=None, axes=None):
        """``flash_select`` for groups [g0, g1) of a layout of ``n_groups``: ``sample_index`` = the layout's samples from
        entry sample_off[g0] on, ``n_samples`` = sample_off[g1] - sample_off[g0]; ``sample_off`` = the whole layout's."""
        self.sync_stream()
        c, keep = self._coords(cell, bmin, axes)
        self._check(self.lib.hy3d_flash_select_range(self.h, _ptr(sample_index), int(n_samples), dims[0], dims[1], dims[2],
                                                     C.byref(c), _ptr(sample_off), int(n_groups), int(g0), int(g1), topk,
                                                     int(merge)), "hy3d_flash_select_range")

    def decode_flash_values(self, index: torch.Tensor, dims, tile_group: torch.Tensor, cell=None, bmin=None,
                            axes=None) -> torch.Tensor:
        """Compact ``decode_flash``: logits of a 128-aligned slice of a padded layout (any value at padding entries)."""
        self.sync_stream()
        c, keep = self._coords(cell, bmin, axes)
        out = torch.empty(index.numel(), dtype=torch.float32, device=self.device)
        self._check(self.lib.hy3d_decode_flash_values(self.h, _ptr(index), index.numel(), dims[0], dims[1], dims[2], C.byref(c),
                                                      _ptr(tile_group), _ptr(out)), "hy3d_decode_flash_values")
        return out

    def decode_flash(self, index: torch.Tensor, dims, tile_group: torch.Tensor, grid: torch.Tensor, cell=None, bmin=None,
                     axes=None):
        self.sync_stream()
        c, keep = self._coords(cell, bmin, axes)
        self._check(self.lib.hy3d_decode_flash(self.h, _ptr(index), index.numel(), dims[0], dims[1], dims[2], C.byref(c),
                                               _ptr(tile_group), _ptr(grid)), "hy3d_decode_flash")

    def flash_layout_bins(self, index: torch.Tensor, dims, cell, bmin, stride: int, with_counts: bool = False):
        """Group-ordered, 128-padded layout of a refined level's active queries (6^3 spatial bins, stable):
        -> (pidx, tile_group, sidx, soff[, counts]), device int32; no host synchronisation."""
        self.sync_stream()
        nq = int(index.numel())
        cap = (nq + 216 * 127 + 127) // 128 * 128
        scap = (nq // stride + 216 + 127) // 128 * 128
        i32 = dict(dtype=torch.int32, device=self.device)
        pidx, tile_group = torch.empty(cap, **i32), torch.empty(cap // 128, **i32)
        sidx, soff = torch.empty(scap, **i32), torch.empty(217, **i32)
        counts = torch.empty(216, **i32) if with_counts else None
        c, keep = self._coords(cell, bmin, None)
        self._check(self.lib.hy3d_flash_layout_bins(self.h, _ptr(index), nq, dims[0], dims[1], dims[2], C.byref(c), int(stride),
                                                    _ptr(pidx), cap, _ptr(tile_group), _ptr(sidx), scap, _ptr(soff),
                                                    _ptr(counts)), "hy3d_flash_layout_bins")
        return (pidx, tile_group, sidx, soff, counts) if with_counts else (pidx, tile_group, sidx, soff)

    def flash_layout_minigrids(self, N: int, mini_grid_num: int, stride: int):
        """Level-0 layout: mini_grid_num^3 mini-grids of the [N]^3 grid -> (pidx, tile_group, sidx, soff)."""
        self.sync_stream()
        m, s = int(mini_grid_num), N // int(mini_grid_num)
        G, padc, nsamp = m ** 3, (s ** 3 + 127) // 128 * 128, (s ** 3 + stride - 1) // stride
        cap, scap = G * padc, (G * nsamp + 127) // 128 * 128
        i32 = dict(dtype=torch.int32, device=self.device)
        pidx, tile_group = torch.empty(cap, **i32), torch.empty(cap // 128, **i32)
        sidx, soff = torch.empty(scap, **i32), torch.empty(G + 1, **i32)
        self._check(self.lib.hy3d_flash_layout_minigrids(self.h, int(N), m, int(stride), _ptr(pidx), cap, _ptr(tile_group),
                                                         _ptr(sidx), scap, _ptr(soff)), "hy3d_flash_layout_minigrids")
        return pidx, tile_group, sidx, soff

    def flash_selection(self, count: int) -> torch.Tensor:
        out = torch.empty(count, dtype=torch.int32, device=self.device)
        self._check(self.lib.hy3d_flash_selection(self.h, _ptr(out), count), "hy3d_flash_selection")
        return out

    def flash_group_tokens(self, n_groups: int) -> torch.Tensor:
        out = torch.empty(n_groups, dtype=torch.int32, device=self.device)
        self._check(self.lib.hy3d_flash_group_tokens(self.h, _ptr(out), n_groups), "hy3d_flash_group_tokens")
        return out

    # ---- octree -------------------------------------------------------------------------------
    def refine_level(self, coarse: torch.Tensor, mc_level: float, last: bool, index: Optional[torch.Tensor],
                     nf: Optional[int] = None) -> int:
        """Active voxels of the fine grid [nf]^3 (default 2n-1; 2n when the level list came from an odd r // 2)."""
        self.sync_stream()
        n = coarse.shape[0]
        cnt = C.c_int64()
        cap = 0 if index is None else index.numel()
        self._check(self.lib.hy3d_refine_level(self.h, _ptr(coarse), n, 2 * n - 1 if nf is None else int(nf), float(mc_level),
                                               int(last), _ptr(index), cap, C.byref(cnt)), "hy3d_refine_level")
        return cnt.value

    def fill(self, grid: torch.Tensor, value: float):
        self.sync_stream()
        self._check(self.lib.hy3d_fill(self.h, _ptr(grid), grid.numel(), float(value)), "hy3d_fill")

    def sentinel_to_nan(self, grid: torch.Tensor, sentinel: float = -10000.0):
        self.sync_stream()
        self._check(self.lib.hy3d_sentinel_to_nan(self.h, _ptr(grid), grid.numel(), float(sentinel)),
                    "hy3d_sentinel_to_nan")

    # ---- marching cubes ------------------------------------------------------------------------
    def set_mc_face_rule(self, rule: str):
        """Ambiguous-face rule of the next count / emit pair, a name of MC_FACE_RULES (mc_count and mc_count_slab set it)."""
        if rule not in MC_FACE_RULES:
            raise ValueError(f"face_rule must be one of {sorted(MC_FACE_RULES)}, got {rule!r}")
        self._check(self.lib.hy3d_set_mc_face_rule(self.h, MC_FACE_RULES[rule]), "hy3d_set_mc_face_rule")

    def mc_count(self, grid: torch.Tensor, level: float, face_rule: str = "sign"):
        self.sync_stream()
        self.set_mc_face_rule(face_rule)
        nv, nf = C.c_int64(), C.c_int64()
        mm = (C.c_float * 3)()
        self._check(self.lib.hy3d_mc_count(self.h, _ptr(grid), grid.shape[0], grid.shape[1], grid.shape[2], float(level),
                                           C.byref(nv), C.byref(nf), mm), "hy3d_mc_count")
        return nv.value, nf.value, (mm[0], mm[1], bool(mm[2]))

    def mc_emit(self, div, mul, add, verts: torch.Tensor, faces: torch.Tensor):
        self.sync_stream()
        d = (C.c_double * 3)(*[float(v) for v in div])
        m = (C.c_double * 3)(*[float(v) for v in mul])
        a = (C.c_double * 3)(*[float(v) for v in add])
        self._check(self.lib.hy3d_mc_emit(self.h, d, m, a, _ptr(verts), _ptr(faces)), "hy3d_mc_emit")

    def mc_count_slab(self, grid: torch.Tensor, own_planes: int, level: float, face_rule: str = "sign"):
        """grid = owned planes followed by the next slab's halo planes; counts of the owned part (see hy3dgeo.h)."""
        self.sync_stream()
        self.set_mc_face_rule(face_rule)
        nv, nf = C.c_int64(), C.c_int64()
        mm = (C.c_float * 3)()
        self._check(self.lib.hy3d_mc_count_slab(self.h, _ptr(grid), grid.shape[0], grid.shape[1], grid.shape[2], int(own_planes),
                                                float(level), C.byref(nv), C.byref(nf), mm), "hy3d_mc_count_slab")
        return nv.value, nf.value, (mm[0], mm[1], bool(mm[2]))

    def mc_emit_slab(self, div, mul, add, plane0: int, id_base: int, verts: torch.Tensor, faces: torch.Tensor):
        self.sync_stream()
        d = (C.c_double * 3)(*[float(v) for v in div])
        m = (C.c_double * 3)(*[float(v) for v in mul])
        a = (C.c_double * 3)(*[float(v) for v in add])
        self._check(self.lib.hy3d_mc_emit_slab(self.h, d, m, a, int(plane0), int(id_base), _ptr(verts), _ptr(faces)), "hy3d_mc_emit_slab")

    def dmc_count(self, grid: torch.Tensor):
        """Dual marching cubes, phase 1 (see hy3dgeo.h): -> (nV, nF, (min, max, nan)) of the fp32 grid, inside iff > 0."""
        self.sync_stream()
        nv, nf = C.c_int64(), C.c_int64()
        mm = (C.c_float * 3)()
        self._check(self.lib.hy3d_dmc_count(self.h, _ptr(grid), grid.shape[0], grid.shape[1], grid.shape[2],
                                            C.byref(nv), C.byref(nf), mm), "hy3d_dmc_count")
        return nv.value, nf.value, (mm[0], mm[1], bool(mm[2]))

    def dmc_emit(self, verts: torch.Tensor, faces: torch.Tensor):
        self.sync_stream()
        self._check(self.lib.hy3d_dmc_emit(self.h, _ptr(verts), _ptr(faces)), "hy3d_dmc_emit")

    def dmc_count_slab(self, slab: torch.Tensor, own_planes: int, plane0: int, n0_global: int):
        """slab = owned planes [plane0, plane0 + own_planes) of a grid of n0_global planes, followed by the next slab's
        halo planes; -> (nV, nF, (min, max, nan)) of the owned part (see hy3dgeo.h: hy3d_dmc_count_slab)."""
        self.sync_stream()
        nv, nf = C.c_int64(), C.c_int64()
        mm = (C.c_float * 3)()
        self._check(self.lib.hy3d_dmc_count_slab(self.h, _ptr(slab), int(own_planes), slab.shape[0] - int(own_planes), slab.shape[1],
                                                 slab.shape[2], int(plane0), int(n0_global), C.byref(nv), C.byref(nf), mm),
                    "hy3d_dmc_count_slab")
        return nv.value, nf.value, (mm[0], mm[1], bool(mm[2]))

    def dmc_emit_slab(self, id_base: int, verts: torch.Tensor, faces: torch.Tensor, bbox: torch.Tensor):
        """Uncentred vertices, faces with global ids, and the slab's ordered-int bounding box (int32 [6], device)."""
        self.sync_stream()
        self._check(self.lib.hy3d_dmc_emit_slab(self.h, int(id_base), _ptr(verts), _ptr(faces), _ptr(bbox)), "hy3d_dmc_emit_slab")

    def dmc_center(self, verts: torch.Tensor, bbox6):
        """verts -= 0.5f * (lo + hi) in place; bbox6 = 6 ordered ints (lo[3], hi[3]) on the host."""
        self.sync_stream()
        box = (C.c_int32 * 6)(*[int(v) for v in bbox6])
        self._check(self.lib.hy3d_dmc_center(self.h, _ptr(verts), verts.shape[0], box), "hy3d_dmc_center")

    def mesh_clean(self, verts: torch.Tensor, faces: torch.Tensor, flip_winding: bool):
        """Device tensors (verts float32 [V,3], faces int32 [F,3]) -> the same mesh without non-finite / unreferenced
        vertices and the faces that used them, winding optionally reversed (see hy3dgeo.h: hy3d_mesh_clean)."""
        self.sync_stream()
        verts, faces = verts.contiguous(), faces.contiguous()
        vo, fo = torch.empty_like(verts), torch.empty_like(faces)
        nv, nf = C.c_int64(), C.c_int64()
        self._check(self.lib.hy3d_mesh_clean(self.h, _ptr(verts), verts.shape[0], _ptr(faces), faces.shape[0], int(bool(flip_winding)),
                                             _ptr(vo), _ptr(fo), C.byref(nv), C.byref(nf)), "hy3d_mesh_clean")
        return vo[: nv.value], fo[: nf.value]

    def _mesh_filter(self, name, verts, faces, *args, extra=()):
        self.sync_stream()
        verts = verts.detach().to(device=self.device, dtype=torch.float32).contiguous()
        faces = faces.detach().to(device=self.device, dtype=torch.int32).contiguous()
        if verts.dim() != 2 or verts.shape[1] != 3 or faces.dim() != 2 or faces.shape[1] != 3:
            raise ValueError(f"{name}: expected verts [V, 3] and faces [F, 3], got {tuple(verts.shape)} and {tuple(faces.shape)}")
        vo, fo = torch.empty_like(verts), torch.empty_like(faces)
        nv, nf = C.c_int64(), C.c_int64()
        self._check(getattr(self.lib, name)(self.h, _ptr(verts), verts.shape[0], _ptr(faces), faces.shape[0], *args,
                                            _ptr(vo), _ptr(fo), C.byref(nv), C.byref(nf), *extra), name)
        return vo[: nv.value], fo[: nf.value]

    def mesh_remove_floaters(self, verts: torch.Tensor, faces: torch.Tensor, min_faces: int):
        """Device tensors -> the mesh without the faces of edge-connected components of fewer than ``min_faces`` faces and
        without the faces touching their vertices; unreferenced vertices dropped, order kept (hy3dgeo.h)."""
        return self._mesh_filter("hy3d_mesh_remove_floaters", verts, faces, int(min_faces))

    def mesh_weld(self, verts: torch.Tensor, faces: torch.Tensor):
        """Device tensors -> the mesh with bit-equal finite vertices merged into the smallest id, faces that collapse
        removed, unreferenced vertices dropped, order kept (hy3dgeo.h)."""
        return self._mesh_filter("hy3d_mesh_weld", verts, faces)

    def mesh_decimate(self, verts: torch.Tensor, faces: torch.Tensor, max_faces: int):
        """Device tensors -> (verts, faces, rounds): quadric edge-collapse decimation to ``max_faces`` faces (``max_faces - 1``
        or ``max_faces`` unless no valid collapse is left); the mesh as given when it has no more faces (hy3dgeo.h)."""
        rounds = C.c_int32()
        vo, fo = self._mesh_filter("hy3d_mesh_decimate", verts, faces, int(max_faces), extra=(C.byref(rounds),))
        return vo, fo, rounds.value

    def mc_cases(self, grid: torch.Tensor, level: float) -> torch.Tensor:
        self.sync_stream()
        out = torch.empty(tuple(s - 1 for s in grid.shape), dtype=torch.uint8, device=self.device)
        self._check(self.lib.hy3d_mc_cases(self.h, _ptr(grid), grid.shape[0], grid.shape[1], grid.shape[2], float(level),
                                           _ptr(out)), "hy3d_mc_cases")
        return out


_tls = threading.local()


def get_context(device) -> GeoContext:
    """Per-(thread, device) context: per-call state never lives on shared objects
    (the reference's processors race under api_server threads, SURVEY §3.5)."""
    device = torch.device(device)
    if device.type != "cuda":
        raise RuntimeError("hy3dgeo runs on CUDA devices only (no CPU fallback)")
    idx = device.index if device.index is not None else torch.cuda.current_device()
    cache = getattr(_tls, "ctx", None)
    if cache is None:
        cache = _tls.ctx = {}
    if idx not in cache:
        cache[idx] = GeoContext(torch.device("cuda", idx))
    return cache[idx]
