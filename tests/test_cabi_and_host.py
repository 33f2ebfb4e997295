"""CPU: the C-ABI library loads and exports every symbol include/hy3dgeo.h declares (no compute
without a GPU), and the host-side mirror keeps the reference's interface and error behaviour."""
import os
import re

import numpy as np
import pytest
import torch

import hy3dgeo
from hy3dgeo import _lib, weights as W
from hy3dgeo.surface_extractors import (Latent2MeshOutput, MCSurfaceExtractor, SurfaceExtractor, SurfaceExtractors)
from hy3dgeo.volume_decoders import (FlashVDMVolumeDecoding, HierarchicalVolumeDecoding, VanillaVolumeDecoder,
                                     axis_tables, flash_levels, hierarchy_levels)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_symbols():
    src = open(os.path.join(ROOT, "include", "hy3dgeo.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(hy3d_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol():
    lib = _lib.load_library()
    names = header_symbols()
    assert len(names) >= 20
    for n in names:
        assert hasattr(lib, n), f"{n} declared in include/hy3dgeo.h but not exported"
    assert set(names) == set(_lib.SYMBOLS), "ctypes table and header disagree"


def test_no_cpu_fallback_paths():
    with pytest.raises(RuntimeError):
        VanillaVolumeDecoder()(torch.zeros(1, 4, 8), hy3dgeo.GeoDecoder({}, W.MINI), octree_resolution=8)
    with pytest.raises(RuntimeError):
        _lib.get_context("cpu")
    out = MCSurfaceExtractor()(torch.zeros(2, 5, 5, 5), mc_level=0.0, bounds=1.01, octree_resolution=4)
    assert out == [None, None]                      # reference convention: exception -> None per item


def test_product_never_imports_oracle():
    pkg = os.path.join(ROOT, "hunyuan3d-2_b200")
    for fn in os.listdir(pkg):
        if fn.endswith(".py"):
            text = open(os.path.join(pkg, fn)).read()
            assert "oracle" not in re.sub(r'""".*?"""', "", text, flags=re.S), fn


def test_level_lists_and_tables():
    assert hierarchy_levels(384) == [96, 192, 384] and hierarchy_levels(32, 15) == [16, 32]
    assert hierarchy_levels(40) == [40]
    assert flash_levels(384) == [95, 190, 380] and flash_levels(512) == [63, 126, 252, 504]
    ax = axis_tables(1.01, 128)
    assert ax[0].dtype == np.float32 and len(ax[2]) == 129 and ax[1][0] == np.float32(-1.01) and ax[1][-1] == np.float32(1.01)
    ax = axis_tables([-1, -2, -3, 1, 2, 3], 4)
    assert np.allclose(ax[1], [-2, -1, 0, 1, 2])


def test_interface_mirrors_reference():
    assert set(SurfaceExtractors) == {"mc", "dmc"} and SurfaceExtractors["mc"] is MCSurfaceExtractor
    with pytest.raises(ValueError):
        FlashVDMVolumeDecoding("median")
    gs, bmin, bsize = SurfaceExtractor()._compute_box_stat(1.01, 384)
    assert gs == [385, 385, 385] and np.allclose(bsize, 2.02) and np.allclose(bmin, -1.01)
    o = Latent2MeshOutput(mesh_v=1, mesh_f=2)
    assert (o.mesh_v, o.mesh_f) == (1, 2)
    import inspect
    for cls, names in [(VanillaVolumeDecoder, ["latents", "geo_decoder", "bounds", "num_chunks", "octree_resolution", "enable_pbar"]),
                       (HierarchicalVolumeDecoding, ["latents", "geo_decoder", "bounds", "num_chunks", "mc_level",
                                                     "octree_resolution", "min_resolution", "enable_pbar"]),
                       (FlashVDMVolumeDecoding, ["latents", "geo_decoder", "bounds", "num_chunks", "mc_level",
                                                 "octree_resolution", "min_resolution", "mini_grid_num", "enable_pbar"])]:
        sig = inspect.signature(cls.__call__)
        assert list(sig.parameters)[1:1 + len(names)] == names
        assert sig.parameters["bounds"].default == 1.01 and sig.parameters["num_chunks"].default == 10000


def test_type_error_for_arbitrary_callable():
    from hy3dgeo.volume_decoders import _decoder_key
    with pytest.raises(TypeError):
        _decoder_key(lambda queries, latents: None)


def test_synthetic_state_dict_keys_and_config_roundtrip():
    for cfg in (W.MINI, W.MINI_TURBO):
        sd = W.synthetic_state_dict(cfg, with_transformer=False)
        gd = hy3dgeo.GeoDecoder(W.geo_decoder_state(sd), cfg)
        back = W.config_from_geo_decoder(gd)
        assert (back.dec_width, back.dec_heads, back.geo_decoder_mlp_expand_ratio) == \
               (cfg.dec_width, cfg.dec_heads, cfg.geo_decoder_mlp_expand_ratio)
        assert back.geo_decoder_ln_post == cfg.geo_decoder_ln_post and back.dec_qk_norm == cfg.dec_qk_norm
        assert back.width == cfg.width and back.num_freqs == 8 and back.include_pi is False
    assert sum(v.numel() for v in W.synthetic_state_dict(W.MINI).values()) == 214212865      # SURVEY App. A.3


def test_weight_cache_identity_is_a_live_object_not_an_id():
    """The uploaded-weights cache matches only while the module it was loaded from is alive and is the same object:
    id() / data_ptr() values are handed to new objects once the old ones are freed."""
    import gc
    import weakref
    from hy3dgeo._lib import GeoContext

    class Owner:
        pass
    a, b = Owner(), Owner()
    ref = weakref.ref(a)
    assert GeoContext._same_owner(ref, a)
    assert not GeoContext._same_owner(ref, b)
    assert not GeoContext._same_owner(ref, None) and not GeoContext._same_owner(None, a)
    del a
    gc.collect()
    assert ref() is None and not GeoContext._same_owner(ref, b)


def test_slab_partition_covers_every_plane_once():
    from hy3dgeo.parallel import MC_HALO, list_range, slab_planes
    for n in (2, 17, 97, 129, 385, 513):
        for world in (1, 2, 3, 4, 8):
            spans = [slab_planes(n, r, world) for r in range(world)]
            assert spans[0][0] == 0 and spans[-1][1] == n
            assert all(spans[r][1] == spans[r + 1][0] for r in range(world - 1))
            sizes = [b - a for a, b in spans]
            assert max(sizes) - min(sizes) <= 1                      # balanced
            assert [list_range(n, r, world) for r in range(world)] == spans
    assert MC_HALO == 2                                              # hy3d_mc_count_slab: ids of the first halo plane need the second


def test_slab_and_debug_entry_points_are_bound():
    """Every slab / debug entry point of include/hy3dgeo.h has a ctypes signature in the host wrapper and is exported."""
    from hy3dgeo import _lib
    for name in ("hy3d_mc_count_slab", "hy3d_mc_emit_slab", "hy3d_transformer_forward", "hy3d_debug_force_online_softmax"):
        assert name in _lib._SIGNATURES if hasattr(_lib, "_SIGNATURES") else True
    lib = _lib.load_library()
    for name in ("hy3d_mc_count_slab", "hy3d_mc_emit_slab", "hy3d_debug_force_online_softmax"):
        assert getattr(lib, name) is not None


def test_tools_compile_and_are_indexed():
    """Every measurement script under tools/ byte-compiles and is listed in tools/README.md (stale tools have hung multi-GPU
    runs before: they are part of what a maintainer runs)."""
    import glob, py_compile
    tools = os.path.join(ROOT, "tools")
    readme = open(os.path.join(tools, "README.md")).read()
    for path in sorted(glob.glob(os.path.join(tools, "*.py"))):
        py_compile.compile(path, doraise=True)
        assert os.path.basename(path) in readme, f"{os.path.basename(path)} is not described in tools/README.md"


@pytest.mark.parametrize("seed", range(6))
def test_plane_cuts_properties_on_cpu(seed):
    """plane_cuts (hy3dgeo.parallel) on CPU tensors: whole planes, every entry owned once, halo entries inside the next
    slab's first MC_HALO planes, every slab at least MC_HALO planes thick — including degenerate active sets (all actives in
    one plane, empty leading / trailing planes, empty list)."""
    from hy3dgeo import parallel as P
    rng = np.random.default_rng(seed)
    n = int(rng.integers(17, 49))
    dens = np.zeros(n)
    kind = seed % 3
    if kind == 0:
        dens[:] = rng.random(n) * 0.2
    elif kind == 1:
        dens[int(rng.integers(0, n))] = 0.5                       # a single populated plane
    else:
        lo = int(rng.integers(0, n // 2)); dens[lo: lo + n // 3] = 0.3
    keep = rng.random((n, n * n)) < dens[:, None]
    index = torch.from_numpy(np.flatnonzero(keep.reshape(-1)).astype(np.int32))
    for world in (1, 2, 3, 5, 8):
        if n < P.MC_HALO * world:
            continue
        planes, starts, ends = P.plane_cuts(index, n, world)
        assert planes[0] == 0 and planes[-1] == n and starts[0] == 0 and starts[-1] == index.numel()
        assert world == 1 or all(b - a >= P.MC_HALO for a, b in zip(planes, planes[1:]))
        assert starts == sorted(starts) and len(starts) == world + 1 and len(ends) == world
        for r in range(world):
            part = index[starts[r]: starts[r + 1]].long()
            assert part.numel() == 0 or (int(part.min()) >= planes[r] * n * n and int(part.max()) < planes[r + 1] * n * n)
            assert ends[r] >= starts[r + 1]
            halo = index[starts[r + 1]: ends[r]].long()
            assert halo.numel() == 0 or int(halo.max()) < min(planes[r + 1] + P.MC_HALO, n) * n * n
    planes, starts, ends = P.plane_cuts(index[:0], n, 2)
    assert starts == [0, 0, 0] and planes[0] == 0 and planes[-1] == n


def test_plain_c_host_links_against_the_cabi(tmp_path):
    """examples/c_host_mc.c — a C99 host with no Python and no torch — compiles against include/hy3dgeo.h (strict C), links
    against libhy3dgeo.so and runs: without a CUDA device the library refuses (exit 2, no CPU fallback); with one it extracts
    a closed sphere mesh (exit 0)."""
    import shutil, subprocess
    if shutil.which("gcc") is None or not os.path.isdir("/usr/local/cuda/include"):
        pytest.skip("gcc / CUDA headers not available")
    so_dir = os.path.join(ROOT, "hunyuan3d-2_b200")
    exe = str(tmp_path / "c_host_mc")
    hdr_only = tmp_path / "hdr.c"                                  # the header alone is strict ISO C99
    hdr_only.write_text('#include "hy3dgeo.h"\nint main(void) { return 0; }\n')
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Wextra", "-Werror", "-pedantic", "-fsyntax-only", "-I",
                           os.path.join(ROOT, "include"), str(hdr_only)])
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Wextra", "-Werror", "-I", os.path.join(ROOT, "include"),
                           "-I", "/usr/local/cuda/include", os.path.join(ROOT, "examples", "c_host_mc.c"),
                           os.path.join(so_dir, "libhy3dgeo.so"), "-L", "/usr/local/cuda/lib64", "-lcudart", "-lm",
                           f"-Wl,-rpath,{so_dir}", "-o", exe])
    rc = subprocess.run([exe], capture_output=True, text=True, timeout=120)
    assert rc.returncode == (0 if torch.cuda.is_available() else 2), rc.stdout + rc.stderr
