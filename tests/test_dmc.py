"""Dual marching cubes (``mc_algo='dmc'``): the generated patch table against the oracle's run-time tracing, the oracle's
surface invariants on CPU, and on the GPU the CUDA kernels bit-exact against ``oracle/dmc.py``, the extractor contract and
the FlashVDM pipeline with its default ``mc_algo``."""
import importlib.util
import os
import re

import numpy as np
import pytest
import torch

from oracle import dmc as OD, mc as OM
from oracle.mesh import assert_same_mesh

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _gen():
    spec = importlib.util.spec_from_file_location("gen_mc_tables", os.path.join(ROOT, "tools", "gen_mc_tables.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


def sphere(n, r=0.6, sharp=20.0):
    x = np.linspace(-1.01, 1.01, n, dtype=np.float32)
    X, Y, Z = np.meshgrid(x, x, x, indexing="ij")
    return np.tanh(sharp * (r - np.sqrt(X * X + Y * Y + Z * Z))).astype(np.float32)


def signed_volume(v, f):
    v = v.astype(np.float64)
    a, b, c = v[f[:, 0]], v[f[:, 1]], v[f[:, 2]]
    return float(np.einsum("ij,ij->i", a, np.cross(b, c)).sum() / 6)


def interior_sign_changes(g):
    ins = g > 0
    n = 0
    for axis in range(3):
        lo, hi = [slice(None)] * 3, [slice(None)] * 3
        lo[axis], hi[axis] = slice(0, -1), slice(1, None)
        flip = ins[tuple(lo)] != ins[tuple(hi)]
        inner = [slice(1, -1) if a != axis else slice(None) for a in range(3)]
        n += int(flip[tuple(inner)].sum())
    return n


def check_invariants(v, f, g):
    """closed genus-0 surface: F = 2V - 4, quads = interior sign-change edges, every edge in exactly two faces"""
    V, F = len(v), len(f)
    assert F == 2 * V - 4 and F == 2 * interior_sign_changes(g)
    e = np.sort(np.concatenate([f[:, [0, 1]], f[:, [1, 2]], f[:, [2, 0]]]).astype(np.int64), 1)
    _, cnt = np.unique(e[:, 0] * V + e[:, 1], return_counts=True)
    assert (cnt == 2).all()
    d = np.concatenate([f[:, [0, 1]], f[:, [1, 2]], f[:, [2, 0]]]).astype(np.int64)       # consistent orientation:
    assert len(np.unique(d[:, 0] * V + d[:, 1])) == len(d)                                # each directed edge once


# ---- CPU -------------------------------------------------------------------------------------------------------------
def test_generated_table_equals_oracle_tracing(tmp_path):
    src = open(os.path.join(ROOT, "hunyuan3d-2_b200", "csrc", "dmc_tables.inc")).read()
    body = lambda name: [int(x) for x in re.findall(r"-?\d+", src.split(name)[1].split("};")[0].split("=", 1)[1])]
    cnt, ep = OD.patch_tables()
    assert body("hy3d_dmc_patch_count[256]") == cnt.tolist()
    assert body("hy3d_dmc_edge_patch[256][12]") == ep.ravel().tolist()
    assert {k: int((cnt == k).sum()) for k in range(5)} == {0: 2, 1: 162, 2: 82, 3: 8, 4: 2}
    assert int((ep >= 0).sum(1).max()) <= 12 and max(int((ep == p).sum(1).max()) for p in range(4)) <= 7
    out = tmp_path / "dmc_tables.inc"                   # the generator reproduces the committed file byte for byte
    _gen().write_dmc_tables(str(out))
    assert out.read_bytes() == open(os.path.join(ROOT, "hunyuan3d-2_b200", "csrc", "dmc_tables.inc"), "rb").read()


def test_oracle_sphere_invariants():
    n = 49
    g = sphere(n)
    vr, f = OD.dual_marching_cubes_raw(g)
    gen = _gen()
    loops = sum(len(gen.trace_loops(int(c))) for c in OM.cube_cases(g, 0.0).ravel() if 0 < c < 255)
    assert len(vr) == loops
    check_invariants(vr, f, g)
    vm, fm, _, _ = OM.marching_cubes(g, 0.0)
    assert np.sign(signed_volume(vr, f)) == np.sign(signed_volume(vm, fm)) != 0
    from scipy.spatial import cKDTree
    d1, _ = cKDTree(vr).query(vm)
    d2, _ = cKDTree(vm).query(vr)
    assert 0.5 * (d1.mean() + d2.mean()) < 0.5                       # Chamfer, index units: below half a cell
    v, f2 = OD.dual_marching_cubes(g)
    assert v.dtype == np.float32 and np.array_equal(f, f2)
    assert np.allclose(v.min(0) + v.max(0), 0, atol=1e-6)             # centred on the bounding box


def test_oracle_errors():
    with pytest.raises(ValueError):
        OD.dual_marching_cubes(np.ones((1, 4, 4), np.float32))
    with pytest.raises(RuntimeError):
        OD.dual_marching_cubes(-np.ones((4, 4, 4), np.float32))


# ---- GPU -------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def dev():
    return torch.device("cuda:0")


@pytest.fixture(scope="module")
def ctx(dev):
    from hy3dgeo import _lib
    return _lib.get_context(dev)


def gpu_dmc(ctx, vol):
    g = torch.from_numpy(np.ascontiguousarray(vol, np.float32)).cuda()
    nv, nf, _ = ctx.dmc_count(g)
    v = torch.empty((nv, 3), dtype=torch.float32, device="cuda")
    f = torch.empty((nf, 3), dtype=torch.int32, device="cuda")
    ctx.dmc_emit(v, f)
    return v.cpu().numpy(), f.cpu().numpy()


NOISE_SHAPES = [(5, 6, 97), (4, 5, 300), (3, 4, 600), (2, 7, 40), (9, 2, 33), (3, 3, 3), (2, 2, 70), (6, 3, 2)]


@pytest.mark.gpu
@pytest.mark.parametrize("shape", NOISE_SHAPES)
def test_cuda_dmc_bit_exact_on_noise(shape, ctx):
    rng = np.random.default_rng(sum(shape))
    for vol in (rng.standard_normal(shape).astype(np.float32),
                rng.integers(-2, 3, size=shape).astype(np.float32)):     # exact zeros (outside) on many crossings
        assert_same_mesh(gpu_dmc(ctx, vol), OD.dual_marching_cubes(vol))


@pytest.mark.gpu
def test_cuda_dmc_sphere_with_nan_and_zero(ctx):
    g = sphere(41)
    g[20, 20, 28] = 0.0                                     # an exact zero on the surface band
    g[5:9, 18:23, 20:30] = np.nan                           # a NaN block across the surface
    got, ref = gpu_dmc(ctx, g), OD.dual_marching_cubes(g)
    assert_same_mesh(got, ref)
    assert np.isnan(got[0]).any() and np.isfinite(got[0]).any()


@pytest.mark.gpu
@pytest.mark.parametrize("n", [257, 385])
def test_cuda_dmc_full_size_invariants(n, ctx):
    g = sphere(n, sharp=8.0)
    v, f = gpu_dmc(ctx, g)
    check_invariants(v, f, g)
    vm, fm, _, _ = OM.marching_cubes(g, 0.0)
    assert np.sign(signed_volume(v, f)) == np.sign(signed_volume(vm, fm)) != 0
    if n == 257:
        assert_same_mesh((v, f), OD.dual_marching_cubes(g))
    else:                                                   # same centre and extent as the MC mesh, normalised
        vmn = vm / (n - 1)
        c = 0.5 * (vmn.min(0) + vmn.max(0))
        got, want = np.stack([v.min(0), v.max(0)]), np.stack([vmn.min(0) - c, vmn.max(0) - c])
        assert np.abs(got - want).max() < 1.0 / (n - 1)


@pytest.mark.gpu
def test_dmc_extractor_contract(dev, tmp_path):
    from hy3dgeo.surface_extractors import DMCSurfaceExtractor, SurfaceExtractors, export_to_trimesh
    assert SurfaceExtractors["dmc"] is DMCSurfaceExtractor
    ext = DMCSurfaceExtractor()
    g = sphere(33)
    ref = OD.dual_marching_cubes(g)
    t = torch.from_numpy(g).to(dev)
    kw = dict(mc_level=0.0, bounds=1.01, octree_resolution=32)
    v, f = ext.run_device(t, **kw)
    assert v.is_cuda and v.dtype == torch.float32 and f.dtype == torch.int32 and v.is_contiguous() and f.is_contiguous()
    out = ext(t[None], **kw)[0]
    assert out.mesh_v.dtype == np.float32 and out.mesh_f.dtype == np.int32 and out.mesh_v.flags.c_contiguous
    assert_same_mesh((out.mesh_v, out.mesh_f), ref)
    assert np.abs(out.mesh_v.min(0) + out.mesh_v.max(0)).max() < 1e-6            # centred on the bounding box
    other = ext(t[None], mc_level=0.3, bounds=[-2, -1, -3, 2, 1, 3], octree_resolution=64)[0]
    assert_same_mesh((other.mesh_v, other.mesh_f), ref)                         # mc_level / bounds play no part
    h = ext(t.half()[None], **kw)[0]                                             # fp16 accepted, converted to fp32
    assert_same_mesh((h.mesh_v, h.mesh_f), OD.dual_marching_cubes(g.astype(np.float16).astype(np.float32)))
    assert ext(torch.stack([-torch.ones_like(t), t]), **kw)[0] is None           # no sign change -> None for that item
    assert ext(torch.zeros((1, 1, 4, 4), device=dev), **kw) == [None]            # dimension below 2 -> None
    gn = g.copy()
    gn[:12] = np.nan                                                              # NaN rim as left by the sparse decoders
    m = ext(torch.from_numpy(gn).to(dev)[None], **kw)[0]
    assert np.isnan(m.mesh_v).any()
    tm = export_to_trimesh(m, dev)
    tv = np.asarray(tm.vertices if hasattr(tm, "vertices") else tm.mesh_v)
    tf = np.asarray(tm.faces if hasattr(tm, "faces") else tm.mesh_f)
    assert np.isfinite(tv).all() and len(tf) > 0 and tf.max() < len(tv)

    import torch.distributed as dist
    from hy3dgeo.parallel import SlabGrid
    own = not dist.is_initialized()
    if own:
        dist.init_process_group("gloo", init_method=f"file://{tmp_path}/store", rank=0, world_size=1)
    try:
        sg = SlabGrid([t.clone()], 0, g.shape[0], g.shape, False)
        s = ext(sg, **kw)[0]
        assert_same_mesh((s.mesh_v, s.mesh_f), ref)
    finally:
        if own:
            dist.destroy_process_group()


@pytest.mark.gpu
def test_flashvdm_default_mc_algo_returns_the_oracle_mesh(gold, dev):
    """``vae.enable_flashvdm_decoder()`` with its defaults selects ``mc_algo='dmc'``: latents2mesh on the mini-turbo decoder
    yields a mesh (not None), equal to the oracle's dual marching cubes of the same device grid."""
    import hy3dgeo
    from hy3dgeo import weights as W
    from hy3dgeo.surface_extractors import DMCSurfaceExtractor
    g = gold("flash_turbo.npz")
    cfg = W.MINI_TURBO
    sd = W.sparsify_field(W.synthetic_state_dict(cfg, seed=0), cfg, int(g["keep_freqs"]), float(g["gain"]), float(g["bias"]))
    vae = hy3dgeo.B200ShapeVAE(cfg, sd, device=dev)
    vae.enable_flashvdm_decoder()
    assert isinstance(vae.surface_extractor, DMCSurfaceExtractor)
    grids = []
    inner = vae.surface_extractor

    def recording(grid_logits, **kw):
        grids.append(grid_logits.clone())
        return inner(grid_logits, **kw)
    vae.surface_extractor = recording
    lat = vae(W.synthetic_latents(cfg, 1, 1234).to(dev))
    out = vae.latents2mesh(lat, bounds=1.01, num_chunks=600, mc_level=0.0, octree_resolution=64, min_resolution=15,
                           enable_pbar=False)
    assert len(out) == 1 and out[0] is not None and len(out[0].mesh_f) > 0
    assert_same_mesh((out[0].mesh_v, out[0].mesh_f), OD.dual_marching_cubes(grids[0][0].cpu().numpy()))


def test_dmc_against_diso():
    """Where diso is importable: same vertex count, bounding box (settles the 1 / (n - 1) scale) and area on fields without
    ambiguous cubes.  diso's triangles, quad split and vertex order are not compared (DESIGN.md §2)."""
    pytest.importorskip("diso", reason="diso is not installed: the dual marching cubes stays unpinned against it")
    if not torch.cuda.is_available():
        pytest.skip("diso runs on CUDA")
    from diso import DiffDMC
    from hy3dgeo.surface_extractors import DMCSurfaceExtractor

    def area(v, f):
        v = v.astype(np.float64)
        return float(np.linalg.norm(np.cross(v[f[:, 1]] - v[f[:, 0]], v[f[:, 2]] - v[f[:, 0]]), axis=1).sum() / 2)
    dmc = DiffDMC(dtype=torch.float32).cuda()
    for n, r in ((49, 0.6), (65, 0.45)):
        g = sphere(n, r=r, sharp=6.0)
        t = torch.from_numpy(g).cuda()
        dv, df = dmc(-t / (n - 1), deform=None, return_quads=False, normalize=True)
        dv = dv - 0.5 * (dv.min(0)[0] + dv.max(0)[0])
        dv, df = dv.cpu().numpy(), df.cpu().numpy()
        v, f = DMCSurfaceExtractor().run(t, octree_resolution=n - 1)
        assert len(v) == len(dv)
        assert np.abs(np.stack([v.min(0), v.max(0)]) - np.stack([dv.min(0), dv.max(0)])).max() < 1e-3
        assert abs(area(v, f) - area(dv, df)) < 1e-2 * area(dv, df)
