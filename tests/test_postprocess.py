"""Mesh post-processing (``FloaterRemover`` / ``DegenerateFaceRemover``): the numpy contract ``oracle/postprocess.py`` on
hand-built meshes and noise-field meshes on CPU; on the GPU ``hy3d_mesh_remove_floaters`` / ``hy3d_mesh_weld`` and the public
classes bit-exact against it, from hand-built meshes up to a full-scale 385^3 marching-cubes mesh."""
import numpy as np
import pytest
import torch
from scipy.ndimage import gaussian_filter

from oracle import dmc as OD, mc as OM, mesh as OMESH, postprocess as PP


def tet(a, b, c, d):
    """the four faces of a tetrahedron over vertex ids a, b, c, d"""
    return [(a, b, c), (a, c, d), (a, d, b), (b, d, c)]


def grid_sheet(n, z=0.0):
    """n x n vertices, 2 (n-1)^2 triangles: one edge-connected component"""
    i, j = np.meshgrid(np.arange(n), np.arange(n), indexing="ij")
    v = np.stack([i.ravel(), j.ravel(), np.full(n * n, z)], 1).astype(np.float32)
    q = (i[:-1, :-1] * n + j[:-1, :-1]).ravel()
    f = np.concatenate([np.stack([q, q + n, q + 1], 1), np.stack([q + 1, q + n, q + n + 1], 1)])
    return v, f.astype(np.int32)


def sheet_with_tet_at_vertex():
    """a 1058-face sheet (min_faces = 5) and a 4-face tetrahedron sharing the sheet's interior vertex 12 * 24 + 12"""
    v, f = grid_sheet(24)
    s = 12 * 24 + 12
    n = len(v)
    extra = np.array([[12.5, 12, 1], [12, 12.5, 1], [12.5, 12.5, 2]], np.float32)
    return np.concatenate([v, extra]), np.concatenate([f, np.array(tet(s, n, n + 1, n + 2), np.int32)]), s


def noise_field(n, seed, quantile, sigma=1.5):
    g = gaussian_filter(np.random.default_rng(seed).standard_normal((n, n, n)), sigma)
    return (g - np.quantile(g, quantile)).astype(np.float32)


def quantised_field(n=48, seed=0):
    """values on multiples of 1/8: many exact zeros, so marching cubes emits coincident vertices"""
    g = gaussian_filter(np.random.default_rng(seed).standard_normal((n, n, n)), 1.5)
    return (np.round(g * 8) / 8).astype(np.float32)


def mc_mesh(vol):
    v, f, _, _ = OM.marching_cubes(vol, 0.0)
    return v.astype(np.float32), f.astype(np.int32)


# ---- CPU: the contract --------------------------------------------------------------------------------------------------
def test_min_faces_formula():
    assert [PP.min_faces_for(F) for F in (0, 199, 200, 399, 400, 1000, 893_000)] == [0, 0, 1, 1, 2, 5, 4465]


def test_oracle_vertex_shared_tet_is_a_floater_and_takes_the_sheet_faces_at_that_vertex():
    v, f, s = sheet_with_tet_at_vertex()
    lab = PP.edge_components(f)
    assert len(np.unique(lab)) == 2 and PP.vertex_components(f, len(v)) == 1
    assert PP.min_faces_for(len(f)) == 5
    vo, fo = PP.remove_floaters(v, f)
    touching = int((f[:-4] == s).any(1).sum())
    assert touching == 6 and len(fo) == len(f) - 4 - touching
    assert len(vo) == len(v) - 4                             # the tet's three own vertices and the shared one
    assert np.array_equal(vo, np.delete(v, [s, len(v) - 3, len(v) - 2, len(v) - 1], axis=0))


def test_oracle_edge_shared_tets_are_one_component():
    f = np.array(tet(0, 1, 2, 3) + tet(0, 1, 4, 5), np.int32)
    assert len(np.unique(PP.edge_components(f))) == 1
    v = np.random.default_rng(0).standard_normal((6, 3)).astype(np.float32)
    vo, fo = PP.remove_floaters(v, f, min_faces=8)
    assert np.array_equal(vo, v) and np.array_equal(fo, f)
    vo, fo = PP.remove_floaters(v, f, min_faces=9)
    assert len(vo) == 0 and len(fo) == 0


def strip(k, base):
    """k triangles in a fan around vertex `base`: one component of k faces over k + 2 vertices"""
    return [(base, base + i + 1, base + i + 2) for i in range(k)]


def test_oracle_component_of_exactly_min_faces_stays():
    v, f = grid_sheet(24)                                    # 1058 faces; with the 7 below F = 1065, min_faces = 5
    n = len(v)
    f = np.concatenate([f, np.array(strip(5, n) + strip(2, n + 7), np.int32)])
    v = np.concatenate([v, np.random.default_rng(1).standard_normal((11, 3)).astype(np.float32)])
    assert PP.min_faces_for(len(f)) == 5
    vo, fo = PP.remove_floaters(v, f)
    assert len(fo) == len(f) - 2 and np.array_equal(fo[-5:], f[-7:-2])
    assert len(vo) == len(v) - 4
    vo, fo = PP.remove_floaters(v, f, min_faces=6)
    assert len(fo) == len(f) - 7


def test_oracle_non_manifold_edge():
    f = np.array([(0, 1, 2), (1, 0, 3), (0, 1, 4), (5, 1, 0), (6, 7, 8)], np.int32)   # edge {0, 1} in four faces
    lab = PP.edge_components(f)
    assert len(set(lab[:4])) == 1 and lab[4] != lab[0]
    v = np.arange(27, dtype=np.float32).reshape(9, 3)
    vo, fo = PP.remove_floaters(v, f, min_faces=2)
    assert np.array_equal(fo, f[:4]) and np.array_equal(vo, v[:6])


def weld_case():
    nan = np.float32(np.nan)
    v = np.array([[0, 0, 0], [-0.0, 0, -0.0], [1, 0, 0], [0, 1, 0], [nan, 0, 0], [nan, 0, 0], [1, 0, 0], [0, 0, np.inf]],
                 np.float32)
    f = np.array([(0, 2, 3), (1, 2, 3), (0, 1, 2), (4, 5, 2), (6, 3, 2), (7, 7, 3), (6, 3, 1)], np.int32)
    return v, f


def test_oracle_weld_signed_zero_and_nan():
    v, f = weld_case()
    assert PP.weld_representatives(v).tolist() == [0, 0, 2, 3, 4, 5, 2, 7]
    vo, fo = PP.weld(v, f)
    # (0,1,2) and (6,3,2) collapse, (7,7,3) is degenerate as given; (1,2,3) becomes a duplicate of (0,2,3) and stays;
    # the two NaN vertices are not merged
    assert fo.tolist() == [[0, 1, 2], [0, 1, 2], [3, 4, 1], [1, 2, 0]]
    assert vo.view(np.uint32).tolist() == v[[0, 2, 3, 4, 5]].view(np.uint32).tolist()


def test_dmc_sheets_touch_at_vertices_so_components_are_edge_connected():
    """On a DMC mesh of a smoothed noise field, sheets touch at single vertices: joining faces by shared vertices would
    merge components that the edge relation keeps apart, and the shared-vertex rule takes faces of large components."""
    vol = noise_field(80, 0, 0.3)
    v, f = OD.dual_marching_cubes(vol)
    lab = PP.edge_components(f)
    assert len(np.unique(lab)) > PP.vertex_components(f, len(v))
    size = np.bincount(lab)
    large = size[lab] >= PP.min_faces_for(len(f))
    _, fo = PP.remove_floaters(v, f)
    assert len(fo) < int(large.sum())


def test_public_classes_reject_other_inputs():
    import hy3dgeo
    for cls in (hy3dgeo.FloaterRemover, hy3dgeo.DegenerateFaceRemover):
        for bad in ("mesh.ply", None, (np.zeros((3, 3)), np.zeros((1, 3), np.int32))):
            with pytest.raises(TypeError):
                cls()(bad)
        with pytest.raises(TypeError):
            cls().run_device(torch.zeros(3, 3), torch.zeros(1, 3, dtype=torch.int32))
    assert "FloaterRemover" in hy3dgeo.__all__ and "DegenerateFaceRemover" in hy3dgeo.__all__
    with pytest.raises(ImportError):
        from hy3dgeo import FaceReducer  # noqa: F401


# ---- GPU ------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def dev():
    return torch.device("cuda:0")


@pytest.fixture(scope="module")
def ctx(dev):
    from hy3dgeo import _lib
    return _lib.get_context(dev)


def gpu(ctx, name, v, f, *args):
    vd = torch.from_numpy(np.ascontiguousarray(v, np.float32)).cuda()
    fd = torch.from_numpy(np.ascontiguousarray(f, np.int32)).cuda()
    vo, fo = getattr(ctx, name)(vd, fd, *args)
    return vo.cpu().numpy(), fo.cpu().numpy()


def assert_same(got, ref):
    (v, f), (vo, fo) = got, ref
    assert v.dtype == np.float32 and f.dtype == np.int32
    assert v.shape == vo.shape and np.array_equal(v.view(np.uint32), np.ascontiguousarray(vo, np.float32).view(np.uint32))
    assert f.shape == fo.shape and np.array_equal(f, fo)


def check_both(ctx, v, f, min_faces=None):
    mf = PP.min_faces_for(len(f)) if min_faces is None else min_faces
    assert_same(gpu(ctx, "mesh_remove_floaters", v, f, mf), PP.remove_floaters(v, f, mf))
    assert_same(gpu(ctx, "mesh_weld", v, f), PP.weld(v, f))


def hand_meshes():
    v, f, _ = sheet_with_tet_at_vertex()
    yield v, f, None
    v6 = np.random.default_rng(0).standard_normal((6, 3)).astype(np.float32)
    ft = np.array(tet(0, 1, 2, 3) + tet(0, 1, 4, 5), np.int32)
    yield v6, ft, 8
    yield v6, ft, 9
    v, f = grid_sheet(24)
    n = len(v)
    yield (np.concatenate([v, np.random.default_rng(1).standard_normal((11, 3)).astype(np.float32)]),
           np.concatenate([f, np.array(strip(5, n) + strip(2, n + 7), np.int32)]), None)
    yield np.arange(27, dtype=np.float32).reshape(9, 3), np.array([(0, 1, 2), (1, 0, 3), (0, 1, 4), (5, 1, 0), (6, 7, 8)],
                                                                   np.int32), 2
    v, f = weld_case()
    yield v, f, 2


@pytest.mark.gpu
def test_cuda_filters_on_hand_built_meshes(ctx):
    for v, f, mf in hand_meshes():
        check_both(ctx, v, f, mf)


@pytest.mark.gpu
@pytest.mark.parametrize("n,seed,q", [(24, 1, 0.5), (48, 2, 0.7), (64, 3, 0.3), (80, 0, 0.3)])
def test_cuda_filters_on_noise_field_meshes(ctx, n, seed, q):
    vol = noise_field(n, seed, q)
    for v, f in (mc_mesh(vol), OD.dual_marching_cubes(vol)):
        check_both(ctx, v, f)
    if n == 80:                                              # DMC components touching at a vertex: the shared-vertex rule bites
        v, f = OD.dual_marching_cubes(vol)
        assert len(np.unique(PP.edge_components(f))) > PP.vertex_components(f, len(v))


@pytest.mark.gpu
def test_cuda_weld_on_quantised_field_meshes(ctx):
    vol = quantised_field()
    for v, f in (mc_mesh(vol), OD.dual_marching_cubes(vol)):
        wv, wf = PP.weld(v, f)
        assert len(wf) < len(f) and len(wv) < len(v)        # coincident vertices are there to weld
        assert_same(gpu(ctx, "mesh_weld", v, f), (wv, wf))
        check_both(ctx, v, f)


def body_with_blobs(n=385):
    """a hollow, bumpy body and 60 small spheres, some of them apart (floaters): ~0.97 M marching-cubes faces at 385^3,
    the mesh size of BASELINE configs[2] (the field of tools/gpu_postprocess_bench.py)"""
    x = np.linspace(-1.01, 1.01, n, dtype=np.float32)
    X, Y, Z = np.meshgrid(x, x, x, indexing="ij")
    R = np.sqrt(X * X + Y * Y + Z * Z)
    d = np.minimum(0.62 + 0.1 * np.sin(20 * X) * np.sin(20 * Y) * np.sin(20 * Z) - R, R - 0.35)
    rng = np.random.default_rng(7)
    for c, r in zip(rng.uniform(-0.95, 0.95, (60, 3)), rng.uniform(0.008, 0.03, 60)):
        d = np.maximum(d, r - np.sqrt((X - c[0]) ** 2 + (Y - c[1]) ** 2 + (Z - c[2]) ** 2))
    return np.tanh(20 * d).astype(np.float32)


@pytest.mark.gpu
def test_cuda_filters_full_scale_mc_mesh_and_determinism(ctx, dev):
    from hy3dgeo.surface_extractors import MCSurfaceExtractor
    g = torch.from_numpy(body_with_blobs()).to(dev)
    v, f = MCSurfaceExtractor(cull_nonfinite=True).run_device(g, mc_level=0.0, bounds=1.01, octree_resolution=384)
    vn, fn = v.cpu().numpy(), f.cpu().numpy()
    assert len(fn) > 800_000
    mf = PP.min_faces_for(len(fn))
    ref = PP.remove_floaters(vn, fn, mf)
    assert len(np.unique(PP.edge_components(fn))) > 1 and len(ref[1]) < len(fn)
    runs = [ctx.mesh_remove_floaters(v, f, mf) for _ in range(2)]
    assert all(torch.equal(a, b) for a, b in zip(runs[0], runs[1]))
    assert_same(tuple(t.cpu().numpy() for t in runs[0]), ref)
    runs = [ctx.mesh_weld(v, f) for _ in range(2)]
    assert all(torch.equal(a, b) for a, b in zip(runs[0], runs[1]))
    assert_same(tuple(t.cpu().numpy() for t in runs[0]), PP.weld(vn, fn))


@pytest.mark.gpu
def test_cuda_filters_everything_removed_and_empty(ctx):
    v = np.random.default_rng(0).standard_normal((1200, 3)).astype(np.float32)
    f = np.arange(1200, dtype=np.int32).reshape(400, 3)      # 400 lone triangles, min_faces = 2
    for got in (gpu(ctx, "mesh_remove_floaters", v, f, PP.min_faces_for(400)), gpu(ctx, "mesh_weld", v, f[:, [0, 0, 1]])):
        assert got[0].shape == (0, 3) and got[1].shape == (0, 3)
    for name, args in (("mesh_remove_floaters", (0,)), ("mesh_weld", ())):
        got = gpu(ctx, name, v, np.zeros((0, 3), np.int32), *args)
        assert got[0].shape == (0, 3) and got[1].shape == (0, 3)


@pytest.mark.gpu
def test_cuda_filters_reject_out_of_range_faces(ctx):
    from hy3dgeo._lib import Hy3dError
    v, f = grid_sheet(24)
    for bad in (len(v), -1, 2 ** 31 - 1):
        fb = f.copy()
        fb[300, 1] = bad
        for name, args in (("mesh_remove_floaters", (5,)), ("mesh_weld", ())):
            with pytest.raises(Hy3dError, match="outside"):
                gpu(ctx, name, v, fb, *args)
    with pytest.raises(Hy3dError):
        gpu(ctx, "mesh_weld", np.zeros((0, 3), np.float32), f[:1])
    check_both(ctx, v, f)                                    # the context stays usable


@pytest.mark.gpu
def test_public_classes(dev):
    import hy3dgeo
    vol = quantised_field(40, 3)
    v, f = mc_mesh(vol)
    m = hy3dgeo.Latent2MeshOutput(mesh_v=v.copy(), mesh_f=f.copy())
    out = hy3dgeo.FloaterRemover()(m)
    assert isinstance(out, hy3dgeo.Latent2MeshOutput) and out is not m
    assert_same((out.mesh_v, out.mesh_f), PP.remove_floaters(v, f))
    out2 = hy3dgeo.DegenerateFaceRemover()(out)
    assert_same((out2.mesh_v, out2.mesh_f), PP.weld(*PP.remove_floaters(v, f)))
    assert np.array_equal(m.mesh_v, v) and np.array_equal(m.mesh_f, f)           # input untouched
    vd, fd = torch.from_numpy(v).to(dev), torch.from_numpy(f).to(dev)
    chained = hy3dgeo.DegenerateFaceRemover().run_device(*hy3dgeo.FloaterRemover().run_device(vd, fd))
    assert chained[0].is_cuda and chained[1].is_cuda
    assert_same(tuple(t.cpu().numpy() for t in chained), (out2.mesh_v, out2.mesh_f))
    trimesh = pytest.importorskip("trimesh")
    tm = trimesh.Trimesh(v, f, process=False)
    t_out = hy3dgeo.DegenerateFaceRemover()(hy3dgeo.FloaterRemover()(tm))
    assert isinstance(t_out, trimesh.Trimesh)
    assert_same((np.asarray(t_out.vertices, np.float32), np.asarray(t_out.faces, np.int32)), (out2.mesh_v, out2.mesh_f))
    assert len(tm.faces) == len(f)


@pytest.mark.gpu
def test_latents2mesh_export_and_postprocess_chain(dev):
    """latents2mesh -> export_to_trimesh -> FloaterRemover -> DegenerateFaceRemover, as the reference's front ends run it,
    equals the same chain through the numpy statements on the same mesh."""
    import hy3dgeo
    from hy3dgeo import weights as W
    cfg = W.MINI
    vae = hy3dgeo.B200ShapeVAE(cfg, W.synthetic_state_dict(cfg, seed=0), device=dev)
    vae.volume_decoder = hy3dgeo.HierarchicalVolumeDecoding()
    lat = vae(W.synthetic_latents(cfg, 1, 1234).to(dev))
    mesh = vae.latents2mesh(lat, bounds=1.01, mc_level=0.0, num_chunks=8000, octree_resolution=32, min_resolution=15,
                            mc_algo="mc", enable_pbar=False)[0]
    assert mesh is not None
    ex = hy3dgeo.export_to_trimesh(mesh, dev)
    out = hy3dgeo.DegenerateFaceRemover()(hy3dgeo.FloaterRemover()(ex))
    get = lambda m: ((np.asarray(m.vertices, np.float32), np.asarray(m.faces, np.int32)) if hasattr(m, "vertices")
                     else (m.mesh_v, m.mesh_f))
    ref = PP.weld(*PP.remove_floaters(*OMESH.export_clean(mesh.mesh_v, mesh.mesh_f, flip_winding=True)))
    assert len(ref[1]) > 0
    assert_same(get(out), ref)
