"""Quadric edge-collapse decimation (``FaceReducer``): the numpy contract ``oracle/decimate.py`` on hand-built and
marching-cubes meshes on CPU; on the GPU ``hy3d_mesh_decimate`` and the public class bit-exact against it, from
hand-built meshes up to the full-scale 385^3 marching-cubes mesh after floater removal and welding."""
import numpy as np
import pytest
import torch

from oracle import decimate as D, dmc as OD, mesh as OMESH, postprocess as PP
from test_postprocess import body_with_blobs, grid_sheet, mc_mesh, noise_field, tet


# ---- helpers --------------------------------------------------------------------------------------------------------------
def edge_faces(f):
    """{(min, max): number of faces}"""
    e = np.sort(np.concatenate([f[:, [0, 1]], f[:, [1, 2]], f[:, [2, 0]]]), 1)
    k, c = np.unique(e, axis=0, return_counts=True)
    return {tuple(x): int(n) for x, n in zip(k, c)}


def assert_closed_oriented(f):
    """every edge in exactly two faces, and each directed edge in exactly one (consistent orientation)"""
    assert set(edge_faces(f).values()) == {2}
    d = np.concatenate([f[:, [0, 1]], f[:, [1, 2]], f[:, [2, 0]]])
    assert len(np.unique(d, axis=0)) == len(d)


def euler_per_component(v, f):
    lab = PP.edge_components(f)
    out = []
    for c in np.unique(lab):
        fc = f[lab == c]
        out.append(len(np.unique(fc)) - len(edge_faces(fc)) + len(fc))
    return sorted(out)


def normals(v, f):
    p = v.astype(np.float64)
    return np.cross(p[f[:, 1]] - p[f[:, 0]], p[f[:, 2]] - p[f[:, 0]])


def grid_axis(n):
    return np.linspace(-1.0, 1.0, n, dtype=np.float32)


def to_world(v, n):
    """marching-cubes vertices are in grid units: map to the [-1, 1] box of grid_axis(n)"""
    return (v.astype(np.float64) * (2.0 / (n - 1)) - 1.0)


def sphere_field(n=48, r=0.7):
    x = grid_axis(n)
    X, Y, Z = np.meshgrid(x, x, x, indexing="ij")
    return (r - np.sqrt(X * X + Y * Y + Z * Z)).astype(np.float32)


def torus_field(n=56, R=0.6, r=0.25):
    x = grid_axis(n)
    X, Y, Z = np.meshgrid(x, x, x, indexing="ij")
    return (r - np.sqrt((np.sqrt(X * X + Y * Y) - R) ** 2 + Z * Z)).astype(np.float32)


def octahedron():
    v = np.array([[1, 0, 0], [-1, 0, 0], [0, 1, 0], [0, -1, 0], [0, 0, 1], [0, 0, -1]], np.float32)
    f = np.array([(0, 2, 4), (2, 1, 4), (1, 3, 4), (3, 0, 4), (2, 0, 5), (1, 2, 5), (3, 1, 5), (0, 3, 5)], np.int32)
    return v, f


def tri_tube(rings=12, radius=0.05, length=2.0):
    """a closed thin tube of triangular cross-section: rings of 3 vertices, end caps of one triangle each"""
    ang = 2 * np.pi * np.arange(3) / 3
    v = np.array([(radius * np.cos(t), radius * np.sin(t), length * k / (rings - 1)) for k in range(rings) for t in ang],
                 np.float32)
    f = []
    for k in range(rings - 1):
        for i in range(3):
            a, b = 3 * k + i, 3 * k + (i + 1) % 3
            f += [(a, b, b + 3), (a, b + 3, a + 3)]
    f += [(0, 2, 1), (3 * rings - 3, 3 * rings - 2, 3 * rings - 1)]
    return v, np.array(f, np.int32)


def two_cones(k=10):
    """two closed cones whose apexes are the same vertex 0 (its faces form two fans)"""
    v, f = [[0, 0, 0]], []
    for s in (1, -1):
        base = len(v)
        ang = 2 * np.pi * np.arange(k) / k
        v += [[np.cos(t), np.sin(t), s * 1.5] for t in ang] + [[0, 0, s * 1.5]]
        c = base + k
        for i in range(k):
            r0, r1 = base + i, base + (i + 1) % k
            f += [(0, r0, r1), (c, r1, r0)] if s > 0 else [(0, r1, r0), (c, r0, r1)]
    return np.array(v, np.float32), np.array(f, np.int32)


# ---- CPU: the contract ------------------------------------------------------------------------------------------------------
def test_at_or_below_target_returns_the_input():
    v, f = grid_sheet(8)
    for T in (len(f), len(f) + 1, 10 ** 9):
        vo, fo, r = D.decimate(v, f, T)
        assert r == 0 and np.array_equal(vo.view(np.uint32), v.view(np.uint32)) and np.array_equal(fo, f)
    with pytest.raises(ValueError):
        D.decimate(v, f, 0)


def test_planar_sheet_keeps_its_boundary_and_plane():
    v, f = grid_sheet(24)
    vo, fo, r = D.decimate(v, f, 300)
    assert r > 0 and len(fo) in (299, 300)
    assert np.all(vo[:, 2] == 0)
    key = lambda p: tuple(p.view(np.uint32))
    border = [key(p) for p in v if p[0] in (0, 23) or p[1] in (0, 23)]
    out = {key(p): i for i, p in enumerate(vo)}
    assert all(b in out for b in border)                                       # bit-identical, never moved

    def boundary_edges(vv, ff):
        return {tuple(sorted((key(vv[a]), key(vv[b])))) for (a, b), c in edge_faces(ff).items() if c == 1}

    assert boundary_edges(vo, fo) == boundary_edges(v, f)


def test_tetrahedron_stays_and_octahedron_stops_at_the_degree_rules():
    v = np.random.default_rng(0).standard_normal((4, 3)).astype(np.float32)
    f = np.array(tet(0, 1, 2, 3), np.int32)
    if np.dot(np.cross(v[1] - v[0], v[2] - v[0]), v[3] - v[0]) > 0:
        v[[1, 2]] = v[[2, 1]]                                                  # outward faces
    vo, fo, r = D.decimate(v, f, 1)
    assert r == 0 and np.array_equal(fo, f) and np.array_equal(vo, v)
    v, f = octahedron()
    vo, fo, r = D.decimate(v, f, 1)
    # every collapse needs deg(a) + deg(b) - 4 >= 3 and wings of degree >= 4: the octahedron goes down to a tetrahedron
    assert len(fo) == 4 and len(vo) == 4 and r == 2
    assert_closed_oriented(fo)


def test_thin_tube_is_not_pinched():
    """collapsing an edge of a triangular cross-section would join two faces back to back: the link condition refuses"""
    v, f = tri_tube()
    ring = {tuple(sorted((3 * k + i, 3 * k + (i + 1) % 3))) for k in range(1, 11) for i in range(3)}
    common = lambda a, b, e: len({w for w in range(len(v)) if tuple(sorted((a, w))) in e and tuple(sorted((b, w))) in e})
    e = edge_faces(f)
    assert all(common(a, b, e) == 3 for a, b in ring)                          # the third ring vertex besides the wings
    trace = []
    vo, fo, r = D.decimate(v, f, 1, trace)
    assert r > 0 and len(fo) < len(f)
    for tv, tf, _ in trace:                                                    # every round: still a closed sphere
        assert_closed_oriented(tf)
        assert euler_per_component(tv, tf) == [2]


def test_two_cones_sharing_a_vertex_keep_it():
    v, f = two_cones()
    vo, fo, r = D.decimate(v, f, 1)
    assert r > 0 and len(fo) < len(f)
    apex = np.nonzero((vo == 0).all(1))[0]
    assert len(apex) == 1
    assert len(np.unique(PP.edge_components(fo))) == 2
    assert all(np.isin(apex[0], fo[PP.edge_components(fo) == c]) for c in np.unique(PP.edge_components(fo)))


# distance of every decimated vertex from the analytic surface, in units of the grid's cell: fixed from a CPU run of the
# oracle at F / 10 (largest distance 0.066 cells on the sphere, 0.091 on the torus; 0.007 and 0.017 before decimation),
# with margin
SURFACE_BOUND_CELLS = 0.15


@pytest.mark.parametrize("name,field,dist,euler", [
    ("sphere", sphere_field, lambda p: np.abs(np.sqrt((p * p).sum(1)) - 0.7), [2]),
    ("torus", torus_field, lambda p: np.abs(np.sqrt((np.sqrt(p[:, 0] ** 2 + p[:, 1] ** 2) - 0.6) ** 2 + p[:, 2] ** 2) - 0.25),
     [0]),
])
def test_closed_mc_meshes_to_a_tenth(name, field, dist, euler):
    vol = field()
    n = vol.shape[0]
    v, f = mc_mesh(vol)
    assert_closed_oriented(f)
    assert euler_per_component(v, f) == euler
    T = len(f) // 10
    trace = []
    vo, fo, r = D.decimate(v, f, T, trace)
    assert len(fo) in (T - 1, T) and r == len(trace)
    assert_closed_oriented(fo)
    assert euler_per_component(vo, fo) == euler
    prev_v, prev_f = v, f
    for tv, tf, kept in trace:                       # no face turns against its normal before the round
        d = (normals(prev_v, prev_f)[kept] * normals(tv, tf)).sum(1)
        assert np.all(d > 0)
        prev_v, prev_f = tv, tf
    cell = 2.0 / (n - 1)
    assert dist(to_world(vo, n)).max() < SURFACE_BOUND_CELLS * cell


def test_face_reducer_rejects_other_inputs():
    import hy3dgeo
    from hy3dgeo.postprocessors import FaceReducer
    for bad in ("mesh.ply", None, (np.zeros((3, 3)), np.zeros((1, 3), np.int32))):
        with pytest.raises(TypeError):
            FaceReducer()(bad)
    with pytest.raises(TypeError):
        FaceReducer().run_device(torch.zeros(3, 3), torch.zeros(1, 3, dtype=torch.int32))
    m = hy3dgeo.Latent2MeshOutput(mesh_v=np.zeros((3, 3), np.float32), mesh_f=np.zeros((1, 3), np.int32))
    for bad in (0, -5):
        with pytest.raises(ValueError):
            FaceReducer()(m, max_facenum=bad)


# ---- GPU ------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def dev():
    return torch.device("cuda:0")


@pytest.fixture(scope="module")
def ctx(dev):
    from hy3dgeo import _lib
    return _lib.get_context(dev)


def gpu_decimate(ctx, v, f, T):
    vd = torch.from_numpy(np.ascontiguousarray(v, np.float32)).cuda()
    fd = torch.from_numpy(np.ascontiguousarray(f, np.int32)).cuda()
    vo, fo, r = ctx.mesh_decimate(vd, fd, T)
    return vo.cpu().numpy(), fo.cpu().numpy(), r


def assert_same(got, ref):
    (v, f, r), (vo, fo, ro) = got, ref
    assert v.dtype == np.float32 and f.dtype == np.int32
    assert r == ro
    assert v.shape == vo.shape and np.array_equal(v.view(np.uint32), np.ascontiguousarray(vo, np.float32).view(np.uint32))
    assert f.shape == fo.shape and np.array_equal(f, fo)


def check(ctx, v, f, T):
    assert_same(gpu_decimate(ctx, v, f, T), D.decimate(v, f, T))


@pytest.mark.gpu
def test_cuda_decimate_hand_built_meshes(ctx):
    v4 = np.random.default_rng(0).standard_normal((4, 3)).astype(np.float32)
    for v, f, T in [(*grid_sheet(24), 300), (*grid_sheet(8), 500), (v4, np.array(tet(0, 1, 2, 3), np.int32), 1),
                    (*octahedron(), 1), (*tri_tube(), 1), (*two_cones(), 1), (*grid_sheet(24), 1)]:
        check(ctx, v, f, T)


@pytest.mark.gpu
@pytest.mark.parametrize("n,seed,q", [(24, 1, 0.5), (48, 2, 0.7), (80, 0, 0.3)])
def test_cuda_decimate_noise_field_meshes(ctx, n, seed, q):
    vol = noise_field(n, seed, q)
    for v, f in (mc_mesh(vol), OD.dual_marching_cubes(vol)):
        for T in (len(f) // 2, len(f) // 20):
            check(ctx, v, f, T)


@pytest.mark.gpu
def test_cuda_decimate_closed_mc_meshes(ctx):
    for field in (sphere_field, torus_field):
        v, f = mc_mesh(field())
        check(ctx, v, f, len(f) // 10)


@pytest.mark.gpu
def test_cuda_decimate_medium_mesh(ctx):
    v, f = mc_mesh(body_with_blobs(161))
    assert 150_000 <= len(f) <= 200_000
    check(ctx, v, f, 10_000)


@pytest.mark.gpu
def test_cuda_decimate_full_scale_and_determinism(ctx, dev):
    from hy3dgeo.surface_extractors import MCSurfaceExtractor
    g = torch.from_numpy(body_with_blobs()).to(dev)
    v, f = MCSurfaceExtractor(cull_nonfinite=True).run_device(g, mc_level=0.0, bounds=1.01, octree_resolution=384)
    v, f = ctx.mesh_weld(*ctx.mesh_remove_floaters(v, f, PP.min_faces_for(f.shape[0])))
    vn, fn = v.cpu().numpy(), f.cpu().numpy()
    assert len(fn) > 800_000
    runs = [ctx.mesh_decimate(v, f, 40_000) for _ in range(2)]
    assert torch.equal(runs[0][0], runs[1][0]) and torch.equal(runs[0][1], runs[1][1]) and runs[0][2] == runs[1][2]
    vo, fo, r = runs[0][0].cpu().numpy(), runs[0][1].cpu().numpy(), runs[0][2]
    assert len(fo) in (39_999, 40_000)
    e_in, e_out = edge_faces(fn), edge_faces(fo)
    assert euler_per_component(vo, fo) == euler_per_component(vn, fn)
    key = lambda p: tuple(p.view(np.uint32))
    bnd = lambda vv, ee: {tuple(sorted((key(vv[a]), key(vv[b])))) for (a, b), c in ee.items() if c == 1}
    assert bnd(vo, e_out) == bnd(vn, e_in)                                     # boundary edges preserved
    assert sum(c > 2 for c in e_out.values()) <= sum(c > 2 for c in e_in.values())
    assert_same((vo, fo, r), D.decimate(vn, fn, 40_000))


@pytest.mark.gpu
def test_cuda_decimate_errors_and_empty(ctx):
    from hy3dgeo._lib import Hy3dError
    v, f = grid_sheet(24)
    for bad in (len(v), -1, 2 ** 31 - 1):
        fb = f.copy()
        fb[300, 1] = bad
        for T in (100, 10_000):
            with pytest.raises(Hy3dError, match="outside"):
                gpu_decimate(ctx, v, fb, T)
    for T in (0, -1):
        with pytest.raises(Hy3dError):
            gpu_decimate(ctx, v, f, T)
    got = gpu_decimate(ctx, np.zeros((0, 3), np.float32), np.zeros((0, 3), np.int32), 10)
    assert got[0].shape == (0, 3) and got[1].shape == (0, 3) and got[2] == 0
    check(ctx, v, f, 300)                                                      # the context stays usable


@pytest.mark.gpu
def test_public_class(dev):
    import hy3dgeo
    from hy3dgeo.postprocessors import FaceReducer
    v, f = mc_mesh(noise_field(48, 2, 0.7))
    ref = D.decimate(v, f, 2000)
    m = hy3dgeo.Latent2MeshOutput(mesh_v=v.copy(), mesh_f=f.copy())
    out = FaceReducer()(m, max_facenum=2000)
    assert isinstance(out, hy3dgeo.Latent2MeshOutput) and out is not m
    assert_same((out.mesh_v, out.mesh_f, ref[2]), ref)
    assert np.array_equal(m.mesh_v, v) and np.array_equal(m.mesh_f, f)           # input untouched
    vd, fd = torch.from_numpy(v).to(dev), torch.from_numpy(f).to(dev)
    chained = FaceReducer().run_device(*hy3dgeo.DegenerateFaceRemover().run_device(
        *hy3dgeo.FloaterRemover().run_device(vd, fd)), max_facenum=2000)
    assert chained[0].is_cuda and chained[1].is_cuda
    host = FaceReducer()(hy3dgeo.DegenerateFaceRemover()(hy3dgeo.FloaterRemover()(m)), max_facenum=2000)
    assert_same((*[t.cpu().numpy() for t in chained], 0), (host.mesh_v, host.mesh_f, 0))
    vs, fs = mc_mesh(noise_field(24, 1, 0.5))
    assert len(fs) <= 40_000
    small = FaceReducer()(hy3dgeo.Latent2MeshOutput(mesh_v=vs, mesh_f=fs))     # default max_facenum: as given
    assert np.array_equal(small.mesh_f, fs) and np.array_equal(small.mesh_v.view(np.uint32), vs.view(np.uint32))
    trimesh = pytest.importorskip("trimesh")
    tm = trimesh.Trimesh(v, f, process=False)
    t_out = FaceReducer()(tm, max_facenum=2000)
    assert isinstance(t_out, trimesh.Trimesh)
    assert_same((np.asarray(t_out.vertices, np.float32), np.asarray(t_out.faces, np.int32), ref[2]), ref)
    assert len(tm.faces) == len(f)


@pytest.mark.gpu
def test_latents2mesh_export_and_postprocess_chain(dev):
    """latents2mesh -> export_to_trimesh -> FloaterRemover -> DegenerateFaceRemover -> FaceReducer, as the reference's
    front ends run it, equals the same chain through the numpy statements on the same mesh."""
    import hy3dgeo
    from hy3dgeo import weights as W
    from hy3dgeo.postprocessors import FaceReducer
    cfg = W.MINI
    vae = hy3dgeo.B200ShapeVAE(cfg, W.synthetic_state_dict(cfg, seed=0), device=dev)
    vae.volume_decoder = hy3dgeo.HierarchicalVolumeDecoding()
    lat = vae(W.synthetic_latents(cfg, 1, 1234).to(dev))
    mesh = vae.latents2mesh(lat, bounds=1.01, mc_level=0.0, num_chunks=8000, octree_resolution=32, min_resolution=15,
                            mc_algo="mc", enable_pbar=False)[0]
    assert mesh is not None
    ex = hy3dgeo.export_to_trimesh(mesh, dev)
    cleaned = PP.weld(*PP.remove_floaters(*OMESH.export_clean(mesh.mesh_v, mesh.mesh_f, flip_winding=True)))
    T = max(len(cleaned[1]) // 3, 1)
    out = FaceReducer()(hy3dgeo.DegenerateFaceRemover()(hy3dgeo.FloaterRemover()(ex)), max_facenum=T)
    get = lambda m: ((np.asarray(m.vertices, np.float32), np.asarray(m.faces, np.int32)) if hasattr(m, "vertices")
                     else (m.mesh_v, m.mesh_f))
    ref = D.decimate(*cleaned, T)
    assert len(ref[1]) < len(cleaned[1])
    assert_same((*get(out), ref[2]), ref)
