"""Marching cubes with the asymptotic decider on ambiguous faces (``face_rule="asymptotic"``, hy3dgeo.h
hy3d_set_mc_face_rule): the generated table against the oracle's run-time loop tracing, hand-built cubes, closed and
consistently oriented meshes on noise, and on the GPU the kernels bit-exact against the oracle in every row layout, in
slabs and on the configs[2] 385^3 field.  A skimage-gated part compares face count and Euler characteristic with
Lewiner on fields whose ambiguous cubes are all MC33 case 3 (golden file made by tools/make_skimage_golden.py)."""
import importlib.util
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

from oracle import mc as OM, mc_face_rule as OF
from oracle.mesh import assert_same_mesh, bits_equal

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "hunyuan3d-2_b200", "csrc")
SKIMAGE_GOLD = os.path.join(ROOT, "tests", "golden", "skimage_mc_face_rule.npz")
CORNERS = [(0, 0, 0), (1, 0, 0), (1, 1, 0), (0, 1, 0), (0, 0, 1), (1, 0, 1), (1, 1, 1), (0, 1, 1)]   # (dx, dy, dz)


def _tool(name):
    spec = importlib.util.spec_from_file_location(name, os.path.join(ROOT, "tools", name + ".py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


def _array(src, name):
    body = re.search(name + r"\[[^=]*=\s*\{(.*?)\};", src, re.S).group(1)
    return [int(v) for v in re.findall(r"-?\d+", body)]


def decider_tables():
    src = open(os.path.join(CSRC, "mc_tables_decider.inc")).read()
    row = int(re.search(r"#define HY3D_MC_DEC_ROW (\d+)", src).group(1))
    faces = np.array(_array(src, "hy3d_mc_face_corner")).reshape(6, 4)
    amb = np.array(_array(src, "hy3d_mc_amb_faces"))
    first = np.array(_array(src, "hy3d_mc_dec_first"))
    tri = np.array(_array(src, "hy3d_mc_dec_tri")).reshape(-1, row)
    return faces, amb, first, tri


def cube(values):
    """2x2x2 volume with corner m (tools/gen_mc_tables.py numbering) = values[m]."""
    vol = np.empty((2, 2, 2), np.float32)
    for m, (dx, dy, dz) in enumerate(CORNERS):
        vol[dz, dy, dx] = values[m]
    return vol


def components(faces):
    parent = {}

    def find(x):
        while parent.setdefault(x, x) != x:
            x = parent[x]
        return x
    for a, b, c in faces:
        parent[find(b)] = find(a)
        parent[find(c)] = find(a)
    return len({find(x) for x in np.unique(faces)})


def ambiguous_face_stats(vol, level):
    """(ambiguous grid faces, those whose inside corners connect) over every face of the grid's cubes, by the contract:
    d = v - level in float32, connect iff d_a d_c > d_b d_d in float64 for inside diagonal (a, c)."""
    d = np.asarray(vol, np.float32) - np.float32(level)
    n_amb = n_con = 0
    for axis in range(3):
        g = np.moveaxis(d, axis, 0)
        for s in range(0, g.shape[0], 16):
            p = g[s:s + 16].astype(np.float64)
            c00, c10, c01, c11 = p[:, :-1, :-1], p[:, 1:, :-1], p[:, :-1, 1:], p[:, 1:, 1:]
            i00, i10, i01, i11 = c00 > 0, c10 > 0, c01 > 0, c11 > 0
            amb = (i00 == i11) & (i10 == i01) & (i00 != i10)
            diag_a, diag_b = c00 * c11, c10 * c01
            con = amb & np.where(i00, diag_a > diag_b, diag_b > diag_a)
            n_amb += int(amb.sum())
            n_con += int(con.sum())
    return n_amb, n_con


# ------------------------------------------------------------------------------------------------------- CPU: tables
def test_decider_table_rows_equal_oracle_tracing():
    """Every case, every decision index: the generated row is what the oracle traces at run time with that face mask;
    decision index 0 is the sign-rule row of mc_tables.inc."""
    faces, amb, first, tri = decider_tables()
    assert faces.tolist() == [[0, 4, 7, 3], [1, 2, 6, 5], [0, 1, 5, 4], [2, 3, 7, 6], [0, 3, 2, 1], [4, 5, 6, 7]]
    src = open(os.path.join(CSRC, "mc_tables.inc")).read()
    sign = np.array(_array(src, "hy3d_mc_tri_table")).reshape(256, -1)
    n_rows = 0
    for cs in range(256):
        ins = [[(cs >> c) & 1 for c in f] for f in faces]
        want_amb = [f for f in range(6) if ins[f][0] == ins[f][2] and ins[f][1] == ins[f][3] and ins[f][0] != ins[f][1]]
        assert amb[cs] == sum(1 << f for f in want_amb), cs
        assert first[cs] == n_rows, cs
        for dec in range(1 << len(want_amb)):
            connect = sum(1 << f for q, f in enumerate(want_amb) if (dec >> q) & 1)
            row = tri[first[cs] + dec]
            got = row[1:1 + 3 * row[0]].reshape(-1, 3)
            assert np.array_equal(got, OF.cube_triangles(cs, connect)), (cs, dec)
            assert (row[1 + 3 * row[0]:] == -1).all()
        assert np.array_equal(tri[first[cs]][:sign.shape[1]], sign[cs])
        n_rows += 1 << len(want_amb)
    assert n_rows == len(tri)


def test_tables_regenerate_byte_identical(tmp_path):
    _tool("gen_mc_tables").main(str(tmp_path))
    for name in ("mc_tables.inc", "dmc_tables.inc", "mc_tables_decider.inc"):
        assert (tmp_path / name).read_bytes() == open(os.path.join(CSRC, name), "rb").read(), name


# -------------------------------------------------------------------------------------------- CPU: hand-built cubes
def mesh_of(values, rule, level=0.0):
    v, f = OF.marching_cubes_raw(cube(values), level, rule)
    return len(f), components(f) if len(f) else 0


@pytest.mark.parametrize("values, level, want", [
    ([2, -1, 2, -1, -1, -1, -1, -1], 0.0, (4, 1)),              # MC33 case 3, 2 * 2 > 1 * 1: connected
    ([0.5, -1, 0.5, -1, -1, -1, -1, -1], 0.0, (2, 2)),          # 0.25 < 1: separated
    ([2.3, -0.7, 2.3, -0.7, -1, -1, -1, -1], 0.3, (4, 1)),      # d = v - level: 4 > 1
    ([1.3, -0.7, 1.3, -0.7, -1, -1, -1, -1], 0.3, (2, 2)),      # d: 1 * 1 == (-1) * (-1): a tie is separated
    ([2, -1, 0.5, -1, -1, -1, -1, -1], 0.0, (2, 2)),            # tie 2 * 0.5 == 1
    ([2, np.nan, 2, -1, -1, -1, -1, -1], 0.0, (2, 2)),          # NaN corner counts outside; NaN product: separated
    ([2, -1, 2, -1, -3, 0.5, -3, 0.5], 0.0, (6, 3)),            # MC33 case 13, only face 4 (corners 0-2) connects
    ([4, -1, 0.5, -1, -1, 0.5, -1, 0.5], 0.0, (10, 1)),         # case 13, the three faces at corner 0 connect
])
def test_hand_built_cubes(values, level, want):
    assert mesh_of(values, "asymptotic", level) == want
    n_in = int((np.array(values) > level).sum())
    assert mesh_of(values, "sign", level) == (n_in, n_in)         # the sign rule cuts off each inside corner


# ---------------------------------------------------------------------------------------------- CPU: noise meshes
def padded_noise(shape, seed, level):
    """Noise with exact level values and NaNs, inside an outside border so the surface is closed."""
    rng = np.random.default_rng(seed)
    vol = np.full(shape, level - 1.0, np.float32)
    inner = rng.standard_normal(tuple(s - 2 for s in shape)).astype(np.float32)
    inner[rng.random(inner.shape) < 0.05] = level
    inner[rng.random(inner.shape) < 0.01] = np.nan
    vol[1:-1, 1:-1, 1:-1] = inner
    return vol


@pytest.mark.parametrize("level", [0.0, 0.3])
def test_noise_mesh_closed_oriented_same_vertices(level):
    vol = padded_noise((30, 31, 33), 5, level)
    n_amb, n_con = ambiguous_face_stats(vol, level)
    assert n_con > 500 and n_amb - n_con > 500                     # both decisions occur many times
    vs, fs = OF.marching_cubes_raw(vol, level, "sign")
    va, fa = OF.marching_cubes_raw(vol, level, "asymptotic")
    assert bits_equal(va, vs)
    assert len(fa) != len(fs)
    # closed and consistently oriented: every directed edge a -> b is matched by one b -> a (as a multiset: where two
    # cubes' fans meet, a welded mesh can use an edge four times, under the sign rule too)
    d = np.concatenate([fa[:, [0, 1]], fa[:, [1, 2]], fa[:, [2, 0]]]).astype(np.int64)
    assert np.array_equal(np.sort(d[:, 0] * len(va) + d[:, 1]), np.sort(d[:, 1] * len(va) + d[:, 0]))


# ------------------------------------------------------------------------------------------------ CPU: interfaces
def test_extractor_face_rule_argument():
    from hy3dgeo.surface_extractors import MCSurfaceExtractor
    assert MCSurfaceExtractor().face_rule == "sign"
    assert MCSurfaceExtractor(face_rule="asymptotic").face_rule == "asymptotic"
    for bad in ("lewiner", "Sign", None, 1):
        with pytest.raises(ValueError):
            MCSurfaceExtractor(face_rule=bad)


def test_setter_exported_and_header_strict_c99(tmp_path):
    from hy3dgeo import _lib
    assert hasattr(_lib.load_library(), "hy3d_set_mc_face_rule") and "hy3d_set_mc_face_rule" in _lib.SYMBOLS
    if shutil.which("gcc") is None:
        pytest.skip("no C compiler")
    src = tmp_path / "rule.c"
    src.write_text("#include <hy3dgeo.h>\nint f(hy3d_ctx* c) { return hy3d_set_mc_face_rule(c, HY3D_MC_FACE_ASYMPTOTIC) + "
                   "HY3D_MC_FACE_SIGN; }\n")
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Wextra", "-Werror", "-pedantic", "-fsyntax-only", "-I",
                           os.path.join(ROOT, "include"), str(src)])


def test_case3_fields_have_only_case3_ambiguity():
    """The skimage comparison fields: every cube with an ambiguous face is MC33 case 3 (two inside corners, one ambiguous
    face), and both decisions occur."""
    _, amb, _, _ = decider_tables()
    for name, (vol, level) in _tool("make_skimage_golden").face_rule_fields().items():
        cases = OM.cube_cases(vol, level).ravel()
        hit = cases[amb[cases] != 0]
        assert len(hit) > 100, name
        assert all(bin(int(c)).count("1") == 2 and bin(int(amb[c])).count("1") == 1 for c in np.unique(hit)), name
        n_amb, n_con = ambiguous_face_stats(vol, level)
        assert 0 < n_con < n_amb, name


# ------------------------------------------------------------------------------------------- skimage (golden-gated)
def _skimage_check(name, v, f, g):
    st = _tool("make_skimage_golden").mesh_stats(v, f)
    assert st["V"] == int(g[name + "_V"]), name
    assert st["F"] == int(g[name + "_F"]) and st["euler"] == int(g[name + "_euler"]), (name, st)


@pytest.mark.skipif(not os.path.exists(SKIMAGE_GOLD), reason="tests/golden/skimage_mc_face_rule.npz absent: scikit-image "
                    "unavailable offline")
def test_oracle_asymptotic_vs_skimage_case3():
    g = np.load(SKIMAGE_GOLD)
    for name, (vol, level) in _tool("make_skimage_golden").face_rule_fields().items():
        v, f, _, _ = OF.marching_cubes(vol, level, face_rule="asymptotic")
        _skimage_check(name, v, f, g)


# ---------------------------------------------------------------------------------------------------------- GPU
@pytest.fixture(scope="module")
def ctx():
    import torch
    from hy3dgeo import _lib
    return _lib.get_context(torch.device("cuda:0"))


def device_mc(ctx, g, level, rule):
    import torch
    nv, nf, _ = ctx.mc_count(g, level, rule)
    v = torch.empty((nv, 3), dtype=torch.float32, device=g.device)
    f = torch.empty((nf, 3), dtype=torch.int32, device=g.device)
    ctx.mc_emit((1, 1, 1), (1, 1, 1), (0, 0, 0), v, f)
    return v.cpu().numpy(), f.cpu().numpy()


def edge_field(shape, seed):
    """Noise (about half of all edges cross 0) with exact zeros and NaNs."""
    rng = np.random.default_rng(seed)
    vol = rng.standard_normal(shape).astype(np.float32)
    vol[rng.random(shape) < 0.05] = 0.0
    vol[rng.random(shape) < 0.01] = np.nan
    return vol


@pytest.mark.gpu
@pytest.mark.parametrize("n2", [97, 300, 600, 1024])             # 4 / 10 / 19 / 32 words: 8-, 16-, 32-, 32-lane rows
def test_gpu_bit_exact_vs_oracle(ctx, n2):
    """Noise rows overflow the 256-entry emit work lists several times per warp."""
    import torch
    vol = edge_field((6, 7, n2), n2)
    g = torch.from_numpy(vol).cuda()
    for level in (0.0, 0.3):
        ref = OF.marching_cubes_raw(vol, level, "asymptotic")
        assert_same_mesh(device_mc(ctx, g, level, "asymptotic"), ref)
        assert_same_mesh(device_mc(ctx, g, level, "sign"), OF.marching_cubes_raw(vol, level, "sign"))
        assert len(ref[1]) != len(OF.marching_cubes_raw(vol, level, "sign")[1])


@pytest.mark.gpu
def test_gpu_case3_fields(ctx):
    import torch
    for name, (vol, level) in _tool("make_skimage_golden").face_rule_fields().items():
        assert_same_mesh(device_mc(ctx, torch.from_numpy(vol).cuda(), level, "asymptotic"),
                         OF.marching_cubes_raw(vol, level, "asymptotic"))


@pytest.mark.gpu
def test_gpu_slabs_concatenate_to_whole_grid(ctx):
    import torch
    from hy3dgeo.parallel import MC_HALO, slab_planes
    from hy3dgeo.surface_extractors import MCSurfaceExtractor
    vol = edge_field((45, 33, 300), 3)
    out = torch.from_numpy(vol).cuda()
    N = vol.shape[0]
    ext = MCSurfaceExtractor(face_rule="asymptotic")
    kw = dict(bounds=1.01, octree_resolution=N - 1)
    v_ref, f_ref = ext.run_device(out, mc_level=0.0, **kw)
    assert_same_mesh((v_ref.cpu().numpy(), f_ref.cpu().numpy()),
                     OF.mc_surface_extract(vol, mc_level=0.0, face_rule="asymptotic", **kw))
    vs, fs, base = [], [], 0
    for r in range(5):
        x0, x1 = slab_planes(N, r, 5)
        slab = out[x0:min(x1 + MC_HALO, N)].contiguous()
        nv, nf, _ = ext.count_slab(slab, x1 - x0, 0.0)
        v, f = ext.emit_slab(nv, nf, x0, base, **kw)
        vs.append(v); fs.append(f); base += nv
    v, f = torch.cat(vs), torch.cat(fs)
    assert torch.equal(v.view(torch.int32), v_ref.view(torch.int32)) and torch.equal(f, f_ref)


@pytest.mark.gpu
def test_gpu_mixed_rules_refused(ctx):
    import torch
    from hy3dgeo import _lib
    g = torch.from_numpy(edge_field((5, 6, 40), 1)).cuda()
    for count_rule, emit_rule in (("sign", "asymptotic"), ("asymptotic", "sign")):
        nv, nf, _ = ctx.mc_count(g, 0.0, count_rule)
        v = torch.empty((nv, 3), dtype=torch.float32, device="cuda")
        f = torch.empty((nf, 3), dtype=torch.int32, device="cuda")
        ctx.set_mc_face_rule(emit_rule)
        with pytest.raises(_lib.Hy3dError, match="face rule"):
            ctx.mc_emit((1, 1, 1), (1, 1, 1), (0, 0, 0), v, f)
    with pytest.raises(ValueError):
        ctx.set_mc_face_rule("lewiner")
    with pytest.raises(_lib.Hy3dError):                              # the C-ABI itself refuses an unknown rule
        ctx._check(ctx.lib.hy3d_set_mc_face_rule(ctx.h, 7), "hy3d_set_mc_face_rule")
    assert_same_mesh(device_mc(ctx, g, 0.0, "asymptotic"), OF.marching_cubes_raw(g.cpu().numpy(), 0.0, "asymptotic"))


@pytest.mark.gpu
def test_gpu_configs2_octree384_field(ctx):
    """configs[2]: the 385^3 NaN-bearing grid HierarchicalVolumeDecoding makes at octree 384 from the full model and the
    benchmark's sparse field; the asymptotic mesh is bit-exact against the oracle."""
    import torch
    import hy3dgeo
    from bench import SPARSE_FULL
    from hy3dgeo import weights as W
    from hy3dgeo.surface_extractors import MCSurfaceExtractor
    from hy3dgeo.volume_decoders import HierarchicalVolumeDecoding
    dev = torch.device("cuda:0")
    cfg = W.FULL
    sd = W.sparsify_field(W.synthetic_state_dict(cfg, seed=0), cfg, **SPARSE_FULL)
    vae = hy3dgeo.B200ShapeVAE(cfg, sd, device=dev)
    lat = vae(W.synthetic_latents(cfg, 1, 1234).to(dev))
    out = HierarchicalVolumeDecoding()(lat, vae.geo_decoder, bounds=1.01, num_chunks=8000, mc_level=0.0,
                                       octree_resolution=384, enable_pbar=False)[0]
    ctx.check_watchdog()
    assert out.shape == (385, 385, 385)
    grid = out.cpu().numpy()
    kw = dict(mc_level=0.0, bounds=1.01, octree_resolution=384)
    v, f = MCSurfaceExtractor(face_rule="asymptotic").run(out, **kw)
    assert_same_mesh((v, f), OF.mc_surface_extract(grid, face_rule="asymptotic", **kw))
    n_amb, n_con = ambiguous_face_stats(grid, 0.0)
    _, f_sign = MCSurfaceExtractor().run(out, **kw)
    print(f"\nconfigs[2] 385^3: {n_amb} ambiguous faces, {n_con} connect; faces asymptotic {len(f)} vs sign {len(f_sign)}")


@pytest.mark.gpu
@pytest.mark.skipif(not os.path.exists(SKIMAGE_GOLD), reason="tests/golden/skimage_mc_face_rule.npz absent: scikit-image "
                    "unavailable offline")
def test_cuda_asymptotic_vs_skimage_case3(ctx):
    import torch
    g = np.load(SKIMAGE_GOLD)
    for name, (vol, level) in _tool("make_skimage_golden").face_rule_fields().items():
        _skimage_check(name, *device_mc(ctx, torch.from_numpy(vol).cuda(), level, "asymptotic"), g)
