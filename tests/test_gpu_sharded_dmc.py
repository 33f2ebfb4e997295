"""GPU: dual marching cubes over a grid cut into slabs along axis 0 (``hy3d_dmc_count_slab`` / ``hy3d_dmc_emit_slab`` /
``hy3d_dmc_center``, ``DMCSurfaceExtractor.run_device`` on a ``SlabGrid``).  The slab entry points on hand-cut slabs, and
the extractor on the grids of the three sharded decoders with world sizes 2 and 3 on ONE device (processes sharing
cuda:0, gloo for the plumbing, as in tests/test_gpu_sharded_flash.py): the mesh must equal the whole grid's bit for bit,
on every rank, without the grid ever being gathered."""
import ctypes as C
import os
import socket
import traceback

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp

from oracle import dmc as OD
from oracle.mesh import assert_same_mesh

pytestmark = pytest.mark.gpu
ERR_ARG = -2


def noise(shape, seed):
    """Normal noise with exact zeros (outside) and NaNs (outside, NaN vertices on their rim)."""
    rng = np.random.default_rng(seed)
    g = rng.standard_normal(shape).astype(np.float32)
    g[rng.random(shape) < 0.15] = 0.0
    g[rng.random(shape) < 0.05] = np.nan
    return g


def _same(a: torch.Tensor, b: torch.Tensor) -> bool:
    """bit equality (NaNs included)"""
    return a.shape == b.shape and a.dtype == b.dtype and torch.equal(a.contiguous().view(torch.int32), b.contiguous().view(torch.int32))


def _same_mesh(a, b) -> bool:
    return a is not None and b is not None and _same(a[0], b[0]) and torch.equal(a[1], b[1])


def whole_dmc(ctx, g):
    nv, nf, _ = ctx.dmc_count(g)
    v = torch.empty((nv, 3), dtype=torch.float32, device=g.device)
    f = torch.empty((nf, 3), dtype=torch.int32, device=g.device)
    ctx.dmc_emit(v, f)
    return v, f


def sliced_dmc(ctx, g, planes):
    """The slab entry points on g cut at ``planes`` (slab r owns [planes[r], planes[r+1]) and reads two halo planes):
    pieces concatenated in slab order, boxes reduced, centred.  -> (verts, faces, per-slab (nV, nF))."""
    n0 = g.shape[0]
    vs, fs, counts, boxes, base = [], [], [], [], 0
    for x0, x1 in zip(planes, planes[1:]):
        slab = g[x0: min(x1 + 2, n0)]
        nv, nf, _ = ctx.dmc_count_slab(slab, x1 - x0, x0, n0)
        v = torch.empty((nv, 3), dtype=torch.float32, device=g.device)
        f = torch.empty((nf, 3), dtype=torch.int32, device=g.device)
        box = torch.empty(6, dtype=torch.int32, device=g.device)
        ctx.dmc_emit_slab(base, v, f, box)
        vs.append(v); fs.append(f); boxes.append(box); counts.append((nv, nf))
        base += nv
    b = torch.stack(boxes).cpu()
    v, f = torch.cat(vs), torch.cat(fs)
    ctx.dmc_center(v, b[:, :3].min(0).values.tolist() + b[:, 3:].max(0).values.tolist())
    return v, f, counts


def cuts_for(n0, seed):
    rng = np.random.default_rng(seed)
    out = [list(range(n0 + 1)),                                   # 1-plane slabs
           [0, 1, n0], [0, n0 - 2, n0], [0, 1, n0 - 2, n0]]       # cuts at planes 1 and N0 - 2
    for k in (2, 3):                                              # uneven cuts
        out.append([0] + sorted(rng.choice(np.arange(1, n0), size=min(k, n0 - 1), replace=False).tolist()) + [n0])
    return out


@pytest.fixture(scope="module")
def dev():
    return torch.device("cuda:0")


@pytest.fixture(scope="module")
def ctx(dev):
    from hy3dgeo import _lib
    return _lib.get_context(dev)


# rows of 97, 300, 600 and 1024 voxels: the 8-, 16- and 32-lane row layouts (4, 10, 19, 32 words)
@pytest.mark.parametrize("shape", [(7, 5, 97), (6, 4, 300), (5, 3, 600), (4, 3, 1024), (9, 6, 33)])
def test_slab_entry_points_concatenate_bit_exact(shape, ctx, dev):
    for s, vol in enumerate((noise(shape, sum(shape)), np.random.default_rng(1).integers(-2, 3, size=shape).astype(np.float32))):
        g = torch.from_numpy(vol).to(dev)
        whole = whole_dmc(ctx, g)
        assert_same_mesh(tuple(t.cpu().numpy() for t in whole), OD.dual_marching_cubes(vol))
        for planes in cuts_for(shape[0], s):
            v, f, _ = sliced_dmc(ctx, g, planes)
            assert _same_mesh((v, f), whole), (shape, s, planes)


def test_slab_without_vertices_still_emits_its_faces(ctx, dev):
    """A slab whose cube planes hold no vertex but whose last edge plane has sign changes along axis 0: its faces use the
    next slab's vertices only.  And a slab without any surface contributes empty pieces."""
    vol = noise((10, 6, 40), 3)
    vol[:3] = 1.0                                      # planes 0..2 inside: cube planes 0, 1 empty
    g = torch.from_numpy(vol).to(dev)
    whole = whole_dmc(ctx, g)
    v, f, counts = sliced_dmc(ctx, g, [0, 1, 2, 10])
    assert _same_mesh((v, f), whole)
    assert counts[0] == (0, 0) and counts[1][0] == 0 and counts[1][1] > 0
    assert_same_mesh((v.cpu().numpy(), f.cpu().numpy()), OD.dual_marching_cubes(vol))


def test_full_size_plane_cuts_bit_exact(ctx, dev):
    """A 385^3 field (a bumpy shell, NaN outside the band a sparse decoder visits) cut by plane_cuts over 3 ranks."""
    from hy3dgeo import parallel as P
    n = 385
    x = torch.linspace(-1.01, 1.01, n, device=dev)
    X, Y, Z = torch.meshgrid(x, x, x, indexing="ij")
    r = torch.sqrt(X * X + Y * Y + Z * Z)
    g = torch.tanh(20 * (0.7 + 0.08 * torch.sin(9 * X) * torch.cos(7 * Y) * torch.sin(5 * Z + 1) - r))
    g = torch.where(g.abs() < 0.95, g, torch.full_like(g, float("nan"))).contiguous()
    index = torch.nonzero(~torch.isnan(g).reshape(-1)).reshape(-1).to(torch.int32)
    planes, _, _ = P.plane_cuts(index, n, 3)
    whole = whole_dmc(ctx, g)
    v, f, counts = sliced_dmc(ctx, g, planes)
    assert len(whole[1]) > 1_000_000 and torch.isnan(whole[0]).any() and all(c[0] > 0 for c in counts)
    assert _same_mesh((v, f), whole)


def test_slab_arguments_rejected(ctx, dev):
    L = ctx.lib
    g = torch.zeros((8, 4, 4), device=dev)
    nv, nf, mm = C.c_int64(), C.c_int64(), (C.c_float * 3)()

    def rc(own, halo, plane0, n0g):
        return L.hy3d_dmc_count_slab(ctx.h, g.data_ptr(), own, halo, 4, 4, plane0, n0g, C.byref(nv), C.byref(nf), mm)
    assert rc(3, 2, -1, 10) == ERR_ARG                 # plane0 < 0
    assert rc(3, 0, 8, 10) == ERR_ARG                  # plane0 + own > n0_global
    assert b"plane0" in L.hy3d_last_error(ctx.h)
    assert rc(0, 2, 2, 10) == ERR_ARG                  # own < 1
    assert rc(3, 1, 2, 10) == ERR_ARG                  # halo missing: two planes follow the slab
    assert rc(3, 0, 6, 10) == ERR_ARG                  # halo missing: one plane follows the slab
    assert rc(3, 3, 2, 7) == ERR_ARG                   # halo past the grid's end
    assert rc(3, 2, 0, 1) == ERR_ARG                   # n0_global < 2
    assert rc(3, 2, 2, 10) == 0 and rc(3, 1, 6, 10) == 0 and rc(3, 0, 7, 10) == 0
    assert L.hy3d_dmc_emit(ctx.h, None, None) != 0      # the whole-grid emit refuses a slab count
    box = torch.empty(6, dtype=torch.int32, device=dev)
    assert L.hy3d_dmc_emit_slab(ctx.h, -1, None, None, box.data_ptr()) == ERR_ARG
    assert L.hy3d_dmc_center(ctx.h, None, -1, (C.c_int32 * 6)()) == ERR_ARG
    ctx.dmc_count(g)                                   # leave a whole-grid count behind


# ---- the extractor on SlabGrids, several processes -----------------------------------------------------------------
def _free_port():
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    return port


def _worker(rank, world, port, q):
    try:
        import torch.distributed as dist
        os.environ["MASTER_ADDR"] = "127.0.0.1"
        os.environ["MASTER_PORT"] = str(port)
        dist.init_process_group("gloo", rank=rank, world_size=world)
        import hy3dgeo
        from hy3dgeo import _lib, parallel as P, weights as W
        from hy3dgeo.surface_extractors import DMCSurfaceExtractor
        from hy3dgeo.volume_decoders import FlashVDMVolumeDecoding
        dev = torch.device("cuda:0")
        torch.cuda.set_device(dev)
        ctx = _lib.get_context(dev)
        dmc = DMCSurfaceExtractor()
        fails = []

        def check(name, cond):
            if not cond:
                fails.append(name)

        gather = P.SlabGrid.to_tensor

        def refuse(self):
            raise AssertionError("SlabGrid.to_tensor called: the grid was gathered")
        P.SlabGrid.to_tensor = refuse                 # any gather inside the extractor fails the comparison below

        def compare(tag, grid):
            check(f"{tag}: SlabGrid", isinstance(grid, P.SlabGrid))
            ref = gather(grid)
            check(f"{tag}: shape", tuple(grid.shape) == tuple(ref.shape))
            for b in range(len(grid)):
                check(f"{tag}: mesh {b}", _same_mesh(dmc.run_device(grid[b]), dmc.run_device(ref[b])))
            outs = dmc(grid)
            check(f"{tag}: plugin call", all(o is not None for o in outs))

        mini = W.MINI
        vae = hy3dgeo.B200ShapeVAE(mini, W.sparsify_field(W.synthetic_state_dict(mini, seed=0), mini, 4, 4.0, 0.3), device=dev)
        lat = vae(W.synthetic_latents(mini, 2, 1234).to(dev))
        base = dict(bounds=1.01, mc_level=0.0, num_chunks=8000, enable_pbar=False)
        # dense slabs without a halo: extract_mesh_sharded's halo exchange
        grid = P.ShardedVanillaVolumeDecoder()(lat, vae.geo_decoder, octree_resolution=21, **base)
        compare("vanilla", grid)
        check("vanilla: no halo", not grid.with_halo)
        sparse = dict(base, octree_resolution=64, min_resolution=15)
        compare("hierarchical", P.ShardedHierarchicalVolumeDecoding()(lat, vae.geo_decoder, **sparse))
        compare("flash mean", P.ShardedFlashVDMVolumeDecoding("mean")(lat, vae.geo_decoder, **sparse))
        turbo = W.MINI_TURBO
        vae_t = hy3dgeo.B200ShapeVAE(turbo, W.sparsify_field(W.synthetic_state_dict(turbo, seed=0), turbo, 2, 60.0, -16.0), device=dev)
        lat_t = vae_t(W.synthetic_latents(turbo, 2, 1234).to(dev))
        compare("flash merge", P.ShardedFlashVDMVolumeDecoding("merge")(lat_t, vae_t.geo_decoder, **sparse))

        # latents2mesh with enable_flashvdm_decoder()'s defaults (mc_algo='dmc'), the decoder swapped for the sharded one
        vae.enable_flashvdm_decoder()
        check("defaults select dmc", isinstance(vae.surface_extractor, DMCSurfaceExtractor))
        outs_ref = vae.latents2mesh(lat[:1], **sparse)
        vae.volume_decoder = P.ShardedFlashVDMVolumeDecoding()
        outs = vae.latents2mesh(lat[:1], **sparse)
        check("latents2mesh on every rank", len(outs) == 1 and outs[0] is not None and outs_ref[0] is not None
              and np.array_equal(outs[0].mesh_f, outs_ref[0].mesh_f)
              and np.array_equal(outs[0].mesh_v.view(np.uint32), outs_ref[0].mesh_v.view(np.uint32)))

        # hand-made SlabGrids: no sign change anywhere -> None on every rank; a rank without surface -> empty pieces
        n = 24
        x0, x1 = P.slab_planes(n, rank, world)
        flat = -torch.ones((n, n, n), device=dev)
        check("no sign change -> None", dmc(P.SlabGrid([flat[x0:x1].clone()], x0, x1 - x0, (n, n, n), False)) == [None])
        try:
            dmc.run_device(P.SlabGrid([flat[x0:x1].clone()], x0, x1 - x0, (n, n, n), False))
            check("no sign change raises", False)
        except RuntimeError:
            pass
        c = torch.linspace(-1, 1, n, device=dev)
        X, Y, Z = torch.meshgrid(c, c, c, indexing="ij")
        ball = (0.3 - torch.sqrt((X - 0.6) ** 2 + Y ** 2 + Z ** 2)).contiguous()     # surface in the last slab only
        nv0, nf0, _ = ctx.dmc_count_slab(ball[x0: min(x1 + 2, n)].contiguous(), x1 - x0, x0, n)
        if rank == 0:
            check("rank 0 has no surface", nv0 == 0 and nf0 == 0)
        mesh = dmc.run_device(P.SlabGrid([ball[x0:x1].clone()], x0, x1 - x0, (n, n, n), False))
        check("empty pieces", _same_mesh(mesh, whole_dmc(ctx, ball)))
        ctx.check_watchdog()
        q.put((rank, fails))
        dist.destroy_process_group()
    except Exception:
        q.put((rank, ["EXCEPTION: " + traceback.format_exc()]))


@pytest.mark.parametrize("world", [2, 3])
def test_dmc_extractor_on_slab_grids_without_gather(world):
    mctx = mp.get_context("spawn")
    q = mctx.Queue()
    port = _free_port()
    procs = [mctx.Process(target=_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    results = dict(q.get(timeout=900) for _ in range(world))
    for p in procs:
        p.join(timeout=60)
    assert results == {r: [] for r in range(world)}, results
