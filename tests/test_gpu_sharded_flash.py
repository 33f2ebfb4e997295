"""GPU: ShardedFlashVDMVolumeDecoding with world sizes 2 and 3 on ONE device (processes sharing cuda:0, gloo for the
plumbing, as in tests/test_gpu_sharded.py).  Uneven partitions on purpose: 64 mini-grids over 3 ranks, spatial bins cut
by rank boundaries and selected by both neighbours.  Grid, visited counts and meshes must equal the single-process
FlashVDMVolumeDecoding's bit for bit."""
import ctypes as C
import os
import socket
import traceback

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp

pytestmark = pytest.mark.gpu

# (config name, sparsify_field arguments, topk_mode, call kwargs): the field settings of the goldens of each model
CASES = [
    ("MINI", (4, 4.0, 0.3), "mean", dict(octree_resolution=64, min_resolution=15)),            # three levels
    ("MINI_TURBO", (2, 60.0, -16.0), "merge", dict(octree_resolution=64, min_resolution=15)),
    ("FULL", (2, 6.0, 1.5), "mean", dict(octree_resolution=64, min_resolution=15)),            # T = 1024 of 3072 tokens
    ("MINI", (4, 4.0, 0.3), "mean", dict(octree_resolution=35, min_resolution=8, mini_grid_num=3)),   # 9^3 level 0, 27 groups
]


def _free_port():
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    return port


def _same(a: torch.Tensor, b: torch.Tensor) -> bool:
    """bit equality (NaNs included)"""
    return a.shape == b.shape and a.dtype == b.dtype and torch.equal(a.contiguous().view(torch.int32), b.contiguous().view(torch.int32))


def _same_mesh(a, b) -> bool:
    return a is not None and b is not None and _same(a[0], b[0]) and torch.equal(a[1], b[1])


def _entry_point_checks(ctx, dev, check):
    from hy3dgeo import _lib, parallel as P
    L, ERR_ARG = ctx.lib, -2
    i32 = torch.zeros(1024, dtype=torch.int32, device=dev)
    f32 = torch.zeros(1024, dtype=torch.float32, device=dev)
    c, _keep = ctx._coords(cell=(0.1, 0.1, 0.1), bmin=(-1.0, -1.0, -1.0))
    for g0, g1 in [(-1, 2), (3, 3), (5, 4), (0, 217)]:
        rc = L.hy3d_flash_select_range(ctx.h, i32.data_ptr(), 8, 8, 8, 8, C.byref(c), i32.data_ptr(), 216, g0, g1, 4, 0)
        check(f"select_range [{g0}, {g1}) rejected", rc == ERR_ARG)
    rc = L.hy3d_decode_flash_values(ctx.h, i32.data_ptr(), 100, 8, 8, 8, C.byref(c), i32.data_ptr(), f32.data_ptr())
    check("decode_flash_values: unaligned length rejected", rc == ERR_ARG)
    for base, ln in [(-1, 5), (0, -1)]:
        rc = L.hy3d_scatter_window(ctx.h, i32.data_ptr(), f32.data_ptr(), 10, base, ln, f32.data_ptr())
        check(f"scatter_window base {base} len {ln} rejected", rc == ERR_ARG)
    # the window: only base <= index < base + len is written; padding skipped; sentinel -> NaN as in hy3d_scatter
    g = torch.Generator().manual_seed(5)
    index = torch.randperm(4000, generator=g)[:1500].to(torch.int32)
    index[::7] = -1
    vals = torch.randn(1500, generator=g)
    vals[3] = -10000.0
    slab = torch.full((1000,), 7.0, device=dev)
    ctx.scatter_window(index.to(dev), vals.to(dev), slab, 1700)
    ref = torch.full((1000,), 7.0)
    keep = (index >= 1700) & (index < 2700)
    ref[(index[keep] - 1700).long()] = torch.where(vals[keep] == -10000.0, torch.tensor(float("nan")), vals[keep])
    check("scatter_window values", _same(slab.cpu(), ref))
    # the level-0 sizes the sharded decoder derives on the host are what the layout kernel writes
    for N, m in [(16, 4), (96, 4), (9, 3)]:
        pidx, tile_group, sidx, soff = ctx.flash_layout_minigrids(N, m, 100)
        counts, soff_h = P.flash_minigrid_sizes(N, m, 100)
        check(f"level-0 sizes {N}/{m}", soff.tolist() == soff_h and tile_group.numel() == sum(-(-q // 128) for q in counts))
    torch.cuda.synchronize()


def _worker(rank, world, port, q):
    try:
        import torch.distributed as dist
        os.environ["MASTER_ADDR"] = "127.0.0.1"
        os.environ["MASTER_PORT"] = str(port)
        dist.init_process_group("gloo", rank=rank, world_size=world)
        import hy3dgeo
        from hy3dgeo import _lib, parallel as P, weights as W
        from hy3dgeo.surface_extractors import DMCSurfaceExtractor, MCSurfaceExtractor
        from hy3dgeo.volume_decoders import FlashVDMVolumeDecoding
        dev = torch.device("cuda:0")
        torch.cuda.set_device(dev)
        ctx = _lib.get_context(dev)
        mc, dmc = MCSurfaceExtractor(), DMCSurfaceExtractor()
        fails = []

        def check(name, cond):
            if not cond:
                fails.append(name)

        _entry_point_checks(ctx, dev, check)
        for ci, (cfg_name, field, mode, extra) in enumerate(CASES):
            tag = f"case{ci} {cfg_name} {mode}"
            cfg = getattr(W, cfg_name)
            sd = W.sparsify_field(W.synthetic_state_dict(cfg, seed=0), cfg, *field)
            vae = hy3dgeo.B200ShapeVAE(cfg, sd, device=dev)
            lat = vae(W.synthetic_latents(cfg, 2, 1234).to(dev))
            kw = dict(bounds=1.01, mc_level=0.0, num_chunks=8000, mc_algo="mc", enable_pbar=False, **extra)
            res = extra["octree_resolution"]
            dref = FlashVDMVolumeDecoding(mode)
            ref = dref(lat, vae.geo_decoder, **kw)
            dec = P.ShardedFlashVDMVolumeDecoding(mode)
            grid = dec(lat, vae.geo_decoder, **kw)
            check(f"{tag}: SlabGrid", isinstance(grid, P.SlabGrid) and tuple(grid.shape) == tuple(ref.shape))
            check(f"{tag}: grid bits", _same(grid.to_tensor(), ref))
            check(f"{tag}: queries", [s["queries"] for s in dec.last_stats] == [s["queries"] for s in dref.last_stats])
            for b in range(2):                  # every real query decoded exactly once across the ranks
                mine = torch.tensor(dec.last_stats[b]["rank_queries"])
                total = torch.empty((world, mine.numel()), dtype=mine.dtype)
                dist.all_gather(list(total.unbind(0)), mine)
                check(f"{tag}: rank_queries {b}", total.sum(0).tolist() == dec.last_stats[b]["queries"])
            gathered = P.ShardedFlashVDMVolumeDecoding(mode, keep_sharded=False)(lat, vae.geo_decoder, **kw)
            check(f"{tag}: gathered variant", isinstance(gathered, torch.Tensor) and _same(gathered, ref))
            for b in range(2):
                mesh = mc.run_device(grid[b], mc_level=0.0, bounds=1.01, octree_resolution=res)
                if rank == 0:
                    check(f"{tag}: mc mesh {b}", _same_mesh(mesh, mc.run_device(ref[b], mc_level=0.0, bounds=1.01, octree_resolution=res)))
                else:
                    check(f"{tag}: mc mesh {b} on dst only", mesh is None)
                check(f"{tag}: dmc mesh {b}", _same_mesh(dmc.run_device(grid[b]), dmc.run_device(ref[b])))
            vae.volume_decoder = FlashVDMVolumeDecoding(mode)
            outs_ref = vae.latents2mesh(lat[:1], **kw)
            vae.volume_decoder = P.ShardedFlashVDMVolumeDecoding(mode)
            outs = vae.latents2mesh(lat[:1], **kw)
            if rank == 0:
                check(f"{tag}: latents2mesh", len(outs) == 1 and outs[0] is not None and outs_ref[0] is not None
                      and np.array_equal(outs[0].mesh_f, outs_ref[0].mesh_f)
                      and np.array_equal(outs[0].mesh_v.view(np.uint32), outs_ref[0].mesh_v.view(np.uint32)))
            else:
                check(f"{tag}: latents2mesh None off rank 0", outs == [None])
            ctx.check_watchdog()
        q.put((rank, fails))
        dist.destroy_process_group()
    except Exception:
        q.put((rank, ["EXCEPTION: " + traceback.format_exc()]))


@pytest.mark.parametrize("world", [2, 3])
def test_sharded_flashvdm_bit_identical(world):
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    results = dict(q.get(timeout=900) for _ in range(world))
    for p in procs:
        p.join(timeout=60)
    assert results == {r: [] for r in range(world)}, results
