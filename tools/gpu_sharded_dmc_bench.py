#!/usr/bin/env python3
"""Dual marching cubes on a grid sharded across GPUs: the old path (``SlabGrid.to_tensor()`` gathers the whole grid on
every rank, then whole-grid DMC on every rank) against the slab path (``DMCSurfaceExtractor.run_device`` on the
``SlabGrid``: slab DMC, bounding-box all-reduce, mesh all-gather).  Grids: 381^3 (FlashVDM octree 384, configs[3] scale)
and 505^3, a bumpy shell with NaN outside the band a sparse decoder visits, cut by ``plane_cuts`` with the two-plane
halo, as ``ShardedFlashVDMVolumeDecoding`` leaves it.  Time per extraction: CUDA events on rank 0 between two barriers,
the two paths alternating, median over --reps after warm-up.  Bytes each rank receives (from shapes and counts): the
grid planes it does not own (old) against the mesh pieces of the other ranks (new, padded as all_gather moves them).
Checks that both paths give the same mesh bit for bit.  Prints the card name and power limit.

    torchrun --nproc_per_node 8 tools/gpu_sharded_dmc_bench.py --out sharded_dmc_8gpu.json
"""
import argparse, json, os, subprocess, sys
import numpy as np, torch
import torch.distributed as dist
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from hy3dgeo import _lib, parallel as P
from hy3dgeo.surface_extractors import DMCSurfaceExtractor

ap = argparse.ArgumentParser()
ap.add_argument("--out", default="sharded_dmc_bench.json")
ap.add_argument("--reps", type=int, default=15)
ap.add_argument("--sizes", default="381,505")
args = ap.parse_args()
dist.init_process_group("nccl")
rank, world = dist.get_rank(), dist.get_world_size()
dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", rank)))
torch.cuda.set_device(dev)
ctx = _lib.get_context(dev)
dmc = DMCSurfaceExtractor()


def field(n):
    x = torch.linspace(-1.01, 1.01, n, device=dev)
    X, Y, Z = torch.meshgrid(x, x, x, indexing="ij")
    g = torch.tanh(20 * (0.7 + 0.08 * torch.sin(9 * X) * torch.cos(7 * Y) * torch.sin(5 * Z + 1) - torch.sqrt(X * X + Y * Y + Z * Z)))
    return torch.where(g.abs() < 0.95, g, torch.full_like(g, float("nan"))).contiguous()


def timed(fn):
    dist.barrier()
    torch.cuda.synchronize(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    res = fn()
    e1.record()
    torch.cuda.synchronize(dev)
    dist.barrier()
    return e0.elapsed_time(e1), res


out = {"world": world, "reps": args.reps, "grids": {}}
if rank == 0:
    q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip()
    out.update(device=torch.cuda.get_device_name(dev), nvidia_smi_name_power_limit_max_sm_clock=q)
    print(out["device"], "|", q, "| world", world, flush=True)
for n in [int(s) for s in args.sizes.split(",")]:
    full = field(n)
    index = torch.nonzero(~torch.isnan(full).reshape(-1)).reshape(-1).to(torch.int32)
    planes, _, _ = P.plane_cuts(index, n, world)
    x0, x1 = planes[rank], planes[rank + 1]
    grid = P.SlabGrid([full[x0: min(x1 + P.MC_HALO, n)].clone()], x0, x1 - x0, (n, n, n), True)
    del full, index
    torch.cuda.empty_cache()
    old = lambda: dmc.run_device(grid.to_tensor()[0])
    new = lambda: dmc.run_device(grid)
    _, a = timed(old)
    _, b = timed(new)
    same = bool(torch.equal(a[0].view(torch.int32), b[0].view(torch.int32)) and torch.equal(a[1], b[1]))
    nv, nf, _ = ctx.dmc_count_slab(grid.slabs[0], x1 - x0, x0, n)
    counts = torch.tensor([nv, nf], dtype=torch.int64, device=dev)
    allc = torch.empty((world, 2), dtype=torch.int64, device=dev)
    dist.all_gather_into_tensor(allc, counts)
    allc = allc.cpu().tolist()
    for _ in range(2):
        timed(old); timed(new)
    t = {"old": [], "new": []}
    for i in range(args.reps):
        for k in (("old", "new") if i % 2 == 0 else ("new", "old")):
            t[k].append(timed(old if k == "old" else new)[0])
    same_all = torch.tensor([int(same)], device=dev)
    dist.all_reduce(same_all, op=dist.ReduceOp.MIN)
    if rank == 0:
        own = [hi - lo for lo, hi in zip(planes, planes[1:])]
        pad_v, pad_f = max(c[0] for c in allc), max(c[1] for c in allc)
        row = {"planes": planes, "V": sum(c[0] for c in allc), "F": sum(c[1] for c in allc), "rank_counts": allc,
               "identical_on_every_rank": bool(same_all.item()),
               "old_ms_median": float(np.median(t["old"])), "new_ms_median": float(np.median(t["new"])),
               "old_ms": [round(v, 4) for v in t["old"]], "new_ms": [round(v, 4) for v in t["new"]],
               # bytes received per rank, worst rank: grid planes owned elsewhere / padded mesh pieces of the other ranks
               "old_bytes_per_rank": max((n - o) * n * n * 4 for o in own),
               "new_bytes_per_rank": (world - 1) * (pad_v * 12 + pad_f * 12)}
        row["speedup"] = round(row["old_ms_median"] / row["new_ms_median"], 3)
        out["grids"][f"{n}^3"] = row
        print(n, {k: v for k, v in row.items() if not k.endswith("_ms")}, flush=True)
    del grid, a, b
    torch.cuda.empty_cache()
if rank == 0:
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
dist.destroy_process_group()
