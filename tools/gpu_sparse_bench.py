#!/usr/bin/env python3
"""BASELINE configs 3/4 on one or more GPUs: octree 384 latents->mesh through the sparse decoders
(Hierarchical, FlashVDM) on a synthetic low-frequency, saturating field (SURVEY §8d recipe: drop the
Fourier frequencies >= 2 from query_proj, choose the output gain/bias from level-0 quantiles so that
~85 % of the voxels saturate below -0.95 and ~5 % lie inside the band).  Prints one JSON line per run, with the card's
name and power limit.  ``--sharded`` runs the sharded Hierarchical and FlashVDM decoders on the same field;
``--timeline`` adds their per-rank stage timeline (separate, synchronising steps after the timed ones).

    python tools/gpu_sparse_bench.py [--model full|mini] [--res 384] [--reps 5]
    torchrun --nproc-per-node N tools/gpu_sparse_bench.py --sharded [--timeline]
"""
import argparse, json, os, subprocess, sys, time
import numpy as np, torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import hy3dgeo
from hy3dgeo import weights as W, _lib
from hy3dgeo.volume_decoders import VanillaVolumeDecoder, HierarchicalVolumeDecoding, FlashVDMVolumeDecoding

ap = argparse.ArgumentParser()
ap.add_argument("--model", default="full")
ap.add_argument("--res", type=int, default=384)
ap.add_argument("--reps", type=int, default=5)
ap.add_argument("--sharded", action="store_true")
ap.add_argument("--timeline", action="store_true")
args = ap.parse_args()
rank, world, lr = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1)), int(os.environ.get("LOCAL_RANK", 0))
dev = torch.device("cuda", lr); torch.cuda.set_device(dev)
if world > 1:
    import torch.distributed as dist
    dist.init_process_group("nccl", device_id=dev)
card = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=name,power.limit", "--format=csv,noheader"],
                      capture_output=True, text=True).stdout.strip()
cfg = W.FULL if args.model == "full" else W.MINI
sd0 = W.sparsify_field(W.synthetic_state_dict(cfg, seed=0), cfg, keep_freqs=2, gain=1.0, bias=0.0)
vae = hy3dgeo.B200ShapeVAE(cfg, sd0, device=dev)
z = W.synthetic_latents(cfg, 1, 1234).to(dev)
lat = vae(z)
g0 = VanillaVolumeDecoder()(lat, vae.geo_decoder, bounds=1.01, octree_resolution=96)[0]
q85, q90 = [float(v) for v in torch.quantile(g0.flatten()[::7].float(), torch.tensor([0.85, 0.90], device=dev))]
gain = 1.9 / (q90 - q85); bias = -0.95 - gain * q85
sd = W.sparsify_field(W.synthetic_state_dict(cfg, seed=0), cfg, keep_freqs=2, gain=gain, bias=bias)
vae = hy3dgeo.B200ShapeVAE(cfg, sd, device=dev)
ctx = _lib.get_context(dev)
kw = dict(bounds=1.01, mc_level=0.0, num_chunks=8000, octree_resolution=args.res, mc_algo="mc", enable_pbar=False)
decs = [("hierarchical", HierarchicalVolumeDecoding()), ("flashvdm_mean", FlashVDMVolumeDecoding("mean"))]
if world > 1 or args.sharded:
    from hy3dgeo.parallel import ShardedFlashVDMVolumeDecoding, ShardedHierarchicalVolumeDecoding
    decs = [("hierarchical_sharded", ShardedHierarchicalVolumeDecoding()), ("flashvdm_mean_sharded", ShardedFlashVDMVolumeDecoding("mean"))]
for name, dec in decs:
    vae.volume_decoder = dec
    for _ in range(2):
        outs = vae.latents2mesh(vae(z), **kw)
    torch.cuda.synchronize()
    ctx.profile_read(); ctx.profile(True)
    t = []
    for _ in range(args.reps):
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(); t0 = time.perf_counter()
        outs = vae.latents2mesh(vae(z), **kw)
        torch.cuda.synchronize(); t.append((time.perf_counter() - t0) * 1e3)
    prof = ctx.profile_read(); ctx.profile(False)
    ctx.check_watchdog()
    st = dec.last_stats[0]
    fams = {k: round(v[0] / args.reps, 3) for k, v in sorted(prof.items(), key=lambda kv: -kv[1][0]) if v[1]}
    per_rank = None
    if args.timeline and world > 1:
        dec.timeline = {}
        for _ in range(args.reps):
            lat_t = vae(z)
            dist.barrier(); dec._t_last = None
            grid = dec(lat_t, vae.geo_decoder, **kw)
            torch.cuda.synchronize(); t2 = time.perf_counter()
            vae.surface_extractor(grid, **kw)
            torch.cuda.synchronize()
            dec.timeline["marching cubes + mesh gather + D2H"] = dec.timeline.get("marching cubes + mesh gather + D2H", 0.0) + (time.perf_counter() - t2) * 1e3
        tab = {k: round(v / args.reps, 3) for k, v in dec.timeline.items()}
        tab["rank_queries"] = dec.last_stats[0]["rank_queries"]
        per_rank = [None] * world
        dist.all_gather_object(per_rank, tab)
        dec.timeline = None
    if rank == 0:
        print(json.dumps({"decoder": name, "card": card, "model": args.model, "res": args.res, "n_gpus": world, "gain": gain, "bias": bias,
                          "levels": st["levels"], "queries": st["queries"], "total_queries": int(sum(st["queries"])),
                          "visited_fraction_last": st["queries"][-1] / (st["levels"][-1] + 1) ** 3,
                          "latents2mesh_ms_median": float(np.median(t)), "latents2mesh_ms_all": [round(x, 2) for x in t],
                          "mesh": None if outs[0] is None else [int(outs[0].mesh_v.shape[0]), int(outs[0].mesh_f.shape[0])],
                          "families_ms": fams, **({"per_rank_timeline_ms": per_rank} if per_rank else {})}), flush=True)
if world > 1:
    dist.destroy_process_group()
