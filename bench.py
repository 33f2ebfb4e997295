#!/usr/bin/env python3
"""Benchmark of the geometry-decoding hot path (latents -> occupancy grid -> mesh).

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--config hier|dense] [--res R] [--dump-outputs DIR]
    torchrun --nnodes=1 --nproc-per-node N ... bench.py --gpus N --steps K --warmup W

Default workload = BASELINE.json configs[2], the configuration the metric ("latents->mesh ms and query pts/sec @octree
384") is quoted on: Hunyuan3D-2 ShapeVAE (3072 latent tokens, width 1024, random-init weights made sparse by the
SURVEY §8d recipe, synthetic latent), HierarchicalVolumeDecoding at octree resolution 384 (levels 97^3 dense -> 193^3 ->
385^3 sparse near-surface refinement) followed by marching cubes on the 385^3 grid.  One "step" = one latents->mesh
pass: latent transformer, K/V projection, the three decoder levels, marching cubes.  On N > 1 GPUs the same job is
partitioned (strong scaling): level 0 by axis-0 slabs, the middle level by equal ranges of the ordered active list, the
last level by plane-aligned slabs that stay on their GPU through marching cubes (ShardedHierarchicalVolumeDecoding +
sharded MCSurfaceExtractor); only mesh pieces travel to rank 0.
`--config dense --res 256|512` runs BASELINE configs[1] / configs[4] (VanillaVolumeDecoder; slabs + halo-exchanged
marching cubes on N > 1).

Metric: decoder query points per second over the whole job = (queries the algorithm evaluates per step) x steps / time;
``ms_per_step`` = ``latents2mesh_ms`` is the other half of BASELINE.json's metric.  Prints ONE JSON line on rank 0.

``value``   : latents resident in HBM, mesh left on the device (CUDA events, max over ranks).
``e2e``     : the public API with HOST buffers: latents from pinned host memory -> B200ShapeVAE.forward -> latents2mesh
              -> numpy mesh; copies inside the timed region.
``roofline``: the decoder kernel family with the largest share of the step (tensor-bound): algorithmic FLOPs / CUDA-event
              time of its launches.  ``roofline_octree`` / ``roofline_mc``: whole-pass HBM fractions of the octree
              refinement (4 n_c^3 + 4 n_f^3 + 8 A bytes per level) and of marching cubes (4 N^3 + 12 V + 12 F).
``cpu_baseline`` / ``--impl reference``: the oracle port of the reference PyTorch fp32 path on the host cores, bounded
              sample (the reference tree itself is absent on the GPU box).

``--dump-outputs DIR`` writes what the last timed step computed (rank 0) as DIR/<name>.npy, every value finite:
``latents`` (ShapeVAE.forward, [tokens, width]); ``grid_visited`` (the volume decoder's grid at the points it evaluated, rows
of (flat grid index, logit): the sparse decoders leave NaN at the others; skipped while the grid stays sharded over the
ranks); ``mesh_v`` / ``mesh_f`` (the marching-cubes mesh without the non-finite vertices along the rim of the visited band
and the faces using them, as ``export_to_trimesh`` / ``MCSurfaceExtractor(cull_nonfinite=True)`` return it).  The inputs
are seeded, so two builds run with the same arguments can be compared output for output.  See ``dump_outputs`` for the
size cap.

bench.py writes nothing into the source tree (which may be read-only): no byte-code caches, no build products.
"""
import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True       # the project's modules are imported from the tree: leave no __pycache__ there

METRIC = "decoder_query_points_per_sec"
UNIT = "pts/s"
CHUNK = 8000          # the reference's num_chunks default in pipelines (pipelines.py:689-693)
# SURVEY §8d sparse-field recipe for the full model, seed 0 / latent seed 1234: query_proj keeps Fourier frequencies < 2,
# output head scaled/shifted so that the level-0 quantiles 0.80 / 0.90 map to -0.95 / +0.95 (tools/gpu_calibrate_sparse.py,
# profiles/r02_calibration_sparse_field.jsonl): octree-384 Hierarchical then visits 11.2 % of the 385^3 grid, 8.34 M queries
# in total — the survey's planning workload (tanh sphere: 11-14 %, 8.18 M).
SPARSE_FULL = dict(keep_freqs=2, gain=9.178747825383368, bias=2.288298721472633)


def flops_per_point(W, M, r, E=51):
    """SURVEY §8: F_pt = 2*51*W + 4*W^2 + 4*M*W + 4*r*W^2 + 2*W."""
    return {"gemm_query_proj": 2 * E * W, "gemm_c_q": 2 * W * W, "attention": 4 * M * W, "gemm_c_proj": 2 * W * W,
            "gemm_c_fc": 2 * r * W * W, "gemm_mlp_proj": 2 * r * W * W, "head": 2 * W}


def executed_flops_per_point(W, M, r):
    """What the kernels actually contract per point (all fp16 MMAs): c_q . query_proj collapsed into one K = 192 GEMM
    (3-term split of the 64-padded Fourier features; the SURVEY formula's 2*51*W + 2*W^2 is never executed as such), c_proj
    K-concatenated with the same 192 columns (x0 recomputed instead of stored)."""
    return {"gemm_c_q": 2 * 192 * W, "attention": 4 * M * W, "gemm_c_proj": 2 * (W + 192) * W, "gemm_c_fc": 2 * r * W * W,
            "gemm_mlp_proj": 2 * r * W * W, "head": 2 * W}


class ClockSampler(threading.Thread):
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag = index, [], False

    def run(self):
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            time.sleep(0.1)

    def summary(self):
        self.stop_flag = True
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unsampled"]}
        sm = sorted(float(r[0]) for r in self.rows if r[0].replace(".", "").isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 3 + i and r[3 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": float(self.rows[0][1]) if self.rows[0][1].replace(".", "").isdigit() else None,
                "power_w_max": max((float(r[2]) for r in self.rows if r[2].replace(".", "").isdigit()), default=None),
                "samples": len(self.rows), "reasons": reasons}


# ------------------------------------------------------------------------------------------------ CPU legs (oracle port)
def cpu_port_setup(cfg, sd, z):
    """Oracle latent transformer on the host (once per latent): returns (latents, seconds)."""
    from oracle import decoder as OD
    torch.set_num_threads(os.cpu_count())
    t0 = time.time()
    lat = OD.shapevae_forward(sd, z, cfg.heads)
    return lat, time.time() - t0


def cpu_port_rate(cfg, sd, lat, seconds, min_chunks=2, res=96):
    """Oracle port of the reference decoder loop on the host cores: chunks of 8000 queries of the workload's dense level
    through CrossAttentionDecoder.forward semantics (K/V re-projected per chunk, as the reference does,
    attention_blocks.py:251-257; the patched HierarchicalVolumeDecoding issues exactly such chunks at every level,
    volume_decoders.py:233-240, 265-271).  Returns (pts/s, chunks, threads)."""
    from hy3dgeo import weights as W
    from oracle import decoder as OD, volume as OV
    torch.set_num_threads(os.cpu_count())
    gsd, fr = W.geo_decoder_state(sd), W.fourier_frequencies(cfg)
    N = res + 1
    ax = OV.axis_tables(1.01, res)
    n, t0, done = 0, time.time(), 0
    while done < min_chunks or time.time() - t0 < seconds:
        lin = (np.arange(done * CHUNK, (done + 1) * CHUNK) + N * N * (N // 3)) % (N ** 3)     # interior planes of the grid
        k = lin % N; j = (lin // N) % N; i = lin // (N * N)
        pts = torch.from_numpy(np.stack([ax[0][i], ax[1][j], ax[2][k]], 1))
        with torch.no_grad():
            OD.geo_decoder_forward(gsd, pts[None], lat, fr, cfg.dec_heads)
        done += 1
        n += CHUNK
    dt = time.time() - t0
    return n / dt, done, torch.get_num_threads()


DUMP_BYTES = 63 * 10 ** 6             # array data; the .npy headers stay well inside the last MB of the 64 MB cap


def dump_outputs(out_dir, arrays, limit=DUMP_BYTES):
    """Writes each tensor of ``arrays`` (name -> tensor, None skipped) as ``out_dir/<name>.npy``: float64 as float64, other
    floating point as float32, integers as float64 (exact for int32).  The tensors are written smallest first and each may
    take an equal share of what is left of ``limit``; one that does not fit is cut to a sample of its rows (dim 0) drawn
    with a fixed seed, so the same shape always keeps the same rows, in their original order."""
    os.makedirs(out_dir, exist_ok=True)
    todo = []
    for name, t in arrays.items():
        if t is not None:
            dt = torch.float32 if t.is_floating_point() and t.dtype != torch.float64 else torch.float64
            todo.append((t.numel() * dt.itemsize, name, t, dt))
    todo.sort(key=lambda x: x[0])
    left = limit
    for i, (_, name, t, dt) in enumerate(todo):
        row_bytes = math.prod(t.shape[1:]) * dt.itemsize
        keep = min(t.shape[0], left // (len(todo) - i) // row_bytes)
        if keep < t.shape[0]:
            rows = np.sort(np.random.default_rng(0).choice(t.shape[0], keep, replace=False))
            t = t[torch.from_numpy(rows).to(t.device)]
        a = t.to(dt).cpu().numpy()
        np.save(os.path.join(out_dir, name + ".npy"), a)
        left -= a.nbytes


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="hier", choices=["hier", "dense"],
                    help="hier: BASELINE configs[2] (Hierarchical, the metric's configuration); dense: configs[1] / configs[4] (Vanilla)")
    ap.add_argument("--res", type=int, default=None, help="octree resolution (default 384 for hier, 256 for dense)")
    ap.add_argument("--model", default="full", choices=["full", "mini"])
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="CPU baseline sample length; 0 skips the CPU leg (tuning runs)")
    ap.add_argument("--norm-gain", type=float, default=1.0,
                    help="multiply the decoder's q_norm / k_norm gains (1.3-1.4 puts the weight-only score bound above 15.9: shows the "
                         "attention kernel's floor with per-head shifts on; changes the field, so a tuning run, not the headline)")
    ap.add_argument("--gather", action="store_true", help="N > 1: gather the grid instead of keeping it sharded through marching cubes")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed as DIR/<name>.npy (float32 / float64, at most 64 MB in all)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the device path (--impl ours)")
    res = args.res if args.res is not None else (384 if args.config == "hier" else 256)

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    import hy3dgeo
    from hy3dgeo import weights as W, _lib
    from hy3dgeo.volume_decoders import hierarchy_levels
    cfg = W.FULL if args.model == "full" else W.MINI
    N = res + 1
    hier = args.config == "hier"
    levels = hierarchy_levels(res) if hier else [res]
    name = f"Hunyuan3D-2{'mini' if args.model == 'mini' else ''} ShapeVAE ({cfg.num_latents} latent tokens, width {cfg.width})"
    if hier:
        workload = (f"{name} HierarchicalVolumeDecoding octree_resolution={res} (levels {[l + 1 for l in levels]}^3, sparse near-surface "
                    f"refinement) + marching cubes")
        weights = (f"random-init seed 0 (hy3dgeo.weights.synthetic_state_dict) + SURVEY §8d sparse-field edit: query_proj keeps Fourier "
                   f"frequencies < {SPARSE_FULL['keep_freqs']}, output_proj gain {SPARSE_FULL['gain']:.6f} bias {SPARSE_FULL['bias']:.6f}")
        partition = (f"x{world}: latent transformer by token ranges (K/V tiles all-gathered per layer), level 0 axis-0 slabs, middle level equal list ranges (all-gathered), last level plane-aligned slabs kept "
                     f"through sharded marching cubes" + (" [--gather: last level all-gathered, MC on rank 0]" if args.gather else "")) if world > 1 else "single GPU"
    else:
        workload = f"{name} VanillaVolumeDecoder octree_resolution={res} + marching cubes"
        weights = "random-init seed 0 (hy3dgeo.weights.synthetic_state_dict)"
        partition = (f"axis-0 slabs x{world}, " + ("gathered on rank 0" if args.gather else "halo-exchanged sharded marching cubes")) if world > 1 else "single GPU"
    if args.norm_gain != 1.0:
        weights += f"; q_norm / k_norm gains x{args.norm_gain}"
    config = {"workload": workload, "grid": [N, N, N], "bounds": 1.01, "mc_level": 0.0, "weights": weights, "latent_seed": 1234,
              "partition": partition,
              "l2": "per-step activations (GBs per 262144-point chunk) and the grids exceed the 126 MB L2; no explicit flush"}

    def make_sd():
        sd = W.synthetic_state_dict(cfg, seed=0)
        if args.norm_gain != 1.0:
            for n in ("q_norm", "k_norm"):
                key = f"geo_decoder.cross_attn_decoder.attn.attention.{n}.weight"
                sd[key] = sd[key] * args.norm_gain
        return W.sparsify_field(sd, cfg, **SPARSE_FULL) if hier else sd

    # -------------------------------------------------------------------------- reference arm
    if args.impl == "reference":
        if rank != 0:
            return
        sd = make_sd()
        z = W.synthetic_latents(cfg, 1, 1234)
        chunks_per_step = 2
        lat, tf_s = cpu_port_setup(cfg, sd, z)                       # latent transformer: once per latent, reported separately
        rates = []
        for s in range(args.warmup + args.steps):
            t0 = time.time()
            r, done, threads = cpu_port_rate(cfg, sd, lat, 0.0, min_chunks=chunks_per_step, res=levels[0])
            if s >= args.warmup:
                rates.append((done * CHUNK, time.time() - t0))
        pts = sum(a for a, _ in rates); secs = sum(b for _, b in rates)
        val = pts / secs
        sample = (f"{chunks_per_step} chunks of {CHUNK} queries of the workload's dense level per step; oracle port of the reference PyTorch "
                  f"fp32 CPU path (K/V re-projected per chunk as the reference does); latent transformer {tf_s:.1f} s once per latent, not "
                  f"in the rate; octree masks / dilations and marching cubes not in the rate")
        print(json.dumps({"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
                          "warmup": args.warmup, "ms_per_step": 1e3 * secs / max(args.steps, 1), "higher_is_better": True,
                          "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config,
                          "cpu_baseline": {"value": val, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
                          "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                          "latent_transformer_s": tf_s}))
        return

    # -------------------------------------------------------------------------------- our arm
    import torch.distributed as dist
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    from hy3dgeo import parallel as P
    from hy3dgeo.volume_decoders import HierarchicalVolumeDecoding, VanillaVolumeDecoder
    sd = make_sd()
    vae = hy3dgeo.B200ShapeVAE(cfg, sd, device=dev)
    if hier:
        vae.volume_decoder = P.ShardedHierarchicalVolumeDecoding(keep_sharded=not args.gather) if world > 1 else HierarchicalVolumeDecoding()
    else:
        vae.volume_decoder = P.ShardedVanillaVolumeDecoder(keep_sharded=not args.gather) if world > 1 else VanillaVolumeDecoder()
    z_host = W.synthetic_latents(cfg, 1, 1234).pin_memory()
    z_dev = z_host.to(dev)
    ctx = _lib.get_context(dev)
    kw = dict(bounds=1.01, mc_level=0.0, num_chunks=CHUNK, octree_resolution=res, mc_algo="mc", enable_pbar=False)
    mesh_bytes = [0]
    mesh_size = [0, 0]

    tf_group = True if world > 1 else None        # N > 1: the latent transformer runs sequence-parallel over the ranks
    last = {}                                     # --dump-outputs: what the latest step_device computed

    def step_device():
        lat = vae(z_dev, group=tf_group)
        grid = vae.volume_decoder(lat, vae.geo_decoder, **kw)
        m = None
        if grid is not None:
            m = vae.surface_extractor.run_device(grid[0], mc_level=0.0, bounds=1.01, octree_resolution=res)
            if m is not None:
                mesh_size[0], mesh_size[1] = m[0].shape[0], m[1].shape[0]
        if args.dump_outputs:
            last.update(latents=lat.reshape(-1, lat.shape[-1]), grid=grid[0].reshape(-1) if isinstance(grid, torch.Tensor) else None,
                        mesh=m)

    def step_e2e():
        outs = vae.latents2mesh(vae(z_host.to(dev, non_blocking=True), group=tf_group), **kw)
        if outs is not None and outs[0] is not None:
            mesh_bytes[0] = outs[0].mesh_v.nbytes + outs[0].mesh_f.nbytes

    def timed(fn, steps, profile=False):
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        if profile:
            ctx.profile_read(); ctx.profile(True)
        l0 = ctx.launches
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        prof = None
        if profile:
            prof = ctx.profile_read(); ctx.profile(False)
        if world > 1:
            dist.barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()), ctx.launches - l0, prof

    warm = max(args.warmup, 3)
    for _ in range(warm):
        step_device()
    ctx.check_watchdog()
    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
    ms, launches, _ = timed(step_device, args.steps)
    clocks = sampler.summary() if sampler else None
    if args.dump_outputs and rank == 0:
        out = {"latents": last["latents"]}
        if last["grid"] is not None:
            visited = torch.nonzero(torch.isfinite(last["grid"])).flatten()
            out["grid_visited"] = torch.stack([visited.double(), last["grid"][visited].double()], 1)
        if last["mesh"] is not None:
            out["mesh_v"], out["mesh_f"] = ctx.mesh_clean(*last["mesh"], flip_winding=False)
        dump_outputs(args.dump_outputs, out)
    # per-family device times from a separate profiled pass (CUDA events around every launch perturb the step by ~1 %)
    ms_prof, _, prof = timed(step_device, min(args.steps, 5), profile=True)
    prof_steps = min(args.steps, 5)
    step_e2e()
    ms_e2e, _, _ = timed(step_e2e, args.steps)
    ctx.check_watchdog()
    st = getattr(vae.volume_decoder, "last_stats", None)
    queries = st[0]["queries"] if st else [N ** 3]
    my_queries = st[0].get("rank_queries", queries) if st else [(P.slab_planes(N, rank, world)[1] - P.slab_planes(N, rank, world)[0]) * N * N]
    total_q = int(sum(queries))
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    value = total_q * args.steps / (ms / 1e3)
    fl = flops_per_point(cfg.dec_width, cfg.num_latents, cfg.geo_decoder_mlp_expand_ratio)
    pts_local = float(sum(my_queries))            # rank 0 times its own share; its families are reported
    fams = {k: v for k, v in prof.items() if v[1] > 0}
    total_fam_ms = sum(v[0] for v in fams.values())
    top = max((k for k in fams if k in fl), key=lambda k: fams[k][0])
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak_tf = peaks.get("bf16_tflops_sustained", 1400.0)
    peak_hbm = peaks.get("hbm_gbs", 6500.0)
    peak_src = "MEASURED_PEAKS.json (bf16_tflops_sustained: kernel timed inside a long step; hbm_gbs)" if peaks else \
        "fallback 1.4 PFLOP/s sustained, 6.5 TB/s (B200_PROFILING.md)"
    top_ms, top_cnt = fams[top]
    achieved = fl[top] * pts_local * prof_steps / (top_ms / 1e3) / 1e12
    traffic = None
    try:
        traffic = json.load(open(os.path.join(ROOT, "profiles", "traffic.json"))).get(top)
    except Exception:
        pass
    chain_ms = sum(fams[k][0] for k in fams if k in fl or k in ("layernorm", "embed"))
    all_tf = sum(fl.values()) * pts_local * prof_steps / (chain_ms / 1e3) / 1e12
    xfl = executed_flops_per_point(cfg.dec_width, cfg.num_latents, cfg.geo_decoder_mlp_expand_ratio)
    exe_tf = sum(xfl.values()) * pts_local * prof_steps / (chain_ms / 1e3) / 1e12
    bound, akern, mbound = ctx.attention_info()
    roofline = {"bound": "tensor", "kernel": top, "achieved": achieved, "peak": peak_tf, "unit": "TFLOP/s", "frac": achieved / peak_tf,
                "traffic": traffic, "peak_source": peak_src, "launches": top_cnt, "avg_launch_ms": top_ms / max(top_cnt, 1),
                "flops_per_point": fl[top], "share_of_step": top_ms / total_fam_ms,
                "decoder_chain_tflops": all_tf, "decoder_chain_frac": all_tf / peak_tf,
                "decoder_chain_tflops_executed": exe_tf, "decoder_chain_frac_executed": exe_tf / peak_tf,
                "flops_note": "achieved / decoder_chain_* use the ALGORITHMIC flops of SURVEY §8 (2*51*W + 4W^2 + 4MW + 4rW^2 + 2W per point); "
                              "*_executed counts what the tensor cores contract: c_q . query_proj runs collapsed as one K=192 GEMM "
                              "(2*192*W instead of 2*51*W + 2W^2), c_proj carries 192 extra K columns; attention is unchanged",
                "families_ms_per_step": {k: round(v[0] / prof_steps, 3) for k, v in sorted(fams.items(), key=lambda kv: -kv[1][0])}}
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": warm,
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f16 operands, f32 accumulate", "data": "synthetic", "config": config,
            "latents2mesh_ms": ms / args.steps, "queries": total_q, "queries_per_level": queries,
            "visited_fraction": queries[-1] / N ** 3, "mesh": {"vertices": mesh_size[0], "faces": mesh_size[1]},
            "attention_kernel": akern, "attention_score_bound": {"from_norm_weights": bound, "measured_max_k_norm": mbound},
            "roofline": roofline}
    # ---- HBM-bound passes, whole-pass fractions (SURVEY §8d algorithmic bytes), rank 0's share
    if hier and "octree" in fams and world == 1:
        ob = sum(4 * (a + 1) ** 3 + 4 * (b + 1) ** 3 + 8 * q for a, b, q in zip(levels, levels[1:], queries[1:]))
        o_ms = fams["octree"][0] / prof_steps
        line["roofline_octree"] = {"bound": "hbm", "achieved": ob / (o_ms / 1e3) / 1e9, "peak": peak_hbm, "unit": "GB/s",
                                   "frac": ob / (o_ms / 1e3) / 1e9 / peak_hbm, "algorithmic_bytes": ob, "ms_per_step": o_ms,
                                   "launches_per_step": fams["octree"][1] / prof_steps,
                                   "formula": "sum over refined levels of 4 n_c^3 + 4 n_f^3 + 8 A (read coarse, write the fine grid incl. sentinel fill, scatter + index list)"}
    mc_f = [k for k in ("mc_bits", "mc_rowcount", "mc_scan", "mc_emit") if k in fams]
    if mc_f and world == 1:
        mb = 4 * N ** 3 + 12 * mesh_size[0] + 12 * mesh_size[1]
        m_ms = sum(fams[k][0] for k in mc_f) / prof_steps
        line["roofline_mc"] = {"bound": "hbm", "achieved": mb / (m_ms / 1e3) / 1e9, "peak": peak_hbm, "unit": "GB/s",
                               "frac": mb / (m_ms / 1e3) / 1e9 / peak_hbm, "algorithmic_bytes": mb, "ms_per_step": m_ms,
                               "formula": "4 N^3 + 12 V + 12 F over classify + count + scan + emit",
                               "classify_pass": {"achieved": 4.0 * N ** 3 / (fams["mc_bits"][0] / fams["mc_bits"][1] / 1e3) / 1e9,
                                                 "frac": 4.0 * N ** 3 / (fams["mc_bits"][0] / fams["mc_bits"][1] / 1e3) / 1e9 / peak_hbm,
                                                 "avg_launch_ms": fams["mc_bits"][0] / fams["mc_bits"][1]} if "mc_bits" in fams else None}
    line["e2e"] = {"value": total_q * args.steps / (ms_e2e / 1e3), "unit": UNIT, "ms_per_step": ms_e2e / args.steps,
                   "h2d_bytes_per_step": z_host.numel() * z_host.element_size(), "d2h_bytes_per_step": mesh_bytes[0]}
    line["gpu_launches"] = launches
    line["clocks"] = clocks
    if world == 1 and args.cpu_seconds > 0:
        lat_cpu, tf_s = cpu_port_setup(cfg, sd, W.synthetic_latents(cfg, 1, 1234))
        rate, chunks, threads = cpu_port_rate(cfg, sd, lat_cpu, args.cpu_seconds, res=levels[0])
        line["cpu_baseline"] = {"value": rate, "unit": UNIT, "cores": threads, "kind": "port",
                                "sample": f"{chunks} chunks of {CHUNK} queries of the workload's dense level (of {total_q} queries per step); oracle "
                                          f"port of the reference fp32 PyTorch CPU path; the decoder part of a full step extrapolates to "
                                          f"{tf_s + total_q / rate:.0f} s (latent transformer {tf_s:.1f} s)"}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
