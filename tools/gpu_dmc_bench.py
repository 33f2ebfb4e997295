#!/usr/bin/env python3
"""Dual vs classic marching cubes on the same grids: whole-extraction device time (count + emit, CUDA events, the two
algorithms alternating, grids cycled so that the field is read from HBM), per-kernel times (torch.profiler, separate
pass), the whole pass as a fraction of the HBM data-sheet bandwidth with algorithmic bytes 4 N^3 + 12 V + 12 F, and
latents2mesh end to end at BASELINE configs[2] with mc_algo 'mc' and 'dmc'.  Grids: tanh sphere at 257^3 / 385^3 / 513^3
and the octree-384 field of bench.py (Hierarchical decode of the calibrated synthetic field, NaN outside the visited band).

    python tools/gpu_dmc_bench.py --out dmc_bench.json
"""
import argparse, json, os, re, subprocess, sys, time
import numpy as np, torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import hy3dgeo
from hy3dgeo import _lib, weights as W
from hy3dgeo.surface_extractors import DMCSurfaceExtractor, MCSurfaceExtractor
from hy3dgeo.volume_decoders import HierarchicalVolumeDecoding

HBM_DATASHEET_GBS = 7700.0                 # HGX B200 data sheet, one GPU (not a measured peak)
SPARSE_FULL = dict(keep_freqs=2, gain=9.178747825383368, bias=2.288298721472633)    # bench.py's calibrated field

ap = argparse.ArgumentParser()
ap.add_argument("--out", default="dmc_bench.json")
ap.add_argument("--reps", type=int, default=20)
args = ap.parse_args()
dev = torch.device("cuda:0")
ctx = _lib.get_context(dev)
q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                   capture_output=True, text=True).stdout.strip()
out = {"device": torch.cuda.get_device_name(dev), "nvidia_smi_name_power_limit_max_sm_clock": q,
       "hbm_reference_GBps": HBM_DATASHEET_GBS, "reps": args.reps, "grids": {}}
print(out["device"], "|", q)


def extract(algo, g):
    if algo == "mc":
        nv, nf, _ = ctx.mc_count(g, 0.0)
        v = torch.empty((nv, 3), dtype=torch.float32, device=dev); f = torch.empty((nf, 3), dtype=torch.int32, device=dev)
        ctx.mc_emit([g.shape[0]] * 3, [2.02] * 3, [-1.01] * 3, v, f)
    else:
        nv, nf, _ = ctx.dmc_count(g)
        v = torch.empty((nv, 3), dtype=torch.float32, device=dev); f = torch.empty((nf, 3), dtype=torch.int32, device=dev)
        ctx.dmc_emit(v, f)
    return nv, nf


def kernel_times(algo, grids, reps=5):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for i in range(reps):
            extract(algo, grids[i % len(grids)])
        torch.cuda.synchronize(dev)
    res = {}
    for e in prof.key_averages():
        m = re.search(r"\b(k_(?:mc|dmc|scan)_[a-z0-9_]+(?:<\d+>)?)", e.key)
        if m:
            t = getattr(e, "self_device_time_total", None) or getattr(e, "self_cuda_time_total", 0.0)
            res[m.group(1)] = res.get(m.group(1), 0.0) + round(t / reps, 2)      # us per extraction
    return res


def bench_grids(name, grids):
    for g in grids[:2]:
        extract("mc", g); extract("dmc", g)
    torch.cuda.synchronize(dev)
    ms = {"mc": [], "dmc": []}
    counts = {}
    for i in range(args.reps):
        for algo in (("mc", "dmc") if i % 2 == 0 else ("dmc", "mc")):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            counts[algo] = extract(algo, grids[i % len(grids)])
            e1.record(); e1.synchronize()
            ms[algo].append(e0.elapsed_time(e1))
    n3 = grids[0].numel()
    row = {"shape": list(grids[0].shape), "buffers_cycled": len(grids)}
    for algo in ("mc", "dmc"):
        us = 1e3 * float(np.median(ms[algo]))
        nv, nf = counts[algo]
        alg = 4.0 * n3 + 12.0 * nv + 12.0 * nf
        row[algo] = {"us_median": round(us, 1), "us_min": round(1e3 * min(ms[algo]), 1), "V": nv, "F": nf,
                     "algorithmic_MB": round(alg / 1e6, 2), "frac_hbm_datasheet": round(alg / (us * 1e-6) / 1e9 / HBM_DATASHEET_GBS, 3),
                     "kernels_us": kernel_times(algo, grids)}
    row["dmc_over_mc"] = round(row["dmc"]["us_median"] / row["mc"]["us_median"], 2)
    out["grids"][name] = row
    print(name, json.dumps(row), flush=True)


for n in (257, 385, 513):
    x = torch.linspace(-1.01, 1.01, n, device=dev)
    r = torch.sqrt(x[:, None, None] ** 2 + x[None, :, None] ** 2 + x[None, None, :] ** 2)
    nbuf = max(2, int(300e6 // (4 * n ** 3)) + 1)             # > 126 MB L2 in total
    bench_grids(f"sphere{n}", [(torch.tanh(20 * (0.6 - r)) + 0.001 * i).contiguous() for i in range(nbuf)])
    del r

# bench.py's octree-384 workload (BASELINE configs[2])
cfg = W.FULL
sd = W.sparsify_field(W.synthetic_state_dict(cfg, seed=0), cfg, **SPARSE_FULL)
vae = hy3dgeo.B200ShapeVAE(cfg, sd, device=dev)
vae.volume_decoder = HierarchicalVolumeDecoding()
lat = vae(W.synthetic_latents(cfg, 1, 1234).to(dev))
kw = dict(bounds=1.01, mc_level=0.0, num_chunks=262144, octree_resolution=384, enable_pbar=False)
grid = vae.volume_decoder(lat, vae.geo_decoder, **kw)[0].contiguous()
out["octree384_nan_fraction"] = float(torch.isnan(grid).float().mean())
bench_grids("octree384", [grid, grid.clone()])

e2e = {"mc": [], "dmc": []}
exts = {"mc": MCSurfaceExtractor(), "dmc": DMCSurfaceExtractor()}
for i in range(2 + 6):
    for algo in (("mc", "dmc") if i % 2 == 0 else ("dmc", "mc")):
        vae.surface_extractor = exts[algo]
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        m = vae.latents2mesh(lat, **kw)[0]
        torch.cuda.synchronize(dev)
        if i >= 2:
            e2e[algo].append(1e3 * (time.perf_counter() - t0))
        assert m is not None
out["latents2mesh_configs2_ms"] = {a: {"median": round(float(np.median(v)), 1), "min": round(min(v), 1)} for a, v in e2e.items()}
out["latents2mesh_configs2_ms"]["workload"] = "FULL ShapeVAE, HierarchicalVolumeDecoding octree 384 (bench.py field), latents given"
print("latents2mesh", json.dumps(out["latents2mesh_configs2_ms"]))
os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
json.dump(out, open(args.out, "w"), indent=1)
