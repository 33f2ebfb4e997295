#!/usr/bin/env python3
"""Marching cubes under the two ambiguous-face rules, ``sign`` and ``asymptotic`` (hy3dgeo.h hy3d_set_mc_face_rule), on the
same grids: whole-extraction device time (count + emit, CUDA events, the two rules alternating, grids cycled so that the
field is read from HBM), per-kernel times (torch.profiler, separate pass), face counts and the number of ambiguous cube
faces that connect.  The asymptotic rule reads the four values of every ambiguous face in the row-count and emit kernels;
this measures what that costs.  Grids: tanh sphere at 385^3, the octree-384 field of bench.py (Hierarchical decode of the
calibrated synthetic field, NaN outside the visited band, BASELINE configs[2]) and a 385^3 noise field (most cubes
ambiguous).  Prints and records the card name and power limit.

    python tools/gpu_mc_face_rule_bench.py --out mc_face_rule_bench.json
"""
import argparse, json, os, re, subprocess, sys
import numpy as np, torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import hy3dgeo
from hy3dgeo import _lib, weights as W
from hy3dgeo.volume_decoders import HierarchicalVolumeDecoding
from bench import SPARSE_FULL

ap = argparse.ArgumentParser()
ap.add_argument("--out", default="mc_face_rule_bench.json")
ap.add_argument("--reps", type=int, default=20)
args = ap.parse_args()
dev = torch.device("cuda:0")
ctx = _lib.get_context(dev)
q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                   capture_output=True, text=True).stdout.strip()
out = {"device": torch.cuda.get_device_name(dev), "nvidia_smi_name_power_limit_max_sm_clock": q, "reps": args.reps,
       "grids": {}}
print(out["device"], "|", q)
RULES = ("sign", "asymptotic")


def extract(rule, g):
    nv, nf, _ = ctx.mc_count(g, 0.0, rule)
    v = torch.empty((nv, 3), dtype=torch.float32, device=dev); f = torch.empty((nf, 3), dtype=torch.int32, device=dev)
    ctx.mc_emit([g.shape[0]] * 3, [2.02] * 3, [-1.01] * 3, v, f)
    return nv, nf


def kernel_times(rule, grids, reps=5):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for i in range(reps):
            extract(rule, grids[i % len(grids)])
        torch.cuda.synchronize(dev)
    res = {}
    for e in prof.key_averages():
        m = re.search(r"\b(k_(?:mc|scan)_[a-z0-9_]+)", e.key)
        if m:
            t = getattr(e, "self_device_time_total", None) or getattr(e, "self_cuda_time_total", 0.0)
            res[m.group(1)] = res.get(m.group(1), 0.0) + round(t / reps, 2)      # us per extraction
    return res


def ambiguous_faces(g):
    """(ambiguous grid faces, those that connect under the asymptotic rule), on the device in float64."""
    n_amb = n_con = 0
    for axis in range(3):
        d = g.movedim(axis, 0)
        for s in range(0, d.shape[0], 32):
            p = d[s:s + 32].double()
            c00, c10, c01, c11 = p[:, :-1, :-1], p[:, 1:, :-1], p[:, :-1, 1:], p[:, 1:, 1:]
            i00, i10, i01, i11 = c00 > 0, c10 > 0, c01 > 0, c11 > 0
            amb = (i00 == i11) & (i10 == i01) & (i00 != i10)
            con = amb & torch.where(i00, c00 * c11 > c10 * c01, c10 * c01 > c00 * c11)
            n_amb += int(amb.sum()); n_con += int(con.sum())
    return n_amb, n_con


def bench_grids(name, grids):
    for g in grids[:2]:
        for rule in RULES:
            extract(rule, g)
    torch.cuda.synchronize(dev)
    ms = {r: [] for r in RULES}
    counts = {}
    for i in range(args.reps):
        for rule in (RULES if i % 2 == 0 else RULES[::-1]):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            counts[rule] = extract(rule, grids[i % len(grids)])
            e1.record(); e1.synchronize()
            ms[rule].append(e0.elapsed_time(e1))
    n_amb, n_con = ambiguous_faces(grids[0])
    row = {"shape": list(grids[0].shape), "buffers_cycled": len(grids), "ambiguous_faces": n_amb, "connected_faces": n_con}
    for rule in RULES:
        nv, nf = counts[rule]
        row[rule] = {"us_median": round(1e3 * float(np.median(ms[rule])), 1), "us_min": round(1e3 * min(ms[rule]), 1),
                     "V": nv, "F": nf, "kernels_us": kernel_times(rule, grids)}
    row["asymptotic_over_sign"] = round(row["asymptotic"]["us_median"] / row["sign"]["us_median"], 3)
    out["grids"][name] = row
    print(name, json.dumps(row), flush=True)


n = 385
nbuf = int(300e6 // (4 * n ** 3)) + 1                     # > 126 MB L2 in total
x = torch.linspace(-1.01, 1.01, n, device=dev)
r = torch.sqrt(x[:, None, None] ** 2 + x[None, :, None] ** 2 + x[None, None, :] ** 2)
bench_grids("sphere385", [(torch.tanh(20 * (0.6 - r)) + 0.001 * i).contiguous() for i in range(nbuf)])
del r
gen = torch.Generator(device=dev).manual_seed(0)
bench_grids("noise385", [torch.randn((n, n, n), device=dev, generator=gen) for _ in range(nbuf)])

cfg = W.FULL                                               # bench.py's octree-384 workload (BASELINE configs[2])
sd = W.sparsify_field(W.synthetic_state_dict(cfg, seed=0), cfg, **SPARSE_FULL)
vae = hy3dgeo.B200ShapeVAE(cfg, sd, device=dev)
lat = vae(W.synthetic_latents(cfg, 1, 1234).to(dev))
kw = dict(bounds=1.01, mc_level=0.0, num_chunks=262144, octree_resolution=384, enable_pbar=False)
grid = HierarchicalVolumeDecoding()(lat, vae.geo_decoder, **kw)[0].contiguous()
bench_grids("octree384", [grid, grid.clone()])
json.dump(out, open(args.out, "w"), indent=1)
print("wrote", args.out)
