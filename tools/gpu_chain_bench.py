#!/usr/bin/env python3
"""Per-kernel-family device time of the tcgen05 decoder chain on a fixed list of query points
(full model unless --model mini).

    python tools/gpu_chain_bench.py [--points 524288] [--reps 3] [--tag name]
"""
import argparse, json, os, sys
import numpy as np, torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import hy3dgeo
from hy3dgeo import weights as W, _lib
from hy3dgeo.volume_decoders import bind

ap = argparse.ArgumentParser()
ap.add_argument("--model", default="full")
ap.add_argument("--points", type=int, default=524288)
ap.add_argument("--reps", type=int, default=3)
ap.add_argument("--tag", default="")
ap.add_argument("--no-pre", action="store_true", help="skip the transformer / K/V timings (short kernel sequence for ncu)")
args = ap.parse_args()
dev = torch.device("cuda:0")
cfg = W.FULL if args.model == "full" else W.MINI
sd = W.synthetic_state_dict(cfg, seed=0)
vae = hy3dgeo.B200ShapeVAE(cfg, sd, device=dev)
z = W.synthetic_latents(cfg, 1, 1234).to(dev)
lat = vae(z)
ctx = bind(lat, vae.geo_decoder)
ctx.prepare_kv(lat[0])
g = torch.Generator(device="cpu").manual_seed(7)
xyz = (torch.rand(args.points, 3, generator=g) * 2.02 - 1.01).to(dev)
def timed(fn, reps=5):
    fn(); torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record(); torch.cuda.synchronize()
    return a.elapsed_time(b) / reps
if not args.no_pre:
    pre = {"transformer_ms": round(timed(lambda: vae(z)), 3)}
    pre["prepare_kv_ms"] = round(timed(lambda: ctx.prepare_kv(lat[0])), 3)
    print(json.dumps(pre), flush=True)
M, Wd, R = cfg.num_latents, cfg.width, 4
flops = {"gemm_c_q": 2 * Wd * Wd, "attention": 4 * M * Wd, "gemm_c_proj": 2 * Wd * Wd,
         "gemm_c_fc": 2 * R * Wd * Wd, "gemm_mlp_proj": 2 * R * Wd * Wd}
for _ in range(2):
    out = ctx.decode_points(xyz)
torch.cuda.synchronize()
ctx.profile_read(); ctx.profile(True)
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
e0.record()
for _ in range(args.reps):
    out = ctx.decode_points(xyz)
e1.record(); torch.cuda.synchronize()
prof = ctx.profile_read(); ctx.profile(False)
wd = ctx.watchdog()
res = {"tag": args.tag, "points": args.points, "total_ms": round(e0.elapsed_time(e1) / args.reps, 3), "watchdog": int(wd[0]),
       "families": {}}
for f, (ms, cnt) in prof.items():
    if cnt:
        d = {"ms": round(ms / args.reps, 3)}
        if f in flops:
            d["tflops"] = round(flops[f] * args.points / (ms / args.reps) / 1e9, 1)
        res["families"][f] = d
print(json.dumps(res), flush=True)
