#!/usr/bin/env python3
"""FloaterRemover / DegenerateFaceRemover at BASELINE configs[2] mesh scale: ``run_device`` of each filter and of the chain
(device time, CUDA events, after warm-up), per-kernel times (torch.profiler, separate pass), the host-to-host call a user
makes on a ``Latent2MeshOutput`` (wall clock, ends in a synchronisation), and the numpy statements of oracle/postprocess.py
on the host for comparison.  pymeshlab is not installed, so the reference filters are not measured.

Meshes: marching cubes and dual marching cubes of one 385^3 field — a hollow, bumpy body (~0.97 M MC faces) plus 60 small
spheres, some of them apart (floaters) — after ``mesh_clean``.  The input mesh (~17 MB) stays in the 126 MB L2 between
passes, as it does right after extraction in the pipeline.

    python tools/gpu_postprocess_bench.py --out postprocess_bench.json
"""
import argparse, json, os, re, subprocess, sys, time
import numpy as np, torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import hy3dgeo
from hy3dgeo import _lib
from oracle import postprocess as PP

ap = argparse.ArgumentParser()
ap.add_argument("--out", default="postprocess_bench.json")
ap.add_argument("--reps", type=int, default=50)
args = ap.parse_args()
dev = torch.device("cuda:0")
ctx = _lib.get_context(dev)
q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                   capture_output=True, text=True).stdout.strip()
out = {"device": torch.cuda.get_device_name(dev), "nvidia_smi_name_power_limit_max_sm_clock": q, "reps": args.reps,
       "pymeshlab": "not measured (not installed)", "meshes": {}}
print(out["device"], "|", q)


def field(n=385):
    x = torch.linspace(-1.01, 1.01, n, device=dev)
    X, Y, Z = x[:, None, None], x[None, :, None], x[None, None, :]
    R = torch.sqrt(X * X + Y * Y + Z * Z)
    d = torch.minimum(0.62 + 0.1 * torch.sin(20 * X) * torch.sin(20 * Y) * torch.sin(20 * Z) - R, R - 0.35)
    rng = np.random.default_rng(7)
    for c, r in zip(rng.uniform(-0.95, 0.95, (60, 3)), rng.uniform(0.008, 0.03, 60)):
        d = torch.maximum(d, float(r) - torch.sqrt((X - float(c[0])) ** 2 + (Y - float(c[1])) ** 2 + (Z - float(c[2])) ** 2))
    return torch.tanh(20 * d).float().contiguous()


def meshes(g):
    ext = hy3dgeo.MCSurfaceExtractor(cull_nonfinite=True)
    yield "mc", ext.run_device(g, mc_level=0.0, bounds=1.01, octree_resolution=384)
    v, f = hy3dgeo.DMCSurfaceExtractor().run_device(g)
    yield "dmc", ctx.mesh_clean(v, f, flip_winding=False)


FR, DR = hy3dgeo.FloaterRemover(), hy3dgeo.DegenerateFaceRemover()
CALLS = {"floaters": lambda v, f: FR.run_device(v, f), "weld": lambda v, f: DR.run_device(v, f),
         "chain": lambda v, f: DR.run_device(*FR.run_device(v, f))}


def device_us(fn, v, f):
    for _ in range(3):
        fn(v, f)
    torch.cuda.synchronize(dev)
    ts = []
    for _ in range(args.reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        res = fn(v, f)
        e1.record(); e1.synchronize()
        ts.append(1e3 * e0.elapsed_time(e1))
    return {"us_median": round(float(np.median(ts)), 1), "us_min": round(min(ts), 1), "V_out": res[0].shape[0],
            "F_out": res[1].shape[0]}


def kernel_us(fn, v, f, reps=10):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn(v, f)
        torch.cuda.synchronize(dev)
    res = {}
    for e in prof.key_averages():
        m = re.search(r"\b(k_[a-z0-9_]+)", e.key)
        t = getattr(e, "self_device_time_total", None) or getattr(e, "self_cuda_time_total", 0.0)
        name = m.group(1) if m else ("memset" if "emset" in e.key else ("memcpy" if "emcpy" in e.key else None))
        if name and t:
            res[name] = round(res.get(name, 0.0) + t / reps, 2)
    return res


def host_s(fn, reps):
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        ts.append(time.perf_counter() - t0)
    return round(float(np.median(ts)) * 1e3, 2)


g = field()
for name, (v, f) in meshes(g):
    vn, fn = v.cpu().numpy(), f.cpu().numpy()
    row = {"V": vn.shape[0], "F": fn.shape[0], "min_faces": PP.min_faces_for(fn.shape[0]),
           "edge_components": int(len(np.unique(PP.edge_components(fn))))}
    for call, fnc in CALLS.items():
        row[call] = device_us(fnc, v, f)
        row[call]["kernels_us"] = kernel_us(fnc, v, f)
    m = hy3dgeo.Latent2MeshOutput(mesh_v=vn, mesh_f=fn)
    FR(m); DR(m)
    row["host_to_host_ms"] = {"FloaterRemover": host_s(lambda: FR(m), 10), "DegenerateFaceRemover": host_s(lambda: DR(m), 10),
                              "chain": host_s(lambda: DR(FR(m)), 10)}
    row["numpy_host_ms"] = {"remove_floaters": host_s(lambda: PP.remove_floaters(vn, fn), 3),
                            "weld": host_s(lambda: PP.weld(vn, fn), 3)}
    got = FR.run_device(v, f)
    ref = PP.remove_floaters(vn, fn)
    row["floaters_equal_numpy"] = bool(np.array_equal(got[1].cpu().numpy(), ref[1]) and
                                       np.array_equal(got[0].cpu().numpy().view(np.uint32), ref[0].view(np.uint32)))
    got = DR.run_device(v, f)
    ref = PP.weld(vn, fn)
    row["weld_equal_numpy"] = bool(np.array_equal(got[1].cpu().numpy(), ref[1]) and
                                   np.array_equal(got[0].cpu().numpy().view(np.uint32), ref[0].view(np.uint32)))
    out["meshes"][name] = row
    print(name, json.dumps(row), flush=True)

os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
json.dump(out, open(args.out, "w"), indent=1)
