#!/usr/bin/env python3
"""FaceReducer at BASELINE configs[2] mesh scale: ``hy3d_mesh_decimate`` on the marching-cubes mesh of the 385^3 field of
tools/gpu_postprocess_bench.py (a hollow, bumpy body plus 60 small spheres, ~0.97 M faces) after ``FloaterRemover`` and
``DegenerateFaceRemover``, as the front ends run them, at the front ends' target of 40 000 faces and at 200 000.

Records per target: device time of ``run_device`` (CUDA events, after warm-up, median of --reps), the rounds (one host
synchronisation each), the host-to-host call a user makes on a ``Latent2MeshOutput`` (wall clock, ends in a
synchronisation), the numpy statement oracle/decimate.py on the host (one run) and whether the two are bit-equal.
pymeshlab is not installed, so the reference filter is not measured.

    python tools/gpu_decimate_bench.py --out profiles/r05_decimate_bench.json
"""
import argparse, json, os, subprocess, sys, time
import numpy as np, torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import hy3dgeo
from hy3dgeo import _lib
from hy3dgeo.postprocessors import FaceReducer
from oracle import decimate as D

ap = argparse.ArgumentParser()
ap.add_argument("--out", default="decimate_bench.json")
ap.add_argument("--reps", type=int, default=10)
ap.add_argument("--targets", default="40000,200000")
args = ap.parse_args()
dev = torch.device("cuda:0")
ctx = _lib.get_context(dev)
q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                   capture_output=True, text=True).stdout.strip()
out = {"device": torch.cuda.get_device_name(dev), "nvidia_smi_name_power_limit_max_sm_clock": q, "reps": args.reps,
       "pymeshlab": "not measured (not installed)", "targets": {}}
print(out["device"], "|", q, flush=True)


def field(n=385):
    x = torch.linspace(-1.01, 1.01, n, device=dev)
    X, Y, Z = x[:, None, None], x[None, :, None], x[None, None, :]
    R = torch.sqrt(X * X + Y * Y + Z * Z)
    d = torch.minimum(0.62 + 0.1 * torch.sin(20 * X) * torch.sin(20 * Y) * torch.sin(20 * Z) - R, R - 0.35)
    rng = np.random.default_rng(7)
    for c, r in zip(rng.uniform(-0.95, 0.95, (60, 3)), rng.uniform(0.008, 0.03, 60)):
        d = torch.maximum(d, float(r) - torch.sqrt((X - float(c[0])) ** 2 + (Y - float(c[1])) ** 2 + (Z - float(c[2])) ** 2))
    return torch.tanh(20 * d).float().contiguous()


FR, DR, RED = hy3dgeo.FloaterRemover(), hy3dgeo.DegenerateFaceRemover(), FaceReducer()
v, f = hy3dgeo.MCSurfaceExtractor(cull_nonfinite=True).run_device(field(), mc_level=0.0, bounds=1.01, octree_resolution=384)
v, f = DR.run_device(*FR.run_device(v, f))
vn, fn = v.cpu().numpy(), f.cpu().numpy()
out["input"] = {"V": vn.shape[0], "F": fn.shape[0], "after": "MC 385^3 -> FloaterRemover -> DegenerateFaceRemover"}
print(json.dumps(out["input"]), flush=True)

for T in [int(t) for t in args.targets.split(",")]:
    for _ in range(2):
        ctx.mesh_decimate(v, f, T)
    torch.cuda.synchronize(dev)
    ts = []
    for _ in range(args.reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        vo, fo, rounds = ctx.mesh_decimate(v, f, T)
        e1.record(); e1.synchronize()
        ts.append(e0.elapsed_time(e1))
    m = hy3dgeo.Latent2MeshOutput(mesh_v=vn, mesh_f=fn)
    RED(m, max_facenum=T)
    hs = []
    for _ in range(3):
        t0 = time.perf_counter()
        RED(m, max_facenum=T)
        hs.append(time.perf_counter() - t0)
    t0 = time.perf_counter()
    ref = D.decimate(vn, fn, T)
    oracle_s = time.perf_counter() - t0
    row = {"V_out": vo.shape[0], "F_out": fo.shape[0], "rounds": rounds,
           "device_ms_median": round(float(np.median(ts)), 2), "device_ms_min": round(min(ts), 2),
           "device_ms_per_round": round(float(np.median(ts)) / max(rounds, 1), 3),
           "host_to_host_ms_median": round(float(np.median(hs)) * 1e3, 2), "numpy_oracle_host_s": round(oracle_s, 1),
           "equal_numpy": bool(ref[2] == rounds and np.array_equal(fo.cpu().numpy(), ref[1]) and
                               np.array_equal(vo.cpu().numpy().view(np.uint32), ref[0].view(np.uint32)))}
    out["targets"][str(T)] = row
    print(T, json.dumps(row), flush=True)

os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
json.dump(out, open(args.out, "w"), indent=1)
