#!/usr/bin/env python3
"""Device-side diagnostics (run on a B200): checks every kernel family against the
oracle, the decoder in both precisions (fp32 SIMT and tcgen05), so that a single GPU trip localises
a bug.  Not a test, not a benchmark."""
import os
import sys
import time
import traceback

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import hy3dgeo  # noqa: E402
from hy3dgeo import weights as W  # noqa: E402
from hy3dgeo import _lib  # noqa: E402
from hy3dgeo.model import B200ShapeVAE  # noqa: E402
from hy3dgeo.volume_decoders import VanillaVolumeDecoder, HierarchicalVolumeDecoding, bind  # noqa: E402
from hy3dgeo.surface_extractors import MCSurfaceExtractor  # noqa: E402
from oracle import decoder as OD, volume as OV, mc as OM  # noqa: E402

dev = torch.device("cuda:0")


def section(name):
    print(f"\n===== {name} =====", flush=True)


def mc_check():
    section("marching cubes vs oracle")
    ctx = _lib.get_context(dev)
    rng = np.random.default_rng(0)
    n = 65
    x = np.linspace(-1.01, 1.01, n, dtype=np.float32)
    X, Y, Z = np.meshgrid(x, x, x, indexing="ij")
    sphere = np.tanh(20 * (0.6 - np.sqrt(X * X + Y * Y + Z * Z))).astype(np.float32)
    noise = rng.standard_normal((33, 40, 70)).astype(np.float32)
    nan = sphere.copy()
    nan[np.abs(nan) > 0.999] = np.nan
    for name, vol in [("sphere65", sphere), ("noise33x40x70", noise), ("sphere+nan", nan)]:
        g = torch.from_numpy(vol).to(dev)
        cases = ctx.mc_cases(g, 0.0).cpu().numpy()
        ok_cases = np.array_equal(cases, OM.cube_cases(vol, 0.0))
        nv, nf, mm = ctx.mc_count(g, 0.0)
        v = torch.empty((nv, 3), dtype=torch.float32, device=dev)
        f = torch.empty((nf, 3), dtype=torch.int32, device=dev)
        ctx.mc_emit([1, 1, 1], [1, 1, 1], [0, 0, 0], v, f)
        v, f = v.cpu().numpy(), f.cpu().numpy()
        vo, fo, _, _ = OM.marching_cubes(vol, 0.0) if not np.isnan(vol).any() else _nan_mc(vol)
        same_v = v.shape == vo.shape and np.array_equal(v.view(np.uint32), vo.view(np.uint32))
        same_f = f.shape == fo.shape and np.array_equal(f, fo)
        print(f"{name}: cases {ok_cases}  V {nv}/{vo.shape[0]}  F {nf}/{fo.shape[0]}  verts bit-exact {same_v}  faces exact {same_f}"
              f"  minmax {mm}")
        if not same_v and v.shape == vo.shape:
            d = np.abs(np.nan_to_num(v) - np.nan_to_num(vo))
            print("   max |dv|", d.max(), "first mismatch", np.argwhere(v.view(np.uint32) != vo.view(np.uint32))[:3])
        if not same_f and f.shape == fo.shape:
            print("   first face mismatches", np.argwhere(f != fo)[:5], f[:3], fo[:3])


def _nan_mc(vol):
    import ctypes
    # the oracle front-end range check chokes on NaN like numpy min/max would not; call through directly
    lib = OM._load()
    pv, pf = ctypes.c_void_p(), ctypes.c_void_p()
    nv, nf = ctypes.c_int64(), ctypes.c_int64()
    vol = np.ascontiguousarray(vol, np.float32)
    lib.hy3d_oracle_mc(vol.ctypes.data, *vol.shape, 0.0, ctypes.byref(pv), ctypes.byref(nv), ctypes.byref(pf), ctypes.byref(nf))
    V, Fc = nv.value, nf.value
    verts = np.ctypeslib.as_array(ctypes.cast(pv, ctypes.POINTER(ctypes.c_float)), shape=(max(V, 1), 3))[:V].copy()
    faces = np.ctypeslib.as_array(ctypes.cast(pf, ctypes.POINTER(ctypes.c_int32)), shape=(max(Fc, 1), 3))[:Fc].copy()
    return verts, faces, None, None


def octree_check():
    section("octree refinement vs oracle")
    ctx = _lib.get_context(dev)
    rng = np.random.default_rng(1)
    n = 33
    x = np.linspace(-1.01, 1.01, n, dtype=np.float32)
    X, Y, Z = np.meshgrid(x, x, x, indexing="ij")
    g = np.tanh(20 * (0.6 - np.sqrt(X * X + Y * Y + Z * Z))).astype(np.float32)
    g2 = g.copy()
    g2[rng.random(g2.shape) < 0.3] = -10000.0
    g3 = rng.standard_normal((17, 17, 17)).astype(np.float32) * 2
    for name, grid in [("sphere33", g), ("sphere33+sentinels", g2), ("noise17", g3)]:
        for last in (False, True):
            want = np.flatnonzero(OV.refine_active_set(grid, 0.0, last).reshape(-1))
            t = torch.from_numpy(grid).to(dev)
            idx = torch.empty(max(want.size * 2, 16), dtype=torch.int32, device=dev)
            cnt = ctx.refine_level(t, 0.0, last, idx)
            got = idx[:cnt].cpu().numpy()
            print(f"{name} last={last}: count {cnt}/{want.size} exact {cnt == want.size and np.array_equal(got, want)}")


def decoder_check(tag, cfg, nq):
    section(f"decoder {tag}: SIMT and tcgen05 vs oracle")
    sd = W.synthetic_state_dict(cfg, seed=0)
    vae = B200ShapeVAE(cfg, sd, device=dev)
    z = W.synthetic_latents(cfg, 1, 1234)
    t0 = time.time()
    lat_o = OD.shapevae_forward(sd, z, cfg.heads)
    lat = vae(z.to(dev))
    print(f"transformer: max|gpu-oracle| {float((lat.cpu() - lat_o).abs().max()):.2e}  (oracle {time.time() - t0:.1f}s)")
    g = torch.Generator().manual_seed(7)
    q = (torch.rand(1, nq, 3, generator=g) * 2 - 1) * 1.01
    gold = np.load(os.path.join(ROOT, "tests", "golden", f"decoder_{tag}.npz"))
    gsd = W.geo_decoder_state(sd)
    ref = OD.geo_decoder_forward(gsd, q, lat_o, W.fourier_frequencies(cfg), cfg.dec_heads)[0, :, 0]
    if np.array_equal(gold["queries"], q.numpy()):
        print(f"oracle vs golden(reference) {float(np.abs(gold['logits'] - ref.numpy()).max()):.2e}")
    ctx = bind(lat, vae.geo_decoder)
    ctx.prepare_kv(lat_o[0].to(dev))
    outs = {}
    for name, prec in [("simt", _lib.PRECISION_FP32_SIMT), ("tc", _lib.PRECISION_FP16_TC)]:
        try:
            ctx.set_precision(prec)
            t0 = time.time()
            o = ctx.decode_points(q[0].to(dev))
            wd = ctx.watchdog()
            torch.cuda.synchronize()
            outs[name] = o.cpu()
            print(f"{name}: max|d| vs oracle {float((outs[name] - ref).abs().max()):.3e}  rms {float((outs[name] - ref).pow(2).mean().sqrt()):.3e}"
                  f"  ({time.time() - t0:.2f}s) watchdog {wd[:5]}  logits std {float(ref.std()):.3f}")
        except Exception:
            traceback.print_exc()
    ctx.set_precision(_lib.PRECISION_FP16_TC)
    return vae, lat_o


def volume_check(vae, lat_o):
    section("volume decoders end to end")
    cfg = vae.cfg
    sd = W.sparsify_field(W.synthetic_state_dict(cfg, seed=0), cfg, keep_freqs=2, gain=6.0, bias=-2.0)
    vae2 = B200ShapeVAE(cfg, sd, device=dev)
    gold = np.load(os.path.join(ROOT, "tests", "golden", "volume_decoder_mini.npz"))
    lat = lat_o.to(dev)
    ctx = _lib.get_context(dev)
    for prec_name, prec in [("simt", _lib.PRECISION_FP32_SIMT), ("tc", _lib.PRECISION_FP16_TC)]:
        try:
            ctx.set_precision(prec)
            h = HierarchicalVolumeDecoding()
            grid = h(lat, vae2.geo_decoder, bounds=1.01, num_chunks=3000, mc_level=0.0, octree_resolution=32, min_resolution=15)[0].cpu().numpy()
            ref = gold["hier32"]
            same = np.array_equal(np.isnan(grid), np.isnan(ref))
            d = np.abs(np.nan_to_num(grid) - np.nan_to_num(ref)).max() if same else float("nan")
            print(f"hier32[{prec_name}]: queries {h.last_stats[0]['queries']} same visited set {same} max|d| {d:.3e}")
            v = VanillaVolumeDecoder()(lat, vae2.geo_decoder, bounds=1.01, octree_resolution=24)
            outs = MCSurfaceExtractor()(v, mc_level=0.0, bounds=1.01, octree_resolution=24)
            g24 = np.load(os.path.join(ROOT, "tests", "golden", "latents2mesh_mini24.npz"))
            print(f"latents2mesh24[{prec_name}]: V {None if outs[0] is None else outs[0].mesh_v.shape} F "
                  f"{None if outs[0] is None else outs[0].mesh_f.shape} golden V {g24['mesh_v'].shape} F {g24['mesh_f'].shape}")
        except Exception:
            traceback.print_exc()
    ctx.set_precision(_lib.PRECISION_FP16_TC)


def speed_check(vae, lat_o):
    section("tcgen05 decoder speed (dense 129^3, mini)")
    ctx = _lib.get_context(dev)
    ctx.set_precision(_lib.PRECISION_FP16_TC)
    lat = lat_o.to(dev)
    dec = VanillaVolumeDecoder()
    for res in (64, 128):
        for rep in range(2):
            torch.cuda.synchronize(); t0 = time.time()
            g = dec(lat, vae.geo_decoder, bounds=1.01, octree_resolution=res)
            torch.cuda.synchronize(); dt = time.time() - t0
            n = (res + 1) ** 3
            fl = n * (21078016 + 4096 * lat.shape[1])
            print(f"res {res}: {dt * 1e3:.1f} ms  {n / dt / 1e6:.2f} Mpts/s  {fl / dt / 1e12:.1f} TFLOP/s  watchdog {ctx.watchdog()[:3]}"
                  f"  finite {bool(torch.isfinite(g).all())}")


if __name__ == "__main__":
    print(torch.cuda.get_device_name(0))
    which = sys.argv[1:] or ["mc", "octree", "mini", "volume", "speed", "full", "turbo"]
    vae = lat = None
    for w in which:
        try:
            if w == "mc":
                mc_check()
            elif w == "octree":
                octree_check()
            elif w == "mini":
                vae, lat = decoder_check("mini", W.MINI, 384)
            elif w == "full":
                decoder_check("full", W.FULL, 256)
            elif w == "turbo":
                decoder_check("turbo", W.MINI_TURBO, 384)
            elif w == "volume" and vae is not None:
                volume_check(vae, lat)
            elif w == "speed" and vae is not None:
                speed_check(vae, lat)
        except Exception:
            traceback.print_exc()
