#!/usr/bin/env python3
"""ORACLE (test infrastructure): generate ``tests/golden/*.npz`` by running the
REAL reference code (imported from /root/reference through ``ref_loader``) on
seeded inputs, and check the restatements in ``oracle/`` against it on the spot.

Run in the build container only:  ``python -m oracle.make_golden``
The reference tree cannot travel to the GPU box, the vectors can.  Weights are
not stored (too large): they are regenerated from ``hy3dgeo.weights`` seeds and
guarded by a checksum stored beside each vector.
"""
from __future__ import annotations

import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import hy3dgeo  # noqa: E402
from hy3dgeo import weights as W  # noqa: E402
from oracle import decoder as OD, volume as OV, mc as OM, ref_loader  # noqa: E402

GOLD = os.path.join(ROOT, "tests", "golden")


def checksum(sd) -> float:
    """Order-independent fingerprint of a state dict (guards RNG drift)."""
    return float(sum(float(v.double().abs().sum()) * (1 + (i % 7)) for i, (k, v) in enumerate(sorted(sd.items()))))


def analytic_field(p: torch.Tensor) -> torch.Tensor:
    """tanh sphere of SURVEY §8c: tanh(20 (0.6 - |p|))."""
    return torch.tanh(20 * (0.6 - p.float().norm(dim=-1)))


class AnalyticDecoder:
    """Fake ``geo_decoder`` for the reference volume decoders (SURVEY §4)."""
    def __call__(self, queries=None, latents=None):
        return analytic_field(queries)[..., None]

    def set_cross_attention_processor(self, p):
        pass


class stable_sort:
    """The reference orders refined FlashVDM queries with ``index.sort()``
    (volume_decoders.py:404), which is not stable; the stride-50/30 sub-sampling
    that follows depends on the tie order, so the reference's own output is
    implementation-defined there (probed: torch 2.11 CPU sort of 618 keys is
    NOT stable).  The canonical order fixed by this project is the stable one
    (SURVEY §7.3-5); goldens are generated with ``Tensor.sort`` defaulting to
    ``stable=True`` for the duration of the reference call.  The reference files
    are untouched."""
    def __enter__(self):
        self._orig = torch.Tensor.sort
        orig = self._orig

        def sort(t, *a, **k):
            if not a and "dim" not in k:
                k.setdefault("stable", True)
            return orig(t, *a, **k)
        torch.Tensor.sort = sort

    def __exit__(self, *exc):
        torch.Tensor.sort = self._orig


def maxdiff(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    m = np.isnan(a) & np.isnan(b)
    return float(np.max(np.abs(np.where(m, 0, a - b)))) if a.size else 0.0


def main():
    torch.set_num_threads(os.cpu_count())
    ns = ref_loader.load()
    os.makedirs(GOLD, exist_ok=True)
    report = []

    # ---------------------------------------------------------------- decoder
    for tag, cfg, nq in [("mini", W.MINI, 384), ("full", W.FULL, 256), ("turbo", W.MINI_TURBO, 384)]:
        sd = W.synthetic_state_dict(cfg, seed=0)
        vae = ref_loader.build_shapevae(ns, cfg, sd)              # strict load: pins key names/shapes
        z = W.synthetic_latents(cfg, batch=1, seed=1234)
        with torch.no_grad():
            lat = vae(z)                                          # ShapeVAE.forward
        g = torch.Generator().manual_seed(7)
        q = (torch.rand(1, nq, 3, generator=g) * 2 - 1) * 1.01
        with torch.no_grad():
            ref = vae.geo_decoder(queries=q, latents=lat)[0, :, 0]
        gsd = W.geo_decoder_state(sd)
        mine = OD.geo_decoder_forward(gsd, q, lat, W.fourier_frequencies(cfg), cfg.dec_heads)[0, :, 0]
        lat_mine = OD.shapevae_forward(sd, z, cfg.heads)
        d_dec, d_lat = maxdiff(ref, mine), maxdiff(lat, lat_mine)
        report.append(f"decoder[{tag}] oracle-vs-reference max|d| logits {d_dec:.2e}  transformer {d_lat:.2e} "
                      f"(|lat|max {float(lat.abs().max()):.1f})")
        assert d_dec < 2e-5 and d_lat < 2e-3 * max(1.0, float(lat.abs().max()) / 50)
        step = max(8, lat.shape[1] // 192)                        # at most 192 token rows: every file stays under 1 MB
        np.savez_compressed(os.path.join(GOLD, f"decoder_{tag}.npz"),
                            queries=q.numpy(), logits=ref.numpy(), latents_out_rows=lat[0, ::step].numpy(),
                            weight_checksum=checksum(sd), seed=0, latent_seed=1234)

    # ------------------------------------------- FlashVDM processors (selection)
    cfg = W.MINI
    sd = W.synthetic_state_dict(cfg, seed=0)
    vae = ref_loader.build_shapevae(ns, cfg, sd)
    z = W.synthetic_latents(cfg, 1, 1234)
    with torch.no_grad():
        lat = vae(z)
    gsd = W.geo_decoder_state(sd)
    g = torch.Generator().manual_seed(11)
    counts = [230, 77, 401]
    q = (torch.rand(1, sum(counts), 3, generator=g) * 2 - 1) * 1.01
    out = {}
    for mode, cls in [("mean", ns.ap.FlashVDMCrossAttentionProcessor), ("merge", ns.ap.FlashVDMTopMCrossAttentionProcessor)]:
        proc = cls()
        vae.geo_decoder.set_cross_attention_processor(proc)
        mine_p = OD.FlashProcessorOracle(mode)
        for state_name, state in [("level0", True), ("bins", ([3, 9, 40], counts))]:
            proc.topk = state if state is True else (list(state[0]), list(state[1]))
            with torch.no_grad():
                ref = vae.geo_decoder(queries=q, latents=lat)[0, :, 0]
            mine_p.topk = state
            mine = OD.geo_decoder_forward(gsd, q, lat, W.fourier_frequencies(cfg), cfg.dec_heads, kv_select=mine_p)[0, :, 0]
            d = maxdiff(ref, mine)
            report.append(f"flash processor[{mode},{state_name}] oracle-vs-reference max|d| {d:.2e}")
            assert d < 2e-5
            out[f"{mode}_{state_name}"] = ref.numpy()
            if mode == "mean":
                out[f"{mode}_{state_name}_sel"] = np.stack([s[0].numpy() for s in mine_p.last_selection]) \
                    if state is True else np.stack([s[0].numpy() for s in mine_p.last_selection])
    vae.geo_decoder.set_cross_attention_processor(ns.ap.CrossAttentionProcessor())
    np.savez_compressed(os.path.join(GOLD, "flash_processors_mini.npz"), queries=q.numpy(),
                        counts=np.array(counts), weight_checksum=checksum(sd), **out)

    # -------------------------------------------------- near-surface extraction
    rng = np.random.default_rng(5)
    grids, masks = [], []
    for t in range(5):
        gnp = rng.standard_normal((11, 12, 13)).astype(np.float32)
        gnp[rng.random(gnp.shape) < 0.15] = -10000.0
        gnp[rng.random(gnp.shape) < 0.05] = 0.0
        alpha = [0.0, 0.0, 0.3, -0.2, 0.0][t]
        import warnings
        with warnings.catch_warnings():
            warnings.simplefilter("ignore")
            ref = ns.vd.extract_near_surface_volume_fn(torch.from_numpy(gnp), alpha).numpy()
        mine = OV.near_surface_mask(gnp, alpha)
        assert np.array_equal(ref, mine), "near-surface restatement differs from reference"
        grids.append(gnp); masks.append(ref)
    report.append("near_surface: 5/5 random grids bit-identical to reference")
    np.savez_compressed(os.path.join(GOLD, "near_surface.npz"), grids=np.stack(grids), masks=np.stack(masks),
                        alphas=np.array([0.0, 0.0, 0.3, -0.2, 0.0], np.float32))

    # ------------------------------------ volume decoders on the analytic field
    fake = AnalyticDecoder()
    lat1 = torch.zeros(1, 4, 8)
    dec = lambda p: analytic_field(p)
    vol = {}
    with torch.no_grad():
        ref = ns.vd.VanillaVolumeDecoder()(lat1, fake, bounds=1.01, num_chunks=5000, octree_resolution=24,
                                           enable_pbar=False)[0].numpy()
    mine = OV.vanilla_decode(dec, 1.01, 5000, 24)
    assert np.array_equal(ref, mine)
    vol["vanilla24"] = ref
    for res, minres in [(64, 15), (128, 63)]:
        with torch.no_grad():
            ref = ns.PatchedHierarchicalVolumeDecoding()(lat1, fake, bounds=1.01, num_chunks=20000, mc_level=0.0,
                                                         octree_resolution=res, min_resolution=minres,
                                                         enable_pbar=False)[0].numpy()
        mine, st = OV.hierarchical_decode(dec, 1.01, 20000, 0.0, res, minres, return_stats=True)
        assert np.array_equal(np.isnan(ref), np.isnan(mine)) and maxdiff(ref, mine) == 0.0
        report.append(f"hierarchical(patched) res {res}: levels {st['levels']} queries {st['queries']} "
                      f"visited {int((~np.isnan(ref)).sum())}  bit-identical")
        vol[f"hier{res}_visited"] = np.array(int((~np.isnan(ref)).sum()))
        vol[f"hier{res}_queries"] = np.array(st["queries"])
        if res == 64:
            vol["hier64"] = ref
    for res, minres in [(64, 15), (128, 63)]:
        fl = ns.vd.FlashVDMVolumeDecoding("mean")
        with torch.no_grad():
            ref = fl(lat1, fake, bounds=1.01, num_chunks=20000, mc_level=0.0, octree_resolution=res,
                     min_resolution=minres, enable_pbar=False)[0].numpy()
        mine, st = OV.flashvdm_decode(lambda p, topk: analytic_field(p), 1.01, 20000, 0.0, res, minres,
                                      return_stats=True)
        assert np.array_equal(np.isnan(ref), np.isnan(mine)) and maxdiff(ref, mine) == 0.0
        report.append(f"flashvdm res {res}: levels {st['levels']} queries {st['queries']} "
                      f"visited {int((~np.isnan(ref)).sum())}  bit-identical")
        vol[f"flash{res}_visited"] = np.array(int((~np.isnan(ref)).sum()))
        vol[f"flash{res}_queries"] = np.array(st["queries"])
        if res == 64:
            vol["flash64"] = ref
    np.savez_compressed(os.path.join(GOLD, "volume_analytic.npz"), **vol)

    # ---------------- volume decoders on the real decoder (sparse random field)
    cfg = W.MINI
    sd = W.sparsify_field(W.synthetic_state_dict(cfg, seed=0), cfg, keep_freqs=2, gain=6.0, bias=-2.0)
    vae = ref_loader.build_shapevae(ns, cfg, sd)
    gsd = W.geo_decoder_state(sd)
    fr = W.fourier_frequencies(cfg)
    with torch.no_grad():
        lat = vae(W.synthetic_latents(cfg, 1, 1234))
    kw = dict(bounds=1.01, num_chunks=3000, mc_level=0.0, octree_resolution=32, min_resolution=15, enable_pbar=False)
    with torch.no_grad():
        ref_h = ns.PatchedHierarchicalVolumeDecoding()(lat, vae.geo_decoder, **kw)[0].numpy()
    dec_real = lambda p: OD.geo_decoder_forward(gsd, p[None], lat, fr, cfg.dec_heads)[0, :, 0]
    mine_h, st = OV.hierarchical_decode(dec_real, 1.01, 3000, 0.0, 32, 15, return_stats=True)
    same_set = np.array_equal(np.isnan(ref_h), np.isnan(mine_h))
    report.append(f"hierarchical on real decoder res 32: queries {st['queries']} visited {int((~np.isnan(ref_h)).sum())} "
                  f"same visited set {same_set}  max|d| {maxdiff(ref_h, mine_h):.2e}")
    assert same_set and maxdiff(ref_h, mine_h) < 5e-5
    out = {"hier32": ref_h}
    for mode in ("mean", "merge"):
        fl = ns.vd.FlashVDMVolumeDecoding(mode)
        with torch.no_grad(), stable_sort():
            ref_f = fl(lat, vae.geo_decoder, **kw)[0].numpy()
        proc = OD.FlashProcessorOracle(mode)

        def dec_group(p, topk, proc=proc):
            proc.topk = topk
            G = p.shape[0]
            return OD.geo_decoder_forward(gsd, p, lat.expand(G, -1, -1), fr, cfg.dec_heads, kv_select=proc)[..., 0]
        mine_f, st = OV.flashvdm_decode(dec_group, 1.01, 3000, 0.0, 32, 15, return_stats=True)
        same_set = np.array_equal(np.isnan(ref_f), np.isnan(mine_f))
        report.append(f"flashvdm[{mode}] on real decoder res 32: levels {st['levels']} queries {st['queries']} "
                      f"same visited set {same_set}  max|d| {maxdiff(ref_f, mine_f):.2e}")
        assert same_set and maxdiff(ref_f, mine_f) < 5e-5
        out[f"flash32_{mode}"] = ref_f
    vae.geo_decoder.set_cross_attention_processor(ns.ap.CrossAttentionProcessor())
    np.savez_compressed(os.path.join(GOLD, "volume_decoder_mini.npz"), weight_checksum=checksum(sd),
                        gain=6.0, bias=-2.0, keep_freqs=2, **out)

    # --------------------- latents2mesh through the reference with the oracle MC
    # (pins the extractor contract: None-on-error, rescale by res+1, dtypes)
    vae.volume_decoder = ns.vd.VanillaVolumeDecoder()
    with torch.no_grad():
        outs = vae.latents2mesh(lat, bounds=1.01, mc_level=0.0, num_chunks=3000, octree_resolution=24,
                                mc_algo="mc", enable_pbar=False)
    assert outs[0] is not None
    grid24 = OV.vanilla_decode(dec_real, 1.01, 3000, 24)
    v2, f2 = OM.mc_surface_extract(grid24, mc_level=0.0, bounds=1.01, octree_resolution=24)
    report.append(f"latents2mesh res 24 via reference + oracle MC: V {outs[0].mesh_v.shape[0]} F {outs[0].mesh_f.shape[0]}"
                  f" dtype {outs[0].mesh_v.dtype}/{outs[0].mesh_f.dtype}; restated extractor max|dv| "
                  f"{maxdiff(outs[0].mesh_v, v2) if outs[0].mesh_v.shape == v2.shape else float('nan'):.2e}")
    np.savez_compressed(os.path.join(GOLD, "latents2mesh_mini24.npz"), mesh_v=outs[0].mesh_v, mesh_f=outs[0].mesh_f,
                        weight_checksum=checksum(sd))

    with open(os.path.join(GOLD, "REPORT.txt"), "w") as f:
        f.write("Generated by oracle/make_golden.py against /root/reference (torch %s)\n" % torch.__version__)
        f.write("\n".join(report) + "\n")
    print("\n".join(report))



# =====================================================================================================================
# Round 2 vectors (``python -m oracle.make_golden r2``): the BASELINE configurations that round 1 left unpinned —
# 3-level and odd-level Hierarchical, FlashVDM on the mini-turbo and the full decoder (mean + merge), include_pi,
# and an end-to-end mesh of >= 10k vertices.  Written to separate files so the round-1 vectors stay byte-identical.
# =====================================================================================================================
SPARSE = {           # (keep_freqs, gain, bias) of hy3dgeo.weights.sparsify_field per decoder config, chosen so that the
    "mini": (4, 4.0, 0.3),       # octree-32/64 levels have a partial band (neither empty nor everything); 13.5k-vertex mesh at 64
    "turbo": (2, 60.0, -16.0),
    "full": (2, 6.0, 1.5),
}


def _flash_pair(ns, vae, lat, gsd, fr, cfg, mode, kw):
    """Reference FlashVDMVolumeDecoding(mode) (stable bin order) and the oracle restatement on the same inputs."""
    fl = ns.vd.FlashVDMVolumeDecoding(mode)
    with torch.no_grad(), stable_sort():
        ref = fl(lat, vae.geo_decoder, **kw)[0].numpy()
    proc = OD.FlashProcessorOracle(mode)

    def dec_group(p, topk, proc=proc):
        proc.topk = topk
        return OD.geo_decoder_forward(gsd, p, lat.expand(p.shape[0], -1, -1), fr, cfg.dec_heads, kv_select=proc)[..., 0]
    mine, st = OV.flashvdm_decode(dec_group, kw["bounds"], kw["num_chunks"], kw["mc_level"], kw["octree_resolution"],
                                  kw["min_resolution"], return_stats=True)
    vae.geo_decoder.set_cross_attention_processor(ns.ap.CrossAttentionProcessor())
    return ref, mine, st


def main_r2():
    torch.set_num_threads(os.cpu_count())
    ns = ref_loader.load()
    report = []
    fake = AnalyticDecoder()
    lat1 = torch.zeros(1, 4, 8)

    # ------------------------------------------------ Hierarchical with odd intermediate levels (r // 2, vd:202-208)
    vol = {}
    for res, minres in [(35, 8), (45, 10), (70, 15)]:
        with torch.no_grad():
            ref = ns.PatchedHierarchicalVolumeDecoding()(lat1, fake, bounds=1.01, num_chunks=20000, mc_level=0.0,
                                                         octree_resolution=res, min_resolution=minres, enable_pbar=False)[0].numpy()
        mine, st = OV.hierarchical_decode(lambda p: analytic_field(p), 1.01, 20000, 0.0, res, minres, return_stats=True)
        assert np.array_equal(np.isnan(ref), np.isnan(mine)) and maxdiff(ref, mine) == 0.0
        report.append(f"hierarchical(patched) res {res}: levels {st['levels']} (grids {[l + 1 for l in st['levels']]}) queries "
                      f"{st['queries']}  bit-identical")
        vol[f"hier{res}_queries"] = np.array(st["queries"])
        if res in (35, 45):
            vol[f"hier{res}"] = ref
    np.savez_compressed(os.path.join(GOLD, "volume_analytic_r2.npz"), **vol)

    # ------------------------------------------------ real mini decoder: 3 levels (octree 64) and odd levels (octree 35)
    cfg = W.MINI
    kf, gain, bias = SPARSE["mini"]
    sd = W.sparsify_field(W.synthetic_state_dict(cfg, seed=0), cfg, keep_freqs=kf, gain=gain, bias=bias)
    vae = ref_loader.build_shapevae(ns, cfg, sd)
    gsd, fr = W.geo_decoder_state(sd), W.fourier_frequencies(cfg)
    with torch.no_grad():
        lat = vae(W.synthetic_latents(cfg, 1, 1234))
    dec_real = lambda p: OD.geo_decoder_forward(gsd, p[None], lat, fr, cfg.dec_heads)[0, :, 0]
    out = {"gain": gain, "bias": bias, "keep_freqs": kf, "weight_checksum": checksum(sd)}
    for res, minres in [(64, 15), (35, 8)]:
        kw = dict(bounds=1.01, num_chunks=8000, mc_level=0.0, octree_resolution=res, min_resolution=minres, enable_pbar=False)
        with torch.no_grad():
            ref = ns.PatchedHierarchicalVolumeDecoding()(lat, vae.geo_decoder, **kw)[0].numpy()
        mine, st = OV.hierarchical_decode(dec_real, 1.01, 8000, 0.0, res, minres, return_stats=True)
        same = np.array_equal(np.isnan(ref), np.isnan(mine))
        report.append(f"hierarchical on real mini decoder res {res}: levels {st['levels']} queries {st['queries']} same visited set {same} "
                      f"max|d| {maxdiff(ref, mine):.2e}")
        assert same and maxdiff(ref, mine) < 5e-5 and len(st["levels"]) == 3
        out[f"hier{res}"] = ref
        out[f"hier{res}_queries"] = np.array(st["queries"])
    # ---- end-to-end mesh: reference latents2mesh (Vanilla, octree 64) with the oracle MC standing in for skimage
    vae.volume_decoder = ns.vd.VanillaVolumeDecoder()
    with torch.no_grad():
        outs = vae.latents2mesh(lat, bounds=1.01, mc_level=0.0, num_chunks=8000, octree_resolution=64, mc_algo="mc", enable_pbar=False)
    assert outs[0] is not None
    grid64 = OV.vanilla_decode(dec_real, 1.01, 8000, 64)
    v2, f2 = OM.mc_surface_extract(grid64, mc_level=0.0, bounds=1.01, octree_resolution=64)
    same_mesh = outs[0].mesh_f.shape == f2.shape and np.array_equal(outs[0].mesh_f, f2)
    report.append(f"latents2mesh res 64 via reference + oracle MC: V {outs[0].mesh_v.shape[0]} F {outs[0].mesh_f.shape[0]}; restated "
                  f"pipeline same faces {same_mesh} max|dv| {maxdiff(outs[0].mesh_v, v2) if outs[0].mesh_v.shape == v2.shape else float('nan'):.2e}")
    assert outs[0].mesh_v.shape[0] >= 10000
    np.savez_compressed(os.path.join(GOLD, "volume_decoder_mini_r2.npz"), **out)
    np.savez_compressed(os.path.join(GOLD, "latents2mesh_mini64.npz"), mesh_v=outs[0].mesh_v, mesh_f=outs[0].mesh_f,
                        gain=gain, bias=bias, keep_freqs=kf, weight_checksum=checksum(sd))

    # ------------------------------------------------ FlashVDM on the mini-turbo decoder (BASELINE config 4) and the full one
    for tag, cfg, cases in [("turbo", W.MINI_TURBO, [(32, 15), (64, 15)]), ("full", W.FULL, [(32, 15)])]:
        kf, gain, bias = SPARSE[tag]
        sd = W.sparsify_field(W.synthetic_state_dict(cfg, seed=0), cfg, keep_freqs=kf, gain=gain, bias=bias)
        vae = ref_loader.build_shapevae(ns, cfg, sd)
        gsd, fr = W.geo_decoder_state(sd), W.fourier_frequencies(cfg)
        with torch.no_grad():
            lat = vae(W.synthetic_latents(cfg, 1, 1234))
        out = {"gain": gain, "bias": bias, "keep_freqs": kf, "weight_checksum": checksum(sd)}
        for res, minres in cases:
            kw = dict(bounds=1.01, num_chunks=600, mc_level=0.0, octree_resolution=res, min_resolution=minres, enable_pbar=False)
            for mode in ("mean", "merge"):
                ref, mine, st = _flash_pair(ns, vae, lat, gsd, fr, cfg, mode, kw)
                same = np.array_equal(np.isnan(ref), np.isnan(mine))
                report.append(f"flashvdm[{mode}] on real {tag} decoder res {res}: levels {st['levels']} queries {st['queries']} "
                              f"same visited set {same} max|d| {maxdiff(ref, mine):.2e}")
                assert same and maxdiff(ref, mine) < 5e-5 * max(1.0, gain / 6.0)
                out[f"flash{res}_{mode}"] = ref
                out[f"flash{res}_{mode}_queries"] = np.array(st["queries"])
        np.savez_compressed(os.path.join(GOLD, f"flash_{tag}.npz"), **out)

    # ------------------------------------------------ include_pi=True decoder (attention_blocks.py:93-94)
    import dataclasses
    cfg = dataclasses.replace(W.MINI, include_pi=True)
    sd = W.synthetic_state_dict(cfg, seed=0)
    vae = ref_loader.build_shapevae(ns, cfg, sd)
    assert abs(float(vae.geo_decoder.fourier_embedder.frequencies[0]) - np.pi) < 1e-6
    with torch.no_grad():
        lat = vae(W.synthetic_latents(cfg, 1, 1234))
        q = (torch.rand(1, 384, 3, generator=torch.Generator().manual_seed(7)) * 2 - 1) * 1.01
        ref = vae.geo_decoder(queries=q, latents=lat)[0, :, 0]
    mine = OD.geo_decoder_forward(W.geo_decoder_state(sd), q, lat, W.fourier_frequencies(cfg), cfg.dec_heads)[0, :, 0]
    report.append(f"decoder[mini, include_pi] oracle-vs-reference max|d| logits {maxdiff(ref, mine):.2e}")
    assert maxdiff(ref, mine) < 2e-5
    np.savez_compressed(os.path.join(GOLD, "decoder_pi.npz"), queries=q.numpy(), logits=ref.numpy(), weight_checksum=checksum(sd),
                        seed=0, latent_seed=1234)

    with open(os.path.join(GOLD, "REPORT_r2.txt"), "w") as f:
        f.write("Generated by `python -m oracle.make_golden r2` against /root/reference (torch %s)\n" % torch.__version__)
        f.write("\n".join(report) + "\n")
    print("\n".join(report))


if __name__ == "__main__":
    if len(sys.argv) > 1 and sys.argv[1] == "r2":
        main_r2()
    else:
        main()
