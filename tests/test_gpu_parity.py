"""GPU parity tests (pytest -m gpu, run on a B200): the CUDA path through the C-ABI against the
oracle on the same seeded inputs, against the committed golden vectors from the real reference,
and — at BASELINE sizes — through size-independent properties.

Tolerances (north_star): logits within 1e-3 abs of the fp32 reference for the O(1)-scale field;
bit-exact cube classification, active-cell sets and face indexing given the same field; Chamfer
distance < 1e-4 of the bbox diagonal.
"""
import os

import numpy as np
import pytest
import torch

import hy3dgeo
from hy3dgeo import _lib, weights as W
from hy3dgeo.surface_extractors import MCSurfaceExtractor
from hy3dgeo.volume_decoders import HierarchicalVolumeDecoding, VanillaVolumeDecoder, bind
from oracle import decoder as OD, mc as OM, volume as OV
from oracle.mesh import bits_equal

pytestmark = pytest.mark.gpu
CFG = {"mini": W.MINI, "full": W.FULL, "turbo": W.MINI_TURBO}
LOGIT_TOL = 1e-3


@pytest.fixture(scope="module")
def dev():
    return torch.device("cuda:0")


@pytest.fixture(scope="module")
def ctx(dev):
    return _lib.get_context(dev)


def sphere(n, r=0.6, sharp=20.0):
    x = np.linspace(-1.01, 1.01, n, dtype=np.float32)
    X, Y, Z = np.meshgrid(x, x, x, indexing="ij")
    return np.tanh(sharp * (r - np.sqrt(X * X + Y * Y + Z * Z))).astype(np.float32)


def gpu_mc(ctx, vol, level, div=(1, 1, 1), mul=(1, 1, 1), add=(0, 0, 0)):
    g = torch.from_numpy(np.ascontiguousarray(vol)).cuda()
    nv, nf, mm = ctx.mc_count(g, level)
    v = torch.empty((nv, 3), dtype=torch.float32, device="cuda")
    f = torch.empty((nf, 3), dtype=torch.int32, device="cuda")
    ctx.mc_emit(div, mul, add, v, f)
    return v.cpu().numpy(), f.cpu().numpy(), mm


# ------------------------------------------------------------------------------ marching cubes
@pytest.mark.parametrize("shape,level", [((2, 2, 2), 0.0), ((3, 5, 33), 0.1), ((17, 9, 32), 0.0), ((9, 31, 65), -0.2),
                                         ((20, 21, 97), 0.0), ((6, 7, 300), 0.05), ((4, 5, 600), 0.0)])
def test_mc_random_fields_bit_exact(ctx, shape, level):
    """Noise fields cross the level on half of all edges: every emit work list overflows its 256 entries several times
    (rows of 97 / 300 / 600 voxels exercise the 8-, 16- and 32-lane row layouts)."""
    rng = np.random.default_rng(sum(shape))
    vol = rng.standard_normal(shape).astype(np.float32)
    assert np.array_equal(ctx.mc_cases(torch.from_numpy(vol).cuda(), level).cpu().numpy(), OM.cube_cases(vol, level))
    v, f, _ = gpu_mc(ctx, vol, level)
    vo, fo = OM.marching_cubes_raw(vol, level)
    assert bits_equal(v, vo) and np.array_equal(f, fo)


def test_mc_sphere_nan_and_exact_zero(ctx):
    vol = sphere(65)
    vol[10, 10, 10] = 0.0                                   # exact level value: "v - level > 0" is false
    v, f, mm = gpu_mc(ctx, vol, 0.0)
    vo, fo = OM.marching_cubes_raw(vol, 0.0)
    assert bits_equal(v, vo) and np.array_equal(f, fo) and f.shape[0] == 2 * v.shape[0] - 4
    assert mm[0] == vol.min() and mm[1] == vol.max() and mm[2] is False
    nanv = vol.copy()
    nanv[np.abs(nanv) > 0.999] = np.nan                     # unvisited voxels of the sparse decoders
    v, f, mm = gpu_mc(ctx, nanv, 0.0)
    vo, fo = OM.marching_cubes_raw(nanv, 0.0)
    assert bits_equal(v, vo) and np.array_equal(f, fo) and mm[2] is True and np.isnan(v).any()


def test_mc_extractor_contract(dev):
    """MCSurfaceExtractor.run/__call__ vs the restated reference call (surface_extractors.py:50-76):
    float64 rescale by res+1 (also when the grid is smaller than res+1, FlashVDM), dtypes, None on error."""
    ext = MCSurfaceExtractor()
    vol = sphere(61)
    for res, bounds in [(60, 1.01), (64, 1.01), (60, [-1.0, -0.5, -2.0, 1.0, 1.5, 2.0])]:
        v, f = ext.run(torch.from_numpy(vol).to(dev), mc_level=0.0, bounds=bounds, octree_resolution=res)
        vo, fo = OM.mc_surface_extract(vol, mc_level=0.0, bounds=bounds, octree_resolution=res)
        assert v.dtype == np.float32 and f.dtype == np.int32 and f.flags["C_CONTIGUOUS"]
        assert bits_equal(v, vo) and np.array_equal(f, fo)
    batch = torch.from_numpy(np.stack([vol, np.full_like(vol, -1.0)])).to(dev)
    outs = ext(batch, mc_level=0.0, bounds=1.01, octree_resolution=60, mc_algo="mc", num_chunks=8000, enable_pbar=False)
    assert outs[0] is not None and outs[1] is None            # level outside the data range -> item is None
    with pytest.raises(ValueError):
        ext.run(batch[1], mc_level=0.0, bounds=1.01, octree_resolution=60)
    half = torch.from_numpy(vol).to(dev).half()               # fp16 grids (reference GPU dtype) are accepted
    v16, f16 = ext.run(half, mc_level=0.0, bounds=1.01, octree_resolution=60)
    assert f16.shape[0] > 0


@pytest.mark.parametrize("shape,parts", [((17, 9, 33), 2), ((24, 12, 40), 3), ((31, 17, 65), 8)])
def test_mc_slabs_concatenate_to_whole_mesh(dev, ctx, shape, parts):
    """Slab forms (hy3d_mc_count_slab / hy3d_mc_emit_slab, the multi-GPU partition of SURVEY §8e): the meshes of
    consecutive axis-0 slabs, each seeing a two-plane halo of the next one, concatenate bit-exactly into the mesh of
    the whole grid (vertex bits, face ids) — random field with NaNs, all ranks emulated on one device."""
    from hy3dgeo.parallel import MC_HALO, slab_planes
    g = torch.randn(shape, generator=torch.Generator().manual_seed(11))
    g[3, 2, 5] = float("nan")
    g = g.to(dev)
    ext = MCSurfaceExtractor()
    kw = dict(bounds=1.01, octree_resolution=shape[0] - 1)
    v_ref, f_ref = ext.run_device(g, mc_level=0.1, **kw)
    vs, fs, base = [], [], 0
    for r in range(parts):
        x0, x1 = slab_planes(shape[0], r, parts)
        slab = g[x0:min(x1 + MC_HALO, shape[0])].contiguous()
        nv, nf, _ = ext.count_slab(slab, x1 - x0, 0.1)
        v, f = ext.emit_slab(nv, nf, x0, base, **kw)
        vs.append(v); fs.append(f); base += nv
    v, f = torch.cat(vs), torch.cat(fs)
    assert v.shape == v_ref.shape and f.shape == f_ref.shape
    assert torch.equal(v.view(torch.int32), v_ref.view(torch.int32)) and torch.equal(f, f_ref)


@pytest.mark.parametrize("n", [257, 385])
def test_mc_full_size_properties(ctx, n):
    """BASELINE grid sizes: V == number of sign-change grid edges, closed genus-0 surface F == 2V-4,
    every face index valid, vertices on the analytic sphere."""
    x = torch.linspace(-1.01, 1.01, n, device="cuda")
    r = torch.sqrt(x[:, None, None] ** 2 + x[None, :, None] ** 2 + x[None, None, :] ** 2)
    g = torch.tanh(20 * (0.6 - r)).contiguous()
    ins = g > 0
    edges = int((ins[1:] != ins[:-1]).sum() + (ins[:, 1:] != ins[:, :-1]).sum() + (ins[:, :, 1:] != ins[:, :, :-1]).sum())
    nv, nf, mm = ctx.mc_count(g, 0.0)
    assert nv == edges and nf == 2 * nv - 4
    v = torch.empty((nv, 3), dtype=torch.float32, device="cuda")
    f = torch.empty((nf, 3), dtype=torch.int32, device="cuda")
    ctx.mc_emit([n - 1] * 3, [2.02] * 3, [-1.01] * 3, v, f)
    assert int(f.min()) == 0 and int(f.max()) == nv - 1
    assert float((v.norm(dim=1) - 0.6).abs().max()) < 2.02 / (n - 1) * 0.05
    e = torch.cat([f[:, [0, 1]], f[:, [1, 2]], f[:, [2, 0]]]).long()
    key = torch.minimum(e[:, 0], e[:, 1]) * nv + torch.maximum(e[:, 0], e[:, 1])
    _, cnt = torch.unique(key, return_counts=True)
    assert bool((cnt == 2).all())                                # watertight


# ------------------------------------------------------------------------------------- octree
def test_refine_matches_oracle(ctx):
    rng = np.random.default_rng(3)
    base = sphere(33)
    holes = base.copy(); holes[rng.random(base.shape) < 0.3] = -10000.0
    noise = (rng.standard_normal((17, 17, 17)) * 2).astype(np.float32)
    zeros = base.copy(); zeros[rng.random(base.shape) < 0.05] = 0.0
    for grid in (base, holes, noise, zeros):
        for level in (0.0, 0.25):
            for last in (False, True):
                want = np.flatnonzero(OV.refine_active_set(grid, level, last).reshape(-1))
                idx = torch.empty(max(2 * want.size, 8), dtype=torch.int32, device="cuda")
                cnt = ctx.refine_level(torch.from_numpy(grid).cuda(), level, last, idx)
                assert cnt == want.size and np.array_equal(idx[:cnt].cpu().numpy(), want)
                assert ctx.refine_level(torch.from_numpy(grid).cuda(), level, last, None) == want.size     # count-only call


def test_refine_counts_match_reference_goldens(ctx, gold):
    """Visited-set sizes produced by the reference itself at octree 128 (SURVEY §8c):
    Hierarchical 65^3 -> 129^3: 294 426;  FlashVDM 64^3 -> 127^3: 286 014."""
    g = gold("volume_analytic.npz")
    for n, key in [(65, "hier128_visited"), (64, "flash128_visited")]:
        coarse = torch.from_numpy(OV.vanilla_decode(lambda p: torch.tanh(20 * (0.6 - p.norm(dim=-1))), 1.01, 10 ** 7, n - 1)).cuda()
        assert ctx.refine_level(coarse, 0.0, True, None) == int(g[key])


def test_fill_scatter_nan(ctx):
    g = torch.empty(1000, device="cuda")
    ctx.fill(g, -10000.0)
    idx = torch.tensor([5, -1, 999, 17], dtype=torch.int32, device="cuda")
    ctx.scatter(idx, torch.tensor([1.0, 2.0, 3.0, 4.0], device="cuda"), g)
    ctx.sentinel_to_nan(g)
    out = g.cpu().numpy()
    assert out[5] == 1 and out[999] == 3 and out[17] == 4 and np.isnan(out).sum() == 997


# ------------------------------------------------------------------------------------ decoder
@pytest.mark.parametrize("tag", ["mini", "turbo", "full"])
def test_decoder_matches_reference_golden(tag, gold, dev, ctx):
    cfg = CFG[tag]
    g = gold(f"decoder_{tag}.npz")
    sd = W.synthetic_state_dict(cfg, seed=0)
    vae = hy3dgeo.B200ShapeVAE(cfg, sd, device=dev)
    lat = vae(W.synthetic_latents(cfg, 1, 1234).to(dev))
    step = lat.shape[1] // g["latents_out_rows"].shape[0]                                  # token rows stored every `step`
    assert np.abs(lat[0, ::step].cpu().numpy() - g["latents_out_rows"]).max() < 1e-3        # ShapeVAE.forward
    c = bind(lat, vae.geo_decoder)
    c.prepare_kv(lat[0])
    q = torch.from_numpy(g["queries"][0]).to(dev)
    for prec, tol in [(_lib.PRECISION_FP32_SIMT, 3e-5), (_lib.PRECISION_FP16_TC, LOGIT_TOL)]:
        c.set_precision(prec)
        out = c.decode_points(q).cpu().numpy()
        c.check_watchdog()
        assert np.abs(out - g["logits"]).max() < tol, (tag, prec, np.abs(out - g["logits"]).max())
    c.set_precision(_lib.PRECISION_FP16_TC)


def test_decoder_ragged_sizes_and_chunks(dev, ctx):
    """Empty, 1, non-multiples of the 128-row tile (odd tile counts leave one CTA of a pair idle), and more than one
    262144-point chunk."""
    CH = 262144
    cfg = W.MINI
    sd = W.synthetic_state_dict(cfg, seed=0, with_transformer=False)
    gd = hy3dgeo.GeoDecoder(W.geo_decoder_state(sd), cfg)
    lat = torch.randn(1, 512, 1024, generator=torch.Generator().manual_seed(3)).to(dev)
    c = bind(lat, gd)
    c.prepare_kv(lat[0])
    gsd, fr = W.geo_decoder_state(sd), W.fourier_frequencies(cfg)
    assert c.decode_points(torch.empty(0, 3, device=dev)).numel() == 0
    pts = (torch.rand(CH + 129, 3, generator=torch.Generator().manual_seed(4)) * 2 - 1) * 1.01
    out = c.decode_points(pts.to(dev)).cpu()
    c.check_watchdog()
    for sl in (slice(0, 1), slice(127, 130), slice(CH - 1, CH + 129)):
        ref = OD.geo_decoder_forward(gsd, pts[None, sl], lat.cpu(), fr, cfg.dec_heads)[0, :, 0]
        assert float((out[sl] - ref).abs().max()) < LOGIT_TOL
    one = c.decode_points(pts[:1].to(dev)).cpu()
    assert float((one - out[:1]).abs().max()) < 1e-6               # result independent of batch composition
    pad = torch.randn(1, 300, 1024, generator=torch.Generator().manual_seed(5)).to(dev)   # token count not a multiple of 128
    c.prepare_kv(pad[0])
    o2 = c.decode_points(pts[:200].to(dev)).cpu()
    ref = OD.geo_decoder_forward(gsd, pts[None, :200], pad.cpu(), fr, cfg.dec_heads)[0, :, 0]
    assert float((o2 - ref).abs().max()) < LOGIT_TOL


# ---------------------------------------------------------------------------- volume decoders
def test_vanilla_grid_layout_and_values(dev):
    cfg = W.MINI
    sd = W.synthetic_state_dict(cfg, seed=0)
    vae = hy3dgeo.B200ShapeVAE(cfg, sd, device=dev)
    z = W.synthetic_latents(cfg, 2, 1234)
    lat_o = OD.shapevae_forward(sd, z, cfg.heads)
    bounds = [-1.0, -0.8, -0.6, 0.9, 1.0, 1.01]
    grid = VanillaVolumeDecoder()(lat_o.to(dev), vae.geo_decoder, bounds=bounds, num_chunks=777, octree_resolution=12,
                                  enable_pbar=False, some_unknown_kwarg=1)
    assert grid.shape == (2, 13, 13, 13) and grid.dtype == torch.float32
    gsd, fr = W.geo_decoder_state(sd), W.fourier_frequencies(cfg)
    for b in range(2):
        ref = OV.vanilla_decode(lambda p: OD.geo_decoder_forward(gsd, p[None], lat_o[b:b + 1], fr, cfg.dec_heads)[0, :, 0],
                                bounds, 5000, 12)
        assert np.abs(grid[b].cpu().numpy() - ref).max() < LOGIT_TOL


def test_hierarchical_matches_patched_reference(gold, dev, ctx, checksum):
    cfg = W.MINI
    g = gold("volume_decoder_mini.npz")
    gain = float(g["gain"])
    sd = W.sparsify_field(W.synthetic_state_dict(cfg, seed=0), cfg, int(g["keep_freqs"]), gain, float(g["bias"]))
    assert checksum(sd) == pytest.approx(float(g["weight_checksum"]), rel=1e-9)
    vae = hy3dgeo.B200ShapeVAE(cfg, sd, device=dev)
    z = W.synthetic_latents(cfg, 1, 1234).to(dev)
    ref = g["hier32"]
    for prec, tol in [(_lib.PRECISION_FP32_SIMT, 1e-4), (_lib.PRECISION_FP16_TC, LOGIT_TOL * gain)]:   # error scales with the head gain
        ctx.set_precision(prec)
        # fp32 leg: fp32 end to end (library fp32 transformer + CUDA-core decoder); tensor leg: tcgen05 transformer + decoder
        lat = vae(z, impl="torch") if prec == _lib.PRECISION_FP32_SIMT else vae(z)
        dec = HierarchicalVolumeDecoding()
        out = dec(lat, vae.geo_decoder, bounds=1.01, num_chunks=3000, mc_level=0.0, octree_resolution=32, min_resolution=15,
                  enable_pbar=False)[0].cpu().numpy()
        assert np.array_equal(np.isnan(out), np.isnan(ref)), "visited set differs from the reference"
        assert np.abs(np.nan_to_num(out) - np.nan_to_num(ref)).max() < tol
        assert dec.last_stats[0]["queries"] == [17 ** 3, int((~np.isnan(ref)).sum())]
    ctx.set_precision(_lib.PRECISION_FP16_TC)


def chamfer(a, b):
    a, b = torch.from_numpy(a).cuda(), torch.from_numpy(b).cuda()
    d = torch.cdist(a, b)
    return float(d.min(1).values.mean() + d.min(0).values.mean()) / 2


def test_latents2mesh_end_to_end(dev, ctx):
    """ShapeVAE.latents2mesh (reference model.py:105-110) through B200ShapeVAE vs the oracle pipeline
    on identical weights/latents: Chamfer < 1e-4 * bbox diagonal; fp32 mode gives the identical mesh."""
    cfg = W.MINI
    sd = W.sparsify_field(W.synthetic_state_dict(cfg, seed=0), cfg, 2, 1.0, 0.0)
    vae = hy3dgeo.B200ShapeVAE(cfg, sd, device=dev)
    z = W.synthetic_latents(cfg, 1, 1234)
    lat_o = OD.shapevae_forward(sd, z, cfg.heads)
    gsd, fr = W.geo_decoder_state(sd), W.fourier_frequencies(cfg)
    res = 40
    grid_o = OV.vanilla_decode(lambda p: OD.geo_decoder_forward(gsd, p[None], lat_o, fr, cfg.dec_heads)[0, :, 0], 1.01, 8000, res)
    vo, fo = OM.mc_surface_extract(grid_o, mc_level=0.0, bounds=1.01, octree_resolution=res)
    kw = dict(bounds=1.01, mc_level=0.0, num_chunks=8000, octree_resolution=res, mc_algo="mc", enable_pbar=False)
    diag = 2.02 * np.sqrt(3)
    for prec in (_lib.PRECISION_FP32_SIMT, _lib.PRECISION_FP16_TC):
        ctx.set_precision(prec)
        # the fp32 leg is fp32 end to end (library fp32 latent transformer + CUDA-core decoder): only then is the
        # mesh expected to be identical; the tensor leg uses the tcgen05 transformer and decoder (Chamfer bound)
        lat = vae(z.to(dev), impl="torch") if prec == _lib.PRECISION_FP32_SIMT else vae(z.to(dev))
        out = vae.latents2mesh(lat, **kw)[0]
        assert out is not None and out.mesh_v.dtype == np.float32 and out.mesh_f.dtype == np.int32
        assert chamfer(out.mesh_v, vo) < 1e-4 * diag
        if prec == _lib.PRECISION_FP32_SIMT and out.mesh_f.shape == fo.shape:
            assert np.array_equal(out.mesh_f, fo)
    ctx.set_precision(_lib.PRECISION_FP16_TC)
    vae.enable_flashvdm_decoder(enabled=False)
    assert type(vae.volume_decoder).__name__ == "VanillaVolumeDecoder"
    with pytest.raises(ValueError):
        vae.enable_flashvdm_decoder(mc_algo="nope")


def test_smoke_entry():
    import __graft_entry__ as g
    g.smoke()


# ---------------------------------------------------------------------------------- latent transformer
@pytest.mark.parametrize("tag", ["mini", "full"])
def test_latent_transformer_matches_oracle_on_both_attention_kernels(tag, dev, ctx):
    """ShapeVAE.forward (reference model.py:186-189; post_kl + 16 pre-LN blocks) on the tcgen05 kernels
    (3-term split GEMMs, folded LayerNorms, fp16 self-attention) vs the fp32 CPU oracle: |latent| <= 6,
    max error < 1e-3 (measured 3.4e-4), rms < 2e-4 (measured 7e-5); both attention kernels."""
    cfg = W.MINI if tag == "mini" else W.FULL
    sd = W.synthetic_state_dict(cfg, seed=0)
    z = W.synthetic_latents(cfg, 1, 1234)
    torch.set_num_threads(os.cpu_count())
    ref = OD.shapevae_forward(sd, z, cfg.heads)
    vae = hy3dgeo.B200ShapeVAE(cfg, sd, device=dev)
    try:
        for online in (False, True):                 # bounded-score kernel (default for these norms), online-softmax kernel
            ctx.debug_force_online_softmax(online)
            lat = vae(z.to(dev)).cpu()
            ctx.check_watchdog()
            d = (lat - ref).abs()
            assert lat.shape == ref.shape and float(d.max()) < 1e-3 and float(d.pow(2).mean().sqrt()) < 2e-4
    finally:
        ctx.debug_force_online_softmax(False)


# ---------------------------------------------------------------------------------- FlashVDM
@pytest.mark.parametrize("mode", ["mean", "merge"])
def test_flashvdm_matches_reference_golden(mode, gold, dev, ctx, checksum):
    """FlashVDMVolumeDecoding(topk_mode) vs the REAL reference (stable bin order) at octree 32:
    identical visited set, logits within tolerance x head gain; snapped grid size 31^3."""
    from hy3dgeo.volume_decoders import FlashVDMVolumeDecoding
    cfg = W.MINI
    g = gold("volume_decoder_mini.npz")
    gain = float(g["gain"])
    sd = W.sparsify_field(W.synthetic_state_dict(cfg, seed=0), cfg, int(g["keep_freqs"]), gain, float(g["bias"]))
    vae = hy3dgeo.B200ShapeVAE(cfg, sd, device=dev)
    z = W.synthetic_latents(cfg, 1, 1234).to(dev)
    ref = g[f"flash32_{mode}"]
    dec = FlashVDMVolumeDecoding(mode)
    kw = dict(bounds=1.01, num_chunks=3000, mc_level=0.0, octree_resolution=32, min_resolution=15, enable_pbar=False)
    # (1) the decoder on the latents the golden was made from (fp32 library transformer, within 1e-5 of the oracle's):
    #     every logit within tolerance
    out = dec(vae(z, impl="torch"), vae.geo_decoder, **kw)[0].cpu().numpy()
    ctx.check_watchdog()
    assert out.shape == ref.shape == (31, 31, 31)
    assert np.array_equal(np.isnan(out), np.isnan(ref))
    assert np.abs(np.nan_to_num(out) - np.nan_to_num(ref)).max() < LOGIT_TOL * gain
    assert dec.last_stats[0]["levels"] == [15, 30]
    # (2) the product path (tcgen05 transformer, latents within 4e-4 of the oracle's): same visited set; the token
    #     selection thresholds (top-k rank / p > 1e-6) may flip a near-tie, which moves a handful of logits of one bin
    out = dec(vae(z), vae.geo_decoder, **kw)[0].cpu().numpy()
    ctx.check_watchdog()
    assert np.array_equal(np.isnan(out), np.isnan(ref))
    err = np.abs(np.nan_to_num(out) - np.nan_to_num(ref))
    assert err.mean() < 1e-4 and err.max() < 5 * LOGIT_TOL * gain
    assert (err > LOGIT_TOL * gain).mean() < 1e-3


def test_flashvdm_level0_selection_and_logits(dev, ctx):
    """Level 0 (64 mini-grids, top-256 of 512 tokens per (mini-grid, head)): the selected token SETS
    equal the oracle processor's except at genuine near-ties; logits within 1e-3 wherever the sets agree."""
    from hy3dgeo.volume_decoders import FlashVDMVolumeDecoding
    cfg = W.MINI
    sd = W.synthetic_state_dict(cfg, seed=0)
    vae = hy3dgeo.B200ShapeVAE(cfg, sd, device=dev)
    z = W.synthetic_latents(cfg, 1, 1234)
    lat_o = OD.shapevae_forward(sd, z, cfg.heads)
    out = FlashVDMVolumeDecoding("mean")(lat_o.to(dev), vae.geo_decoder, bounds=1.01, octree_resolution=32, min_resolution=31,
                                         enable_pbar=False)[0].cpu().numpy()
    assert out.shape == (32, 32, 32) and not np.isnan(out).any()
    gsd, fr = W.geo_decoder_state(sd), W.fourier_frequencies(cfg)
    proc = OD.FlashProcessorOracle("mean")
    sels = []

    def dec_group(p, topk):
        proc.topk = topk
        o = OD.geo_decoder_forward(gsd, p, lat_o.expand(p.shape[0], -1, -1), fr, cfg.dec_heads, kv_select=proc)[..., 0]
        sels.append(proc.last_selection[0])
        return o
    ref = OV.flashvdm_decode(dec_group, 1.01, 200000, 0.0, 32, 31)
    sel_ref = torch.cat(sels, 0).numpy()
    G, H, T = sel_ref.shape
    assert (G, H, T) == (64, 16, 256)
    sel = ctx.flash_selection(G * H * T).cpu().numpy().reshape(G, H, T)
    assert bool((ctx.flash_group_tokens(G).cpu().numpy() == T).all())
    bad_groups = {g for g in range(G) for h in range(H) if set(sel[g, h]) != set(sel_ref[g, h])}
    ndiff = sum(len(set(sel[g, h]) ^ set(sel_ref[g, h])) // 2 for g in range(G) for h in range(H))
    assert ndiff <= 8, f"{ndiff} selected tokens differ from the fp32 reference selection"
    order = OV.flash_minigrid_order(32, 4)
    for g in range(G):
        d = np.abs(out.reshape(-1)[order[g]] - ref.reshape(-1)[order[g]]).max()
        assert d < (LOGIT_TOL if g not in bad_groups else 2e-2), (g, d)


@pytest.mark.parametrize("case", ["shell", "random", "flat_axis", "tiny", "empty"])
def test_flash_layout_bins_matches_reference_restatement(case, dev, ctx):
    """hy3d_flash_layout_bins: bin ids, stable order, padding, per-tile group and stride samples, bit for bit."""
    rng = np.random.default_rng(11)
    n = 97
    if case == "shell":
        g = np.linalg.norm(np.stack(np.meshgrid(*[np.arange(n)] * 3, indexing="ij"), -1) - 48.0, axis=-1)
        index = np.nonzero((np.abs(g - 30.0) < 2.0).reshape(-1))[0]
    elif case == "random":
        index = np.sort(rng.choice(n ** 3, 70001, replace=False))
    elif case == "flat_axis":                                    # max == min on axis 0: NaN bin component -> clamped ids
        index = np.sort(rng.choice(n * n, 5000, replace=False)) + 40 * n * n
    elif case == "tiny":
        index = np.array([5, 77, 4000, 900000], np.int64)
    else:
        index = np.zeros(0, np.int64)
    index = index.astype(np.int32)
    cell = (np.full(3, 2.02) / (n - 1)).astype(np.float32)
    bmin = np.full(3, -1.01, np.float32)
    for stride in (50, 30):
        pidx, tg, sidx, soff, counts = ctx.flash_layout_bins(torch.from_numpy(index).to(dev), (n, n, n), cell, bmin, stride, with_counts=True)
        if len(index):
            rp, rt, rs, ro, rc = OV.flash_layout_reference(index, n, cell, bmin, stride)
        else:
            rp, rt = np.full(pidx.numel(), -1, np.int32), np.full(tg.numel(), 215, np.int32)
            rs, ro, rc = np.zeros(0, np.int32), np.zeros(217, np.int32), np.zeros(216, np.int32)
        assert np.array_equal(counts.cpu().numpy(), rc)
        assert np.array_equal(soff.cpu().numpy(), ro)
        assert np.array_equal(pidx.cpu().numpy(), rp)
        s = sidx.cpu().numpy()
        assert np.array_equal(s[:len(rs)], rs) and bool((s[len(rs):] == -1).all())
        # tiles past the last bin hold only padding; the reference restatement leaves them at G-1 too
        assert np.array_equal(tg.cpu().numpy(), rt)


def test_flash_layout_minigrids_matches_oracle_order(dev, ctx):
    N, m, stride = 32, 4, 100
    pidx, tg, sidx, soff = ctx.flash_layout_minigrids(N, m, stride)
    order = OV.flash_minigrid_order(N, m)                         # [64, 512]
    G, s3 = order.shape
    padc = (s3 + 127) // 128 * 128
    p = pidx.cpu().numpy().reshape(G, padc)
    assert np.array_equal(p[:, :s3], order.astype(np.int32)) and bool((p[:, s3:] == -1).all())
    assert np.array_equal(tg.cpu().numpy(), np.repeat(np.arange(G, dtype=np.int32), padc // 128))
    ns = (s3 + stride - 1) // stride
    assert np.array_equal(soff.cpu().numpy(), np.arange(G + 1, dtype=np.int32) * ns)
    sv = sidx.cpu().numpy()
    assert np.array_equal(sv[:G * ns].reshape(G, ns), order[:, ::stride].astype(np.int32)) and bool((sv[G * ns:] == -1).all())


def test_flash_topk_ties_go_to_the_lower_token(dev, ctx):
    """Radix-select top-k (k_sim_topk): latent tokens 256..511 are exact copies of tokens 0..255, so every similarity is
    tied pairwise.  The selection must hold T distinct tokens per (mini-grid, head), and whenever the copy i + 256 is taken
    its original i (equal key, lower index) is taken too — the count of threshold ties is exact."""
    cfg = W.MINI
    sd = W.synthetic_state_dict(cfg, seed=0, with_transformer=False)
    gd = hy3dgeo.GeoDecoder(W.geo_decoder_state(sd), cfg)
    half = torch.randn(1, 256, 1024, generator=torch.Generator().manual_seed(21))
    lat = torch.cat([half, half], 1).to(dev)
    c = bind(lat, gd)
    c.prepare_kv(lat[0])
    N0, m, T = 32, 4, 200                                   # T not a multiple of anything convenient
    pidx, tg, sidx, soff = c.flash_layout_minigrids(N0, m, 100)
    axes = OV.axis_tables(1.01, N0 - 1)
    c.flash_select(sidx, (N0, N0, N0), soff, m ** 3, T, False, axes=axes)
    G, H = m ** 3, cfg.dec_heads
    sel = c.flash_selection(G * H * T).cpu().numpy().reshape(G, H, T)
    c.check_watchdog()
    assert sel.min() >= 0 and sel.max() < 512
    for g in range(G):
        for h in range(H):
            row = sel[g, h]
            chosen = set(row.tolist())
            assert len(chosen) == T
            assert bool((np.diff(row) > 0).all())            # emitted in ascending token order
            assert all((t - 256) in chosen for t in chosen if t >= 256), (g, h)


# ------------------------------------------------------------------ round 2: BASELINE configurations (goldens *_r2)
def test_refine_odd_levels_matches_oracle(ctx):
    """Fine grids of 2n voxels per axis (the coarse level is an odd r // 2, reference vd:202-208): indices are laid out on the
    (r+1)^3 grid, the up-sampled voxels sit at 2c, dilations are clipped at the fine grid's faces."""
    rng = np.random.default_rng(5)
    base = sphere(18)
    noise = (rng.standard_normal((9, 9, 9)) * 2).astype(np.float32)
    for grid in (base, noise):
        n = grid.shape[0]
        for nf in (2 * n - 1, 2 * n):
            for last in (False, True):
                want = np.flatnonzero(OV.refine_active_set(grid, 0.0, last, nf=nf).reshape(-1))
                idx = torch.empty(max(2 * want.size, 8), dtype=torch.int32, device="cuda")
                cnt = ctx.refine_level(torch.from_numpy(grid).cuda(), 0.0, last, idx, nf)
                assert cnt == want.size and np.array_equal(idx[:cnt].cpu().numpy(), want)
    with pytest.raises(_lib.Hy3dError):
        ctx.refine_level(torch.from_numpy(base).cuda(), 0.0, True, None, 2 * 18 + 1)


def _sparse_vae(tag, g, dev):
    cfg = CFG[tag]
    sd = W.sparsify_field(W.synthetic_state_dict(cfg, seed=0), cfg, int(g["keep_freqs"]), float(g["gain"]), float(g["bias"]))
    return cfg, sd, hy3dgeo.B200ShapeVAE(cfg, sd, device=dev)


@pytest.mark.parametrize("res,minres", [(64, 15), (35, 8)])
def test_hierarchical_three_levels_matches_patched_reference(res, minres, gold, dev, ctx, checksum):
    """BASELINE config 3's structure — 3 levels, expand_num = 1 on the middle one (reference vd:250-259) — and the odd-level
    list [8, 17, 35] on the real mini decoder against the patched reference: identical visited set, logits within
    tolerance x head gain, per-level query counts."""
    g = gold("volume_decoder_mini_r2.npz")
    gain = float(g["gain"])
    cfg, sd, vae = _sparse_vae("mini", g, dev)
    assert checksum(sd) == pytest.approx(float(g["weight_checksum"]), rel=1e-9)
    z = W.synthetic_latents(cfg, 1, 1234).to(dev)
    ref = g[f"hier{res}"]
    for prec, tol in [(_lib.PRECISION_FP32_SIMT, 1e-4), (_lib.PRECISION_FP16_TC, LOGIT_TOL * gain)]:
        ctx.set_precision(prec)
        exact = prec == _lib.PRECISION_FP32_SIMT
        lat = vae(z, impl="torch") if exact else vae(z)
        dec = HierarchicalVolumeDecoding(keep_levels=True)
        out = dec(lat, vae.geo_decoder, bounds=1.01, num_chunks=8000, mc_level=0.0, octree_resolution=res, min_resolution=minres,
                  enable_pbar=False)[0].cpu().numpy()
        ctx.check_watchdog()
        assert out.shape == ref.shape and len(dec.last_stats[0]["levels"]) == 3
        OV.check_sparse_levels(dec, out, ref, tol, exact=exact)
        if exact:
            assert dec.last_stats[0]["queries"] == list(g[f"hier{res}_queries"])
    ctx.set_precision(_lib.PRECISION_FP16_TC)


@pytest.mark.parametrize("tag,res", [("turbo", 32), ("turbo", 64), ("full", 32)])
@pytest.mark.parametrize("mode", ["mean", "merge"])
def test_flashvdm_turbo_and_full_match_reference_golden(tag, res, mode, gold, dev, ctx, checksum):
    """FlashVDMVolumeDecoding on BASELINE config 4's decoder (mini-turbo: latents_proj, no q/k norm -> online-softmax
    attention kernel, expand ratio 1, top-256) and on the full decoder (3072 tokens, top-1024), both selection modes,
    2 and 3 levels, against the REAL reference (stable bin order)."""
    from hy3dgeo.volume_decoders import FlashVDMVolumeDecoding
    g = gold(f"flash_{tag}.npz")
    gain = float(g["gain"])
    cfg, sd, vae = _sparse_vae(tag, g, dev)
    assert checksum(sd) == pytest.approx(float(g["weight_checksum"]), rel=1e-9)
    z = W.synthetic_latents(cfg, 1, 1234).to(dev)
    ref = g[f"flash{res}_{mode}"]
    dec = FlashVDMVolumeDecoding(mode, keep_levels=True)
    kw = dict(bounds=1.01, num_chunks=600, mc_level=0.0, octree_resolution=res, min_resolution=15, enable_pbar=False)
    gsd, fr = W.geo_decoder_state(sd), W.fourier_frequencies(cfg)
    torch.set_num_threads(os.cpu_count())

    def oracle_steps(lat, lv):
        """the reference algorithm (oracle, pinned to the reference by tests/test_oracle_golden.py) on the SAME latents,
        level by level on the DEVICE's own previous level.  The active set, the 6^3 binning and the every-50th / 30th
        sampling are discontinuous in the coarse logits: a sub-tolerance difference that flips one voxel at a threshold
        shifts the sampling phase of its bin, hence the selected tokens and every logit of that bin (measured: bins
        whose selection then differs by up to 15 tokens per head, tools/gpu_flash_bins_debug.py) — the reference is just
        as sensitive to its own rounding.  Given the same field nothing of that is left: what remains between the two is
        the decoder arithmetic and genuine near-ties of the selection at the precision of the sampled q (~1e-6)."""
        lat_c = lat.cpu()
        proc = OD.FlashProcessorOracle(mode)

        def dec_group(p, topk):
            proc.topk = topk
            return OD.geo_decoder_forward(gsd, p, lat_c.expand(p.shape[0], -1, -1), fr, cfg.dec_heads, kv_select=proc)[..., 0]
        levels = dec.last_stats[0]["levels"]
        want = [OV.flashvdm_decode(dec_group, 1.01, 600, 0.0, levels[0], 10 ** 9)]      # level 0 alone: the 64 mini-grids
        for k, r in enumerate(levels[1:]):
            want.append(OV.flashvdm_level(dec_group, lv[k], 1.01, r, r == levels[-1], 600, 0.0)[0])
        return want

    for leg, lat in [("fp32 library transformer", vae(z, impl="torch")), ("tcgen05 transformer (product path)", vae(z))]:
        out = dec(lat, vae.geo_decoder, **kw)[0].cpu().numpy()
        ctx.check_watchdog()
        levels = dec.last_stats[0]["levels"]
        assert out.shape == ref.shape and levels == [15, 30, 60][: len(levels)]
        lv = [g_.cpu().numpy() for g_ in dec.last_levels]
        assert np.array_equal(~np.isnan(out), lv[-1] != OV.SENTINEL)
        for k, want in enumerate(oracle_steps(lat, lv)):
            vis = lv[k] != OV.SENTINEL
            assert np.array_equal(vis, want != OV.SENTINEL), f"{leg}: level {k} active set is not the reference logic's for the same field"
            err = np.abs(lv[k][vis] - want[vis])
            # at most 0.1 % of a level's voxels in bins with a genuine near-tie (never beyond 5 x tolerance)
            assert err.max() < 5 * LOGIT_TOL * gain and (err > LOGIT_TOL * gain).mean() <= 1e-3, (leg, k, err.max(), (err > LOGIT_TOL * gain).mean())
        # against the reference's own output (golden; latents differ by 1e-5 / 4e-4, logits by fp16-operand rounding):
        # the visited sets agree up to threshold flips (< 1 %), the error on the common voxels is small on average
        vis, rvis = ~np.isnan(out), ~np.isnan(ref)
        assert (vis ^ rvis).sum() < 0.01 * rvis.sum(), leg
        both = vis & rvis
        assert np.abs(out[both] - ref[both]).mean() < 5e-4 * gain, (leg, np.abs(out[both] - ref[both]).mean())


def test_decoder_include_pi_matches_reference_golden(gold, dev, ctx):
    """FourierEmbedder(include_pi=True) (attention_blocks.py:93-94): frequencies pi * 2^k, arguments up to +-407 rad."""
    import dataclasses
    cfg = dataclasses.replace(W.MINI, include_pi=True)
    g = gold("decoder_pi.npz")
    sd = W.synthetic_state_dict(cfg, seed=0)
    vae = hy3dgeo.B200ShapeVAE(cfg, sd, device=dev)
    lat = vae(W.synthetic_latents(cfg, 1, 1234).to(dev))
    c = bind(lat, vae.geo_decoder)
    c.prepare_kv(lat[0])
    q = torch.from_numpy(g["queries"][0]).to(dev)
    for prec, tol in [(_lib.PRECISION_FP32_SIMT, 3e-5), (_lib.PRECISION_FP16_TC, LOGIT_TOL)]:
        c.set_precision(prec)
        out = c.decode_points(q).cpu().numpy()
        c.check_watchdog()
        assert np.abs(out - g["logits"]).max() < tol, (prec, np.abs(out - g["logits"]).max())
    c.set_precision(_lib.PRECISION_FP16_TC)


def test_latents2mesh_end_to_end_golden_13k_vertices(gold, dev, ctx, checksum):
    """ShapeVAE.latents2mesh at octree 64 against the mesh the REFERENCE's latents2mesh produced (13 552 vertices; its
    marching cubes is the oracle's — skimage is absent, parity unpinned there): fp32 chain = identical faces and
    vertices within 1e-4; tensor chain within the Chamfer bound with a vertex count within 1 %."""
    m = gold("latents2mesh_mini64.npz")
    cfg, sd, vae = _sparse_vae("mini", m, dev)
    assert checksum(sd) == pytest.approx(float(m["weight_checksum"]), rel=1e-9)
    z = W.synthetic_latents(cfg, 1, 1234).to(dev)
    kw = dict(bounds=1.01, mc_level=0.0, num_chunks=8000, octree_resolution=64, mc_algo="mc", enable_pbar=False)
    diag = 2.02 * np.sqrt(3)
    sub = np.random.default_rng(0).choice(m["mesh_v"].shape[0], 6000, replace=False)
    for prec in (_lib.PRECISION_FP32_SIMT, _lib.PRECISION_FP16_TC):
        ctx.set_precision(prec)
        lat = vae(z, impl="torch") if prec == _lib.PRECISION_FP32_SIMT else vae(z)
        out = vae.latents2mesh(lat, **kw)[0]
        ctx.check_watchdog()
        assert out is not None and out.mesh_v.dtype == np.float32 and out.mesh_f.dtype == np.int32
        if prec == _lib.PRECISION_FP32_SIMT:
            assert np.array_equal(out.mesh_f, m["mesh_f"])
            assert np.abs(out.mesh_v - m["mesh_v"]).max() < 1e-4
        else:
            assert abs(out.mesh_v.shape[0] - m["mesh_v"].shape[0]) < 0.01 * m["mesh_v"].shape[0]
            a, b = torch.from_numpy(m["mesh_v"][sub]).cuda(), torch.from_numpy(out.mesh_v).cuda()
            assert float(torch.cdist(a, b).min(1).values.mean()) < 1e-4 * diag
            a, b = torch.from_numpy(out.mesh_v[::3]).cuda(), torch.from_numpy(m["mesh_v"]).cuda()
            assert float(torch.cdist(a, b).min(1).values.mean()) < 1e-4 * diag
    ctx.set_precision(_lib.PRECISION_FP16_TC)


# ---------------------------------------------------------------- mesh clean-up (the step right after the path, §8f rank 3)
def test_mesh_clean_matches_export_to_trimesh_restatement(dev, ctx):
    """hy3d_mesh_clean / MCSurfaceExtractor(cull_nonfinite) / hy3dgeo.export_to_trimesh vs the numpy restatement of
    export_to_trimesh's arithmetic (pipelines.py:95-110: winding flip, then trimesh dropping non-finite vertices, their faces
    and unreferenced vertices): bit-identical arrays, on a sparse-decoder-like grid (NaN outside a band) and on edge cases."""
    from oracle import mesh as OMESH
    vol = sphere(49)
    vol[np.abs(vol) > 0.9995] = np.nan                       # unvisited voxels of the sparse decoders -> NaN vertices at the rim
    vol[10:14, 20:30, 20:30] = np.nan                        # a hole in the band
    ext = MCSurfaceExtractor()
    g = torch.from_numpy(vol).to(dev)
    v, f = ext.run_device(g, mc_level=0.0, bounds=1.01, octree_resolution=48)
    vn, fn = v.cpu().numpy(), f.cpu().numpy()
    assert np.isnan(vn).any()
    for flip in (False, True):
        vo, fo = ctx.mesh_clean(v, f, flip_winding=flip)
        wv, wf = OMESH.export_clean(vn, fn, flip_winding=flip)
        assert bits_equal(vo.cpu().numpy(), wv) and np.array_equal(fo.cpu().numpy(), wf)
        assert np.isfinite(vo.cpu().numpy()).all() and int(fo.max()) == vo.shape[0] - 1
    v2, f2 = MCSurfaceExtractor(cull_nonfinite=True).run(g, mc_level=0.0, bounds=1.01, octree_resolution=48)
    wv, wf = OMESH.export_clean(vn, fn, flip_winding=False)
    assert bits_equal(v2, wv) and np.array_equal(f2, wf)
    out = hy3dgeo.export_to_trimesh([hy3dgeo.Latent2MeshOutput(mesh_v=vn, mesh_f=fn), None])
    assert out[1] is None
    wv, wf = OMESH.export_clean(vn, fn, flip_winding=True)
    ov, of = (np.asarray(out[0].vertices, np.float32), np.asarray(out[0].faces, np.int32)) if hasattr(out[0], "vertices") else (out[0].mesh_v, out[0].mesh_f)
    assert bits_equal(ov, wv) and np.array_equal(of, wf)
    # nothing to remove: the mesh comes back unchanged (winding aside); every face removed: empty mesh
    clean = sphere(33)
    v, f = ext.run_device(torch.from_numpy(clean).to(dev), mc_level=0.0, bounds=1.01, octree_resolution=32)
    vo, fo = ctx.mesh_clean(v, f, flip_winding=True)
    assert torch.equal(vo, v) and torch.equal(fo, f.flip(1))
    vo, fo = ctx.mesh_clean(torch.full_like(v, float("nan")), f, flip_winding=False)
    assert vo.shape[0] == 0 and fo.shape[0] == 0


# ------------------------------------------------- attention: measured score bounds, per-head shift, exact redo pass
def _scaled_norms(cfg, gain, seed=0):
    sd = W.synthetic_state_dict(cfg, seed=seed, with_transformer=False)
    c = "geo_decoder.cross_attn_decoder.attn.attention."
    for n in ("q_norm", "k_norm"):
        sd[c + n + ".weight"] = sd[c + n + ".weight"] * gain
    return sd


def test_attention_large_norm_gains_use_measured_bounds(dev, ctx):
    """A checkpoint whose q/k-norm gains put the weight-only score bound above 15.9 (here x1.4 each: ~30) still runs the
    bounded-score kernel: each head's scores are shifted by its MEASURED bound (max ||k|| of the latent set) minus 15.9, so
    exp2 cannot overflow fp16, and rows too far below the bound are recomputed exactly.  Logits vs the fp32 device path."""
    cfg = W.MINI
    sd = _scaled_norms(cfg, 1.4)
    gd = hy3dgeo.GeoDecoder(W.geo_decoder_state(sd), cfg)
    lat = torch.randn(1, 512, 1024, generator=torch.Generator().manual_seed(3)).to(dev)
    c = bind(lat, gd)
    c.prepare_kv(lat[0])
    wb, kern, mb = c.attention_info()
    assert 15.9 < wb < 40 and kern.startswith("bounded-score + per-head shift") and mb < wb
    pts = ((torch.rand(3000, 3, generator=torch.Generator().manual_seed(4)) * 2 - 1) * 1.01).to(dev)
    c.set_precision(_lib.PRECISION_FP32_SIMT)
    ref = c.decode_points(pts).cpu()
    c.set_precision(_lib.PRECISION_FP16_TC)
    out = c.decode_points(pts).cpu()
    c.check_watchdog()
    assert float((out - ref).abs().max()) < LOGIT_TOL
    assert c.debug_attn_redo() == 0                      # ordinary latents: nothing is far enough below the bound
    gsd, fr = W.geo_decoder_state(sd), W.fourier_frequencies(cfg)
    o = OD.geo_decoder_forward(gsd, pts[None, :256].cpu(), lat.cpu(), fr, cfg.dec_heads)[0, :, 0]
    assert float((out[:256] - o).abs().max()) < LOGIT_TOL
    # gains beyond the shift range (weight-only bound > 40): the online-softmax kernel, same answers
    sd2 = _scaled_norms(cfg, 2.0)
    gd2 = hy3dgeo.GeoDecoder(W.geo_decoder_state(sd2), cfg)
    c = bind(lat, gd2)
    c.prepare_kv(lat[0])
    assert c.attention_info()[1] == "online-softmax"
    c.set_precision(_lib.PRECISION_FP32_SIMT); ref = c.decode_points(pts[:512]).cpu()
    c.set_precision(_lib.PRECISION_FP16_TC); out = c.decode_points(pts[:512]).cpu()
    assert float((out - ref).abs().max()) < LOGIT_TOL


def test_attention_redo_pass_recomputes_rows_far_below_the_bound(dev, ctx):
    """Adversarial latents (all tokens nearly identical): every key of a head points the same way, so for half of the
    queries ALL scores sit far below the head's bound; after the shift their probabilities underflow fp16.  The kernel flags
    those (query tile, head pair) items on the device and the online-softmax kernel recomputes them: results stay exact."""
    cfg = W.MINI
    sd = _scaled_norms(cfg, 1.5)
    gd = hy3dgeo.GeoDecoder(W.geo_decoder_state(sd), cfg)
    g = torch.Generator().manual_seed(5)
    row = torch.randn(1, 1, 1024, generator=g)
    lat = (row + 1e-3 * torch.randn(1, 512, 1024, generator=g)).to(dev)
    c = bind(lat, gd)
    c.prepare_kv(lat[0])
    assert c.attention_info()[1].startswith("bounded-score + per-head shift")
    pts = ((torch.rand(1500, 3, generator=torch.Generator().manual_seed(6)) * 2 - 1) * 1.01).to(dev)
    c.set_precision(_lib.PRECISION_FP32_SIMT)
    ref = c.decode_points(pts).cpu()
    c.set_precision(_lib.PRECISION_FP16_TC)
    out = c.decode_points(pts).cpu()
    c.check_watchdog()
    assert c.debug_attn_redo() > 0, "the adversarial case was meant to exercise the redo pass"
    assert float((out - ref).abs().max()) < LOGIT_TOL
