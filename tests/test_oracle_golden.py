"""CPU: the oracle restatements against the golden vectors produced by the REAL reference
(oracle/make_golden.py, run where /root/reference exists).  This is what pins the oracle on
machines where the reference tree is absent."""
import numpy as np
import pytest
import torch

import hy3dgeo  # noqa: F401
from hy3dgeo import weights as W
from oracle import decoder as OD, volume as OV, mc as OM

CFG = {"mini": W.MINI, "full": W.FULL, "turbo": W.MINI_TURBO}


def analytic(p):
    return torch.tanh(20 * (0.6 - p.float().norm(dim=-1)))


@pytest.mark.parametrize("tag", ["mini", "turbo", "full"])
def test_decoder_and_transformer_match_reference(tag, gold, checksum):
    cfg = CFG[tag]
    g = gold(f"decoder_{tag}.npz")
    sd = W.synthetic_state_dict(cfg, seed=int(g["seed"]))
    assert checksum(sd) == pytest.approx(float(g["weight_checksum"]), rel=1e-9), "weight RNG drifted"
    z = W.synthetic_latents(cfg, 1, int(g["latent_seed"]))
    lat = OD.shapevae_forward(sd, z, cfg.heads)
    step = lat.shape[1] // g["latents_out_rows"].shape[0]                             # token rows stored every `step`
    assert np.abs(lat[0, ::step].numpy() - g["latents_out_rows"]).max() < 1e-4        # ShapeVAE.forward
    q = torch.from_numpy(g["queries"])
    out = OD.geo_decoder_forward(W.geo_decoder_state(sd), q, lat, W.fourier_frequencies(cfg), cfg.dec_heads)[0, :, 0]
    assert np.abs(out.numpy() - g["logits"]).max() < 2e-5                            # CrossAttentionDecoder.forward


def test_flash_processors_match_reference(gold, checksum):
    cfg = W.MINI
    g = gold("flash_processors_mini.npz")
    sd = W.synthetic_state_dict(cfg, seed=0)
    assert checksum(sd) == pytest.approx(float(g["weight_checksum"]), rel=1e-9)
    lat = OD.shapevae_forward(sd, W.synthetic_latents(cfg, 1, 1234), cfg.heads)
    q = torch.from_numpy(g["queries"])
    counts = [int(c) for c in g["counts"]]
    gsd, fr = W.geo_decoder_state(sd), W.fourier_frequencies(cfg)
    for mode in ("mean", "merge"):
        proc = OD.FlashProcessorOracle(mode)
        for name, state in [("level0", True), ("bins", ([3, 9, 40], counts))]:
            proc.topk = state
            out = OD.geo_decoder_forward(gsd, q, lat, fr, cfg.dec_heads, kv_select=proc)[0, :, 0]
            assert np.abs(out.numpy() - g[f"{mode}_{name}"]).max() < 2e-5, (mode, name)


def test_near_surface_bit_exact(gold):
    g = gold("near_surface.npz")
    for grid, mask, alpha in zip(g["grids"], g["masks"], g["alphas"]):
        assert np.array_equal(OV.near_surface_mask(grid, float(alpha)), mask)


def test_volume_decoders_on_analytic_field(gold):
    g = gold("volume_analytic.npz")
    assert np.array_equal(OV.vanilla_decode(analytic, 1.01, 5000, 24), g["vanilla24"])
    h, st = OV.hierarchical_decode(analytic, 1.01, 20000, 0.0, 64, 15, return_stats=True)
    assert np.array_equal(np.isnan(h), np.isnan(g["hier64"]))
    assert np.array_equal(np.nan_to_num(h), np.nan_to_num(g["hier64"]))
    assert st["queries"] == list(g["hier64_queries"])
    f, st = OV.flashvdm_decode(lambda p, topk: analytic(p), 1.01, 20000, 0.0, 64, 15, return_stats=True)
    assert np.array_equal(np.isnan(f), np.isnan(g["flash64"]))
    assert np.array_equal(np.nan_to_num(f), np.nan_to_num(g["flash64"]))
    assert st["levels"] == [15, 30, 60] and st["queries"] == list(g["flash64_queries"])


def test_octree_counts_at_reference_resolution(gold):
    """SURVEY §8c golden numbers produced by the reference: res 128 visited sets."""
    g = gold("volume_analytic.npz")
    h, st = OV.hierarchical_decode(analytic, 1.01, 200000, 0.0, 128, 63, return_stats=True)
    assert int((~np.isnan(h)).sum()) == int(g["hier128_visited"]) == 294426
    f, st = OV.flashvdm_decode(lambda p, topk: analytic(p), 1.01, 200000, 0.0, 128, 63, return_stats=True)
    assert int((~np.isnan(f)).sum()) == int(g["flash128_visited"]) == 286014
    assert f.shape == (127, 127, 127)


def test_level_lists():
    assert OV.hierarchy_levels(384) == [96, 192, 384]
    assert OV.flash_levels(384) == [95, 190, 380]
    assert OV.flash_levels(512) == [63, 126, 252, 504]
    assert OV.flash_levels(128) == [63, 126]


def test_volume_decoders_on_real_decoder(gold, checksum):
    cfg = W.MINI
    g = gold("volume_decoder_mini.npz")
    sd = W.sparsify_field(W.synthetic_state_dict(cfg, seed=0), cfg, int(g["keep_freqs"]), float(g["gain"]), float(g["bias"]))
    assert checksum(sd) == pytest.approx(float(g["weight_checksum"]), rel=1e-9)
    lat = OD.shapevae_forward(sd, W.synthetic_latents(cfg, 1, 1234), cfg.heads)
    gsd, fr = W.geo_decoder_state(sd), W.fourier_frequencies(cfg)
    dec = lambda p: OD.geo_decoder_forward(gsd, p[None], lat, fr, cfg.dec_heads)[0, :, 0]
    h = OV.hierarchical_decode(dec, 1.01, 3000, 0.0, 32, 15)
    assert np.array_equal(np.isnan(h), np.isnan(g["hier32"]))
    assert np.abs(np.nan_to_num(h) - np.nan_to_num(g["hier32"])).max() < 5e-5
    for mode in ("mean", "merge"):
        proc = OD.FlashProcessorOracle(mode)

        def dec_group(p, topk):
            proc.topk = topk
            return OD.geo_decoder_forward(gsd, p, lat.expand(p.shape[0], -1, -1), fr, cfg.dec_heads, kv_select=proc)[..., 0]
        f = OV.flashvdm_decode(dec_group, 1.01, 3000, 0.0, 32, 15)
        assert np.array_equal(np.isnan(f), np.isnan(g[f"flash32_{mode}"]))
        assert np.abs(np.nan_to_num(f) - np.nan_to_num(g[f"flash32_{mode}"])).max() < 5e-5


# ---- marching cubes: PARITY UNPINNED against skimage; LUT-independent invariants (SURVEY App. D) ----

def sphere(n=49):
    x = np.linspace(-1.01, 1.01, n, dtype=np.float32)
    X, Y, Z = np.meshgrid(x, x, x, indexing="ij")
    return np.tanh(20 * (0.6 - np.sqrt(X * X + Y * Y + Z * Z))).astype(np.float32)


def sign_change_edges(vol, level=0.0):
    ins = (vol - np.float32(level)) > 0
    return int((ins[1:] != ins[:-1]).sum() + (ins[:, 1:] != ins[:, :-1]).sum() + (ins[:, :, 1:] != ins[:, :, :-1]).sum())


def test_mc_oracle_invariants_closed_surface():
    vol = sphere()
    v, f, _, _ = OM.marching_cubes(vol, 0.0)
    assert v.dtype == np.float32 and f.dtype == np.int32
    assert v.shape[0] == sign_change_edges(vol)                    # one welded vertex per sign-change edge
    assert f.shape[0] == 2 * v.shape[0] - 4                        # closed genus-0 surface
    e = np.concatenate([f[:, [0, 1]], f[:, [1, 2]], f[:, [2, 0]]])
    _, cnt = np.unique(np.sort(e, 1), axis=0, return_counts=True)
    assert (cnt == 2).all()                                        # watertight manifold
    assert len(np.unique(e, axis=0)) == len(e)                     # consistently oriented
    a, b, c = (v[f[:, i]].astype(np.float64) for i in range(3))
    assert np.einsum("ij,ij->i", a, np.cross(b, c)).sum() < 0      # raw winding: normals toward higher values
    # every vertex lies on its grid edge at the linear-interpolation parameter
    frac = v - np.floor(v)
    assert ((frac > 1e-6).sum(1) <= 1).all()
    r = np.linalg.norm((v / 48.0) * 2.02 - 1.01, axis=1)
    assert np.abs(r - 0.6).max() < 2e-3


def test_mc_oracle_random_field_watertight_inside():
    rng = np.random.default_rng(0)
    vol = rng.standard_normal((14, 15, 16)).astype(np.float32)
    v, f, _, _ = OM.marching_cubes(vol, 0.1)
    assert v.shape[0] == sign_change_edges(vol, 0.1)
    cases = OM.cube_cases(vol, 0.1)
    assert cases.shape == (13, 14, 15)
    used = np.zeros(v.shape[0], bool)
    used[f.reshape(-1)] = True
    assert used.all()


def test_mc_oracle_errors_and_nan():
    vol = sphere(17)
    with pytest.raises(ValueError):
        OM.marching_cubes(vol, 5.0)
    vol2 = vol.copy()
    vol2[vol2 > 0.9] = np.nan                                      # NaN next to positive values (sparse decoders)
    v, f, _, _ = OM.marching_cubes(vol2, 0.0)                      # range check disabled by NaN, like skimage
    assert np.isnan(v).any() and f.shape[0] > 0


def test_extractor_rescale_matches_reference_contract(gold):
    g = gold("latents2mesh_mini24.npz")
    assert g["mesh_v"].dtype == np.float32 and g["mesh_f"].dtype == np.int32
    # vertices / (res+1) * size + min : everything inside the (shrunk) box
    assert g["mesh_v"].min() >= -1.01 and g["mesh_v"].max() <= 1.01 * (24 / 25) + 1e-6


# ---- round-2 vectors (oracle/make_golden.py r2): BASELINE configurations ---------------------------------------------

def _flash_oracle(gsd, lat, fr, heads, mode, res, minres):
    proc = OD.FlashProcessorOracle(mode)

    def dec_group(p, topk):
        proc.topk = topk
        return OD.geo_decoder_forward(gsd, p, lat.expand(p.shape[0], -1, -1), fr, heads, kv_select=proc)[..., 0]
    return OV.flashvdm_decode(dec_group, 1.01, 600, 0.0, res, minres, return_stats=True)


def test_hierarchical_odd_levels_match_reference(gold):
    """Levels built with r // 2 (reference vd:202-208) need not double: 35 -> [8, 17, 35] = grids 9, 18 (= 2n), 36 (= 2n).
    The reference scatters at 2c into the (r+1)^3 grid and dilates with zero padding at ITS faces."""
    g = gold("volume_analytic_r2.npz")
    for res, minres in [(35, 8), (45, 10)]:
        h, st = OV.hierarchical_decode(analytic, 1.01, 20000, 0.0, res, minres, return_stats=True)
        assert h.shape == (res + 1,) * 3 and st["queries"] == list(g[f"hier{res}_queries"])
        assert np.array_equal(np.isnan(h), np.isnan(g[f"hier{res}"]))
        assert np.array_equal(np.nan_to_num(h), np.nan_to_num(g[f"hier{res}"]))
    assert OV.hierarchy_levels(390) == [97, 195, 390] and OV.hierarchy_levels(70, 15) == [17, 35, 70]
    _, st = OV.hierarchical_decode(analytic, 1.01, 200000, 0.0, 70, 15, return_stats=True)
    assert st["queries"] == list(g["hier70_queries"])


def test_three_level_hierarchical_and_mesh_on_real_decoder(gold, checksum):
    """3 levels with expand_num=1 on the middle one (vd:250-259) and odd levels on the real mini decoder; the octree-64
    dense field gives the >= 10k-vertex end-to-end mesh the reference's latents2mesh produced (MC = oracle, unpinned)."""
    cfg = W.MINI
    g = gold("volume_decoder_mini_r2.npz")
    sd = W.sparsify_field(W.synthetic_state_dict(cfg, seed=0), cfg, int(g["keep_freqs"]), float(g["gain"]), float(g["bias"]))
    assert checksum(sd) == pytest.approx(float(g["weight_checksum"]), rel=1e-9)
    lat = OD.shapevae_forward(sd, W.synthetic_latents(cfg, 1, 1234), cfg.heads)
    gsd, fr = W.geo_decoder_state(sd), W.fourier_frequencies(cfg)
    dec = lambda p: OD.geo_decoder_forward(gsd, p[None], lat, fr, cfg.dec_heads)[0, :, 0]
    for res, minres in [(64, 15), (35, 8)]:
        h, st = OV.hierarchical_decode(dec, 1.01, 8000, 0.0, res, minres, return_stats=True)
        ref = g[f"hier{res}"]
        assert len(st["levels"]) == 3 and st["queries"] == list(g[f"hier{res}_queries"])
        assert np.array_equal(np.isnan(h), np.isnan(ref))
        assert np.abs(np.nan_to_num(h) - np.nan_to_num(ref)).max() < 5e-5
    m = gold("latents2mesh_mini64.npz")
    assert m["mesh_v"].shape[0] >= 10000 and m["mesh_f"].max() == m["mesh_v"].shape[0] - 1
    grid = OV.vanilla_decode(dec, 1.01, 8000, 64)
    v, f = OM.mc_surface_extract(grid, mc_level=0.0, bounds=1.01, octree_resolution=64)
    assert np.array_equal(f, m["mesh_f"]) and np.abs(v - m["mesh_v"]).max() < 1e-4


@pytest.mark.parametrize("tag,res", [("turbo", 32), ("turbo", 64), ("full", 32)])
def test_flashvdm_turbo_and_full_match_reference(tag, res, gold, checksum):
    """BASELINE config 4 (mini-turbo: no q/k norm, latents_proj, expand 1, top-256) and the full decoder (top-1024,
    attention_processors.py:40-45), both selection modes."""
    cfg = CFG[tag]
    g = gold(f"flash_{tag}.npz")
    sd = W.sparsify_field(W.synthetic_state_dict(cfg, seed=0), cfg, int(g["keep_freqs"]), float(g["gain"]), float(g["bias"]))
    assert checksum(sd) == pytest.approx(float(g["weight_checksum"]), rel=1e-9)
    torch.set_num_threads(8)
    lat = OD.shapevae_forward(sd, W.synthetic_latents(cfg, 1, 1234), cfg.heads)
    gsd, fr = W.geo_decoder_state(sd), W.fourier_frequencies(cfg)
    for mode in ("mean", "merge"):
        f, st = _flash_oracle(gsd, lat, fr, cfg.dec_heads, mode, res, 15)
        ref = g[f"flash{res}_{mode}"]
        assert st["queries"] == list(g[f"flash{res}_{mode}_queries"])
        assert np.array_equal(np.isnan(f), np.isnan(ref))
        assert np.abs(np.nan_to_num(f) - np.nan_to_num(ref)).max() < 5e-5 * max(1.0, float(g["gain"]) / 6.0)


def test_decoder_include_pi_matches_reference(gold, checksum):
    import dataclasses
    cfg = dataclasses.replace(W.MINI, include_pi=True)
    g = gold("decoder_pi.npz")
    sd = W.synthetic_state_dict(cfg, seed=0)
    assert checksum(sd) == pytest.approx(float(g["weight_checksum"]), rel=1e-9)
    fr = W.fourier_frequencies(cfg)
    assert abs(float(fr[0]) - np.pi) < 1e-6
    lat = OD.shapevae_forward(sd, W.synthetic_latents(cfg, 1, 1234), cfg.heads)
    out = OD.geo_decoder_forward(W.geo_decoder_state(sd), torch.from_numpy(g["queries"]), lat, fr, cfg.dec_heads)[0, :, 0]
    assert np.abs(out.numpy() - g["logits"]).max() < 2e-5
