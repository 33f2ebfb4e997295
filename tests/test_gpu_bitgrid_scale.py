"""GPU tests of the bit-grid kernels (octree refinement, marching cubes, dual marching cubes) against the oracle, exactly,
at the two places they can go wrong unnoticed by the small-grid tests of test_gpu_parity.py / test_dmc.py:

  * the shape edges of the bit-row layouts: rows that fill their 32-bit words exactly or overrun them by one voxel, the
    8- / 16- / 32-lane row layouts of the MC / DMC row kernels (8, 16, 32 words per row and one more), row counts at the
    4096-row scan-chunk edge and above the 1024 chunks one block of ``k_scan_chunks`` sums in one pass;
  * the BASELINE configurations at full size, stage by stage, each stage fed with what the device itself produced at the
    stage before (its own coarse level, its own grid): octree 384 Hierarchical (configs[2]), dense octree 256 / 512
    (configs[1] / [4], the 513^3 grid also cut into 8 slabs), FlashVDM octree 384 levels (configs[3]).

Decoder values at full size are sampled (first / last list entries, every 262 144-th list position +-1 — the decoder's
chunk edges — and random ones) and compared with the float64 oracle on the device's own latents; the measured errors are
printed (run with -s to see them).
"""
import os

import numpy as np
import pytest
import torch

import hy3dgeo
from hy3dgeo import _lib, weights as W
from hy3dgeo.surface_extractors import DMCSurfaceExtractor, MCSurfaceExtractor
from hy3dgeo.volume_decoders import FlashVDMVolumeDecoding, HierarchicalVolumeDecoding, VanillaVolumeDecoder, refine_level
from oracle import decoder as OD, dmc as ODMC, mc as OM, volume as OV
from oracle.mesh import assert_same_mesh, bits_equal

pytestmark = pytest.mark.gpu
LOGIT_TOL = 1e-3                 # the suite's logit tolerance for the O(1)-scale field, times the head gain
CHUNK = 262144                   # points per decoder launch chunk


@pytest.fixture(scope="module")
def dev():
    return torch.device("cuda:0")


@pytest.fixture(scope="module")
def ctx(dev):
    return _lib.get_context(dev)


def device_mc(ctx, g, level):
    """Raw marching cubes of the device grid ``g`` (vertices in index units, as the oracle's) -> host arrays."""
    nv, nf, _ = ctx.mc_count(g, level)
    v = torch.empty((nv, 3), dtype=torch.float32, device=g.device)
    f = torch.empty((nf, 3), dtype=torch.int32, device=g.device)
    ctx.mc_emit((1, 1, 1), (1, 1, 1), (0, 0, 0), v, f)
    return v.cpu().numpy(), f.cpu().numpy()


def device_dmc(ctx, g):
    nv, nf, _ = ctx.dmc_count(g)
    v = torch.empty((nv, 3), dtype=torch.float32, device=g.device)
    f = torch.empty((nf, 3), dtype=torch.int32, device=g.device)
    ctx.dmc_emit(v, f)
    return v.cpu().numpy(), f.cpu().numpy()


def shell(n, r=0.6, sharp=20.0):
    x = np.linspace(-1.01, 1.01, n, dtype=np.float32)
    return np.tanh(sharp * (r - np.sqrt(x[:, None, None] ** 2 + x[None, :, None] ** 2 + x[None, None, :] ** 2))).astype(np.float32)


# ------------------------------------------------------------------------------- octree refinement: word edges
REFINE_N = [31, 32, 33, 63, 64, 65, 95, 96, 97, 127, 128, 129]     # coarse rows of 1-5 words: short, exact, one over


def refine_field(kind, n):
    rng = np.random.default_rng(n)
    if kind == "shell":
        return shell(n)
    if kind == "band":                                  # |g| < BAND everywhere: every fine voxel is active
        return rng.uniform(-0.9, 0.9, (n, n, n)).astype(np.float32)
    if kind == "flat":                                  # far from the level: nothing is active
        return np.full((n, n, n), 5.0, np.float32)
    g = (rng.standard_normal((n, n, n)) * 2).astype(np.float32)
    if kind == "holes":                                 # unvisited voxels of a sparse level
        g[rng.random(g.shape) < 0.3] = OV.SENTINEL
    return g


@pytest.mark.parametrize("kind", ["shell", "noise", "holes", "band", "flat"])
@pytest.mark.parametrize("n", REFINE_N)
def test_refine_word_edges_match_oracle(ctx, n, kind):
    """hy3d_refine_level for fine grids 2n-1 and 2n, dilated and last levels: the exact ordered index list, nothing written
    past it, the count-only call; and with a capacity below the count, the first `cap` entries right, nothing written at or
    past `cap`, the full count returned."""
    grid = refine_field(kind, n)
    g = torch.from_numpy(grid).cuda()
    for nf in (2 * n - 1, 2 * n):
        for last in (False, True):
            want = np.flatnonzero(OV.refine_active_set(grid, 0.0, last, nf=nf).reshape(-1)).astype(np.int32)
            if kind == "band":
                assert want.size == nf ** 3
            if kind == "flat":
                assert want.size == 0
            buf = torch.full((want.size + 64,), -7, dtype=torch.int32, device="cuda")
            cnt = ctx.refine_level(g, 0.0, last, buf, nf)
            out = buf.cpu().numpy()
            assert cnt == want.size and np.array_equal(out[:cnt], want), (nf, last)
            assert (out[cnt:] == -7).all(), (nf, last)
            assert ctx.refine_level(g, 0.0, last, None, nf) == want.size
            if want.size > 1:
                cap = want.size // 2 + 1
                buf.fill_(-7)
                assert ctx.refine_level(g, 0.0, last, buf[:cap], nf) == want.size
                out = buf.cpu().numpy()
                assert np.array_equal(out[:cap], want[:cap]) and (out[cap:] == -7).all(), (nf, last, cap)


# ------------------------------------------------------------------ marching cubes / dual marching cubes: layout edges
def edge_field(shape, seed, offset=0.0):
    """Noise (about half of all edges cross 0) with exact zeros ("g > 0" is false at the level) and NaNs."""
    rng = np.random.default_rng(seed)
    vol = (rng.standard_normal(shape) + offset).astype(np.float32)
    vol[rng.random(shape) < 0.05] = 0.0
    vol[rng.random(shape) < 0.01] = np.nan
    return vol


N2_EDGES = [32, 64, 255, 256, 257, 511, 512, 513, 1023, 1024]       # 1, 2, 8, 8 / 9, 16 / 17, 32 words per row
ROW_EDGES = [(63, 65, 40), (64, 64, 40), (17, 241, 40)]             # 4095, 4096, 4097 rows: one scan chunk and one over


@pytest.mark.parametrize("shape", [(3, 5, n2) for n2 in N2_EDGES] + ROW_EDGES)
def test_mc_dmc_layout_edges_bit_exact(ctx, shape):
    vol = edge_field(shape, sum(shape))
    g = torch.from_numpy(vol).cuda()
    for level in (0.0, 0.3):
        assert_same_mesh(device_mc(ctx, g, level), OM.marching_cubes_raw(vol, level))
    assert_same_mesh(device_dmc(ctx, g), ODMC.dual_marching_cubes(vol))


def test_mc_dmc_more_than_1024_scan_chunks_bit_exact(ctx):
    """2048 x 2049 rows of 2 voxels: 1025 chunks of 4096 rows, so the chunk-sum scan runs a second 1024-block pass and
    the last chunk is half full.  Offset noise keeps the mesh at ~2.6 M vertices, present in every chunk."""
    shape = (2048, 2049, 2)
    vol = edge_field(shape, 7, offset=1.5)
    g = torch.from_numpy(vol).cuda()
    assert_same_mesh(device_mc(ctx, g, 0.0), OM.marching_cubes_raw(vol, 0.0))
    assert_same_mesh(device_dmc(ctx, g), ODMC.dual_marching_cubes(vol))


def test_mc_dmc_reject_rows_over_1024_voxels(ctx):
    g = torch.from_numpy(edge_field((3, 3, 1025), 1)).cuda()
    with pytest.raises(_lib.Hy3dError):
        ctx.mc_count(g, 0.0)
    with pytest.raises(_lib.Hy3dError):
        ctx.dmc_count(g)


# -------------------------------------------------------------------------------- BASELINE configurations, full size
@pytest.fixture(scope="module")
def full_sd():
    return W.synthetic_state_dict(W.FULL, seed=0)


def sample_positions(length, seed, total=4096):
    """List positions to check: first, last, every CHUNK-th +-1, random ones up to `total`, ascending."""
    edges = [m * CHUNK + d for m in range(1, (length - 1) // CHUNK + 1) for d in (-1, 0, 1)]
    rng = np.random.default_rng(seed)
    pos = np.concatenate([[0, length - 1], edges, rng.integers(0, length, max(total - len(edges) - 2, 0))])
    return np.unique(pos[(pos >= 0) & (pos < length)]).astype(np.int64)


class LogitCheck:
    """Device logits against the float64 oracle decoder on the device's own latents, at the float32 coordinates the
    product forms."""

    def __init__(self, cfg, sd, lat):
        torch.set_num_threads(os.cpu_count())
        self.cfg = cfg
        self.gsd = {k: v.double() for k, v in W.geo_decoder_state(sd).items()}
        self.fr = W.fourier_frequencies(cfg).double()
        self.lat = lat.detach().cpu().double().reshape(1, *lat.shape[-2:])

    def __call__(self, got, pts, tol, rms_tol, what):
        ref = torch.cat([OD.geo_decoder_forward(self.gsd, torch.from_numpy(pts[s:s + 1024]).double()[None], self.lat, self.fr,
                                                self.cfg.dec_heads)[0, :, 0] for s in range(0, len(pts), 1024)]).numpy()
        err = np.abs(got.astype(np.float64) - ref)
        mx, rms = float(err.max()), float(np.sqrt((err ** 2).mean()))
        print(f"\n{what}: {len(pts)} points, logit error max {mx:.3e} rms {rms:.3e} (|logit| max {np.abs(ref).max():.2f})")
        assert mx < tol and rms < rms_tol, (what, mx, rms)
        return mx, rms


def dense_points(res, flat):
    """float32 coordinates of flat indices of the dense (res+1)^3 grid: the linspace axis tables (reference vd:131-133)."""
    ax = OV.axis_tables(1.01, res)
    N = res + 1
    return np.stack([ax[0][flat // (N * N)], ax[1][(flat // N) % N], ax[2][flat % N]], 1)


def test_hierarchical_octree384_full_size(dev, ctx, full_sd):
    """configs[2]: HierarchicalVolumeDecoding at octree 384 (97 -> 193 -> 385) on the full model and the benchmark's sparse
    field.  Each level's visited set is refine_active_set of the device's own previous level; ~4096 logits per level
    against the float64 oracle; MC and DMC of the 385^3 NaN-bearing grid bit-exact against the oracles."""
    from bench import SPARSE_FULL
    cfg = W.FULL
    sd = W.sparsify_field(full_sd, cfg, **SPARSE_FULL)
    gain = SPARSE_FULL["gain"]
    vae = hy3dgeo.B200ShapeVAE(cfg, sd, device=dev)
    lat = vae(W.synthetic_latents(cfg, 1, 1234).to(dev))
    dec = HierarchicalVolumeDecoding(keep_levels=True)
    out = dec(lat, vae.geo_decoder, bounds=1.01, num_chunks=8000, mc_level=0.0, octree_resolution=384, enable_pbar=False)[0]
    ctx.check_watchdog()
    assert dec.last_stats[0]["levels"] == [96, 192, 384] and out.shape == (385, 385, 385)
    grid = out.cpu().numpy()
    OV.check_sparse_levels(dec, grid)
    check = LogitCheck(cfg, sd, lat[0])
    lv = [g.cpu().numpy() for g in dec.last_levels]
    for k, r in enumerate([96, 192, 384]):
        flat = np.arange(lv[k].size) if k == 0 else np.flatnonzero(lv[k].reshape(-1) != OV.SENTINEL)
        assert 0 < len(flat) < lv[k].size // 4 or k == 0
        sel = flat[sample_positions(len(flat), k)]
        if k == 0:
            pts = dense_points(r, sel)
        else:
            pts = OV.refined_coords(np.stack(np.unravel_index(sel, lv[k].shape), 1), 1.01, r)
        # measured on one B200: max 4.7e-3 / 5.1e-3 / 4.7e-3, rms 1.35e-3 / 1.39e-3 / 1.37e-3 (gain 9.18)
        check(lv[k].reshape(-1)[sel], pts, LOGIT_TOL * gain, LOGIT_TOL * gain / 4, f"configs[2] level {k} ({r + 1}^3)")
    del lv
    v, f = MCSurfaceExtractor().run(out, mc_level=0.0, bounds=1.01, octree_resolution=384)
    assert np.isnan(v).any()
    assert_same_mesh((v, f), OM.mc_surface_extract(grid, mc_level=0.0, bounds=1.01, octree_resolution=384))
    del v, f
    assert_same_mesh(DMCSurfaceExtractor().run(out), ODMC.dual_marching_cubes(grid))


@pytest.mark.parametrize("res", [256, 512])
def test_dense_full_size(res, dev, ctx, full_sd):
    """configs[1] / configs[4]: VanillaVolumeDecoder at octree 256 / 512 on the full model.  Sampled logits (corners, the
    decoder's chunk edges, random voxels) against the float64 oracle; MC and DMC of the 257^3 / 513^3 grid bit-exact against
    the oracles (513: 17-word rows, the 32-lane layout); at 513 the grid cut into 8 slabs with a halo concatenates to the
    whole-grid mesh bit for bit."""
    from hy3dgeo.parallel import MC_HALO, slab_planes
    cfg = W.FULL
    vae = hy3dgeo.B200ShapeVAE(cfg, full_sd, device=dev)
    lat = vae(W.synthetic_latents(cfg, 1, 1234).to(dev))
    out = VanillaVolumeDecoder()(lat, vae.geo_decoder, bounds=1.01, num_chunks=8000, octree_resolution=res, enable_pbar=False)[0]
    ctx.check_watchdog()
    N = res + 1
    assert out.shape == (N, N, N)
    corners = np.array([((i * N) + j) * N + k for i in (0, N - 1) for j in (0, N - 1) for k in (0, N - 1)])
    sel = np.unique(np.concatenate([corners, sample_positions(N ** 3, res)]))
    got = out.reshape(-1)[torch.from_numpy(sel).to(dev)].cpu().numpy()
    # measured on one B200: max 3.9e-4 / 4.0e-4, rms 1.03e-4 / 1.02e-4 at octree 256 / 512
    LogitCheck(cfg, full_sd, lat[0])(got, dense_points(res, sel), LOGIT_TOL, LOGIT_TOL / 4, f"dense octree {res} ({N}^3)")

    ext = MCSurfaceExtractor()
    kw = dict(mc_level=0.0, bounds=1.01, octree_resolution=res)
    v_ref, f_ref = ext.run_device(out, **kw)
    grid = out.cpu().numpy()
    vo, fo = OM.mc_surface_extract(grid, **kw)
    assert bits_equal(v_ref.cpu().numpy(), vo) and np.array_equal(f_ref.cpu().numpy(), fo)
    del vo, fo
    if res == 512:
        vs, fs, base = [], [], 0
        for r in range(8):
            x0, x1 = slab_planes(N, r, 8)
            slab = out[x0:min(x1 + MC_HALO, N)].contiguous()
            nv, nf, _ = ext.count_slab(slab, x1 - x0, 0.0)
            v, f = ext.emit_slab(nv, nf, x0, base, bounds=1.01, octree_resolution=res)
            vs.append(v); fs.append(f); base += nv
            del slab
        v, f = torch.cat(vs), torch.cat(fs)
        del vs, fs
        assert v.shape == v_ref.shape and f.shape == f_ref.shape
        assert torch.equal(v.view(torch.int32), v_ref.view(torch.int32)) and torch.equal(f, f_ref)
        del v, f
    del v_ref, f_ref
    assert_same_mesh(DMCSurfaceExtractor().run(out), ODMC.dual_marching_cubes(grid))


def test_flashvdm_octree384_levels_and_layout(gold, dev, ctx):
    """configs[3] levels: FlashVDMVolumeDecoding at octree 384 (96 -> 191 -> 381) on the mini-turbo decoder.  Each level's
    visited set is refine_active_set of the device's own previous level; the bin layout of the device's own index lists
    at 191 and 381 bit for bit against the restatement, sample strides 50 ('mean') and 30 ('merge').
    The field is the suite's mini-turbo sparse field (flash_turbo.npz): the full model's calibration (bench.SPARSE_FULL)
    would put every mini-turbo logit far above the level, leaving nothing to refine."""
    g = gold("flash_turbo.npz")
    cfg = W.MINI_TURBO
    sd = W.sparsify_field(W.synthetic_state_dict(cfg, seed=0), cfg, int(g["keep_freqs"]), float(g["gain"]), float(g["bias"]))
    vae = hy3dgeo.B200ShapeVAE(cfg, sd, device=dev)
    lat = vae(W.synthetic_latents(cfg, 1, 1234).to(dev))
    dec = FlashVDMVolumeDecoding("mean", keep_levels=True)
    out = dec(lat, vae.geo_decoder, bounds=1.01, num_chunks=8000, mc_level=0.0, octree_resolution=384, enable_pbar=False)[0]
    ctx.check_watchdog()
    assert dec.last_stats[0]["levels"] == [95, 190, 380] and out.shape == (381, 381, 381)
    OV.check_sparse_levels(dec, out.cpu().numpy())
    del out
    bmin = np.full(3, -1.01, np.float32)
    for k in (1, 2):
        coarse, n = dec.last_levels[k - 1], dec.last_levels[k].shape[0]
        index = refine_level(ctx, coarse, 0.0, last=(k == 2), nf=n)
        idx = index.cpu().numpy()
        assert np.array_equal(idx, np.flatnonzero(dec.last_levels[k].cpu().numpy().reshape(-1) != OV.SENTINEL))
        print(f"\nconfigs[3] level {k} ({n}^3): {len(idx)} visited voxels")
        assert 0 < len(idx) < n ** 3 // 4
        cell = (np.full(3, 2.02) / (n - 1)).astype(np.float32)
        for stride in (50, 30):
            pidx, tg, sidx, soff, counts = ctx.flash_layout_bins(index, (n, n, n), cell, bmin, stride, with_counts=True)
            rp, rt, rs, ro, rc = OV.flash_layout_reference(idx, n, cell, bmin, stride)
            assert np.array_equal(counts.cpu().numpy(), rc)
            assert np.array_equal(soff.cpu().numpy(), ro)
            assert np.array_equal(pidx.cpu().numpy(), rp)
            s = sidx.cpu().numpy()
            assert np.array_equal(s[:len(rs)], rs) and bool((s[len(rs):] == -1).all())
            assert np.array_equal(tg.cpu().numpy(), rt)
