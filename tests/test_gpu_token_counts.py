"""The tcgen05 attention paths along the token-count axis, against a float64 oracle.

The number of latent tokens M decides every partial-tile path of the attention code: the zero K/V padding rows of the
last 128-token tile, the per-64-column-half `valid` masks of both softmax kernels, the measured per-head score bound over
M rows, the KV-chunk indexing of the sequence-parallel transformer, and the FlashVDM radix select / gather / merge mask.
The number of 128-query tiles decides the duplicate, unstored tile of the shared-K/V attention and the idle CTA of a
GEMM pair.  Each test below moves one of those and compares with `oracle/decoder.py` evaluated in float64, or with the
same call on a fresh context (bit for bit), so that a failure points at one kernel.

Tolerances are the project's: decoder logits within 1e-3 (max) and 2.5e-4 (rms) of float64; latent transformer within
1e-3 / 2e-4.  Every comparison prints its max / rms error (run pytest with -s to see them).
"""
import dataclasses
import functools
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import hy3dgeo
from hy3dgeo import _lib, weights as W
from oracle import decoder as OD, volume as OV

LOGIT_MAX, LOGIT_RMS = 1e-3, 2.5e-4
TF_MAX, TF_RMS = 1e-3, 2e-4
CH = 262144                                       # query chunk of the decoder (decode_tc_impl)

# token counts: every count of valid columns on both sides of the 64-column half boundary, and M on both sides of 128,
# 256 and 4096 (the largest set the FlashVDM selection takes)
DECODER_MS = [1, 63, 64, 65, 127, 128, 129, 191, 192, 193, 255, 257, 383, 385, 1000, 2049, 4095, 4096, 4097]
QUERY_COUNTS = [1, 129, 383]                      # 1 and 3 query tiles: odd counts leave a duplicate, unstored tile


def decoder64(gsd, queries, latents, freqs, heads, kv_select=None):
    """``oracle.decoder.geo_decoder_forward`` with every input in float64 (state dict, queries, latents, frequencies)."""
    return OD.geo_decoder_forward({k: v.double() for k, v in gsd.items()}, queries.double(), latents.double(), freqs.double(),
                                  heads, kv_select)


def _err(out, ref):
    d = (out.detach().cpu().double() - ref.double()).abs()
    return float(d.max()), float(d.pow(2).mean().sqrt())


def _check(label, out, ref, max_tol, rms_tol):
    mx, rms = _err(out, ref)
    print(f"[token-counts] {label}: max {mx:.3e} rms {rms:.3e}")
    assert mx < max_tol and rms < rms_tol, (label, mx, rms)


def _latents(M, width=1024):
    return torch.randn(M, width, generator=torch.Generator().manual_seed(1000 + M))


def _points(n, seed=7):
    return (torch.rand(n, 3, generator=torch.Generator().manual_seed(seed)) * 2 - 1) * 1.01


def _decoder_state(kind):
    """(cfg, decoder state dict) of a decoder kind: 'mini' (q/k norm: bounded-score kernel), 'turbo' (latents_proj, no
    q/k norm: online-softmax kernel), 'shifted' (mini with q/k norm gains x 1.4: bounded-score with per-head shift)."""
    cfg = W.MINI_TURBO if kind == "turbo" else W.MINI
    sd = W.synthetic_state_dict(cfg, seed=0, with_transformer=False)
    if kind == "shifted":
        c = "geo_decoder.cross_attn_decoder.attn.attention."
        for n in ("q_norm", "k_norm"):
            sd[c + n + ".weight"] = sd[c + n + ".weight"] * 1.4
    return cfg, W.geo_decoder_state(sd)


def _context(dev, kind):
    cfg, gsd = _decoder_state(kind)
    c = _lib.GeoContext(dev)
    c.set_decoder(gsd, cfg)
    c.set_precision(_lib.PRECISION_FP16_TC)
    return c


@functools.lru_cache(maxsize=None)
def _decoder_ref(kind, M, npts=max(QUERY_COUNTS)):
    torch.set_num_threads(os.cpu_count())
    cfg, gsd = _decoder_state(kind)
    return decoder64(gsd, _points(npts)[None], _latents(M)[None], W.fourier_frequencies(cfg), cfg.dec_heads)[0, :, 0]


# ------------------------------------------------------------------------------------------------ float64 oracle (CPU)
def test_float64_oracle_matches_fp32_oracle_and_reference_golden(gold, checksum):
    """The float64 oracle the GPU tests below compare with: on the mini golden's queries it agrees with the fp32 oracle
    within 1e-5, and both agree with the logits the reference produced."""
    torch.set_num_threads(os.cpu_count())
    cfg = W.MINI
    g = gold("decoder_mini.npz")
    sd = W.synthetic_state_dict(cfg, seed=int(g["seed"]))
    assert checksum(sd) == pytest.approx(float(g["weight_checksum"]), rel=1e-9)
    lat = OD.shapevae_forward(sd, W.synthetic_latents(cfg, 1, int(g["latent_seed"])), cfg.heads)
    gsd, fr = W.geo_decoder_state(sd), W.fourier_frequencies(cfg)
    q = torch.from_numpy(g["queries"])
    out32 = OD.geo_decoder_forward(gsd, q, lat, fr, cfg.dec_heads)[0, :, 0]
    out64 = decoder64(gsd, q, lat, fr, cfg.dec_heads)[0, :, 0]
    assert out64.dtype == torch.float64
    gl = torch.from_numpy(g["logits"]).double()
    assert float((out64 - out32.double()).abs().max()) < 1e-5
    assert float((out32.double() - gl).abs().max()) < 2e-5
    assert float((out64 - gl).abs().max()) < 2e-5


# ------------------------------------------------------------------------- A. decoder cross-attention at ragged M
KERNELS = {"mini": "bounded-score", "turbo": "online-softmax", "mini-forced-online": "online-softmax",
           "shifted": "bounded-score + per-head shift + exact redo"}
CASES_A = [(k, M) for k in ("mini", "turbo", "mini-forced-online") for M in DECODER_MS] + [("shifted", M) for M in (65, 300, 4097)]


@pytest.fixture(scope="module")
def dev():
    return torch.device("cuda:0")


@pytest.fixture(scope="module")
def contexts(dev):
    made = {}

    def get(kind):
        if kind not in made:
            made[kind] = _context(dev, kind)
        return made[kind]
    yield get
    for c in made.values():
        c.close()


def _decode(c, pts):
    out = c.decode_points(pts).cpu()
    c.check_watchdog()
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("kernel,M", CASES_A)
def test_decoder_attention_at_ragged_token_counts(kernel, M, dev, contexts):
    """Logits of 1, 129 and 383 queries against M latent tokens vs float64, on each attention kernel: the K/V padding
    rows, the valid-column masks of the last tile (both 64-column halves), the duplicate query tile."""
    kind = "mini" if kernel == "mini-forced-online" else kernel
    c = contexts(kind)
    c.prepare_kv(_latents(M).to(dev))
    ref = _decoder_ref("mini" if kernel == "mini-forced-online" else kernel, M)
    pts = _points(max(QUERY_COUNTS)).to(dev)
    forced = kernel == "mini-forced-online"
    try:
        c.debug_force_online_softmax(forced)
        assert c.attention_info()[1] == KERNELS[kernel]
        for P in QUERY_COUNTS:
            _check(f"decoder {kernel} M={M} P={P}", _decode(c, pts[:P]), ref[:P], LOGIT_MAX, LOGIT_RMS)
    finally:
        c.debug_force_online_softmax(False)


@pytest.mark.gpu
@pytest.mark.parametrize("kernel", ["mini", "turbo", "mini-forced-online"])
def test_decoder_attention_across_the_query_chunk(kernel, dev, contexts):
    """128 k + 1 queries over two 262144-point chunks (the second one of 3 query tiles) at M = 385."""
    M = 385
    kind = "mini" if kernel == "mini-forced-online" else kernel
    cfg, gsd = _decoder_state(kind)
    c = contexts(kind)
    lat = _latents(M)
    c.prepare_kv(lat.to(dev))
    pts = _points(CH + 257, seed=8)
    try:
        c.debug_force_online_softmax(kernel == "mini-forced-online")
        assert c.attention_info()[1] == KERNELS[kernel]
        out = _decode(c, pts.to(dev))
    finally:
        c.debug_force_online_softmax(False)
    torch.set_num_threads(os.cpu_count())
    for sl in (slice(0, 1), slice(127, 130), slice(CH - 1, CH + 257)):
        ref = decoder64(gsd, pts[None, sl], lat[None], W.fourier_frequencies(cfg), cfg.dec_heads)[0, :, 0]
        _check(f"decoder {kernel} M={M} P={CH + 257} rows {sl.start}:{sl.stop}", out[sl], ref, LOGIT_MAX, LOGIT_RMS)


# ------------------------------------------------------------------------- B. state carried between calls on one context
def _bits(t):
    return t.contiguous().view(torch.int32)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["mini", "shifted"])
def test_decoder_state_does_not_leak_between_token_counts(kind, dev):
    """Workspaces are grow-only (ws[], kv.ktile, kv.k32): M = 4096, then 300, then 4096 again on one context, each
    bit-identical to the same call on a fresh context — logits and the measured score bound of attention_info()."""
    c = _context(dev, kind)
    try:
        for M, P in [(4096, 1000), (300, 383), (4096, 1000)]:
            lat, pts = _latents(M).to(dev), _points(P).to(dev)
            c.prepare_kv(lat)
            out = _decode(c, pts)
            info = c.attention_info()
            f = _context(dev, kind)
            try:
                f.prepare_kv(lat)
                want = _decode(f, pts)
                assert info == f.attention_info(), (M, info, f.attention_info())
            finally:
                f.close()
            assert torch.equal(_bits(out), _bits(want)), f"M={M}: logits differ from a fresh context's"
    finally:
        c.close()


# ------------------------------------------------------------------------- C. latent transformer at odd tile counts
CFG_TF = dataclasses.replace(W.FULL, num_decoder_layers=4)


@functools.lru_cache(maxsize=1)
def _tf_state():
    return W.synthetic_state_dict(CFG_TF, seed=0)


def _tf_latents(B, M):
    return torch.randn(B, M, CFG_TF.embed_dim, generator=torch.Generator().manual_seed(77 + M))


@functools.lru_cache(maxsize=None)
def _tf_ref(M):
    torch.set_num_threads(os.cpu_count())
    sd = {k: v.double() for k, v in _tf_state().items()}
    return OD.shapevae_forward(sd, _tf_latents(2, M).double(), CFG_TF.heads)


@pytest.mark.gpu
@pytest.mark.parametrize("online", [False, True], ids=["bounded-score", "online-softmax"])
@pytest.mark.parametrize("M", [128, 384, 640, 1024])
def test_latent_transformer_at_odd_tile_counts(M, online, dev):
    """B200ShapeVAE.forward (4-layer FULL, batch 2) at 1, 3, 5 and 8 token tiles vs float64: odd tile counts leave one
    CTA of a GEMM pair idle and a duplicate query tile in the self-attention."""
    vae = hy3dgeo.B200ShapeVAE(CFG_TF, _tf_state(), device=dev)
    ctx = _lib.get_context(dev)
    try:
        ctx.debug_force_online_softmax(online)
        lat = vae(_tf_latents(2, M).to(dev)).cpu()
        ctx.check_watchdog()
    finally:
        ctx.debug_force_online_softmax(False)
    ref = _tf_ref(M)
    assert lat.shape == ref.shape
    _check(f"transformer {'online' if online else 'bounded'} M={M}", lat, ref, TF_MAX, TF_RMS)


@pytest.mark.gpu
def test_latent_transformer_rejects_token_counts_off_the_tile(dev):
    vae = hy3dgeo.B200ShapeVAE(CFG_TF, _tf_state(), device=dev)
    with pytest.raises(RuntimeError):
        vae(_tf_latents(1, 200).to(dev))


@pytest.mark.gpu
def test_transformer_state_does_not_leak_between_token_counts(dev):
    """3072, then 384, then 3072 tokens on one context: each bit-identical to the same call on a fresh context."""
    c = _lib.GeoContext(dev)
    try:
        c.set_transformer(_tf_state(), CFG_TF)
        for M in (3072, 384, 3072):
            z = _tf_latents(1, M)[0].to(dev)
            out = c.transformer_forward(z)
            f = _lib.GeoContext(dev)
            try:
                f.set_transformer(_tf_state(), CFG_TF)
                want = f.transformer_forward(z)
            finally:
                f.close()
            assert torch.equal(_bits(out), _bits(want)), f"M={M}: latents differ from a fresh context's"
    finally:
        c.close()


@pytest.mark.gpu
@pytest.mark.parametrize("parts,Ml", [(3, 128), (4, 128), (3, 384)])
def test_sequence_parallel_transformer_emulated_on_one_device(parts, Ml, dev):
    """hy3d_transformer_begin / layer_kv / layer_rest / end with `parts` contexts on one device, one per emulated rank;
    the all-gather of the K/V chunks is done with torch copies.  The concatenated rows are bit-identical to the
    single-context pass: the kv_tpr / kv_chunk_stride tile indexing at odd part counts and one tile per part."""
    cfg, sd = CFG_TF, _tf_state()
    M, H, L = parts * Ml, cfg.heads, cfg.num_decoder_layers
    z = _tf_latents(1, M)[0].to(dev)
    ctxs = [_lib.GeoContext(dev) for _ in range(parts)]
    try:
        for c in ctxs:
            c.set_transformer(sd, cfg)
        want = ctxs[0].transformer_forward(z)
        chunk = 2 * H * (Ml // 128) * 16384                     # [2 (K, V^T)][H][Ml / 128][16 KB] per part
        bufs = [torch.empty(parts * chunk, dtype=torch.uint8, device=dev) for _ in range(parts)]
        zl = [z[r * Ml:(r + 1) * Ml].contiguous() for r in range(parts)]
        outs = [torch.empty(Ml, cfg.width, dtype=torch.float32, device=dev) for _ in range(parts)]
        for r, c in enumerate(ctxs):
            c.sync_stream()
            c._check(c.lib.hy3d_transformer_begin(c.h, _lib._ptr(zl[r]), Ml, parts, r), "hy3d_transformer_begin")
        for l in range(L):
            for r, c in enumerate(ctxs):
                c._check(c.lib.hy3d_transformer_layer_kv(c.h, l, _lib._ptr(bufs[r])), "hy3d_transformer_layer_kv")
            for r in range(parts):
                for s in range(parts):
                    if s != r:
                        bufs[s][r * chunk:(r + 1) * chunk].copy_(bufs[r][r * chunk:(r + 1) * chunk])
            for r, c in enumerate(ctxs):
                c._check(c.lib.hy3d_transformer_layer_rest(c.h, l, _lib._ptr(bufs[r])), "hy3d_transformer_layer_rest")
        for r, c in enumerate(ctxs):
            c._check(c.lib.hy3d_transformer_end(c.h, _lib._ptr(outs[r])), "hy3d_transformer_end")
        for c in ctxs:
            c.check_watchdog()
        got = torch.cat(outs, 0)
        assert torch.equal(_bits(got), _bits(want)), [
            float((got[r * Ml:(r + 1) * Ml] - want[r * Ml:(r + 1) * Ml]).abs().max()) for r in range(parts)]
    finally:
        for c in ctxs:
            c.close()


# ------------------------------------------------------------------------- D. FlashVDM selection and grouped decoding
N0, MINI_GRIDS, STRIDE = 32, 4, 100
EPS_FACTOR = 32


def _q_side(gsd, pts, freqs, heads):
    """x0 and q of geo_decoder_forward (its first and third lines) for points [P, 3]: q [H, P, d]."""
    x0 = F.linear(OD.fourier_embed(pts[None], freqs), gsd["query_proj.weight"], gsd["query_proj.bias"])
    return x0, OD.q_heads(gsd, x0, heads)[0]


def _grid_points(axes, flat):
    i0, rem = np.divmod(flat, N0 * N0)
    i1, i2 = np.divmod(rem, N0)
    return torch.from_numpy(np.stack([axes[0][i0], axes[1][i1], axes[2][i2]], 1).astype(np.float32))


def _gather_heads(x, ids):
    """x [H, M, d], ids [H, n] -> [H, n, d]"""
    return torch.gather(x, 1, ids[..., None].expand(-1, -1, x.shape[-1]))


def _check_near_ties(name, dev_ids, ref_mask, dist, eps):
    """The device set may differ from the float64 set only by tokens whose float64 `dist` to the threshold is <= eps."""
    got = np.zeros_like(ref_mask)
    got[dev_ids] = True
    diff = np.nonzero(got ^ ref_mask)[0]
    assert diff.size == 0 or float(dist[diff].max()) <= eps, (name, diff[:8], dist[diff].max(), eps)
    return diff.size


@pytest.mark.gpu
@pytest.mark.parametrize("M", [300, 1000, 2049, 4096])
def test_flash_selection_and_grouped_decode_at_ragged_token_counts(M, dev, contexts):
    """Level-0 layout (64 mini-grids of 512 queries, every 100th sampled), budgets T in {1, 127, 128, 129, M // 3, M} and
    merge mode, on the mini decoder.

    Selection: the mean of the sampled q per group (float64 oracle q) dotted with the float64 k; each (group, head) device
    set equals the float64 top-T except for swaps of tokens whose float64 similarity lies within eps of the T-th value.
    eps: the device's sampled q and k come from 3-term split fp16 GEMMs with fp32 accumulation (hy3d_tc_sample_q,
    hy3d_tc_project_kv), fp32-grade — the dropped lo x lo product is 2^-22 relative, the tensor-core accumulation rounds
    no better than fp32.  So eps = 32 x the measured error of the same similarities in fp32 (CPU oracle, same inputs):
    about an order of magnitude of head-room over "a few times fp32".  Merge mode: tokens whose head-averaged
    probability exceeds 1e-6 for a sample, same argument in log space (|ln(p / 1e-6)| <= 2 eps, from the score and the
    log-sum-exp).

    Grouped decode: two query tiles of different groups (one with padding entries) through decode_flash_values; every
    logit vs the float64 oracle run with the DEVICE's own selection (read back with flash_selection), so the plain
    tolerance applies."""
    torch.set_num_threads(os.cpu_count())
    cfg, gsd = _decoder_state("mini")
    H, fr = cfg.dec_heads, W.fourier_frequencies(cfg)
    c = contexts("mini")
    lat = _latents(M)
    c.prepare_kv(lat.to(dev))
    pidx, tg, sidx, soff = c.flash_layout_minigrids(N0, MINI_GRIDS, STRIDE)
    G = MINI_GRIDS ** 3
    axes = OV.axis_tables(1.01, N0 - 1)
    soff_h = soff.cpu().numpy()
    samp = sidx.cpu().numpy()[: soff_h[-1]]
    pidx_h = pidx.cpu().numpy().reshape(G, -1)
    Mpad = (M + 127) // 128 * 128

    # float64 and fp32 oracle: k, v of the latent set; q of the sampled queries
    sd64 = {k: v.double() for k, v in gsd.items()}
    k64, v64 = (t[0] for t in OD.kv_heads(sd64, lat[None].double(), H))
    k32 = OD.kv_heads(gsd, lat[None], H)[0][0]
    spts = _grid_points(axes, samp)
    q64 = _q_side(sd64, spts.double(), fr.double(), H)[1]
    q32 = _q_side(gsd, spts, fr, H)[1]
    qbar64 = torch.stack([q64[:, soff_h[g]:soff_h[g + 1]].mean(1) for g in range(G)])        # [G, H, d]
    qbar32 = torch.stack([q32[:, soff_h[g]:soff_h[g + 1]].mean(1) for g in range(G)])
    sim64 = torch.einsum("ghd,hmd->ghm", qbar64, k64).numpy()
    sim32 = torch.einsum("ghd,hmd->ghm", qbar32, k32).double().numpy()
    eps = EPS_FACTOR * float(np.abs(sim32 - sim64).max())

    rng = np.random.default_rng(M)

    def decode_two_tiles(label, select_ids):
        """select_ids(g) -> LongTensor [H, n] of the device's tokens of group g"""
        gs = rng.choice(G, 2, replace=False)
        ks = rng.integers(0, pidx_h.shape[1] // 128, 2)
        idx = np.concatenate([pidx_h[g, 128 * k:128 * (k + 1)] for g, k in zip(gs, ks)]).astype(np.int32)
        idx[-13:] = -1                                                # padding entries of a layout
        out = c.decode_flash_values(torch.from_numpy(idx).to(dev), (N0, N0, N0),
                                    torch.from_numpy(gs.astype(np.int32)).to(dev), axes=axes).cpu()
        c.check_watchdog()
        valid = idx >= 0
        x0, q = _q_side(sd64, _grid_points(axes, idx[valid]).double(), fr.double(), H)
        rows = [np.arange(0, 128), np.arange(128, 256 - 13)]
        attn = torch.empty(H, int(valid.sum()), 64, dtype=torch.float64)
        for g, r in zip(gs, rows):
            ids = select_ids(int(g))
            attn[:, r] = OD.sdpa(q[:, r], _gather_heads(k64, ids), _gather_heads(v64, ids))
        ref = OD.decoder_tail(sd64, x0, attn[None], ln_post=True)[0, :, 0]
        _check(f"flash {label} M={M}", out[torch.from_numpy(valid)], ref, LOGIT_MAX, LOGIT_RMS)

    for T in sorted({1, 127, 128, 129, M // 3, M}):
        c.flash_select(sidx, (N0, N0, N0), soff, G, T, False, axes=axes)
        sel = c.flash_selection(G * H * T).cpu().numpy().reshape(G, H, T)
        assert bool((c.flash_group_tokens(G).cpu().numpy() == T).all())
        assert sel.min() >= 0 and sel.max() < M and bool((np.diff(sel, axis=-1) > 0).all())   # distinct, ascending
        swaps = 0
        for g in range(G):
            for h in range(H):
                s = sim64[g, h]
                kth = np.partition(s, M - T)[M - T]                                            # T-th largest
                ref = np.zeros(M, bool)
                ref[np.argsort(-s, kind="stable")[:T]] = True
                swaps += _check_near_ties(f"mean M={M} T={T} g={g} h={h}", sel[g, h], ref, np.abs(s - kth), eps)
        print(f"[token-counts] flash select mean M={M} T={T}: {swaps} near-tie tokens differ (eps {eps:.2e})")
        decode_two_tiles(f"mean T={T}", lambda g: torch.from_numpy(sel[g]).long())

    # merge mode: one token set per group, shared by all heads
    c.flash_select(sidx, (N0, N0, N0), soff, G, 1, True, axes=axes)
    ntok = c.flash_group_tokens(G).cpu().numpy()
    msel = c.flash_selection(G * Mpad).cpu().numpy().reshape(G, Mpad)
    assert bool((ntok >= 1).all()) and bool((ntok <= M).all())
    swaps, leps = 0, 0.0
    for g in range(G):
        s0, s1 = soff_h[g], soff_h[g + 1]
        lg64 = q64[:, s0:s1] @ k64.transpose(-1, -2)                                            # [H, S, M] unscaled
        lg32 = (q32[:, s0:s1] @ k32.transpose(-1, -2)).double()
        leps = max(leps, EPS_FACTOR * float((lg32 - lg64).abs().max()))
        pmax = lg64.softmax(-1).mean(0).max(0).values.numpy()
        ids = msel[g, :ntok[g]]
        assert ids.min() >= 0 and ids.max() < M and bool((np.diff(ids) > 0).all())
        swaps += _check_near_ties(f"merge M={M} g={g}", ids, pmax > 1e-6, np.abs(np.log(np.maximum(pmax, 1e-300) / 1e-6)), 2 * leps)
    print(f"[token-counts] flash select merge M={M}: set sizes {int(ntok.min())}..{int(ntok.max())}, {swaps} near-threshold tokens differ")
    decode_two_tiles("merge", lambda g: torch.from_numpy(msel[g, :ntok[g]]).long().expand(H, -1))


@pytest.mark.gpu
def test_flash_selection_rejects_more_than_4096_tokens(dev, contexts):
    c = contexts("mini")
    c.prepare_kv(_latents(4097).to(dev))
    _, _, sidx, soff = c.flash_layout_minigrids(N0, MINI_GRIDS, STRIDE)
    axes = OV.axis_tables(1.01, N0 - 1)
    for merge in (False, True):
        with pytest.raises(_lib.Hy3dError):
            c.flash_select(sidx, (N0, N0, N0), soff, MINI_GRIDS ** 3, 128, merge, axes=axes)
