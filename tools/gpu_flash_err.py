import os, sys, numpy as np, torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import hy3dgeo
from hy3dgeo import weights as W, _lib
from hy3dgeo.volume_decoders import FlashVDMVolumeDecoding
dev = torch.device('cuda:0')
g = np.load(os.path.join(ROOT, 'tests', 'golden', 'volume_decoder_mini.npz'))
cfg = W.MINI
gain = float(g["gain"])
sd = W.sparsify_field(W.synthetic_state_dict(cfg, seed=0), cfg, int(g["keep_freqs"]), gain, float(g["bias"]))
vae = hy3dgeo.B200ShapeVAE(cfg, sd, device=dev)
ctx = _lib.get_context(dev)
for impl in ("tc", "torch"):
    lat = vae(W.synthetic_latents(cfg, 1, 1234).to(dev), impl=impl)
    for bits, poly in ((0, 1), (0, 0), (32, 0), (0x10000, 1), (0x10020, 0)):
        ctx.debug_experiment(bits, poly)
        for mode in ("mean", "merge"):
            dec = FlashVDMVolumeDecoding(mode)
            out = dec(lat, vae.geo_decoder, bounds=1.01, num_chunks=3000, mc_level=0.0, octree_resolution=32, min_resolution=15, enable_pbar=False)[0].cpu().numpy()
            ref = g[f"flash32_{mode}"]
            same = np.array_equal(np.isnan(out), np.isnan(ref))
            err = np.abs(np.nan_to_num(out) - np.nan_to_num(ref))
            print(impl, hex(bits), poly, mode, "nan-equal", same, "max err", err.max(), "mean err", err.mean(), "n>6e-3", int((err > 6e-3).sum()), flush=True)
