"""ORACLE (test infrastructure, never shipped): CPU restatement of the reference's
volume decoders — dense grid generation, near-surface extraction, the
coarse-to-fine octree refinement and the FlashVDM query binning.

Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s CPU-baseline legs
may import this.  Reference: ``hy3dgen/shapegen/models/autoencoders/volume_decoders.py``
(cited as ``vd:LINE``).  Pinned by ``oracle/make_golden.py`` against the
reference classes (Hierarchical with the int64-coordinate defect at vd:262-264
patched to float32, see SURVEY §0.3 / Appendix E).

``decode`` arguments are callables ``f(points[P,3] float32 tensor) -> logits[P]``
so the same code runs against the decoder oracle or an analytic field.
"""
from __future__ import annotations

from typing import Callable, List, Sequence, Tuple, Union

import numpy as np
import torch

SENTINEL = -10000.0
BAND = 0.95


def normalize_bounds(bounds) -> np.ndarray:
    """vd:158-161 — a Python float b means the cube [-b, b]^3."""
    if isinstance(bounds, float):
        bounds = [-bounds, -bounds, -bounds, bounds, bounds, bounds]
    return np.asarray(bounds, dtype=np.float64)


def axis_tables(bounds, res: int) -> List[np.ndarray]:
    """vd:131-133 — per-axis ``np.linspace(min, max, res+1, dtype=float32)``
    (float64 arithmetic, then one rounding to float32)."""
    b = normalize_bounds(bounds)
    return [np.linspace(b[a], b[a + 3], int(res) + 1, dtype=np.float32) for a in range(3)]


def dense_points(bounds, res: int) -> np.ndarray:
    """vd:122-138 — meshgrid 'ij', flat index (i*N + j)*N + k, columns x,y,z."""
    x, y, z = axis_tables(bounds, res)
    xs, ys, zs = np.meshgrid(x, y, z, indexing="ij")
    return np.stack((xs, ys, zs), axis=-1).reshape(-1, 3)


def hierarchy_levels(octree_resolution: int, min_resolution: int = 63) -> List[int]:
    """vd:202-208."""
    res, r = [], int(octree_resolution)
    if r < min_resolution:
        res.append(r)
    while r >= min_resolution:
        res.append(r)
        r //= 2
    res.reverse()
    return res


def flash_levels(octree_resolution: int, min_resolution: int = 63, mini_grid_num: int = 4) -> List[int]:
    """vd:310-319 — level 0 snapped to a multiple of mini_grid_num minus 1 (Python
    ``round``: banker's rounding), later levels r0 * 2^i."""
    res = hierarchy_levels(octree_resolution, min_resolution)
    res[0] = round(res[0] / mini_grid_num) * mini_grid_num - 1
    for i in range(1, len(res)):
        res[i] = res[0] * 2 ** i
    return res


def near_surface_mask(g: np.ndarray, alpha: float) -> np.ndarray:
    """vd:29-119 restated: ``val = g + alpha``; a voxel is flagged when it is valid
    (val > -9000) and the sign of any of its 6 axis neighbours (index clamped at
    the border; an invalid neighbour is replaced by the voxel's own value)
    differs from its own sign.  sign(0) = 0 is its own class (torch.sign)."""
    val = (g + np.float32(alpha)).astype(np.float32)
    valid = val > -9000
    s = np.sign(val)
    diff = np.zeros(val.shape, dtype=bool)
    n = val.shape
    for axis in range(3):
        for shift in (1, -1):
            idx = np.clip(np.arange(n[axis]) + shift, 0, n[axis] - 1)
            nb = np.take(val, idx, axis=axis)
            nb = np.where(nb > -9000, nb, val)
            diff |= np.sign(nb) != s
    return (diff & valid).astype(np.int32)


def box3(mask: np.ndarray) -> np.ndarray:
    """3x3x3 all-ones Conv3d with zero padding, thresholded > 0 (vd:224-225,254-259)."""
    m = mask.astype(bool)
    out = np.zeros_like(m)
    p = np.pad(m, 1)
    n0, n1, n2 = m.shape
    for a in range(3):
        for b in range(3):
            for c in range(3):
                out |= p[a:a + n0, b:b + n1, c:c + n2]
    return out


def refine_active_set(grid: np.ndarray, mc_level: float, last: bool, nf: int = None) -> np.ndarray:
    """One coarse->fine step of vd:247-260 / vd:378-391 (SURVEY Appendix B).
    ``grid`` is the coarse level [n,n,n]; returns the boolean fine mask [nf,nf,nf]
    of voxels to query.  ``nf`` = r + 1 of the next level (vd:243): 2n-1 when the
    resolution doubles exactly (default), 2n when the coarse level is an odd r // 2
    (vd:202-208); the scatter at 2c (vd:256) and the zero-padded dilations (vd:258)
    act on that grid."""
    act = (near_surface_mask(grid, mc_level) > 0) | (np.abs(grid) < BAND)
    if not last:
        act = box3(act)
    n = grid.shape[0]
    nf = 2 * (n - 1) + 1 if nf is None else int(nf)
    up = np.zeros((nf, nf, nf), dtype=bool)
    cx, cy, cz = np.nonzero(act)
    up[cx * 2, cy * 2, cz * 2] = True
    up = box3(up)
    if last:
        up = box3(up)
    return up


def refined_coords(idx: np.ndarray, bounds, res: int) -> np.ndarray:
    """vd:394-396 (the float32 form; Hierarchical's vd:262-264 is patched to
    this): ``float32(idx) * float32(bbox_size / res) + float32(bbox_min)``,
    elementwise fp32 multiply then add."""
    b = normalize_bounds(bounds)
    cell = ((b[3:] - b[:3]) / res).astype(np.float32)
    return (idx.astype(np.float32) * cell + b[:3].astype(np.float32)).astype(np.float32)


Decode = Callable[[torch.Tensor], torch.Tensor]


def _decode_chunks(decode: Decode, pts: np.ndarray, num_chunks: int) -> np.ndarray:
    out = []
    for s in range(0, pts.shape[0], num_chunks):
        out.append(decode(torch.from_numpy(pts[s:s + num_chunks])).reshape(-1).numpy())
    return np.concatenate(out).astype(np.float32) if out else np.zeros((0,), np.float32)


def vanilla_decode(decode: Decode, bounds=1.01, num_chunks=10000, octree_resolution=None) -> np.ndarray:
    """vd:141-182 for one latent -> float32 [N,N,N]."""
    N = int(octree_resolution) + 1
    pts = dense_points(bounds, octree_resolution)
    return _decode_chunks(decode, pts, num_chunks).reshape(N, N, N)


def hierarchical_decode(decode: Decode, bounds=1.01, num_chunks=10000, mc_level=0.0,
                        octree_resolution=None, min_resolution=63, return_stats=False):
    """vd:185-277 (patched coordinates) for one latent -> float32 [N,N,N], NaN = unvisited."""
    levels = hierarchy_levels(octree_resolution, min_resolution)
    N0 = levels[0] + 1
    grid = _decode_chunks(decode, dense_points(bounds, levels[0]), num_chunks).reshape(N0, N0, N0)
    stats = {"levels": levels, "queries": [N0 ** 3]}
    for r in levels[1:]:
        up = refine_active_set(grid, mc_level, last=(r == levels[-1]), nf=r + 1)
        idx = np.stack(np.nonzero(up), axis=1)                 # lexicographic (torch.where order)
        vals = _decode_chunks(decode, refined_coords(idx, bounds, r), num_chunks)
        nxt = np.full(up.shape, SENTINEL, dtype=np.float32)
        nxt[up] = vals
        grid = nxt
        stats["queries"].append(int(idx.shape[0]))
    grid = grid.copy()
    grid[grid == SENTINEL] = np.nan
    return (grid, stats) if return_stats else grid


# ----------------------------------------------------------------------------
# FlashVDM geometry (vd:280-435)
# ----------------------------------------------------------------------------

def flash_minigrid_order(N: int, mini_grid_num: int = 4) -> np.ndarray:
    """vd:343-354 — permutation mapping (mini-grid, inner) order to the dense
    flat index.  Returns int64 [mini^3, (N/mini)^3] of dense linear indices."""
    m, s = mini_grid_num, N // mini_grid_num
    lin = np.arange(N ** 3, dtype=np.int64).reshape(m, s, m, s, m, s)
    return lin.transpose(0, 2, 4, 1, 3, 5).reshape(m ** 3, s ** 3)


def flash_bins(pts: np.ndarray, query_grid_num: int = 6) -> np.ndarray:
    """vd:398-403 — bin id of each refined query from its own bounding box:
    ``floor((p - min) / (max - min) * (6 - 0.001))`` per axis in float32, id =
    36 bx + 6 by + bz."""
    p = torch.from_numpy(pts)
    mn = p.min(0).values
    mx = p.max(0).values
    v = (p - mn) / (mx - mn) * (query_grid_num - 0.001)
    i = torch.floor(v).long()
    return (i[:, 0] * query_grid_num ** 2 + i[:, 1] * query_grid_num + i[:, 2]).numpy()


def flash_pack_bins(bin_ids: Sequence[int], counts: Sequence[int], num_chunks: int):
    """vd:408-427 — consecutive whole bins packed into calls while
    ``sum + count < num_chunks`` (the first bin of a call is always accepted).
    Returns a list of (ids, counts) per decoder call."""
    calls, cur, total = [], [[], []], 0
    for b, c in zip(bin_ids, counts):
        if total + c < num_chunks or total == 0:
            total += c
            cur[0].append(b)
            cur[1].append(c)
        else:
            calls.append(cur)
            cur, total = [[b], [c]], c
    if total > 0:
        calls.append(cur)
    return calls


def flashvdm_level(decode_group: Callable, grid: np.ndarray, bounds, r: int, last: bool, num_chunks: int = 10000,
                   mc_level: float = 0.0):
    """One refined level of vd:373-431: ``grid`` is the previous level (sentinel -10000 = unvisited) -> the level of
    resolution ``r`` in the same form, the number of queries and the per-call (bin ids, counts).  Exposed on its own so
    that a device implementation can be checked level by level on ITS OWN previous level: the active set, the 6^3
    binning and the stride sampling are discontinuous in the coarse values, so two implementations whose logits differ
    below tolerance may legitimately diverge after a threshold flip — but never given the same field."""
    up = refine_active_set(grid, mc_level, last=last)
    idx = np.stack(np.nonzero(up), axis=1)
    P = refined_coords(idx, bounds, r)
    bins = flash_bins(P)
    order_ = np.argsort(bins, kind="stable")               # vd:404 (stable on CPU, SURVEY §7.3-5)
    Ps = P[order_]
    ub, uc = np.unique(bins, return_counts=True)
    calls = flash_pack_bins(ub.tolist(), uc.tolist(), num_chunks)
    vals_sorted = np.empty(Ps.shape[0], dtype=np.float32)
    start = 0
    for ids, cnts in calls:
        n = int(sum(cnts))
        out = decode_group(torch.from_numpy(Ps[None, start:start + n]), (ids, cnts)).numpy()
        vals_sorted[start:start + n] = out.reshape(-1)
        start += n
    vals = np.empty_like(vals_sorted)
    vals[order_] = vals_sorted
    nxt = np.full(up.shape, SENTINEL, dtype=np.float32)
    nxt[up] = vals
    return nxt, int(idx.shape[0]), calls


def flashvdm_decode(decode_group: Callable, bounds=1.01, num_chunks=10000, mc_level=0.0,
                    octree_resolution=None, min_resolution=63, mini_grid_num=4, return_stats=False):
    """vd:291-435 for one latent -> float32 [N',N',N'], NaN = unvisited.

    ``decode_group(points[G,P,3] tensor, topk)`` evaluates the decoder with the
    FlashVDM processor state ``topk`` (True for level-0 mini-grids where the
    leading dim is the mini-grid batch; ``(ids, counts)`` for refined levels
    where G == 1) and returns logits [G,P].
    """
    levels = flash_levels(octree_resolution, min_resolution, mini_grid_num)
    N0 = levels[0] + 1
    pts = dense_points(bounds, levels[0])
    order = flash_minigrid_order(N0, mini_grid_num)             # [64, s^3]
    nb = max(num_chunks // order.shape[1], 1)                   # vd:356
    flat = np.empty(N0 ** 3, dtype=np.float32)
    for s in range(0, order.shape[0], nb):
        sel = order[s:s + nb]
        out = decode_group(torch.from_numpy(pts[sel]), True).numpy()
        flat[sel.reshape(-1)] = out.reshape(-1)
    grid = flat.reshape(N0, N0, N0)
    stats = {"levels": levels, "queries": [N0 ** 3], "calls": []}
    for r in levels[1:]:
        grid, nq, calls = flashvdm_level(decode_group, grid, bounds, r, r == levels[-1], num_chunks, mc_level)
        stats["queries"].append(nq)
        stats["calls"].append([(list(i), list(c)) for i, c in calls])
    grid = grid.copy()
    grid[grid == SENTINEL] = np.nan
    return (grid, stats) if return_stats else grid


def flash_layout_reference(index: np.ndarray, n: int, cell: np.ndarray, bmin: np.ndarray, stride: int):
    """Host restatement of vd:394-412 for the padded layout of ``hy3d_flash_layout_bins``: oracle bin ids, stable sort,
    128-padding, samples -> (padded index, per-tile group, samples, sample offsets, per-bin counts)."""
    idx = np.stack(np.unravel_index(index.astype(np.int64), (n, n, n)), 1)
    pts = (idx.astype(np.float32) * cell.astype(np.float32) + bmin.astype(np.float32)).astype(np.float32)
    with np.errstate(all="ignore"):
        bins = flash_bins(pts)
    bins = np.clip(bins, 0, 215)
    order = np.argsort(bins, kind="stable")
    counts = np.bincount(bins, minlength=216)
    cap = (len(index) + 216 * 127 + 127) // 128 * 128
    pidx = np.full(cap, -1, np.int32)
    tile_group = np.full(cap // 128, 215, np.int32)
    samples, soff, pos, at = [], [0], 0, 0
    for g in range(216):
        members = index[order[at:at + counts[g]]]
        at += counts[g]
        pc = (counts[g] + 127) // 128 * 128
        pidx[pos:pos + counts[g]] = members
        tile_group[pos // 128:(pos + pc) // 128] = g
        pos += pc
        samples.append(members[::stride])
        soff.append(soff[-1] + len(samples[-1]))
    return pidx, tile_group, np.concatenate(samples).astype(np.int32), np.asarray(soff, np.int32), counts.astype(np.int32)


def check_sparse_levels(dec, out, ref=None, tol=None, mc_level=0.0, exact=False, tie_frac=0.0):
    """A sparse decoder's grid against the reference's.  The active sets are a discontinuous function of the coarse
    values (sign changes, |v| < 0.95), so with fp16-operand logits (error up to `tol`) a voxel within `tol` of a threshold
    may flip and carry its fine neighbourhood in or out of the visited set.  What must hold:
      * exact (fp32 chain): the visited set IS the reference's;
      * always: every level's visited set is exactly what the reference logic (oracle, bit-pinned to the reference) derives
        from OUR previous level — "active-cell sets bit-exact given the same field";
      * every voxel both visited agrees within `tol`; the sets differ on < 1 % of the visited voxels.
    `dec` ran with ``keep_levels=True``; `ref` None checks the level chain alone (no reference grid at that size).
    `tie_frac` (FlashVDM only): the fraction of voxels allowed above `tol` (never above 5 x `tol`) — a near-tie of the KV
    selection (rank 256 vs 257 of the mean similarity, p vs 1e-6) resolves differently under 1e-5 changes of the latents
    and moves the logits of that one bin; the reference is exactly as sensitive to its own latents."""
    vis = ~np.isnan(out)
    lv = [g.cpu().numpy() for g in dec.last_levels]
    for k in range(len(lv) - 1):
        want = refine_active_set(lv[k], mc_level, last=(k == len(lv) - 2), nf=lv[k + 1].shape[0])
        assert np.array_equal(want, lv[k + 1] != SENTINEL), f"level {k + 1}: active set is not the reference logic's for the same field"
    assert np.array_equal(vis, lv[-1] != SENTINEL)
    if ref is None:
        return
    rvis = ~np.isnan(ref)
    if exact:
        assert np.array_equal(vis, rvis), "visited set differs from the reference"
    both = vis & rvis
    assert (vis ^ rvis).sum() < 0.01 * rvis.sum(), ((vis ^ rvis).sum(), rvis.sum())
    err = np.abs(out[both] - ref[both])
    if tie_frac > 0:
        assert err.max() < 5 * tol and (err > tol).mean() <= tie_frac, (err.max(), (err > tol).mean())
    else:
        assert err.max() < tol, err.max()
