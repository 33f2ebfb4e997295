"""Multi-GPU sharding of the volume decoders: one process per GPU, ``torch.distributed``
(NCCL over NVLink; gloo in the CPU tests) for the plumbing.

The reference has no multi-device path (SURVEY §2.2).  Query points are independent given the
K/V of the latent, so the grid is partitioned into slabs along axis 0 (the slowest-varying,
contiguous one) and the ordered active list of a refined level into equal contiguous ranges.
Exchange steps (the only collectives):
  * dense / level-0 slabs  -> all ranks (all_gather of equal padded slabs) or -> rank 0 (gather);
  * refined-level values   -> all ranks (all_gather of equal padded value ranges);
  * latents are replicated by the caller (each rank receives the same ``latents``; use
    ``broadcast_latents`` when only rank 0 holds them).
Marching cubes either runs on rank 0 over the assembled grid (at 385^3 the grid is 228 MB, ~0.3 ms
over NVLink) or stays sharded (``extract_mesh_sharded``): every rank keeps its slab, receives a
two-plane halo from its upper neighbour, extracts the part of the mesh it owns with globally
consistent vertex ids, and only the mesh pieces travel to rank 0 (BASELINE config 5).

The communication helpers take any decode callables, so the host logic is testable on CPU with
gloo and a fake field (tests/test_parallel_gloo.py).
"""
from __future__ import annotations

import bisect
import itertools
from typing import Callable, List, Optional, Sequence, Tuple

import numpy as np
import torch
import torch.distributed as dist

from .volume_decoders import (NAN, SENTINEL, axis_tables, bind, flash_levels, flash_topk_budget, hierarchy_levels, normalize_bounds,
                              refine_level)


def slab_planes(n_planes: int, rank: int, world: int) -> Tuple[int, int]:
    """Planes [x0, x1) of an axis-0 partition into ``world`` near-equal slabs."""
    base, rem = divmod(n_planes, world)
    x0 = rank * base + min(rank, rem)
    return x0, x0 + base + (1 if rank < rem else 0)


def list_range(n: int, rank: int, world: int) -> Tuple[int, int]:
    """Contiguous share [a, b) of an ordered list of n queries."""
    return slab_planes(n, rank, world)


def _staged(t: torch.Tensor, group) -> bool:
    """CUDA tensors under a gloo group (the 2-process tests that share one GPU) travel through host memory: gloo
    moves device tensors for broadcast / all_reduce only.  Under NCCL nothing is staged."""
    return t.is_cuda and dist.get_backend(group) == "gloo"


def _peer(group, r: int) -> int:
    """Global rank of group rank ``r``: P2POp / send / recv / broadcast name their peers by GLOBAL rank even when a
    sub-group is passed."""
    return r if group is None else dist.get_global_rank(group, r)


def _run_p2p(sends, recvs, group):
    """One batched group of point-to-point copies.  sends / recvs: lists of (tensor, group_rank); recv tensors may be
    views (slices of a larger buffer) — they are filled in place."""
    if not sends and not recvs:
        return
    ops, fix = [], []
    for t, r in sends:
        t = t.contiguous()
        ops.append(dist.P2POp(dist.isend, t.cpu() if _staged(t, group) else t, _peer(group, r), group))
    for t, r in recvs:
        if _staged(t, group) or not t.is_contiguous():
            buf = torch.empty(t.shape, dtype=t.dtype, device="cpu" if _staged(t, group) else t.device)
            fix.append((t, buf))
            ops.append(dist.P2POp(dist.irecv, buf, _peer(group, r), group))
        else:
            ops.append(dist.P2POp(dist.irecv, t, _peer(group, r), group))
    for q in dist.batch_isend_irecv(ops):
        q.wait()
    for t, buf in fix:
        t.copy_(buf)


def agree(ok: bool, device, group=None) -> bool:
    """True iff ``ok`` on every rank (one tiny all_reduce): lets all ranks leave a collective sequence together when
    one of them failed, instead of the healthy ones blocking in the next exchange."""
    flag = torch.tensor([0 if ok else 1], dtype=torch.int32, device="cpu" if dist.get_backend(group) == "gloo" else device)
    dist.all_reduce(flag, op=dist.ReduceOp.MAX, group=group)
    return int(flag.item()) == 0


def broadcast_latents(latents: Optional[torch.Tensor], shape, device, group=None, src: int = 0) -> torch.Tensor:
    """``src`` is a group rank."""
    if latents is None:
        latents = torch.empty(shape, dtype=torch.float32, device=device)
    latents = latents.contiguous()
    dist.broadcast(latents, src=_peer(group, src), group=group)
    return latents


def all_gather_ranges(local: torch.Tensor, counts: List[int], group=None) -> torch.Tensor:
    """Concatenate per-rank 1-D tensors of (known) different lengths on every rank: equal padded
    chunks through one all_gather, then trimmed."""
    world = dist.get_world_size(group)
    pad = max(counts) if counts else 0
    staged = _staged(local, group)
    dev = "cpu" if staged else local.device
    buf = torch.zeros(pad, dtype=local.dtype, device=dev)
    buf[: local.numel()] = local
    out = torch.empty(world * pad, dtype=local.dtype, device=dev)
    if buf.is_cuda:
        dist.all_gather_into_tensor(out, buf, group=group)
    else:
        dist.all_gather(list(out.view(world, pad).unbind(0)), buf, group=group)
    return torch.cat([out[r * pad: r * pad + counts[r]] for r in range(world)]).to(local.device)


def decode_dense_sharded(decode_range: Callable[[int, int, torch.Tensor], None], N: Tuple[int, int, int], device,
                         group=None, to_all: bool = True) -> Optional[torch.Tensor]:
    """``decode_range(first, count, out)`` fills ``out[:count]`` with the logits of flat indices
    [first, first+count).  Every rank decodes its slab; returns the full [n0,n1,n2] grid on every
    rank (to_all) or on rank 0 only (others get None)."""
    rank, world = dist.get_rank(group), dist.get_world_size(group)
    n0, n1, n2 = N
    plane = n1 * n2
    x0, x1 = slab_planes(n0, rank, world)
    local = torch.empty((x1 - x0) * plane, dtype=torch.float32, device=device)
    if x1 > x0:
        decode_range(x0 * plane, (x1 - x0) * plane, local)
    counts = [(b - a) * plane for a, b in (slab_planes(n0, r, world) for r in range(world))]
    if to_all:
        return all_gather_ranges(local, counts, group).view(n0, n1, n2)
    # one batched group of point-to-point copies (a single NCCL group launch; sizes differ per rank)
    sends, recvs, grid = [], [], None
    if rank == 0:
        grid = torch.empty(n0 * plane, dtype=torch.float32, device=device)
        grid[: counts[0]] = local
        off = counts[0]
        for r in range(1, world):
            if counts[r]:
                recvs.append((grid[off: off + counts[r]], r))
            off += counts[r]
    elif local.numel():
        sends.append((local, 0))
    _run_p2p(sends, recvs, group)
    return grid.view(n0, n1, n2) if rank == 0 else None


MC_HALO = 2      # planes of the next slab a rank needs (hy3dgeo.h: hy3d_mc_count_slab)


def exchange_halo(local: torch.Tensor, halo: int = MC_HALO, group=None) -> torch.Tensor:
    """``local`` = this rank's planes [p, n1, n2] of an axis-0 partition (every slab at least ``halo`` planes deep).
    Returns them followed by the first ``halo`` planes of the next rank's slab (nothing on the last rank): one
    batched send/recv between neighbours, N^2 * halo * 4 bytes per rank."""
    rank, world = dist.get_rank(group), dist.get_world_size(group)
    if world == 1:
        return local
    if local.shape[0] < halo:
        raise ValueError(f"slab of {local.shape[0]} planes is thinner than the {halo}-plane halo")
    sends, recv = [], None
    if rank > 0:
        sends.append((local[:halo], rank - 1))
    if rank < world - 1:
        recv = torch.empty((halo,) + tuple(local.shape[1:]), dtype=local.dtype, device=local.device)
    _run_p2p(sends, [] if recv is None else [(recv, rank + 1)], group)
    return local if recv is None else torch.cat([local, recv], 0)


def extract_mesh_sharded(local: torch.Tensor, plane0: int, count_slab: Callable, emit_slab: Callable, mc_level: float,
                         group=None, dst: int = 0, with_halo: bool = False):
    """Marching cubes over a grid that stays partitioned along axis 0.

    local      : this rank's planes [plane0, plane0 + p) of the grid, [p, n1, n2]; with ``with_halo`` the tensor
                 already ends with the next slab's first MC_HALO planes (ranks that decoded or hold them anyway)
    count_slab : (slab_with_halo, own_planes) -> (nV, nF, (vmin, vmax, has_nan))     (MCSurfaceExtractor.count_slab)
    emit_slab  : (nV, nF, plane0, id_base) -> (verts [nV, 3] float32, faces [nF, 3] int32), face ids global
    Returns (verts, faces) on ``dst`` (a group rank) — exactly the mesh of the whole grid: rank pieces are contiguous
    ranges of the global lexicographic vertex / face order — and None elsewhere; with ``dst=None`` every rank receives
    the mesh (one all-gather of the vertex pieces and one of the face pieces).  Raises the errors of
    ``skimage.measure.marching_cubes`` (level outside the data range, no surface) on every rank alike; ``mc_level=None``
    skips the range check (dual marching cubes has no level).  A rank whose own kernels fail makes ALL ranks raise before
    the mesh exchange (nobody is left blocked in a collective)."""
    rank, world = dist.get_rank(group), dist.get_world_size(group)
    own = local.shape[0] - (MC_HALO if with_halo and rank < world - 1 else 0)
    slab = local if with_halo else exchange_halo(local, MC_HALO, group)
    err, nv, nf, vmin, vmax, has_nan = None, 0, 0, float("nan"), float("nan"), False
    try:
        nv, nf, (vmin, vmax, has_nan) = count_slab(slab, own)
    except Exception as e:          # noqa: BLE001 - re-raised below, on every rank
        err = e
    inf = float("inf")
    mine = torch.tensor([nv, nf, vmin if vmin == vmin else inf, vmax if vmax == vmax else -inf, float(has_nan), float(err is not None)],
                        dtype=torch.float64, device="cpu" if _staged(local, group) else local.device)
    allst = torch.empty((world, 6), dtype=torch.float64, device=mine.device)
    dist.all_gather(list(allst.unbind(0)), mine, group=group)
    allst = allst.cpu()
    if err is not None:
        raise err
    if bool(allst[:, 5].max() > 0):
        raise RuntimeError("marching cubes failed on another rank of the group")
    nvs, nfs = [int(v) for v in allst[:, 0]], [int(v) for v in allst[:, 1]]
    gmin, gmax, any_nan = float(allst[:, 2].min()), float(allst[:, 3].max()), bool(allst[:, 4].max() > 0)
    if mc_level is not None and not any_nan and (mc_level < gmin or mc_level > gmax):
        raise ValueError("Surface level must be within volume data range.")
    if sum(nfs) == 0 and sum(nvs) == 0:        # marching cubes has faces iff it has vertices; a DMC mesh may have no face
        raise RuntimeError("No surface found at the given iso value.")
    verts = faces = None
    try:
        verts, faces = emit_slab(nv, nf, plane0, sum(nvs[:rank]))
    except Exception as e:          # noqa: BLE001
        err = e
    if not agree(err is None, local.device, group):
        raise err if err is not None else RuntimeError("marching cubes failed on another rank of the group")
    if dst is None:
        V = all_gather_ranges(verts.reshape(-1), [3 * v for v in nvs], group).view(-1, 3)
        F = all_gather_ranges(faces.reshape(-1), [3 * f for f in nfs], group).view(-1, 3) if sum(nfs) else faces
        return V, F
    # mesh pieces -> dst: one batched group of point-to-point copies (sizes differ per rank)
    sends, recvs, V, F = [], [], None, None
    if rank == dst:
        V = torch.empty((sum(nvs), 3), dtype=torch.float32, device=local.device)
        F = torch.empty((sum(nfs), 3), dtype=torch.int32, device=local.device)
        vo, fo = 0, 0
        for r in range(world):
            if r == rank:
                V[vo: vo + nvs[r]] = verts
                F[fo: fo + nfs[r]] = faces
            else:
                if nvs[r]:
                    recvs.append((V[vo: vo + nvs[r]], r))
                if nfs[r]:
                    recvs.append((F[fo: fo + nfs[r]], r))
            vo += nvs[r]; fo += nfs[r]
    else:
        if nv:
            sends.append((verts, dst))
        if nf:
            sends.append((faces, dst))
    _run_p2p(sends, recvs, group)
    return (V, F) if rank == dst else None


def decode_list_sharded(decode_values: Callable[[torch.Tensor], torch.Tensor], index: torch.Tensor, group=None) -> torch.Tensor:
    """``decode_values(index_slice) -> logits`` for an ordered index list known identically on all
    ranks; each rank evaluates its contiguous share, the values are all-gathered."""
    rank, world = dist.get_rank(group), dist.get_world_size(group)
    n = index.numel()
    a, b = list_range(n, rank, world)
    vals = decode_values(index[a:b]) if b > a else torch.empty(0, dtype=torch.float32, device=index.device)
    counts = [hi - lo for lo, hi in (list_range(n, r, world) for r in range(world))]
    return all_gather_ranges(vals, counts, group)


class SlabGrid:
    """A batch of occupancy grids left partitioned along axis 0 across a process group — the opaque grid of SURVEY §8b:
    it answers ``shape`` / ``len`` / ``[i]`` like the ``[B, N, N, N]`` tensor the reference decoders return, the B200
    ``MCSurfaceExtractor`` and ``DMCSurfaceExtractor`` recognise it and extract the mesh slab by slab (``extract_mesh_sharded``), and
    ``to_tensor()`` materialises the ordinary tensor on every rank for any other consumer.

    slabs[b]  : this rank's planes [plane0, plane0 + own) of item b, followed by the next slab's first MC_HALO planes
                when ``with_halo`` (ranks that evaluated them anyway), float32 [p, n1, n2]
    """

    def __init__(self, slabs: List[torch.Tensor], plane0, own, dims: Tuple[int, int, int], with_halo: bool, group=None,
                 dtype=torch.float32):
        B = len(slabs)
        self.slabs, self.dims, self.with_halo, self.group, self.dtype = slabs, tuple(dims), with_halo, group, dtype
        self.plane0s = list(plane0) if isinstance(plane0, (list, tuple)) else [int(plane0)] * B      # per item: the cuts of a
        self.owns = list(own) if isinstance(own, (list, tuple)) else [int(own)] * B                  # sparse level differ

    @property
    def plane0(self) -> int:
        return self.plane0s[0]

    @property
    def own(self) -> int:
        return self.owns[0]

    @property
    def shape(self):
        return torch.Size((len(self.slabs),) + self.dims)

    def __len__(self):
        return len(self.slabs)

    def __getitem__(self, b: int) -> "SlabGrid":
        return SlabGrid([self.slabs[b]], self.plane0s[b], self.owns[b], self.dims, self.with_halo, self.group, self.dtype)

    def to_tensor(self) -> torch.Tensor:
        """The whole batch [B, n0, n1, n2] on every rank (one all_gather of the owned planes per item)."""
        world = dist.get_world_size(self.group)
        n0, n1, n2 = self.dims
        B = len(self.slabs)
        meta = torch.tensor(self.owns, dtype=torch.int64, device="cpu" if _staged(self.slabs[0], self.group) else self.slabs[0].device)
        owns = torch.empty((world, B), dtype=torch.int64, device=meta.device)
        dist.all_gather(list(owns.unbind(0)), meta, group=self.group)
        owns = owns.cpu()
        return torch.stack([all_gather_ranges(sl[: self.owns[b]].reshape(-1), [int(v) * n1 * n2 for v in owns[:, b]], self.group)
                            .view(n0, n1, n2) for b, sl in enumerate(self.slabs)], 0).to(self.dtype)


class ShardedVanillaVolumeDecoder:
    """VanillaVolumeDecoder (reference volume_decoders.py:141-182) over a process group; same call signature.
    ``keep_sharded`` (default): every rank keeps its slab and a ``SlabGrid`` is returned on all ranks — marching cubes
    then runs per slab behind a two-plane halo exchange (BASELINE config 5).  Otherwise the slabs are gathered and
    the grid is returned on rank 0 (float32 [B,N,N,N]), None elsewhere."""

    def __init__(self, group=None, keep_sharded: bool = True):
        self.group = group
        self.keep_sharded = keep_sharded

    @torch.no_grad()
    def __call__(self, latents, geo_decoder, bounds=1.01, num_chunks=10000, octree_resolution=None, enable_pbar=True,
                 **kwargs):
        ctx = bind(latents, geo_decoder)
        axes = axis_tables(bounds, octree_resolution)
        N = int(octree_resolution) + 1
        rank, world = dist.get_rank(self.group), dist.get_world_size(self.group)
        outs = []
        if self.keep_sharded:
            if N < MC_HALO * world:        # decided identically on every rank: nobody is left waiting in the halo exchange
                raise ValueError(f"{N} planes cannot be split into {world} slabs of at least {MC_HALO} planes")
            x0, x1 = slab_planes(N, rank, world)
            for b in range(latents.shape[0]):
                ctx.prepare_kv(latents[b])
                local = torch.empty((x1 - x0, N, N), dtype=torch.float32, device=latents.device)
                ctx.decode_dense(axes, x0 * N * N, (x1 - x0) * N * N, local)
                outs.append(local)
            return SlabGrid(outs, x0, x1 - x0, (N, N, N), False, self.group)
        for b in range(latents.shape[0]):
            ctx.prepare_kv(latents[b])
            g = decode_dense_sharded(lambda first, count, out: ctx.decode_dense(axes, first, count, out), (N, N, N),
                                     latents.device, self.group, to_all=False)
            outs.append(g)
        if rank != 0:
            return None
        return torch.stack(outs, 0)


def plane_cuts(index: torch.Tensor, n: int, world: int, halo: int = MC_HALO):
    """Partition an ordered (lexicographic) active list of an [n,n,n] grid into ``world`` runs of WHOLE planes holding
    near-equal numbers of queries (variable-thickness slabs = balanced decoder work, SURVEY §8e): the ideal cut
    r * len / world is moved back to the start of its plane.  Returns host lists (planes, starts, ends): rank r owns
    planes [planes[r], planes[r+1]) = list entries [starts[r], starts[r+1]) and additionally evaluates the entries up to
    ends[r] (the actives of the next ``halo`` planes, which its marching-cubes slab needs).  One host read-back.
    Every slab is at least ``halo`` planes thick (the halo of rank r must lie inside rank r+1's slab)."""
    cnt, nn = index.numel(), n * n
    dev = index.device
    if cnt == 0 or world == 1:
        planes = [slab_planes(n, r, world)[0] for r in range(world)] + [n]
    else:
        pos = torch.tensor([r * cnt // world for r in range(1, world)], device=dev)
        planes = [0] + [int(v) for v in (index[pos] // nn).cpu()] + [n]
        for r in range(1, world):                       # strictly increasing by >= halo planes, leaving room for the rest
            planes[r] = min(max(planes[r], planes[r - 1] + halo), n - halo * (world - r))
    if any(b - a < halo for a, b in zip(planes, planes[1:])) and world > 1:
        raise ValueError(f"{n} planes cannot be split into {world} slabs of at least {halo} planes")
    keys = torch.tensor([p * nn for p in planes] + [min(p + halo, n) * nn for p in planes[1:]], dtype=index.dtype, device=dev)
    at = [int(v) for v in torch.searchsorted(index, keys).cpu()] if cnt else [0] * (2 * world + 1)
    return planes, at[: world + 1], at[world + 1:]


class _StageTimeline:
    """Diagnostics of the sharded sparse decoders: with ``self.timeline`` a dict, ``_tick(name)`` adds the wall time since the
    previous tick to stage ``name`` (ms, accumulated; synchronises the device; tools/gpu_hier_timeline.py)."""
    timeline = None

    def _tick(self, name, dev):
        if self.timeline is None:
            return
        import time
        torch.cuda.synchronize(dev)
        now = time.perf_counter()
        if getattr(self, "_t_last", None) is not None and name:
            self.timeline[name] = self.timeline.get(name, 0.0) + (now - self._t_last) * 1e3
        self._t_last = now


class ShardedHierarchicalVolumeDecoding(_StageTimeline):
    """HierarchicalVolumeDecoding (reference :185-277, patched coordinates) over a process group.

    Coarse levels: every rank evaluates its share (level 0: an axis-0 slab; refined levels: an equal contiguous range
    of the ordered active list), the values are all-gathered and every rank holds the whole level — the next active
    set is derived identically everywhere from it.
    Last level (``keep_sharded``, default): the grid is cut at plane boundaries into slabs holding near-equal numbers of
    active voxels; the decoder work is split into exactly equal ranges of the ordered list, and the values that fall
    into another rank's slab (or its two-plane marching-cubes halo) change hands in one batched point-to-point exchange
    (a few % of the list).  Each rank fills only its own slab and returns a ``SlabGrid`` — no all-gather of the values, no
    full-resolution grid anywhere; the mesh is then extracted slab by slab.  With ``keep_sharded=False`` the
    last level is gathered like the others and the ordinary tensor is returned on all ranks."""

    def __init__(self, group=None, keep_sharded: bool = True, timeline: bool = False):
        self.group = group
        self.keep_sharded = keep_sharded
        self.timeline = {} if timeline else None      # diagnostics: stage -> accumulated ms (synchronising; tools/gpu_hier_timeline.py)

    @torch.no_grad()
    def __call__(self, latents, geo_decoder, bounds=1.01, num_chunks=10000, mc_level=0.0, octree_resolution=None,
                 min_resolution=63, enable_pbar=True, **kwargs):
        self._tick(None, latents.device)
        ctx = bind(latents, geo_decoder)
        levels = hierarchy_levels(octree_resolution, min_resolution)
        b6 = normalize_bounds(bounds)
        bbox_min, bbox_size = b6[:3], b6[3:] - b6[:3]
        bmin32 = bbox_min.astype(np.float32)
        rank, world = dist.get_rank(self.group), dist.get_world_size(self.group)
        sharded_last = self.keep_sharded and len(levels) > 1 and levels[-1] + 1 >= MC_HALO * world
        outs, plane0s, owns = [], [], []
        self.last_stats = []
        for b in range(latents.shape[0]):
            ctx.prepare_kv(latents[b])
            self._tick("kv_prepare", latents.device)
            n0 = levels[0] + 1
            ax = axis_tables(bounds, levels[0])
            grid = decode_dense_sharded(lambda first, count, out: ctx.decode_dense(ax, first, count, out), (n0, n0, n0),
                                        latents.device, self.group, to_all=True).contiguous()
            self._tick("level0 decode + all_gather", latents.device)
            queries, mine = [n0 ** 3], [(slab_planes(n0, rank, world)[1] - slab_planes(n0, rank, world)[0]) * n0 * n0]
            for r in levels[1:]:
                n = r + 1
                last = r == levels[-1]
                index = refine_level(ctx, grid, mc_level, last=last, nf=n)
                self._tick(f"refine -> {n}^3 (replicated)", latents.device)
                cell = (bbox_size / r).astype(np.float32)
                queries.append(int(index.numel()))
                if last and sharded_last:
                    planes, starts, ends = plane_cuts(index, n, world)
                    self._tick("plane cuts", latents.device)
                    plane0, own = planes[rank], planes[rank + 1] - planes[rank]
                    p_hi = min(planes[rank + 1] + MC_HALO, n)
                    lo, hi = starts[rank], ends[rank]             # list entries whose values this rank's slab (+ halo) needs
                    # decoder work is split into EQUAL ranges of the list (plane-aligned slabs differ by up to +-8 % in
                    # queries at octree 384 on 8 GPUs); the few values that fall into a neighbour's slab change hands
                    # in one batched point-to-point exchange (every rank knows all the boundaries)
                    cnt = int(index.numel())
                    rng = [list_range(cnt, q, world) for q in range(world)]
                    a, bq = rng[rank]
                    vals = ctx.decode_list_values(index[a:bq], (n, n, n), cell, bmin32) if bq > a else \
                        torch.empty(0, dtype=torch.float32, device=latents.device)
                    need = torch.empty(hi - lo, dtype=torch.float32, device=latents.device)
                    sends, recvs = [], []
                    for q in range(world):
                        s0, s1 = max(a, starts[q]), min(bq, ends[q])          # mine, needed by q
                        r0, r1 = max(rng[q][0], lo), min(rng[q][1], hi)       # q's, needed by me
                        if q == rank:
                            if r1 > r0:
                                need[r0 - lo: r1 - lo] = vals[r0 - a: r1 - a]
                            continue
                        if s1 > s0:
                            sends.append((vals[s0 - a: s1 - a], q))
                        if r1 > r0:
                            recvs.append((need[r0 - lo: r1 - lo], q))
                    _run_p2p(sends, recvs, self.group)
                    slab = torch.empty((p_hi - plane0, n, n), dtype=torch.float32, device=latents.device)
                    ctx.fill(slab, float("nan"))           # unvisited = NaN from the start: no sentinel sweep afterwards
                    if hi > lo:
                        ctx.scatter(index[lo:hi], need, slab, base=plane0 * n * n)
                    part = index[a:bq]
                    grid = slab
                    plane0s.append(plane0); owns.append(own)
                    mine.append(int(part.numel()))
                    self._tick("last level decode (own slab)", latents.device)
                    break
                vals = decode_list_sharded(lambda idx: ctx.decode_list_values(idx, (n, n, n), cell, bmin32), index, self.group)
                nxt = torch.empty((n, n, n), dtype=torch.float32, device=latents.device)
                ctx.fill(nxt, SENTINEL)
                ctx.scatter(index, vals, nxt)
                grid = nxt
                a, bb = list_range(index.numel(), rank, world)
                mine.append(bb - a)
                self._tick(f"level {n}^3 decode + all_gather + scatter", latents.device)
            if not sharded_last:
                ctx.sentinel_to_nan(grid, SENTINEL)
            outs.append(grid)
            self.last_stats.append({"levels": levels, "queries": queries, "rank_queries": mine})
        if sharded_last:
            N = levels[-1] + 1
            return SlabGrid(outs, plane0s, owns, (N, N, N), True, self.group, latents.dtype)
        return torch.stack(outs, 0).to(latents.dtype)


def flash_partition(tiles_per_group: Sequence[int], world: int) -> List[Tuple[int, int, int, int]]:
    """Split the tiles of a group-ordered, 128-padded FlashVDM list into ``world`` contiguous runs whose tile counts differ
    by at most one (decoder work balanced to within one tile).  Returns per rank (t0, t1, g0, g1): tiles [t0, t1) and the
    groups [g0, g1) they use, from the group of the first tile to the group of the last.  A group cut by a boundary is
    selected by both neighbours; a rank without tiles gets (t0, t0, 0, 0)."""
    ends = list(itertools.accumulate(int(t) for t in tiles_per_group))
    total = ends[-1] if ends else 0
    parts = []
    for r in range(world):
        t0, t1 = list_range(total, r, world)
        if t1 == t0:
            parts.append((t0, t1, 0, 0))
        else:                                   # group of tile t = the first group whose tiles end past t
            parts.append((t0, t1, bisect.bisect_right(ends, t0), bisect.bisect_right(ends, t1 - 1) + 1))
    return parts


def flash_minigrid_sizes(N: int, mini_grid_num: int, stride: int = 100) -> Tuple[List[int], List[int]]:
    """Host image of the level-0 layout hy3d_flash_layout_minigrids writes: (queries per mini-grid, sample offsets [G+1]).
    Every mini-grid holds s^3 queries (s = N / mini_grid_num) padded to whole tiles and ceil(s^3 / stride) samples."""
    m = int(mini_grid_num)
    s3 = (int(N) // m) ** 3
    nsamp = -(-s3 // int(stride))
    return [s3] * m ** 3, [g * nsamp for g in range(m ** 3 + 1)]


def _tile_queries(counts: Sequence[int], t0: int, t1: int) -> int:
    """Real (non-padding) queries in tiles [t0, t1) of a padded list whose groups hold ``counts`` queries."""
    q, a = 0, 0
    for c in counts:
        k = -(-int(c) // 128)
        lo, hi = max(t0, a), min(t1, a + k)
        if hi > lo:
            q += min(c, 128 * (hi - a)) - min(c, 128 * (lo - a))
        a += k
    return q


class ShardedFlashVDMVolumeDecoding(_StageTimeline):
    """FlashVDMVolumeDecoding (reference volume_decoders.py:280-435) over a process group; same call signature, and the
    same grid bit for bit (NaNs included).

    Every rank holds the same K/V, refined active list and group layout (level 0: mini_grid_num^3 mini-grids; refined
    levels: 6^3 spatial bins), all cheap and deterministic.  The padded list's tiles are split into contiguous runs of
    near-equal length (``flash_partition``); each rank selects the K/V tokens of the groups its run touches (a group cut
    by a boundary is selected by both neighbours, identically) and decodes its run into compact values, which are
    all-gathered.  Level 0 and intermediate levels are then scattered into the whole grid on every rank.  The last level
    (``keep_sharded``, default, more than one level): each rank scatters into its plane-aligned slab (``plane_cuts``) plus
    the two-plane marching-cubes halo only and a ``SlabGrid`` is returned — no full-resolution grid on any rank.
    Otherwise the ordinary latents.dtype tensor is returned on every rank.  A refined level adds one host read-back (the
    216 bin counts and sample offsets) to what the single-GPU decoder synchronises on.

    ``last_stats[b]``: levels, queries (as FlashVDMVolumeDecoding), rank_queries (real queries this rank decoded)."""

    def __init__(self, topk_mode='mean', group=None, keep_sharded: bool = True, timeline: bool = False):
        if topk_mode not in ['mean', 'merge']:
            raise ValueError(f'Unsupported topk_mode {topk_mode}, available: {["mean", "merge"]}')
        self.topk_mode = topk_mode
        self.group = group
        self.keep_sharded = keep_sharded
        self.timeline = {} if timeline else None

    def _level(self, ctx, dims, layout, soff_h, counts, topk, merge, coords):
        """Select + decode this rank's run of a level's layout; -> (values of the whole padded list, this rank's queries)."""
        pidx, tile_group, sidx, soff = layout
        rank, world = dist.get_rank(self.group), dist.get_world_size(self.group)
        parts = flash_partition([-(-c // 128) for c in counts], world)
        t0, t1, g0, g1 = parts[rank]
        vals = torch.empty(0, dtype=torch.float32, device=pidx.device)
        if t1 > t0:
            ctx.flash_select_range(sidx[soff_h[g0]:], soff_h[g1] - soff_h[g0], dims, soff, len(counts), g0, g1, topk, merge, **coords)
            vals = ctx.decode_flash_values(pidx[t0 * 128: t1 * 128], dims, tile_group[t0:t1], **coords)
        vals = all_gather_ranges(vals, [(b - a) * 128 for a, b, _, _ in parts], self.group)
        return vals, _tile_queries(counts, t0, t1)

    @torch.no_grad()
    def __call__(self, latents, geo_decoder, bounds=1.01, num_chunks=10000, mc_level=0.0, octree_resolution=None,
                 min_resolution=63, mini_grid_num=4, enable_pbar=True, **kwargs):
        dev = latents.device
        self._tick(None, dev)
        ctx = bind(latents, geo_decoder)
        levels = flash_levels(octree_resolution, min_resolution, mini_grid_num)
        b6 = normalize_bounds(bounds)
        bbox_min, bbox_size = b6[:3], b6[3:] - b6[:3]
        bmin32 = bbox_min.astype(np.float32)
        merge = self.topk_mode == 'merge'
        rank, world = dist.get_rank(self.group), dist.get_world_size(self.group)
        sharded_last = self.keep_sharded and len(levels) > 1 and levels[-1] + 1 >= MC_HALO * world
        T = flash_topk_budget(latents.shape[1])
        outs, plane0s, owns = [], [], []
        self.last_stats = []
        for b in range(latents.shape[0]):
            ctx.prepare_kv(latents[b])
            self._tick("kv_prepare (replicated)", dev)
            # ---- level 0: mini-grids; sizes known on the host (level 0 is 'mean' in both modes, as in FlashVDMVolumeDecoding)
            N0 = levels[0] + 1
            layout = ctx.flash_layout_minigrids(N0, mini_grid_num, 100)
            counts, soff_h = flash_minigrid_sizes(N0, mini_grid_num, 100)
            self._tick("level0 layout (replicated)", dev)
            vals, mine0 = self._level(ctx, (N0, N0, N0), layout, soff_h, counts, T, False, dict(axes=axis_tables(bounds, levels[0])))
            grid = torch.empty((N0, N0, N0), dtype=torch.float32, device=dev)
            ctx.scatter(layout[0][: vals.numel()], vals, grid)
            self._tick("level0 select + decode + all_gather + scatter", dev)
            queries, mine = [N0 ** 3], [mine0]
            # ---- refined levels: 6^3 spatial bins of the active queries
            for r in levels[1:]:
                n = r + 1
                last = r == levels[-1]
                index = refine_level(ctx, grid, mc_level, last=last, nf=n)
                self._tick(f"refine -> {n}^3 (replicated)", dev)
                cell = (bbox_size / r).astype(np.float32)
                nq = int(index.numel())
                queries.append(nq)
                if nq:                  # nq is the same on every rank: an empty level is skipped by all alike
                    *layout, counts_d = ctx.flash_layout_bins(index, (n, n, n), cell, bmin32, 30 if merge else 50, with_counts=True)
                    meta = torch.cat([counts_d, layout[3]]).tolist()          # one small read-back: 216 counts + 217 offsets
                    self._tick(f"level {n}^3 layout + count read-back (replicated)", dev)
                    vals, m = self._level(ctx, (n, n, n), layout, meta[216:], meta[:216], T, merge, dict(cell=cell, bmin=bmin32))
                    self._tick(f"level {n}^3 select + decode + all_gather", dev)
                mine.append(m if nq else 0)
                if last and sharded_last:
                    planes, _, _ = plane_cuts(index, n, world)
                    plane0, own = planes[rank], planes[rank + 1] - planes[rank]
                    slab = torch.empty((min(planes[rank + 1] + MC_HALO, n) - plane0, n, n), dtype=torch.float32, device=dev)
                    ctx.fill(slab, NAN)
                    if nq:
                        ctx.scatter_window(layout[0][: vals.numel()], vals, slab, plane0 * n * n)
                    grid = slab
                    plane0s.append(plane0); owns.append(own)
                    self._tick("last level scatter (own slab)", dev)
                    break
                nxt = torch.empty((n, n, n), dtype=torch.float32, device=dev)
                ctx.fill(nxt, NAN if last else SENTINEL)
                if nq:
                    ctx.scatter(layout[0][: vals.numel()], vals, nxt)
                grid = nxt
                self._tick(f"level {n}^3 scatter", dev)
            outs.append(grid)
            self.last_stats.append({"levels": levels, "queries": queries, "rank_queries": mine})
        if sharded_last:
            N = levels[-1] + 1
            return SlabGrid(outs, plane0s, owns, (N, N, N), True, self.group, latents.dtype)
        return torch.stack(outs, 0).to(latents.dtype)


def vanilla_latents2mesh_sharded(latents, geo_decoder, surface_extractor=None, group=None, bounds=1.01, mc_level=0.0,
                                 octree_resolution=None, **kwargs):
    """VanillaVolumeDecoder + MCSurfaceExtractor with the grid left in place (BASELINE config 5): every rank decodes
    its slab, marching cubes runs per slab behind a two-plane halo exchange, rank 0 receives the mesh pieces.
    Returns ``list[Latent2MeshOutput | None]`` on rank 0 (the reference's per-item error convention) and None elsewhere."""
    from .surface_extractors import MCSurfaceExtractor
    ext = surface_extractor if surface_extractor is not None else MCSurfaceExtractor()
    kw = dict(bounds=bounds, mc_level=mc_level, octree_resolution=octree_resolution, **kwargs)
    grid = ShardedVanillaVolumeDecoder(group, keep_sharded=True)(latents, geo_decoder, **kw)
    outs = ext(grid, **kw)
    return outs if dist.get_rank(group) == 0 else None


def latents2mesh_data_parallel(vae, latents, group=None, dst: int = 0, **kwargs):
    """Batched latents, whole meshes per GPU (BASELINE config 4): item b of ``latents`` [B, M, C] is decoded by
    rank ``b % world`` with ``vae.latents2mesh`` (any volume decoder, FlashVDM included — it is batch-1 per call in
    the reference too, volume_decoders.py:361); the ``Latent2MeshOutput`` objects are gathered on ``dst`` in batch
    order (``None`` elsewhere).  No data-path collective: only the final object gather."""
    rank, world = dist.get_rank(group), dist.get_world_size(group)
    B = latents.shape[0]
    mine = {}
    for b in range(rank, B, world):
        mine[b] = vae.latents2mesh(latents[b:b + 1], **kwargs)[0]
    gathered = [None] * world if rank == dst else None
    dist.gather_object(mine, gathered, dst=dst, group=group)
    if rank != dst:
        return None
    out = [None] * B
    for part in gathered:
        for b, o in part.items():
            out[b] = o
    return out
