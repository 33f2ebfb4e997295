"""ORACLE (test infrastructure): dual marching cubes in numpy, the contract of ``DMCSurfaceExtractor`` and
``hy3d_dmc_count`` / ``hy3d_dmc_emit`` (DESIGN.md §2).  PARITY UNPINNED against ``diso.DiffDMC`` (absent here): this is
the project's own statement of the dual surface, not a transcription of diso.

Contract
  * inside iff g > 0 (NaN => outside);
  * one vertex per (cube, patch).  A patch is one connected piece of the cube's iso-surface: crossing edges sharing a
    cube face are joined by that face's iso-segment; on an ambiguous face (diagonal corners inside) the inside corners are
    separated, i.e. the two edges at each inside corner are joined.  Patches are numbered by their smallest edge id.
    The patches are derived here at run time, NOT read from csrc/dmc_tables.inc, so a parity test checks that table;
  * vertex = mean of the crossings of the patch's edges; crossing on an edge from its lower corner a to its upper corner b
    at a + t, t = g_a / (g_a - g_b), all in float64: summed in ascending edge id, divided by the edge count, divided by
    (n_axis - 1) per axis, rounded once to float32; then the fp32 centring v - 0.5f * (lo + hi) with lo / hi the per-axis
    min / max over the non-NaN vertices;
  * one quad per grid edge with a sign change whose four incident cubes lie inside the grid, through the patch vertex of
    each of those cubes that contains the edge, split along its first diagonal into two triangles, oriented like the
    marching-cubes table of csrc/mc_tables.inc;
  * vertices in lexicographic (cube, patch) order, faces in lexicographic (edge owner voxel, edge axis) order."""
from __future__ import annotations

import numpy as np

# corner m: offsets (dx, dy, dz) with x = array axis 2, y = axis 1, z = axis 0 (SURVEY App. D)
CORNERS = [(0, 0, 0), (1, 0, 0), (1, 1, 0), (0, 1, 0), (0, 0, 1), (1, 0, 1), (1, 1, 1), (0, 1, 1)]
EDGES = [(0, 1), (1, 2), (2, 3), (3, 0), (4, 5), (5, 6), (6, 7), (7, 4), (0, 4), (1, 5), (2, 6), (3, 7)]


def _edge_geometry():
    """per edge: (lower corner, upper corner, lower-corner offset in array axes (o0, o1, o2), array axis)"""
    out = []
    for a, b in EDGES:
        lo, hi = (a, b) if sum(CORNERS[a]) < sum(CORNERS[b]) else (b, a)
        x, y, z = CORNERS[lo]
        d = [abs(p - q) for p, q in zip(CORNERS[a], CORNERS[b])].index(1)
        out.append((lo, hi, (z, y, x), 2 - d))
    return out


EDGE_GEOM = _edge_geometry()
EDGE_AT = {(g[2], g[3]): e for e, g in enumerate(EDGE_GEOM)}          # (offset, axis) -> cube edge id


def case_patches(case: int):
    """Patch index of each of the 12 edges (-1: no crossing) of sign configuration `case`."""
    ins = [(case >> m) & 1 for m in range(8)]
    cross = [e for e, (a, b) in enumerate(EDGES) if ins[a] != ins[b]]
    parent = list(range(12))

    def find(e):
        while parent[e] != e:
            e = parent[e]
        return e

    def join(e, f):
        parent[find(e)] = find(f)
    for axis in range(3):
        for side in (0, 1):
            face = [m for m in range(8) if CORNERS[m][axis] == side]
            fe = [e for e in cross if EDGES[e][0] in face and EDGES[e][1] in face]
            if len(fe) == 2:
                join(fe[0], fe[1])
            elif len(fe) == 4:                             # ambiguous face: separate the inside corners
                for m in face:
                    if ins[m]:
                        at = [e for e in fe if m in EDGES[e]]
                        join(at[0], at[1])
    roots = sorted({find(e) for e in cross}, key=lambda r: min(e for e in cross if find(e) == r))
    patch = [-1] * 12
    for e in cross:
        patch[e] = roots.index(find(e))
    return patch


def patch_tables():
    """(count[256], edge_patch[256, 12]) int8 — what tools/gen_mc_tables.py writes to csrc/dmc_tables.inc."""
    ep = np.array([case_patches(c) for c in range(256)], dtype=np.int8)
    return (ep.max(axis=1) + 1).astype(np.int8), ep


def dual_marching_cubes_raw(grid: np.ndarray):
    """-> (verts float64 [V,3] in index units, faces int32 [F,3]) before normalisation and centring."""
    g = np.ascontiguousarray(grid, dtype=np.float32)
    if g.ndim != 3:
        raise ValueError("Input volume should be a 3D array.")
    n0, n1, n2 = g.shape
    if min(g.shape) < 2:
        raise ValueError("dual marching cubes needs at least 2 samples per axis")
    inside = g > 0
    cnt_tab, ep_tab = patch_tables()
    case = np.zeros((n0 - 1, n1 - 1, n2 - 1), dtype=np.int32)
    for m, (x, y, z) in enumerate(CORNERS):
        case |= inside[z:z + n0 - 1, y:y + n1 - 1, x:x + n2 - 1].astype(np.int32) << m
    npatch = cnt_tab[case].astype(np.int64)
    vbase = np.concatenate([[0], np.cumsum(npatch.ravel())[:-1]]).reshape(case.shape)
    V = int(npatch.sum())
    if V == 0:
        raise RuntimeError("No surface found at the given iso value.")

    # vertices: lexicographic (cube, patch)
    act = np.flatnonzero(npatch.ravel())
    ci, cj, ck = np.unravel_index(act, case.shape)
    cs = case.ravel()[act]
    g64 = g.astype(np.float64)
    verts = np.empty((V, 3), dtype=np.float64)
    for p in range(int(npatch.max())):
        sel = npatch.ravel()[act] > p
        i, j, k, c = ci[sel], cj[sel], ck[sel], cs[sel]
        acc = np.zeros((len(c), 3))
        cnt = np.zeros(len(c))
        for e, (lo, hi, off, axis) in enumerate(EDGE_GEOM):
            m = ep_tab[c, e] == p
            if not m.any():
                continue
            a = np.stack([i + off[0], j + off[1], k + off[2]], 1)
            b = a.copy()
            b[:, axis] += 1
            ga, gb = g64[a[:, 0], a[:, 1], a[:, 2]], g64[b[:, 0], b[:, 1], b[:, 2]]
            with np.errstate(invalid="ignore", divide="ignore"):
                t = ga / (ga - gb)
            pt = a.astype(np.float64)
            pt[:, axis] = pt[:, axis] + t
            acc[m] = acc[m] + pt[m]
            cnt[m] += 1
        verts[vbase.ravel()[act[sel]] + p] = acc / cnt[:, None]

    # faces: one quad per interior sign-change edge, lexicographic (owner voxel, axis)
    keys, quads = [], []
    for axis in range(3):
        u, v = (axis + 1) % 3, (axis + 2) % 3
        lo = [slice(None)] * 3
        hi = [slice(None)] * 3
        lo[axis], hi[axis] = slice(0, g.shape[axis] - 1), slice(1, None)
        flip = inside[tuple(lo)] != inside[tuple(hi)]
        pi, pj, pk = np.nonzero(flip)
        P = np.stack([pi, pj, pk], 1)
        ok = (P[:, u] >= 1) & (P[:, u] <= g.shape[u] - 2) & (P[:, v] >= 1) & (P[:, v] <= g.shape[v] - 2)
        P = P[ok]
        ids = []
        for du, dv in ((0, 0), (1, 0), (1, 1), (0, 1)):          # counter-clockwise around +axis
            B = P.copy()
            B[:, u] -= du
            B[:, v] -= dv
            off = [0, 0, 0]
            off[u], off[v] = du, dv
            e = EDGE_AT[(tuple(off), axis)]
            c = case[B[:, 0], B[:, 1], B[:, 2]]
            ids.append(vbase[B[:, 0], B[:, 1], B[:, 2]] + ep_tab[c, e])
        q = np.stack(ids, 1)
        lower_in = inside[P[:, 0], P[:, 1], P[:, 2]]
        q = np.where(lower_in[:, None], q[:, ::-1], q)           # same orientation as the marching-cubes table
        keys.append((np.ravel_multi_index(P.T, g.shape).astype(np.int64) * 3 + axis) if len(P) else np.zeros(0, np.int64))
        quads.append(q.reshape(-1, 4))
    keys, quads = np.concatenate(keys), np.concatenate(quads)
    quads = quads[np.argsort(keys, kind="stable")]
    faces = np.stack([quads[:, [0, 1, 2]], quads[:, [0, 2, 3]]], 1).reshape(-1, 3).astype(np.int32)
    return verts, faces


def dual_marching_cubes(grid: np.ndarray):
    """-> (verts float32 [V,3], faces int32 [F,3]): normalised to the unit cube and centred on the bounding box."""
    verts, faces = dual_marching_cubes_raw(grid)
    n = np.array(np.shape(grid), dtype=np.float64) - 1.0
    v = (verts / n).astype(np.float32)
    with np.errstate(invalid="ignore"):
        lo, hi = np.nanmin(v, axis=0), np.nanmax(v, axis=0)
    c = np.float32(0.5) * (lo + hi)
    return (v - c).astype(np.float32), faces


def dmc_surface_extract(grid_logit: np.ndarray, **kwargs):
    """``DMCSurfaceExtractor.run`` on the host: ``mc_level`` and ``bounds`` play no part (as in the reference)."""
    return dual_marching_cubes(grid_logit)
