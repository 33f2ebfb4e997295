"""The ownership rule of dual marching cubes over a grid cut into slabs along axis 0 (``hy3d_dmc_count_slab`` /
``hy3d_dmc_emit_slab``), stated on CPU against ``oracle/dmc.py``.  A slab owning planes [x0, x1) of N0 holds the vertices
of the cubes based at [x0, x1) and the faces of the edges in planes [x0 + 1, x1 + 1) (from 0 on the first slab, to N0 on
the last).  Then every piece is a contiguous range of the whole mesh, its faces reference only the cube planes [x0, x1],
and it is what the oracle gives on the slab plus a two-plane halo of the next slab, with ids shifted by the vertices of
the earlier slabs: no lower halo is read."""
import numpy as np
import pytest

from oracle import dmc as OD


def noise(shape, seed):
    """Normal noise with exact zeros (outside) and NaNs (outside, NaN vertices on their rim)."""
    rng = np.random.default_rng(seed)
    g = rng.standard_normal(shape).astype(np.float32)
    g[rng.random(shape) < 0.15] = 0.0
    g[rng.random(shape) < 0.05] = np.nan
    return g


def plane_counts(g):
    """(vertices per cube plane [N0 - 1], faces per edge plane [N0]) of the oracle's mesh of g."""
    n0, n1, n2 = g.shape
    inside = g > 0
    case = np.zeros((n0 - 1, n1 - 1, n2 - 1), dtype=np.int32)
    for m, (x, y, z) in enumerate(OD.CORNERS):
        case |= inside[z:z + n0 - 1, y:y + n1 - 1, x:x + n2 - 1].astype(np.int32) << m
    cnt, _ = OD.patch_tables()
    vp = cnt[case].astype(np.int64).sum((1, 2))
    fp = np.zeros(n0, dtype=np.int64)
    for axis in range(3):
        lo, hi = [slice(None)] * 3, [slice(None)] * 3
        lo[axis], hi[axis] = slice(0, g.shape[axis] - 1), slice(1, None)
        P = np.stack(np.nonzero(inside[tuple(lo)] != inside[tuple(hi)]), 1)
        u, v = (axis + 1) % 3, (axis + 2) % 3
        P = P[(P[:, u] >= 1) & (P[:, u] <= g.shape[u] - 2) & (P[:, v] >= 1) & (P[:, v] <= g.shape[v] - 2)]
        np.add.at(fp, P[:, 0], 2)
    return vp, fp


def slab_ranges(x0, x1, n0):
    """(cube planes, edge planes) a slab owning [x0, x1) of n0 planes emits."""
    return (x0, min(x1, n0 - 1)), (0 if x0 == 0 else x0 + 1, min(x1 + 1, n0))


SHAPES = [(9, 7, 11), (6, 5, 40), (12, 4, 4), (5, 9, 33), (2, 6, 6), (3, 3, 3)]


@pytest.mark.parametrize("shape", SHAPES)
def test_slab_pieces_are_contiguous_ranges_of_the_oracle_mesh(shape):
    g = noise(shape, sum(shape))
    v, f = OD.dual_marching_cubes_raw(g)
    vp, fp = plane_counts(g)
    n0 = shape[0]
    assert vp.sum() == len(v) and fp.sum() == len(f)
    vcum, fcum = np.concatenate([[0], np.cumsum(vp)]), np.concatenate([[0], np.cumsum(fp)])
    for x0 in range(n0):
        for x1 in range(x0 + 1, n0 + 1):
            (c0, c1), (e0, e1) = slab_ranges(x0, x1, n0)
            base, V = vcum[c0], vcum[c1] - vcum[c0]
            vx1 = vp[x1] if x1 < n0 - 1 else 0                    # vertices of the halo cube plane x1
            piece = f[fcum[e0]: fcum[e1]]
            assert piece.size == 0 or (piece.min() >= base and piece.max() < base + V + vx1), (x0, x1)
            # the slab's piece is the oracle mesh of the slab + two halo planes, restricted to its planes, ids shifted
            hi = min(x1 + 2, n0)
            if hi - x0 < 2:
                assert V == 0 and piece.size == 0
                continue
            sub = g[x0:hi]
            svp, sfp = plane_counts(sub)
            assert svp[: x1 - x0].sum() == V and np.array_equal(svp[: c1 - c0], vp[c0:c1])
            if not (svp.sum() or sfp.sum()):
                assert piece.size == 0
                continue
            try:
                sv, sf = OD.dual_marching_cubes_raw(sub)
            except RuntimeError:                                   # no vertex in the slab at all
                assert V == 0 and piece.size == 0
                continue
            scum = np.concatenate([[0], np.cumsum(sfp)])
            lf = sf[scum[e0 - x0]: scum[e1 - x0]]
            assert np.array_equal(lf + base, piece), (x0, x1)
            sv = sv[: V].copy()
            sv[:, 0] += x0
            assert np.allclose(sv, v[base: base + V], atol=1e-9, equal_nan=True)


@pytest.mark.parametrize("shape", SHAPES[:4])
def test_slab_pieces_concatenate_to_the_oracle_mesh(shape):
    """Cut at every plane 1 .. N0 - 1 and at uneven multi-way cuts: the pieces in slab order are the whole mesh."""
    g = noise(shape, 7 * sum(shape))
    v, f = OD.dual_marching_cubes_raw(g)
    vp, fp = plane_counts(g)
    n0 = shape[0]
    vcum, fcum = np.concatenate([[0], np.cumsum(vp)]), np.concatenate([[0], np.cumsum(fp)])
    rng = np.random.default_rng(0)
    cuts = [[0, c, n0] for c in range(1, n0)]
    cuts += [[0] + sorted(rng.choice(np.arange(1, n0), size=min(k, n0 - 1), replace=False).tolist()) + [n0] for k in (2, 3, 5)]
    for planes in cuts:
        vs, fs = [], []
        for x0, x1 in zip(planes, planes[1:]):
            (c0, c1), (e0, e1) = slab_ranges(x0, x1, n0)
            vs.append(v[vcum[c0]: vcum[c1]])
            fs.append(f[fcum[e0]: fcum[e1]])
        assert np.array_equal(np.concatenate(vs), v, equal_nan=True) and np.array_equal(np.concatenate(fs), f), planes
