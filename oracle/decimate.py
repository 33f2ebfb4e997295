"""ORACLE (test infrastructure, never shipped): numpy statement of the third mesh filter of the reference's
``hy3dgen/shapegen/postprocessors.py``, ``FaceReducer``, that ``hy3dgeo.FaceReducer`` / ``hy3d_mesh_decimate`` implement on
the GPU bit for bit.

PARITY UNPINNED: the reference runs pymeshlab's ``meshing_decimation_quadric_edge_collapse(targetfacenum=max_facenum,
qualitythr=1.0, preserveboundary=True, boundaryweight=3, preservenormal=True, preservetopology=True, autoclean=True)``,
vcglib's sequential heap-ordered collapse, which is not available here.  What follows is the project's own statement of
what those parameters intend, in rounds of independent collapses that a GPU runs deterministically.

Input V float32 [nV, 3], F int32 [nF, 3], target T >= 1.  If nF <= T the mesh is returned as given.  Otherwise, in rounds,
each starting from the compacted mesh of the previous one:
  1. frozen vertices (never moved, never removed): on an edge with one face or with three or more; incident faces not one
     closed fan; in a face with a repeated id; a non-finite coordinate.
  2. quadrics, once, on the input: per face n = (p1-p0) x (p2-p0) in float64; a face whose three vertices are finite and
     0 < |n| < inf contributes the plane quadric of n/|n|, d = -n.p0 / |n|; a vertex sums its faces in ascending face id.
  3. candidates: edge (a, b), a < b, numbered in (a, b) order, with exactly two faces (a, b, c) and (b, a, d); a, b not
     frozen; common neighbours exactly {c, d}; deg(a) + deg(b) - 4 >= 3, deg(c) >= 4, deg(d) >= 4.
  4. position: Cramer's minimiser of Q = Qa + Qb when |det A| >= 1e-12, pa, pb, the midpoint: the cheapest, ties to that
     order; rounded to float32, and everything below uses the rounded position.
  5. validity and cost: every other face of the two stars with a, b replaced by p must keep n_old . n_new > 0 (so a NaN
     product is invalid too); quality |n| / (longest edge)^2; cost = max(pQp, 1e-15) / min(qmin, 1.0).
  6. ranking by (cost, edge id); m1[v] = smallest rank of a valid edge at v, m2[v] = min of m1 over v and its neighbours; an
     edge is selected iff its rank equals m2[a] and m2[b]; only the ceil((F - T) / 2) lowest-ranked selected edges apply.
  7. apply: a takes p and Qa + Qb, b becomes a, the edge's two faces go; vertices and faces are compacted in order.
  8. stop when F <= T or when a round applies nothing (that round's compaction is kept; ``rounds`` does not count it).

Float64 arithmetic is written out operation by operation (no np.dot / @ / einsum); the kernels use the same order.
"""
from __future__ import annotations

import numpy as np

QUALITYTHR = 1.0
DET_MIN = 1e-12
COST_MIN = 1e-15


def _cross(ux, uy, uz, wx, wy, wz):
    return uy * wz - uz * wy, uz * wx - ux * wz, ux * wy - uy * wx


def _norm(x, y, z):
    return np.sqrt((x * x + y * y) + z * z)


def _tri_normal(p0, p1, p2):
    """(p1 - p0) x (p2 - p0) of float64 [K, 3] corner arrays, as three columns"""
    return _cross(p1[:, 0] - p0[:, 0], p1[:, 1] - p0[:, 1], p1[:, 2] - p0[:, 2],
                  p2[:, 0] - p0[:, 0], p2[:, 1] - p0[:, 1], p2[:, 2] - p0[:, 2])


def face_quadrics(v: np.ndarray, f: np.ndarray) -> np.ndarray:
    """[F, 10] (aa, ab, ac, ad, bb, bc, bd, cc, cd, dd) of each face's unit plane; zero where the face does not count."""
    p = v.astype(np.float64)
    p0, p1, p2 = p[f[:, 0]], p[f[:, 1]], p[f[:, 2]]
    nx, ny, nz = _tri_normal(p0, p1, p2)
    ln = _norm(nx, ny, nz)
    ok = np.isfinite(v).all(1)[f].all(1) & (ln > 0) & (ln < np.inf)
    safe = np.where(ok, ln, 1.0)
    a, b, c = nx / safe, ny / safe, nz / safe
    d = -((a * p0[:, 0] + b * p0[:, 1]) + c * p0[:, 2])
    q = np.stack([a * a, a * b, a * c, a * d, b * b, b * c, b * d, c * c, c * d, d * d], 1)
    q[~ok] = 0.0
    return q


def _csr(f: np.ndarray, n: int):
    """vertex -> incident face ids in ascending order: (start [n + 1], faces [3F], corner slot in the face [3F])"""
    cv = f.reshape(-1).astype(np.int64)
    order = np.argsort(cv, kind="stable")
    return np.searchsorted(cv[order], np.arange(n + 1)), (order // 3).astype(np.int64), (order % 3).astype(np.int64)


def vertex_quadrics(v: np.ndarray, f: np.ndarray) -> np.ndarray:
    fq = face_quadrics(v, f)
    start, cf, _ = _csr(f, len(v))
    Q = np.zeros((len(v), 10), np.float64)
    cnt = np.diff(start)
    for k in range(int(cnt.max()) if len(cnt) else 0):       # ascending face id, one addition per step
        has = np.nonzero(cnt > k)[0]
        Q[has] = Q[has] + fq[cf[start[has] + k]]
    return Q


def _det3(m00, m01, m02, m10, m11, m12, m20, m21, m22):
    return (m00 * (m11 * m22 - m12 * m21) - m01 * (m10 * m22 - m12 * m20)) + m02 * (m10 * m21 - m11 * m20)


def _energy(q, x, y, z):
    t0 = ((q[:, 0] * x + q[:, 1] * y) + q[:, 2] * z) + q[:, 3]
    t1 = ((q[:, 1] * x + q[:, 4] * y) + q[:, 5] * z) + q[:, 6]
    t2 = ((q[:, 2] * x + q[:, 5] * y) + q[:, 7] * z) + q[:, 8]
    t3 = ((q[:, 3] * x + q[:, 6] * y) + q[:, 8] * z) + q[:, 9]
    return ((x * t0 + y * t1) + z * t2) + t3


def _position(q, pa, pb):
    """float32 [K, 3] collapse positions: the cheapest of (minimiser, pa, pb, midpoint), ties to that order"""
    det = _det3(q[:, 0], q[:, 1], q[:, 2], q[:, 1], q[:, 4], q[:, 5], q[:, 2], q[:, 5], q[:, 7])
    has = np.abs(det) >= DET_MIN
    sd = np.where(has, det, 1.0)
    bx, by, bz = -q[:, 3], -q[:, 6], -q[:, 8]
    ox = _det3(bx, q[:, 1], q[:, 2], by, q[:, 4], q[:, 5], bz, q[:, 5], q[:, 7]) / sd
    oy = _det3(q[:, 0], bx, q[:, 2], q[:, 1], by, q[:, 5], q[:, 2], bz, q[:, 7]) / sd
    oz = _det3(q[:, 0], q[:, 1], bx, q[:, 1], q[:, 4], by, q[:, 2], q[:, 5], bz) / sd
    a, b = pa.astype(np.float64), pb.astype(np.float64)
    mid = (a + b) * 0.5
    best = a.copy()
    cost = _energy(q, a[:, 0], a[:, 1], a[:, 2])
    for c in (b, mid):
        e = _energy(q, c[:, 0], c[:, 1], c[:, 2])
        take = e < cost
        best[take], cost[take] = c[take], e[take]
    e = _energy(q, ox, oy, oz)
    take = has & (e <= cost)                                 # the minimiser comes first: it wins ties
    best[take] = np.stack([ox, oy, oz], 1)[take]
    return best.astype(np.float32)


def _compact(v, Q, f, keep_f):
    f = f[keep_f]
    ref = np.zeros(len(v), dtype=bool)
    ref[f.reshape(-1)] = True
    remap = np.cumsum(ref) - 1
    return (np.ascontiguousarray(v[ref]), Q[ref], np.ascontiguousarray(remap[f].astype(np.int32).reshape(-1, 3)),
            np.nonzero(keep_f)[0])


def frozen_vertices(v, f, start, cf, cs, elo, ehi, ecnt):
    """bool [nV]: the vertices no collapse may move or remove (contract step 1)"""
    n = len(v)
    frozen = ~np.isfinite(v).all(1)
    rep = (f[:, 0] == f[:, 1]) | (f[:, 1] == f[:, 2]) | (f[:, 0] == f[:, 2])
    frozen[f[rep].reshape(-1)] = True
    bad = ecnt != 2
    frozen[elo[bad]] = True
    frozen[ehi[bad]] = True
    # one closed fan: the link edges x -> y of the faces (v, x, y) at v form a single cycle through all of them
    cnt = np.diff(start)
    frozen |= cnt == 0
    cv = np.repeat(np.arange(n, dtype=np.int64), cnt)
    src = f[cf, (cs + 1) % 3].astype(np.int64)
    tgt = f[cf, (cs + 2) % 3].astype(np.int64)
    ks, kt = cv * n + src, cv * n + tgt
    ok = np.ones(n, bool)
    for k in (ks, kt):
        s = np.sort(k)
        dup = s[1:] == s[:-1]
        ok[(s[1:][dup] // n)] = False
    order = np.argsort(ks, kind="stable")
    sks = ks[order]
    pos = np.minimum(np.searchsorted(sks, kt), len(sks) - 1) if len(sks) else np.zeros(0, np.int64)
    found = sks[pos] == kt if len(sks) else np.zeros(0, bool)
    ok[cv[~found]] = False
    succ = order[pos]
    good = ok[cv]
    # cycles of the successor permutation (pointer doubling): the smallest corner index on each corner's cycle
    lab = np.arange(len(cv))
    jump = np.where(good, succ, lab)
    for _ in range(int(np.ceil(np.log2(max(int(cnt.max()) if len(cnt) else 1, 1)))) + 1):
        lab = np.minimum(lab, lab[jump])
        jump = jump[jump]
    ncyc = np.bincount(cv[good & (lab == np.arange(len(cv)))], minlength=n)
    ok &= ncyc == 1
    frozen |= ~ok
    return frozen


def one_round(v, Q, f, T):
    """-> (v, Q, f, kept face ids of the input, collapses applied)"""
    n, m = len(v), len(f)
    start, cf, cs = _csr(f, n)
    a3 = f.reshape(-1).astype(np.int64)
    b3 = f[:, [1, 2, 0]].reshape(-1).astype(np.int64)
    nd = a3 != b3
    key = np.minimum(a3, b3) * (1 << 32) + np.maximum(a3, b3)
    hf = np.repeat(np.arange(m, dtype=np.int64), 3)
    key, hf = key[nd], hf[nd]
    order = np.argsort(key, kind="stable")
    skey, sface = key[order], hf[order]
    ukey, first, ecnt = np.unique(skey, return_index=True, return_counts=True)
    elo, ehi = ukey >> 32, ukey & 0xffffffff
    deg = np.bincount(elo, minlength=n) + np.bincount(ehi, minlength=n)
    frozen = frozen_vertices(v, f, start, cf, cs, elo, ehi, ecnt)

    # candidates (step 3)
    E = len(ukey)
    cand = np.nonzero((ecnt == 2) & ~frozen[elo] & ~frozen[ehi])[0]
    a, b = elo[cand], ehi[cand]
    f1, f2 = sface[first[cand]], sface[first[cand] + 1]

    def directed(t):                                          # face t holds a -> b
        g = f[t].astype(np.int64)
        return (((g[:, 0] == a) & (g[:, 1] == b)) | ((g[:, 1] == a) & (g[:, 2] == b)) | ((g[:, 2] == a) & (g[:, 0] == b)))

    d1, d2 = directed(f1), directed(f2)
    fab = np.where(d1, f1, f2)
    fba = np.where(d1, f2, f1)
    c = f[fab].astype(np.int64).sum(1) - a - b
    d = f[fba].astype(np.int64).sum(1) - a - b
    ok = (d1 != d2) & (c != d) & (deg[a] + deg[b] - 4 >= 3) & (deg[c] >= 4) & (deg[d] >= 4)
    # link condition: a's neighbours that are also b's neighbours must be exactly {c, d}
    nb_src = np.concatenate([elo, ehi])
    nb_dst = np.concatenate([ehi, elo])
    no = np.argsort(nb_src, kind="stable")
    nstart = np.searchsorted(nb_src[no], np.arange(n + 1))
    ndst = nb_dst[no]
    cnt_a = nstart[a + 1] - nstart[a]
    ci = np.repeat(np.arange(len(cand)), cnt_a)
    w = ndst[np.repeat(nstart[a], cnt_a) + (np.arange(int(cnt_a.sum())) - np.repeat(np.cumsum(cnt_a) - cnt_a, cnt_a))]
    bb = b[ci]
    k2 = np.minimum(bb, w) * (1 << 32) + np.maximum(bb, w)
    p = np.minimum(np.searchsorted(ukey, k2), max(E - 1, 0))
    common = np.bincount(ci[ukey[p] == k2], minlength=len(cand)) if E else np.zeros(len(cand), np.int64)
    ok &= common == 2
    sel = np.nonzero(ok)[0]
    cand, a, b, f1, f2 = cand[sel], a[sel], b[sel], f1[sel], f2[sel]
    K = len(cand)

    # position, validity and cost (steps 4, 5)
    q = Q[a] + Q[b]
    pos = _position(q, v[a], v[b])
    sa, sb = start[a + 1] - start[a], start[b + 1] - start[b]
    idx, owner = [], []
    for s0, cntk in ((start[a], sa), (start[b], sb)):
        off = np.arange(int(cntk.sum())) - np.repeat(np.cumsum(cntk) - cntk, cntk)
        idx.append(cf[np.repeat(s0, cntk) + off])
        owner.append(np.repeat(np.arange(K), cntk))
    t = np.concatenate(idx)
    o = np.concatenate(owner)
    srt = np.argsort(o, kind="stable")
    t, o = t[srt], o[srt]
    keep = (t != f1[o]) & (t != f2[o])
    t, o = t[keep], o[keep]
    P = v.astype(np.float64)
    g = f[t]
    old = [P[g[:, i]] for i in range(3)]
    pn = pos[o].astype(np.float64)
    new = [np.where(((g[:, i] == a[o]) | (g[:, i] == b[o]))[:, None], pn, old[i]) for i in range(3)]
    nox, noy, noz = _tri_normal(*old)
    nnx, nny, nnz = _tri_normal(*new)
    dot = (nox * nnx + noy * nny) + noz * nnz
    l2 = []
    for i in range(3):
        u, w3 = new[i], new[(i + 1) % 3]
        dx, dy, dz = w3[:, 0] - u[:, 0], w3[:, 1] - u[:, 1], w3[:, 2] - u[:, 2]
        l2.append((dx * dx + dy * dy) + dz * dz)
    qual = _norm(nnx, nny, nnz) / np.maximum(np.maximum(l2[0], l2[1]), l2[2])
    valid = np.ones(K, bool)
    valid[o[~(dot > 0)]] = False
    qmin = np.full(K, np.inf)
    np.minimum.at(qmin, o, qual)
    pd = pos.astype(np.float64)
    e = _energy(q, pd[:, 0], pd[:, 1], pd[:, 2])
    cost = np.where(e > COST_MIN, e, COST_MIN) / np.minimum(qmin, QUALITYTHR)

    vs = np.nonzero(valid)[0]
    if len(vs) == 0:
        vo, Qo, fo, kept = _compact(v, Q, f, np.ones(m, bool))
        return vo, Qo, fo, kept, 0
    # ranking and selection (step 6)
    order = np.lexsort((cand[vs], cost[vs]))
    rank = np.empty(len(vs), np.int64)
    rank[order] = np.arange(len(vs))
    BIG = np.iinfo(np.int64).max
    m1 = np.full(n, BIG)
    np.minimum.at(m1, a[vs], rank)
    np.minimum.at(m1, b[vs], rank)
    m2 = m1.copy()
    np.minimum.at(m2, elo, m1[ehi])
    np.minimum.at(m2, ehi, m1[elo])
    chosen = np.nonzero((rank == m2[a[vs]]) & (rank == m2[b[vs]]))[0]
    chosen = chosen[np.argsort(rank[chosen])][: (m - T + 1) // 2]
    ch = vs[chosen]
    # apply (step 7)
    v = v.copy()
    Q = Q.copy()
    v[a[ch]] = pos[ch]
    Q[a[ch]] = q[ch]
    redirect = np.arange(n)
    redirect[b[ch]] = a[ch]
    keep_f = np.ones(m, bool)
    keep_f[f1[ch]] = False
    keep_f[f2[ch]] = False
    vo, Qo, fo, kept = _compact(v, Q, redirect[f].astype(np.int32), keep_f)
    return vo, Qo, fo, kept, len(ch)


def decimate(v: np.ndarray, f: np.ndarray, max_faces: int, trace: list | None = None):
    """FaceReducer -> (vertices float32, faces int32, rounds).  ``trace``, if a list, receives (v, f, kept) per round: the
    round's output and, for each of its faces, the id of the face it came from in the round's input."""
    v = np.ascontiguousarray(v, np.float32).reshape(-1, 3)
    f = np.ascontiguousarray(f, np.int32).reshape(-1, 3)
    T = int(max_faces)
    if T < 1:
        raise ValueError("max_faces < 1")
    if len(f) <= T:
        return v.copy(), f.copy(), 0
    if f.min() < 0 or f.max() >= len(v):
        raise ValueError(f"face index outside [0, {len(v)})")
    with np.errstate(divide="ignore", invalid="ignore"):     # degenerate faces of refused collapses
        Q = vertex_quadrics(v, f)
        return _rounds(v, Q, f, T, trace)


def _rounds(v, Q, f, T, trace):
    rounds = 0
    while len(f) > T:
        v, Q, f, kept, applied = one_round(v, Q, f, T)
        if trace is not None:
            trace.append((v, f, kept))
        if not applied:
            break
        rounds += 1
    return v, f, rounds
