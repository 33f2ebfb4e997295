#!/usr/bin/env python3
"""Generate the 256-case marching-cubes triangle table used by the CUDA emit kernel.

No table is copied from anywhere: it is *derived* here by tracing, for every
sign configuration, the oriented iso-contour loops on the six cube faces and
fan-triangulating each loop.  Ambiguous faces (diagonal corners inside) are
resolved by one fixed rule that depends only on the four corner signs of that
face — "inside corners are separated" — so the two cubes sharing a face always
agree and the extracted surface is watertight (the classic Lorensen table is
not).  skimage's Lewiner variant resolves those faces from the values instead;
see DESIGN.md "marching cubes: parity unpinned".  For that value-based choice
(the asymptotic decider, the opt-in `face_rule="asymptotic"`) the same tracing
runs once per combination of per-face choices: mc_tables_decider.inc.

Conventions (SURVEY Appendix D): cube corner m has offsets (dx,dy,dz) with
x = array axis 2 (fastest), y = axis 1, z = axis 0:
  v0(0,0,0) v1(1,0,0) v2(1,1,0) v3(0,1,0) v4(0,0,1) v5(1,0,1) v6(1,1,1) v7(0,1,1)
case bit m is set iff value(v_m) - level > 0.
Edge e joins CORNER pairs EDGES[e]; the edge is *owned* by its lower corner.

Output: hunyuan3d-2_b200/csrc/mc_tables.inc, dmc_tables.inc and
mc_tables_decider.inc (checked in; regenerate with
`python tools/gen_mc_tables.py [output directory]`).  The C oracles
(oracle/mc_oracle.c, and oracle/mc_face_rule.c for the face rules) do NOT read
these tables: they trace loops at run time, so a parity test between the two
checks the tables.
"""
import itertools
import os
import sys

CORNERS = [(0, 0, 0), (1, 0, 0), (1, 1, 0), (0, 1, 0), (0, 0, 1), (1, 0, 1), (1, 1, 1), (0, 1, 1)]
EDGES = [(0, 1), (1, 2), (2, 3), (3, 0), (4, 5), (5, 6), (6, 7), (7, 4), (0, 4), (1, 5), (2, 6), (3, 7)]
EDGE_ID = {frozenset(e): i for i, e in enumerate(EDGES)}


def face_cycles():
    """Corner cycles of the 6 faces, counter-clockwise seen from outside the cube."""
    faces = []
    for axis in range(3):
        for side in (0, 1):
            cs = [i for i, c in enumerate(CORNERS) if c[axis] == side]
            # order the 4 corners around the face
            u, v = [a for a in range(3) if a != axis]
            cs.sort(key=lambda i: (CORNERS[i][u], CORNERS[i][v]))
            cyc = [cs[0], cs[2], cs[3], cs[1]]          # (0,0) (1,0) (1,1) (0,1) in (u,v)
            # Newell normal
            n = [0.0, 0.0, 0.0]
            for a, b in zip(cyc, cyc[1:] + cyc[:1]):
                pa, pb = CORNERS[a], CORNERS[b]
                n[0] += (pa[1] - pb[1]) * (pa[2] + pb[2])
                n[1] += (pa[2] - pb[2]) * (pa[0] + pb[0])
                n[2] += (pa[0] - pb[0]) * (pa[1] + pb[1])
            outward = 1 if side == 1 else -1
            if n[axis] * outward < 0:
                cyc = cyc[::-1]
            # canonical rotation: start at the smallest corner id
            k = cyc.index(min(cyc))
            faces.append(cyc[k:] + cyc[:k])
    return faces


FACES = face_cycles()


def face_segments(case, cyc, connect_inside=False):
    """Directed iso-segments (edge_from, edge_to) on one face; the inside region is
    on the left when seen from outside."""
    ins = [(case >> c) & 1 for c in cyc]
    e = [EDGE_ID[frozenset((cyc[m], cyc[(m + 1) % 4]))] for m in range(4)]
    io = [m for m in range(4) if ins[m] and not ins[(m + 1) % 4]]      # in -> out edges
    oi = [m for m in range(4) if not ins[m] and ins[(m + 1) % 4]]      # out -> in edges
    if len(io) == 0:
        return []
    if len(io) == 1:
        return [(e[io[0]], e[oi[0]])]
    segs = []
    for m in io:                       # corner cyc[m] is inside, cyc[m+1] outside
        if connect_inside:
            segs.append((e[m], e[(m + 1) % 4]))      # cut off the outside corner m+1
        else:
            segs.append((e[m], e[(m - 1) % 4]))      # cut off the inside corner m
    return segs


def trace_loops(case, connect=0):
    """Iso-contour loops of one cube.  Bit f of `connect` set: ambiguous face FACES[f] connects its inside corners."""
    nxt = {}
    for f, cyc in enumerate(FACES):
        for a, b in face_segments(case, cyc, bool((connect >> f) & 1)):
            assert a not in nxt
            nxt[a] = b
    loops, seen = [], set()
    for start in sorted(nxt):
        if start in seen:
            continue
        loop, e = [], start
        while e not in seen:
            seen.add(e)
            loop.append(e)
            e = nxt[e]
        assert e == start
        loops.append(loop)
    return loops


def triangles(case, flip, connect=0):
    tris = []
    for loop in trace_loops(case, connect):
        for m in range(1, len(loop) - 1):
            t = (loop[0], loop[m], loop[m + 1])
            tris.append((t[0], t[2], t[1]) if flip else t)
    return tris


def build(flip=True):
    return [triangles(c, flip) for c in range(256)]


def ambiguous_faces(case):
    """Indices into FACES of the faces whose inside corners are diagonal, ascending."""
    out = []
    for f, cyc in enumerate(FACES):
        ins = [(case >> c) & 1 for c in cyc]
        if ins[0] == ins[2] and ins[1] == ins[3] and ins[0] != ins[1]:
            out.append(f)
    return out


def decision_connect(case, dec):
    """Face mask for trace_loops from decision index `dec`: bit q of dec is the choice of the q-th ambiguous face."""
    return sum(1 << f for q, f in enumerate(ambiguous_faces(case)) if (dec >> q) & 1)


def build_decider(flip=True):
    """Per case, 2^k triangle lists (k ambiguous faces), one per decision index."""
    return [[triangles(c, flip, decision_connect(c, dec)) for dec in range(1 << len(ambiguous_faces(c)))] for c in range(256)]


def write_decider_tables(out):
    table = build_decider(flip=True)
    assert all(rows[0] == tris for rows, tris in zip(table, build(flip=True)))     # no face connected: the sign-rule table
    maxt = max(len(t) for rows in table for t in rows)
    nrows = sum(len(rows) for rows in table)
    with open(out, "w") as f:
        f.write("// GENERATED by tools/gen_mc_tables.py — do not edit.\n")
        f.write("// Marching cubes with the asymptotic decider on ambiguous faces.  Faces f = 0..5 (corner cycles\n")
        f.write("// hy3d_mc_face_corner[f], counter-clockwise seen from outside).  Per case c: hy3d_mc_amb_faces[c] = mask of its\n")
        f.write("// ambiguous faces (inside corners diagonal); with k of them, rows hy3d_mc_dec_first[c] + d, d = 0 .. 2^k - 1, of\n")
        f.write("// hy3d_mc_dec_tri hold its triangles when bit q of d says whether the q-th ambiguous face (ascending f) connects its\n")
        f.write("// inside corners.  Row d = 0 is the row of mc_tables.inc.  Row: triangle count, 3 edge ids per triangle, -1 padded.\n")
        f.write(f"#define HY3D_MC_DEC_MAX_TRIS {maxt}\n")
        f.write(f"#define HY3D_MC_DEC_ROW {1 + 3 * maxt}\n")
        f.write(f"#define HY3D_MC_DEC_ROWS {nrows}\n")
        f.write("HY3D_MC_DEC_QUAL signed char hy3d_mc_face_corner[6][4] = {\n")
        f.write("  " + ",".join("{" + ",".join(str(c) for c in cyc) + "}" for cyc in FACES) + "};\n")
        masks = [sum(1 << fc for fc in ambiguous_faces(c)) for c in range(256)]
        f.write("HY3D_MC_DEC_QUAL unsigned char hy3d_mc_amb_faces[256] = {\n")
        for c0 in range(0, 256, 32):
            f.write("  " + ",".join(str(v) for v in masks[c0:c0 + 32]) + ",\n")
        f.write("};\n")
        first, acc = [], 0
        for rows in table:
            first.append(acc)
            acc += len(rows)
        f.write("HY3D_MC_DEC_QUAL short hy3d_mc_dec_first[256] = {\n")
        for c0 in range(0, 256, 16):
            f.write("  " + ",".join(str(v) for v in first[c0:c0 + 16]) + ",\n")
        f.write("};\n")
        f.write("HY3D_MC_DEC_QUAL signed char hy3d_mc_dec_tri[HY3D_MC_DEC_ROWS][HY3D_MC_DEC_ROW] = {\n")
        for c, rows in enumerate(table):
            for dec, tris in enumerate(rows):
                row = [len(tris)] + [e for t in tris for e in t]
                row += [-1] * (1 + 3 * maxt - len(row))
                f.write("  {" + ",".join(f"{v:2d}" for v in row) + "},\n")
        f.write("};\n")
    print(f"wrote {os.path.normpath(out)}; {nrows} rows, max triangles per cube = {maxt}")


def main(outdir=None):
    table = build(flip=True)
    maxt = max(len(t) for t in table)
    here = os.path.dirname(os.path.abspath(__file__))
    outdir = outdir or os.path.join(here, "..", "hunyuan3d-2_b200", "csrc")
    out = os.path.join(outdir, "mc_tables.inc")
    with open(out, "w") as f:
        f.write("// GENERATED by tools/gen_mc_tables.py — do not edit.\n")
        f.write("// 256-case marching-cubes table derived by face-loop tracing (fixed ambiguous-face rule:\n")
        f.write("// inside corners separated).  Row c: triangle count, then 3 edge ids per triangle, -1 padded.\n")
        f.write(f"#define HY3D_MC_MAX_TRIS {maxt}\n")
        f.write(f"#define HY3D_MC_ROW {1 + 3 * maxt}\n")
        f.write("HY3D_MC_TABLE_QUAL signed char hy3d_mc_tri_table[256][HY3D_MC_ROW] = {\n")
        for c, tris in enumerate(table):
            row = [len(tris)] + [e for t in tris for e in t]
            row += [-1] * (1 + 3 * maxt - len(row))
            f.write("  {" + ",".join(f"{v:2d}" for v in row) + "},\n")
        f.write("};\n")
        # edge geometry: owner corner offset (dz,dy,dx) = (axis0,axis1,axis2) and axis of each edge
        f.write("// edge e: owner voxel offset along (axis0, axis1, axis2) and the array axis it runs along\n")
        f.write("HY3D_MC_TABLE_QUAL signed char hy3d_mc_edge_owner[12][4] = {\n")
        for a, b in EDGES:
            pa, pb = CORNERS[a], CORNERS[b]
            lo = tuple(min(x, y) for x, y in zip(pa, pb))
            d = [abs(x - y) for x, y in zip(pa, pb)].index(1)      # 0:x 1:y 2:z
            axis = 2 - d                                         # array axis
            f.write(f"  {{{lo[2]},{lo[1]},{lo[0]},{axis}}},\n")
        f.write("};\n")
    print(f"wrote {os.path.normpath(out)}; max triangles per cube = {maxt}")
    print("faces (ccw from outside):", FACES)
    write_dmc_tables(os.path.join(outdir, "dmc_tables.inc"))
    write_decider_tables(os.path.join(outdir, "mc_tables_decider.inc"))


def dmc_patches(case):
    """Dual marching cubes: one patch (= one dual vertex) per traced loop, loops in trace_loops order (ascending
    smallest edge id).  Returns the patch index of each of the 12 edges, -1 where the edge has no crossing."""
    patch = [-1] * 12
    for p, loop in enumerate(trace_loops(case)):
        for e in loop:
            assert patch[e] == -1          # no edge belongs to two loops
            patch[e] = p
    return patch


def write_dmc_tables(out):
    rows = [dmc_patches(c) for c in range(256)]
    counts = [max(r) + 1 for r in rows]
    with open(out, "w") as f:
        f.write("// GENERATED by tools/gen_mc_tables.py — do not edit.\n")
        f.write("// Dual marching cubes: per case the number of patches (iso-contour loops of mc_tables.inc, one dual vertex\n")
        f.write("// each) and the patch of each of the 12 cube edges (-1: no crossing).  Patches are numbered in ascending\n")
        f.write("// order of their smallest edge id.\n")
        f.write(f"#define HY3D_DMC_MAX_PATCHES {max(counts)}\n")
        f.write("HY3D_DMC_TABLE_QUAL signed char hy3d_dmc_patch_count[256] = {\n")
        for c0 in range(0, 256, 32):
            f.write("  " + ",".join(str(v) for v in counts[c0:c0 + 32]) + ",\n")
        f.write("};\n")
        f.write("HY3D_DMC_TABLE_QUAL signed char hy3d_dmc_edge_patch[256][12] = {\n")
        for r in rows:
            f.write("  {" + ",".join(f"{v:2d}" for v in r) + "},\n")
        f.write("};\n")
    hist = {k: counts.count(k) for k in sorted(set(counts))}
    print(f"wrote {os.path.normpath(out)}; cases per patch count = {hist}")


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else None)
