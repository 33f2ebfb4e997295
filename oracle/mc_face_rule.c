/* ORACLE (test infrastructure, never shipped): marching cubes with a choice of rule for ambiguous faces, the contract
 * of MCSurfaceExtractor(face_rule=...) / hy3d_set_mc_face_rule.
 *
 * An ambiguous face has its two inside corners on one diagonal and its two outside corners on the other.
 *   face rule 0, "sign": the inside corners are separated (each is cut off) -- exactly mc_oracle.c;
 *   face rule 1, "asymptotic": the asymptotic decider of Lewiner's face test (skimage.measure.marching_cubes,
 *     method="lewiner").  With d = v - level in float32, inside diagonal (a, c) and outside diagonal (b, d), the
 *     inside corners connect iff
 *         (double)d_a * (double)d_c > (double)d_b * (double)d_d
 *     A product of two floats is exact in float64, so the comparison is exact; equality or any NaN => separated.
 *     Both cubes that share a face evaluate the same comparison, so the mesh stays watertight.
 * Lewiner's interior tests (a vertex inside the cube, MC33 cases 4, 6, 7, 10, 12, 13) are not restated.
 *
 * Vertices (one per sign-change edge, same interpolation, order and welding) are mc_oracle.c's: this file includes it
 * and takes the vertex array from hy3d_oracle_mc.  Per cube, the face decisions choose the loops the iso-contour
 * tracing produces; each loop is fan-triangulated from its first edge; triangles in cube order.  Like mc_oracle.c it
 * traces at run time and does NOT read the generated tables (hunyuan3d-2_b200/csrc/mc_tables_decider.inc).
 *
 * Build: oracle/mc_face_rule.py (gcc -O2 -ffp-contract=off, as oracle/Makefile).
 */
#include "mc_oracle.c"

/* Triangles of one cube as edge ids; returns the count (<= 10).  Bit f of `connect` set: the ambiguous face FACE[f]
 * connects its inside corners (each outside corner is cut off); clear: each inside corner is cut off. */
static int cube_triangles_connect(int cs, int connect, int tri[10][3]) {
    int nxt[12];
    for (int e = 0; e < 12; ++e) nxt[e] = -1;
    for (int f = 0; f < 6; ++f) {
        int in[4], ed[4];
        for (int m = 0; m < 4; ++m) {
            in[m] = (cs >> FACE[f][m]) & 1;
            ed[m] = edge_between(FACE[f][m], FACE[f][(m + 1) & 3]);
        }
        int nio = 0, io[2], oi[2], noi = 0;
        for (int m = 0; m < 4; ++m) {
            if (in[m] && !in[(m + 1) & 3]) io[nio++] = m;
            if (!in[m] && in[(m + 1) & 3]) oi[noi++] = m;
        }
        if (nio == 1) nxt[ed[io[0]]] = ed[oi[0]];
        else if (nio == 2)
            for (int q = 0; q < 2; ++q) nxt[ed[io[q]]] = ed[((connect >> f) & 1) ? (io[q] + 1) & 3 : (io[q] + 3) & 3];
    }
    int seen[12] = {0}, nt = 0;
    for (int s = 0; s < 12; ++s) {
        if (nxt[s] < 0 || seen[s]) continue;
        int loop[12], n = 0, e = s;
        while (!seen[e]) { seen[e] = 1; loop[n++] = e; e = nxt[e]; }
        for (int m = 1; m + 1 < n; ++m) {          /* fan, reversed winding (as mc_oracle.c) */
            tri[nt][0] = loop[0]; tri[nt][1] = loop[m + 1]; tri[nt][2] = loop[m]; ++nt;
        }
    }
    return nt;
}

/* Asymptotic decider of one cube: bit f set iff face f is ambiguous and its inside corners connect.  d[m] = v - level
 * (float32) of corner m. */
static int face_connect(int cs, const float d[8]) {
    int connect = 0;
    for (int f = 0; f < 6; ++f) {
        const int* c = FACE[f];
        const int i0 = (cs >> c[0]) & 1, i1 = (cs >> c[1]) & 1;
        if (i0 == i1 || ((cs >> c[2]) & 1) != i0 || ((cs >> c[3]) & 1) != i1) continue;   /* not ambiguous */
        const int a = i0 ? 0 : 1;                  /* inside diagonal: face corners a, a + 2 */
        const double in_p = (double)d[c[a]] * (double)d[c[a + 2]];
        const double out_p = (double)d[c[a + 1]] * (double)d[c[(a + 3) & 3]];
        if (in_p > out_p) connect |= 1 << f;
    }
    return connect;
}

/* Triangles of case cs with face mask `connect` into tri[10][3] (the table test); returns the count. */
int hy3d_oracle_cube_triangles(int cs, int connect, int32_t* tri) {
    int t[10][3];
    const int nt = cube_triangles_connect(cs, connect, t);
    for (int q = 0; q < nt; ++q) for (int c = 0; c < 3; ++c) tri[3 * q + c] = t[q][c];
    return nt;
}

/* hy3d_oracle_mc with a face rule (0 sign, 1 asymptotic).  Returns 0 on success; buffers as hy3d_oracle_mc's. */
int hy3d_oracle_mc_rule(const float* vol, int n0, int n1, int n2, float level, int face_rule,
                        float** verts_out, int64_t* nV_out, int32_t** faces_out, int64_t* nF_out) {
    if (face_rule != 0 && face_rule != 1) return -2;
    int32_t* sign_faces = NULL;
    int64_t nF_sign = 0;
    int rc = hy3d_oracle_mc(vol, n0, n1, n2, level, verts_out, nV_out, &sign_faces, &nF_sign);
    if (rc) return rc;
    free(sign_faces);
    const int64_t s0 = (int64_t)n1 * n2, s1 = n2;
    const int64_t nvox = (int64_t)n0 * n1 * n2;
    int32_t* eid = (int32_t*)malloc(sizeof(int32_t) * 3 * (size_t)nvox);   /* edge -> vertex id, as hy3d_oracle_mc */
    if (!eid) return -1;
    int32_t nV = 0;
    for (int i = 0; i < n0; ++i) for (int j = 0; j < n1; ++j) for (int k = 0; k < n2; ++k) {
        int64_t p = i * s0 + j * s1 + k;
        int a = inside(vol[p], level);
        eid[3*p+0] = (i + 1 < n0 && inside(vol[p + s0], level) != a) ? nV++ : -1;
        eid[3*p+1] = (j + 1 < n1 && inside(vol[p + s1], level) != a) ? nV++ : -1;
        eid[3*p+2] = (k + 1 < n2 && inside(vol[p + 1],  level) != a) ? nV++ : -1;
    }
    int64_t capF = 1024, nF = 0;
    int32_t* faces = (int32_t*)malloc(sizeof(int32_t) * 3 * (size_t)capF);
    for (int i = 0; i + 1 < n0; ++i) for (int j = 0; j + 1 < n1; ++j) for (int k = 0; k + 1 < n2; ++k) {
        int cs = 0;
        float d[8];
        for (int m = 0; m < 8; ++m) {
            int64_t p = (i + CORNER[m][2]) * s0 + (j + CORNER[m][1]) * s1 + (k + CORNER[m][0]);
            cs |= inside(vol[p], level) << m;
            d[m] = vol[p] - level;
        }
        if (cs == 0 || cs == 255) continue;
        int tri[10][3];
        int nt = cube_triangles_connect(cs, face_rule == 1 ? face_connect(cs, d) : 0, tri);
        if (nF + nt > capF) { capF *= 2; faces = (int32_t*)realloc(faces, sizeof(int32_t) * 3 * (size_t)capF); }
        for (int t = 0; t < nt; ++t) {
            for (int c = 0; c < 3; ++c) {
                int e = tri[t][c];
                const int* ca = CORNER[EDGE[e][0]]; const int* cb = CORNER[EDGE[e][1]];
                int ox = ca[0] < cb[0] ? ca[0] : cb[0], oy = ca[1] < cb[1] ? ca[1] : cb[1], oz = ca[2] < cb[2] ? ca[2] : cb[2];
                int axis = (ca[2] != cb[2]) ? 0 : (ca[1] != cb[1]) ? 1 : 2;     /* array axis */
                int64_t p = (i + oz) * s0 + (j + oy) * s1 + (k + ox);
                faces[3*nF + c] = eid[3*p + axis];
            }
            ++nF;
        }
    }
    free(eid);
    *faces_out = faces; *nF_out = nF;
    return 0;
}
