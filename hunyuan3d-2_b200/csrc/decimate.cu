// Quadric edge-collapse decimation on the device: FaceReducer of hy3dgen/shapegen/postprocessors.py (contract:
// oracle/decimate.py, which these kernels meet bit for bit).  The mesh is decimated in rounds of independent collapses;
// every round starts from the compacted mesh of the previous one:
//   k_corners        per face: vertex -> corner keys, undirected half-edge keys (min * n + max), repeated ids freeze
//   radix sorts      corners by vertex (stable: ascending face id per vertex) and half-edges by key (stable: by face id)
//   k_vstart         vertex -> corner CSR offsets (lower bound of each vertex id)
//   k_quadrics       first round only: per-vertex sum of the unit plane quadrics of its faces, ascending face id
//   k_edges          per edge (first half-edge of a key run): degrees; an edge without exactly two faces freezes both ends
//   k_fan            per vertex: one closed fan of distinct faces and finite coordinates, or frozen
//   k_candidates     per edge: topology rules, the float32-rounded position, validity (no face flips) and cost
//   radix sort       (cost bits, edge id) -> rank = sorted position
//   k_m1, k_m2       min-propagation of ranks over vertices and their neighbours; k_select: rank == m2[a] == m2[b]
//   scan, k_apply    the ceil((F - T) / 2) lowest-ranked selected collapses move a, merge the quadrics, redirect b to a
//   k_redirect       faces rewritten through the redirection, the two faces of every collapsed edge dropped
//   compact          order-preserving compaction of meshcompact.cuh, quadrics carried; the round's one host synchronisation
// Float64 arithmetic goes through __dadd_rn / __dsub_rn / __dmul_rn / __ddiv_rn / __dsqrt_rn in the oracle's order, so no
// FMA is contracted; every other decision is a minimum, a count or a stable sort, independent of scheduling.
#include "common.cuh"
#include "meshcompact.cuh"

#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

namespace {

constexpr unsigned long long KEY_NONE = ~0ull;
constexpr double DET_MIN = 1e-12, COST_MIN = 1e-15, QUALITYTHR = 1.0;

__device__ __forceinline__ double A(double x, double y) { return __dadd_rn(x, y); }
__device__ __forceinline__ double S(double x, double y) { return __dsub_rn(x, y); }
__device__ __forceinline__ double M(double x, double y) { return __dmul_rn(x, y); }

struct d3 { double x, y, z; };
__device__ __forceinline__ d3 load3(const float* __restrict__ v, int i) {
  return {(double)v[3 * i], (double)v[3 * i + 1], (double)v[3 * i + 2]};
}
__device__ __forceinline__ d3 cross3(d3 u, d3 w) {
  return {S(M(u.y, w.z), M(u.z, w.y)), S(M(u.z, w.x), M(u.x, w.z)), S(M(u.x, w.y), M(u.y, w.x))};
}
__device__ __forceinline__ d3 tri_normal(d3 p0, d3 p1, d3 p2) {
  return cross3({S(p1.x, p0.x), S(p1.y, p0.y), S(p1.z, p0.z)}, {S(p2.x, p0.x), S(p2.y, p0.y), S(p2.z, p0.z)});
}
__device__ __forceinline__ double sq3(d3 n) { return A(A(M(n.x, n.x), M(n.y, n.y)), M(n.z, n.z)); }
__device__ __forceinline__ double dist2(d3 u, d3 w) { return sq3({S(w.x, u.x), S(w.y, u.y), S(w.z, u.z)}); }

__device__ __forceinline__ double det3(double m00, double m01, double m02, double m10, double m11, double m12, double m20,
                                       double m21, double m22) {
  return A(S(M(m00, S(M(m11, m22), M(m12, m21))), M(m01, S(M(m10, m22), M(m12, m20)))), M(m02, S(M(m10, m21), M(m11, m20))));
}

// p^T Q p with p = (x, y, z, 1), Q = (aa, ab, ac, ad, bb, bc, bd, cc, cd, dd)
__device__ __forceinline__ double energy(const double* q, double x, double y, double z) {
  const double t0 = A(A(A(M(q[0], x), M(q[1], y)), M(q[2], z)), q[3]);
  const double t1 = A(A(A(M(q[1], x), M(q[4], y)), M(q[5], z)), q[6]);
  const double t2 = A(A(A(M(q[2], x), M(q[5], y)), M(q[7], z)), q[8]);
  const double t3 = A(A(A(M(q[3], x), M(q[6], y)), M(q[8], z)), q[9]);
  return A(A(A(M(x, t0), M(y, t1)), M(z, t2)), t3);
}

__device__ __forceinline__ bool has_repeat(int a, int b, int c) { return a == b || b == c || a == c; }

// Per face: corner keys (vertex id, value = corner 3f + i), half-edge keys (min * n + max, value = face; KEY_NONE when the
// two ids are equal), vertices of a face with a repeated id frozen.  An out-of-range face raises *err and gets no keys.
__global__ void __launch_bounds__(256) k_corners(const int32_t* __restrict__ faces, long long nF, long long nV,
                                                  unsigned* __restrict__ vkey, unsigned* __restrict__ vval,
                                                  unsigned long long* __restrict__ hkey, unsigned* __restrict__ hval,
                                                  uint8_t* __restrict__ frozen, int* __restrict__ err) {
  const long long f = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (f >= nF) return;
  const int v[3] = {faces[3 * f], faces[3 * f + 1], faces[3 * f + 2]};
  const bool ok = face_in_range(v[0], v[1], v[2], nV);
  if (!ok) *err = 1;
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    const int a = v[i], b = v[(i + 1) % 3];
    vkey[3 * f + i] = ok ? (unsigned)a : 0xffffffffu;
    vval[3 * f + i] = (unsigned)(3 * f + i);
    hkey[3 * f + i] = ok && a != b ? (unsigned long long)min(a, b) * (unsigned long long)nV + (unsigned long long)max(a, b) : KEY_NONE;
    hval[3 * f + i] = (unsigned)f;
  }
  if (ok && has_repeat(v[0], v[1], v[2])) { frozen[v[0]] = 1; frozen[v[1]] = 1; frozen[v[2]] = 1; }
}

// vstart[v] = first sorted corner of vertex v (v in [0, nV])
__global__ void __launch_bounds__(256) k_vstart(const unsigned* __restrict__ skey, long long nC, long long nV, int* __restrict__ vstart,
                                                 const int* __restrict__ err) {
  const long long v = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (v > nV || *err) return;
  long long lo = 0, hi = nC;
  while (lo < hi) {
    const long long mid = (lo + hi) >> 1;
    if (skey[mid] < (unsigned)v) lo = mid + 1; else hi = mid;
  }
  vstart[v] = (int)lo;
}

// Unit plane quadric of face f (zero unless its vertices are finite and 0 < |n| < inf).
__device__ __forceinline__ void face_quadric(const float* __restrict__ verts, const int32_t* __restrict__ faces, int f, double q[10]) {
  const int i0 = faces[3 * f], i1 = faces[3 * f + 1], i2 = faces[3 * f + 2];
  const d3 p0 = load3(verts, i0), n = tri_normal(p0, load3(verts, i1), load3(verts, i2));
  const double ln = __dsqrt_rn(sq3(n));
  if (!(finite3(verts, i0) && finite3(verts, i1) && finite3(verts, i2) && ln > 0.0 && ln < __longlong_as_double(0x7ff0000000000000ll))) {
#pragma unroll
    for (int j = 0; j < 10; ++j) q[j] = 0.0;
    return;
  }
  const double a = __ddiv_rn(n.x, ln), b = __ddiv_rn(n.y, ln), c = __ddiv_rn(n.z, ln);
  const double d = -A(A(M(a, p0.x), M(b, p0.y)), M(c, p0.z));
  q[0] = M(a, a); q[1] = M(a, b); q[2] = M(a, c); q[3] = M(a, d); q[4] = M(b, b);
  q[5] = M(b, c); q[6] = M(b, d); q[7] = M(c, c); q[8] = M(c, d); q[9] = M(d, d);
}

__global__ void __launch_bounds__(128) k_quadrics(const float* __restrict__ verts, long long nV, const int32_t* __restrict__ faces,
                                                   const int* __restrict__ vstart, const unsigned* __restrict__ corner,
                                                   double* __restrict__ Q, const int* __restrict__ err) {
  const long long v = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= nV || *err) return;
  double acc[10];
#pragma unroll
  for (int j = 0; j < 10; ++j) acc[j] = 0.0;
  for (int s = vstart[v]; s < vstart[v + 1]; ++s) {
    double q[10];
    face_quadric(verts, faces, (int)(corner[s] / 3), q);
#pragma unroll
    for (int j = 0; j < 10; ++j) acc[j] = A(acc[j], q[j]);
  }
#pragma unroll
  for (int j = 0; j < 10; ++j) Q[10 * v + j] = acc[j];
}

__device__ __forceinline__ bool is_head(const unsigned long long* __restrict__ hk, long long h) {
  return hk[h] != KEY_NONE && (h == 0 || hk[h - 1] != hk[h]);
}

__device__ __forceinline__ int run_length(const unsigned long long* __restrict__ hk, long long h, long long nC) {
  int c = 1;
  while (h + c < nC && hk[h + c] == hk[h]) ++c;
  return c;
}

// Per edge: both ends gain a neighbour; an edge with one face or three or more freezes both ends.
__global__ void __launch_bounds__(256) k_edges(const unsigned long long* __restrict__ hk, long long nC, long long nV,
                                                int* __restrict__ deg, uint8_t* __restrict__ frozen, const int* __restrict__ err) {
  const long long h = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (h >= nC || *err || !is_head(hk, h)) return;
  const int a = (int)(hk[h] / (unsigned long long)nV), b = (int)(hk[h] % (unsigned long long)nV);
  atomicAdd(deg + a, 1);
  atomicAdd(deg + b, 1);
  if (run_length(hk, h, nC) != 2) { frozen[a] = 1; frozen[b] = 1; }
}

// Link edge x -> y of the corner of `v` at sorted position s: the face is (v, x, y) rotated.
__device__ __forceinline__ void link_edge(const int32_t* __restrict__ faces, unsigned corner, int& x, int& y) {
  const unsigned f = corner / 3, i = corner % 3;
  x = faces[3 * f + (i + 1) % 3];
  y = faces[3 * f + (i + 2) % 3];
}

// A vertex stays free iff its coordinates are finite and its link edges form one cycle through all of them (one closed
// fan): no two share a source, no two share a target, and the walk from the first returns to it after exactly k steps.
__global__ void __launch_bounds__(128) k_fan(const float* __restrict__ verts, long long nV, const int32_t* __restrict__ faces,
                                              const int* __restrict__ vstart, const unsigned* __restrict__ corner,
                                              uint8_t* __restrict__ frozen, const int* __restrict__ err) {
  const long long v = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= nV || *err || frozen[v]) return;
  const int s0 = vstart[v], k = vstart[v + 1] - s0;
  bool ok = k > 0 && finite3(verts, v);
  for (int i = 0; ok && i < k; ++i) {
    int xi, yi;
    link_edge(faces, corner[s0 + i], xi, yi);
    for (int j = i + 1; j < k; ++j) {
      int xj, yj;
      link_edge(faces, corner[s0 + j], xj, yj);
      if (xi == xj || yi == yj) { ok = false; break; }
    }
  }
  int cur = 0;
  for (int step = 1; ok && step <= k; ++step) {
    int x, y;
    link_edge(faces, corner[s0 + cur], x, y);
    int nxt = -1;
    for (int j = 0; j < k; ++j) {
      int xj, yj;
      link_edge(faces, corner[s0 + j], xj, yj);
      if (xj == y) { nxt = j; break; }
    }
    if (nxt < 0 || (nxt == 0) != (step == k)) ok = false;
    cur = nxt;
  }
  if (!ok) frozen[v] = 1;
}

__device__ __forceinline__ bool directed(const int32_t* __restrict__ faces, int f, int a, int b) {
  const int g0 = faces[3 * f], g1 = faces[3 * f + 1], g2 = faces[3 * f + 2];
  return (g0 == a && g1 == b) || (g1 == a && g2 == b) || (g2 == a && g0 == b);
}

// Faces of the star of `v` other than f1, f2 with a and b replaced by p: all keep n_old . n_new > 0 -> smallest quality.
__device__ __forceinline__ bool star_ok(const float* __restrict__ verts, const int32_t* __restrict__ faces,
                                       const int* __restrict__ vstart, const unsigned* __restrict__ corner, int v, int a, int b,
                                       int f1, int f2, d3 p, double& qmin) {
  for (int s = vstart[v]; s < vstart[v + 1]; ++s) {
    const int f = (int)(corner[s] / 3);
    if (f == f1 || f == f2) continue;
    const int g0 = faces[3 * f], g1 = faces[3 * f + 1], g2 = faces[3 * f + 2];
    const d3 o0 = load3(verts, g0), o1 = load3(verts, g1), o2 = load3(verts, g2);
    const d3 n0 = (g0 == a || g0 == b) ? p : o0, n1 = (g1 == a || g1 == b) ? p : o1, n2 = (g2 == a || g2 == b) ? p : o2;
    const d3 no = tri_normal(o0, o1, o2), nn = tri_normal(n0, n1, n2);
    const double dot = A(A(M(no.x, nn.x), M(no.y, nn.y)), M(no.z, nn.z));
    if (!(dot > 0.0)) return false;
    const double l2 = fmax(fmax(dist2(n0, n1), dist2(n1, n2)), dist2(n2, n0));
    const double qual = __ddiv_rn(__dsqrt_rn(sq3(nn)), l2);
    if (qual < qmin) qmin = qual;
  }
  return true;
}

// Per edge: the contract's candidate rules, position, validity and cost.  ckey[h] = cost bits (KEY_NONE when not a valid
// candidate), cval[h] = h, pos[h] = the float32 position.
__global__ void __launch_bounds__(128, 1) k_candidates(const float* __restrict__ verts, long long nV, const int32_t* __restrict__ faces,
                                                     const int* __restrict__ vstart, const unsigned* __restrict__ corner,
                                                     const unsigned long long* __restrict__ hk, const unsigned* __restrict__ hface,
                                                     long long nC, const int* __restrict__ deg, const uint8_t* __restrict__ frozen,
                                                     const double* __restrict__ Q, unsigned long long* __restrict__ ckey,
                                                     unsigned* __restrict__ cval, float* __restrict__ pos, const int* __restrict__ err) {
  const long long h = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (h >= nC) return;
  ckey[h] = KEY_NONE;
  cval[h] = (unsigned)h;
  if (*err || !is_head(hk, h) || run_length(hk, h, nC) != 2) return;
  const int a = (int)(hk[h] / (unsigned long long)nV), b = (int)(hk[h] % (unsigned long long)nV);
  if (frozen[a] || frozen[b]) return;
  const int f1 = (int)hface[h], f2 = (int)hface[h + 1];
  const bool d1 = directed(faces, f1, a, b), d2 = directed(faces, f2, a, b);
  if (d1 == d2) return;
  const int fab = d1 ? f1 : f2, fba = d1 ? f2 : f1;
  const int c = faces[3 * fab] + faces[3 * fab + 1] + faces[3 * fab + 2] - a - b;
  const int d = faces[3 * fba] + faces[3 * fba + 1] + faces[3 * fba + 2] - a - b;
  if (c == d || deg[a] + deg[b] - 4 < 3 || deg[c] < 4 || deg[d] < 4) return;
  int common = 0;                                           // a, b free: their neighbours are the sources of their link edges
  for (int s = vstart[a]; s < vstart[a + 1]; ++s) {
    int x, y;
    link_edge(faces, corner[s], x, y);
    for (int t = vstart[b]; t < vstart[b + 1]; ++t) {
      int xb, yb;
      link_edge(faces, corner[t], xb, yb);
      common += xb == x;
    }
  }
  if (common != 2) return;

  double q[10];
#pragma unroll
  for (int j = 0; j < 10; ++j) q[j] = A(Q[10 * a + j], Q[10 * b + j]);
  const d3 pa = load3(verts, a), pb = load3(verts, b);
  const d3 mid = {M(A(pa.x, pb.x), 0.5), M(A(pa.y, pb.y), 0.5), M(A(pa.z, pb.z), 0.5)};
  d3 best = pa;
  double e = energy(q, pa.x, pa.y, pa.z);
  const double eb = energy(q, pb.x, pb.y, pb.z);
  if (eb < e) { best = pb; e = eb; }
  const double em = energy(q, mid.x, mid.y, mid.z);
  if (em < e) { best = mid; e = em; }
  const double det = det3(q[0], q[1], q[2], q[1], q[4], q[5], q[2], q[5], q[7]);
  if (fabs(det) >= DET_MIN) {
    const double bx = -q[3], by = -q[6], bz = -q[8];
    const d3 o = {__ddiv_rn(det3(bx, q[1], q[2], by, q[4], q[5], bz, q[5], q[7]), det),
                  __ddiv_rn(det3(q[0], bx, q[2], q[1], by, q[5], q[2], bz, q[7]), det),
                  __ddiv_rn(det3(q[0], q[1], bx, q[1], q[4], by, q[2], q[5], bz), det)};
    if (energy(q, o.x, o.y, o.z) <= e) best = o;
  }
  const float px = __double2float_rn(best.x), py = __double2float_rn(best.y), pz = __double2float_rn(best.z);
  const d3 p = {(double)px, (double)py, (double)pz};
  double qmin = __longlong_as_double(0x7ff0000000000000ll);
  if (!star_ok(verts, faces, vstart, corner, a, a, b, f1, f2, p, qmin)) return;
  if (!star_ok(verts, faces, vstart, corner, b, a, b, f1, f2, p, qmin)) return;
  const double en = energy(q, p.x, p.y, p.z);
  const double cost = __ddiv_rn(en > COST_MIN ? en : COST_MIN, qmin < QUALITYTHR ? qmin : QUALITYTHR);
  ckey[h] = (unsigned long long)__double_as_longlong(cost);
  pos[3 * h] = px; pos[3 * h + 1] = py; pos[3 * h + 2] = pz;
}

__device__ __forceinline__ void edge_ends(const unsigned long long* __restrict__ hk, unsigned h, long long nV, int& a, int& b) {
  a = (int)(hk[h] / (unsigned long long)nV);
  b = (int)(hk[h] % (unsigned long long)nV);
}

// m1[v] = smallest rank (sorted position r) of a valid edge at v
__global__ void __launch_bounds__(256) k_m1(const unsigned long long* __restrict__ skey, const unsigned* __restrict__ sval,
                                             const unsigned long long* __restrict__ hk, long long nC, long long nV, int* __restrict__ m1,
                                             const int* __restrict__ err) {
  const long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= nC || *err || skey[r] == KEY_NONE) return;
  int a, b;
  edge_ends(hk, sval[r], nV, a, b);
  atomicMin(m1 + a, (int)r);
  atomicMin(m1 + b, (int)r);
}

// m2 (= m1 on entry) lowered by m1 of every neighbour
__global__ void __launch_bounds__(256) k_m2(const unsigned long long* __restrict__ hk, long long nC, long long nV,
                                             const int* __restrict__ m1, int* __restrict__ m2, const int* __restrict__ err) {
  const long long h = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (h >= nC || *err || !is_head(hk, h)) return;
  int a, b;
  edge_ends(hk, (unsigned)h, nV, a, b);
  atomicMin(m2 + a, m1[b]);
  atomicMin(m2 + b, m1[a]);
}

__global__ void __launch_bounds__(256) k_select(const unsigned long long* __restrict__ skey, const unsigned* __restrict__ sval,
                                                 const unsigned long long* __restrict__ hk, long long nC, long long nV,
                                                 const int* __restrict__ m2, int* __restrict__ sel, const int* __restrict__ err) {
  const long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= nC) return;
  int s = 0;
  if (!*err && skey[r] != KEY_NONE) {
    int a, b;
    edge_ends(hk, sval[r], nV, a, b);
    s = m2[a] == (int)r && m2[b] == (int)r;
  }
  sel[r] = s;
}

// The `limit` lowest-ranked selected collapses: a takes p and Qa + Qb, b is redirected to a, the edge's faces are dropped.
// Selected edges share no vertex and no neighbour, so every thread writes its own a, b and faces.
__global__ void __launch_bounds__(256) k_apply(const unsigned* __restrict__ sval, const int* __restrict__ sel, const int* __restrict__ pre,
                                                long long limit, const unsigned long long* __restrict__ hk, const unsigned* __restrict__ hface,
                                                long long nC, long long nV, const float* __restrict__ pos, float* __restrict__ verts,
                                                double* __restrict__ Q, int* __restrict__ redirect, uint8_t* __restrict__ fdrop) {
  const long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= nC || !sel[r] || pre[r] >= limit) return;
  const unsigned h = sval[r];
  int a, b;
  edge_ends(hk, h, nV, a, b);
#pragma unroll
  for (int j = 0; j < 3; ++j) verts[3 * a + j] = pos[3 * h + j];
#pragma unroll
  for (int j = 0; j < 10; ++j) Q[10 * a + j] = A(Q[10 * a + j], Q[10 * b + j]);
  redirect[b] = a;
  fdrop[hface[h]] = 1;
  fdrop[hface[h + 1]] = 1;
}

__global__ void __launch_bounds__(256) k_redirect(const int32_t* __restrict__ faces, long long nF, const int* __restrict__ redirect,
                                                   const uint8_t* __restrict__ fdrop, int32_t* __restrict__ out, uint8_t* __restrict__ fkeep,
                                                   uint8_t* __restrict__ vref, const int* __restrict__ err) {
  const long long f = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (f >= nF) return;
  if (*err || fdrop[f]) { fkeep[f] = 0; return; }
  fkeep[f] = 1;
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    const int v = faces[3 * f + i], r = redirect[v];
    const int w = r >= 0 ? r : v;
    out[3 * f + i] = w;
    vref[w] = 1;
  }
}

__global__ void __launch_bounds__(256) k_check_range(const int32_t* __restrict__ faces, long long nF, long long nV, int* __restrict__ err) {
  const long long f = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (f < nF && !face_in_range(faces[3 * f], faces[3 * f + 1], faces[3 * f + 2], nV)) *err = 1;
}

int bits_for(unsigned long long n) {                        // smallest b with 2^b > n
  int b = 0;
  while (b < 64 && (n >> b) != 0) ++b;
  return b;
}

}  // namespace

extern "C" int hy3d_mesh_decimate(hy3d_ctx* ctx, const float* d_verts, int64_t nV, const int32_t* d_faces, int64_t nF, int64_t max_faces,
                                  float* d_verts_out, int32_t* d_faces_out, int64_t* h_nv_out, int64_t* h_nf_out, int32_t* h_rounds) {
  if (!ctx || nV < 0 || nF < 0 || !h_nv_out || !h_nf_out || !h_rounds) return HY3D_ERR_ARG;
  *h_nv_out = 0; *h_nf_out = 0; *h_rounds = 0;
  if (max_faces < 1) return hy3d_fail(ctx, HY3D_ERR_ARG, "max_faces < 1");
  if (nF > 0 && nV == 0) return hy3d_fail(ctx, HY3D_ERR_ARG, "face index outside [0, 0)");
  if ((nV && (!d_verts || !d_verts_out)) || (nF && (!d_faces || !d_faces_out))) return HY3D_ERR_ARG;
  if (nV > 2147483647LL) return hy3d_fail(ctx, HY3D_ERR_UNSUPPORTED, "vertex ids exceed int32");
  if (nF > 715827882LL) return hy3d_fail(ctx, HY3D_ERR_UNSUPPORTED, "corner ids (3 nF) exceed 32 bits");
  HY3D_CUDA(ctx, cudaSetDevice(ctx->device));
  const long long nC0 = 3 * nF;
  cudaStream_t st = ctx->stream;

  // CUB temporary storage: the largest of the three sorts and the scan at the first round's sizes
  size_t tmp_bytes = 0, b;
  HY3D_CUDA(ctx, cub::DeviceRadixSort::SortPairs(nullptr, b, (unsigned*)nullptr, (unsigned*)nullptr, (unsigned*)nullptr,
                                                 (unsigned*)nullptr, (int)nC0, 0, 32, st));
  tmp_bytes = b;
  HY3D_CUDA(ctx, cub::DeviceRadixSort::SortPairs(nullptr, b, (unsigned long long*)nullptr, (unsigned long long*)nullptr,
                                                 (unsigned*)nullptr, (unsigned*)nullptr, (int)nC0, 0, 64, st));
  tmp_bytes = b > tmp_bytes ? b : tmp_bytes;
  HY3D_CUDA(ctx, cub::DeviceScan::ExclusiveSum(nullptr, b, (int*)nullptr, (int*)nullptr, (int)nC0, st));
  tmp_bytes = b > tmp_bytes ? b : tmp_bytes;

  Compaction cp;
  float* V[2]; double* Q[2]; int32_t *F[2], *ftmp;
  unsigned *vkey[2], *vval[2], *hval[2], *cval[2];
  unsigned long long *hkey[2], *ckey[2];
  float* pos; uint8_t *frozen, *fdrop; int *vstart, *deg, *m1, *m2, *redirect, *sel, *pre, *err;
  void* tmp;
  int rc = carve_scratch(ctx, nV, nF, cp, [&](Carver& c) {
    for (int i = 0; i < 2; ++i) {
      V[i] = c.take<float>(3 * nV); Q[i] = c.take<double>(10 * nV); F[i] = c.take<int32_t>(nC0);
      vkey[i] = c.take<unsigned>(nC0); vval[i] = c.take<unsigned>(nC0); hkey[i] = c.take<unsigned long long>(nC0);
      hval[i] = c.take<unsigned>(nC0); ckey[i] = c.take<unsigned long long>(nC0); cval[i] = c.take<unsigned>(nC0);
    }
    ftmp = c.take<int32_t>(nC0); pos = c.take<float>(3 * nC0); sel = c.take<int>(nC0); pre = c.take<int>(nC0);
    frozen = c.take<uint8_t>(nV); fdrop = c.take<uint8_t>(nF); vstart = c.take<int>(nV + 1); deg = c.take<int>(nV);
    m1 = c.take<int>(nV); m2 = c.take<int>(nV); redirect = c.take<int>(nV); err = c.take<int>(1);
    tmp = c.take<char>(tmp_bytes);
  });
  if (rc) return rc;
  HY3D_CUDA(ctx, cudaMemsetAsync(err, 0, sizeof(int), st));

  if (nF <= max_faces) {                                    // returned as given (face ids still checked)
    if (nF) {
      HY3D_PROF(ctx, FAM_MC_EMIT);
      k_check_range<<<(unsigned)ceil_div64(nF, 256), 256, 0, st>>>(d_faces, nF, nV, err);
      HY3D_LAUNCH_CHECK(ctx);
      HY3D_CUDA(ctx, cudaMemcpyAsync(d_faces_out, d_faces, 12 * nF, cudaMemcpyDeviceToDevice, st));
    }
    if (nV) HY3D_CUDA(ctx, cudaMemcpyAsync(d_verts_out, d_verts, 12 * nV, cudaMemcpyDeviceToDevice, st));
    int* perr = reinterpret_cast<int*>(ctx->pinned);
    HY3D_CUDA(ctx, cudaMemcpyAsync(perr, err, 4, cudaMemcpyDeviceToHost, st));
    HY3D_CUDA(ctx, cudaStreamSynchronize(st));
    if (*perr) return hy3d_fail(ctx, HY3D_ERR_ARG, "face index outside [0, %lld)", (long long)nV);
    *h_nv_out = nV; *h_nf_out = nF;
    return HY3D_OK;
  }

  HY3D_CUDA(ctx, cudaMemcpyAsync(V[0], d_verts, 12 * nV, cudaMemcpyDeviceToDevice, st));
  long long n = nV, m = nF;
  int cur = 0, rounds = 0;
  const int32_t* Fc = d_faces;
  for (bool first = true; m > max_faces; first = false) {
    const long long nC = 3 * m;
    const unsigned gC = (unsigned)ceil_div64(nC, 256), gV = (unsigned)ceil_div64(n + 1, 256), gF = (unsigned)ceil_div64(m, 256);
    const unsigned gC128 = (unsigned)ceil_div64(nC, 128), gV128 = (unsigned)ceil_div64(n, 128);
    cp.sizes(n, m);
    HY3D_CUDA(ctx, cudaMemsetAsync(frozen, 0, n, st));
    HY3D_CUDA(ctx, cudaMemsetAsync(deg, 0, 4 * n, st));
    HY3D_CUDA(ctx, cudaMemsetAsync(m1, 0x7f, 4 * n, st));   // 0x7f7f7f7f: above every rank
    HY3D_CUDA(ctx, cudaMemsetAsync(redirect, 0xff, 4 * n, st));
    HY3D_CUDA(ctx, cudaMemsetAsync(fdrop, 0, m, st));
    HY3D_CUDA(ctx, cudaMemsetAsync(cp.vref, 0, n, st));
    HY3D_PROF(ctx, FAM_MC_EMIT);
    k_corners<<<gF, 256, 0, st>>>(Fc, m, n, vkey[0], vval[0], hkey[0], hval[0], frozen, err);
    HY3D_LAUNCH_CHECK(ctx);
    size_t tb = tmp_bytes;
    HY3D_PROF(ctx, FAM_MC_SCAN);
    HY3D_CUDA(ctx, cub::DeviceRadixSort::SortPairs(tmp, tb, vkey[0], vkey[1], vval[0], vval[1], (int)nC, 0, bits_for(n), st));
    HY3D_LAUNCH_CHECK(ctx);
    tb = tmp_bytes;
    HY3D_PROF(ctx, FAM_MC_SCAN);
    HY3D_CUDA(ctx, cub::DeviceRadixSort::SortPairs(tmp, tb, hkey[0], hkey[1], hval[0], hval[1], (int)nC, 0,
                                                   bits_for((unsigned long long)n * n), st));
    HY3D_LAUNCH_CHECK(ctx);
    const unsigned* corner = vval[1];
    const unsigned long long* hk = hkey[1];
    HY3D_PROF(ctx, FAM_MC_EMIT);
    k_vstart<<<gV, 256, 0, st>>>(vkey[1], nC, n, vstart, err);
    HY3D_LAUNCH_CHECK(ctx);
    if (first) {
      HY3D_PROF(ctx, FAM_MC_EMIT);
      k_quadrics<<<gV128, 128, 0, st>>>(V[0], n, Fc, vstart, corner, Q[0], err);
      HY3D_LAUNCH_CHECK(ctx);
    }
    HY3D_PROF(ctx, FAM_MC_EMIT);
    k_edges<<<gC, 256, 0, st>>>(hk, nC, n, deg, frozen, err);
    HY3D_LAUNCH_CHECK(ctx);
    HY3D_PROF(ctx, FAM_MC_EMIT);
    k_fan<<<gV128, 128, 0, st>>>(V[cur], n, Fc, vstart, corner, frozen, err);
    HY3D_LAUNCH_CHECK(ctx);
    HY3D_PROF(ctx, FAM_MC_EMIT);
    k_candidates<<<gC128, 128, 0, st>>>(V[cur], n, Fc, vstart, corner, hk, hval[1], nC, deg, frozen, Q[cur], ckey[0], cval[0], pos, err);
    HY3D_LAUNCH_CHECK(ctx);
    tb = tmp_bytes;
    HY3D_PROF(ctx, FAM_MC_SCAN);
    HY3D_CUDA(ctx, cub::DeviceRadixSort::SortPairs(tmp, tb, ckey[0], ckey[1], cval[0], cval[1], (int)nC, 0, 64, st));
    HY3D_LAUNCH_CHECK(ctx);
    HY3D_PROF(ctx, FAM_MC_EMIT);
    k_m1<<<gC, 256, 0, st>>>(ckey[1], cval[1], hk, nC, n, m1, err);
    HY3D_LAUNCH_CHECK(ctx);
    HY3D_CUDA(ctx, cudaMemcpyAsync(m2, m1, 4 * n, cudaMemcpyDeviceToDevice, st));
    HY3D_PROF(ctx, FAM_MC_EMIT);
    k_m2<<<gC, 256, 0, st>>>(hk, nC, n, m1, m2, err);
    HY3D_LAUNCH_CHECK(ctx);
    HY3D_PROF(ctx, FAM_MC_EMIT);
    k_select<<<gC, 256, 0, st>>>(ckey[1], cval[1], hk, nC, n, m2, sel, err);
    HY3D_LAUNCH_CHECK(ctx);
    tb = tmp_bytes;
    HY3D_PROF(ctx, FAM_MC_SCAN);
    HY3D_CUDA(ctx, cub::DeviceScan::ExclusiveSum(tmp, tb, sel, pre, (int)nC, st));
    HY3D_LAUNCH_CHECK(ctx);
    HY3D_PROF(ctx, FAM_MC_EMIT);
    k_apply<<<gC, 256, 0, st>>>(cval[1], sel, pre, (m - max_faces + 1) / 2, hk, hval[1], nC, n, pos, V[cur], Q[cur], redirect, fdrop);
    HY3D_LAUNCH_CHECK(ctx);
    HY3D_PROF(ctx, FAM_MC_EMIT);
    k_redirect<<<gF, 256, 0, st>>>(Fc, m, redirect, fdrop, ftmp, cp.fkeep, cp.vref, err);
    HY3D_LAUNCH_CHECK(ctx);
    int64_t nn, mm;
    rc = compact(ctx, cp, V[cur], n, ftmp, m, 0, err, V[1 - cur], F[1 - cur], &nn, &mm, Q[cur], Q[1 - cur]);
    if (rc) return rc;
    cur = 1 - cur;
    Fc = F[cur];
    const bool applied = mm < m;
    n = nn; m = mm;
    if (!applied) break;
    ++rounds;
  }
  HY3D_CUDA(ctx, cudaMemcpyAsync(d_verts_out, V[cur], 12 * n, cudaMemcpyDeviceToDevice, st));
  HY3D_CUDA(ctx, cudaMemcpyAsync(d_faces_out, Fc, 12 * m, cudaMemcpyDeviceToDevice, st));
  *h_nv_out = n; *h_nf_out = m; *h_rounds = rounds;
  return HY3D_OK;
}
