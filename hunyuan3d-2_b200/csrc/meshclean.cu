// Mesh clean-up on the device, before the mesh crosses PCIe: what the step right after the hot path does on the host —
// export_to_trimesh (reference hy3dgen/shapegen/pipelines.py:95-110): `mesh_f[:, ::-1]` (winding flip) followed by
// trimesh.Trimesh(v, f) whose default processing drops non-finite vertices together with every face that references one,
// and keeps only referenced vertices, re-indexing the faces (SURVEY §8f rank 3).  The sparse volume decoders leave NaN at
// unvisited voxels, so their meshes carry NaN vertices along the band's rim (SURVEY §0.5); here they never leave the GPU.
//
//   k_face_flags   per face: all three vertices finite?  -> keep bit + marks its vertices referenced      (12 F read)
//   k_keep_counts  per 1024-element block: kept vertices (finite & referenced) / kept faces              (V + F bytes)
//   k_scan_counts  exclusive scan of the block counts (one block), totals
//   k_emit         order-preserving compaction: vertices copied, faces re-indexed and (optionally) flipped (12 V + 12 F in / out)
// Integer / byte work, HBM-bound: algorithmic bytes 24 V + 24 F.  (trimesh also merges vertices closer than 1e-8; the
// marching-cubes output is welded already, see INTEGRATION.md for the one corner case.)
//
// The two filters of hy3dgen/shapegen/postprocessors.py that are graph / hash work (contract: oracle/postprocess.py) end in
// the same compaction:
//   hy3d_mesh_remove_floaters  edge table (open addressing, key (min, max) of the undirected edge, slot = smallest face on it)
//                              -> union-find over faces sharing an edge (label = smallest face id of the component) -> sizes
//                              -> vertices of small components selected -> faces touching a selected vertex dropped
//   hy3d_mesh_weld             position table (key = the three fp32 bit patterns, -0 == +0, non-finite never merged, slot =
//                              smallest vertex id) -> faces rewritten through it -> faces with two equal ids dropped
// Both are deterministic whatever the scheduling: every value kept is a minimum or a count.
#include "common.cuh"

#include "meshcompact.cuh"

namespace {


__global__ void __launch_bounds__(256) k_face_flags(const float* __restrict__ verts, long long nV, const int32_t* __restrict__ faces,
                                                     long long nF, uint8_t* __restrict__ fkeep, uint8_t* __restrict__ vref) {
  const long long f = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (f >= nF) return;
  const int a = faces[3 * f], b = faces[3 * f + 1], c = faces[3 * f + 2];
  const bool ok = (unsigned)a < (unsigned long long)nV && (unsigned)b < (unsigned long long)nV && (unsigned)c < (unsigned long long)nV &&
                  finite3(verts, a) && finite3(verts, b) && finite3(verts, c);
  fkeep[f] = ok;
  if (ok) { vref[a] = 1; vref[b] = 1; vref[c] = 1; }          // same value from every writer: a benign race
}


// ---- floater removal: connected components of faces that share an undirected edge ---------------------------------
constexpr unsigned long long EDGE_EMPTY = ~0ull;

__device__ __forceinline__ unsigned long long mix64(unsigned long long k) {   // murmur3 finaliser
  k ^= k >> 33; k *= 0xff51afd7ed558ccdull; k ^= k >> 33; k *= 0xc4ceb9fe1a85ec53ull; k ^= k >> 33;
  return k;
}


__device__ __forceinline__ unsigned long long edge_key(int a, int b) {
  return a < b ? ((unsigned long long)a << 32) | (unsigned)b : ((unsigned long long)b << 32) | (unsigned)a;
}

// Slot of edge {a, b} in the open-addressing table; inserts the key if `insert`, else the key must be present.
__device__ __forceinline__ unsigned long long edge_slot(unsigned long long* keys, unsigned long long mask, unsigned long long key,
                                                        bool insert) {
  for (unsigned long long h = mix64(key) & mask;; h = (h + 1) & mask) {
    unsigned long long cur = keys[h];                       // a slot goes EMPTY -> key once: a stale EMPTY is caught by the CAS
    if (insert && cur == EDGE_EMPTY) {
      cur = atomicCAS(keys + h, EDGE_EMPTY, key);
      if (cur == EDGE_EMPTY) return h;
    }
    if (cur == key) return h;
  }
}

// Per face: its three non-degenerate edges into the table, each slot keeping the smallest face id on that edge; parent = self.
__global__ void __launch_bounds__(256) k_edge_insert(const int32_t* __restrict__ faces, long long nF, long long nV,
                                                      unsigned long long* keys, unsigned* __restrict__ minface,
                                                      unsigned long long mask, int* __restrict__ parent, int* __restrict__ err) {
  const long long f = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (f >= nF) return;
  parent[f] = (int)f;
  const int v[3] = {faces[3 * f], faces[3 * f + 1], faces[3 * f + 2]};
  if (!face_in_range(v[0], v[1], v[2], nV)) { *err = 1; return; }
#pragma unroll
  for (int e = 0; e < 3; ++e) {
    const int a = v[e], b = v[(e + 1) % 3];
    if (a != b) atomicMin(minface + edge_slot(keys, mask, edge_key(a, b), true), (unsigned)f);
  }
}

// Union-find with parent[x] <= x: a root is the smallest face id of its tree.  Path halving writes only ancestors.
__device__ __forceinline__ int uf_find(int* parent, int x) {
  int p = __ldcg(parent + x);
  while (p != x) {
    const int g = __ldcg(parent + p);
    if (g != p) parent[x] = g;
    x = p;
    p = g;
  }
  return x;
}

// Read-only walk to the root, used once every union is done: a path-halving write could overwrite a label already stored.
__device__ __forceinline__ int uf_root(const int* parent, int x) {
  for (int p; (p = __ldcg(parent + x)) != x;) x = p;
  return x;
}

__device__ __forceinline__ void uf_union(int* parent, int a, int b) {
  for (;;) {
    a = uf_find(parent, a);
    b = uf_find(parent, b);
    if (a == b) return;
    if (a < b) { const int t = a; a = b; b = t; }
    if (atomicCAS(parent + a, a, b) == a) return;           // hook the larger root under the smaller one
  }
}

__global__ void __launch_bounds__(256) k_edge_union(const int32_t* __restrict__ faces, long long nF, long long nV,
                                                     unsigned long long* keys, const unsigned* __restrict__ minface,
                                                     unsigned long long mask, int* parent) {
  const long long f = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (f >= nF) return;
  const int v[3] = {faces[3 * f], faces[3 * f + 1], faces[3 * f + 2]};
  if (!face_in_range(v[0], v[1], v[2], nV)) return;         // never inserted (k_edge_insert)
#pragma unroll
  for (int e = 0; e < 3; ++e) {
    const int a = v[e], b = v[(e + 1) % 3];
    if (a == b) continue;
    const int g = (int)minface[edge_slot(keys, mask, edge_key(a, b), false)];
    if (g != f) uf_union(parent, (int)f, g);
  }
}

// label = root = smallest face id of the component (independent of scheduling); component sizes, one atomic per label and warp
__global__ void __launch_bounds__(256) k_face_label(long long nF, int* parent, int* __restrict__ size) {
  const long long f = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const unsigned live = __ballot_sync(0xffffffffu, f < nF);   // taken before the finds diverge
  if (f >= nF) return;
  const int r = uf_root(parent, (int)f);
  parent[f] = r;                                            // the only write to parent[] in this kernel: it ends as the labels
  const unsigned same = __match_any_sync(live, r);
  if ((threadIdx.x & 31) == __ffs(same) - 1) atomicAdd(size + r, __popc(same));
}

// vertices of faces in components of fewer than min_faces faces are selected (same value from every writer)
__global__ void __launch_bounds__(256) k_select_small(const int32_t* __restrict__ faces, long long nF, long long nV,
                                                       const int* __restrict__ label, const int* __restrict__ size,
                                                       long long min_faces, uint8_t* __restrict__ vsel) {
  const long long f = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (f >= nF || size[label[f]] >= min_faces) return;
  const int a = faces[3 * f], b = faces[3 * f + 1], c = faces[3 * f + 2];
  if (face_in_range(a, b, c, nV)) { vsel[a] = 1; vsel[b] = 1; vsel[c] = 1; }
}

// a face survives iff none of its vertices is selected; survivors mark their vertices referenced
__global__ void __launch_bounds__(256) k_keep_unselected(const int32_t* __restrict__ faces, long long nF, long long nV,
                                                          const uint8_t* __restrict__ vsel, uint8_t* __restrict__ fkeep,
                                                          uint8_t* __restrict__ vref) {
  const long long f = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (f >= nF) return;
  const int a = faces[3 * f], b = faces[3 * f + 1], c = faces[3 * f + 2];
  const bool ok = face_in_range(a, b, c, nV) && !(vsel[a] | vsel[b] | vsel[c]);
  fkeep[f] = ok;
  if (ok) { vref[a] = 1; vref[b] = 1; vref[c] = 1; }
}

// ---- weld: vertices with bit-equal finite positions (-0.0 == +0.0) -> the smallest such vertex id -------------------
__device__ __forceinline__ bool weld_key(const float* __restrict__ verts, long long v, unsigned k[3]) {
#pragma unroll
  for (int d = 0; d < 3; ++d) {
    const unsigned u = __float_as_uint(verts[3 * v + d]);
    k[d] = u == 0x80000000u ? 0u : u;
  }
  return ((k[0] & 0x7f800000u) != 0x7f800000u) && ((k[1] & 0x7f800000u) != 0x7f800000u) && ((k[2] & 0x7f800000u) != 0x7f800000u);
}

// Table of vertex ids, -1 = empty.  A slot only ever holds ids of one position: it is claimed by CAS and then lowered by
// atomicMin among equal keys, so after this kernel it holds the smallest id of its position.  slot_of[v] = v's slot.
__global__ void __launch_bounds__(256) k_weld_insert(const float* __restrict__ verts, long long nV, int* slots, unsigned long long mask,
                                                      unsigned* __restrict__ slot_of) {
  const long long v = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= nV) return;
  unsigned k[3];
  if (!weld_key(verts, v, k)) return;                       // non-finite: its own representative (k_weld_rep)
  const unsigned long long hk = mix64(((unsigned long long)k[0] << 32 | k[1]) ^ mix64(k[2]));
  for (unsigned long long h = hk & mask;; h = (h + 1) & mask) {
    int cur = slots[h];
    if (cur == -1) {
      cur = atomicCAS(slots + h, -1, (int)v);
      if (cur == -1) { slot_of[v] = (unsigned)h; return; }
    }
    unsigned o[3];
    weld_key(verts, cur, o);
    if (o[0] == k[0] && o[1] == k[1] && o[2] == k[2]) {
      atomicMin(slots + h, (int)v);
      slot_of[v] = (unsigned)h;
      return;
    }
  }
}

__global__ void __launch_bounds__(256) k_weld_rep(const float* __restrict__ verts, long long nV, const int* __restrict__ slots,
                                                   const unsigned* __restrict__ slot_of, int32_t* __restrict__ rep) {
  const long long v = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= nV) return;
  unsigned k[3];
  rep[v] = weld_key(verts, v, k) ? slots[slot_of[v]] : (int32_t)v;
}

// faces rewritten through the representatives; a face with two equal indices is dropped; survivors mark their vertices
__global__ void __launch_bounds__(256) k_weld_faces(const int32_t* __restrict__ faces, long long nF, long long nV,
                                                     const int32_t* __restrict__ rep, int32_t* __restrict__ welded,
                                                     uint8_t* __restrict__ fkeep, uint8_t* __restrict__ vref, int* __restrict__ err) {
  const long long f = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (f >= nF) return;
  const int a = faces[3 * f], b = faces[3 * f + 1], c = faces[3 * f + 2];
  if (!face_in_range(a, b, c, nV)) { *err = 1; fkeep[f] = 0; return; }
  const int ra = rep[a], rb = rep[b], rc = rep[c];
  welded[3 * f] = ra; welded[3 * f + 1] = rb; welded[3 * f + 2] = rc;
  const bool ok = ra != rb && rb != rc && ra != rc;
  fkeep[f] = ok;
  if (ok) { vref[ra] = 1; vref[rb] = 1; vref[rc] = 1; }
}


// Arguments of the floater and weld entry points.  Returns HY3D_OK to proceed, 1 for an empty result (counts already 0).
int check_mesh_args(hy3d_ctx* ctx, const float* d_verts, long long nV, const int32_t* d_faces, long long nF, const float* d_verts_out,
                    const int32_t* d_faces_out, int64_t* h_nv_out, int64_t* h_nf_out) {
  if (!ctx || nV < 0 || nF < 0 || !h_nv_out || !h_nf_out) return HY3D_ERR_ARG;
  *h_nv_out = 0; *h_nf_out = 0;
  if (nF == 0) return 1;
  if (nV == 0) return hy3d_fail(ctx, HY3D_ERR_ARG, "face index outside [0, 0)");
  if (!d_verts || !d_faces || !d_verts_out || !d_faces_out) return HY3D_ERR_ARG;
  if (nV > 2147483647LL) return hy3d_fail(ctx, HY3D_ERR_UNSUPPORTED, "vertex ids exceed int32");
  if (nF > 2147483647LL) return hy3d_fail(ctx, HY3D_ERR_UNSUPPORTED, "face ids exceed int32");
  return HY3D_OK;
}

unsigned long long pow2_at_least(unsigned long long n) {
  unsigned long long c = 1024;
  while (c < n) c <<= 1;
  return c;
}

}  // namespace

extern "C" int hy3d_mesh_clean(hy3d_ctx* ctx, const float* d_verts, int64_t nV, const int32_t* d_faces, int64_t nF, int32_t flip_winding,
                               float* d_verts_out, int32_t* d_faces_out, int64_t* h_nv_out, int64_t* h_nf_out) {
  if (!ctx || nV < 0 || nF < 0 || !h_nv_out || !h_nf_out) return HY3D_ERR_ARG;
  *h_nv_out = 0; *h_nf_out = 0;
  if (nV == 0 || nF == 0) return HY3D_OK;
  if (!d_verts || !d_faces || !d_verts_out || !d_faces_out) return HY3D_ERR_ARG;
  if (nV > 2147483647LL) return hy3d_fail(ctx, HY3D_ERR_UNSUPPORTED, "vertex ids exceed int32");
  HY3D_CUDA(ctx, cudaSetDevice(ctx->device));
  Compaction cp;
  int rc = carve_scratch(ctx, nV, nF, cp, [](Carver&) {});
  if (rc) return rc;
  HY3D_CUDA(ctx, cudaMemsetAsync(cp.vref, 0, nV, ctx->stream));
  HY3D_PROF(ctx, FAM_MC_EMIT);
  k_face_flags<<<(unsigned)ceil_div64(nF, 256), 256, 0, ctx->stream>>>(d_verts, nV, d_faces, nF, cp.fkeep, cp.vref);
  HY3D_LAUNCH_CHECK(ctx);
  return compact(ctx, cp, d_verts, nV, d_faces, nF, flip_winding ? 1 : 0, nullptr, d_verts_out, d_faces_out, h_nv_out, h_nf_out);
}

extern "C" int hy3d_mesh_remove_floaters(hy3d_ctx* ctx, const float* d_verts, int64_t nV, const int32_t* d_faces, int64_t nF,
                                         int64_t min_faces, float* d_verts_out, int32_t* d_faces_out, int64_t* h_nv_out,
                                         int64_t* h_nf_out) {
  int rc = check_mesh_args(ctx, d_verts, nV, d_faces, nF, d_verts_out, d_faces_out, h_nv_out, h_nf_out);
  if (rc) return rc > 0 ? HY3D_OK : rc;
  if (min_faces < 0) return hy3d_fail(ctx, HY3D_ERR_ARG, "min_faces < 0");
  HY3D_CUDA(ctx, cudaSetDevice(ctx->device));
  const unsigned long long cap = pow2_at_least(6ull * (unsigned long long)nF);     // >= 2x the 3F half-edges
  Compaction cp;
  unsigned long long* keys;
  unsigned* minface;
  int *parent, *size, *err;
  uint8_t* vsel;
  rc = carve_scratch(ctx, nV, nF, cp, [&](Carver& c) {
    keys = c.take<unsigned long long>(cap); minface = c.take<unsigned>(cap);        // adjacent: one 0xff fill
    size = c.take<int>(nF); vsel = c.take<uint8_t>(nV); err = c.take<int>(1);
    parent = c.take<int>(nF);
  });
  if (rc) return rc;
  const size_t zero_bytes = reinterpret_cast<char*>(parent) - reinterpret_cast<char*>(size);   // size, vsel, err
  HY3D_CUDA(ctx, cudaMemsetAsync(keys, 0xff, reinterpret_cast<char*>(size) - reinterpret_cast<char*>(keys), ctx->stream));
  HY3D_CUDA(ctx, cudaMemsetAsync(size, 0, zero_bytes, ctx->stream));
  HY3D_CUDA(ctx, cudaMemsetAsync(cp.vref, 0, nV, ctx->stream));
  const unsigned gF = (unsigned)ceil_div64(nF, 256);
  HY3D_PROF(ctx, FAM_MC_EMIT);
  k_edge_insert<<<gF, 256, 0, ctx->stream>>>(d_faces, nF, nV, keys, minface, cap - 1, parent, err);
  HY3D_LAUNCH_CHECK(ctx);
  HY3D_PROF(ctx, FAM_MC_EMIT);
  k_edge_union<<<gF, 256, 0, ctx->stream>>>(d_faces, nF, nV, keys, minface, cap - 1, parent);
  HY3D_LAUNCH_CHECK(ctx);
  HY3D_PROF(ctx, FAM_MC_EMIT);
  k_face_label<<<gF, 256, 0, ctx->stream>>>(nF, parent, size);
  HY3D_LAUNCH_CHECK(ctx);
  HY3D_PROF(ctx, FAM_MC_EMIT);
  k_select_small<<<gF, 256, 0, ctx->stream>>>(d_faces, nF, nV, parent, size, (long long)min_faces, vsel);
  HY3D_LAUNCH_CHECK(ctx);
  HY3D_PROF(ctx, FAM_MC_EMIT);
  k_keep_unselected<<<gF, 256, 0, ctx->stream>>>(d_faces, nF, nV, vsel, cp.fkeep, cp.vref);
  HY3D_LAUNCH_CHECK(ctx);
  return compact(ctx, cp, d_verts, nV, d_faces, nF, 0, err, d_verts_out, d_faces_out, h_nv_out, h_nf_out);
}

extern "C" int hy3d_mesh_weld(hy3d_ctx* ctx, const float* d_verts, int64_t nV, const int32_t* d_faces, int64_t nF, float* d_verts_out,
                              int32_t* d_faces_out, int64_t* h_nv_out, int64_t* h_nf_out) {
  int rc = check_mesh_args(ctx, d_verts, nV, d_faces, nF, d_verts_out, d_faces_out, h_nv_out, h_nf_out);
  if (rc) return rc > 0 ? HY3D_OK : rc;
  HY3D_CUDA(ctx, cudaSetDevice(ctx->device));
  const unsigned long long cap = pow2_at_least(2ull * (unsigned long long)nV);     // <= 2^32: slot ids fit in 32 bits
  Compaction cp;
  int *slots, *err;
  unsigned* slot_of;
  int32_t *rep, *welded;
  rc = carve_scratch(ctx, nV, nF, cp, [&](Carver& c) {
    slots = c.take<int>(cap); slot_of = c.take<unsigned>(nV); rep = c.take<int32_t>(nV); welded = c.take<int32_t>(3 * (size_t)nF);
    err = c.take<int>(1);
  });
  if (rc) return rc;
  HY3D_CUDA(ctx, cudaMemsetAsync(slots, 0xff, cap * sizeof(int), ctx->stream));
  HY3D_CUDA(ctx, cudaMemsetAsync(err, 0, sizeof(int), ctx->stream));
  HY3D_CUDA(ctx, cudaMemsetAsync(cp.vref, 0, nV, ctx->stream));
  const unsigned gV = (unsigned)ceil_div64(nV, 256), gF = (unsigned)ceil_div64(nF, 256);
  HY3D_PROF(ctx, FAM_MC_EMIT);
  k_weld_insert<<<gV, 256, 0, ctx->stream>>>(d_verts, nV, slots, cap - 1, slot_of);
  HY3D_LAUNCH_CHECK(ctx);
  HY3D_PROF(ctx, FAM_MC_EMIT);
  k_weld_rep<<<gV, 256, 0, ctx->stream>>>(d_verts, nV, slots, slot_of, rep);
  HY3D_LAUNCH_CHECK(ctx);
  HY3D_PROF(ctx, FAM_MC_EMIT);
  k_weld_faces<<<gF, 256, 0, ctx->stream>>>(d_faces, nF, nV, rep, welded, cp.fkeep, cp.vref, err);
  HY3D_LAUNCH_CHECK(ctx);
  return compact(ctx, cp, d_verts, nV, welded, nF, 0, err, d_verts_out, d_faces_out, h_nv_out, h_nf_out);
}
