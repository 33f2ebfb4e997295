// Order-preserving compaction of a mesh (block counts -> scan -> emit) and the scratch layout shared by the mesh
// filters of meshclean.cu and decimate.cu (each translation unit gets its own copy of these kernels).
#pragma once
#include "common.cuh"

namespace {

constexpr int CL_BLOCK = 1024;

__device__ __forceinline__ bool finite3(const float* __restrict__ v, long long i) {
  const float x = v[3 * i], y = v[3 * i + 1], z = v[3 * i + 2];
  return (fabsf(x) <= 3.402823466e38f) && (fabsf(y) <= 3.402823466e38f) && (fabsf(z) <= 3.402823466e38f);   // false for NaN / inf
}

// blockIdx.y = 0: vertices (keep = referenced; a referenced vertex is finite by construction), 1: faces
__global__ void __launch_bounds__(256) k_keep_counts(const uint8_t* __restrict__ vref, long long nV, const uint8_t* __restrict__ fkeep,
                                                      long long nF, int* __restrict__ cntV, int* __restrict__ cntF) {
  const uint8_t* src = blockIdx.y ? fkeep : vref;
  const long long n = blockIdx.y ? nF : nV;
  const long long base = (long long)blockIdx.x * CL_BLOCK;
  if (base >= n) return;
  int c = 0;
  for (int t = threadIdx.x; t < CL_BLOCK; t += 256) c += (base + t < n) ? src[base + t] : 0;
  __shared__ int red[8];
  for (int o = 16; o; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = c;
  __syncthreads();
  if (threadIdx.x == 0) {
    int s = 0;
    for (int w = 0; w < 8; ++w) s += red[w];
    (blockIdx.y ? cntF : cntV)[blockIdx.x] = s;
  }
}

// exclusive scan of n counts by one block per array (blockIdx.x selects it); out[n] = total
__global__ void __launch_bounds__(1024) k_scan_counts(const int* __restrict__ in0, int n0, long long* __restrict__ out0,
                                                       const int* __restrict__ in1, int n1, long long* __restrict__ out1) {
  const int* in = blockIdx.x ? in1 : in0;
  long long* out = blockIdx.x ? out1 : out0;
  const int n = blockIdx.x ? n1 : n0;
  __shared__ long long part[1024];
  const int tid = threadIdx.x, per = (n + 1023) / 1024, lo = tid * per, hi = min(lo + per, n);
  long long s = 0;
  for (int i = lo; i < hi; ++i) s += in[i];
  part[tid] = s;
  __syncthreads();
  for (int off = 1; off < 1024; off <<= 1) {
    long long v = tid >= off ? part[tid - off] : 0;
    __syncthreads();
    part[tid] += v;
    __syncthreads();
  }
  long long run = tid ? part[tid - 1] : 0;
  for (int i = lo; i < hi; ++i) { out[i] = run; run += in[i]; }
  if (tid == 1023) out[n] = part[1023];
}

// block-local exclusive scan of 1024 keep flags (4 per thread) + the block's offset -> new position of every kept element
__device__ __forceinline__ void block_positions(const uint8_t* __restrict__ keep, long long base, long long n, long long blockoff,
                                                bool k[4], long long pos[4]) {
  __shared__ int wsum[8];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int c = 0;
#pragma unroll
  for (int u = 0; u < 4; ++u) { const long long e = base + threadIdx.x * 4 + u; k[u] = e < n && keep[e]; c += k[u]; }
  int incl = c;
  for (int o = 1; o < 32; o <<= 1) { int t = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += t; }
  if (lane == 31) wsum[warp] = incl;
  __syncthreads();
  long long p = blockoff + incl - c;
  for (int w = 0; w < warp; ++w) p += wsum[w];
#pragma unroll
  for (int u = 0; u < 4; ++u) { pos[u] = p; p += k[u]; }
  __syncthreads();
}

// WITH_Q: the per-vertex quadrics qin (10 doubles per vertex) are carried along with the positions to qout (decimate.cu)
template <bool WITH_Q>
__global__ void __launch_bounds__(256) k_emit_verts(const float* __restrict__ verts, long long nV, const uint8_t* __restrict__ vref,
                                                     const long long* __restrict__ offV, float* __restrict__ out, int32_t* __restrict__ remap,
                                                     const double* __restrict__ qin, double* __restrict__ qout) {
  const long long base = (long long)blockIdx.x * CL_BLOCK;
  bool k[4]; long long pos[4];
  block_positions(vref, base, nV, offV[blockIdx.x], k, pos);
#pragma unroll
  for (int u = 0; u < 4; ++u) {
    const long long e = base + threadIdx.x * 4 + u;
    if (e >= nV) continue;
    remap[e] = k[u] ? (int32_t)pos[u] : -1;
    if (k[u]) { out[3 * pos[u]] = verts[3 * e]; out[3 * pos[u] + 1] = verts[3 * e + 1]; out[3 * pos[u] + 2] = verts[3 * e + 2]; }
    if (WITH_Q && k[u]) {
#pragma unroll
      for (int j = 0; j < 10; ++j) qout[10 * pos[u] + j] = qin[10 * e + j];
    }
  }
}

__global__ void __launch_bounds__(256) k_emit_faces(const int32_t* __restrict__ faces, long long nF, const uint8_t* __restrict__ fkeep,
                                                     const long long* __restrict__ offF, const int32_t* __restrict__ remap, int flip,
                                                     int32_t* __restrict__ out) {
  const long long base = (long long)blockIdx.x * CL_BLOCK;
  bool k[4]; long long pos[4];
  block_positions(fkeep, base, nF, offF[blockIdx.x], k, pos);
#pragma unroll
  for (int u = 0; u < 4; ++u) {
    const long long e = base + threadIdx.x * 4 + u;
    if (e >= nF || !k[u]) continue;
    const int a = remap[faces[3 * e]], b = remap[faces[3 * e + 1]], c = remap[faces[3 * e + 2]];
    out[3 * pos[u]] = flip ? c : a; out[3 * pos[u] + 1] = b; out[3 * pos[u] + 2] = flip ? a : c;
  }
}

__device__ __forceinline__ bool face_in_range(int a, int b, int c, long long nV) {
  return (unsigned)a < (unsigned long long)nV && (unsigned)b < (unsigned long long)nV && (unsigned)c < (unsigned long long)nV;
}

// ---- scratch layout and the order-preserving compaction shared by the three entry points --------------------------
struct Carver {                                             // 256-byte aligned pieces of one scratch allocation
  uintptr_t base;
  size_t off = 0;
  template <class T> T* take(size_t n) {
    T* p = reinterpret_cast<T*>(base + off);
    off += (n * sizeof(T) + 255) / 256 * 256;
    return p;
  }
};

struct Compaction {
  uint8_t* vref;       // [nV] vertex kept (referenced by a kept face)
  uint8_t* fkeep;      // [nF] face kept
  int32_t* remap;      // [nV] old -> new vertex id
  int *cntV, *cntF;    // per CL_BLOCK block
  long long *offV, *offF;
  int nbV, nbF;
  void sizes(long long nV, long long nF) { nbV = (int)ceil_div64(nV, CL_BLOCK); nbF = (int)ceil_div64(nF, CL_BLOCK); }
  void carve(Carver& c, long long nV, long long nF) {
    sizes(nV, nF);
    vref = c.take<uint8_t>(nV); fkeep = c.take<uint8_t>(nF); remap = c.take<int32_t>(nV);
    cntV = c.take<int>(nbV); cntF = c.take<int>(nbF); offV = c.take<long long>(nbV + 1); offF = c.take<long long>(nbF + 1);
  }
};

// Lays out the compaction buffers and then whatever `more` takes, in one grow-only scratch allocation.
template <class F>
int carve_scratch(hy3d_ctx* ctx, long long nV, long long nF, Compaction& cp, F&& more) {
  Carver dry{0};
  cp.carve(dry, nV, nF);
  more(dry);
  HY3D_CUDA(ctx, ctx->scratch.reserve(dry.off));
  Carver c{reinterpret_cast<uintptr_t>(ctx->scratch.p)};
  cp.carve(c, nV, nF);
  more(c);
  return HY3D_OK;
}

// vref / fkeep set: counts -> scan -> emit (faces read from `faces`, re-indexed, optionally flipped; quadrics d_q carried to
// d_q_out when given), then the one host synchronisation, which also reads back the device error flag `d_err` (may be null).
int compact(hy3d_ctx* ctx, const Compaction& cp, const float* d_verts, long long nV, const int32_t* d_faces, long long nF, int flip,
            const int* d_err, float* d_verts_out, int32_t* d_faces_out, int64_t* h_nv_out, int64_t* h_nf_out,
            const double* d_q = nullptr, double* d_q_out = nullptr) {
  HY3D_PROF(ctx, FAM_MC_EMIT);
  k_keep_counts<<<dim3((unsigned)(cp.nbV > cp.nbF ? cp.nbV : cp.nbF), 2), 256, 0, ctx->stream>>>(cp.vref, nV, cp.fkeep, nF, cp.cntV,
                                                                                              cp.cntF);
  HY3D_LAUNCH_CHECK(ctx);
  HY3D_PROF(ctx, FAM_MC_SCAN);
  k_scan_counts<<<2, 1024, 0, ctx->stream>>>(cp.cntV, cp.nbV, cp.offV, cp.cntF, cp.nbF, cp.offF);
  HY3D_LAUNCH_CHECK(ctx);
  HY3D_PROF(ctx, FAM_MC_EMIT);
  if (d_q) k_emit_verts<true><<<cp.nbV, 256, 0, ctx->stream>>>(d_verts, nV, cp.vref, cp.offV, d_verts_out, cp.remap, d_q, d_q_out);
  else k_emit_verts<false><<<cp.nbV, 256, 0, ctx->stream>>>(d_verts, nV, cp.vref, cp.offV, d_verts_out, cp.remap, nullptr, nullptr);
  HY3D_LAUNCH_CHECK(ctx);
  HY3D_PROF(ctx, FAM_MC_EMIT);
  k_emit_faces<<<cp.nbF, 256, 0, ctx->stream>>>(d_faces, nF, cp.fkeep, cp.offF, cp.remap, flip, d_faces_out);
  HY3D_LAUNCH_CHECK(ctx);
  long long* pl = reinterpret_cast<long long*>(ctx->pinned);
  HY3D_CUDA(ctx, cudaMemcpyAsync(pl, cp.offV + cp.nbV, 8, cudaMemcpyDeviceToHost, ctx->stream));
  HY3D_CUDA(ctx, cudaMemcpyAsync(pl + 1, cp.offF + cp.nbF, 8, cudaMemcpyDeviceToHost, ctx->stream));
  int* perr = reinterpret_cast<int*>(pl + 2);
  *perr = 0;
  if (d_err) HY3D_CUDA(ctx, cudaMemcpyAsync(perr, d_err, 4, cudaMemcpyDeviceToHost, ctx->stream));
  HY3D_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  if (*perr) return hy3d_fail(ctx, HY3D_ERR_ARG, "face index outside [0, %lld)", nV);
  *h_nv_out = pl[0]; *h_nf_out = pl[1];
  return HY3D_OK;
}

}  // namespace
