// Pieces of the marching-cubes count phase shared by mc.cu and dmc.cu: the bit-grid classify pass, the bit-row
// edge masks and the scans of the per-row counts.
#pragma once
#include <cfloat>

#include "common.cuh"

namespace {

__device__ __forceinline__ int f2ord(float f) { int i = __float_as_int(f); return i >= 0 ? i : i ^ 0x7fffffff; }
__host__ __device__ __forceinline__ float ord2f(int i) {
  int b = i >= 0 ? i : i ^ 0x7fffffff;
#ifdef __CUDA_ARCH__
  return __int_as_float(b);
#else
  float f; memcpy(&f, &b, 4); return f;
#endif
}

constexpr int BITS_WARPS = 8;
constexpr int BITS_T = 32;         // 32-voxel words per warp iteration: 32 independent 128 B loads in flight per warp (4 KB)

// The field is streamed as ONE flat array (no row structure, no integer division): lane l of a warp
// loads elements 32*t + l of its 1024-element chunk, so every request is a full 128-byte line and one
// ballot yields one word of the flat bitstream (bit e of the stream = voxel with flat index e); lane t keeps
// word t, so the chunk's 32 words leave as one coalesced 128-byte store.
// Row-aligned words are recovered later by a funnel shift (load_bits).
// "v - level > 0" (skimage) is evaluated as v > level: identical for every pair of floats (gradual underflow keeps
// v - level != 0 when v != level; NaN compares false either way).  fminf / fmaxf drop NaN operands, so the extrema
// need no branch; the NaN flag is one compare per element.
// stats: [0] ordered-int min, [1] ordered-int max, [2] nan flag.
__global__ void __launch_bounds__(BITS_WARPS * 32) k_mc_bits(const float* __restrict__ grid, long long total, float level,
                                                             uint32_t* __restrict__ bits, long long nwords, int* __restrict__ stats) {
  const int lane = threadIdx.x & 31;
  const long long warp0 = (long long)blockIdx.x * BITS_WARPS + (threadIdx.x >> 5);
  const long long nwarps = (long long)gridDim.x * BITS_WARPS;
  const long long nchunks = (nwords + BITS_T - 1) / BITS_T;
  const long long nfull = total / (BITS_T * 32);          // chunks that lie entirely inside the field
  float mn = INFINITY, mx = -INFINITY; int nanf = 0;
  for (long long c = warp0; c < nchunks; c += nwarps) {
    const float* src = grid + c * (BITS_T * 32) + lane;
    float v[BITS_T];
    if (c < nfull) {
#pragma unroll
      for (int t = 0; t < BITS_T; ++t) v[t] = __ldcs(src + t * 32);          // streamed once: evict-first
    } else {
      const long long e0 = c * (BITS_T * 32) + lane;
#pragma unroll
      for (int t = 0; t < BITS_T; ++t) v[t] = (e0 + t * 32 < total) ? __ldcs(src + t * 32) : -INFINITY;   // padding: bit 0, no effect on max
    }
    uint32_t mine = 0;
#pragma unroll
    for (int t = 0; t < BITS_T; ++t) {
      const uint32_t m = __ballot_sync(0xffffffffu, v[t] > level);
      if (lane == t) mine = m;
      nanf |= (v[t] != v[t]);
      mx = fmaxf(mx, v[t]);
    }
    if (c < nfull) {
#pragma unroll
      for (int t = 0; t < BITS_T; ++t) mn = fminf(mn, v[t]);
    } else {
      const long long e0 = c * (BITS_T * 32) + lane;
#pragma unroll
      for (int t = 0; t < BITS_T; ++t) if (e0 + t * 32 < total) mn = fminf(mn, v[t]);
    }
    if (c * BITS_T + lane < nwords) bits[c * BITS_T + lane] = mine;
  }
  for (int o = 16; o; o >>= 1) {
    mn = fminf(mn, __shfl_xor_sync(0xffffffffu, mn, o));
    mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    nanf |= __shfl_xor_sync(0xffffffffu, nanf, o);
  }
  __shared__ float smn[BITS_WARPS], smx[BITS_WARPS];
  __shared__ int snan[BITS_WARPS];
  if (lane == 0) { smn[threadIdx.x >> 5] = mn; smx[threadIdx.x >> 5] = mx; snan[threadIdx.x >> 5] = nanf; }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < BITS_WARPS; ++w) { mn = fminf(mn, smn[w]); mx = fmaxf(mx, smx[w]); nanf |= snan[w]; }
    // same-address atomics serialise in L2: only blocks that improve the running extrema issue one
    if (mn <= mx) {
      if (f2ord(mn) < *(volatile int*)&stats[0]) atomicMin(&stats[0], f2ord(mn));
      if (f2ord(mx) > *(volatile int*)&stats[1]) atomicMax(&stats[1], f2ord(mx));
    }
    if (nanf && !*(volatile int*)&stats[2]) atomicOr(&stats[2], 1);
  }
}

struct RowMasks { uint32_t m0, m1, m2; };

// bit k of result = x[k+1] (x_next supplies bit 0 of the following word)
__device__ __forceinline__ uint32_t shl1(uint32_t x, uint32_t x_next) { return (x >> 1) | (x_next << 31); }

// word w (voxels 32w .. 32w+31) of row (i,j), cut out of the flat bitstream; bits past the row end are 0
__device__ __forceinline__ uint32_t load_bits(const uint32_t* __restrict__ bits, int n0, int n1, int n2, int i, int j, int w) {
  if (i >= n0 || j >= n1 || w * 32 >= n2) return 0u;
  const long long start = ((long long)i * n1 + j) * n2 + w * 32;
  const long long idx = start >> 5;
  const int sh = (int)(start & 31);
  const uint32_t lo = __ldg(bits + idx), hi = __ldg(bits + idx + 1);      // the stream is padded by two zero words
  uint32_t v = __funnelshift_r(lo, hi, sh);
  const int valid = n2 - w * 32;
  if (valid < 32) v &= (1u << valid) - 1u;
  return v;
}

// A bit row of n2 voxels is handled by LPR lanes (word = lane % LPR), LPR = 8, 16 or 32 >= words per row: a warp works on
// 32 / LPR rows at once (385^3: 13 words -> 2 rows per warp; <= 256 voxels: 4 rows) instead of idling the lanes past the row.
// All shuffles use `width = LPR` segments; every lane of the warp executes them (inactive rows carry zero masks).
template <int LPR>
__device__ __forceinline__ uint32_t next_word(uint32_t x) {        // word (lane + 1) of the same row, 0 past the segment
  const uint32_t n = __shfl_down_sync(0xffffffffu, x, 1, LPR);
  return ((threadIdx.x & (LPR - 1)) == LPR - 1) ? 0u : n;
}

// sign-change edge masks of row (i,j), word = lane % LPR.  r = this row, rj = row (i,j+1), ri = row (i+1,j).
template <int LPR>
__device__ __forceinline__ RowMasks edge_masks(uint32_t r, uint32_t rj, uint32_t ri, bool has_j, bool has_i, uint32_t inrow,
                                               uint32_t validk) {
  const uint32_t rn = next_word<LPR>(r);
  RowMasks m;
  m.m2 = (r ^ shl1(r, rn)) & validk;
  m.m1 = has_j ? ((r ^ rj) & inrow) : 0u;
  m.m0 = has_i ? ((r ^ ri) & inrow) : 0u;
  return m;
}

template <int LPR>
__device__ __forceinline__ int seg_excl_scan(int v) {              // exclusive scan inside each LPR-lane segment
  int incl = v;
  const int sub = threadIdx.x & (LPR - 1);
#pragma unroll
  for (int o = 1; o < LPR; o <<= 1) { int t = __shfl_up_sync(0xffffffffu, incl, o, LPR); if (sub >= o) incl += t; }
  return incl - v;
}

__device__ __forceinline__ int cube_case(uint32_t a, uint32_t sa, uint32_t b, uint32_t sb, uint32_t c, uint32_t sc, uint32_t d,
                                         uint32_t sd, int k) {
  return ((a >> k) & 1) | (((sa >> k) & 1) << 1) | (((sb >> k) & 1) << 2) | (((b >> k) & 1) << 3) | (((c >> k) & 1) << 4) |
         (((sc >> k) & 1) << 5) | (((sd >> k) & 1) << 6) | (((d >> k) & 1) << 7);
}

// Exclusive scans of the two per-row count arrays (blockIdx.y selects the array), three small launches:
// per-4096-chunk local scans + chunk sums, scan of the chunk sums, offset add.  out[n] = total.
constexpr int SCAN_CHUNK = 4096;

__device__ __forceinline__ long long block_excl_scan_1024(long long v, long long* total) {
  __shared__ long long wsum[32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  long long incl = v;
  for (int o = 1; o < 32; o <<= 1) { long long t = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += t; }
  __syncthreads();
  if (lane == 31) wsum[warp] = incl;
  __syncthreads();
  if (warp == 0) {
    long long w = wsum[lane], wi = w;
    for (int o = 1; o < 32; o <<= 1) { long long t = __shfl_up_sync(0xffffffffu, wi, o); if (lane >= o) wi += t; }
    wsum[lane] = wi - w;
    if (lane == 31) *total = wi;
  }
  __syncthreads();
  return incl - v + wsum[warp];
}

__global__ void __launch_bounds__(1024) k_scan_local(const int* __restrict__ in0, const int* __restrict__ in1, int n,
                                                     long long* __restrict__ out0, long long* __restrict__ out1,
                                                     long long* __restrict__ csum, int nchunks) {
  const int* in = blockIdx.y ? in1 : in0;
  long long* out = blockIdx.y ? out1 : out0;
  __shared__ long long tot;
  const int base = blockIdx.x * SCAN_CHUNK + threadIdx.x * 4;
  int v[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) v[i] = base + i < n ? in[base + i] : 0;
  const long long mine = (long long)v[0] + v[1] + v[2] + v[3];
  long long ex = block_excl_scan_1024(mine, &tot);
#pragma unroll
  for (int i = 0; i < 4; ++i) { if (base + i < n) out[base + i] = ex; ex += v[i]; }
  if (threadIdx.x == 0) csum[blockIdx.y * nchunks + blockIdx.x] = tot;
}

__global__ void __launch_bounds__(1024) k_scan_chunks(long long* __restrict__ csum, int nchunks, long long* __restrict__ out0,
                                                      long long* __restrict__ out1, int n) {
  long long* cs = csum + blockIdx.x * nchunks;
  long long* out = blockIdx.x ? out1 : out0;
  __shared__ long long tot;
  long long carry = 0;
  for (int c0 = 0; c0 < nchunks; c0 += 1024) {
    const int c = c0 + threadIdx.x;
    const long long v = c < nchunks ? cs[c] : 0;
    const long long ex = block_excl_scan_1024(v, &tot);
    if (c < nchunks) cs[c] = carry + ex;
    carry += tot;
    __syncthreads();
  }
  if (threadIdx.x == 0) out[n] = carry;
}

__global__ void __launch_bounds__(1024) k_scan_add(long long* __restrict__ out0, long long* __restrict__ out1,
                                                   const long long* __restrict__ csum, int nchunks, int n) {
  long long* out = blockIdx.y ? out1 : out0;
  const long long off = csum[blockIdx.y * nchunks + blockIdx.x];
  const int base = blockIdx.x * SCAN_CHUNK + threadIdx.x * 4;
#pragma unroll
  for (int i = 0; i < 4; ++i) if (base + i < n) out[base + i] += off;
}

}  // namespace
