// Coarse-to-fine octree refinement: replaces extract_near_surface_volume_fn + the Conv3d
// dilations + torch.where of the reference (volume_decoders.py:29-119, :245-260, :376-391;
// restated in SURVEY App. B).  All integer/bit work, HBM/L2-bound: the coarse grid is read once, everything after that
// happens on bit rows (1 bit per voxel, rows padded to 32-bit words), no float grids, no byte masks, no host round trips
// except the final count.
//
//   coarse grid G[n^3] --k_coarse_bits--> act bits [n*n rows][ceil(n/32)]                     (near-surface | band mask)
//   [not last level]   --k_dilate_bits--> 3x3x3 box dilation in bit space (word-parallel shifts / ORs of 9 rows)
//   fine mask: the x2 up-sampling followed by 1 or 2 box dilations collapses to "any active coarse voxel c with
//   |2c - f|_inf <= r" (r = 1 or 2).  Along k that is, for a whole 32-voxel fine word at once,
//       even f = 2m: a[m] (r = 1) or a[m-1] | a[m] | a[m+1] (r = 2);   odd f = 2m+1: a[m] | a[m+1]
//   on the 18 coarse bits under the word, bit-interleaved back to 32 fine bits; along i and j the same rule picks 1-3
//   coarse rows per axis, OR-ed before the k rule.                --k_fine_words--> fine bits [nf*nf rows][ceil(nf/32)]
//   --k_scan_i32--> offsets of 256-word blocks --k_words_emit--> ordered flat indices (torch.where order)
#include "common.cuh"

namespace {

__device__ __forceinline__ int sgn(float v) { return (v > 0.f) - (v < 0.f); }

// one block per coarse row (i, j), one thread per k (blockDim = 32 * words per row): 1 bit per voxel
__global__ void k_coarse_bits(const float* __restrict__ g, int n, int wpr, float alpha, uint32_t* __restrict__ act) {
  const int row = blockIdx.x, i = row / n, j = row - i * n, k = threadIdx.x;
  bool on = false;
  if (k < n) {
    const long long t = (long long)row * n + k;
    const float gv = g[t];
    const float val = __fadd_rn(gv, alpha);
    const bool valid = val > -9000.f;
    const int s = sgn(val);
    bool diff = false;
    const long long sn[3] = {(long long)n * n, n, 1};
    const int idx[3] = {i, j, k};
#pragma unroll
    for (int a = 0; a < 3; ++a) {
#pragma unroll
      for (int d = -1; d <= 1; d += 2) {
        int c = idx[a] + d;
        c = c < 0 ? 0 : (c > n - 1 ? n - 1 : c);                 // replicate padding
        float nb = __fadd_rn(g[t + (long long)(c - idx[a]) * sn[a]], alpha);
        if (!(nb > -9000.f)) nb = val;                           // invalid neighbour -> own value
        diff |= sgn(nb) != s;
      }
    }
    on = (diff && valid) || (fabsf(gv) < HY3D_BAND);
  }
  const uint32_t m = __ballot_sync(0xffffffffu, on);
  if ((threadIdx.x & 31) == 0) act[(size_t)row * wpr + (threadIdx.x >> 5)] = m;
}

// 3x3x3 box dilation on bit rows (zero beyond the grid): thread per (row, word)
__global__ void k_dilate_bits(const uint32_t* __restrict__ in, int n, int wpr, uint32_t* __restrict__ out) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (long long)n * n * wpr) return;
  const int w = (int)(t % wpr); const int row = (int)(t / wpr); const int i = row / n, j = row - i * n;
  uint32_t x = 0, l = 0, r = 0;
  for (int a = max(i - 1, 0); a <= min(i + 1, n - 1); ++a)
    for (int b = max(j - 1, 0); b <= min(j + 1, n - 1); ++b) {
      const uint32_t* p = in + ((size_t)a * n + b) * wpr;
      x |= p[w];
      if (w > 0) l |= p[w - 1];
      if (w + 1 < wpr) r |= p[w + 1];
    }
  uint32_t d = x | (x << 1) | (x >> 1) | (l >> 31) | (r << 31);
  const int valid = n - w * 32;
  if (valid < 32) d &= (1u << valid) - 1u;
  out[t] = d;
}

__device__ __forceinline__ uint32_t spread16(uint32_t x) {      // bit s of x -> bit 2s
  x &= 0xFFFFu;
  x = (x | (x << 8)) & 0x00FF00FFu;
  x = (x | (x << 4)) & 0x0F0F0F0Fu;
  x = (x | (x << 2)) & 0x33333333u;
  x = (x | (x << 1)) & 0x55555555u;
  return x;
}

constexpr int FW_BLOCK = 256;                      // fine words per block (= per scan element)

// thread per fine word (fine row (fi, fj), word w): 32 fine voxels from the 18 coarse bits under them, OR-ed over the
// coarse rows within reach in i and j.  Also the block's population count for the ordered compaction.
__global__ void __launch_bounds__(FW_BLOCK) k_fine_words(const uint32_t* __restrict__ act, int n, int wpr_c, int nf, int wpr_f,
                                                          int reach, long long nwords, uint32_t* __restrict__ words,
                                                          int* __restrict__ blockcnt) {
  const long long L = (long long)blockIdx.x * FW_BLOCK + threadIdx.x;
  uint32_t out = 0;
  if (L < nwords) {
    const int w = (int)(L % wpr_f); const int row = (int)(L / wpr_f); const int fi = row / nf, fj = row - fi * nf;
    // coarse index range per axis: ceil((f - reach) / 2) .. floor((f + reach) / 2), clipped
    int lo[2], hi[2];
    const int f2[2] = {fi, fj};
#pragma unroll
    for (int a = 0; a < 2; ++a) {
      const int l = f2[a] - reach, h = f2[a] + reach;
      lo[a] = l <= 0 ? 0 : (l + 1) >> 1;
      hi[a] = min(h >> 1, n - 1);
    }
    const int start = 16 * w - 1;                  // window bit t <-> coarse k = start + t, t = 0 .. 17
    uint32_t a18 = 0;
    for (int ci = lo[0]; ci <= hi[0]; ++ci)
      for (int cj = lo[1]; cj <= hi[1]; ++cj) {
        const uint32_t* p = act + ((size_t)ci * n + cj) * wpr_c;
        uint32_t win;
        if (start < 0) win = p[0] << 1;
        else {
          const int idx = start >> 5, sh = start & 31;
          const uint32_t w0 = p[idx], w1 = idx + 1 < wpr_c ? p[idx + 1] : 0u;
          win = __funnelshift_r(w0, w1, sh);
        }
        a18 |= win;
      }
    const uint32_t e = reach == 2 ? (a18 | (a18 >> 1) | (a18 >> 2)) : (a18 >> 1);      // even fine voxels 2m (m = 16 w + s)
    const uint32_t o = (a18 >> 1) | (a18 >> 2);                                         // odd fine voxels 2m + 1
    out = spread16(e) | (spread16(o) << 1);
    const int valid = nf - w * 32;
    if (valid < 32) out &= (1u << valid) - 1u;
    words[L] = out;
  }
  int c = __popc(out);
  __shared__ int red[FW_BLOCK / 32];
  for (int s = 16; s; s >>= 1) c += __shfl_xor_sync(0xffffffffu, c, s);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = c;
  __syncthreads();
  if (threadIdx.x == 0) {
    int t = 0;
    for (int q = 0; q < FW_BLOCK / 32; ++q) t += red[q];
    blockcnt[blockIdx.x] = t;
  }
}

// exclusive scan of int counts by ONE block (n up to a few hundred thousand); total -> out[n]
__global__ void __launch_bounds__(1024) k_scan_i32(const int* __restrict__ in, int n, long long* __restrict__ out) {
  __shared__ long long part[1024];
  const int tid = threadIdx.x;
  const int per = (n + 1023) / 1024;
  const int lo = tid * per, hi = min(lo + per, n);
  long long s = 0;
  for (int i = lo; i < hi; ++i) s += in[i];
  part[tid] = s;
  __syncthreads();
  for (int off = 1; off < 1024; off <<= 1) {                 // Hillis-Steele inclusive scan
    long long v = tid >= off ? part[tid - off] : 0;
    __syncthreads();
    part[tid] += v;
    __syncthreads();
  }
  long long run = tid ? part[tid - 1] : 0;
  for (int i = lo; i < hi; ++i) { out[i] = run; run += in[i]; }
  if (tid == 1023) out[n] = part[1023];
}

// ordered compaction of the row-aligned fine words: warp = 32 consecutive words (lane holds one), every set bit becomes
// the flat index (row * nf + 32 w + bit) at its rank — coalesced stores, no atomics
__global__ void __launch_bounds__(FW_BLOCK) k_words_emit(const uint32_t* __restrict__ words, long long nwords, int nf, int wpr_f,
                                                          const long long* __restrict__ blockoff, int32_t* __restrict__ index,
                                                          long long cap) {
  __shared__ int wc[FW_BLOCK / 32];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long L = (long long)blockIdx.x * FW_BLOCK + threadIdx.x;
  const uint32_t my = L < nwords ? words[L] : 0u;
  int c = __popc(my), incl = c;
  for (int o = 1; o < 32; o <<= 1) { int v = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += v; }
  if (lane == 31) wc[warp] = incl;
  __syncthreads();
  long long off = blockoff[blockIdx.x];
  for (int q = 0; q < warp; ++q) off += wc[q];
  const int excl = incl - c;
  const int row = (int)(L / wpr_f), w = (int)(L - (long long)row * wpr_f);
  const int base = L < nwords ? row * nf + 32 * w : 0;          // flat index of this word's bit 0 (nf^3 < 2^31)
  for (int it = 0; it < 32; ++it) {
    const uint32_t m = __shfl_sync(0xffffffffu, my, it);
    if (m == 0u) continue;                                       // (uniform)
    const int e = __shfl_sync(0xffffffffu, excl, it);
    const int b0 = __shfl_sync(0xffffffffu, base, it);
    if ((m >> lane) & 1u) {
      const long long pos = off + e + __popc(m & ((1u << lane) - 1u));
      if (pos < cap) index[pos] = b0 + lane;
    }
  }
}

__global__ void k_fill_f32(float* __restrict__ p, long long n, float v) {
  long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  long long stride = (long long)gridDim.x * blockDim.x;
  for (; t < n; t += stride) p[t] = v;
}

// entries outside the window [base, base + len) of the whole grid (padding -1 included) are skipped
__global__ void k_scatter_f32(const int32_t* __restrict__ index, const float* __restrict__ vals, long long n, long long base,
                              long long len, float* __restrict__ grid) {
  long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n) return;
  int i = index[t];
  if (i < base || i - base >= len) return;
  float v = vals[t];
  if (v == HY3D_SENTINEL) v = __int_as_float(0x7fc00000);    // a logit equal to the sentinel is "unvisited" downstream (volume_decoders.py:275)
  grid[i - base] = v;
}

__global__ void k_sentinel_nan(float* __restrict__ p, long long n, float sentinel) {
  long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  long long stride = (long long)gridDim.x * blockDim.x;
  const float nanv = __int_as_float(0x7fc00000);
  for (; t < n; t += stride) { float v = p[t]; if (v == sentinel) p[t] = nanv; }
}

}  // namespace

extern "C" {

int hy3d_refine_level(hy3d_ctx* ctx, const float* d_coarse, int32_t n, int32_t nf, float mc_level, int32_t last_level,
                      int32_t* d_index, int64_t cap, int64_t* h_count) {
  if (!ctx || !d_coarse || n < 2 || !h_count || cap < 0 || (cap > 0 && !d_index)) return HY3D_ERR_ARG;
  // the fine grid is (r+1)^3 with r = 2 r_c or 2 r_c + 1 (levels are built with r // 2, volume_decoders.py:202-208):
  // every up-sampled voxel 2c must exist (nf >= 2n - 1) and every fine voxel must have a coarse parent f >> 1 (nf <= 2n)
  if (nf < 2 * n - 1 || nf > 2 * n) return hy3d_fail(ctx, HY3D_ERR_ARG, "fine grid %d^3 does not refine a %d^3 grid (need 2n-1 or 2n)", nf, n);
  HY3D_CUDA(ctx, cudaSetDevice(ctx->device));
  const long long nfine = (long long)nf * nf * nf;
  if (nfine > 2147483647LL) return hy3d_fail(ctx, HY3D_ERR_UNSUPPORTED, "fine grid too large for int32 indices");
  if (n > 1024) return hy3d_fail(ctx, HY3D_ERR_UNSUPPORTED, "coarse grids above 1024^3 are not supported");
  const int wpr_c = (n + 31) / 32, wpr_f = (nf + 31) / 32;
  const long long cwords = (long long)n * n * wpr_c;
  const long long nwords = (long long)nf * nf * wpr_f;
  const int nblocks = (int)ceil_div64(nwords, FW_BLOCK);
  HY3D_CUDA(ctx, ctx->scratch.reserve((size_t)cwords * 4 * 2 + 512));
  HY3D_CUDA(ctx, ctx->scratch2.reserve((size_t)nwords * 4 + (size_t)nblocks * 4 + (size_t)(nblocks + 1) * 8 + 1024));
  uint32_t* act = ctx->scratch.as<uint32_t>();
  uint32_t* act2 = act + ((cwords + 63) / 64 * 64);
  uint32_t* words = ctx->scratch2.as<uint32_t>();
  int* blockcnt = reinterpret_cast<int*>(words + ((nwords + 63) / 64 * 64));
  long long* blockoff = reinterpret_cast<long long*>(blockcnt + ((nblocks + 63) / 64 * 64));
  HY3D_PROF(ctx, FAM_OCTREE);
  k_coarse_bits<<<(unsigned)(n * n), wpr_c * 32, 0, ctx->stream>>>(d_coarse, n, wpr_c, mc_level, act);
  HY3D_LAUNCH_CHECK(ctx);
  const uint32_t* mask = act;
  if (!last_level) {
    HY3D_PROF(ctx, FAM_OCTREE);
    k_dilate_bits<<<(unsigned)ceil_div64(cwords, 256), 256, 0, ctx->stream>>>(act, n, wpr_c, act2);
    HY3D_LAUNCH_CHECK(ctx);
    mask = act2;
  }
  const int reach = last_level ? 2 : 1;
  HY3D_PROF(ctx, FAM_OCTREE);
  k_fine_words<<<nblocks, FW_BLOCK, 0, ctx->stream>>>(mask, n, wpr_c, nf, wpr_f, reach, nwords, words, blockcnt);
  HY3D_LAUNCH_CHECK(ctx);
  HY3D_PROF(ctx, FAM_OCTREE);
  k_scan_i32<<<1, 1024, 0, ctx->stream>>>(blockcnt, nblocks, blockoff);
  HY3D_LAUNCH_CHECK(ctx);
  if (cap > 0) {
    HY3D_PROF(ctx, FAM_OCTREE);
    k_words_emit<<<nblocks, FW_BLOCK, 0, ctx->stream>>>(words, nwords, nf, wpr_f, blockoff, d_index, cap);
    HY3D_LAUNCH_CHECK(ctx);
  }
  long long* pinned = reinterpret_cast<long long*>(ctx->pinned);
  HY3D_CUDA(ctx, cudaMemcpyAsync(pinned, blockoff + nblocks, sizeof(long long), cudaMemcpyDeviceToHost, ctx->stream));
  if (int rc = hy3d_watchdog_enqueue(ctx)) return rc;
  HY3D_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  *h_count = pinned[0];
  return hy3d_watchdog_check(ctx);        // the coarse grid came from the tensor kernels: a barrier timeout there invalidates it
}

int hy3d_fill(hy3d_ctx* ctx, float* d_grid, int64_t n, float value) {
  if (!ctx || n < 0 || (n > 0 && !d_grid)) return HY3D_ERR_ARG;
  if (n == 0) return HY3D_OK;
  HY3D_CUDA(ctx, cudaSetDevice(ctx->device));
  int blocks = (int)(ceil_div64(n, 256) < (long long)ctx->num_sms * 16 ? ceil_div64(n, 256) : (long long)ctx->num_sms * 16);
  HY3D_PROF(ctx, FAM_OCTREE);
  k_fill_f32<<<blocks, 256, 0, ctx->stream>>>(d_grid, n, value);
  HY3D_LAUNCH_CHECK(ctx);
  return HY3D_OK;
}

int hy3d_scatter(hy3d_ctx* ctx, const int32_t* d_index, const float* d_values, int64_t n, int64_t base, float* d_grid) {
  if (!ctx || n < 0 || base < 0 || (n > 0 && (!d_index || !d_values || !d_grid))) return HY3D_ERR_ARG;
  if (n == 0) return HY3D_OK;
  HY3D_CUDA(ctx, cudaSetDevice(ctx->device));
  HY3D_PROF(ctx, FAM_OCTREE);
  k_scatter_f32<<<(unsigned)ceil_div64(n, 256), 256, 0, ctx->stream>>>(d_index, d_values, n, base, LLONG_MAX, d_grid);
  HY3D_LAUNCH_CHECK(ctx);
  return HY3D_OK;
}

int hy3d_scatter_window(hy3d_ctx* ctx, const int32_t* d_index, const float* d_values, int64_t n, int64_t base, int64_t len,
                        float* d_grid) {
  if (!ctx || n < 0 || base < 0 || len < 0 || (n > 0 && len > 0 && (!d_index || !d_values || !d_grid))) return HY3D_ERR_ARG;
  if (n == 0 || len == 0) return HY3D_OK;
  HY3D_CUDA(ctx, cudaSetDevice(ctx->device));
  HY3D_PROF(ctx, FAM_OCTREE);
  k_scatter_f32<<<(unsigned)ceil_div64(n, 256), 256, 0, ctx->stream>>>(d_index, d_values, n, base, len, d_grid);
  HY3D_LAUNCH_CHECK(ctx);
  return HY3D_OK;
}

int hy3d_sentinel_to_nan(hy3d_ctx* ctx, float* d_grid, int64_t n, float sentinel) {
  if (!ctx || n < 0 || (n > 0 && !d_grid)) return HY3D_ERR_ARG;
  if (n == 0) return HY3D_OK;
  HY3D_CUDA(ctx, cudaSetDevice(ctx->device));
  int blocks = (int)(ceil_div64(n, 256) < (long long)ctx->num_sms * 16 ? ceil_div64(n, 256) : (long long)ctx->num_sms * 16);
  HY3D_PROF(ctx, FAM_OCTREE);
  k_sentinel_nan<<<blocks, 256, 0, ctx->stream>>>(d_grid, n, sentinel);
  HY3D_LAUNCH_CHECK(ctx);
  return HY3D_OK;
}

}  // extern "C"
