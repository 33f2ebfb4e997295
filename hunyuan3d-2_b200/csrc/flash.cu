// FlashVDM adaptive KV selection on the device: replaces FlashVDMCrossAttentionProcessor /
// FlashVDMTopMCrossAttentionProcessor (reference attention_processors.py:35-96) as driven by
// FlashVDMVolumeDecoding (volume_decoders.py:343-371, 398-428).
//
// A "group" is one mini-grid (level 0) or one of the 6^3 spatial bins (refined levels).  Per group:
//   mean  mode: sim[h][t] = (mean over sub-sampled queries of q_h) . k_h[t]   (unscaled, == the mean of
//               the per-query similarities by linearity), keep the T largest tokens per (group, head);
//   merge mode: tokens whose head-averaged softmax probability exceeds 1e-6 for any sub-sampled query,
//               one set shared by all heads.
// The selected K / V^T rows are gathered into per-group UMMA tiles that the attention kernel streams
// exactly like the full K/V (AttnTC.tile_group / group_ntok).
// The sub-sampled q is produced by hy3d_tc_sample_q at ~fp32 accuracy (3-term split fp16 GEMMs), so
// that the token *sets* agree with the fp32 reference except at genuine near-ties.
#include "common.cuh"
#include "tc_ptx.cuh"

namespace {

constexpr int TILE_BYTES = 16384;

// qbar[g][c] = mean over samples of group g of qs[s][c].  off = the sample offsets of the selected groups; qs row 0 is the
// sample at off[0] (a range of groups starting past group 0 has its samples' q rows only)
__global__ void k_group_mean(const float* __restrict__ qs, const int* __restrict__ off, int W, float* __restrict__ qbar) {
  const int g = blockIdx.x;
  const int s0 = off[g] - off[0], s1 = off[g + 1] - off[0];
  for (int c = threadIdx.x; c < W; c += blockDim.x) {
    float acc = 0.f;
    for (int s = s0; s < s1; ++s) acc += qs[(size_t)s * W + c];
    qbar[(size_t)g * W + c] = s1 > s0 ? acc / (float)(s1 - s0) : 0.f;
  }
}

// one block per (group, head): similarities to all M (<= 4096) tokens, then the T largest by radix select on the
// order-preserving integer image of the keys (4 passes of 8 bits over a shared-memory histogram); ties at the
// threshold go to the lower token index (torch.topk's set on distinct keys; ties are measure-zero in fp32).
// Output: the T token ids in ascending order -> sel[g][h][0..T) (the attention is order-independent).
__global__ void __launch_bounds__(1024) k_sim_topk(const float* __restrict__ qbar, const float* __restrict__ k32, int H, int M, int T,
                                                    int* __restrict__ sel, int* __restrict__ ntok) {
  constexpr int PER = 4;                        // tokens per thread, consecutive (M <= 4096)
  __shared__ float qv[64];
  __shared__ unsigned hist[256];
  __shared__ unsigned sh_prefix, sh_need;
  __shared__ int wsum[32];
  const int g = blockIdx.x / H, h = blockIdx.x % H;
  if (threadIdx.x < 64) qv[threadIdx.x] = qbar[(size_t)g * H * 64 + h * 64 + threadIdx.x];
  if (threadIdx.x == 0) { sh_prefix = 0u; sh_need = (unsigned)T; }
  __syncthreads();
  unsigned key[PER];
#pragma unroll
  for (int i = 0; i < PER; ++i) {
    const int t = threadIdx.x * PER + i;
    key[i] = 0u;                                // below every real key (real keys are >= 0x00800000 after the flip of -inf)
    if (t < M) {
      const float4* kr = reinterpret_cast<const float4*>(k32 + ((size_t)h * M + t) * 64);
      float acc = 0.f;
#pragma unroll
      for (int d4 = 0; d4 < 16; ++d4) {
        float4 kv = __ldg(kr + d4);
        acc = fmaf(qv[4 * d4], kv.x, acc); acc = fmaf(qv[4 * d4 + 1], kv.y, acc);
        acc = fmaf(qv[4 * d4 + 2], kv.z, acc); acc = fmaf(qv[4 * d4 + 3], kv.w, acc);
      }
      const unsigned u = __float_as_uint(acc);
      key[i] = (u & 0x80000000u) ? ~u : (u | 0x80000000u);
      if (key[i] == 0u) key[i] = 1u;            // keep 0 for "no token" (only a NaN with all mantissa bits could map there)
    }
  }
  // threshold = the T-th largest key: fix 8 bits per pass, from the top
  for (int pass = 0; pass < 4; ++pass) {
    const int shift = 24 - 8 * pass;
    if (threadIdx.x < 256) hist[threadIdx.x] = 0u;
    __syncthreads();
    const unsigned prefix = sh_prefix;
    const unsigned himask = pass == 0 ? 0u : (0xffffffffu << (shift + 8));
#pragma unroll
    for (int i = 0; i < PER; ++i)
      if (key[i] != 0u && (key[i] & himask) == prefix) atomicAdd(&hist[(key[i] >> shift) & 255u], 1u);
    __syncthreads();
    if (threadIdx.x < 32) {                     // one warp: walk the 256 buckets from the top until `need` is covered
      unsigned need = sh_need;
      unsigned c[8]; unsigned tot = 0;
#pragma unroll
      for (int j = 0; j < 8; ++j) { c[j] = hist[255 - (threadIdx.x * 8 + j)]; tot += c[j]; }
      unsigned incl = tot;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) { const unsigned v = __shfl_up_sync(0xffffffffu, incl, o); if ((int)threadIdx.x >= o) incl += v; }
      unsigned before = incl - tot;             // keys in buckets above this lane's eight
      if (before < need && need <= incl) {
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          if (before < need && need <= before + c[j]) {
            sh_prefix = prefix | ((unsigned)(255 - (threadIdx.x * 8 + j)) << shift);
            sh_need = need - before;            // how many keys of this bucket still belong to the top T
          }
          before += c[j];
        }
      }
    }
    __syncthreads();
  }
  const unsigned thr = sh_prefix;
  const int ties = (int)sh_need;                // keys == thr to take, lowest token ids first
  // ordered compaction: packed scan of (greater, equal) flags
  int gt = 0, eq = 0;
#pragma unroll
  for (int i = 0; i < PER; ++i) { gt += key[i] > thr; eq += (key[i] == thr); }
  int packed = gt | (eq << 16);
  int incl = packed;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) { const int v = __shfl_up_sync(0xffffffffu, incl, o); if ((int)(threadIdx.x & 31) >= o) incl += v; }
  if ((threadIdx.x & 31) == 31) wsum[threadIdx.x >> 5] = incl;
  __syncthreads();
  if (threadIdx.x < 32) {
    const int v = wsum[threadIdx.x];
    int s = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const int u = __shfl_up_sync(0xffffffffu, s, o); if ((int)threadIdx.x >= o) s += u; }
    wsum[threadIdx.x] = s - v;
  }
  __syncthreads();
  const int excl = wsum[threadIdx.x >> 5] + incl - packed;
  int ngt = excl & 0xffff, neq = excl >> 16;
  int* out = sel + ((size_t)g * H + h) * T;
#pragma unroll
  for (int i = 0; i < PER; ++i) {
    const bool is_gt = key[i] > thr, is_eq = key[i] == thr;
    if (is_gt || (is_eq && neq < ties)) out[ngt + min(neq, ties)] = threadIdx.x * PER + i;
    ngt += is_gt; neq += is_eq;
  }
  if (h == 0 && threadIdx.x == 0) ntok[g] = T;
}

// merge mode: one block per sub-sampled query; flags tokens with head-averaged probability > thresh
__global__ void __launch_bounds__(256) k_merge_flags(const float* __restrict__ qs, const int* __restrict__ off, int G, int H, int M,
                                                     const float* __restrict__ k32, float thresh, uint32_t* __restrict__ mask,
                                                     int mwords) {
  const int s = blockIdx.x, s0 = off[0];        // qs row s = sample s0 + s (see k_group_mean)
  if (s >= off[G] - s0) return;
  __shared__ int gsh;
  __shared__ float qv[64];
  __shared__ float red[8];
  if (threadIdx.x == 0) { int g = 0; while (g + 1 < G && off[g + 1] - s0 <= s) ++g; gsh = g; }
  constexpr int PER = 16;                      // tokens per thread (M <= 4096)
  float acc[PER];
#pragma unroll
  for (int i = 0; i < PER; ++i) acc[i] = 0.f;
  const int W = H * 64;
  for (int h = 0; h < H; ++h) {
    __syncthreads();
    if (threadIdx.x < 64) qv[threadIdx.x] = qs[(size_t)s * W + h * 64 + threadIdx.x];
    __syncthreads();
    float lg[PER];
    float mx = -INFINITY;
#pragma unroll
    for (int i = 0; i < PER; ++i) {
      const int t = threadIdx.x + i * 256;
      lg[i] = -INFINITY;
      if (t < M) {
        const float4* kr = reinterpret_cast<const float4*>(k32 + ((size_t)h * M + t) * 64);
        float a = 0.f;
#pragma unroll
        for (int d4 = 0; d4 < 16; ++d4) {
          float4 kv = __ldg(kr + d4);
          a = fmaf(qv[4 * d4], kv.x, a); a = fmaf(qv[4 * d4 + 1], kv.y, a); a = fmaf(qv[4 * d4 + 2], kv.z, a); a = fmaf(qv[4 * d4 + 3], kv.w, a);
        }
        lg[i] = a;
      }
      mx = fmaxf(mx, lg[i]);
    }
    for (int o = 16; o; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = mx;
    __syncthreads();
    mx = red[0];
#pragma unroll
    for (int w = 1; w < 8; ++w) mx = fmaxf(mx, red[w]);
    __syncthreads();
    float sum = 0.f;
#pragma unroll
    for (int i = 0; i < PER; ++i) { lg[i] = expf(lg[i] - mx); sum += lg[i]; }
    for (int o = 16; o; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = sum;
    __syncthreads();
    sum = 0.f;
#pragma unroll
    for (int w = 0; w < 8; ++w) sum += red[w];
    const float inv = 1.f / sum;
#pragma unroll
    for (int i = 0; i < PER; ++i) acc[i] += lg[i] * inv;
  }
  const int g = gsh;
  const float invH = 1.f / (float)H;
#pragma unroll
  for (int i = 0; i < PER; ++i) {
    const int t = threadIdx.x + i * 256;
    if (t < M && acc[i] * invH > thresh) atomicOr(&mask[(size_t)g * mwords + (t >> 5)], 1u << (t & 31));
  }
}

// ordered list of the set bits of each group's mask -> sel[g][0..n), ntok[g] = max(n, 1)
__global__ void __launch_bounds__(128) k_mask_compact(const uint32_t* __restrict__ mask, int mwords, int stride, int* __restrict__ sel,
                                                      int* __restrict__ ntok) {
  const int g = blockIdx.x;
  __shared__ int pre[129];
  const int w = threadIdx.x;
  const uint32_t m = w < mwords ? mask[(size_t)g * mwords + w] : 0u;
  pre[w + 1] = __popc(m);
  if (w == 0) pre[0] = 0;
  __syncthreads();
  if (w == 0) for (int i = 1; i <= 128; ++i) pre[i] += pre[i - 1];
  __syncthreads();
  int pos = pre[w];
  for (uint32_t t = m; t; t &= t - 1) sel[(size_t)g * stride + pos++] = w * 32 + __ffs(t) - 1;
  if (w == 0) {
    int n = pre[128];
    if (n == 0) { sel[(size_t)g * stride] = 0; n = 1; }
    ntok[g] = n;
  }
}

// gather selected tokens into per-group K and V^T tiles (same images as k_build_kv in decoder_tc.cu)
__global__ void k_gather_kv(const float* __restrict__ k32, const float* __restrict__ vT32, int H, int M, int nkv,
                            const int* __restrict__ sel, long long sel_sg, long long sel_sh, const int* __restrict__ ntok,
                            uint8_t* __restrict__ kt, uint8_t* __restrict__ vt, long long total) {
  long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= total) return;
  const long long per_head = (long long)nkv * 128 * 8;
  const long long gh = t / per_head; const long long rem = t % per_head;
  const int g = (int)(gh / H), h = (int)(gh % H);
  const int n = ntok[g];
  const int* s = sel + g * sel_sg + h * sel_sh;
  {
    const int slot = (int)(rem / 8), c16 = (int)(rem % 8);
    const int tok = slot < n ? s[slot] : -1;
    float v[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) v[i] = tok >= 0 ? k32[((size_t)h * M + tok) * 64 + c16 * 8 + i] : 0.f;
    uint8_t* tile = kt + ((size_t)gh * nkv + slot / 128) * TILE_BYTES;
    uint4 u; u.x = tc::pack_h2(v[0], v[1]); u.y = tc::pack_h2(v[2], v[3]); u.z = tc::pack_h2(v[4], v[5]); u.w = tc::pack_h2(v[6], v[7]);
    *reinterpret_cast<uint4*>(tile + tc::sw128_off(slot % 128, c16)) = u;
  }
  {
    const int d = (int)(rem % 64); const int tc8 = (int)(rem / 64);
    const int slot0 = tc8 * 8, j = slot0 / 128, kbk = (slot0 % 128) / 64, c16 = (slot0 % 64) / 8;
    float v[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int slot = slot0 + i;
      const int tok = slot < n ? s[slot] : -1;
      v[i] = tok >= 0 ? vT32[((size_t)h * 64 + d) * M + tok] : 0.f;
    }
    uint8_t* tile = vt + ((size_t)gh * nkv + j) * TILE_BYTES + kbk * (TILE_BYTES / 2);
    uint4 u; u.x = tc::pack_h2(v[0], v[1]); u.y = tc::pack_h2(v[2], v[3]); u.z = tc::pack_h2(v[4], v[5]); u.w = tc::pack_h2(v[6], v[7]);
    *reinterpret_cast<uint4*>(tile + tc::sw128_off(d, c16)) = u;
  }
}

int make_source(hy3d_ctx* ctx, const hy3d_coords* c, const int32_t* d_index, int32_t n0, int32_t n1, int32_t n2, QuerySource& s) {
  s = QuerySource{};
  s.index = d_index; s.n0 = n0; s.n1 = n1; s.n2 = n2;
  if (c->mode == 2) {
    s.mode = 2;
    for (int a = 0; a < 3; ++a) { s.cell[a] = c->cell[a]; s.bmin[a] = c->bmin[a]; }
  } else if (c->mode == 3) {
    if (!c->axis0 || !c->axis1 || !c->axis2) return hy3d_fail(ctx, HY3D_ERR_ARG, "axis tables missing");
    s.mode = 3;
    if (int rc = hy3d_upload_axes(ctx, c->axis0, c->axis1, c->axis2, n0, n1, n2)) return rc;
    s.axis = ctx->ws[11].as<float>();
  } else {
    return hy3d_fail(ctx, HY3D_ERR_ARG, "coords.mode must be 2 (idx*cell+bmin) or 3 (axis tables)");
  }
  return 0;
}

}  // namespace

extern "C" {

int hy3d_flash_select(hy3d_ctx* ctx, const int32_t* d_sample_index, int64_t n_samples, int32_t n0, int32_t n1, int32_t n2,
                      const hy3d_coords* coords, const int32_t* d_sample_off, int32_t G, int32_t topk, int32_t merge_mode) {
  return hy3d_flash_select_range(ctx, d_sample_index, n_samples, n0, n1, n2, coords, d_sample_off, G, 0, G, topk, merge_mode);
}

// groups [g0, g1) of a layout: d_sample_index = the layout's sample list from entry d_sample_off[g0] on, d_sample_off = the
// whole layout's offsets; the selection is stored under the local group ids 0 .. g1-g0-1 and hy3d_decode_flash(_values)
// subtracts g0 from every tile's group
int hy3d_flash_select_range(hy3d_ctx* ctx, const int32_t* d_sample_index, int64_t n_samples, int32_t n0, int32_t n1, int32_t n2,
                            const hy3d_coords* coords, const int32_t* d_sample_off, int32_t G_all, int32_t g0, int32_t g1,
                            int32_t topk, int32_t merge_mode) {
  if (!ctx || !d_sample_index || !coords || !d_sample_off || G_all <= 0 || n_samples <= 0) return HY3D_ERR_ARG;
  if (g0 < 0 || g1 <= g0 || g1 > G_all) return hy3d_fail(ctx, HY3D_ERR_ARG, "group range [%d, %d) outside [0, %d)", g0, g1, G_all);
  const int G = g1 - g0;
  d_sample_off += g0;
  if (!ctx->w.set || !ctx->kv.ready) return hy3d_fail(ctx, HY3D_ERR_STATE, "weights / K,V not prepared");
  if (ctx->precision != HY3D_PRECISION_FP16_TC) return hy3d_fail(ctx, HY3D_ERR_UNSUPPORTED, "FlashVDM runs on the tcgen05 path only");
  HY3D_CUDA(ctx, cudaSetDevice(ctx->device));
  DecoderWeights& w = ctx->w;
  KVSelState& ks = ctx->kvsel;
  ks.ready = false;
  const int W = w.W, H = w.H, M = ctx->kv.M, Mpad = ctx->kv.Mpad;
  if (M > 4096) return hy3d_fail(ctx, HY3D_ERR_UNSUPPORTED, "KV selection supports at most 4096 tokens");
  if (!merge_mode && (topk <= 0 || topk > M)) return hy3d_fail(ctx, HY3D_ERR_ARG, "bad topk");
  const long long Sp = (n_samples + 127) / 128 * 128;
  HY3D_CUDA(ctx, ks.qs.reserve((size_t)Sp * W * 4));
  QuerySource src;
  if (int rc = make_source(ctx, coords, d_sample_index, n0, n1, n2, src)) return rc;
  if (int rc = hy3d_tc_sample_q(ctx, src, n_samples, ks.qs.as<float>())) return rc;
  HY3D_CUDA(ctx, ks.ntok.reserve((size_t)G * 4));
  const float* k32 = ctx->kv.k32.as<float>();
  const float* vT32 = ctx->kv.v32.as<float>();
  long long sel_sg, sel_sh;
  if (!merge_mode) {
    const int T = topk;
    ks.nkv = (T + 127) / 128;
    HY3D_CUDA(ctx, ks.qbar.reserve((size_t)G * W * 4));
    HY3D_CUDA(ctx, ks.sel.reserve((size_t)G * H * T * 4));
    HY3D_PROF(ctx, FAM_SELECT);
    k_group_mean<<<G, 256, 0, ctx->stream>>>(ks.qs.as<float>(), d_sample_off, W, ks.qbar.as<float>());
    HY3D_LAUNCH_CHECK(ctx);
    HY3D_PROF(ctx, FAM_SELECT);
    k_sim_topk<<<G * H, 1024, 0, ctx->stream>>>(ks.qbar.as<float>(), k32, H, M, T, ks.sel.as<int>(), ks.ntok.as<int>());
    HY3D_LAUNCH_CHECK(ctx);
    sel_sg = (long long)H * T; sel_sh = T;
  } else {
    ks.nkv = Mpad / 128;
    const int mwords = (M + 31) / 32;
    HY3D_CUDA(ctx, ks.mask.reserve((size_t)G * mwords * 4));
    HY3D_CUDA(ctx, ks.sel.reserve((size_t)G * Mpad * 4));
    HY3D_CUDA(ctx, cudaMemsetAsync(ks.mask.p, 0, (size_t)G * mwords * 4, ctx->stream));
    HY3D_PROF(ctx, FAM_SELECT);
    k_merge_flags<<<(unsigned)n_samples, 256, 0, ctx->stream>>>(ks.qs.as<float>(), d_sample_off, G, H, M, k32, 1e-6f, ks.mask.as<uint32_t>(), mwords);
    HY3D_LAUNCH_CHECK(ctx);
    HY3D_PROF(ctx, FAM_SELECT);
    k_mask_compact<<<G, 128, 0, ctx->stream>>>(ks.mask.as<uint32_t>(), mwords, Mpad, ks.sel.as<int>(), ks.ntok.as<int>());
    HY3D_LAUNCH_CHECK(ctx);
    sel_sg = Mpad; sel_sh = 0;
  }
  const size_t bytes = (size_t)G * H * ks.nkv * TILE_BYTES;
  HY3D_CUDA(ctx, ks.ktile.reserve(bytes));
  HY3D_CUDA(ctx, ks.vtile.reserve(bytes));
  const long long total = (long long)G * H * ks.nkv * 128 * 8;
  HY3D_PROF(ctx, FAM_SELECT);
  k_gather_kv<<<(unsigned)ceil_div64(total, 256), 256, 0, ctx->stream>>>(k32, vT32, H, M, ks.nkv, ks.sel.as<int>(), sel_sg, sel_sh,
                                                                         ks.ntok.as<int>(), ks.ktile.as<uint8_t>(), ks.vtile.as<uint8_t>(), total);
  HY3D_LAUNCH_CHECK(ctx);
  ks.G = G;
  ks.g0 = g0;
  ks.ready = true;
  return HY3D_OK;
}

int hy3d_decode_flash(hy3d_ctx* ctx, const int32_t* d_index, int64_t n, int32_t n0, int32_t n1, int32_t n2,
                      const hy3d_coords* coords, const int32_t* d_tile_group, float* d_grid) {
  if (!ctx || n < 0 || !coords) return HY3D_ERR_ARG;
  if (n == 0) return HY3D_OK;
  if (!d_index || !d_tile_group || !d_grid || (n % 128) != 0) return hy3d_fail(ctx, HY3D_ERR_ARG, "padded list must be a multiple of 128");
  if (ctx->precision != HY3D_PRECISION_FP16_TC) return hy3d_fail(ctx, HY3D_ERR_UNSUPPORTED, "FlashVDM runs on the tcgen05 path only");
  HY3D_CUDA(ctx, cudaSetDevice(ctx->device));
  QuerySource src;
  if (int rc = make_source(ctx, coords, d_index, n0, n1, n2, src)) return rc;
  return hy3d_decode_tc_groups(ctx, src, n, d_grid, 1, d_tile_group);
}

int hy3d_decode_flash_values(hy3d_ctx* ctx, const int32_t* d_index, int64_t n, int32_t n0, int32_t n1, int32_t n2,
                             const hy3d_coords* coords, const int32_t* d_tile_group, float* d_values) {
  if (!ctx || n < 0 || !coords) return HY3D_ERR_ARG;
  if (n == 0) return HY3D_OK;
  if (!d_index || !d_tile_group || !d_values || (n % 128) != 0) return hy3d_fail(ctx, HY3D_ERR_ARG, "padded list must be a multiple of 128");
  if (ctx->precision != HY3D_PRECISION_FP16_TC) return hy3d_fail(ctx, HY3D_ERR_UNSUPPORTED, "FlashVDM runs on the tcgen05 path only");
  HY3D_CUDA(ctx, cudaSetDevice(ctx->device));
  QuerySource src;
  if (int rc = make_source(ctx, coords, d_index, n0, n1, n2, src)) return rc;
  return hy3d_decode_tc_groups(ctx, src, n, d_values, 0, d_tile_group);
}

// selected token ids of the last hy3d_flash_select (selection-parity tests): mean mode int32 [G,H,T]
int hy3d_flash_selection(hy3d_ctx* ctx, int32_t* d_out, int64_t count) {
  if (!ctx || !d_out) return HY3D_ERR_ARG;
  if (!ctx->kvsel.ready) return hy3d_fail(ctx, HY3D_ERR_STATE, "no KV selection prepared");
  if ((size_t)count * 4 > ctx->kvsel.sel.cap) return hy3d_fail(ctx, HY3D_ERR_ARG, "count exceeds the selection buffer");
  HY3D_CUDA(ctx, cudaMemcpyAsync(d_out, ctx->kvsel.sel.p, (size_t)count * 4, cudaMemcpyDeviceToDevice, ctx->stream));
  return HY3D_OK;
}

int hy3d_flash_group_tokens(hy3d_ctx* ctx, int32_t* d_out, int32_t G) {
  if (!ctx || !d_out || G <= 0) return HY3D_ERR_ARG;
  if (!ctx->kvsel.ready || G > ctx->kvsel.G) return hy3d_fail(ctx, HY3D_ERR_STATE, "no KV selection prepared");
  HY3D_CUDA(ctx, cudaMemcpyAsync(d_out, ctx->kvsel.ntok.p, (size_t)G * 4, cudaMemcpyDeviceToDevice, ctx->stream));
  return HY3D_OK;
}

}  // extern "C"
