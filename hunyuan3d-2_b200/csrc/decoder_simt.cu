// fp32 CUDA-core decoder: the exact-order device reference (HY3D_PRECISION_FP32_SIMT) and the
// per-latent K/V projection shared with the tcgen05 path.
//
// Restates CrossAttentionDecoder.forward (reference attention_blocks.py:483-493, formula in
// SURVEY App. A.2) as a chain of plain kernels.  It is deliberately simple: its job is to be
// right, so that the tcgen05 kernels (decoder_tc.cu) can be checked stage by stage on the device.
#include "common.cuh"

namespace {

// ------------------------------------------------------------------------------------------
// Fourier embedding + query_proj (attention_blocks.py:112-130, :457, :485)
// ------------------------------------------------------------------------------------------
constexpr int EQ_PTS = 16;

__global__ void k_embed_qproj(QuerySource src, long long n, int F, int include_pi, const float* __restrict__ Wqp,
                              const float* __restrict__ bqp, int W, float* __restrict__ x0) {
  __shared__ float e[EQ_PTS][64];
  const int E = 3 * (2 * F + 1);
  long long p0 = (long long)blockIdx.x * EQ_PTS;
  for (int t = threadIdx.x; t < EQ_PTS * 3 * F; t += blockDim.x) {
    int pt = t / (3 * F), r = t % (3 * F), a = r / F, f = r % F;
    long long q = p0 + pt;
    float c[3] = {0.f, 0.f, 0.f};
    long long oi;
    if (q < n) hy3d_query_point(src, q, c[0], c[1], c[2], oi);
    float freq = exp2f((float)f);
    if (include_pi) freq *= 3.14159265358979323846f;   // torch: float32(2^f) * float32(pi)
    float arg = __fmul_rn(c[a], freq);
    e[pt][3 + a * F + f] = sinf(arg);
    e[pt][3 + 3 * F + a * F + f] = cosf(arg);
    if (f == 0) e[pt][a] = c[a];
  }
  __syncthreads();
  for (int nn = threadIdx.x; nn < W; nn += blockDim.x) {
    float acc[EQ_PTS];
#pragma unroll
    for (int pt = 0; pt < EQ_PTS; ++pt) acc[pt] = 0.f;
    const float* w = Wqp + (size_t)nn * E;
    for (int c = 0; c < E; ++c) {
      float wv = w[c];
#pragma unroll
      for (int pt = 0; pt < EQ_PTS; ++pt) acc[pt] = fmaf(e[pt][c], wv, acc[pt]);
    }
    float b = bqp[nn];
#pragma unroll
    for (int pt = 0; pt < EQ_PTS; ++pt)
      if (p0 + pt < n) x0[(size_t)(p0 + pt) * W + nn] = acc[pt] + b;
  }
}

// ------------------------------------------------------------------------------------------
// Row LayerNorm, one warp per row (two-pass, fp32).  In-place allowed.
// ------------------------------------------------------------------------------------------
__global__ void k_layernorm(const float* __restrict__ x, long long rows, int len, long long ldx,
                            const float* __restrict__ g, const float* __restrict__ b, float eps, float post_scale,
                            float* __restrict__ y, long long ldy) {
  long long row = (long long)blockIdx.x * (blockDim.x / 32) + threadIdx.x / 32;
  int lane = threadIdx.x & 31;
  if (row >= rows) return;
  const float* xr = x + row * ldx;
  float s = 0.f;
  for (int c = lane; c < len; c += 32) s += xr[c];
  for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  float mean = s / len, v = 0.f;
  for (int c = lane; c < len; c += 32) { float d = xr[c] - mean; v += d * d; }
  for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  float rstd = rsqrtf(v / len + eps);
  float* yr = y + row * ldy;
  for (int c = lane; c < len; c += 32) {
    float t = (xr[c] - mean) * rstd;
    if (g) t = t * g[c] + b[c];
    yr[c] = t * post_scale;
  }
}

// ------------------------------------------------------------------------------------------
// Generic SGEMM  C[M,N] = A[M,K] * B[N,K]^T (+bias) (+gelu) (+residual), batched over z.
// 64x64x16 tiles, 256 threads, 4x4 micro-tiles.
// ------------------------------------------------------------------------------------------
struct GemmArgs {
  const float* A; long long lda, sA;
  const float* B; long long ldb, sB;
  float* C; long long ldc, sC;
  const float* bias;
  const float* resid; long long ldr, sR;
  long long M; int N, K;
  int gelu;
  float alpha;
};

__device__ __forceinline__ float gelu_erf(float x) { return 0.5f * x * (1.f + erff(x * 0.70710678118654752440f)); }

__global__ void __launch_bounds__(256) k_sgemm(GemmArgs g) {
  __shared__ float As[16][64 + 4];
  __shared__ float Bs[16][64 + 4];
  const int z = blockIdx.z;
  const float* A = g.A + z * g.sA;
  const float* B = g.B + z * g.sB;
  float* C = g.C + z * g.sC;
  const long long m0 = (long long)blockIdx.y * 64;
  const int n0 = blockIdx.x * 64;
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  float acc[4][4] = {};
  for (int k0 = 0; k0 < g.K; k0 += 16) {
    for (int t = threadIdx.x; t < 64 * 16; t += 256) {
      int r = t >> 4, c = t & 15;
      long long m = m0 + r; int n = n0 + r; int k = k0 + c;
      As[c][r] = (m < g.M && k < g.K) ? A[m * g.lda + k] : 0.f;
      Bs[c][r] = (n < g.N && k < g.K) ? B[(long long)n * g.ldb + k] : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < 16; ++kk) {
      float a[4], b[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) { a[i] = As[kk][ty * 4 + i]; b[i] = Bs[kk][tx * 4 + i]; }
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    long long m = m0 + ty * 4 + i;
    if (m >= g.M) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      int n = n0 + tx * 4 + j;
      if (n >= g.N) continue;
      float v = acc[i][j] * g.alpha;
      if (g.bias) v += g.bias[n];
      if (g.gelu) v = gelu_erf(v);
      if (g.resid) v += g.resid[z * g.sR + m * g.ldr + n];
      C[m * g.ldc + n] = v;
    }
  }
}

// softmax over rows of length len (in place), one warp per row
__global__ void k_softmax_rows(float* __restrict__ s, long long rows, int len) {
  long long row = (long long)blockIdx.x * (blockDim.x / 32) + threadIdx.x / 32;
  int lane = threadIdx.x & 31;
  if (row >= rows) return;
  float* r = s + row * (long long)len;
  float m = -INFINITY;
  for (int c = lane; c < len; c += 32) m = fmaxf(m, r[c]);
  for (int o = 16; o; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  float sum = 0.f;
  for (int c = lane; c < len; c += 32) { float e = expf(r[c] - m); r[c] = e; sum += e; }
  for (int o = 16; o; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
  float inv = 1.f / sum;
  for (int c = lane; c < len; c += 32) r[c] *= inv;
}

// [ln_post] + output_proj (attention_blocks.py:490-492), one warp per row; scatter per out_mode.
__global__ void k_head_out(const float* __restrict__ x, long long rows, int W, const float* __restrict__ g,
                           const float* __restrict__ b, const float* __restrict__ wout, const float* __restrict__ bout,
                           QuerySource src, float* __restrict__ out, int out_mode) {
  long long row = (long long)blockIdx.x * (blockDim.x / 32) + threadIdx.x / 32;
  int lane = threadIdx.x & 31;
  if (row >= rows) return;
  const float* xr = x + row * (long long)W;
  float dot = 0.f;
  if (g) {
    float s = 0.f;
    for (int c = lane; c < W; c += 32) s += xr[c];
    for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    float mean = s / W, v = 0.f;
    for (int c = lane; c < W; c += 32) { float d = xr[c] - mean; v += d * d; }
    for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    float rstd = rsqrtf(v / W + 1e-5f);
    for (int c = lane; c < W; c += 32) dot += ((xr[c] - mean) * rstd * g[c] + b[c]) * wout[c];
  } else {
    for (int c = lane; c < W; c += 32) dot += xr[c] * wout[c];
  }
  for (int o = 16; o; o >>= 1) dot += __shfl_xor_sync(0xffffffffu, dot, o);
  if (lane == 0) {
    long long oi = row;
    float v = dot + bout[0];
    if (out_mode == 1) {
      oi = src.index[row];
      if (oi < 0) return;
      if (v == HY3D_SENTINEL) v = __int_as_float(0x7fc00000);      // see k_head_final (decoder_tc.cu)
    }
    out[oi] = v;
  }
}

// split c_kv output [M, 2W] into per-head k [H,M,D] and v^T [H,D,M] (attention_blocks.py:205-208)
__global__ void k_split_kv(const float* __restrict__ kv, int M, int H, int D, float* __restrict__ k, float* __restrict__ vT) {
  long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  long long total = (long long)M * H * D;
  if (t >= total) return;
  int d = t % D; long long r = t / D; int h = r % H; int m = r / H;
  const float* row = kv + (size_t)m * (2 * H * D) + (size_t)h * 2 * D;
  k[((size_t)h * M + m) * D + d] = row[d];
  vT[((size_t)h * D + d) * M + m] = row[D + d];
}

int sgemm(hy3d_ctx* ctx, const GemmArgs& g, int batch) {
  dim3 grid((g.N + 63) / 64, (unsigned)((g.M + 63) / 64), batch);
  k_sgemm<<<grid, 256, 0, ctx->stream>>>(g);
  HY3D_LAUNCH_CHECK(ctx);
  return 0;
}

int layernorm(hy3d_ctx* ctx, const float* x, long long rows, int len, long long ldx, const float* g, const float* b,
              float eps, float post_scale, float* y, long long ldy) {
  int wpb = 8;
  k_layernorm<<<(unsigned)ceil_div64(rows, wpb), wpb * 32, 0, ctx->stream>>>(x, rows, len, ldx, g, b, eps, post_scale, y, ldy);
  HY3D_LAUNCH_CHECK(ctx);
  return 0;
}

}  // namespace

// ------------------------------------------------------------------------------------------
// Per-latent K/V (fp32): [latents_proj] -> ln_2 -> c_kv -> split -> k_norm
// ------------------------------------------------------------------------------------------
int hy3d_simt_prepare_kv(hy3d_ctx* ctx, const float* d_latents, int M) {
  HY3D_PROF(ctx, FAM_KV);   // times the first launch only; the K/V family total is read from its share of the step
  DecoderWeights& w = ctx->w;
  const int W = w.W, H = w.H, D = w.D;
  HY3D_CUDA(ctx, ctx->ws[0].reserve((size_t)M * W * 4));
  HY3D_CUDA(ctx, ctx->ws[1].reserve((size_t)M * 2 * W * 4));
  HY3D_CUDA(ctx, ctx->kv.k32.reserve((size_t)H * M * D * 4));
  HY3D_CUDA(ctx, ctx->kv.v32.reserve((size_t)H * M * D * 4));
  float* lat = ctx->ws[0].as<float>();
  float* kvbuf = ctx->ws[1].as<float>();
  const float* src = d_latents;
  long long ld = w.LW;
  if (w.has_latents_proj) {
    GemmArgs g{};
    g.A = d_latents; g.lda = w.LW; g.B = w.lp_w; g.ldb = w.LW; g.C = lat; g.ldc = W; g.bias = w.lp_b;
    g.M = M; g.N = W; g.K = w.LW; g.alpha = 1.f;
    if (int rc = sgemm(ctx, g, 1)) return rc;
    src = lat; ld = W;
  }
  if (int rc = layernorm(ctx, src, M, W, ld, w.ln2_w, w.ln2_b, 1e-6f, 1.f, lat, W)) return rc;
  {
    GemmArgs g{};
    g.A = lat; g.lda = W; g.B = w.ckv_w; g.ldb = W; g.C = kvbuf; g.ldc = 2 * W; g.bias = w.ckv_b;
    g.M = M; g.N = 2 * W; g.K = W; g.alpha = 1.f;
    if (int rc = sgemm(ctx, g, 1)) return rc;
  }
  long long total = (long long)M * H * D;
  k_split_kv<<<(unsigned)ceil_div64(total, 256), 256, 0, ctx->stream>>>(kvbuf, M, H, D, ctx->kv.k32.as<float>(),
                                                                        ctx->kv.v32.as<float>());
  HY3D_LAUNCH_CHECK(ctx);
  if (w.qk_norm) {
    float* k = ctx->kv.k32.as<float>();
    if (int rc = layernorm(ctx, k, (long long)H * M, D, D, w.kn_w, w.kn_b, 1e-6f, 1.f, k, D)) return rc;
  }
  ctx->kv.M = M;
  ctx->kv.Mpad = (M + 127) / 128 * 128;
  ctx->kv.ready = true;
  return 0;
}

// ------------------------------------------------------------------------------------------
// Full fp32 decode of n query points
// ------------------------------------------------------------------------------------------
int hy3d_decode_simt(hy3d_ctx* ctx, const QuerySource& src_in, long long n, float* d_out, int out_mode) {
  DecoderWeights& w = ctx->w;
  const int W = w.W, H = w.H, D = w.D, R = w.R, M = ctx->kv.M;
  const long long CH = 2048;
  HY3D_CUDA(ctx, ctx->ws[2].reserve((size_t)CH * W * 4));          // x (residual stream)
  HY3D_CUDA(ctx, ctx->ws[3].reserve((size_t)CH * W * 4));          // ln / q
  HY3D_CUDA(ctx, ctx->ws[4].reserve((size_t)CH * W * 4));          // attention output
  HY3D_CUDA(ctx, ctx->ws[5].reserve((size_t)CH * W * R * 4));      // mlp hidden
  HY3D_CUDA(ctx, ctx->ws[6].reserve((size_t)CH * H * M * 4));      // scores
  float* x = ctx->ws[2].as<float>();
  float* t = ctx->ws[3].as<float>();
  float* a = ctx->ws[4].as<float>();
  float* h = ctx->ws[5].as<float>();
  float* s = ctx->ws[6].as<float>();
  for (long long p0 = 0; p0 < n; p0 += CH) {
    long long P = (n - p0 < CH) ? (n - p0) : CH;
    QuerySource src = src_in;
    if (src.mode == 0) src.xyz += 3 * p0;
    else if (src.mode == 1) src.first += p0;
    else src.index += p0;
    k_embed_qproj<<<(unsigned)ceil_div64(P, EQ_PTS), 256, 0, ctx->stream>>>(src, P, w.F, w.include_pi, w.qp_w, w.qp_b, W, x);
    HY3D_LAUNCH_CHECK(ctx);
    if (int rc = layernorm(ctx, x, P, W, W, w.ln1_w, w.ln1_b, 1e-6f, 1.f, t, W)) return rc;
    {   // q = c_q(ln_1(x))   (written to a, then head-normed in place)
      GemmArgs g{};
      g.A = t; g.lda = W; g.B = w.cq_w; g.ldb = W; g.C = a; g.ldc = W; g.bias = w.cq_b; g.M = P; g.N = W; g.K = W; g.alpha = 1.f;
      if (int rc = sgemm(ctx, g, 1)) return rc;
    }
    if (w.qk_norm)
      if (int rc = layernorm(ctx, a, P * H, D, D, w.qn_w, w.qn_b, 1e-6f, 1.f, a, D)) return rc;
    {   // scores[h] = q_h k_h^T / sqrt(D)
      GemmArgs g{};
      g.A = a; g.lda = W; g.sA = D; g.B = ctx->kv.k32.as<float>(); g.ldb = D; g.sB = (long long)M * D;
      g.C = s; g.ldc = M; g.sC = P * (long long)M; g.M = P; g.N = M; g.K = D; g.alpha = rsqrtf((float)D);
      if (int rc = sgemm(ctx, g, H)) return rc;
    }
    k_softmax_rows<<<(unsigned)ceil_div64(P * H, 8), 256, 0, ctx->stream>>>(s, P * H, M);
    HY3D_LAUNCH_CHECK(ctx);
    {   // o_h = softmax(scores) v_h   -> t[:, h*D:(h+1)*D]
      GemmArgs g{};
      g.A = s; g.lda = M; g.sA = P * (long long)M; g.B = ctx->kv.v32.as<float>(); g.ldb = M; g.sB = (long long)D * M;
      g.C = t; g.ldc = W; g.sC = D; g.M = P; g.N = D; g.K = M; g.alpha = 1.f;
      if (int rc = sgemm(ctx, g, H)) return rc;
    }
    {   // x1 = x0 + c_proj(attn)
      GemmArgs g{};
      g.A = t; g.lda = W; g.B = w.cproj_w; g.ldb = W; g.C = x; g.ldc = W; g.bias = w.cproj_b; g.resid = x; g.ldr = W;
      g.M = P; g.N = W; g.K = W; g.alpha = 1.f;
      if (int rc = sgemm(ctx, g, 1)) return rc;
    }
    if (int rc = layernorm(ctx, x, P, W, W, w.ln3_w, w.ln3_b, 1e-6f, 1.f, t, W)) return rc;
    {   // h = gelu(c_fc(ln_3 x1))
      GemmArgs g{};
      g.A = t; g.lda = W; g.B = w.fc_w; g.ldb = W; g.C = h; g.ldc = (long long)W * R; g.bias = w.fc_b; g.gelu = 1;
      g.M = P; g.N = W * R; g.K = W; g.alpha = 1.f;
      if (int rc = sgemm(ctx, g, 1)) return rc;
    }
    {   // x2 = x1 + c_proj(h)
      GemmArgs g{};
      g.A = h; g.lda = (long long)W * R; g.B = w.mp_w; g.ldb = (long long)W * R; g.C = x; g.ldc = W; g.bias = w.mp_b;
      g.resid = x; g.ldr = W; g.M = P; g.N = W; g.K = W * R; g.alpha = 1.f;
      if (int rc = sgemm(ctx, g, 1)) return rc;
    }
    float* outp = d_out + (out_mode == 0 ? p0 : 0);
    k_head_out<<<(unsigned)ceil_div64(P, 8), 256, 0, ctx->stream>>>(x, P, W, w.ln_post ? w.lnp_w : nullptr, w.lnp_b, w.out_w,
                                                                   w.out_b, src, outp, out_mode);
    HY3D_LAUNCH_CHECK(ctx);
  }
  return 0;
}
