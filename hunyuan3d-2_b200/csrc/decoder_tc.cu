// tcgen05 / TMEM decoder (HY3D_PRECISION_FP16_TC): CrossAttentionDecoder.forward (reference
// attention_blocks.py:483-493, SURVEY App. A.2) for batches of query points, fp16 operands with
// fp32 accumulation in tensor memory.
//
// Memory layout: every operand tile is ONE contiguous 16/32 KB block already in the 128-byte-swizzled K-major
// form the UMMA descriptors expect, so a single copy drops it into shared memory — a 1-D bulk copy (cp.async.bulk,
// SASS UBLKCP) in the attention kernel, a tensor-map TMA over "rows of 128 bytes" (UTMALDG) in the CTA-pair GEMM:
//   "T16"  fp16 activations  [P/128][K/64][128 rows x 64 cols, SW128]        (16 KB tiles)
//   "B16"  fp16 weights      [N/256][K/64][256 rows x 64 cols, SW128]        (32 KB tiles)
//   "R32"  fp32 residual     [P/128][N/4][128 rows][4]   (row-per-thread epilogues read/write 512 B
//                                                          contiguous per warp instruction)
//   K      fp16 [group][head][M/128][128 tok x 64, SW128]      V^T fp16 [group][head][M/128][2][64 d x 64 tok, SW128]
//
// Stage chain per chunk of 262144 points (one launch each, activations through HBM/L2; the chain is
// compute-bound: ~30 KB/point of traffic vs 33.7 MFLOP/point).  The three LayerNorms never run as kernels: ln_1 / ln_3
// are folded into the consuming GEMM (raw operand, gamma in the weights, per-row statistics from the producer's
// epilogue or, for ln_1, from the embed kernel), ln_post into the head.  x0 = query_proj(e) is never formed:
//   k_embed_tc       Fourier features, fp16 hi/lo split; ln_1 statistics of x0   -> T16 [., 3], row (mean, rstd)
//   k_gemm_tc<Q>     c_q . query_proj collapsed (K = 192, ln_1 folded), per-head q_norm, * scale * log2e
//                                                                                -> T16 q (k-block == head)
//   k_attn_fast / k_attn_tc   softmax(q k^T) v, 2 heads in flight per CTA (attention_tc.cuh)  -> T16
//   k_gemm_tc<RES>   x0 + c_proj: [attn | e] [W_o | W_qp]^T (K = W + 192)          -> R32 x1, T16 raw x1, row stats
//   k_gemm_tc<GELU>  c_fc (ln_3 folded) + erf-GELU                                -> T16 h
//   k_gemm_tc<RES>   mlp.c_proj + residual: only row stats + dot with gamma_post * w_out leave the kernel
//   k_head_final     [ln_post] + output_proj from those statistics               -> logits (dense or scattered)
// (k_finish_stats merges a producer's per-64-column partial statistics once per row before each folded GEMM;
//  k_ln_tc is the unfolded LayerNorm, used by the fp32-grade q of the FlashVDM token selection.)
#include <cuda.h>
#include "common.cuh"
#include "tc_ptx.cuh"

using namespace tc;

namespace {

constexpr int TILE_M = 128;
constexpr int TILE_BYTES = 16384;          // 128 x 64 fp16
constexpr int BN = 256;                    // GEMM N tile
constexpr int BTILE_BYTES = BN * 128;      // 256 x 64 fp16
constexpr int GEMM_CL = 2;                // CTAs per cluster: 2 = one MMA pair (product); 4 = two pairs sharing the B tile by multicast TMA (measured 5-10 % slower: only 33 such clusters = 132 of 148 SMs are co-resident)
constexpr int GEMM_STAGES = 5;            // 32 KB per stage and CTA: A tile + half of the B tile (+ 64 KB of output staging)
constexpr int GEMM_THREADS = 640;          // warp0 producer, warp1 mma, warp2 tmem, warp3 idle, warps 4..19 epilogue
constexpr int ST_PER_TILE = 4;             // row-statistic slots per 256-column tile (one per epilogue warp column quarter)
constexpr int ST_COLS = BN / ST_PER_TILE;  // columns per slot (64)
constexpr float LOG2E = 1.4426950408889634f;

enum { EPI_X0 = 0, EPI_Q = 1, EPI_RES = 2, EPI_GELU = 3, EPI_QF32 = 4, EPI_QKV = 5 };

struct GemmTC {
  const uint8_t* A;      // T16 tiles [Mb][KB]  (k-blocks 0 .. KB1-1 when a second operand is concatenated along K)
  const uint8_t* A2;     // optional second A operand, T16 tiles [Mb][KB - KB1]: k-blocks KB1 .. KB-1 (K-concatenated GEMM)
  int KB1;               // k-blocks taken from A (0 = all)
  const uint8_t* B;      // B16 tiles [Nb][KB]
  int Mb, Nb, KB, N;
  const float* bias;     // [N] or null
  const float* Rin;      // R32 (EPI_RES)
  float* Rout;           // R32 (EPI_X0, EPI_RES)
  uint8_t* Tout;         // T16 (EPI_Q, EPI_GELU)
  float* Fout;           // row-major fp32 [P, N] (EPI_QF32)
  const float* qn_w; const float* qn_b; int qk_norm; float qscale;   // EPI_Q
  // LayerNorm folded into this GEMM: the A operand is the RAW row (fp16), W was pre-multiplied by gamma,
  // so  LN(x) W^T = rstd * (x W'^T - mean * cs) + (beta W^T + bias);  row statistics come as S partial
  // (mean, M2) slots written by the producer's epilogue and are merged here (Chan et al.), deterministically.
  const float* st_in; int st_slots; int st_np; const float* cs; float ln_eps;
  const float2* ln_mr;   // per row (mean, rstd): merged from st_in by k_finish_stats (set by launch_gemm), or given directly
  // statistics of the rows this GEMM produces (EPI_X0 / EPI_RES): slot nb * 4 + column quarter <- (mean, M2[, dot with dotw]) of 64 columns
  float* st_out; int st_k; const float* dotw;
  uint8_t* Tcopy;        // fp16 T16 copy of the fp32 rows written to Rout (operand of the next GEMM)
  int split_out;         // Tcopy / Tout(GELU) written as [hi | lo | hi] (3 * N/64 k-blocks): operand of a 3-term split GEMM
  // EPI_QKV (latent transformer): output columns are [q (W) | k (W) | v (W)], head-contiguous
  uint8_t* Kout; uint8_t* Vout; const float* kn_w; const float* kn_b; int nkv; int Wq;
  int part0;             // 0: columns [q | k | v] (latent transformer); 1: columns [k | v] (decoder c_kv)
  float* K32; float* V32T; int Mtok;   // optional fp32 copies k [H, Mtok, 64], v^T [H, 64, Mtok] (FlashVDM selection); rows >= Mtok are written as zeros
};

// merge S partial (mean, M2) pairs of n_p samples each -> (mean, rstd)   (Chan et al., deterministic order)
// `st` = S records of `stride` floats (mean, M2[, dot]); record i at st + i * stride.  The whole row record block
// (S * stride floats, 16-byte aligned) is read with 128-bit loads: a thread per row would otherwise issue S * stride
// scalar loads that no warp-mate shares a sector with.
template <int kStride>
__device__ __forceinline__ void merge_row_stats(const float* __restrict__ st, int S, int n_p, float eps, float& mean, float& rstd,
                                                float* dot = nullptr) {
  constexpr int kMaxS = 16;                       // widths up to 1024 (64-column slots) take the vector path
  if (S <= kMaxS && ((S * kStride) & 3) == 0) {
    float v[kMaxS * kStride];
#pragma unroll
    for (int i = 0; i < kMaxS * kStride / 4; ++i)
      if (4 * i < S * kStride) {
        const float4 t = __ldg(reinterpret_cast<const float4*>(st) + i);
        v[4 * i] = t.x; v[4 * i + 1] = t.y; v[4 * i + 2] = t.z; v[4 * i + 3] = t.w;
      }
    float ms = 0.f, d = 0.f;
#pragma unroll
    for (int i = 0; i < kMaxS; ++i)
      if (i < S) { ms += v[i * kStride]; if (kStride == 3) d += v[i * kStride + kStride - 1]; }
    mean = ms / (float)S;
    float M2 = 0.f;
#pragma unroll
    for (int i = 0; i < kMaxS; ++i)
      if (i < S) { const float dd = v[i * kStride] - mean; M2 += v[i * kStride + 1] + (float)n_p * dd * dd; }
    rstd = rsqrtf(M2 / (float)(S * n_p) + eps);
    if (dot) *dot = d;
    return;
  }
  float ms = 0.f, d = 0.f;
  for (int i = 0; i < S; ++i) { ms += __ldg(st + i * kStride); if (kStride == 3) d += __ldg(st + i * kStride + 2); }
  mean = ms / (float)S;
  float M2 = 0.f;
  for (int i = 0; i < S; ++i) { const float dd = __ldg(st + i * kStride) - mean; M2 += __ldg(st + i * kStride + 1) + (float)n_p * dd * dd; }
  rstd = rsqrtf(M2 / (float)(S * n_p) + eps);
  if (dot) *dot = d;
}

// exact-erf GELU (reference attention_blocks.py:177) without erff's two divergent branches:
//   gelu(x) = max(x, 0) - |x| * erfc(|x| / sqrt2) / 2,   erfc(t) = 2^(-t g(t)),  g a minimax fit on [0, 4]
// (beyond t = 4 the correction is < 1e-8 |x| and the clamp keeps it there).  The 1/2 rides in the exponent.
// kDeg = 5: |gelu err| < 1e-7 (fp32-grade, latent transformer);  kDeg = 3: < 9e-6, far below the fp16
// rounding of the stored activation (decoder MLP) for two FFMA less per element.
template <int kDeg>
__device__ __forceinline__ float gelu_erf(float x) {
  const float ax = fabsf(x);
  const float t = fminf(ax * 0.70710678118654752440f, 4.0f);
  float g;
  if constexpr (kDeg == 5) {
    g = -2.39272936e-04f;
    g = fmaf(g, t, 4.18474770e-03f); g = fmaf(g, t, -3.19086965e-02f); g = fmaf(g, t, 1.50579343e-01f);
    g = fmaf(g, t, 9.17831750e-01f); g = fmaf(g, t, 1.62796776e+00f);
  } else {
    g = -1.664811e-02f;
    g = fmaf(g, t, 1.2936552e-01f); g = fmaf(g, t, 9.2985345e-01f); g = fmaf(g, t, 1.62573555e+00f);
  }
  const float e = ex2(fmaf(-t, g, -1.0f));        // erfc(|x| / sqrt2) / 2
  return fmaxf(x, 0.f) - ax * e;
}

// gelu_erf<3> of two values with the polynomial on packed f32x2 instructions (FMUL2 / FFMA2: one issue slot for the pair):
// 8 instead of 12.5 issue slots per element in the c_fc epilogue, which is what paces that GEMM (epilogue ~ MMA time).
__device__ __forceinline__ void gelu_erf3_pair(float x0, float x1, float& y0, float& y1) {
  float u0, u1;
  unpack_f2(mul_f2(pack_f2(x0, x1), pack_f2(0.70710678118654752440f, 0.70710678118654752440f)), u0, u1);
  const uint64_t t = pack_f2(fminf(fabsf(u0), 4.0f), fminf(fabsf(u1), 4.0f));
  uint64_t g = fma_f2(pack_f2(1.664811e-02f, 1.664811e-02f), t, pack_f2(-1.2936552e-01f, -1.2936552e-01f));     // -g(t)
  g = fma_f2(g, t, pack_f2(-9.2985345e-01f, -9.2985345e-01f));
  g = fma_f2(g, t, pack_f2(-1.62573555e+00f, -1.62573555e+00f));
  float a0, a1;
  unpack_f2(fma_f2(t, g, pack_f2(-1.0f, -1.0f)), a0, a1);             // -t g(t) - 1
  y0 = fmaf(-fabsf(x0), ex2(a0), fmaxf(x0, 0.f));
  y1 = fmaf(-fabsf(x1), ex2(a1), fmaxf(x1, 0.f));
}

__device__ __forceinline__ void store_t16_chunk(uint8_t* tile, int r, int c16, const float* v) {
  uint4 u;
  u.x = pack_h2(v[0], v[1]); u.y = pack_h2(v[2], v[3]); u.z = pack_h2(v[4], v[5]); u.w = pack_h2(v[6], v[7]);
  *reinterpret_cast<uint4*>(tile + sw128_off(r, c16)) = u;
}

// fp16 hi/lo split stores of 8 values: chunk c16 of row r in tiles (hi) t0, (lo) t1, (hi) t2
__device__ __forceinline__ void store_t16_split(uint8_t* t0, uint8_t* t1, uint8_t* t2, int r, int c16, const float* v) {
  float hi[8], lo[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) { hi[i] = __half2float(__float2half_rn(v[i])); lo[i] = v[i] - hi[i]; }
  store_t16_chunk(t0, r, c16, hi);
  store_t16_chunk(t1, r, c16, lo);
  store_t16_chunk(t2, r, c16, hi);
}


// ------------------------------------------------------------------------------------------
// Persistent warp-specialised GEMM:  C[P, N] = A[P, K] * W[N, K]^T with a fused epilogue.
// ------------------------------------------------------------------------------------------
// One MMA spans a CTA pair (cta_group::2): the pair computes a 256 x 256 tile, each CTA holding 128 rows of A, 128 of the
// 256 B rows and its 128 x 256 accumulator.  Per k-block each SM moves 32 KB into and out of its shared memory instead
// of 48 KB: with single-SM MMAs the TMA fills plus the operand reads already take ~190 B/clk of shared-memory
// bandwidth and every epilogue load/store slowed the tensor pipe (full kernel 30 % slower than max(MMA-only,
// epilogue-only)).  Barrier protocol (s = smem stage, acc = accumulator buffer):
//   FULL(s)   (leader) TMA bytes of BOTH CTAs' stage s, 64 KB -> leader MMA warp
//   EMPTY(s)  multicast tcgen05.commit of the leader          -> both producers
//   TFULL(a)  multicast tcgen05.commit of the leader          -> both CTAs' epilogue warps
//   TEMPTY(a) (leader) 16 local + 16 remote epilogue arrivals -> leader MMA warp
template <int EPI>
__global__ void __cluster_dims__(GEMM_CL, 1, 1) __launch_bounds__(GEMM_THREADS, 1)
k_gemm_tc(GemmTC g, const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmA2, const __grid_constant__ CUtensorMap tmB) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sA = smem;                                      // [STAGES][16 KB]  this CTA's 128 rows of A
  uint8_t* sB = smem + GEMM_STAGES * TILE_BYTES;           // [STAGES][16 KB]  this CTA's 128 of the 256 B rows
  uint8_t* sOut = smem + GEMM_STAGES * 2 * TILE_BYTES;     // [4 column quarters][16 KB]  fp16 output tiles staged for bulk stores
  uint64_t* bars = reinterpret_cast<uint64_t*>(sOut + ST_PER_TILE * TILE_BYTES);
  const uint32_t bar0 = smem_u32(bars);
  auto FULL = [&](int s) { return bar0 + 8u * s; };
  auto EMPTY = [&](int s) { return bar0 + 8u * (GEMM_STAGES + s); };
  auto TFULL = [&](int a) { return bar0 + 8u * (2 * GEMM_STAGES + a); };
  auto TEMPTY = [&](int a) { return bar0 + 8u * (2 * GEMM_STAGES + 2 + a); };
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * GEMM_STAGES + 4);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (threadIdx.x == 0) {
    for (int s = 0; s < GEMM_STAGES; ++s) { mbar_init(FULL(s), 1); mbar_init(EMPTY(s), GEMM_CL / 2); }
    for (int a = 0; a < 2; ++a) { mbar_init(TFULL(a), 1); mbar_init(TEMPTY(a), 32); }
    fence_barrier_init();
  }
  if (warp == 2) { tmem_alloc2(smem_u32(tmem_slot), 512); tmem_relinquish2(); }
  fence_before_sync();
  cluster_sync();                      // the peer's barriers must exist before anything is signalled to them
  fence_after_sync();
  const uint32_t tmem = *tmem_slot;
  // work item p of cluster c: tile pair (m-blocks 2 (p / Nb) + {0, 1}, n-block p % Nb); this CTA holds m-block + rank
  // (GEMM_CL = 4: two pairs with the same n-block; each CTA fetches a QUARTER of the B tile and multicasts it to the CTA of the
  //  other pair that holds the same B half — 24 KB instead of 32 KB of L2 -> SM traffic per CTA and k-block)
  const int crank = (int)cluster_ctarank();
  const int rank = crank & 1, pair = crank >> 1;          // position inside the MMA pair, pair inside the cluster
  const int npairs = ((g.Mb + GEMM_CL - 1) / GEMM_CL) * g.Nb;
  const int cid = blockIdx.x / GEMM_CL, ncl = gridDim.x / GEMM_CL;
  const uint16_t mask_all = (uint16_t)((1u << GEMM_CL) - 1), mask_pair = (uint16_t)(3u << (2 * pair));

  if (warp == 0) {
    int s = 0; uint32_t ph = 0;
    for (int p = cid; p < npairs; p += ncl) {
      int mb = GEMM_CL * (p / g.Nb) + crank; const int nb = p % g.Nb;
      if (mb >= g.Mb) mb = g.Mb - 1;   // ragged tile count: the idle CTAs still feed their share of B (their results are dropped)
      // operands through the tensor maps tmA / tmA2 / tmB: A tile (mb, kb) = tile index mb KB + kb,
      // this CTA's half of B tile (nb, kb) = rows [(nb KB + kb) 256 + 128 rank, +128)
      const int kb1 = g.KB1 ? g.KB1 : g.KB;
      // tensor-map rows are 2 KB: a 16 KB tile = 8 rows
      const int arow = mb * kb1 * 8, a2row = mb * (g.KB - kb1) * 8;
      const int brow = nb * g.KB * 16 + rank * 8 + (GEMM_CL == 4 ? pair * 4 : 0);
      for (int kb = 0; kb < g.KB; ++kb) {
        mbar_wait(EMPTY(s), ph ^ 1);
        if (elect_one()) {
          // both CTAs' copies complete on the LEADER's FULL(s) (64 KB per stage): no software relay on the critical path
          if (rank == 0) mbar_arrive_expect_tx(FULL(s), 4 * TILE_BYTES);
          if (kb < kb1) tma2d_g2s_pair(smem_u32(sA + s * TILE_BYTES), &tmA, 0, arow + kb * 8, FULL(s));
          else tma2d_g2s_pair(smem_u32(sA + s * TILE_BYTES), &tmA2, 0, a2row + (kb - kb1) * 8, FULL(s));
          if (GEMM_CL == 4)
            tma2d_g2s_pair_multicast(smem_u32(sB + s * TILE_BYTES + pair * (TILE_BYTES / 2)), &tmB, 0, brow + kb * 16, FULL(s),
                                     (uint16_t)((1u << crank) | (1u << (crank ^ 2))));
          else
            tma2d_g2s_pair(smem_u32(sB + s * TILE_BYTES), &tmB, 0, brow + kb * 16, FULL(s));
        }
        __syncwarp();
        if (++s == GEMM_STAGES) { s = 0; ph ^= 1; }
      }
    }
  } else if (warp == 1 && rank != 0) {
    // peer CTA: the leader issues the pair's MMAs
  } else if (warp == 1) {
    const uint32_t idesc = make_idesc_f16(2 * TILE_M, BN);
    int s = 0; uint32_t ph = 0;
    int it = 0;
    for (int p = cid; p < npairs; p += ncl, ++it) {
      const int acc = it & 1;
      const uint32_t aph = (it >> 1) & 1;
      mbar_wait(TEMPTY(acc), aph ^ 1);
      fence_after_sync();
      const uint32_t d = tmem + acc * BN;
      for (int kb = 0; kb < g.KB; ++kb) {
        mbar_wait(FULL(s), ph);
        fence_after_sync();
        const uint64_t ad = make_desc_sw128(smem_u32(sA + s * TILE_BYTES));
        const uint64_t bd = make_desc_sw128(smem_u32(sB + s * TILE_BYTES));
        if (elect_one()) {
#pragma unroll
          for (int k = 0; k < 4; ++k) mma2_f16_ss(d, ad + 2 * k, bd + 2 * k, idesc, (kb | k) != 0);
          mma2_commit_multicast(EMPTY(s), mask_all);
          if (kb == g.KB - 1) mma2_commit_multicast(TFULL(acc), mask_pair);
        }
        __syncwarp();
        if (++s == GEMM_STAGES) { s = 0; ph ^= 1; }
      }
    }
  } else if (warp >= 4) {
    // ---------------- epilogue: 16 warps = 4 TMEM lane quadrants x 4 column quarters of 64 ----------------
    // (four warps per scheduler: the TMEM-load -> constants -> math -> store chain of one warp hides behind the others)
    const int q = warp & 3;                 // TMEM lane quadrant this warp may access
    const int cq = (warp - 4) >> 2;         // 64-column quarter of the 256-wide tile
    const int r = q * 32 + lane;            // row inside the tile
    int it = 0;
    for (int p = cid; p < npairs; p += ncl, ++it) {
      const int mb = GEMM_CL * (p / g.Nb) + crank, nb = p % g.Nb;
      const int acc = it & 1;
      const uint32_t aph = (it >> 1) & 1;
      mbar_wait(TFULL(acc), aph);
      fence_after_sync();
      if (mb >= g.Mb) {
        fence_before_sync(); __syncwarp();
        if (lane == 0) { if (rank == 0) mbar_arrive(TEMPTY(acc)); else mbar_arrive_remote(TEMPTY(acc), crank & ~1); }
        continue;
      }
      const uint32_t tcol = tmem + acc * BN + cq * 64 + ((uint32_t)(q * 32) << 16);
      const int c0 = nb * BN + cq * 64;     // first global column of this warp's quarter
      float ln_mean = 0.f, ln_rstd = 1.f;
      if (g.ln_mr) { const float2 mr = __ldg(g.ln_mr + (size_t)mb * TILE_M + r); ln_mean = mr.x; ln_rstd = mr.y; }
      const float nm = -ln_rstd * ln_mean;
      // 32 accumulator columns [c0 + 32 ch, +32) -> x: + bias, or the folded LayerNorm  rstd * a + (bb - rstd * mean * cs)
      auto load32 = [&](int ch, float* x, bool fold) {
        uint32_t v[32];
        HY3D_TMEM_LD32(tcol + ch * 32, v);
        tmem_wait_ld();
        const float4* b4 = reinterpret_cast<const float4*>(g.bias + c0 + ch * 32);
        const float4* c4 = reinterpret_cast<const float4*>(g.cs + c0 + ch * 32);
#pragma unroll
        for (int i4 = 0; i4 < 8; ++i4) {
          float4 bv = g.bias ? __ldg(b4 + i4) : make_float4(0.f, 0.f, 0.f, 0.f);
          const float a0 = __uint_as_float(v[4 * i4]), a1 = __uint_as_float(v[4 * i4 + 1]);
          const float a2 = __uint_as_float(v[4 * i4 + 2]), a3 = __uint_as_float(v[4 * i4 + 3]);
          if (fold) {           // rstd * a + (nm * cs + b) on packed pairs: 2 FFMA2 per pair instead of 4 FFMA
            const float4 cv = __ldg(c4 + i4);
            const uint64_t r2 = pack_f2(ln_rstd, ln_rstd), n2 = pack_f2(nm, nm);
            unpack_f2(fma_f2(r2, pack_f2(a0, a1), fma_f2(n2, pack_f2(cv.x, cv.y), pack_f2(bv.x, bv.y))), x[4 * i4], x[4 * i4 + 1]);
            unpack_f2(fma_f2(r2, pack_f2(a2, a3), fma_f2(n2, pack_f2(cv.z, cv.w), pack_f2(bv.z, bv.w))), x[4 * i4 + 2], x[4 * i4 + 3]);
          } else {
            x[4 * i4] = a0 + bv.x; x[4 * i4 + 1] = a1 + bv.y; x[4 * i4 + 2] = a2 + bv.z; x[4 * i4 + 3] = a3 + bv.w;
          }
        }
      };
      // fp16 T16 output tile (128 rows x 64 columns = this column quarter) of the tile: the quarter's four warps write
      // their rows into the staging tile, then one thread hands the 16 KB to the bulk-copy engine
      uint8_t* sOq = sOut + cq * TILE_BYTES;
      auto stage_begin = [&]() {          // the previous bulk store must have finished reading the staging tile
        if (q == 0 && lane == 0) bulk_wait_read();
        named_bar_sync(1 + cq, 128);
      };
      auto stage_chunk = [&](int ch, const float* x) {
#pragma unroll
        for (int c16 = 0; c16 < 4; ++c16) store_t16_chunk(sOq, r, ch * 4 + c16, x + 8 * c16);
      };
      auto stage_flush = [&](uint8_t* gtile) {
        fence_proxy_async_smem();
        named_bar_sync(1 + cq, 128);
        if (q == 0 && lane == 0) bulk_s2g(gtile, smem_u32(sOq), TILE_BYTES);
      };
      if constexpr (EPI == EPI_Q || EPI == EPI_QF32 || EPI == EPI_QKV) {
        // this warp's 64 columns are exactly one head: per-head LayerNorm (q_norm / k_norm) in two passes over TMEM
        const bool fold = g.ln_mr != nullptr;
        int part = 0, cpart = 0;                            // 0 q, 1 k, 2 v (EPI_QKV); q otherwise
        if constexpr (EPI == EPI_QKV) { cpart = c0 / g.Wq; part = cpart + g.part0; }
        const float* nw = part == 1 ? g.kn_w : g.qn_w;
        const float* nbp = part == 1 ? g.kn_b : g.qn_b;
        const float oscale = part == 0 ? g.qscale : 1.f;
        const bool norm = g.qk_norm && part < 2;
        float mean = 0.f, rs = oscale;
        if (norm) {
          float s1 = 0.f, s2 = 0.f;
#pragma unroll 1
          for (int ch = 0; ch < 2; ++ch) {
            float x[32];
            load32(ch, x, fold);
#pragma unroll
            for (int i = 0; i < 32; ++i) { s1 += x[i]; s2 = fmaf(x[i], x[i], s2); }
          }
          mean = s1 * (1.f / 64.f);
          rs = rsqrtf(fmaxf(s2 * (1.f / 64.f) - mean * mean, 0.f) + 1e-6f) * oscale;
        }
        const int row = mb * TILE_M + r;
        const bool pad = (EPI == EPI_QKV) && g.Mtok > 0 && row >= g.Mtok;      // padding tokens: exact zeros
        const int h = (EPI == EPI_QKV) ? (c0 - cpart * g.Wq) >> 6 : c0 >> 6;
#pragma unroll 1
        for (int ch = 0; ch < 2; ++ch) {
          float x[32];
          load32(ch, x, fold);
          if (norm) {
#pragma unroll
            for (int i4 = 0; i4 < 8; ++i4) {                // (x - mean) * (rstd * scale * gamma) + scale * beta
              const float4 gw = __ldg(reinterpret_cast<const float4*>(nw) + ch * 8 + i4);
              const float4 gb = __ldg(reinterpret_cast<const float4*>(nbp) + ch * 8 + i4);
              x[4 * i4] = fmaf(x[4 * i4] - mean, rs * gw.x, gb.x * oscale);
              x[4 * i4 + 1] = fmaf(x[4 * i4 + 1] - mean, rs * gw.y, gb.y * oscale);
              x[4 * i4 + 2] = fmaf(x[4 * i4 + 2] - mean, rs * gw.z, gb.z * oscale);
              x[4 * i4 + 3] = fmaf(x[4 * i4 + 3] - mean, rs * gw.w, gb.w * oscale);
            }
          } else {
#pragma unroll
            for (int i = 0; i < 32; ++i) x[i] *= oscale;
          }
          if (pad) {
#pragma unroll
            for (int i = 0; i < 32; ++i) x[i] = 0.f;
          }
          if constexpr (EPI == EPI_QF32) {
            float4* o = reinterpret_cast<float4*>(g.Fout + (size_t)row * g.N + c0 + ch * 32);
#pragma unroll
            for (int i4 = 0; i4 < 8; ++i4) o[i4] = make_float4(x[4 * i4], x[4 * i4 + 1], x[4 * i4 + 2], x[4 * i4 + 3]);
          } else if (part == 2) {                           // v: V^T tiles [H][nkv][2][64 d x 64 tok] — transposed 2-byte stores
            if (g.V32T && row < g.Mtok) {
              float* o = g.V32T + ((size_t)h * 64 + ch * 32) * g.Mtok + row;
#pragma unroll
              for (int d = 0; d < 32; ++d) o[(size_t)d * g.Mtok] = x[d];
            }
            uint8_t* tile = g.Vout + ((size_t)h * g.nkv + mb) * TILE_BYTES + (r >> 6) * (TILE_BYTES / 2) + (r & 7) * 2;
            const int c16 = (r & 63) >> 3;
#pragma unroll
            for (int d = 0; d < 32; ++d) *reinterpret_cast<__half*>(tile + sw128_off(ch * 32 + d, c16)) = __float2half_rn(x[d]);
          } else {                                          // q (T16 [Mb][heads], k-block == head) or k (K tiles [H][nkv])
            if (part == 1 && g.K32 && row < g.Mtok) {
              float4* o = reinterpret_cast<float4*>(g.K32 + ((size_t)h * g.Mtok + row) * 64 + ch * 32);
#pragma unroll
              for (int i4 = 0; i4 < 8; ++i4) o[i4] = make_float4(x[4 * i4], x[4 * i4 + 1], x[4 * i4 + 2], x[4 * i4 + 3]);
            }
            uint8_t* tile = part == 1 ? g.Kout + ((size_t)h * g.nkv + mb) * TILE_BYTES
                                      : g.Tout + ((size_t)mb * ((EPI == EPI_QKV ? g.Wq : g.N) / 64) + h) * TILE_BYTES;
            if (ch == 0) stage_begin();
            stage_chunk(ch, x);
            if (ch == 1) stage_flush(tile);
          }
        }
      } else {
        float rn = 0.f, rmean = 0.f, rM2 = 0.f, rdot = 0.f;  // running statistics of this thread's 64 output columns
#pragma unroll 1
        for (int ch = 0; ch < 2; ++ch) {
          const int c = c0 + ch * 32;
          float x[32];
          load32(ch, x, (EPI == EPI_GELU) && g.ln_mr != nullptr);
          if constexpr (EPI == EPI_GELU) {
            if (g.split_out) {
#pragma unroll
              for (int i = 0; i < 32; ++i) x[i] = gelu_erf<5>(x[i]);
            } else {
#pragma unroll
              for (int i = 0; i < 32; i += 2) gelu_erf3_pair(x[i], x[i + 1], x[i], x[i + 1]);
            }
            const int KBn = g.N / 64;
            uint8_t* tile = g.Tout + ((size_t)mb * (g.split_out ? 3 : 1) * KBn + (c >> 6)) * TILE_BYTES;
            if (g.split_out) {
#pragma unroll
              for (int c16 = 0; c16 < 4; ++c16)
                store_t16_split(tile, tile + (size_t)KBn * TILE_BYTES, tile + (size_t)2 * KBn * TILE_BYTES, r, ch * 4 + c16, x + 8 * c16);
            } else {
              if (ch == 0) stage_begin();
              stage_chunk(ch, x);
              if (ch == 1) stage_flush(tile);
            }
          } else {
            // R32: [mb][c/4][row][4]
            const size_t base = ((size_t)mb * (g.N / 4) + (c >> 2)) * TILE_M + r;
#pragma unroll
            for (int i4 = 0; i4 < 8; ++i4) {
              float4 o = make_float4(x[4 * i4], x[4 * i4 + 1], x[4 * i4 + 2], x[4 * i4 + 3]);
              const size_t idx = base + (size_t)i4 * TILE_M;
              if (EPI == EPI_RES && g.Rin) {
                const float4 rr = __ldg(reinterpret_cast<const float4*>(g.Rin) + idx);
                o.x += rr.x; o.y += rr.y; o.z += rr.z; o.w += rr.w;
                x[4 * i4] = o.x; x[4 * i4 + 1] = o.y; x[4 * i4 + 2] = o.z; x[4 * i4 + 3] = o.w;
              }
              if (g.Rout) reinterpret_cast<float4*>(g.Rout)[idx] = o;
            }
            if (g.Tcopy) {
              const int KBn = g.N / 64;
              uint8_t* tile = g.Tcopy + ((size_t)mb * (g.split_out ? 3 : 1) * KBn + (c >> 6)) * TILE_BYTES;
              if (g.split_out) {
#pragma unroll
                for (int c16 = 0; c16 < 4; ++c16)
                  store_t16_split(tile, tile + (size_t)KBn * TILE_BYTES, tile + (size_t)2 * KBn * TILE_BYTES, r, ch * 4 + c16, x + 8 * c16);
              } else {
                if (ch == 0) stage_begin();
                stage_chunk(ch, x);
                if (ch == 1) stage_flush(tile);
              }
            }
            if (g.st_out) {
              float cs_ = 0.f;
#pragma unroll
              for (int i = 0; i < 32; ++i) cs_ += x[i];
              const float cm = cs_ * (1.f / 32.f);
              float cM2 = 0.f;
#pragma unroll
              for (int i = 0; i < 32; ++i) { const float d = x[i] - cm; cM2 += d * d; }
              const float delta = cm - rmean, tot = rn + 32.f;
              rmean += delta * 32.f / tot;
              rM2 += cM2 + delta * delta * rn * 32.f / tot;
              rn = tot;
              if (g.st_k == 3) {
#pragma unroll
                for (int i4 = 0; i4 < 8; ++i4) {
                  const float4 dw = __ldg(reinterpret_cast<const float4*>(g.dotw + c) + i4);
                  rdot = fmaf(x[4 * i4], dw.x, rdot); rdot = fmaf(x[4 * i4 + 1], dw.y, rdot);
                  rdot = fmaf(x[4 * i4 + 2], dw.z, rdot); rdot = fmaf(x[4 * i4 + 3], dw.w, rdot);
                }
              }
            }
          }
        }
        if constexpr (EPI == EPI_X0 || EPI == EPI_RES) {
          if (g.st_out) {                                    // slot nb * 4 + cq  <-  (mean, M2[, dot]) of 64 columns
            float* so = g.st_out + (((size_t)mb * TILE_M + r) * (ST_PER_TILE * g.Nb) + nb * ST_PER_TILE + cq) * g.st_k;
            so[0] = rmean; so[1] = rM2;
            if (g.st_k == 3) so[2] = rdot;
          }
        }
      }
      fence_before_sync();
      __syncwarp();
      if (lane == 0) { if (rank == 0) mbar_arrive(TEMPTY(acc)); else mbar_arrive_remote(TEMPTY(acc), crank & ~1); }
    }
  }
  if (warp >= 4 && (warp & 3) == 0 && lane == 0) bulk_wait_all();   // staged output tiles have reached global memory
  fence_before_sync();
  cluster_sync();                      // the peer may still be signalling this CTA's barriers
  if (warp == 2) tmem_dealloc2(tmem, 512);
}

constexpr size_t GEMM_SMEM = 1024 + GEMM_STAGES * 2 * TILE_BYTES + ST_PER_TILE * TILE_BYTES + 256;

#include "attention_tc.cuh"

// ------------------------------------------------------------------------------------------
// Small HBM-bound stages around the GEMMs
// ------------------------------------------------------------------------------------------
// Fourier embedding (attention_blocks.py:112-130) -> T16 with K = 192: [e_hi | e_lo | e_hi]; column E (the first padding
// column) carries the constant 1 that multiplies the bias column of the collapsed c_q . query_proj weight (see QStats).
// With `qs`: also the ln_1 statistics (mean, rstd) of x0 = query_proj(e) — x0 itself is never formed.  Both are closed forms
// in e (E = 51 numbers):  mean = e . wbar + bbar,  var = e^T Gc e + 2 e . hc + cc  with the CENTRED second moments of the
// query_proj rows (no cancellation), evaluated here on the CUDA cores (2.7 kFLOP per point).
struct QStats { const float* wbar; const float* hc; const float* Gc; const float* scal; int E; };   // wbar[64], hc[64], Gc[64][64], scal = {bbar, cc}

// kF > 0: number of Fourier frequencies known at compile time (8 for every Hunyuan3D-2 checkpoint): the feature vector and
// the quadratic form are fully unrolled with static indices, so e[] lives in registers and the centred Gram matrix is read
// from shared memory as broadcast 128-bit loads of its upper triangle (off-diagonals doubled): ~1.4 k FMA per point.
// kF = 0: generic loops (e[] in local memory), any F.
template <int kF>
__global__ void __launch_bounds__(128) k_embed_tc(QuerySource src, long long n, int F, float pi_mul, uint8_t* __restrict__ T,
                                                  QStats qs, float ln_eps, float2* __restrict__ ln_mr) {
  constexpr int kE = 3 + 6 * kF, kES = (kE + 3) & ~3;          // static embedding width, Gram row stride (kF > 0)
  __shared__ __align__(16) float sG[64 * 64 + 2 * 64];
  const int r = threadIdx.x;
  if (ln_mr) {
    if constexpr (kF > 0) {
      for (int t = r; t < kE * kES; t += 128) {
        const int a = t / kES, bb = t % kES;
        sG[t] = (bb < a || bb >= kE) ? 0.f : (bb == a ? 1.f : 2.f) * qs.Gc[a * 64 + bb];
      }
    } else {
      for (int t = r; t < qs.E * qs.E; t += 128) sG[t] = qs.Gc[(t / qs.E) * 64 + (t % qs.E)];
    }
    for (int t = r; t < 64; t += 128) { sG[64 * 64 + t] = qs.wbar[t]; sG[64 * 64 + 64 + t] = qs.hc[t]; }
    __syncthreads();
  }
  // persistent over 128-row tiles: the Gram matrix is staged once per block, not once per tile
  const int ntiles = (int)((n + TILE_M - 1) / TILE_M);
  for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
  const long long qi = (long long)tile * TILE_M + r;
  float c[3] = {0.f, 0.f, 0.f};
  long long oi;
  if (qi < n) hy3d_query_point(src, qi, c[0], c[1], c[2], oi);
  float e[64];
#pragma unroll
  for (int i = 0; i < 64; ++i) e[i] = 0.f;
  e[0] = c[0]; e[1] = c[1]; e[2] = c[2];
  if constexpr (kF > 0) {
#pragma unroll
    for (int a = 0; a < 3; ++a)
#pragma unroll
      for (int f = 0; f < kF; ++f) {
        float s, co;
        sincosf(__fmul_rn(c[a], (float)(1 << f) * pi_mul), &s, &co);
        e[3 + a * kF + f] = s;
        e[3 + 3 * kF + a * kF + f] = co;
      }
  } else {
    for (int a = 0; a < 3; ++a)
      for (int f = 0; f < F; ++f) {
        float s, co;
        sincosf(__fmul_rn(c[a], exp2f((float)f) * pi_mul), &s, &co);
        e[3 + a * F + f] = s;
        e[3 + 3 * F + a * F + f] = co;
      }
  }
  if (ln_mr) {
    const float* wb = sG + 64 * 64; const float* hc = wb + 64;
    float mean = __ldg(qs.scal), lin = 0.f, quad = 0.f;
    if constexpr (kF > 0) {
#pragma unroll
      for (int a = 0; a < kE; ++a) {
        float t = 0.f;
#pragma unroll
        for (int b4 = a & ~3; b4 < kES; b4 += 4) {
          const float4 u = *reinterpret_cast<const float4*>(sG + a * kES + b4);
          t = fmaf(u.x, e[b4], t); t = fmaf(u.y, e[b4 + 1], t); t = fmaf(u.z, e[b4 + 2], t); t = fmaf(u.w, e[b4 + 3], t);
        }
        quad = fmaf(e[a], t, quad);
        mean = fmaf(e[a], wb[a], mean);
        lin = fmaf(e[a], hc[a], lin);
      }
    } else {
      const int E = qs.E;
      for (int a = 0; a < E; ++a) {
        const float ea = e[a];
        float t = 0.f;
        for (int b = 0; b < E; ++b) t = fmaf(sG[a * E + b], e[b], t);
        quad = fmaf(ea, t, quad);
        mean = fmaf(ea, wb[a], mean);
        lin = fmaf(ea, hc[a], lin);
      }
    }
    const float var = fmaxf(quad + 2.f * lin + __ldg(qs.scal + 1), 0.f);
    ln_mr[qi] = make_float2(mean, rsqrtf(var + ln_eps));          // rows past n: statistics of the zero point, never used
  }
  {
    const int ec = kF > 0 ? kE : 3 + 6 * F;
    if (ec < 64) e[ec] = 1.0f;                                      // constant column (bias of the collapsed weight)
  }
  uint8_t* t0 = T + (size_t)tile * 3 * TILE_BYTES;
#pragma unroll
  for (int c16 = 0; c16 < 8; ++c16) {
    float hi[8], lo[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      float v = e[c16 * 8 + i];
      float h = __half2float(__float2half_rn(v));
      hi[i] = h; lo[i] = v - h;
    }
    store_t16_chunk(t0, r, c16, hi);
    store_t16_chunk(t0 + TILE_BYTES, r, c16, lo);
    store_t16_chunk(t0 + 2 * TILE_BYTES, r, c16, hi);
  }
  }
}

// LayerNorm over N columns: R32 -> T16 (one thread per row, one block per 128-row tile)
// kSplit: the row is written as [hi | lo | hi] (3 * N/64 k-blocks) for the 3-term split GEMM.
template <bool kSplit>
__global__ void __launch_bounds__(128) k_ln_tc(const float* __restrict__ R, int N, const float* __restrict__ gam,
                                                const float* __restrict__ bet, float eps, uint8_t* __restrict__ T) {
  const int r = threadIdx.x;
  const float4* x = reinterpret_cast<const float4*>(R) + (size_t)blockIdx.x * (N / 4) * TILE_M + r;
  const int n4 = N / 4;
  const float shift = __ldg(&x[0]).x;
  float s = 0.f, ss = 0.f;
#pragma unroll 8
  for (int c = 0; c < n4; ++c) {
    float4 v = __ldg(&x[(size_t)c * TILE_M]);
    float a0 = v.x - shift, a1 = v.y - shift, a2 = v.z - shift, a3 = v.w - shift;
    s += (a0 + a1) + (a2 + a3);
    ss += (a0 * a0 + a1 * a1) + (a2 * a2 + a3 * a3);
  }
  const float ms = s / N;
  const float mean = shift + ms;
  const float var = fmaxf(ss / N - ms * ms, 0.f);
  const float rstd = rsqrtf(var + eps);
  const int KBn = N / 64;
  uint8_t* tbase = T + (size_t)blockIdx.x * (kSplit ? 3 : 1) * KBn * TILE_BYTES;
#pragma unroll 4
  for (int c8 = 0; c8 < N / 8; ++c8) {
    float4 v0 = __ldg(&x[(size_t)(2 * c8) * TILE_M]), v1 = __ldg(&x[(size_t)(2 * c8 + 1) * TILE_M]);
    const float4 g0 = __ldg(reinterpret_cast<const float4*>(gam) + 2 * c8), g1 = __ldg(reinterpret_cast<const float4*>(gam) + 2 * c8 + 1);
    const float4 b0 = __ldg(reinterpret_cast<const float4*>(bet) + 2 * c8), b1 = __ldg(reinterpret_cast<const float4*>(bet) + 2 * c8 + 1);
    float o[8];
    o[0] = (v0.x - mean) * rstd * g0.x + b0.x; o[1] = (v0.y - mean) * rstd * g0.y + b0.y;
    o[2] = (v0.z - mean) * rstd * g0.z + b0.z; o[3] = (v0.w - mean) * rstd * g0.w + b0.w;
    o[4] = (v1.x - mean) * rstd * g1.x + b1.x; o[5] = (v1.y - mean) * rstd * g1.y + b1.y;
    o[6] = (v1.z - mean) * rstd * g1.z + b1.z; o[7] = (v1.w - mean) * rstd * g1.w + b1.w;
    if constexpr (kSplit) {
      float hi[8], lo[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) { hi[i] = __half2float(__float2half_rn(o[i])); lo[i] = o[i] - hi[i]; }
      store_t16_chunk(tbase + (size_t)(c8 >> 3) * TILE_BYTES, r, c8 & 7, hi);
      store_t16_chunk(tbase + (size_t)(KBn + (c8 >> 3)) * TILE_BYTES, r, c8 & 7, lo);
      store_t16_chunk(tbase + (size_t)(2 * KBn + (c8 >> 3)) * TILE_BYTES, r, c8 & 7, hi);
    } else {
      store_t16_chunk(tbase + (size_t)(c8 >> 3) * TILE_BYTES, r, c8 & 7, o);
    }
  }
}

// logits from the per-row partial statistics of x2 written by the last GEMM's epilogue:
// [ln_post](x2) . wout + bout = rstd * (dot(x2, gamma*wout) - mean * C1) + C2   (C1 = sum gamma*wout, C2 = beta.wout + bout)
__global__ void __launch_bounds__(128) k_head_final(const float* __restrict__ st, int S, int n_p, int ln_post, const float* __restrict__ c12,
                                                     QuerySource src, long long n, float* __restrict__ out, int out_mode) {
  const long long qi = (long long)blockIdx.x * TILE_M + threadIdx.x;
  if (qi >= n) return;
  float mean, rstd, dot;
  merge_row_stats<3>(st + (size_t)qi * S * 3, S, n_p, 1e-5f, mean, rstd, &dot);
  const float v = ln_post ? rstd * (dot - mean * __ldg(c12)) + __ldg(c12 + 1) : dot + __ldg(c12 + 1);
  long long oi = qi;
  float w = v;
  if (out_mode == 1) {
    oi = src.index[qi];
    if (oi < 0) return;
    // scattered into a sparse level: a logit that equals the "unvisited" sentinel IS unvisited to everything downstream
    // (volume_decoders.py:275 turns it into NaN; the next refinement treats both alike) — written as NaN right here, so the
    // last level can be pre-filled with NaN and needs no full-grid sentinel pass afterwards
    if (v == HY3D_SENTINEL) w = __int_as_float(0x7fc00000);
  }
  out[oi] = w;
}

// head constants: dotw = gamma_post * wout (or wout), c12 = {sum dotw, beta_post . wout + bout}
__global__ void __launch_bounds__(256) k_head_consts(const float* __restrict__ gam, const float* __restrict__ bet,
                                                      const float* __restrict__ wout, const float* __restrict__ bout, int W,
                                                      float* __restrict__ dotw, float* __restrict__ c12) {
  __shared__ float r1[256], r2[256];
  float a = 0.f, b = 0.f;
  for (int k = threadIdx.x; k < W; k += 256) {
    const float d = gam ? gam[k] * wout[k] : wout[k];
    dotw[k] = d; a += d;
    if (bet) b = fmaf(bet[k], wout[k], b);
  }
  r1[threadIdx.x] = a; r2[threadIdx.x] = b;
  __syncthreads();
  for (int o = 128; o; o >>= 1) { if (threadIdx.x < o) { r1[threadIdx.x] += r1[threadIdx.x + o]; r2[threadIdx.x] += r2[threadIdx.x + o]; } __syncthreads(); }
  if (threadIdx.x == 0) { c12[0] = r1[0]; c12[1] = r2[0] + bout[0]; }
}

__global__ void k_add_vec(const float* __restrict__ a, const float* __restrict__ b, int n, float* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = (a ? a[i] : 0.f) + (b ? b[i] : 0.f);
}

// LayerNorm fold: Wf[j][k] = gamma[k] * W[j][k];  cs[j] = sum_k fp16(Wf[j][k]);  bb[j] = sum_k beta[k] W[j][k] + bias[j]
// (one warp per output row j)
// permH > 0: source rows are [head][q|k|v][64] (c_qkv, attention_blocks.py:318-321; parts = 3) or [head][k|v][64] (c_kv, :205-208;
// parts = 2), output rows [q | k | v] / [k | v] head-contiguous.
// exact_cs: column sums of the unrounded folded weight (3-term split GEMMs) instead of its fp16 rounding.
__global__ void k_fold_ln(const float* __restrict__ Wsrc, const float* __restrict__ gam, const float* __restrict__ bet,
                          const float* __restrict__ bias, int N, int K, float* __restrict__ Wf, float* __restrict__ cs,
                          float* __restrict__ bb, int permH, int exact_cs, int parts = 3) {
  const int j = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (j >= N) return;
  int jd = j;
  if (permH) { const int hs = 64 * parts, h = j / hs, p = (j % hs) / 64, d = j % 64; jd = p * (permH * 64) + h * 64 + d; }
  float a = 0.f, b = 0.f;
  for (int k = lane; k < K; k += 32) {
    const float w = Wsrc[(size_t)j * K + k];
    const float wf = gam ? gam[k] * w : w;
    Wf[(size_t)jd * K + k] = wf;
    a += exact_cs ? wf : __half2float(__float2half_rn(wf));
    if (bet) b = fmaf(bet[k], w, b);
  }
  for (int o = 16; o; o >>= 1) { a += __shfl_xor_sync(0xffffffffu, a, o); b += __shfl_xor_sync(0xffffffffu, b, o); }
  if (lane == 0) { cs[jd] = a; bb[jd] = b + (bias ? bias[j] : 0.f); }
}

// c_q . query_proj collapsed (both are linear, ln_1 between them only scales / shifts rows):
//   c_q(ln_1(x0)) = rstd (x0 W'^T - mean cs) + bb   (the LayerNorm fold)   and   x0 = e Wqp^T + bqp
//   =>  x0 W'^T = e (W' Wqp)^T + W' bqp =: e Wc^T + d        — a K = 51 contraction instead of K = 1024, x0 never formed.
// Wc_out[j][c] = sum_k Wf[j][k] Wqp[k][c] (c < E),  Wc_out[j][E] = d[j] = sum_k Wf[j][k] bqp[k]   (float64 accumulation)
__global__ void k_combine_q(const float* __restrict__ Wf, const float* __restrict__ Wqp, const float* __restrict__ bqp, int W, int E,
                            float* __restrict__ Wc) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= W * (E + 1)) return;
  const int j = t / (E + 1), c = t % (E + 1);
  double acc = 0.0;
  for (int k = 0; k < W; ++k) acc += (double)Wf[(size_t)j * W + k] * (double)(c < E ? Wqp[(size_t)k * E + c] : bqp[k]);
  Wc[t] = (float)acc;
}
// centred moments of the query_proj rows for the closed-form ln_1 statistics of x0 (k_embed_tc): one block
__global__ void __launch_bounds__(256) k_qstats_consts(const float* __restrict__ Wqp, const float* __restrict__ bqp, int W, int E,
                                                        float* __restrict__ wbar, float* __restrict__ hc, float* __restrict__ Gc,
                                                        float* __restrict__ scal) {
  __shared__ double sw[64];
  __shared__ double sb;
  for (int a = threadIdx.x; a < 64; a += 256) {
    double m = 0.0;
    if (a < E) { for (int c = 0; c < W; ++c) m += Wqp[(size_t)c * E + a]; m /= W; }
    sw[a] = m; wbar[a] = (float)m;
  }
  if (threadIdx.x == 0) { double m = 0.0; for (int c = 0; c < W; ++c) m += bqp[c]; sb = m / W; }
  __syncthreads();
  for (int t = threadIdx.x; t < 64 * 64; t += 256) {
    const int a = t / 64, b = t % 64;
    double g = 0.0;
    if (a < E && b < E) { for (int c = 0; c < W; ++c) g += ((double)Wqp[(size_t)c * E + a] - sw[a]) * ((double)Wqp[(size_t)c * E + b] - sw[b]); g /= W; }
    Gc[t] = (float)g;
  }
  for (int a = threadIdx.x; a < 64; a += 256) {
    double h = 0.0;
    if (a < E) { for (int c = 0; c < W; ++c) h += ((double)Wqp[(size_t)c * E + a] - sw[a]) * ((double)bqp[c] - sb); h /= W; }
    hc[a] = (float)h;
  }
  if (threadIdx.x == 0) {
    double v = 0.0;
    for (int c = 0; c < W; ++c) v += ((double)bqp[c] - sb) * ((double)bqp[c] - sb);
    scal[0] = (float)sb; scal[1] = (float)(v / W);
  }
}

// ---- operand image builders ----------------------------------------------------------------
// fp32 row-major W[N, K] (ld = ldw) -> B16 tiles.  mode 0: plain.  mode 1: query_proj split:
// K_out = 192 = [W_hi | W_hi | W_lo] over the first E columns (zero padded to 64).  mode 2: the same
// 3-term split for a full [N, K/3] matrix.  kbs: k-blocks per 256-row block of `out` (0 = K / 64; more when the image is
// one part of a K-concatenated operand).
__global__ void k_build_b16(const float* __restrict__ Wsrc, int N, int K, int ldw, int mode, int E, uint8_t* __restrict__ out,
                            int kbs = 0) {
  const int KB = K / 64;
  long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;    // one 16-byte chunk per thread
  long long total = (long long)N * (K / 8);
  if (t >= total) return;
  const int c8 = (int)(t % (K / 8)); const int n = (int)(t / (K / 8));
  const int kb = c8 >> 3, c16 = c8 & 7;
  float v[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    int k = c8 * 8 + i;
    float w;
    if (mode == 0) w = Wsrc[(size_t)n * ldw + k];
    else if (mode == 2) {                      // [W_hi | W_hi | W_lo], each K/3 wide
      const int Ks = K / 3, part = k / Ks;
      float full = Wsrc[(size_t)n * ldw + (k - part * Ks)];
      float hi = __half2float(__float2half_rn(full));
      w = part < 2 ? hi : full - hi;
    } else {
      int part = k / 64, kk = k % 64;
      float full = kk < E ? Wsrc[(size_t)n * ldw + kk] : 0.f;
      float hi = __half2float(__float2half_rn(full));
      w = part < 2 ? hi : full - hi;
    }
    v[i] = w;
  }
  uint8_t* tile = out + ((size_t)(n / BN) * (kbs ? kbs : KB) + kb) * BTILE_BYTES;
  store_t16_chunk(tile, n % BN, c16, v);
}

// k32 [H, M, 64] -> K tiles; vT32 [H, 64, M] -> V^T tiles (zero padded to Mpad tokens)
__global__ void k_build_kv(const float* __restrict__ k32, const float* __restrict__ vT32, int H, int M, int nkv,
                           uint8_t* __restrict__ kt, uint8_t* __restrict__ vt) {
  long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;    // one 16-byte chunk of K and of V^T per thread
  const long long per_head = (long long)nkv * 128 * 8;
  if (t >= per_head * H) return;
  const int h = (int)(t / per_head); long long rem = t % per_head;
  {  // K: row = token, chunk over d
    const int tok = (int)(rem / 8), c16 = (int)(rem % 8);
    float v[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) v[i] = tok < M ? k32[((size_t)h * M + tok) * 64 + c16 * 8 + i] : 0.f;
    uint8_t* tile = kt + ((size_t)h * nkv + tok / 128) * TILE_BYTES;
    store_t16_chunk(tile, tok % 128, c16, v);
  }
  {  // V^T: row = d, chunk over 8 tokens
    const int d = (int)(rem % 64); const int tc8 = (int)(rem / 64);          // token chunk index over all padded tokens
    const int tok0 = tc8 * 8, j = tok0 / 128, kbk = (tok0 % 128) / 64, c16 = (tok0 % 64) / 8;
    float v[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) v[i] = (tok0 + i) < M ? vT32[((size_t)h * 64 + d) * M + tok0 + i] : 0.f;
    uint8_t* tile = vt + ((size_t)h * nkv + j) * TILE_BYTES + kbk * (TILE_BYTES / 2);
    store_t16_chunk(tile, d, c16, v);
  }
}

// Tensor map over an operand image viewed as a plain 2-D byte array (every UMMA tile is a contiguous 16 KB block, already
// swizzled in memory): box = one 16 KB tile, no hardware swizzle.  cuTensorMapEncodeTiled comes
// from the driver through the runtime (no link-time libcuda dependency).
int make_rows_map(hy3d_ctx* ctx, CUtensorMap* m, const void* base, uint64_t rows, int box_rows = 8) {
  typedef CUresult (*encode_fn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
  if (!ctx->tmap_encode) {
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult q;
    HY3D_CUDA(ctx, cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q));
    if (!fn || q != cudaDriverEntryPointSuccess) return hy3d_fail(ctx, HY3D_ERR_CUDA, "cuTensorMapEncodeTiled unavailable");
    ctx->tmap_encode = fn;
  }
  const encode_fn encode = reinterpret_cast<encode_fn>(ctx->tmap_encode);
  // `rows` counts 128-byte rows; the map itself uses rows of 256 x 8 bytes (2 KB): a 16 KB tile = box of 8 such rows, so the
  // TMA unit walks 8 long rows per tile instead of 128 short ones
  const cuuint64_t dims[2] = {256, rows / 16};
  const cuuint64_t strides[1] = {2048};
  const cuuint32_t box[2] = {256, (cuuint32_t)box_rows};     // 8 rows of 2 KB = one 16 KB tile (4 = half of it)
  const cuuint32_t estr[2] = {1, 1};
  // 256 B L2 promotion, the widest: every box row is 2 KB of contiguous bytes that the copy reads whole
  const CUresult r = encode(m, CU_TENSOR_MAP_DATA_TYPE_UINT64, 2, const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                            CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return hy3d_fail(ctx, HY3D_ERR_CUDA, "cuTensorMapEncodeTiled failed (%d)", (int)r);
  return 0;
}

// (mean, rstd) per row from the S partial (mean, M2) slots a producer epilogue wrote: once per row here, instead of
// S strided loads per row in every consumer tile (which made the consumer epilogues LSU-bound)
__global__ void k_finish_stats(const float* __restrict__ st, int S, int n_p, float eps, long long rows, float2* __restrict__ out) {
  const long long row = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (row >= rows) return;
  float mean, rstd;
  merge_row_stats<2>(st + row * S * 2, S, n_p, eps, mean, rstd);
  out[row] = make_float2(mean, rstd);
}

template <int EPI>
int launch_gemm(hy3d_ctx* ctx, const GemmTC& g, int fam) {
  HY3D_CUDA(ctx, cudaFuncSetAttribute(k_gemm_tc<EPI>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)GEMM_SMEM));
  int& max_clusters = ctx->gemm_max_clusters[EPI];                 // co-resident 2-CTA clusters (persistent grid)
  if (max_clusters == 0) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(ctx->num_sms / GEMM_CL * GEMM_CL); cfg.blockDim = dim3(GEMM_THREADS); cfg.dynamicSmemBytes = GEMM_SMEM;
    int n = 0;
    if (cudaOccupancyMaxActiveClusters(&n, k_gemm_tc<EPI>, &cfg) != cudaSuccess || n <= 0) { n = ctx->num_sms / GEMM_CL; (void)cudaGetLastError(); }
    max_clusters = n < ctx->num_sms / GEMM_CL ? n : ctx->num_sms / GEMM_CL;
    if (getenv("HY3D_VERBOSE")) fprintf(stderr, "[hy3dgeo] k_gemm_tc<%d>: %d co-resident %d-CTA clusters\n", EPI, max_clusters, GEMM_CL);
  }
  const int pairs = ((g.Mb + GEMM_CL - 1) / GEMM_CL) * g.Nb;        // one group of GEMM_CL vertically adjacent tiles per cluster iteration
  const int grid = GEMM_CL * (pairs < max_clusters ? pairs : max_clusters);
  HY3D_PROF(ctx, fam);
  GemmTC gd = g;
  if (g.st_in) {
    const long long rows = (long long)g.Mb * TILE_M;
    HY3D_CUDA(ctx, ctx->ln_mr.reserve((size_t)rows * sizeof(float2)));
    gd.ln_mr = ctx->ln_mr.as<float2>();
    k_finish_stats<<<(unsigned)ceil_div64(rows, 256), 256, 0, ctx->stream>>>(g.st_in, g.st_slots, g.st_np, g.ln_eps, rows, ctx->ln_mr.as<float2>());
    ctx->launches++;
  }
  CUtensorMap tmA, tmA2, tmB;
  const int kb1 = g.KB1 ? g.KB1 : g.KB;
  if (int rc = make_rows_map(ctx, &tmA, g.A, (uint64_t)g.Mb * kb1 * 128)) return rc;
  if (int rc = make_rows_map(ctx, &tmA2, g.A2 ? g.A2 : g.A, (uint64_t)g.Mb * (g.A2 ? g.KB - kb1 : kb1) * 128)) return rc;
  if (int rc = make_rows_map(ctx, &tmB, g.B, (uint64_t)g.Nb * g.KB * 256, GEMM_CL == 4 ? 4 : 8)) return rc;
  k_gemm_tc<EPI><<<grid, GEMM_THREADS, GEMM_SMEM, ctx->stream>>>(gd, tmA, tmA2, tmB);
  HY3D_LAUNCH_CHECK(ctx);
  return 0;
}

// Attention launch: the bounded-score kernel when `fast` (see attention_tc.cuh), else the online-softmax kernel.
template <class K>
int launch_attn_kernel(hy3d_ctx* ctx, K kern, const AttnTC& a, int threads) {
  HY3D_CUDA(ctx, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ATT_SMEM));
  const int items = a.share_kv ? ((a.Pb + 1) / 2) * a.H : a.Pb * (a.H / 2);
  const int grid = items < ctx->num_sms ? items : ctx->num_sms;
  kern<<<grid, threads, ATT_SMEM, ctx->stream>>>(a);
  return 0;
}
int launch_attn(hy3d_ctx* ctx, AttnTC a, bool fast, int fam, bool shifted = false) {
  if (ctx->force_online_softmax) fast = false;
  KVState& kv = ctx->kv;
  if (fast && shifted) {                                   // decoder attention with measured per-head bounds (k_head_shift)
    const size_t items = (size_t)a.Pb * (a.H / 2);
    HY3D_CUDA(ctx, kv.redo.reserve((1 + 2 * items) * sizeof(int)));
    HY3D_CUDA(ctx, cudaMemsetAsync(kv.redo.p, 0, (1 + 2 * items) * sizeof(int), ctx->stream));
    a.head_shift = kv.head_shift.as<float>();
    a.redo_count = kv.redo.as<int>(); a.redo_list = a.redo_count + 1; a.redo_flag = a.redo_list + items;
  }
  HY3D_PROF(ctx, fam);
  // one K/V set for all query tiles (no per-tile KV groups): pairs of query tiles share every K/V tile they stream
  a.share_kv = a.tile_group == nullptr ? 1 : 0;
  const int rc = fast ? launch_attn_kernel(ctx, k_attn_fast, a, ATT_FAST_THREADS) : launch_attn_kernel(ctx, k_attn_tc<0>, a, ATT_THREADS);
  if (rc) return rc;
  HY3D_LAUNCH_CHECK(ctx);
  if (fast && shifted) {
    // exact redo of the (query tile, head pair) items the bounded-score kernel flagged (rows whose probabilities all fell
    // below 2^-12 of their head's bound — normally none): the online-softmax kernel over the device work list.  A launch
    // with an empty list costs a few microseconds; no host round trip decides anything.
    AttnTC r = a;
    r.share_kv = 0; r.head_shift = nullptr; r.redo_count = nullptr; r.redo_list = nullptr; r.redo_flag = nullptr;
    r.work_count = a.redo_count; r.work_list = a.redo_list;
    HY3D_PROF(ctx, fam);
    HY3D_CUDA(ctx, cudaFuncSetAttribute(k_attn_tc<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ATT_SMEM));
    const int items = a.Pb * (a.H / 2);
    k_attn_tc<0><<<items < ctx->num_sms ? items : ctx->num_sms, ATT_THREADS, ATT_SMEM, ctx->stream>>>(r);
    HY3D_LAUNCH_CHECK(ctx);
  }
  return 0;
}

// Upper bound of |q . k| * scale * log2e for LayerNorm-ed q and k (over d = 64 head dims, affine (w, b)):
// ||w * xhat + b|| <= sqrt(d) * max|w| + ||b||.  Reads the 4 x 64 norm parameters back once, at weight-load time.
int attn_score_bound(hy3d_ctx* ctx, const float* qw, const float* qb, const float* kw, const float* kb, float* bound, float* qbound = nullptr) {
  float h[4][64];
  const float* src[4] = {qw, qb, kw, kb};
  HY3D_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  for (int i = 0; i < 4; ++i) HY3D_CUDA(ctx, cudaMemcpy(h[i], src[i], sizeof(float) * 64, cudaMemcpyDeviceToHost));
  float n[2];
  for (int i = 0; i < 2; ++i) {
    float mw = 0.f, nb = 0.f;
    for (int d = 0; d < 64; ++d) { mw = fmaxf(mw, fabsf(h[2 * i][d])); nb += h[2 * i + 1][d] * h[2 * i + 1][d]; }
    n[i] = 8.f * mw + sqrtf(nb);
  }
  *bound = n[0] * n[1] * 0.125f * LOG2E;
  if (qbound) *qbound = n[0];
  return 0;
}

// Per head: max over tokens of ||k_t|| (the K the attention kernel will see, after k_norm) -> the head's true score bound
// B_h = qbound * max||k|| * scale * log2e and its shift c_h = max(0, B_h - 15.9): exp2(s - c_h) can then never overflow fp16
// whatever the norm gains of the checkpoint are.  k32: fp32 [H, M, 64].  out: shift[H] then bound[H].
constexpr float ATT_SHIFT_MAX_BOUND = 40.f;     // beyond this the weight-only bound sends the decoder to the online-softmax kernel
__global__ void __launch_bounds__(256) k_head_shift(const float* __restrict__ k32, int M, float qbound, float* __restrict__ out, int H) {
  const int h = blockIdx.x;
  float mx = 0.f;
  for (int t = threadIdx.x; t < M; t += 256) {
    const float4* kr = reinterpret_cast<const float4*>(k32 + ((size_t)h * M + t) * 64);
    float s = 0.f;
#pragma unroll
    for (int d4 = 0; d4 < 16; ++d4) { const float4 v = __ldg(kr + d4); s = fmaf(v.x, v.x, s); s = fmaf(v.y, v.y, s); s = fmaf(v.z, v.z, s); s = fmaf(v.w, v.w, s); }
    mx = fmaxf(mx, s);
  }
  __shared__ float red[8];
  for (int o = 16; o; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = mx;
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < 8; ++w) mx = fmaxf(mx, red[w]);
    // fp16 rounding of q and k (2^-11 relative each) and of the product sum: 0.2 % head-room on the bound
    const float b = qbound * sqrtf(mx) * 0.125f * LOG2E * 1.002f;
    out[h] = fmaxf(b - ATT_FAST_BOUND, 0.f);
    out[H + h] = b;
  }
}

}  // namespace

// ------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------
int hy3d_tc_prepare_weights(hy3d_ctx* ctx) {
  DecoderWeights& w = ctx->w;
  if (w.D != 64 || w.W % 256 || (w.W * w.R) % 256) {
    // the tcgen05 path is specialised to head_dim 64 and widths that tile by 256; other shapes can
    // only run in HY3D_PRECISION_FP32_SIMT
    w.t_qp = nullptr;
    return 0;
  }
  const size_t W = w.W, R = w.R;
  const size_t n_qp = W * 192, n_fc = R * W * W, n_mp = R * W * W, n_cq3 = 3 * W * W;
  const size_t n_ckv3 = 2 * W * 3 * W, n_lp3 = w.has_latents_proj ? W * 3 * (size_t)w.LW : 0;
  const size_t n_cpx = W * (W + 192);                               // [c_proj | query_proj split] concatenated along K
  const size_t n_cqx = W * 192;                                     // c_q . query_proj collapsed: [Wc_hi | Wc_hi | Wc_lo]
  HY3D_CUDA(ctx, w.tc.reserve((n_qp + n_fc + n_mp + n_cq3 + n_ckv3 + n_lp3 + n_cpx + n_cqx) * 2));
  __half* p_qp = w.tc.as<__half>(); __half* p_fc = p_qp + n_qp; __half* p_mp = p_fc + n_fc; __half* p_cq3 = p_mp + n_mp;
  __half* p_ckv3 = p_cq3 + n_cq3; __half* p_lp3 = p_ckv3 + n_ckv3; __half* p_cpx = p_lp3 + n_lp3; __half* p_cqx = p_cpx + n_cpx;
  auto build = [&](const float* src, int N, int K, int ldw, int mode, __half* dst, int kbs = 0) -> int {
    long long total = (long long)N * (K / 8);
    k_build_b16<<<(unsigned)ceil_div64(total, 256), 256, 0, ctx->stream>>>(src, N, K, ldw, mode, w.E, reinterpret_cast<uint8_t*>(dst), kbs);
    HY3D_LAUNCH_CHECK(ctx);
    return 0;
  };
  // ln_1 folded into c_q, ln_3 into c_fc, ln_post into the head (see GemmTC)
  const size_t n_qs = 64 + 64 + 64 * 64 + 64 + W * 64 + W;          // wbar, hc, Gc, scalars, Wc rows (E + 1 <= 64 columns), exact cs
  HY3D_CUDA(ctx, w.fold.reserve((W + R * W + R * W + W + 64 + 4 * W + W + n_qs) * sizeof(float)));
  HY3D_CUDA(ctx, ctx->ws[10].reserve(R * W * W * sizeof(float)));
  float* fb = w.fold.as<float>();
  float* bb_q = fb; float* cs_fc = bb_q + W; float* bb_fc = cs_fc + R * W; float* dotw = bb_fc + R * W; float* c12 = dotw + W;
  float* Wf = ctx->ws[10].as<float>();
  if (int rc = build(w.qp_w, (int)W, 192, w.E, 1, p_qp)) return rc;
  {   // collapsed c_q . query_proj + the closed-form ln_1 statistics of x0
    float* qsb = c12 + 64 + 4 * W + W;
    float* wbar = qsb; float* hcv = wbar + 64; float* Gc = hcv + 64; float* scal = Gc + 64 * 64; float* Wc = scal + 64;
    float* cs_qx = Wc + W * 64;
    const int E1 = w.E + 1;
    if (E1 > 64) return hy3d_fail(ctx, HY3D_ERR_UNSUPPORTED, "Fourier embedding wider than 63 columns");
    // the collapsed product is fp32-grade (3-term split): its LayerNorm fold needs the EXACT column sums of the folded weight
    k_fold_ln<<<(unsigned)((W + 7) / 8), 256, 0, ctx->stream>>>(w.cq_w, w.ln1_w, w.ln1_b, w.cq_b, (int)W, (int)W, Wf, cs_qx, bb_q, 0, 1);
    HY3D_LAUNCH_CHECK(ctx);
    k_combine_q<<<(unsigned)((W * E1 + 255) / 256), 256, 0, ctx->stream>>>(Wf, w.qp_w, w.qp_b, (int)W, w.E, Wc);
    HY3D_LAUNCH_CHECK(ctx);
    k_qstats_consts<<<1, 256, 0, ctx->stream>>>(w.qp_w, w.qp_b, (int)W, w.E, wbar, hcv, Gc, scal);
    HY3D_LAUNCH_CHECK(ctx);
    const int saveE = w.E;
    w.E = E1;                                                        // k_build_b16 mode 1 reads w.E valid columns
    const int rc = build(Wc, (int)W, 192, E1, 1, p_cqx);
    w.E = saveE;
    if (rc) return rc;
    w.t_cqx = p_cqx; w.qs_wbar = wbar; w.qs_hc = hcv; w.qs_Gc = Gc; w.qs_scal = scal; w.cs_qx = cs_qx;
  }
  k_fold_ln<<<(unsigned)((R * W + 7) / 8), 256, 0, ctx->stream>>>(w.fc_w, w.ln3_w, w.ln3_b, w.fc_b, (int)(R * W), (int)W, Wf, cs_fc, bb_fc, 0, 0);
  HY3D_LAUNCH_CHECK(ctx);
  if (int rc = build(Wf, (int)(R * W), (int)W, (int)W, 0, p_fc)) return rc;
  k_head_consts<<<1, 256, 0, ctx->stream>>>(w.ln_post ? w.lnp_w : nullptr, w.ln_post ? w.lnp_b : nullptr, w.out_w, w.out_b, (int)W, dotw, c12);
  HY3D_LAUNCH_CHECK(ctx);
  w.bb_q = bb_q; w.cs_fc = cs_fc; w.bb_fc = bb_fc; w.dotw = dotw; w.c12 = c12;
  if (int rc = build(w.mp_w, (int)W, (int)(R * W), (int)(R * W), 0, p_mp)) return rc;
  if (int rc = build(w.cq_w, (int)W, (int)(3 * W), (int)W, 2, p_cq3)) return rc;
  w.t_qp = p_qp; w.t_fc = p_fc; w.t_mp = p_mp; w.t_cq3 = p_cq3;
  w.attn_bound = INFINITY; w.attn_qbound = INFINITY; w.attn_fast = false;
  if (w.qk_norm) {
    if (int rc = attn_score_bound(ctx, w.qn_w, w.qn_b, w.kn_w, w.kn_b, &w.attn_bound, &w.attn_qbound)) return rc;
    // bounded-score kernel whenever q/k norms bound the scores at all; above 15.9 (weight-only bound) the per-head shift from
    // the MEASURED max ||k|| of each latent set (k_head_shift) keeps exp2 inside fp16 and an exact redo pass covers the rows
    // whose scores sit far below their head's bound (hy3d_tc_head_shift, launch_attn)
    w.attn_fast = w.attn_bound <= ATT_SHIFT_MAX_BOUND;
  }
  if (getenv("HY3D_VERBOSE")) fprintf(stderr, "[hy3dgeo] decoder attention score bound (weights) %.3f -> %s kernel\n", w.attn_bound, w.attn_fast ? "bounded-score" : "online-softmax");
  // per-latent K/V projection on the tensor path (hy3d_tc_project_kv): ln_2 folded into c_kv, rows permuted
  // [head][k|v][64] -> [k | v], 3-term split (fp32-grade: K/V feed every query and the FlashVDM token selection)
  w.t_ckv3 = nullptr; w.t_lp3 = nullptr;
  if (w.LW % 64 == 0 && (!w.has_latents_proj || w.LW % 64 == 0)) {
    float* cs_kv = c12 + 64; float* bb_kv = cs_kv + 2 * W;
    k_fold_ln<<<(unsigned)((2 * W + 7) / 8), 256, 0, ctx->stream>>>(w.ckv_w, w.ln2_w, w.ln2_b, w.has_ckv_b ? w.ckv_b : nullptr, (int)(2 * W),
                                                                    (int)W, Wf, cs_kv, bb_kv, w.H, 1, 2);
    HY3D_LAUNCH_CHECK(ctx);
    if (int rc = build(Wf, (int)(2 * W), (int)(3 * W), (int)W, 2, p_ckv3)) return rc;
    if (w.has_latents_proj)
      if (int rc = build(w.lp_w, (int)W, (int)(3 * w.LW), (int)w.LW, 2, p_lp3)) return rc;
    w.t_ckv3 = p_ckv3; w.t_lp3 = w.has_latents_proj ? p_lp3 : nullptr; w.cs_kv = cs_kv; w.bb_kv = bb_kv;
  }
  // x1 = x0 + c_proj(attn) + b  as ONE GEMM over K = W + 192: [attn | e_hi | e_lo | e_hi] [W_o | W_qp,hi | W_qp,hi | W_qp,lo]^T
  // + (b_o + b_qp) — the fp32 x0 never travels through HBM.  Per 256-row block the image holds the W / 64 k-blocks of c_proj,
  // then the 3 of the query_proj split.
  {
    const int kb_o = (int)W / 64;
    if (int rc = build(w.cproj_w, (int)W, (int)W, (int)W, 0, p_cpx, kb_o + 3)) return rc;
    if (int rc = build(w.qp_w, (int)W, 192, w.E, 1, p_cpx + (size_t)kb_o * (BTILE_BYTES / 2), kb_o + 3)) return rc;
    float* b_cpx = c12 + 64 + 4 * W;
    k_add_vec<<<(unsigned)((W + 255) / 256), 256, 0, ctx->stream>>>(w.cproj_b, w.qp_b, (int)W, b_cpx);
    HY3D_LAUNCH_CHECK(ctx);
    w.t_cpx = p_cpx; w.b_cpx = b_cpx;
  }
  return 0;
}

// Measured per-head score bounds of the K just prepared (kv.k32) -> kv.head_shift; see k_head_shift.
int hy3d_tc_head_shift(hy3d_ctx* ctx) {
  DecoderWeights& w = ctx->w;
  KVState& kv = ctx->kv;
  kv.shifted = false;
  if (!w.attn_fast) return 0;
  HY3D_CUDA(ctx, kv.head_shift.reserve((size_t)2 * w.H * sizeof(float)));
  HY3D_PROF(ctx, FAM_KV);
  k_head_shift<<<w.H, 256, 0, ctx->stream>>>(kv.k32.as<float>(), kv.M, w.attn_qbound, kv.head_shift.as<float>(), w.H);
  HY3D_LAUNCH_CHECK(ctx);
  kv.shifted = w.attn_bound > ATT_FAST_BOUND;          // weight-only bound already safe: every c_h is 0, no redo pass needed
  return 0;
}

int hy3d_tc_prepare_kv(hy3d_ctx* ctx) {
  DecoderWeights& w = ctx->w;
  if (!w.t_qp) return 0;
  KVState& kv = ctx->kv;
  const int nkv = kv.Mpad / 128;
  size_t bytes = (size_t)w.H * nkv * TILE_BYTES;
  HY3D_CUDA(ctx, kv.ktile.reserve(bytes));
  HY3D_CUDA(ctx, kv.vtile.reserve(bytes));
  long long total = (long long)w.H * nkv * 128 * 8;
  HY3D_PROF(ctx, FAM_KV);
  k_build_kv<<<(unsigned)ceil_div64(total, 256), 256, 0, ctx->stream>>>(kv.k32.as<float>(), kv.v32.as<float>(), w.H, kv.M, nkv,
                                                                        kv.ktile.as<uint8_t>(), kv.vtile.as<uint8_t>());
  HY3D_LAUNCH_CHECK(ctx);
  return hy3d_tc_head_shift(ctx);
}

namespace {
// fp32 rows [M, K] -> T16 split [hi | lo | hi]
__global__ void k_rows_to_t16_split(const float* __restrict__ src, int M, int K, uint8_t* __restrict__ T) {
  long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;      // one 8-element chunk per thread
  const int c8n = K / 8;
  const long long rows_p = (long long)((M + 127) / 128) * 128;
  if (t >= rows_p * c8n) return;
  const int c8 = (int)(t % c8n); const long long row = t / c8n;
  const int KBn = K / 64;
  float v[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) v[i] = row < M ? src[row * K + c8 * 8 + i] : 0.f;
  uint8_t* t0 = T + ((size_t)(row / 128) * 3 * KBn + (c8 >> 3)) * TILE_BYTES;
  store_t16_split(t0, t0 + (size_t)KBn * TILE_BYTES, t0 + (size_t)2 * KBn * TILE_BYTES, (int)(row % 128), c8 & 7, v);
}

}  // namespace

namespace {
// per-row (mean, M2) of fp32 rows [M, K] in the slot format of GemmTC::st_in: slot s covers columns [64 s, 64 s + 64)
__global__ void k_row_slot_stats(const float* __restrict__ src, int M, int K, float* __restrict__ st) {
  const long long wi = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31, S = K / ST_COLS;
  const long long rows_p = (long long)((M + 127) / 128) * 128;
  if (wi >= rows_p * S) return;
  const long long row = wi / S; const int slot = (int)(wi % S);
  float2 v = make_float2(0.f, 0.f);
  if (row < M) v = reinterpret_cast<const float2*>(src + row * K + slot * ST_COLS)[lane];
  float sum = v.x + v.y;
  for (int o = 16; o; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
  const float mean = sum * (1.f / ST_COLS);
  const float a = v.x - mean, b = v.y - mean;
  float m2 = a * a + b * b;
  for (int o = 16; o; o >>= 1) m2 += __shfl_xor_sync(0xffffffffu, m2, o);
  if (lane == 0) { st[(row * S + slot) * 2] = mean; st[(row * S + slot) * 2 + 1] = m2; }
}
}  // namespace

// K/V of one latent set on the tensor path (reference attention_blocks.py:487-488 latents_proj, :237/:291 ln_2, :257 c_kv,
// :205-211 per-head split + k_norm): fp16 K / V^T tile images for the attention kernel plus fp32 copies for the FlashVDM
// token selection, in two launches (three with latents_proj) instead of the fp32 SIMT GEMMs.
int hy3d_tc_project_kv(hy3d_ctx* ctx, const float* d_latents, int M) {
  DecoderWeights& w = ctx->w;
  if (!w.t_qp || !w.t_ckv3) return hy3d_fail(ctx, HY3D_ERR_UNSUPPORTED, "tcgen05 K/V projection unavailable for this decoder shape");
  KVState& kv = ctx->kv;
  const int W = w.W, H = w.H, LW = w.LW;
  const int Mb = (M + 127) / 128, nkv = Mb, S = W / ST_COLS;   // statistic slots (k_row_slot_stats / latents_proj epilogue)
  const size_t Mp = (size_t)Mb * 128;
  HY3D_CUDA(ctx, kv.k32.reserve((size_t)H * M * 64 * 4));
  HY3D_CUDA(ctx, kv.v32.reserve((size_t)H * M * 64 * 4));
  HY3D_CUDA(ctx, kv.ktile.reserve((size_t)H * nkv * TILE_BYTES));
  HY3D_CUDA(ctx, kv.vtile.reserve((size_t)H * nkv * TILE_BYTES));
  HY3D_CUDA(ctx, ctx->ws[0].reserve(Mp * 3 * (size_t)(LW > W ? LW : W) * 2));    // T16 split of the latents / projected latents
  HY3D_CUDA(ctx, ctx->ws[1].reserve(Mp * 3 * (size_t)W * 2 + Mp * S * 2 * 4));    // second T16 split + row statistics
  uint8_t* tl = ctx->ws[0].as<uint8_t>();
  uint8_t* tp = ctx->ws[1].as<uint8_t>();
  float* st = reinterpret_cast<float*>(tp + Mp * 3 * (size_t)W * 2);
  const uint8_t* a_kv = tl;
  {
    long long total = (long long)Mp * (LW / 8);
    HY3D_PROF(ctx, FAM_KV);
    k_rows_to_t16_split<<<(unsigned)ceil_div64(total, 256), 256, 0, ctx->stream>>>(d_latents, M, LW, tl);
    HY3D_LAUNCH_CHECK(ctx);
  }
  if (w.has_latents_proj) {                                   // L = latents Wlp^T + blp; statistics for the folded ln_2 from the epilogue
    GemmTC g{};
    g.Mb = Mb; g.A = tl; g.B = reinterpret_cast<const uint8_t*>(w.t_lp3); g.KB = 3 * LW / 64; g.N = W; g.Nb = W / BN; g.bias = w.lp_b;
    g.Tcopy = tp; g.split_out = 1; g.st_out = st; g.st_k = 2;
    if (int rc = launch_gemm<EPI_X0>(ctx, g, FAM_KV)) return rc;
    a_kv = tp;
  } else {
    long long warps = (long long)Mp * S;
    HY3D_PROF(ctx, FAM_KV);
    k_row_slot_stats<<<(unsigned)ceil_div64(warps * 32, 256), 256, 0, ctx->stream>>>(d_latents, M, W, st);
    HY3D_LAUNCH_CHECK(ctx);
  }
  GemmTC g{};
  g.Mb = Mb; g.A = a_kv; g.B = reinterpret_cast<const uint8_t*>(w.t_ckv3); g.KB = 3 * W / 64; g.N = 2 * W; g.Nb = 2 * W / BN; g.bias = w.bb_kv;
  g.st_in = st; g.st_slots = S; g.st_np = ST_COLS; g.cs = w.cs_kv; g.ln_eps = 1e-6f;
  g.Kout = kv.ktile.as<uint8_t>(); g.Vout = kv.vtile.as<uint8_t>(); g.nkv = nkv; g.Wq = W; g.part0 = 1;
  g.kn_w = w.kn_w; g.kn_b = w.kn_b; g.qk_norm = w.qk_norm ? 1 : 0; g.qscale = 1.f;
  g.K32 = kv.k32.as<float>(); g.V32T = kv.v32.as<float>(); g.Mtok = M;
  if (int rc = launch_gemm<EPI_QKV>(ctx, g, FAM_KV)) return rc;
  kv.M = M; kv.Mpad = (int)Mp; kv.ready = true;
  return hy3d_tc_head_shift(ctx);
}

static int decode_tc_impl(hy3d_ctx* ctx, const QuerySource& src_in, long long n, float* d_out, int out_mode, const int* d_tile_group) {
  DecoderWeights& w = ctx->w;
  if (!w.t_qp)
    return hy3d_fail(ctx, HY3D_ERR_UNSUPPORTED, "tcgen05 path needs head_dim 64 and widths that are multiples of 256");
  const int W = w.W, H = w.H, R = w.R;
  const int S = ST_PER_TILE * (W / BN);                         // statistic slots per row (one per 64 output columns)
  // points per chunk (a multiple of 256: whole CTA-pair tiles); the activations of one chunk are what the stages hand over
  // through L2 / HBM.  131072 measured 1 % slower, 32768 7 % slower.
  const long long CH = 262144;
  const long long chmax = n < CH ? (n + 127) / 128 * 128 : CH;
  HY3D_CUDA(ctx, ctx->ws[2].reserve((size_t)chmax * W * 4));          // R32 residual stream
  HY3D_CUDA(ctx, ctx->ws[3].reserve((size_t)chmax * W * 2));          // T16 q, then raw x1
  HY3D_CUDA(ctx, ctx->ws[4].reserve((size_t)chmax * W * 2));          // T16 attention output
  HY3D_CUDA(ctx, ctx->ws[5].reserve((size_t)chmax * W * R * 2));      // T16 h
  HY3D_CUDA(ctx, ctx->ws[9].reserve((size_t)chmax * S * 5 * 4));      // row statistics: x1 (2), x2 (3) per slot
  HY3D_CUDA(ctx, ctx->ws[6].reserve((size_t)chmax * 192 * 2));        // T16 Fourier features [hi | lo | hi] (kept for the fused c_proj)
  HY3D_CUDA(ctx, ctx->ln_mr.reserve((size_t)chmax * sizeof(float2)));  // ln_1 statistics of x0 (k_embed_tc)
  float* x = ctx->ws[2].as<float>();
  uint8_t* ta = ctx->ws[3].as<uint8_t>();
  uint8_t* tq = ctx->ws[4].as<uint8_t>();
  uint8_t* th = ctx->ws[5].as<uint8_t>();
  uint8_t* te = ctx->ws[6].as<uint8_t>();
  float* st3 = ctx->ws[9].as<float>();
  float* stp = st3 + (size_t)chmax * S * 2;
  const float pi_mul = w.include_pi ? 3.14159265358979323846f : 1.f;
  for (long long p0 = 0; p0 < n; p0 += CH) {
    const long long P = (n - p0 < CH) ? (n - p0) : CH;
    const int Pb = (int)((P + 127) / 128);
    QuerySource src = src_in;
    if (src.mode == 0) src.xyz += 3 * p0;
    else if (src.mode == 1) src.first += p0;
    else src.index += p0;
    // q = q_norm(c_q(ln_1(query_proj(e)))) * scale * log2e as ONE K = 192 GEMM: c_q . query_proj collapsed into Wc (the
    // LayerNorm between them only scales and shifts rows; its statistics are closed forms in e, computed by the embed
    // kernel).  x0 is never formed, q is fp32-grade (x0 used to be rounded to fp16 on its way into c_q).
    QStats qs{w.qs_wbar, w.qs_hc, w.qs_Gc, w.qs_scal, w.E};
    HY3D_PROF(ctx, FAM_EMBED);
    if (w.F == 8) k_embed_tc<8><<<(Pb < ctx->num_sms * 8 ? Pb : ctx->num_sms * 8), 128, 0, ctx->stream>>>(src, P, w.F, pi_mul, te, qs, 1e-6f, ctx->ln_mr.as<float2>());
    else k_embed_tc<0><<<(Pb < ctx->num_sms * 8 ? Pb : ctx->num_sms * 8), 128, 0, ctx->stream>>>(src, P, w.F, pi_mul, te, qs, 1e-6f, ctx->ln_mr.as<float2>());
    HY3D_LAUNCH_CHECK(ctx);
    GemmTC g{};
    g.Mb = Pb; g.A = te; g.B = reinterpret_cast<const uint8_t*>(w.t_cqx); g.KB = 3; g.N = W; g.Nb = W / BN; g.bias = w.bb_q; g.Tout = ta;
    g.ln_mr = ctx->ln_mr.as<float2>(); g.cs = w.cs_qx; g.ln_eps = 1e-6f;
    g.qn_w = w.qn_w; g.qn_b = w.qn_b; g.qk_norm = w.qk_norm ? 1 : 0; g.qscale = rsqrtf((float)w.D) * LOG2E;
    if (int rc = launch_gemm<EPI_Q>(ctx, g, FAM_GEMM_CQ)) return rc;
    {
      AttnTC a{};
      a.Q = ta; a.O = tq; a.Pb = Pb; a.H = H;
      if (d_tile_group) {
        a.K = ctx->kvsel.ktile.as<uint8_t>(); a.V = ctx->kvsel.vtile.as<uint8_t>(); a.nkv = ctx->kvsel.nkv;
        a.tile_group = d_tile_group + p0 / 128; a.group_ntok = ctx->kvsel.ntok.as<int>(); a.group_base = ctx->kvsel.g0;
      } else {
        a.K = ctx->kv.ktile.as<uint8_t>(); a.V = ctx->kv.vtile.as<uint8_t>(); a.nkv = ctx->kv.Mpad / 128; a.ntok = ctx->kv.M;
      }
      if (int rc = launch_attn(ctx, a, w.attn_fast, FAM_ATTN, ctx->kv.shifted)) return rc;
    }
    // x1 = x0 + c_proj(attn) = [attn | e] [W_o | W_qp]^T + (b_o + b_qp): K-concatenated, no fp32 x0 in memory;
    // fp32 residual + raw fp16 copy + statistics for the folded ln_3
    g = GemmTC{}; g.Mb = Pb;
    g.A = tq; g.KB1 = W / 64; g.A2 = te; g.KB = W / 64 + 3; g.B = reinterpret_cast<const uint8_t*>(w.t_cpx); g.bias = w.b_cpx;
    g.N = W; g.Nb = W / BN; g.Rout = x; g.Tcopy = ta; g.st_out = st3; g.st_k = 2;
    if (int rc = launch_gemm<EPI_RES>(ctx, g, FAM_GEMM_CPROJ)) return rc;
    // h = gelu(c_fc(ln_3 x1))                      (ln_3 folded)
    g = GemmTC{}; g.Mb = Pb;
    g.A = ta; g.B = reinterpret_cast<const uint8_t*>(w.t_fc); g.KB = W / 64; g.N = W * R; g.Nb = W * R / BN; g.bias = w.bb_fc; g.Tout = th;
    g.st_in = st3; g.st_slots = S; g.st_np = ST_COLS; g.cs = w.cs_fc; g.ln_eps = 1e-6f;
    if (int rc = launch_gemm<EPI_GELU>(ctx, g, FAM_GEMM_FC)) return rc;
    // x2 = x1 + c_proj(h): never stored — only its row statistics and its dot with gamma_post * w_out, from which
    // k_head_final forms [ln_post] + output_proj
    g = GemmTC{}; g.Mb = Pb;
    g.A = th; g.B = reinterpret_cast<const uint8_t*>(w.t_mp); g.KB = W * R / 64; g.N = W; g.Nb = W / BN; g.bias = w.mp_b;
    g.Rin = x; g.st_out = stp; g.st_k = 3; g.dotw = w.dotw;
    if (int rc = launch_gemm<EPI_RES>(ctx, g, FAM_GEMM_MLP)) return rc;
    float* outp = d_out + (out_mode == 0 ? p0 : 0);
    HY3D_PROF(ctx, FAM_HEAD);
    k_head_final<<<Pb, 128, 0, ctx->stream>>>(stp, S, ST_COLS, w.ln_post ? 1 : 0, w.c12, src, P, outp, out_mode);
    HY3D_LAUNCH_CHECK(ctx);
  }
  return 0;
}

int hy3d_decode_tc(hy3d_ctx* ctx, const QuerySource& src, long long n, float* d_out, int out_mode) {
  return decode_tc_impl(ctx, src, n, d_out, out_mode, nullptr);
}

int hy3d_decode_tc_groups(hy3d_ctx* ctx, const QuerySource& src, long long n, float* d_out, int out_mode, const int* d_tile_group) {
  if (!ctx->kvsel.ready) return hy3d_fail(ctx, HY3D_ERR_STATE, "no KV selection prepared");
  return decode_tc_impl(ctx, src, n, d_out, out_mode, d_tile_group);
}

// Front of the chain for the sub-sampled queries that drive the FlashVDM KV selection, at ~fp32
// accuracy: embed -> query_proj (split) -> ln_1 (split output) -> c_q (3-term split, K = 3W) -> q_norm.
int hy3d_tc_sample_q(hy3d_ctx* ctx, const QuerySource& src_in, long long n, float* d_q) {
  DecoderWeights& w = ctx->w;
  if (!w.t_qp) return hy3d_fail(ctx, HY3D_ERR_UNSUPPORTED, "tcgen05 path unavailable for this decoder shape");
  const int W = w.W;
  const long long CH = 32768;
  const long long chmax = n < CH ? (n + 127) / 128 * 128 : CH;
  HY3D_CUDA(ctx, ctx->ws[7].reserve((size_t)chmax * W * 4));
  HY3D_CUDA(ctx, ctx->ws[8].reserve((size_t)chmax * W * 2 * 3));
  float* x = ctx->ws[7].as<float>();
  uint8_t* ta = ctx->ws[8].as<uint8_t>();
  const float pi_mul = w.include_pi ? 3.14159265358979323846f : 1.f;
  for (long long p0 = 0; p0 < n; p0 += CH) {
    const long long P = (n - p0 < CH) ? (n - p0) : CH;
    const int Pb = (int)((P + 127) / 128);
    QuerySource src = src_in;
    if (src.mode == 0) src.xyz += 3 * p0;
    else if (src.mode == 1) src.first += p0;
    else src.index += p0;
    HY3D_PROF(ctx, FAM_SELECT);
    k_embed_tc<0><<<(Pb < ctx->num_sms * 8 ? Pb : ctx->num_sms * 8), 128, 0, ctx->stream>>>(src, P, w.F, pi_mul, ta, QStats{}, 0.f, nullptr);
    HY3D_LAUNCH_CHECK(ctx);
    GemmTC g{};
    g.Mb = Pb; g.A = ta; g.B = reinterpret_cast<const uint8_t*>(w.t_qp); g.KB = 3; g.N = W; g.Nb = W / BN; g.bias = w.qp_b; g.Rout = x;
    if (int rc = launch_gemm<EPI_X0>(ctx, g, FAM_SELECT)) return rc;
    HY3D_PROF(ctx, FAM_SELECT);
    k_ln_tc<true><<<Pb, 128, 0, ctx->stream>>>(x, W, w.ln1_w, w.ln1_b, 1e-6f, ta);
    HY3D_LAUNCH_CHECK(ctx);
    g = GemmTC{}; g.Mb = Pb;
    g.A = ta; g.B = reinterpret_cast<const uint8_t*>(w.t_cq3); g.KB = 3 * W / 64; g.N = W; g.Nb = W / BN; g.bias = w.cq_b;
    g.Fout = d_q + (size_t)p0 * W; g.qn_w = w.qn_w; g.qn_b = w.qn_b; g.qk_norm = w.qk_norm ? 1 : 0; g.qscale = 1.f;
    if (int rc = launch_gemm<EPI_QF32>(ctx, g, FAM_SELECT)) return rc;
  }
  return 0;
}

// ------------------------------------------------------------------------------------------
// Latent transformer: post_kl + L pre-LN self-attention blocks (reference model.py:186-189,
// attention_blocks.py:301-432) on the same kernels.  Every GEMM is a 3-term split (fp32-grade);
// the LayerNorms are folded into c_qkv / c_fc; c_qkv's output columns are permuted to [q | k | v].
// ------------------------------------------------------------------------------------------
namespace {

__global__ void k_r32_to_rows(const float* __restrict__ R, long long rows, int W, float* __restrict__ out) {
  long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= rows * (W / 4)) return;
  const long long row = t / (W / 4); const int c4 = (int)(t % (W / 4));
  const float4 v = reinterpret_cast<const float4*>(R)[((row / 128) * (W / 4) + c4) * 128 + (row % 128)];
  reinterpret_cast<float4*>(out)[row * (W / 4) + c4] = v;
}

}  // namespace

extern "C" int hy3d_set_transformer_weights(hy3d_ctx* ctx, const hy3d_transformer_desc* d) {
  if (!ctx || !d || !d->layer) return HY3D_ERR_ARG;
  HY3D_CUDA(ctx, cudaSetDevice(ctx->device));
  TransformerState& t = ctx->tf;
  t.set = false;
  const size_t W = d->width, H = d->heads, L = d->layers, E = d->embed_dim, R = 4;
  if (W % 256 || H == 0 || W / H != 64 || E % 64 || L == 0)
    return hy3d_fail(ctx, HY3D_ERR_UNSUPPORTED, "tcgen05 transformer needs head_dim 64, width %% 256 == 0, embed_dim %% 64 == 0");
  t.L = (int)L; t.W = (int)W; t.H = (int)H; t.E = (int)E; t.qk_norm = d->qk_norm;
  const size_t n_pk = W * 3 * E, n_qkv = 3 * W * 3 * W, n_proj = W * 3 * W, n_fc = R * W * 3 * W, n_p2 = W * 3 * R * W;
  HY3D_CUDA(ctx, t.tc.reserve((n_pk + L * (n_qkv + n_proj + n_fc + n_p2)) * 2));
  const size_t f_layer = 3 * W + 3 * W + W + R * W + R * W + W + 4 * 64;
  HY3D_CUDA(ctx, t.f32.reserve((W + L * f_layer + 64) * sizeof(float)));
  HY3D_CUDA(ctx, ctx->ws[10].reserve(R * W * W * sizeof(float)));
  float* Wf = ctx->ws[10].as<float>();
  __half* hp = t.tc.as<__half>();
  float* fp = t.f32.as<float>();
  auto build = [&](const float* src, size_t N, size_t K3, size_t ldw, __half* dst) -> int {   // mode 2: [hi | hi | lo]
    long long total = (long long)N * (K3 / 8);
    k_build_b16<<<(unsigned)ceil_div64(total, 256), 256, 0, ctx->stream>>>(src, (int)N, (int)K3, (int)ldw, 2, 0, reinterpret_cast<uint8_t*>(dst));
    HY3D_LAUNCH_CHECK(ctx);
    return 0;
  };
  auto copyf = [&](const float* src, size_t n, float* dst) -> int {
    HY3D_CUDA(ctx, cudaMemcpyAsync(dst, src, n * sizeof(float), cudaMemcpyDeviceToDevice, ctx->stream));
    return 0;
  };
  if (!d->post_kl_w || !d->post_kl_b) return hy3d_fail(ctx, HY3D_ERR_ARG, "post_kl missing");
  if (int rc = build(d->post_kl_w, W, 3 * E, E, hp)) return rc;
  t.t_postkl = reinterpret_cast<const uint8_t*>(hp); hp += n_pk;
  if (int rc = copyf(d->post_kl_b, W, fp)) return rc;
  t.b_postkl = fp; fp += W;
  t.t_qkv.assign(L, nullptr); t.t_proj.assign(L, nullptr); t.t_fc.assign(L, nullptr); t.t_proj2.assign(L, nullptr);
  t.cs_qkv.assign(L, nullptr); t.bb_qkv.assign(L, nullptr); t.b_proj.assign(L, nullptr); t.cs_fc.assign(L, nullptr);
  t.bb_fc.assign(L, nullptr); t.b_proj2.assign(L, nullptr); t.qn_w.assign(L, nullptr); t.qn_b.assign(L, nullptr);
  t.kn_w.assign(L, nullptr); t.kn_b.assign(L, nullptr); t.attn_fast.assign(L, 0);
  for (size_t l = 0; l < L; ++l) {
    const hy3d_transformer_layer& y = d->layer[l];
    if (!y.ln1_w || !y.ln1_b || !y.c_qkv_w || !y.c_proj_w || !y.c_proj_b || !y.ln2_w || !y.ln2_b || !y.c_fc_w || !y.c_fc_b ||
        !y.mlp_proj_w || !y.mlp_proj_b)
      return hy3d_fail(ctx, HY3D_ERR_ARG, "transformer layer %d: a required tensor is NULL", (int)l);
    if (d->qk_norm && !(y.q_norm_w && y.q_norm_b && y.k_norm_w && y.k_norm_b))
      return hy3d_fail(ctx, HY3D_ERR_ARG, "transformer layer %d: q/k norm missing", (int)l);
    float* cs_qkv = fp; float* bb_qkv = cs_qkv + 3 * W; float* b_proj = bb_qkv + 3 * W; float* cs_fc = b_proj + W;
    float* bb_fc = cs_fc + R * W; float* b_p2 = bb_fc + R * W; float* nrm = b_p2 + W;
    fp += f_layer;
    // c_qkv: ln_1 folded, rows permuted [head][q|k|v] -> [q | k | v]
    k_fold_ln<<<(unsigned)((3 * W + 7) / 8), 256, 0, ctx->stream>>>(y.c_qkv_w, y.ln1_w, y.ln1_b, y.c_qkv_b, (int)(3 * W), (int)W, Wf, cs_qkv,
                                                                    bb_qkv, (int)H, 1);
    HY3D_LAUNCH_CHECK(ctx);
    if (int rc = build(Wf, 3 * W, 3 * W, W, hp)) return rc;
    t.t_qkv[l] = reinterpret_cast<const uint8_t*>(hp); hp += n_qkv;
    if (int rc = build(y.c_proj_w, W, 3 * W, W, hp)) return rc;
    t.t_proj[l] = reinterpret_cast<const uint8_t*>(hp); hp += n_proj;
    k_fold_ln<<<(unsigned)((R * W + 7) / 8), 256, 0, ctx->stream>>>(y.c_fc_w, y.ln2_w, y.ln2_b, y.c_fc_b, (int)(R * W), (int)W, Wf, cs_fc,
                                                                    bb_fc, 0, 1);
    HY3D_LAUNCH_CHECK(ctx);
    if (int rc = build(Wf, R * W, 3 * W, W, hp)) return rc;
    t.t_fc[l] = reinterpret_cast<const uint8_t*>(hp); hp += n_fc;
    if (int rc = build(y.mlp_proj_w, W, 3 * R * W, R * W, hp)) return rc;
    t.t_proj2[l] = reinterpret_cast<const uint8_t*>(hp); hp += n_p2;
    if (int rc = copyf(y.c_proj_b, W, b_proj)) return rc;
    if (int rc = copyf(y.mlp_proj_b, W, b_p2)) return rc;
    if (d->qk_norm) {
      if (int rc = copyf(y.q_norm_w, 64, nrm)) return rc;
      if (int rc = copyf(y.q_norm_b, 64, nrm + 64)) return rc;
      if (int rc = copyf(y.k_norm_w, 64, nrm + 128)) return rc;
      if (int rc = copyf(y.k_norm_b, 64, nrm + 192)) return rc;
    }
    t.cs_qkv[l] = cs_qkv; t.bb_qkv[l] = bb_qkv; t.b_proj[l] = b_proj; t.cs_fc[l] = cs_fc; t.bb_fc[l] = bb_fc; t.b_proj2[l] = b_p2;
    t.qn_w[l] = nrm; t.qn_b[l] = nrm + 64; t.kn_w[l] = nrm + 128; t.kn_b[l] = nrm + 192;
    if (d->qk_norm) {
      float bound = INFINITY;
      if (int rc = attn_score_bound(ctx, y.q_norm_w, y.q_norm_b, y.k_norm_w, y.k_norm_b, &bound)) return rc;
      t.attn_fast[l] = bound <= ATT_FAST_BOUND ? 1 : 0;       // (weight-only bound: the self-attention launches are 16 x 90 us)
    }
  }
  HY3D_CUDA(ctx, cudaStreamSynchronize(ctx->stream));      // the fold scratch (ws[10]) is reused by other calls
  t.set = true;
  return HY3D_OK;
}

// ---- the forward pass in four steps, so that a latent set can be split by token ranges across GPUs (sequence parallel):
// every GEMM, LayerNorm and residual acts on rows independently; only self-attention needs all tokens' K / V, which the
// ranks exchange as ready-made tile images — one all-gather per layer, done by the host between layer_kv and layer_rest.
// K / V exchange buffer: [parts][2 (K, V^T)][H][Ml / 128][16 KB]; chunk `part` is written by this rank.
static size_t tf_chunk_bytes(const TransformerState& t) { return (size_t)2 * t.H * (t.Ml / 128) * TILE_BYTES; }

extern "C" int hy3d_transformer_begin(hy3d_ctx* ctx, const float* d_z_local, int32_t Ml, int32_t parts, int32_t part) {
  if (!ctx || !d_z_local || Ml <= 0 || parts <= 0 || part < 0 || part >= parts) return HY3D_ERR_ARG;
  TransformerState& t = ctx->tf;
  if (!t.set) return hy3d_fail(ctx, HY3D_ERR_STATE, "transformer weights not set");
  if (Ml % 128) return hy3d_fail(ctx, HY3D_ERR_UNSUPPORTED, "token count (per part) must be a multiple of 128");
  HY3D_CUDA(ctx, cudaSetDevice(ctx->device));
  t.Ml = Ml; t.parts = parts; t.part = part;
  const int W = t.W, R = t.R, E = t.E, Mb = Ml / 128, S = ST_PER_TILE * (W / BN);
  const size_t Mp = (size_t)Ml;
  HY3D_CUDA(ctx, t.x.reserve(Mp * W * 4));
  HY3D_CUDA(ctx, t.ta.reserve(Mp * 3 * W * 2));
  HY3D_CUDA(ctx, t.tq.reserve(Mp * W * 2));
  HY3D_CUDA(ctx, t.to.reserve(Mp * 3 * W * 2));
  HY3D_CUDA(ctx, t.th.reserve(Mp * 3 * R * W * 2));
  HY3D_CUDA(ctx, t.st.reserve(Mp * S * 2 * 2 * 4));
  HY3D_CUDA(ctx, t.tz.reserve(Mp * 3 * E * 2));
  {
    long long total = (long long)Ml * (E / 8);
    HY3D_PROF(ctx, FAM_KV);
    k_rows_to_t16_split<<<(unsigned)ceil_div64(total, 256), 256, 0, ctx->stream>>>(d_z_local, Ml, E, t.tz.as<uint8_t>());
    HY3D_LAUNCH_CHECK(ctx);
  }
  GemmTC g{};
  g.Mb = Mb; g.A = t.tz.as<uint8_t>(); g.B = t.t_postkl; g.KB = 3 * E / 64; g.N = W; g.Nb = W / BN; g.bias = t.b_postkl;
  g.Rout = t.x.as<float>(); g.Tcopy = t.ta.as<uint8_t>(); g.split_out = 1; g.st_out = t.st.as<float>(); g.st_k = 2;
  return launch_gemm<EPI_X0>(ctx, g, FAM_KV);
}

extern "C" int hy3d_transformer_layer_kv(hy3d_ctx* ctx, int32_t l, void* d_kv_all) {
  if (!ctx || !d_kv_all) return HY3D_ERR_ARG;
  TransformerState& t = ctx->tf;
  if (!t.set || t.Ml <= 0 || l < 0 || l >= t.L) return hy3d_fail(ctx, HY3D_ERR_STATE, "hy3d_transformer_begin has not been called / bad layer");
  const int W = t.W, Mb = t.Ml / 128, S = ST_PER_TILE * (W / BN);
  float* stA = t.st.as<float>();
  uint8_t* chunk = static_cast<uint8_t*>(d_kv_all) + (size_t)t.part * tf_chunk_bytes(t);
  GemmTC g{}; g.Mb = Mb;                                       // q, k, v = split(c_qkv(ln_1 x)), q/k norms
  g.A = t.ta.as<uint8_t>(); g.B = t.t_qkv[l]; g.KB = 3 * W / 64; g.N = 3 * W; g.Nb = 3 * W / BN; g.bias = t.bb_qkv[l];
  g.st_in = stA; g.st_slots = S; g.st_np = ST_COLS; g.cs = t.cs_qkv[l]; g.ln_eps = 1e-6f;
  g.Tout = t.tq.as<uint8_t>(); g.Kout = chunk; g.Vout = chunk + (size_t)t.H * Mb * TILE_BYTES; g.nkv = Mb; g.Wq = W;
  g.qn_w = t.qn_w[l]; g.qn_b = t.qn_b[l]; g.kn_w = t.kn_w[l]; g.kn_b = t.kn_b[l]; g.qk_norm = t.qk_norm;
  g.qscale = rsqrtf(64.f) * LOG2E;
  return launch_gemm<EPI_QKV>(ctx, g, FAM_KV);
}

extern "C" int hy3d_transformer_layer_rest(hy3d_ctx* ctx, int32_t l, const void* d_kv_all) {
  if (!ctx || !d_kv_all) return HY3D_ERR_ARG;
  TransformerState& t = ctx->tf;
  if (!t.set || t.Ml <= 0 || l < 0 || l >= t.L) return hy3d_fail(ctx, HY3D_ERR_STATE, "hy3d_transformer_begin has not been called / bad layer");
  const int W = t.W, H = t.H, R = t.R, Mb = t.Ml / 128, S = ST_PER_TILE * (W / BN);
  float* x = t.x.as<float>();
  uint8_t *ta = t.ta.as<uint8_t>(), *to = t.to.as<uint8_t>(), *th = t.th.as<uint8_t>();
  float* stA = t.st.as<float>(); float* stB = stA + (size_t)t.Ml * S * 2;
  {
    AttnTC a{};                                                // local query tiles against the K / V of ALL parts
    a.Q = t.tq.as<uint8_t>(); a.O = to; a.Pb = Mb; a.H = H; a.split_out = 1;
    a.K = static_cast<const uint8_t*>(d_kv_all); a.V = a.K + (size_t)H * Mb * TILE_BYTES;
    a.nkv = Mb * t.parts; a.ntok = t.Ml * t.parts; a.kv_tpr = Mb; a.kv_chunk_stride = (long long)tf_chunk_bytes(t);
    if (int rc = launch_attn(ctx, a, t.attn_fast[l] != 0, FAM_KV)) return rc;
  }
  GemmTC g{}; g.Mb = Mb;                                       // x += c_proj(attn)
  g.A = to; g.B = t.t_proj[l]; g.KB = 3 * W / 64; g.N = W; g.Nb = W / BN; g.bias = t.b_proj[l];
  g.Rin = x; g.Rout = x; g.Tcopy = ta; g.split_out = 1; g.st_out = stB; g.st_k = 2;
  if (int rc = launch_gemm<EPI_RES>(ctx, g, FAM_KV)) return rc;
  g = GemmTC{}; g.Mb = Mb;                                     // h = gelu(c_fc(ln_2 x))
  g.A = ta; g.B = t.t_fc[l]; g.KB = 3 * W / 64; g.N = R * W; g.Nb = R * W / BN; g.bias = t.bb_fc[l];
  g.st_in = stB; g.st_slots = S; g.st_np = ST_COLS; g.cs = t.cs_fc[l]; g.ln_eps = 1e-6f; g.Tout = th; g.split_out = 1;
  if (int rc = launch_gemm<EPI_GELU>(ctx, g, FAM_KV)) return rc;
  g = GemmTC{}; g.Mb = Mb;                                     // x += c_proj(h)
  g.A = th; g.B = t.t_proj2[l]; g.KB = 3 * R * W / 64; g.N = W; g.Nb = W / BN; g.bias = t.b_proj2[l];
  g.Rin = x; g.Rout = x; g.Tcopy = ta; g.split_out = 1; g.st_out = stA; g.st_k = 2;
  return launch_gemm<EPI_RES>(ctx, g, FAM_KV);
}

extern "C" int hy3d_transformer_end(hy3d_ctx* ctx, float* d_out_local) {
  if (!ctx || !d_out_local) return HY3D_ERR_ARG;
  TransformerState& t = ctx->tf;
  if (!t.set || t.Ml <= 0) return hy3d_fail(ctx, HY3D_ERR_STATE, "hy3d_transformer_begin has not been called");
  long long total = (long long)t.Ml * (t.W / 4);
  HY3D_PROF(ctx, FAM_KV);
  k_r32_to_rows<<<(unsigned)ceil_div64(total, 256), 256, 0, ctx->stream>>>(t.x.as<float>(), t.Ml, t.W, d_out_local);
  HY3D_LAUNCH_CHECK(ctx);
  return HY3D_OK;
}

extern "C" int hy3d_transformer_forward(hy3d_ctx* ctx, const float* d_z, int32_t M, float* d_out) {
  if (!ctx || !d_z || !d_out || M <= 0) return HY3D_ERR_ARG;
  TransformerState& t = ctx->tf;
  if (!t.set) return hy3d_fail(ctx, HY3D_ERR_STATE, "transformer weights not set");
  if (int rc = hy3d_transformer_begin(ctx, d_z, M, 1, 0)) return rc;
  HY3D_CUDA(ctx, t.kt.reserve(tf_chunk_bytes(t)));            // one part: the exchange buffer is private
  for (int l = 0; l < t.L; ++l) {
    if (int rc = hy3d_transformer_layer_kv(ctx, l, t.kt.p)) return rc;
    if (int rc = hy3d_transformer_layer_rest(ctx, l, t.kt.p)) return rc;
  }
  return hy3d_transformer_end(ctx, d_out);
}

int hy3d_watchdog_enqueue(hy3d_ctx* ctx) {
  int* rec = reinterpret_cast<int*>(ctx->pinned) + 128;
  HY3D_CUDA(ctx, cudaMemcpyFromSymbolAsync(rec, hy3d_wd, sizeof(int) * 8, 0, cudaMemcpyDeviceToHost, ctx->stream));
  return 0;
}

int hy3d_watchdog_check(hy3d_ctx* ctx) {
  const int* rec = reinterpret_cast<const int*>(ctx->pinned) + 128;
  if (!rec[0]) return 0;
  const int blk = rec[1], thr = rec[2], bar = rec[3], par = rec[4];
  int zero[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  cudaMemcpyToSymbol(hy3d_wd, zero, sizeof(zero));
  return hy3d_fail(ctx, HY3D_ERR_STATE, "tcgen05 kernel barrier timeout (block %d thread %d barrier 0x%x parity %d): the results of the "
                   "decoder launches before this call are invalid", blk, thr, bar, par);
}

extern "C" int hy3d_debug_watchdog(hy3d_ctx* ctx, int32_t h_out[8]) {
  if (!ctx || !h_out) return HY3D_ERR_ARG;
  HY3D_CUDA(ctx, cudaSetDevice(ctx->device));
  HY3D_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  HY3D_CUDA(ctx, cudaMemcpyFromSymbol(h_out, hy3d_wd, sizeof(int) * 8));
  int zero[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  HY3D_CUDA(ctx, cudaMemcpyToSymbol(hy3d_wd, zero, sizeof(zero)));
  return HY3D_OK;
}
