// Shared declarations of libhy3dgeo.so (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_fp16.h>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/hy3dgeo.h"

#define HY3D_SENTINEL (-10000.0f)
#define HY3D_BAND 0.95f

struct DevBuf {                       // grow-only device scratch
  void* p = nullptr;
  size_t cap = 0;
  cudaError_t reserve(size_t bytes) {
    if (bytes <= cap) return cudaSuccess;
    if (p) cudaFree(p);
    p = nullptr; cap = 0;
    cudaError_t e = cudaMalloc(&p, bytes);
    if (e == cudaSuccess) cap = bytes;
    return e;
  }
  void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
  template <class T> T* as() const { return reinterpret_cast<T*>(p); }
};

// Decoder weights kept on the device.  fp32 copies feed the SIMT path and the per-latent K/V
// projection; fp16 UMMA-tiled copies feed the tcgen05 path (built in decoder_tc.cu).
struct DecoderWeights {
  bool set = false;
  int W = 0, H = 0, D = 0, R = 0, LW = 0, F = 0, E = 0;   // width, heads, head dim, mlp ratio, latent width, freqs, embed dim
  bool include_pi = false, ln_post = true, qk_norm = true;
  bool has_latents_proj = false, has_cq_b = false, has_ckv_b = false;
  float freqs[16];
  DevBuf f32;                         // one slab holding all fp32 tensors
  const float *qp_w, *qp_b, *lp_w, *lp_b, *ln1_w, *ln1_b, *ln2_w, *ln2_b, *ln3_w, *ln3_b;
  const float *cq_w, *cq_b, *ckv_w, *ckv_b, *cproj_w, *cproj_b, *qn_w, *qn_b, *kn_w, *kn_b;
  const float *fc_w, *fc_b, *mp_w, *mp_b, *lnp_w, *lnp_b, *out_w, *out_b;
  // tcgen05 operand images (decoder_tc.cu)
  DevBuf tc;
  const __half *t_qp, *t_fc, *t_mp;                       // B tiles
  DevBuf fold;                        // LayerNorm-folded epilogue constants (decoder_tc.cu)
  const float *bb_q, *cs_fc, *bb_fc, *dotw, *c12;
  const __half *t_ckv3, *t_lp3;                           // c_kv (ln_2 folded, [k | v] rows) and latents_proj, 3-term split
  const float *cs_kv, *bb_kv;
  const __half* t_cqx = nullptr;                         // c_q . query_proj collapsed into one K = 192 image (x0 never formed)
  const float *qs_wbar = nullptr, *qs_hc = nullptr, *qs_Gc = nullptr, *qs_scal = nullptr;   // closed-form ln_1 statistics of x0
  const float* cs_qx = nullptr;                          // exact column sums of the gamma-folded c_q weight (collapsed path)
  const __half* t_cpx; const float* b_cpx;               // [c_proj | query_proj] K-concatenated image and b_o + b_qp (fused residual)
  const __half* t_cq3;
  float attn_bound = 0.f;              // upper bound of |q.k| scale log2e from the q/k norm WEIGHTS alone (inf without qk_norm)
  float attn_qbound = 0.f;             // upper bound of ||q|| (after q_norm) from the q-norm weights: sqrt(d) max|w| + ||b||
  bool attn_fast = false;              // q/k norms present: the bounded-score attention kernel applies (attention_tc.cuh), with a
                                       // per-head shift from the measured max ||k|| (KVState::head_shift) when the weight-only bound is above 15.9
};

struct KVState {
  bool ready = false;
  int M = 0;                          // tokens
  int Mpad = 0;                       // tokens padded to 128
  DevBuf k32, v32;                    // fp32 [H, M, D] (after k_norm) — SIMT path + selection
  DevBuf ktile, vtile;                // fp16 UMMA tiles — tcgen05 path
  DevBuf head_shift;                  // float [H] per-head score shift c_h of the bounded-score attention kernel + float [H] measured score bounds
  bool shifted = false;               // some c_h may be > 0: the exact redo pass follows every bounded-score launch
  DevBuf redo;                        // int [1 + items] count + list of (query tile, head pair) items to recompute, then int flags per item
};

// FlashVDM per-group K/V selection (attention_processors.py:35-96): gathered token subsets as UMMA tiles
struct KVSelState {
  bool ready = false;
  int G = 0, nkv = 0;                 // groups, 128-token tiles per (group, head)
  int g0 = 0;                         // layout group of local group 0 (hy3d_flash_select_range)
  DevBuf ktile, vtile;                // [G][H][nkv][16 KB]
  DevBuf ntok;                        // int [G] valid tokens per group
  DevBuf sel;                         // int [G][H][T] (mean) or [G][Mpad] (merge) selected token ids
  DevBuf qs, qbar, mask;              // sampled q fp32 [S, W]; group means [G, W]; merge-mode token bitmasks
};

// Latent transformer (ShapeVAE.forward, reference model.py:186-189) on the tcgen05 path
struct TransformerState {
  bool set = false;
  int L = 0, W = 0, H = 0, E = 0, R = 4, qk_norm = 0;
  int Ml = 0, parts = 1, part = 0;     // forward pass in progress: local tokens, token-range parts (GPUs), this part
  DevBuf tc;                          // fp16 B16 images, 3-term split: post_kl, per layer c_qkv (LN-folded, rows permuted), c_proj, c_fc (LN-folded), mlp.c_proj
  DevBuf f32;                         // per layer: cs_qkv, bb_qkv, b_proj, cs_fc, bb_fc, b_proj2, q/k norm; post_kl bias
  std::vector<const uint8_t*> t_qkv, t_proj, t_fc, t_proj2;
  std::vector<int> attn_fast;         // per layer: bounded attention scores (see DecoderWeights::attn_fast)
  std::vector<const float*> cs_qkv, bb_qkv, b_proj, cs_fc, bb_fc, b_proj2, qn_w, qn_b, kn_w, kn_b;
  const uint8_t* t_postkl = nullptr;
  const float* b_postkl = nullptr;
  DevBuf x, ta, tq, to, th, kt, vt, st, tz;   // activations of one forward pass
};

struct McState {
  bool counted = false;
  const float* grid = nullptr;
  int n0 = 0, n1 = 0, n2 = 0, words = 0;
  int own_planes = 0;                 // slab mode: planes [0, own_planes) are owned, the rest is the next slab's halo
  float level = 0.f;
  int rule = HY3D_MC_FACE_SIGN;       // hy3d_set_mc_face_rule: applies to the next count / emit pair
  int counted_rule = HY3D_MC_FACE_SIGN;   // the rule the last count ran under: an emit under another rule is refused
  long long nV = 0, nF = 0;
  DevBuf bits, rowcnt, rowoff, stats;
};

struct DmcState {                     // dual marching cubes (dmc.cu): hy3d_dmc_count[_slab] -> hy3d_dmc_emit[_slab]
  bool counted = false;
  const float* grid = nullptr;
  int n0 = 0, n1 = 0, n2 = 0, words = 0;   // n0: local planes (owned + read halo)
  int plane0 = 0, N0 = 0, own = 0;    // slab: global index of local plane 0, global plane count, owned planes
  long long nV = 0, nF = 0;           // owned vertices, faces
  long long nVall = 0;                // vertices of every local cube plane (the owned ones and the halo's first)
  DevBuf bits, rowcnt, rowoff, stats, rec;
};

// Per-kernel-family device timing with CUDA events on the launch stream (bench.py roofline).  The numbering is part of the
// C-ABI (hy3d_profile_read): FAM_GEMM_QPROJ and FAM_LN keep their slots although no launch records them any more.
enum { FAM_EMBED = 0, FAM_GEMM_QPROJ, FAM_LN, FAM_GEMM_CQ, FAM_ATTN, FAM_GEMM_CPROJ, FAM_GEMM_FC, FAM_GEMM_MLP, FAM_HEAD,
       FAM_MC_BITS, FAM_MC_ROWCOUNT, FAM_MC_SCAN, FAM_MC_EMIT, FAM_OCTREE, FAM_KV, FAM_SELECT, FAM_COUNT };
struct ProfRec { int fam; cudaEvent_t e0, e1; };
struct Prof {
  int on = 0, cur = -1;
  std::vector<ProfRec> recs;
  std::vector<cudaEvent_t> pool;
  double ms[FAM_COUNT] = {};
  long long cnt[FAM_COUNT] = {};
};

struct hy3d_ctx {
  int device = 0;
  cudaStream_t stream = nullptr;
  int precision = HY3D_PRECISION_FP16_TC;
  int num_sms = 148;
  long long launches = 0;
  std::string err;
  DecoderWeights w;
  KVState kv;
  KVSelState kvsel;
  TransformerState tf;
  McState mc;
  DmcState dmc;
  DevBuf ws[12];                      // decoder workspaces
  DevBuf scratch, scratch2;           // octree / misc
  DevBuf ln_mr;                       // per-row (mean, rstd) of the LayerNorm folded into the running GEMM
  void* pinned = nullptr;             // small pinned host buffer for read-backs (4 KB; ints 128..135 = watchdog record)
  Prof prof;
  // per-context launch state of the tcgen05 path (was function-local statics: one context per thread and device)
  void* tmap_encode = nullptr;        // cuTensorMapEncodeTiled entry point
  int gemm_max_clusters[8] = {0, 0, 0, 0, 0, 0, 0, 0};   // co-resident CTA pairs per GEMM epilogue variant
  std::vector<float> axis_host;       // last per-axis coordinate tables uploaded to ws[11] (skips the upload when unchanged)
  int force_online_softmax = 0;       // hy3d_debug_force_online_softmax: tests run the online-softmax kernel as a reference
};

int hy3d_fail(hy3d_ctx* ctx, int code, const char* fmt, ...);
// tcgen05 watchdog (tc_ptx.cuh): enqueue the read-back of the record before a stream synchronisation that happens anyway,
// check it after — a barrier timeout inside a tensor kernel turns into an error of the next synchronising call.
int hy3d_watchdog_enqueue(hy3d_ctx* ctx);
int hy3d_watchdog_check(hy3d_ctx* ctx);
// per-axis coordinate tables (n0 + n1 + n2 floats) resident in ws[11]; uploaded only when they changed
int hy3d_upload_axes(hy3d_ctx* ctx, const float* h0, const float* h1, const float* h2, int n0, int n1, int n2);

#define HY3D_CUDA(ctx, expr)                                                                   \
  do {                                                                                         \
    cudaError_t _e = (expr);                                                                   \
    if (_e != cudaSuccess)                                                                     \
      return hy3d_fail(ctx, HY3D_ERR_CUDA, "%s:%d %s -> %s", __FILE__, __LINE__, #expr,        \
                       cudaGetErrorString(_e));                                                \
  } while (0)

static inline void hy3d_prof_begin(hy3d_ctx* ctx, int fam) {
  Prof& p = ctx->prof;
  if (!p.on) return;
  ProfRec r; r.fam = fam;
  for (cudaEvent_t* e : {&r.e0, &r.e1}) {
    if (!p.pool.empty()) { *e = p.pool.back(); p.pool.pop_back(); }
    else cudaEventCreate(e);
  }
  cudaEventRecord(r.e0, ctx->stream);
  p.recs.push_back(r);
  p.cur = (int)p.recs.size() - 1;
}
static inline void hy3d_prof_end(hy3d_ctx* ctx) {
  Prof& p = ctx->prof;
  if (!p.on || p.cur < 0) return;
  cudaEventRecord(p.recs[p.cur].e1, ctx->stream);
  p.cur = -1;
}
#define HY3D_PROF(ctx, fam) hy3d_prof_begin(ctx, fam)

#define HY3D_LAUNCH_CHECK(ctx)                                                                 \
  do {                                                                                         \
    (ctx)->launches++;                                                                         \
    hy3d_prof_end(ctx);                                                                        \
    HY3D_CUDA(ctx, cudaGetLastError());                                                        \
  } while (0)

static inline int64_t ceil_div64(int64_t a, int64_t b) { return (a + b - 1) / b; }

// ---- decoder entry points implemented per precision --------------------------------------
struct QuerySource {
  int mode;                 // 0 explicit xyz, 1 dense grid range, 2 index list (idx*cell+bmin), 3 index list (axis tables)
  const float* xyz;         // mode 0
  const float* axis;        // mode 1: device table [n0 + n1 + n2]
  const int32_t* index;     // mode 2
  int n0, n1, n2;
  long long first;          // mode 1
  float cell[3], bmin[3];   // mode 2
};
// out_mode 0: out[q] = logit ; 1: out[index[q]] = logit (skip index < 0)
int hy3d_decode_simt(hy3d_ctx* ctx, const QuerySource& src, long long n, float* d_out, int out_mode);
int hy3d_decode_tc(hy3d_ctx* ctx, const QuerySource& src, long long n, float* d_out, int out_mode);
int hy3d_tc_prepare_weights(hy3d_ctx* ctx);
// decode with per-q-tile KV groups (tile_group: device int per 128-query tile of the whole list) from ctx->kvsel
int hy3d_decode_tc_groups(hy3d_ctx* ctx, const QuerySource& src, long long n, float* d_out, int out_mode, const int* d_tile_group);
// q after q_norm (unscaled), ~fp32 accuracy via 3-term split fp16 tensor GEMMs: d_q row-major [ceil128(n), W]
int hy3d_tc_sample_q(hy3d_ctx* ctx, const QuerySource& src, long long n, float* d_q);
int hy3d_tc_prepare_kv(hy3d_ctx* ctx);
int hy3d_tc_head_shift(hy3d_ctx* ctx);
int hy3d_tc_project_kv(hy3d_ctx* ctx, const float* d_latents, int M);   // tensor-path K/V projection (replaces simt prepare + tc prepare)
int hy3d_simt_prepare_kv(hy3d_ctx* ctx, const float* d_latents, int M);

__device__ __forceinline__ void hy3d_query_point(const QuerySource& s, long long q, float& x, float& y, float& z,
                                                 long long& out_idx) {
  if (s.mode == 0) {
    x = s.xyz[3 * q]; y = s.xyz[3 * q + 1]; z = s.xyz[3 * q + 2]; out_idx = q;
  } else if (s.mode == 1) {
    long long lin = s.first + q;
    int k = (int)(lin % s.n2); long long t = lin / s.n2;
    int j = (int)(t % s.n1); int i = (int)(t / s.n1);
    x = s.axis[i]; y = s.axis[s.n0 + j]; z = s.axis[s.n0 + s.n1 + k]; out_idx = q;
  } else {
    int lin = s.index[q];
    out_idx = lin;
    if (lin < 0) { x = y = z = 0.f; return; }
    int k = lin % s.n2; int t = lin / s.n2;
    int j = t % s.n1; int i = t / s.n1;
    if (s.mode == 3) { x = s.axis[i]; y = s.axis[s.n0 + j]; z = s.axis[s.n0 + s.n1 + k]; return; }
    // volume_decoders.py:394-396: float32(idx) * float32(cell) + float32(bbox_min), no FMA contraction
    x = __fadd_rn(__fmul_rn((float)i, s.cell[0]), s.bmin[0]);
    y = __fadd_rn(__fmul_rn((float)j, s.cell[1]), s.bmin[1]);
    z = __fadd_rn(__fmul_rn((float)k, s.cell[2]), s.bmin[2]);
  }
}
