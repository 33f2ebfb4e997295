// C-ABI glue of libhy3dgeo.so: context, weights, decoder entry points (include/hy3dgeo.h).
#include <cstdarg>

#include "common.cuh"

int hy3d_fail(hy3d_ctx* ctx, int code, const char* fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  if (ctx) ctx->err = buf;
  return code;
}

extern "C" {

int hy3d_profile(hy3d_ctx* ctx, int enable) {
  if (!ctx) return HY3D_ERR_ARG;
  ctx->prof.on = enable ? 1 : 0;
  return HY3D_OK;
}

int hy3d_profile_read(hy3d_ctx* ctx, double h_ms[16], int64_t h_count[16]) {
  if (!ctx || !h_ms || !h_count) return HY3D_ERR_ARG;
  HY3D_CUDA(ctx, cudaSetDevice(ctx->device));
  HY3D_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  Prof& p = ctx->prof;
  for (auto& r : p.recs) {
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, r.e0, r.e1) == cudaSuccess) { p.ms[r.fam] += ms; p.cnt[r.fam]++; }
    p.pool.push_back(r.e0); p.pool.push_back(r.e1);
  }
  p.recs.clear(); p.cur = -1;
  for (int f = 0; f < 16; ++f) { h_ms[f] = p.ms[f]; h_count[f] = p.cnt[f]; p.ms[f] = 0; p.cnt[f] = 0; }
  return HY3D_OK;
}

int hy3d_debug_force_online_softmax(hy3d_ctx* ctx, int enable) {
  if (!ctx) return HY3D_ERR_ARG;
  ctx->force_online_softmax = enable ? 1 : 0;
  return HY3D_OK;
}

}  // extern "C"

// The tables are a few KB and change only with (bounds, resolution): they are kept in ws[11] and re-uploaded only when
// their contents differ from the last upload.  Then the stream is drained first (kernels of earlier calls may still read
// the old tables) and the copy is synchronous (pageable source) — the common repeated call costs no synchronisation.
int hy3d_upload_axes(hy3d_ctx* ctx, const float* h0, const float* h1, const float* h2, int n0, int n1, int n2) {
  const size_t na = (size_t)n0 + n1 + n2;
  std::vector<float>& tab = ctx->axis_host;
  const bool same = tab.size() == na + 3 && tab[0] == (float)n0 && tab[1] == (float)n1 && tab[2] == (float)n2 &&
                    !memcmp(tab.data() + 3, h0, n0 * sizeof(float)) && !memcmp(tab.data() + 3 + n0, h1, n1 * sizeof(float)) &&
                    !memcmp(tab.data() + 3 + n0 + n1, h2, n2 * sizeof(float)) && ctx->ws[11].p;
  if (same) return 0;
  HY3D_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  HY3D_CUDA(ctx, ctx->ws[11].reserve(na * sizeof(float)));
  tab.resize(na + 3);
  tab[0] = (float)n0; tab[1] = (float)n1; tab[2] = (float)n2;
  memcpy(tab.data() + 3, h0, n0 * sizeof(float));
  memcpy(tab.data() + 3 + n0, h1, n1 * sizeof(float));
  memcpy(tab.data() + 3 + n0 + n1, h2, n2 * sizeof(float));
  HY3D_CUDA(ctx, cudaMemcpyAsync(ctx->ws[11].p, tab.data() + 3, na * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
  HY3D_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return 0;
}

extern "C" {

int hy3d_create(int device, void* cuda_stream, hy3d_ctx** out) {
  if (!out) return HY3D_ERR_ARG;
  *out = nullptr;
  int count = 0;
  if (cudaGetDeviceCount(&count) != cudaSuccess || device < 0 || device >= count) return HY3D_ERR_CUDA;
  if (cudaSetDevice(device) != cudaSuccess) return HY3D_ERR_CUDA;
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return HY3D_ERR_CUDA;
  if (prop.major != 10) return HY3D_ERR_UNSUPPORTED;        // sm_100a only: no other code path exists
  hy3d_ctx* ctx = new hy3d_ctx();
  ctx->device = device;
  ctx->stream = (cudaStream_t)cuda_stream;
  ctx->num_sms = prop.multiProcessorCount;
  if (cudaMallocHost(&ctx->pinned, 4096) != cudaSuccess) { delete ctx; return HY3D_ERR_CUDA; }
  *out = ctx;
  return HY3D_OK;
}

void hy3d_destroy(hy3d_ctx* ctx) {
  if (!ctx) return;
  cudaSetDevice(ctx->device);
  cudaStreamSynchronize(ctx->stream);
  ctx->w.f32.release(); ctx->w.tc.release();
  ctx->kv.k32.release(); ctx->kv.v32.release(); ctx->kv.ktile.release(); ctx->kv.vtile.release();
  ctx->kv.head_shift.release(); ctx->kv.redo.release();
  ctx->mc.bits.release(); ctx->mc.rowcnt.release(); ctx->mc.rowoff.release(); ctx->mc.stats.release();
  { DmcState& d = ctx->dmc; for (DevBuf* b : {&d.bits, &d.rowcnt, &d.rowoff, &d.stats, &d.rec}) b->release(); }
  for (auto& b : ctx->ws) b.release();
  { TransformerState& t = ctx->tf; for (DevBuf* b : {&t.tc, &t.f32, &t.x, &t.ta, &t.tq, &t.to, &t.th, &t.kt, &t.vt, &t.st, &t.tz}) b->release(); }
  ctx->w.fold.release();
  { KVSelState& k = ctx->kvsel; k.ktile.release(); k.vtile.release(); k.ntok.release(); k.sel.release(); k.qs.release(); k.qbar.release(); k.mask.release(); }
  ctx->scratch.release(); ctx->scratch2.release(); ctx->ln_mr.release();
  for (auto& r : ctx->prof.recs) { cudaEventDestroy(r.e0); cudaEventDestroy(r.e1); }
  for (auto e : ctx->prof.pool) cudaEventDestroy(e);
  if (ctx->pinned) cudaFreeHost(ctx->pinned);
  delete ctx;
}

int hy3d_set_stream(hy3d_ctx* ctx, void* s) {
  if (!ctx) return HY3D_ERR_ARG;
  ctx->stream = (cudaStream_t)s;
  return HY3D_OK;
}

const char* hy3d_last_error(const hy3d_ctx* ctx) { return ctx ? ctx->err.c_str() : "null context"; }

int hy3d_set_precision(hy3d_ctx* ctx, int precision) {
  if (!ctx) return HY3D_ERR_ARG;
  if (precision != HY3D_PRECISION_FP32_SIMT && precision != HY3D_PRECISION_FP16_TC)
    return hy3d_fail(ctx, HY3D_ERR_ARG, "unknown precision %d", precision);
  ctx->precision = precision;
  return HY3D_OK;
}

int hy3d_set_mc_face_rule(hy3d_ctx* ctx, int rule) {
  if (!ctx) return HY3D_ERR_ARG;
  if (rule != HY3D_MC_FACE_SIGN && rule != HY3D_MC_FACE_ASYMPTOTIC) return hy3d_fail(ctx, HY3D_ERR_ARG, "unknown face rule %d", rule);
  ctx->mc.rule = rule;
  return HY3D_OK;
}

int64_t hy3d_launch_count(const hy3d_ctx* ctx) { return ctx ? ctx->launches : 0; }

int hy3d_attention_info(hy3d_ctx* ctx, float* h_score_bound, int32_t* h_bounded_kernel, float* h_measured_bound) {
  if (!ctx || !h_score_bound || !h_bounded_kernel) return HY3D_ERR_ARG;
  *h_score_bound = ctx->w.attn_bound;
  const bool fast = ctx->w.attn_fast && !ctx->force_online_softmax;
  *h_bounded_kernel = !fast ? 0 : (ctx->kv.shifted ? 2 : 1);
  if (h_measured_bound) {
    *h_measured_bound = ctx->w.attn_bound;
    if (ctx->w.attn_fast && ctx->kv.ready && ctx->kv.head_shift.p) {        // largest per-head bound of the current latent set
      const int H = ctx->w.H;
      std::vector<float> b(2 * (size_t)H);
      HY3D_CUDA(ctx, cudaSetDevice(ctx->device));
      HY3D_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
      HY3D_CUDA(ctx, cudaMemcpy(b.data(), ctx->kv.head_shift.p, b.size() * sizeof(float), cudaMemcpyDeviceToHost));
      float mx = 0.f;
      for (int h = 0; h < H; ++h) mx = b[H + h] > mx ? b[H + h] : mx;
      *h_measured_bound = mx;
    }
  }
  return HY3D_OK;
}

int hy3d_debug_attn_redo(hy3d_ctx* ctx, int32_t* h_items) {
  if (!ctx || !h_items) return HY3D_ERR_ARG;
  *h_items = 0;
  if (!ctx->kv.redo.p) return HY3D_OK;
  HY3D_CUDA(ctx, cudaSetDevice(ctx->device));
  HY3D_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  HY3D_CUDA(ctx, cudaMemcpy(h_items, ctx->kv.redo.p, sizeof(int32_t), cudaMemcpyDeviceToHost));
  return HY3D_OK;
}

int hy3d_set_decoder_weights(hy3d_ctx* ctx, const hy3d_decoder_desc* d) {
  if (!ctx || !d) return HY3D_ERR_ARG;
  HY3D_CUDA(ctx, cudaSetDevice(ctx->device));
  DecoderWeights& w = ctx->w;
  w.set = false;
  ctx->kv.ready = false;
  if (d->width <= 0 || d->heads <= 0 || d->width % d->heads) return hy3d_fail(ctx, HY3D_ERR_ARG, "bad width/heads");
  if (d->num_freqs < 1 || d->num_freqs > 10) return hy3d_fail(ctx, HY3D_ERR_ARG, "num_freqs must be in [1,10]");
  w.W = d->width; w.H = d->heads; w.D = d->width / d->heads; w.R = d->mlp_ratio; w.LW = d->latent_width;
  w.F = d->num_freqs; w.E = 3 * (2 * w.F + 1);
  w.include_pi = d->include_pi != 0; w.ln_post = d->ln_post != 0; w.qk_norm = d->qk_norm != 0;
  w.has_latents_proj = d->latents_proj_w != nullptr;
  if (!w.has_latents_proj && w.LW != w.W) return hy3d_fail(ctx, HY3D_ERR_ARG, "latent_width != width needs latents_proj");
  if (w.ln_post && !(d->ln_post_w && d->ln_post_b)) return hy3d_fail(ctx, HY3D_ERR_ARG, "ln_post weights missing");
  if (w.qk_norm && !(d->q_norm_w && d->q_norm_b && d->k_norm_w && d->k_norm_b))
    return hy3d_fail(ctx, HY3D_ERR_ARG, "q/k norm weights missing");
  for (int f = 0; f < w.F; ++f) w.freqs[f] = (float)(1u << f) * (w.include_pi ? 3.14159265358979323846f : 1.f);

  const long long W = w.W, R = w.R, D = w.D, LW = w.LW, E = w.E;
  struct Item { const float* src; long long n; const float** dst; };
  Item items[] = {
      {d->query_proj_w, W * E, &w.qp_w},     {d->query_proj_b, W, &w.qp_b},
      {d->latents_proj_w, W * LW, &w.lp_w},  {d->latents_proj_b, W, &w.lp_b},
      {d->ln1_w, W, &w.ln1_w}, {d->ln1_b, W, &w.ln1_b}, {d->ln2_w, W, &w.ln2_w}, {d->ln2_b, W, &w.ln2_b},
      {d->ln3_w, W, &w.ln3_w}, {d->ln3_b, W, &w.ln3_b},
      {d->c_q_w, W * W, &w.cq_w},            {d->c_q_b, W, &w.cq_b},
      {d->c_kv_w, 2 * W * W, &w.ckv_w},      {d->c_kv_b, 2 * W, &w.ckv_b},
      {d->c_proj_w, W * W, &w.cproj_w},      {d->c_proj_b, W, &w.cproj_b},
      {d->q_norm_w, D, &w.qn_w}, {d->q_norm_b, D, &w.qn_b}, {d->k_norm_w, D, &w.kn_w}, {d->k_norm_b, D, &w.kn_b},
      {d->c_fc_w, R * W * W, &w.fc_w},       {d->c_fc_b, R * W, &w.fc_b},
      {d->mlp_proj_w, R * W * W, &w.mp_w},   {d->mlp_proj_b, W, &w.mp_b},
      {d->ln_post_w, W, &w.lnp_w},           {d->ln_post_b, W, &w.lnp_b},
      {d->out_w, W, &w.out_w},               {d->out_b, 1, &w.out_b},
  };
  const float* required[] = {d->query_proj_w, d->query_proj_b, d->ln1_w, d->ln1_b, d->ln2_w, d->ln2_b, d->ln3_w, d->ln3_b,
                             d->c_q_w, d->c_kv_w, d->c_proj_w, d->c_proj_b, d->c_fc_w, d->c_fc_b, d->mlp_proj_w,
                             d->mlp_proj_b, d->out_w, d->out_b};
  for (const float* p : required)
    if (!p) return hy3d_fail(ctx, HY3D_ERR_ARG, "a required decoder tensor is NULL");
  size_t total = 0;
  for (auto& it : items) total += it.src ? (size_t)((it.n + 63) / 64 * 64) : 0;
  HY3D_CUDA(ctx, w.f32.reserve(total * sizeof(float)));
  float* base = w.f32.as<float>();
  size_t off = 0;
  for (auto& it : items) {
    if (!it.src) { *it.dst = nullptr; continue; }
    HY3D_CUDA(ctx, cudaMemcpyAsync(base + off, it.src, (size_t)it.n * sizeof(float), cudaMemcpyDeviceToDevice, ctx->stream));
    *it.dst = base + off;
    off += (size_t)((it.n + 63) / 64 * 64);
  }
  w.has_cq_b = d->c_q_b != nullptr;
  w.has_ckv_b = d->c_kv_b != nullptr;
  w.set = true;
  int rc = hy3d_tc_prepare_weights(ctx);
  if (rc) { w.set = false; return rc; }
  return HY3D_OK;
}

int hy3d_prepare_kv(hy3d_ctx* ctx, const float* d_latents, int32_t M) {
  if (!ctx || !d_latents || M <= 0) return HY3D_ERR_ARG;
  if (!ctx->w.set) return hy3d_fail(ctx, HY3D_ERR_STATE, "decoder weights not set");
  HY3D_CUDA(ctx, cudaSetDevice(ctx->device));
  // tensor path: K/V projected by the split-precision tcgen05 GEMMs; HY3D_PRECISION_FP32_SIMT (the on-device
  // fp32 statement used as a cross-check) and shapes the tensor path does not tile keep the CUDA-core projection
  if (ctx->precision != HY3D_PRECISION_FP32_SIMT && ctx->w.t_qp && ctx->w.t_ckv3)
    return hy3d_tc_project_kv(ctx, d_latents, M);
  if (int rc = hy3d_simt_prepare_kv(ctx, d_latents, M)) return rc;
  return hy3d_tc_prepare_kv(ctx);
}

static int decode(hy3d_ctx* ctx, const QuerySource& src, long long n, float* d_out, int out_mode) {
  if (!ctx->w.set) return hy3d_fail(ctx, HY3D_ERR_STATE, "decoder weights not set");
  if (!ctx->kv.ready) return hy3d_fail(ctx, HY3D_ERR_STATE, "hy3d_prepare_kv has not been called");
  if (n == 0) return HY3D_OK;
  HY3D_CUDA(ctx, cudaSetDevice(ctx->device));
  if (ctx->precision == HY3D_PRECISION_FP32_SIMT) return hy3d_decode_simt(ctx, src, n, d_out, out_mode);
  return hy3d_decode_tc(ctx, src, n, d_out, out_mode);
}

int hy3d_decode_points(hy3d_ctx* ctx, const float* d_xyz, int64_t n, float* d_out) {
  if (!ctx || n < 0 || (n > 0 && (!d_xyz || !d_out))) return HY3D_ERR_ARG;
  QuerySource s{};
  s.mode = 0; s.xyz = d_xyz;
  return decode(ctx, s, n, d_out, 0);
}

int hy3d_decode_dense(hy3d_ctx* ctx, const float* h0, const float* h1, const float* h2, int32_t n0, int32_t n1, int32_t n2,
                      int64_t first, int64_t count, float* d_out) {
  if (!ctx || !h0 || !h1 || !h2 || n0 <= 0 || n1 <= 0 || n2 <= 0 || first < 0 || count < 0) return HY3D_ERR_ARG;
  if (first + count > (int64_t)n0 * n1 * n2) return hy3d_fail(ctx, HY3D_ERR_ARG, "range exceeds grid");
  if (count == 0) return HY3D_OK;
  if (!d_out) return HY3D_ERR_ARG;
  HY3D_CUDA(ctx, cudaSetDevice(ctx->device));
  if (int rc = hy3d_upload_axes(ctx, h0, h1, h2, n0, n1, n2)) return rc;
  QuerySource s{};
  s.mode = 1; s.axis = ctx->ws[11].as<float>(); s.n0 = n0; s.n1 = n1; s.n2 = n2; s.first = first;
  return decode(ctx, s, count, d_out, 0);
}

int hy3d_decode_list(hy3d_ctx* ctx, const int32_t* d_index, int64_t n, int32_t n0, int32_t n1, int32_t n2,
                     const float h_cell[3], const float h_bmin[3], float* d_grid) {
  if (!ctx || n < 0 || !h_cell || !h_bmin) return HY3D_ERR_ARG;
  if (n == 0) return HY3D_OK;
  if (!d_index || !d_grid) return HY3D_ERR_ARG;
  if ((int64_t)n0 * n1 * n2 > 2147483647LL) return hy3d_fail(ctx, HY3D_ERR_UNSUPPORTED, "grid too large for int32 indices");
  QuerySource s{};
  s.mode = 2; s.index = d_index; s.n0 = n0; s.n1 = n1; s.n2 = n2;
  for (int a = 0; a < 3; ++a) { s.cell[a] = h_cell[a]; s.bmin[a] = h_bmin[a]; }
  return decode(ctx, s, n, d_grid, 1);
}

int hy3d_decode_list_values(hy3d_ctx* ctx, const int32_t* d_index, int64_t n, int32_t n0, int32_t n1, int32_t n2,
                            const float h_cell[3], const float h_bmin[3], float* d_values) {
  if (!ctx || n < 0 || !h_cell || !h_bmin) return HY3D_ERR_ARG;
  if (n == 0) return HY3D_OK;
  if (!d_index || !d_values) return HY3D_ERR_ARG;
  QuerySource s{};
  s.mode = 2; s.index = d_index; s.n0 = n0; s.n1 = n1; s.n2 = n2;
  for (int a = 0; a < 3; ++a) { s.cell[a] = h_cell[a]; s.bmin[a] = h_bmin[a]; }
  return decode(ctx, s, n, d_values, 0);
}

}  // extern "C"
