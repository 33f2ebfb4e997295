/* hy3dgeo.h — C-ABI of libhy3dgeo.so: B200-native (sm_100a) geometry decoding for
 * Hunyuan3D-2 (latents -> occupancy grid -> mesh).
 *
 * The reference has no FFI for this path: it is Python calling torch and skimage.
 * Each entry point below names the reference Python interface it replaces
 * (paths relative to /root/reference/hy3dgen/shapegen/models/autoencoders/).
 * The host-side mirror of those interfaces (same class names, kwargs and error
 * behaviour) lives in hunyuan3d-2_b200/{volume_decoders,surface_extractors}.py
 * and binds this header through ctypes (see INTEGRATION.md).
 *
 * Conventions
 *   - plain pointers and sizes only; every `const float* d_*` / `float* d_*` is a
 *     DEVICE pointer on the context's device, `h_*` is a HOST pointer;
 *   - all work is enqueued on the context's stream (hy3d_set_stream); the only
 *     host synchronisations are the explicit size read-backs documented below;
 *   - return value 0 = success, negative = error (hy3d_last_error gives text);
 *     nothing throws across the ABI;
 *   - a context is NOT thread-safe: one context per (host thread, device);
 *   - there is no CPU fallback anywhere behind this ABI.
 */
#ifndef HY3DGEO_H
#define HY3DGEO_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define HY3D_OK 0
#define HY3D_ERR_CUDA (-1)
#define HY3D_ERR_ARG (-2)
#define HY3D_ERR_STATE (-3)
#define HY3D_ERR_UNSUPPORTED (-4)

typedef struct hy3d_ctx hy3d_ctx;

/* Arithmetic of the decoder's dense contractions. */
#define HY3D_PRECISION_FP32_SIMT 0 /* fp32 CUDA-core kernels: exact-order reference on the device      */
#define HY3D_PRECISION_FP16_TC 1   /* fp16 operands, fp32 accumulate on tcgen05/TMEM (the product path) */

/* Weights of CrossAttentionDecoder (attention_blocks.py:435-476), fp32 DEVICE pointers in
 * PyTorch nn.Linear layout [out_features, in_features] row-major, names as in its
 * state_dict (SURVEY App. A.3).  Optional tensors are NULL when absent. */
typedef struct hy3d_decoder_desc {
  int32_t width;        /* decoder width Wd = query_proj.weight.shape[0]                   */
  int32_t heads;        /* cross_attn_decoder.attn.heads                                  */
  int32_t mlp_ratio;    /* c_fc.weight.shape[0] / Wd                                      */
  int32_t latent_width; /* width of the incoming latents (= Wd * downsample_ratio)        */
  int32_t num_freqs;    /* FourierEmbedder.num_freqs (attention_blocks.py:72-98)          */
  int32_t include_pi;   /* frequencies *= pi                                              */
  int32_t ln_post;      /* enable_ln_post (attention_blocks.py:471-473)                   */
  int32_t qk_norm;      /* q_norm / k_norm present (attention_blocks.py:197-198)          */
  const float* query_proj_w;   const float* query_proj_b;     /* [Wd, 3*(2F+1)], [Wd]    */
  const float* latents_proj_w; const float* latents_proj_b;   /* [Wd, latent_width] / NULL */
  const float* ln1_w; const float* ln1_b;                     /* [Wd]                     */
  const float* ln2_w; const float* ln2_b;                     /* [Wd]                     */
  const float* ln3_w; const float* ln3_b;                     /* [Wd]                     */
  const float* c_q_w;    const float* c_q_b;                  /* [Wd, Wd], bias or NULL   */
  const float* c_kv_w;   const float* c_kv_b;                 /* [2Wd, Wd], bias or NULL  */
  const float* c_proj_w; const float* c_proj_b;               /* [Wd, Wd], [Wd]           */
  const float* q_norm_w; const float* q_norm_b;               /* [Wd/heads] or NULL       */
  const float* k_norm_w; const float* k_norm_b;               /* [Wd/heads] or NULL       */
  const float* c_fc_w;     const float* c_fc_b;               /* [r*Wd, Wd], [r*Wd]       */
  const float* mlp_proj_w; const float* mlp_proj_b;           /* [Wd, r*Wd], [Wd]         */
  const float* ln_post_w;  const float* ln_post_b;            /* [Wd] or NULL             */
  const float* out_w;      const float* out_b;                /* [1, Wd], [1]             */
} hy3d_decoder_desc;

/* ---- context -------------------------------------------------------------------------- */
int hy3d_create(int device, void* cuda_stream, hy3d_ctx** out);
void hy3d_destroy(hy3d_ctx* ctx);
int hy3d_set_stream(hy3d_ctx* ctx, void* cuda_stream);
const char* hy3d_last_error(const hy3d_ctx* ctx);
/* HY3D_PRECISION_*; default HY3D_PRECISION_FP16_TC. */
int hy3d_set_precision(hy3d_ctx* ctx, int precision);
/* Count of kernels this library has launched on ctx since creation (bench `gpu_launches`). */
int64_t hy3d_launch_count(const hy3d_ctx* ctx);

/* Which attention kernel runs for the loaded decoder weights and the K/V prepared last (bench / diagnostics; synchronises the
 * stream when h_measured_bound is given).  *h_score_bound = upper bound of |q.k| * scale * log2(e) from the q/k-norm WEIGHTS
 * alone (+inf without q/k norm); *h_measured_bound = the same with the measured max ||k|| of the current latent set per head
 * (largest over heads); *h_bounded_kernel = 0 online-softmax kernel, 1 bounded-score kernel, 2 bounded-score kernel with
 * per-head score shifts and the exact redo pass (weight-only bound above 15.9; csrc/attention_tc.cuh). */
int hy3d_attention_info(hy3d_ctx* ctx, float* h_score_bound, int32_t* h_bounded_kernel, float* h_measured_bound);

/* ---- latent transformer: replaces ShapeVAE.forward = post_kl + Transformer (model.py:186-189,
 * attention_blocks.py:301-432).  fp32 DEVICE pointers, nn.Linear layout, state_dict names
 * transformer.resblocks.{l}.* (SURVEY App. A.3).  c_qkv_b may be NULL (qkv_bias False). ---------- */
typedef struct hy3d_transformer_layer {
  const float* ln1_w; const float* ln1_b;
  const float* c_qkv_w; const float* c_qkv_b;          /* [3W, W]; rows viewed [head][q64|k64|v64] (attention_blocks.py:318-321) */
  const float* c_proj_w; const float* c_proj_b;        /* [W, W] */
  const float* q_norm_w; const float* q_norm_b; const float* k_norm_w; const float* k_norm_b;   /* [64] or NULL */
  const float* ln2_w; const float* ln2_b;
  const float* c_fc_w; const float* c_fc_b;            /* [4W, W] */
  const float* mlp_proj_w; const float* mlp_proj_b;    /* [W, 4W] */
} hy3d_transformer_layer;
typedef struct hy3d_transformer_desc {
  int32_t width, heads, layers, embed_dim, qk_norm;
  const float* post_kl_w; const float* post_kl_b;      /* [W, embed_dim], [W] */
  const hy3d_transformer_layer* layer;                 /* HOST array of `layers` entries */
} hy3d_transformer_desc;
int hy3d_set_transformer_weights(hy3d_ctx* ctx, const hy3d_transformer_desc* desc);
/* d_z: fp32 [M, embed_dim] (already divided by scale_factor, pipelines.py:657); d_out: fp32 [M, W]. M % 128 == 0. */
int hy3d_transformer_forward(hy3d_ctx* ctx, const float* d_z, int32_t M, float* d_out);

/* Sequence-parallel form of the same forward pass (no reference counterpart: the reference is single-device; SURVEY §8e).
 * The M tokens of a latent set are split into `parts` equal ranges (M / parts a multiple of 128), one per GPU; every GEMM,
 * LayerNorm and residual acts on rows, only self-attention needs all tokens' K / V.  Per layer the host runs
 *   hy3d_transformer_layer_kv   -> this part's K / V^T tile images into chunk `part` of the exchange buffer,
 *   [all-gather of the chunks across the GPUs — NCCL, done by the caller; in place],
 *   hy3d_transformer_layer_rest -> attention of the local queries against all K / V, c_proj, MLP.
 * Exchange buffer (DEVICE, caller-owned): [parts][2 (K, V^T)][heads][M / parts / 128][16 KB] bytes.
 * hy3d_transformer_forward is exactly begin(parts = 1) + the layer loop on a private buffer + end. */
int hy3d_transformer_begin(hy3d_ctx* ctx, const float* d_z_local, int32_t tokens_local, int32_t parts, int32_t part);
int hy3d_transformer_layer_kv(hy3d_ctx* ctx, int32_t layer, void* d_kv_all);
int hy3d_transformer_layer_rest(hy3d_ctx* ctx, int32_t layer, const void* d_kv_all);
int hy3d_transformer_end(hy3d_ctx* ctx, float* d_out_local);

/* ---- decoder: replaces CrossAttentionDecoder.forward (attention_blocks.py:483-493) ---- */
/* Copies / re-lays-out the weights into the context (fp16 UMMA tiles + fp32 originals). */
int hy3d_set_decoder_weights(hy3d_ctx* ctx, const hy3d_decoder_desc* desc);
/* Per-latent work hoisted out of the query loop: [latents_proj] -> ln_2 -> c_kv -> k_norm
 * (attention_blocks.py:487-488, 296, 257, 205-211).  d_latents: fp32 [M, latent_width]. */
int hy3d_prepare_kv(hy3d_ctx* ctx, const float* d_latents, int32_t M);
/* logits for explicit points.  d_xyz: fp32 [n,3]; d_out: fp32 [n]. */
int hy3d_decode_points(hy3d_ctx* ctx, const float* d_xyz, int64_t n, float* d_out);
/* Dense grid, replaces VanillaVolumeDecoder.__call__'s loop (volume_decoders.py:162-180) for
 * the flat index range [first, first+count) of an [n0,n1,n2] grid (index (i*n1+j)*n2+k).
 * h_axis{0,1,2}: HOST per-axis coordinate tables (np.linspace, volume_decoders.py:131-133).
 * d_out receives `count` logits (d_out[0] is flat index `first`). */
int hy3d_decode_dense(hy3d_ctx* ctx, const float* h_axis0, const float* h_axis1, const float* h_axis2,
                      int32_t n0, int32_t n1, int32_t n2, int64_t first, int64_t count, float* d_out);
/* Sparse list, replaces the refined-level loops (volume_decoders.py:262-274, 394-431):
 * point p = float32(ijk) * cell + bmin (fp32 mul then add), ijk from the flat index
 * d_index[q] of an [n0,n1,n2] grid; result scattered to d_grid[d_index[q]].
 * Entries with d_index[q] < 0 are padding and are skipped. */
int hy3d_decode_list(hy3d_ctx* ctx, const int32_t* d_index, int64_t n, int32_t n0, int32_t n1, int32_t n2,
                     const float h_cell[3], const float h_bmin[3], float* d_grid);

/* Same queries as hy3d_decode_list, compact result: d_values[q] = logit of d_index[q] (used when
 * the ordered list is split across ranks and the values are all-gathered before the scatter). */
int hy3d_decode_list_values(hy3d_ctx* ctx, const int32_t* d_index, int64_t n, int32_t n0, int32_t n1, int32_t n2,
                            const float h_cell[3], const float h_bmin[3], float* d_values);
/* d_grid[d_index[q] - base] = d_values[q] (reference: next_logits[nidx] = grid_logits, volume_decoders.py:273).
 * `base` = flat index of d_grid[0] in the whole grid (0, or the first voxel of a slab kept by one GPU);
 * every non-negative d_index[q] must be >= base.  Entries with d_index[q] < 0 are skipped. */
int hy3d_scatter(hy3d_ctx* ctx, const int32_t* d_index, const float* d_values, int64_t n, int64_t base, float* d_grid);
/* Windowed form of hy3d_scatter for a slab of a grid that is partitioned across GPUs: d_grid holds the flat indices
 * [base, base + len) of the whole grid; only the entries with base <= d_index[q] < base + len are written (as
 * d_grid[d_index[q] - base], a logit equal to the -10000 sentinel as NaN, like hy3d_scatter), all others are skipped. */
int hy3d_scatter_window(hy3d_ctx* ctx, const int32_t* d_index, const float* d_values, int64_t n, int64_t base, int64_t len,
                        float* d_grid);

/* ---- FlashVDM: replaces FlashVDMVolumeDecoding's decoder calls (volume_decoders.py:343-371,
 * 398-431) and the processors of attention_processors.py:35-96 ------------------------------ */
/* How the points of an index list get their coordinates: mode 2 = float32(ijk)*cell + bmin
 * (refined levels, volume_decoders.py:394-396), mode 3 = per-axis HOST tables (level 0 mini-grids). */
typedef struct hy3d_coords {
  int32_t mode;
  float cell[3];
  float bmin[3];
  const float* axis0; const float* axis1; const float* axis2;
} hy3d_coords;
/* KV selection for G groups (mini-grids or spatial bins).  d_sample_index: flat grid indices of the
 * sub-sampled queries (every 100th / 50th / 30th query of each group, in group order; -1 = padding),
 * d_sample_off[g]..d_sample_off[g+1] delimits group g (DEVICE int32 [G+1]).  merge_mode 0: top-`topk`
 * tokens per (group, head) by mean similarity; 1: union of tokens with head-averaged probability
 * > 1e-6, shared by all heads.  The result lives in the context until the next call. */
int hy3d_flash_select(hy3d_ctx* ctx, const int32_t* d_sample_index, int64_t n_samples, int32_t n0, int32_t n1, int32_t n2,
                      const hy3d_coords* coords, const int32_t* d_sample_off, int32_t G, int32_t topk, int32_t merge_mode);
/* Decode a group-ordered, 128-padded index list (-1 = padding) with the selected K/V of each
 * tile's group (d_tile_group: DEVICE int32 [n/128]); logits scattered to d_grid[d_index[q]]. */
int hy3d_decode_flash(hy3d_ctx* ctx, const int32_t* d_index, int64_t n, int32_t n0, int32_t n1, int32_t n2,
                      const hy3d_coords* coords, const int32_t* d_tile_group, float* d_grid);
/* Multi-GPU forms (no reference counterpart: the reference is single-device; SURVEY §8e).  One GPU selects and decodes a
 * contiguous run of tiles of a layout; the groups its tiles use are [g0, g1).
 * hy3d_flash_select_range: hy3d_flash_select restricted to groups [g0, g1) of a layout of G groups.  d_sample_off is the
 * whole layout's DEVICE int32 [G+1]; d_sample_index points at that layout's sample d_sample_off[g0] and n_samples =
 * d_sample_off[g1] - d_sample_off[g0] (known to the caller: no host synchronisation).  Each group's selection is exactly
 * the one hy3d_flash_select makes for it; it is stored under the local ids 0 .. g1-g0-1, and until the next selection
 * hy3d_decode_flash and hy3d_decode_flash_values take a tile's K/V from local group d_tile_group[t] - g0
 * (hy3d_flash_select = the range [0, G)).  A bad range returns HY3D_ERR_ARG.
 * hy3d_decode_flash_values: hy3d_decode_flash with a compact result, d_values[q] = logit of d_index[q] (any value at
 * padding entries); d_index / d_tile_group may be a 128-aligned slice of a layout. */
int hy3d_flash_select_range(hy3d_ctx* ctx, const int32_t* d_sample_index, int64_t n_samples, int32_t n0, int32_t n1, int32_t n2,
                            const hy3d_coords* coords, const int32_t* d_sample_off, int32_t G, int32_t g0, int32_t g1,
                            int32_t topk, int32_t merge_mode);
int hy3d_decode_flash_values(hy3d_ctx* ctx, const int32_t* d_index, int64_t n, int32_t n0, int32_t n1, int32_t n2,
                             const hy3d_coords* coords, const int32_t* d_tile_group, float* d_values);
/* Query layout of a refined FlashVDM level, all on the device (no host synchronisation): replaces
 * volume_decoders.py:394-412 -- bin id of every active query (float32 op for op: floor((p - min) /
 * (max - min) * (6 - 0.001)) per axis, 6^3 = 216 bins, ids clamped to [0, 215]), STABLE sort by bin,
 * per-bin slices and the q[:, :, ::stride] sub-sampling.  d_index: the level's ordered active indices
 * (hy3d_refine_level); coords must be mode 2.  Outputs (DEVICE int32): d_pidx[cap] every bin starting on
 * a multiple of 128, -1 = padding; d_tile_group[cap/128]; d_sidx[scap] every stride-th query of each bin,
 * -1 = padding; d_soff[217]; d_counts[216] (optional, may be NULL).  Static capacities:
 * cap >= round128(n + 216*127), scap >= n/stride + 216. */
int hy3d_flash_layout_bins(hy3d_ctx* ctx, const int32_t* d_index, int64_t n, int32_t n0, int32_t n1, int32_t n2,
                           const hy3d_coords* coords, int32_t stride, int32_t* d_pidx, int64_t cap, int32_t* d_tile_group,
                           int32_t* d_sidx, int64_t scap, int32_t* d_soff, int32_t* d_counts);
/* The same layout for level 0: mini_grid_num^3 mini-grids of (N/mini_grid_num)^3 voxels each, queries of a
 * mini-grid in lexicographic order (volume_decoders.py:343-356).  cap = G*round128(s^3),
 * scap >= G*ceil(s^3/stride), d_soff[G+1]. */
int hy3d_flash_layout_minigrids(hy3d_ctx* ctx, int32_t N, int32_t mini_grid_num, int32_t stride, int32_t* d_pidx, int64_t cap,
                                int32_t* d_tile_group, int32_t* d_sidx, int64_t scap, int32_t* d_soff);
/* Selected token ids / per-group token counts of the last hy3d_flash_select (parity tests). */
int hy3d_flash_selection(hy3d_ctx* ctx, int32_t* d_out, int64_t count);
int hy3d_flash_group_tokens(hy3d_ctx* ctx, int32_t* d_out, int32_t G);

/* ---- octree refinement: replaces volume_decoders.py:29-119 and :245-260 / :376-391 ----- */
/* Active fine voxels of one coarse->fine step (SURVEY App. B): near-surface | band mask,
 * dilation, x2 up-sampling, dilation, ordered compaction.  d_coarse: fp32 [n,n,n] (sentinel
 * -10000 = unvisited).  The fine grid is [nf]^3 with nf = r + 1 of the next level: 2n-1 when the
 * resolution doubles exactly, 2n when the coarser level came from an odd r // 2
 * (volume_decoders.py:202-208, e.g. 390 -> 195 -> 97); up-sampled voxels sit at 2c and the
 * dilations are clipped at the fine grid's faces, as the zero-padded Conv3d of the reference is.
 * Writes the lexicographically ordered flat fine indices ((i*nf + j)*nf + k) to d_index
 * (capacity `cap`), returns their number in *h_count (HOST; this call synchronises the stream
 * once).  If the count exceeds cap nothing is written past cap and *h_count still holds the
 * true count. */
int hy3d_refine_level(hy3d_ctx* ctx, const float* d_coarse, int32_t n, int32_t nf, float mc_level, int32_t last_level,
                      int32_t* d_index, int64_t cap, int64_t* h_count);
int hy3d_fill(hy3d_ctx* ctx, float* d_grid, int64_t n, float value);
/* grid[grid == sentinel] = NaN (volume_decoders.py:275, :433). */
int hy3d_sentinel_to_nan(hy3d_ctx* ctx, float* d_grid, int64_t n, float sentinel);

/* ---- marching cubes: replaces MCSurfaceExtractor.run (surface_extractors.py:68-76) ------ */
/* Phase 1: classify + count.  d_grid: fp32 [n0,n1,n2]; inside test `v - level > 0`, NaN =>
 * outside.  Returns vertex/face counts and the finite min/max of the field in HOST
 * variables (synchronises the stream once).  h_minmax[2] = 1 if the grid holds NaN. */
int hy3d_mc_count(hy3d_ctx* ctx, const float* d_grid, int32_t n0, int32_t n1, int32_t n2, float level,
                  int64_t* h_num_verts, int64_t* h_num_faces, float h_minmax[3]);
/* Phase 2: emit the welded, indexed mesh of the grid given to the last hy3d_mc_count.
 * Vertex v (index units, array-axis order) is written as
 *   float32( double(v) / h_div[a] * h_mul[a] + h_add[a] )   per axis a
 * which is the reference's `vertices / grid_size * bbox_size + bbox_min` (float64, :75).
 * d_verts: fp32 [V,3]; d_faces: int32 [F,3]. */
int hy3d_mc_emit(hy3d_ctx* ctx, const double h_div[3], const double h_mul[3], const double h_add[3],
                 float* d_verts, int32_t* d_faces);
/* Slab forms for grids partitioned along axis 0 across GPUs (no reference counterpart: the reference is single-device;
 * SURVEY §8e).  d_grid holds planes [plane0, plane0 + n0) of the whole grid: the first `own_planes` are OWNED by this
 * slab, the rest (two planes, fewer at the end of the grid) are the next slab's first planes, kept as a halo.  Counted
 * and emitted: the vertices on edges starting at owned voxels and the triangles of cubes based at owned planes.  Vertex
 * and face orders are the global lexicographic ones, so the meshes of consecutive slabs concatenate into exactly the
 * mesh hy3d_mc_count / hy3d_mc_emit produce for the whole grid when each slab passes
 *   id_base = number of vertices owned by all earlier slabs
 * (faces of the last owned plane reference vertices of the first halo plane: their ids continue past this slab's own
 * count, which is why the halo is two planes deep — the ids depend on that plane's axis-0 edges too). */
int hy3d_mc_count_slab(hy3d_ctx* ctx, const float* d_grid, int32_t n0, int32_t n1, int32_t n2, int32_t own_planes, float level,
                       int64_t* h_num_verts, int64_t* h_num_faces, float h_minmax[3]);
int hy3d_mc_emit_slab(hy3d_ctx* ctx, const double h_div[3], const double h_mul[3], const double h_add[3], int32_t plane0,
                      int64_t id_base, float* d_verts, int32_t* d_faces);
/* ---- dual marching cubes: replaces DMCSurfaceExtractor.run (surface_extractors.py:79-94), i.e. diso.DiffDMC(sdf =
 * -logits / res, normalize=True) + center_vertices (:29-34) + the reversed winding ------------------------------------
 * Phase 1: classify + count.  d_grid: fp32 [n0,n1,n2]; inside test `g > 0` (iso-value 0 of sdf = -logit / res), NaN =>
 * outside.  Returns in HOST variables the vertex count (one per iso-surface patch of every cube, the patches of
 * mc_tables.inc's loops), the face count (two per sign-change edge whose four cubes lie inside the grid) and the finite
 * min/max of the field, h_minmax[2] = 1 if the grid holds NaN (synchronises the stream once). */
int hy3d_dmc_count(hy3d_ctx* ctx, const float* d_grid, int32_t n0, int32_t n1, int32_t n2, int64_t* h_num_verts,
                   int64_t* h_num_faces, float h_minmax[3]);
/* Phase 2: emit the mesh of the grid given to the last hy3d_dmc_count.  Vertex = mean of its patch's edge crossings
 * (float64, divided by n_axis - 1 per axis: the grid spans the unit cube), rounded to fp32, then centred on the bounding
 * box of the non-NaN vertices in fp32; vertices in lexicographic (cube, patch) order, faces (two triangles per quad) in
 * lexicographic (edge owner voxel, edge axis) order, oriented like hy3d_mc_emit's.  d_verts: fp32 [V,3]; d_faces:
 * int32 [F,3]. */
int hy3d_dmc_emit(hy3d_ctx* ctx, float* d_verts, int32_t* d_faces);
/* ---- mesh clean-up: the device side of export_to_trimesh (hy3dgen/shapegen/pipelines.py:95-110) ---------------------
 * `mesh_f[:, ::-1]` (flip_winding != 0) and what trimesh.Trimesh(v, f)'s default processing does to a mesh with
 * non-finite vertices: faces that reference a NaN / inf vertex are dropped, then vertices that are non-finite or no longer
 * referenced, and the faces are re-indexed; the order of the survivors is preserved.  d_verts fp32 [nV,3], d_faces int32
 * [nF,3]; the outputs need room for nV / nF entries and must not alias the inputs.  Returns the new counts in HOST
 * variables (synchronises the stream once). */
int hy3d_mesh_clean(hy3d_ctx* ctx, const float* d_verts, int64_t nV, const int32_t* d_faces, int64_t nF, int32_t flip_winding,
                    float* d_verts_out, int32_t* d_faces_out, int64_t* h_num_verts_out, int64_t* h_num_faces_out);
/* ---- mesh post-processing: FloaterRemover / DegenerateFaceRemover (hy3dgen/shapegen/postprocessors.py) --------------------
 * Same buffers, output order and single synchronisation as hy3d_mesh_clean (no winding flip): surviving faces keep their
 * order and winding, vertices are kept iff a surviving face references them, in their original order.  Vertex and face ids
 * above int32 return HY3D_ERR_UNSUPPORTED; a face index outside [0, nV) is never dereferenced and returns HY3D_ERR_ARG; a
 * mesh that becomes empty returns counts 0.
 * Floaters, replacing pymeshlab's compute_selection_by_small_disconnected_components_per_face(nbfaceratio) +
 * compute_selection_transfer_face_to_vertex(inclusive=False) + meshing_remove_selected_vertices_and_faces: faces are
 * connected iff they share an undirected edge {a, b}, a != b (any number of faces per edge); a component of fewer than
 * min_faces faces is small (FloaterRemover passes int(0.005 * nF)); every vertex of a small component's face is selected
 * and every face with a selected vertex is removed. */
int hy3d_mesh_remove_floaters(hy3d_ctx* ctx, const float* d_verts, int64_t nV, const int32_t* d_faces, int64_t nF,
                              int64_t min_faces, float* d_verts_out, int32_t* d_faces_out, int64_t* h_num_verts_out,
                              int64_t* h_num_faces_out);
/* Weld, replacing DegenerateFaceRemover's pymeshlab / trimesh round trip: every vertex is replaced by the smallest vertex id
 * with the same three fp32 bit patterns (-0.0 taken as +0.0; a vertex with a non-finite coordinate is never merged), then
 * a face with two equal ids is removed.  Collinear and duplicate faces are kept; there is no distance tolerance. */
int hy3d_mesh_weld(hy3d_ctx* ctx, const float* d_verts, int64_t nV, const int32_t* d_faces, int64_t nF, float* d_verts_out,
                   int32_t* d_faces_out, int64_t* h_num_verts_out, int64_t* h_num_faces_out);
/* Quadric edge-collapse decimation, replacing FaceReducer's pymeshlab meshing_decimation_quadric_edge_collapse(
 * targetfacenum=max_faces, qualitythr=1.0, preserveboundary=True, boundaryweight=3, preservenormal=True,
 * preservetopology=True, autoclean=True); contract oracle/decimate.py, parity with pymeshlab unpinned.  nF <= max_faces:
 * the mesh is copied as given.  Otherwise rounds of independent collapses, each on the compacted mesh of the previous one:
 * vertices on boundary or non-manifold edges, without one closed fan, in a face with a repeated id or non-finite never move;
 * a candidate edge (a, b) has exactly two oppositely oriented faces (a, b, c) and (b, a, d), free ends, common neighbours
 * exactly {c, d}, deg(a) + deg(b) - 4 >= 3 and deg(c), deg(d) >= 4; a takes the float32-rounded cheapest of the minimiser of
 * Qa + Qb (unit plane quadrics of the input, |det| >= 1e-12), pa, pb and the midpoint; the collapse is invalid if a face
 * of the two stars would get n_old . n_new <= 0; cost = max(pQp, 1e-15) / min(worst new face quality, 1).  Edges ranked
 * by (cost, edge id) are selected when their rank is the smallest over both ends and their neighbours, and at most
 * ceil((F - max_faces) / 2) of them apply, so the result has max_faces - 1 or max_faces faces unless a round finds no
 * valid collapse (the mesh is then returned with more faces).  Same buffers, int32 rules and output order as
 * hy3d_mesh_weld; max_faces < 1 and a face index outside [0, nV) return HY3D_ERR_ARG.  *h_rounds = rounds that applied
 * collapses.  One host synchronisation per round (the new counts and the error flag); the final copies into the output
 * buffers are enqueued on the context's stream after the last one. */
int hy3d_mesh_decimate(hy3d_ctx* ctx, const float* d_verts, int64_t nV, const int32_t* d_faces, int64_t nF, int64_t max_faces,
                       float* d_verts_out, int32_t* d_faces_out, int64_t* h_num_verts_out, int64_t* h_num_faces_out,
                       int32_t* h_rounds);
/* Table-independent classification for parity tests: 8-bit case per cube, [n0-1,n1-1,n2-1]. */
int hy3d_mc_cases(hy3d_ctx* ctx, const float* d_grid, int32_t n0, int32_t n1, int32_t n2, float level,
                  uint8_t* d_cases);

/* ---- measurement ----------------------------------------------------------------------- */
/* Device timing per kernel family with CUDA events recorded on the launch stream around every
 * launch (enable=1).  hy3d_profile_read synchronises, returns and clears the totals:
 * h_ms[f] milliseconds and h_count[f] launches of family f.  Families: 0 embed, 1 gemm query_proj,
 * 2 layernorm, 3 gemm c_q, 4 attention, 5 gemm c_proj, 6 gemm c_fc, 7 gemm mlp.c_proj, 8 head,
 * 9 mc bits, 10 mc rowcount, 11 mc scan, 12 mc emit, 13 octree, 14 kv prepare, 15 kv select. */
int hy3d_profile(hy3d_ctx* ctx, int enable);
int hy3d_profile_read(hy3d_ctx* ctx, double h_ms[16], int64_t h_count[16]);

/* ---- diagnostics ---------------------------------------------------------------------- */
/* Synchronises the stream and returns + clears the tensor-path watchdog record:
 * h_out[0] != 0 means an mbarrier wait timed out inside a tcgen05 kernel (results of that
 * launch are invalid); h_out[1..4] = block, thread, barrier shared address, parity. */
int hy3d_debug_watchdog(hy3d_ctx* ctx, int32_t h_out[8]);
/* Keep (enable=1) the per-stage activations of the last decoded chunk for hy3d_debug_fetch.
 * Stage ids: 0 x0, 1 ln_1(x0), 2 q after q_norm (the tcgen05 path stores q*scale*log2e),
 * 3 attention output, 4 x1, 5 ln_3(x1), 6 MLP hidden, 7 x2.  Costs one device copy per stage. */
int hy3d_debug_retain(hy3d_ctx* ctx, int enable);
/* Kernel-tuning experiments (tools/gpu_chain_bench.py): `bits` disables parts of the tcgen05 kernels
 * (1 GEMM epilogue, 2 GEMM MMAs, 4 GEMM epilogue stores) so that their cost can be measured by difference — results
 * are garbage while those are set; 0x20 forces the online-softmax attention kernel, 0x40 runs the instrumented
 * bounded-score attention kernel (hy3d_debug_timers), 0x10000 the CUDA-core K/V projection (results stay valid);
 * 0x100 gives every attention stream its own K/V ring even when all query tiles share one K/V set;
 * `attn_poly` = pairs of every 8 pairs of attention exponentials evaluated as packed polynomials on the FMA pipe
 * (0 none, 1 .. 6 = that many pairs, 8 = all; other values select the default, 2 = a quarter of the exponentials).
 * Defaults (0, 2) are the product configuration. */
int hy3d_debug_experiment(hy3d_ctx* ctx, int bits, int attn_poly);
/* Phase clocks accumulated by the instrumented attention kernel (experiment bit 0x40), returned and cleared:
 * per head stream a (0, 1) h_out[8a + i] = SM cycles one softmax thread of CTA 0 spent in phase i
 * (0 wait S, 1 load S, 2 exponentials, 3 wait PV, 4 store P, 5 finalize), h_out[8a + 7] = KV tiles. */
int hy3d_debug_timers(hy3d_ctx* ctx, uint64_t h_out[32]);
/* (query tile, head pair) items the exact redo pass recomputed after the LAST bounded-score attention launch with per-head
 * shifts (normally 0; see hy3d_attention_info).  Synchronises the stream. */
int hy3d_debug_attn_redo(hy3d_ctx* ctx, int32_t* h_items);
/* Row-major fp32 [rows, *h_width] copy of a retained stage, whatever its internal layout. */
int hy3d_debug_fetch(hy3d_ctx* ctx, int stage, float* d_out, int64_t rows, int32_t* h_width);

#ifdef __cplusplus
}
#endif
#endif /* HY3DGEO_H */
