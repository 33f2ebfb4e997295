// Attention of the tcgen05 decoder chain and of the latent transformer (reference
// attention_processors.py:29-32 SDPA; attention_blocks.py:184-215 / :301-345): softmax(q k^T) v per head,
// head dim 64, 128-query tiles, fp16 operands, fp32 accumulation in tensor memory.
// Included by decoder_tc.cu inside its anonymous namespace (uses TILE_BYTES, store_t16_* and tc::).
//
// One CTA iteration = two independent *streams* of one (128-query tile, head) each:
//   share_kv = 1 (plain decoding, the latent transformer): the two streams are two QUERY TILES of the SAME head and consume
//                the same K / V^T tiles from ONE ring of 10 slots, loaded once by one producer warp — half the L2 -> SM
//                traffic and half the shared-memory fill bandwidth of giving each stream its own copy (the K/V of a head
//                used to be re-streamed from L2 for every 128 queries: ~31 B/clk/SM, three quarters of the L2 ceiling);
//   share_kv = 0 (FlashVDM: neighbouring query tiles may belong to different KV groups): the two streams are two HEADS of
//                one query tile, each with its own producer warp and ring of 5 slots.
//   producer warp  (warp 0 / 2a): Q tile(s), then K(0), K(1), V(0), K(2), V(1), ... through a ring of 16 KB slots
//                               (1-D bulk copies: every tile is one contiguous SW128 K-major image)
//   MMA warp       (warp 2a+1): S = Q K(j)^T  (4 x tcgen05.mma 128x128x16, A and B from shared memory)
//                               O += P(j) V(j) (8 x tcgen05.mma 128x64x16, A = P from TENSOR memory, B = V^T)
//   softmax warps:              S -> registers, exponentials, P -> tensor memory as packed fp16 pairs
// so that neither stream's waits block the other and the tensor pipe interleaves their MMAs.
// Both single-thread roles run with the whole warp converged and issue through one elected lane (tc::elect_one):
// under a divergent `if (lane == 0)` ptxas wraps every tcgen05.mma in a ~100-cycle uniform-register waterfall,
// which alone capped this kernel at ~30 % of the tensor peak.
// TMEM columns: S[a] (fp32, 128) at a*128; P[a] (fp16 pairs, 64) at 256 + a*64; O[a] (fp32, 64) at 384 + a*64.
// P never crosses shared memory, whose bandwidth (operand reads + TMA fills) is the scarce resource here.
//
// Two softmax bodies:
//  * k_attn_fast — used when the scores are provably bounded: with q_norm / k_norm (LayerNorm over the 64 head
//    dims, reference attention_blocks.py:197-198,210-211) |q.k| * scale * log2e <= B, a constant of the norm
//    weights (attn_score_bound).  For B <= 15.9 no exp2(s) can overflow fp16, so the softmax needs NO running
//    maximum, no subtraction and no rescaling of O: p = exp2(s) directly — mathematically the same softmax (the
//    common factor cancels in O / l).  Probabilities below 2^-14 are fp16 subnormals (absolute error <= 2^-25,
//    i.e. <= 2^-9 of the row's largest term even in the worst case of a row whose every score sits at -B; rows
//    whose best score is >= -5 — every row of a trained or random model — lose < 2^-20 per term).  Two threads per
//    query row (16 softmax warps) halve the serial latency of each stream; per pair of elements the instruction
//    stream is 2 MUFU.EX2 + FADD2 + F2FP, or the packed polynomial (3 FADD2 + 3 FFMA2 + 2 IMAD + FADD2 + F2FP) for
//    kPoly of every 8 pairs.  Heads whose measured bound exceeds 15.9 subtract a per-head shift first (head_shift) and
//    rows that end up far below it are flagged for an exact redo by k_attn_tc (redo_list).
//  * k_attn_tc — online softmax with a running maximum (lazy rescale) for everything else (no q/k norm, norm gains
//    beyond the shift range, the redo pass).  Same two-threads-per-row layout; the halves of a row exchange their
//    tile maximum through shared memory.
#pragma once

constexpr int ATT_SLOTS = 5;               // K / V^T ring per stream, 16 KB each
constexpr int TM_S0 = 0, TM_P0 = 256, TM_O0 = 384;
constexpr int ATT_THREADS = 640;           // k_attn_tc: 4 role warps + 2 x 8 softmax warps (two threads per row)
constexpr int ATT_FAST_THREADS = 640;      // k_attn_fast: 4 role warps + 2 x 8 softmax warps
constexpr float ATT_FAST_BOUND = 15.9f;    // exp2(15.9) = 61147 < 65504: no fp16 overflow, ever

struct AttnTC {
  const uint8_t* Q;      // T16 [Pb][H]  (q already scaled by 1/sqrt(d) * log2e)
  const uint8_t* K;      // [group][H][nkv][16 KB]
  const uint8_t* V;      // [group][H][nkv][16 KB]  (V^T: 2 x [64 d x 64 tok] per tile)
  uint8_t* O;            // T16 [Pb][H]
  const int* tile_group; // per q-tile KV group or null
  const int* group_ntok; // valid tokens per group or null
  int Pb, H, nkv, ntok;  // nkv = tiles per (group, head); ntok = valid tokens when group_ntok == null
  int group_base;        // K / V / group_ntok hold groups group_base, group_base + 1, ... (tile_group values are absolute)
  int split_out;         // O written as [hi | lo | hi] over 3H k-blocks (operand of a 3-term split GEMM)
  int share_kv;          // 1: streams = two query tiles of one head sharing every K/V tile; 0: two heads of one query tile
  // K / V gathered from several GPUs (sequence-parallel latent transformer): tile j of head h lives in chunk j / kv_tpr at
  // K + (j / kv_tpr) * kv_chunk_stride + (h * kv_tpr + j % kv_tpr) * 16 KB (same for V).  kv_tpr = 0: one chunk of nkv tiles.
  int kv_tpr; long long kv_chunk_stride;
  int no_pipe;           // experiment: load both 32-column halves of S before any exponential (no software pipeline)
  // bounded-score kernel with measured bounds: p = exp2(s - head_shift[h]); rows whose sum falls below ntok * 2^-14 (all their
  // scores far below the head's bound: the fp16 probabilities would be subnormal) flag their (tile, head pair) for an exact redo
  const float* head_shift;      // [H] or null (no shift)
  int* redo_count; int* redo_list; int* redo_flag;      // device work list filled by the bounded-score kernel (or null)
  // online-softmax kernel in list mode: items come from a device work list written by an earlier launch
  const int* work_count; const int* work_list;
  unsigned long long* timers;   // k_attn_fast<.., true>: phase clocks of CTA 0 (see hy3d_debug_timers)
};

struct AttnBars {                          // mbarrier addresses (shared window), per stream a
  uint32_t b0;
  static constexpr int NB = 2 * ATT_SLOTS + 6;
  __device__ __forceinline__ uint32_t kvfull(int a, int s) const { return b0 + 8u * (a * NB + s); }
  __device__ __forceinline__ uint32_t kvempty(int a, int s) const { return b0 + 8u * (a * NB + ATT_SLOTS + s); }
  // shared ring (share_kv): slot s in [0, 2 SLOTS) uses stream (s / SLOTS)'s barrier s % SLOTS
  __device__ __forceinline__ uint32_t kvfull_sh(int s) const { return kvfull(s >= ATT_SLOTS, s >= ATT_SLOTS ? s - ATT_SLOTS : s); }
  __device__ __forceinline__ uint32_t kvempty_sh(int s) const { return kvempty(s >= ATT_SLOTS, s >= ATT_SLOTS ? s - ATT_SLOTS : s); }
  __device__ __forceinline__ uint32_t qfull(int a) const { return b0 + 8u * (a * NB + 2 * ATT_SLOTS); }
  __device__ __forceinline__ uint32_t qempty(int a) const { return b0 + 8u * (a * NB + 2 * ATT_SLOTS + 1); }
  __device__ __forceinline__ uint32_t sfull(int a) const { return b0 + 8u * (a * NB + 2 * ATT_SLOTS + 2); }
  __device__ __forceinline__ uint32_t sempty(int a) const { return b0 + 8u * (a * NB + 2 * ATT_SLOTS + 3); }
  __device__ __forceinline__ uint32_t pfull(int a) const { return b0 + 8u * (a * NB + 2 * ATT_SLOTS + 4); }
  __device__ __forceinline__ uint32_t pvdone(int a) const { return b0 + 8u * (a * NB + 2 * ATT_SLOTS + 5); }
};

constexpr int ATT_TILES_BYTES = (2 + 2 * ATT_SLOTS) * TILE_BYTES;      // Q[2] + K/V ring[2][SLOTS]
constexpr size_t ATT_SMEM = 1024 + ATT_TILES_BYTES + 512 + 2048 + 4096; // + barriers / TMEM slot + row-sum exchange + tile-maximum exchange (k_attn_tc)

// Shared prologue: barriers, TMEM.  `softmax_warps` = arrivals expected on SEMPTY / PFULL per stream.
__device__ __forceinline__ uint32_t attn_setup(uint8_t* smem, AttnBars& B, int softmax_warps, int share_kv) {
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + ATT_TILES_BYTES);
  B.b0 = smem_u32(bars);
  asm volatile("" : "+r"(B.b0));        // opaque: otherwise every barrier use re-derives the shared-window address from special registers
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * AttnBars::NB);
  const int warp = threadIdx.x >> 5;
  if (threadIdx.x == 0) {
    for (int a = 0; a < 2; ++a) {
      for (int s = 0; s < ATT_SLOTS; ++s) { mbar_init(B.kvfull(a, s), 1); mbar_init(B.kvempty(a, s), share_kv ? 2 : 1); }   // shared slot: released by both streams' MMAs
      mbar_init(B.qfull(a), 1); mbar_init(B.qempty(a), 1);
      mbar_init(B.sfull(a), 1); mbar_init(B.sempty(a), softmax_warps); mbar_init(B.pfull(a), softmax_warps); mbar_init(B.pvdone(a), 1);
    }
    fence_barrier_init();
  }
  if (warp == 2) { tmem_alloc(smem_u32(tmem_slot), 512); tmem_relinquish(); }
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  return *tmem_slot;
}

// Work item -> (query tile, head) of stream a.  share_kv: item = (pair of query tiles, head), stream a takes tile 2 pair + a
// (an odd tile count leaves the last pair's second stream on a duplicate of the last tile; it computes but does not store).
struct AttnItem { int qt, h; bool store; };
__device__ __forceinline__ int attn_num_items(const AttnTC& g) {
  if (g.work_count) return *g.work_count;           // list mode (uniform: every thread reads the same word)
  return g.share_kv ? ((g.Pb + 1) >> 1) * g.H : g.Pb * (g.H >> 1);
}
__device__ __forceinline__ AttnItem attn_item(const AttnTC& g, int item, int a) {
  AttnItem it;
  if (g.work_list) {                                // entry = query tile * (H / 2) + head pair
    const int HP = g.H >> 1, e = g.work_list[item];
    it.qt = e / HP; it.h = (e - it.qt * HP) * 2 + a; it.store = true;
  } else if (g.share_kv) {
    const int pr = item / g.H, q = 2 * pr + a;
    it.h = item - pr * g.H; it.store = q < g.Pb; it.qt = it.store ? q : g.Pb - 1;
  } else {
    const int HP = g.H >> 1;
    it.qt = item / HP; it.h = (item - it.qt * HP) * 2 + a; it.store = true;
  }
  return it;
}

// Producer warp of stream a (whole warp converged).  share_kv: called once (a = 0) and feeds both streams.
__device__ __forceinline__ void attn_producer(const AttnTC& g, const AttnBars& B, uint8_t* smem, int a) {
  const bool sh = g.share_kv != 0;
  uint32_t ring32 = smem_u32(smem + 2 * TILE_BYTES + (sh ? 0 : a * ATT_SLOTS * TILE_BYTES)), q32 = smem_u32(smem);
  asm volatile("" : "+r"(ring32), "+r"(q32));
  const int nslots = sh ? 2 * ATT_SLOTS : ATT_SLOTS;
  const int nitems = attn_num_items(g), nkv = g.nkv;
  int s = 0; uint32_t ph = 0, qph = 0;
  auto push = [&](const uint8_t* src) {
    const uint32_t full = sh ? B.kvfull_sh(s) : B.kvfull(a, s), empty = sh ? B.kvempty_sh(s) : B.kvempty(a, s);
    mbar_wait(empty, ph ^ 1);
    if (elect_one()) {
      mbar_arrive_expect_tx(full, TILE_BYTES);
      bulk_g2s(ring32 + s * TILE_BYTES, src, TILE_BYTES, full);
    }
    __syncwarp();
    if (++s == nslots) { s = 0; ph ^= 1; }
  };
  for (int item = blockIdx.x; item < nitems; item += gridDim.x) {
    AttnItem it = attn_item(g, item, a);
    for (int aa = a; aa < (sh ? 2 : a + 1); ++aa) {           // Q tile of each stream this producer feeds
      const AttnItem iq = attn_item(g, item, aa);
      mbar_wait(B.qempty(aa), qph ^ 1);
      if (elect_one()) {
        mbar_arrive_expect_tx(B.qfull(aa), TILE_BYTES);
        bulk_g2s(q32 + aa * TILE_BYTES, g.Q + ((size_t)iq.qt * g.H + iq.h) * TILE_BYTES, TILE_BYTES, B.qfull(aa));
      }
      __syncwarp();
    }
    qph ^= 1;
    const int grp = g.tile_group ? g.tile_group[it.qt] - g.group_base : 0;
    const int tpr = g.kv_tpr ? g.kv_tpr : nkv;
    const size_t head_off = ((size_t)grp * g.H + it.h) * tpr * TILE_BYTES;
    auto tile = [&](const uint8_t* base, int j) {
      return g.kv_tpr ? base + (size_t)(j / tpr) * g.kv_chunk_stride + head_off + (size_t)(j % tpr) * TILE_BYTES
                      : base + head_off + (size_t)j * TILE_BYTES;
    };
    push(tile(g.K, 0));
    for (int j = 0; j < nkv; ++j) {
      if (j + 1 < nkv) push(tile(g.K, j + 1));
      push(tile(g.V, j));
    }
  }
}

// MMA-issuing warp of stream a (whole warp converged, one elected lane issues).
__device__ __forceinline__ void attn_mma(const AttnTC& g, const AttnBars& B, uint8_t* smem, uint32_t tmem, int a) {
  const bool sh = g.share_kv != 0;
  uint8_t* sQ = smem + a * TILE_BYTES;
  const int nslots = sh ? 2 * ATT_SLOTS : ATT_SLOTS;
  const int nitems = attn_num_items(g), nkv = g.nkv;
  const uint32_t idesc_s = make_idesc_f16(128, 128);
  const uint32_t idesc_o = make_idesc_f16(128, 64);
  uint32_t d_s = tmem + TM_S0 + a * 128, d_o = tmem + TM_O0 + a * 64, a_p = tmem + TM_P0 + a * 64;
  uint64_t qd = make_desc_sw128(smem_u32(sQ));
  // descriptor of ring slot 0; slot s adds s * TILE_BYTES / 16 to the address field.  Opaque (see attn_setup): this warp's
  // wake-up -> MMA issue path is on the serial chain of the stream.
  uint64_t ring_d = make_desc_sw128(smem_u32(smem + 2 * TILE_BYTES + (sh ? 0 : a * ATT_SLOTS * TILE_BYTES)));
  asm volatile("" : "+r"(d_s), "+r"(d_o), "+r"(a_p), "+l"(qd), "+l"(ring_d));
  int s = 0; uint32_t ph = 0, qph = 0, sph = 0, pph = 0;
  // instrumented launches (hy3d_debug_timers): cycles this warp waits for 0 K tile, 1 S buffer free, 2 V tile, 3 P stored
  const bool tmr = g.timers != nullptr && blockIdx.x == 0;
  long long tw[4] = {0, 0, 0, 0}, t0 = 0;
  auto tick = [&](int i) { if (tmr) { const long long t_ = clock64(); tw[i] += t_ - t0; t0 = t_; } };
  auto issue_s = [&]() {
    const uint32_t full = sh ? B.kvfull_sh(s) : B.kvfull(a, s), empty = sh ? B.kvempty_sh(s) : B.kvempty(a, s);
    if (tmr) t0 = clock64();
    mbar_wait(full, ph);
    tick(0);
    mbar_wait(B.sempty(a), sph ^ 1); sph ^= 1;
    tick(1);
    fence_after_sync();
    const uint64_t bd = ring_d + (uint64_t)(s * (TILE_BYTES / 16));
    if (elect_one()) {
#pragma unroll
      for (int k = 0; k < 4; ++k) mma_f16_ss(d_s, qd + 2 * k, bd + 2 * k, idesc_s, k != 0);
      mma_commit(empty);
      mma_commit(B.sfull(a));
    }
    __syncwarp();
    if (++s == nslots) { s = 0; ph ^= 1; }
  };
  auto issue_pv = [&](int j) {
    const uint32_t full = sh ? B.kvfull_sh(s) : B.kvfull(a, s), empty = sh ? B.kvempty_sh(s) : B.kvempty(a, s);
    if (tmr) t0 = clock64();
    mbar_wait(full, ph);
    tick(2);
    mbar_wait(B.pfull(a), pph); pph ^= 1;
    tick(3);
    fence_after_sync();
    const uint64_t bd = ring_d + (uint64_t)(s * (TILE_BYTES / 16));
    if (elect_one()) {
#pragma unroll
      for (int k = 0; k < 8; ++k)                      // 16 tokens (8 TMEM columns of fp16 pairs) per MMA
        mma_f16_ts(d_o, a_p + 8 * k, bd + (k >> 2) * (TILE_BYTES / 2 / 16) + 2 * (k & 3), idesc_o, (j | k) != 0);
      mma_commit(empty);
      mma_commit(B.pvdone(a));
    }
    __syncwarp();
    if (++s == nslots) { s = 0; ph ^= 1; }
  };
  for (int item = blockIdx.x; item < nitems; item += gridDim.x) {
    mbar_wait(B.qfull(a), qph); qph ^= 1;
    fence_after_sync();
    issue_s();
    for (int j = 0; j < nkv; ++j) {
      if (j + 1 < nkv) issue_s();
      else { if (elect_one()) mma_commit(B.qempty(a)); __syncwarp(); }   // all S MMAs of this item issued: Q may be refilled once they finish
      issue_pv(j);
    }
  }
  if (tmr && (threadIdx.x & 31) == 0)
    for (int i = 0; i < 4; ++i) atomicAdd(&g.timers[16 + a * 4 + i], (unsigned long long)tw[i]);
}

// exp2 on the FMA/ALU pipes (Cody-Waite split + degree-3 minimax on [-0.5, 0.5], max rel. error 1.6e-4, below the
// fp16 rounding of the stored probability): takes kPoly of every 8 exponentials off the SFU.
__device__ __forceinline__ float exp2_poly(float x) {
  x = fmaxf(x, -126.f);
  const float t = x + 12582912.f;                 // round to nearest integer in the low mantissa bits
  const float f = x - (t - 12582912.f);
  float p = fmaf(5.360121652e-02f, f, 2.423726171e-01f);
  p = fmaf(p, f, 6.935024858e-01f);
  p = fmaf(p, f, 9.999481440e-01f);
  return __int_as_float(__float_as_int(p) + (__float_as_int(t) << 23));
}
template <int kPoly>
__device__ __forceinline__ bool exp_on_fma(int i) {
  // 16-element patterns of the online-softmax kernel: kPoly 1 = 2/16, 5 = 3/16, 2 = 4/16, 3 = 6/16, 4 = 8/16
  constexpr unsigned kMask = kPoly == 0 ? 0x0000u : kPoly == 1 ? 0x1010u : kPoly == 5 ? 0x0842u : kPoly == 2 ? 0x2222u : kPoly == 3 ? 0x5252u
                           : kPoly == 4 ? 0xAAAAu : 0xEEEEu;
  return ((kMask >> (i & 15)) & 1u) != 0;
}
// Bounded-score kernel: whole PAIRS of adjacent exponentials go to the FMA pipe so that the polynomial runs on packed
// f32x2 instructions (FADD2 / FFMA2: both lanes for one issue slot) — kPairs of every 8 pairs (= 2 kPairs / 16 elements).
template <int kPairs>
__device__ __forceinline__ bool pair_on_fma(int pair) {
  constexpr unsigned kMask = kPairs <= 0 ? 0x00u : kPairs == 1 ? 0x10u : kPairs == 2 ? 0x44u : kPairs == 3 ? 0x54u : kPairs == 4 ? 0xAAu
                           : kPairs == 5 ? 0xB5u : kPairs == 6 ? 0xEEu : 0xFFu;
  return ((kMask >> (pair & 7)) & 1u) != 0;
}
// exp2 of two finite scores (|x| <= 15.9, no clamp needed) on the FMA pipe: 3 FADD2 + 3 FFMA2 + 2 integer ops for the pair
__device__ __forceinline__ void exp2_poly2(float x0, float x1, float& p0, float& p1) {
  const uint64_t kMagic = pack_f2(12582912.f, 12582912.f);
  const uint64_t c3 = pack_f2(5.360121652e-02f, 5.360121652e-02f), c2 = pack_f2(2.423726171e-01f, 2.423726171e-01f);
  const uint64_t c1 = pack_f2(6.935024858e-01f, 6.935024858e-01f), c0 = pack_f2(9.999481440e-01f, 9.999481440e-01f);
  const uint64_t x = pack_f2(x0, x1);
  const uint64_t t = add_f2(x, kMagic);                // integer part in the low mantissa bits
  const uint64_t f = sub_f2(x, sub_f2(t, kMagic));     // fraction in [-0.5, 0.5]
  uint64_t p = fma_f2(c3, f, c2);
  p = fma_f2(p, f, c1);
  p = fma_f2(p, f, c0);
  float pa, pb, ta, tb;
  unpack_f2(p, pa, pb); unpack_f2(t, ta, tb);
  p0 = __int_as_float(__float_as_int(pa) + (__float_as_int(ta) << 23));
  p1 = __int_as_float(__float_as_int(pb) + (__float_as_int(tb) << 23));
}

// ------------------------------------------------------------------------------------------
// Bounded scores: no running maximum, two threads per query row.
// ------------------------------------------------------------------------------------------
template <int kPoly, bool kTimers>
__global__ void __launch_bounds__(ATT_FAST_THREADS, 1) k_attn_fast(AttnTC g) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  AttnBars B;
  const uint32_t tmem = attn_setup(smem, B, 8, g.share_kv);
  float* lsum = reinterpret_cast<float*>(smem + ATT_TILES_BYTES + 512);   // [2 streams][2 halves][128 rows]
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nitems = attn_num_items(g), nkv = g.nkv;

  // Registers move inside the CTA's launch allocation (640 x 96): the role warpgroup gives up 40 per thread, the four
  // softmax warpgroups take 8 more each (128 x 56 + 512 x 104 <= 640 x 96) — at 96 the softmax loop spilled and the
  // compiler re-derived every barrier / TMEM address from %tid and the shared window base at each use.
  if (warp < 4) {
    reg_dealloc<56>();
    if ((warp & 1) == 0) { if (!g.share_kv || warp == 0) attn_producer(g, B, smem, warp >> 1); }   // shared ring: one producer
    else attn_mma(g, B, smem, tmem, warp >> 1);
  } else {
    reg_alloc<104>();
    const int a = (warp - 4) >> 3;                      // head stream
    const int hh = ((warp - 4) >> 2) & 1;               // column half: tokens [64 hh, 64 hh + 64) of every KV tile
    const int q = warp & 3;                             // TMEM lane quadrant
    const int r = q * 32 + lane;                        // query row
    const uint32_t lane_off = (uint32_t)(q * 32) << 16;
    const uint32_t t_s = tmem + TM_S0 + a * 128 + hh * 64 + lane_off;
    const uint32_t t_p = tmem + TM_P0 + a * 64 + hh * 32 + lane_off;
    const uint32_t t_o = tmem + TM_O0 + a * 64 + hh * 32 + lane_off;
    // Opaque copies: left to itself the compiler re-derives the barrier addresses (S2UR %cluster_ctarank / shared-window
    // base, align, add) and the TMEM addresses (S2R %tid, shifts) at every use inside the tile loop — ~100 of its ~330
    // instructions per tile, several of them long-latency special-register reads on the stream's serial chain.
    uint32_t bar_sfull = B.sfull(a), bar_sempty = B.sempty(a), bar_pfull = B.pfull(a), bar_pvdone = B.pvdone(a);
    uint32_t ts_ = t_s, tp_ = t_p, lane0 = lane == 0;
    int col0 = hh * 64;                                  // first token column of this thread inside a KV tile
    asm volatile("" : "+r"(bar_sfull), "+r"(bar_sempty), "+r"(bar_pfull), "+r"(bar_pvdone), "+r"(ts_), "+r"(tp_), "+r"(lane0), "+r"(col0));
    uint32_t sfull_ph = 0, pv_ph = 0;
    long long tk0 = 0, tk[6] = {0, 0, 0, 0, 0, 0};
#define HY3D_TICK(i) if constexpr (kTimers) { const long long t_ = clock64(); tk[i] += t_ - tk0; tk0 = t_; }
    for (int item = blockIdx.x; item < nitems; item += gridDim.x) {
      const AttnItem wi = attn_item(g, item, a);
      const int qt = wi.qt, h = wi.h;
      const int ntok = g.group_ntok ? g.group_ntok[g.tile_group ? g.tile_group[qt] - g.group_base : 0] : g.ntok;
      uint64_t l2 = 0ull;                                // packed (even columns, odd columns) row sums: one FADD2 per pair
      const float cshift = g.head_shift ? g.head_shift[h] : 0.f;       // 0 unless the head's measured score bound exceeds 15.9
      const uint64_t cshift2 = pack_f2(cshift, cshift);
      if constexpr (kTimers) tk0 = clock64();
      // Every barrier round trip of these warps queues behind the MUFU instructions already in the SM's MIO pipe (the
      // kernel's bottleneck): a wait costs ~450 clk even when the barrier completed long ago (instrumented: wait S 497,
      // wait PV 482 clk per tile of 2840).  So the two MMA-completion barriers are PROBED in the middle of the
      // exponentials — the probes travel in the shadow of that work — and the blocking waits run only if a probe failed.
      bool s_ready = false;                              // S(j) already known complete
      for (int j = 0; j < nkv; ++j) {
        if (!s_ready) mbar_wait(bar_sfull, sfull_ph);
        sfull_ph ^= 1;
        fence_after_sync();
        HY3D_TICK(0)
        // software pipeline over the two 32-column halves of this thread's 64 scores: the second tcgen05.ld is in flight
        // while the first half's exponentials run (one TMEM round trip per tile off the stream's serial chain)
        uint32_t sv[64];
        HY3D_TMEM_LD32(ts_, sv);
        if (g.no_pipe) {                                 // (experiment bit 0x200: both halves up front, S released before any exponential)
          HY3D_TMEM_LD32(ts_ + 32, (sv + 32)); tmem_wait_ld();
          fence_before_sync();
          __syncwarp();
          if (lane0) mbar_arrive(bar_sempty);
        } else { tmem_wait_ld(); HY3D_TMEM_LD32(ts_ + 32, (sv + 32)); }
        HY3D_TICK(1)
        const int valid = ntok - j * 128 - col0;     // columns >= valid are padding tokens (last tile of a ragged count)
        bool pv_ok = j == 0, s_ok = false;
        if (cshift != 0.f) {                           // (warp-uniform) s - c_h: one FADD2 per pair, only for heads that need it
#pragma unroll
          for (int i = 0; i < 16; ++i) {
            float x0, x1;
            unpack_f2(sub_f2(pack_f2(__uint_as_float(sv[2 * i]), __uint_as_float(sv[2 * i + 1])), cshift2), x0, x1);
            sv[2 * i] = __float_as_uint(x0); sv[2 * i + 1] = __float_as_uint(x1);
          }
        }
        auto exp_pairs = [&](int i0, int i1) {         // in place: sv[i] <- packed (p[2i], p[2i+1])
          if (valid >= 64) {
#pragma unroll
            for (int i = i0; i < i1; ++i) {
              if (i == 24) {                           // probes: PV(j-1) consumed the previous P?  S(j+1) computed?
                if (j > 0) pv_ok = mbar_test_wait(bar_pvdone, pv_ph);
                if (j + 1 < nkv) s_ok = mbar_test_wait(bar_sfull, sfull_ph);
              }
              const float x0 = __uint_as_float(sv[2 * i]), x1 = __uint_as_float(sv[2 * i + 1]);
              float p0, p1;
              if (pair_on_fma<kPoly>(i)) exp2_poly2(x0, x1, p0, p1);
              else { p0 = ex2(x0); p1 = ex2(x1); }
              l2 = add_f2(l2, pack_f2(p0, p1));
              sv[i] = pack_h2(p0, p1);
            }
          } else {                                     // ragged last tile: padding columns contribute p = 0
#pragma unroll
            for (int i = i0; i < i1; ++i) {
              const float p0 = 2 * i < valid ? ex2(__uint_as_float(sv[2 * i])) : 0.f;
              const float p1 = 2 * i + 1 < valid ? ex2(__uint_as_float(sv[2 * i + 1])) : 0.f;
              l2 = add_f2(l2, pack_f2(p0, p1));
              sv[i] = pack_h2(p0, p1);
            }
          }
        };
        exp_pairs(0, 16);
        if (!g.no_pipe) {
          HY3D_TMEM_WAIT_LD32((sv + 32));              // second half has landed (tied to its registers)
          fence_before_sync();
          __syncwarp();
          if (lane0) mbar_arrive(bar_sempty);          // S is in registers: the next S MMA may overwrite it
        }
        if (cshift != 0.f) {
#pragma unroll
          for (int i = 16; i < 32; ++i) {
            float x0, x1;
            unpack_f2(sub_f2(pack_f2(__uint_as_float(sv[2 * i]), __uint_as_float(sv[2 * i + 1])), cshift2), x0, x1);
            sv[2 * i] = __float_as_uint(x0); sv[2 * i + 1] = __float_as_uint(x1);
          }
        }
        exp_pairs(16, 32);
        HY3D_TICK(2)
        if (j > 0) { if (!pv_ok) mbar_wait(bar_pvdone, pv_ph); pv_ph ^= 1; }   // PV(j-1) has consumed the previous P
        s_ready = s_ok;
        HY3D_TICK(3)
        HY3D_TMEM_ST32(tp_, sv);
        tmem_wait_st();
        fence_before_sync();
        __syncwarp();
        if (lane0) mbar_arrive(bar_pfull);
        HY3D_TICK(4)
      }
      // ---- finalize: row sums of the two column halves through shared memory, O / l -> fp16 tile (q-tile, head) ----
      float* ls = lsum + a * 256;
      { float l0, l1; unpack_f2(l2, l0, l1); ls[hh * 128 + r] = l0 + l1; }
      asm volatile("bar.sync %0, 256;" ::"r"(1 + a) : "memory");
      const float lrow = ls[r] + ls[128 + r];
      const float inv = 1.f / lrow;
      if (g.redo_count && cshift != 0.f && lrow < (float)ntok * 0x1p-14f && hh == 0) {
        // fp16 probabilities below 2^-14 are subnormal (absolute error up to 2^-25 each): with ntok of them the row sum is
        // only guaranteed to 2^-11 relative (the precision of a normal fp16 term) while it stays above ntok * 2^-14.  Rows
        // below that — every score far under the head's bound — are recomputed exactly: flag the (tile, head pair)
        const int e = qt * (g.H >> 1) + (h >> 1);
        if (atomicExch(&g.redo_flag[e], 1) == 0) g.redo_list[atomicAdd(g.redo_count, 1)] = e;
      }
      mbar_wait(bar_pvdone, pv_ph); pv_ph ^= 1;
      fence_after_sync();
      uint8_t* tile = g.O + ((size_t)qt * (g.split_out ? 3 : 1) * g.H + h) * TILE_BYTES;
      {
        uint32_t ov[32];
        HY3D_TMEM_LD32(t_o, ov);
        tmem_wait_ld();
        float x[32];
#pragma unroll
        for (int i = 0; i < 32; ++i) x[i] = __uint_as_float(ov[i]) * inv;
        if (!wi.store) {
          // duplicate of the last query tile (odd tile count in share_kv mode): computed, not stored
        } else if (g.split_out) {
#pragma unroll
          for (int c16 = 0; c16 < 4; ++c16)
            store_t16_split(tile, tile + (size_t)g.H * TILE_BYTES, tile + (size_t)2 * g.H * TILE_BYTES, r, hh * 4 + c16, x + 8 * c16);
        } else {
#pragma unroll
          for (int c16 = 0; c16 < 4; ++c16) store_t16_chunk(tile, r, hh * 4 + c16, x + 8 * c16);
        }
      }
      fence_before_sync();
      asm volatile("bar.sync %0, 256;" ::"r"(1 + a) : "memory");   // ls[] is reused by the next item
      HY3D_TICK(5)
      if constexpr (kTimers) {
        if (g.timers && lane == 0 && q == 0 && hh == 0 && blockIdx.x == 0) {
#pragma unroll
          for (int i = 0; i < 6; ++i) { atomicAdd(&g.timers[a * 8 + i], (unsigned long long)tk[i]); tk[i] = 0; }
          atomicAdd(&g.timers[a * 8 + 7], (unsigned long long)nkv);
        }
      }
    }
#undef HY3D_TICK
  }
  fence_before_sync();
  __syncthreads();
  if (warp == 2) tmem_dealloc(tmem, 512);
}

// ------------------------------------------------------------------------------------------
// General case: online softmax with a running maximum (decoders without q/k norm, norm gains beyond the shift range, and
// the exact redo pass of the bounded-score kernel).  Same thread layout as k_attn_fast: two threads per query row, each
// owning 64 of the 128 key columns of a KV tile (16 softmax warps instead of round 1's 8: twice the warps to hide the
// TMEM / MUFU latencies).  The two halves of a row agree on the running maximum through shared memory once per tile
// (double-buffered by tile parity, one 256-thread named barrier per stream), so they take the same lazy-rescale
// decisions and feed ONE P tile / O accumulator.
// ------------------------------------------------------------------------------------------
template <int kPoly>
__global__ void __launch_bounds__(ATT_THREADS, 1) k_attn_tc(AttnTC g) {
  constexpr float kLazy = 8.f;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  AttnBars B;
  const uint32_t tmem = attn_setup(smem, B, 8, g.share_kv);
  float* lsum = reinterpret_cast<float*>(smem + ATT_TILES_BYTES + 512);   // [2 streams][2 halves][128 rows] row sums (finalize)
  float* mxs = lsum + 512;                                                // [2 parities][2 streams][2 halves][128 rows] tile maxima
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nitems = attn_num_items(g), nkv = g.nkv;

  if (warp < 4) {
    reg_dealloc<56>();
    if ((warp & 1) == 0) { if (!g.share_kv || warp == 0) attn_producer(g, B, smem, warp >> 1); }
    else attn_mma(g, B, smem, tmem, warp >> 1);
  } else {
    reg_alloc<104>();
    const int a = (warp - 4) >> 3;                      // head stream
    const int hh = ((warp - 4) >> 2) & 1;               // column half: tokens [64 hh, 64 hh + 64) of every KV tile
    const int q = warp & 3;                             // TMEM lane quadrant
    const int r = q * 32 + lane;                        // query row
    const uint32_t lane_off = (uint32_t)(q * 32) << 16;
    uint32_t bar_sfull = B.sfull(a), bar_sempty = B.sempty(a), bar_pfull = B.pfull(a), bar_pvdone = B.pvdone(a);
    uint32_t ts_ = tmem + TM_S0 + a * 128 + hh * 64 + lane_off, tp_ = tmem + TM_P0 + a * 64 + hh * 32 + lane_off;
    uint32_t to_ = tmem + TM_O0 + a * 64 + hh * 32 + lane_off, lane0 = lane == 0;
    int col0 = hh * 64;
    float* mine = mxs + (a * 2 + hh) * 128 + r;         // + parity * 512
    float* other = mxs + (a * 2 + (hh ^ 1)) * 128 + r;
    asm volatile("" : "+r"(bar_sfull), "+r"(bar_sempty), "+r"(bar_pfull), "+r"(bar_pvdone), "+r"(ts_), "+r"(tp_), "+r"(to_), "+r"(lane0), "+r"(col0));   // opaque copies, see k_attn_fast
    uint32_t sfull_ph = 0, pv_ph = 0;
    for (int item = blockIdx.x; item < nitems; item += gridDim.x) {
      const AttnItem wi = attn_item(g, item, a);
      const int qt = wi.qt, h = wi.h;
      const int ntok = g.group_ntok ? g.group_ntok[g.tile_group ? g.tile_group[qt] - g.group_base : 0] : g.ntok;
      float m = -INFINITY;
      uint64_t l2 = 0ull;                               // packed (even, odd column) partial row sums of this half
      for (int j = 0; j < nkv; ++j) {
        mbar_wait(bar_sfull, sfull_ph); sfull_ph ^= 1;
        fence_after_sync();
        uint32_t sv[64];
        HY3D_TMEM_LD32(ts_, sv); HY3D_TMEM_LD32(ts_ + 32, (sv + 32));
        tmem_wait_ld();
        fence_before_sync();
        __syncwarp();
        if (lane0) mbar_arrive(bar_sempty);
        const int valid = ntok - j * 128 - col0;        // columns >= valid are padding tokens
        if (valid < 64) {                               // only the last tile of a ragged token count
#pragma unroll
          for (int i = 0; i < 64; ++i)
            if (i >= valid) sv[i] = 0xff800000u;        // -inf
        }
        float mx4[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};   // 4 independent max chains (3-input FMNMX)
#pragma unroll
        for (int i = 0; i < 64; i += 8) {
#pragma unroll
          for (int u = 0; u < 4; ++u)
            mx4[u] = fmaxf(mx4[u], fmaxf(__uint_as_float(sv[i + 2 * u]), __uint_as_float(sv[i + 2 * u + 1])));
        }
        float mx = fmaxf(fmaxf(mx4[0], mx4[1]), fmaxf(mx4[2], mx4[3]));
        // the other half's maximum of this tile (slot = tile parity: a slot is rewritten only two barriers later)
        mine[(j & 1) * 512] = mx;
        asm volatile("bar.sync %0, 256;" ::"r"(1 + a) : "memory");
        mx = fmaxf(mx, other[(j & 1) * 512]);
        bool need = false;
        float m_new = m;
        if (j == 0) { m_new = mx; }
        else if (mx > m + kLazy) { m_new = mx; need = true; }   // lazy rescale: keep the old max while p <= 2^kLazy
        // PV(j-1) must be complete before O is rescaled or the single P buffer is overwritten.  The rescale is rare (lazy
        // threshold): normally the wait is deferred until this tile's probabilities sit packed in registers.
        bool waited = (j == 0);
        if (j > 0 && __any_sync(0xffffffffu, need)) {    // both halves of these 32 rows see the same row maxima: same decision
          mbar_wait(bar_pvdone, pv_ph); pv_ph ^= 1; waited = true;
          fence_after_sync();
          const float sc = need ? ex2(m - m_new) : 1.f;
          { float l0, l1; unpack_f2(l2, l0, l1); l2 = pack_f2(l0 * sc, l1 * sc); }
          uint32_t ov[32];
          HY3D_TMEM_LD32(to_, ov);
          tmem_wait_ld();
#pragma unroll
          for (int i = 0; i < 32; ++i) ov[i] = __float_as_uint(__uint_as_float(ov[i]) * sc);
          HY3D_TMEM_ST32(to_, ov);
          tmem_wait_st();
        }
        m = m_new;
        const uint64_t m2 = pack_f2(m, m);
#pragma unroll
        for (int i = 0; i < 32; ++i) {                       // in place: sv[i] <- packed (p[2i], p[2i+1])
          float x0, x1;
          unpack_f2(sub_f2(pack_f2(__uint_as_float(sv[2 * i]), __uint_as_float(sv[2 * i + 1])), m2), x0, x1);
          float p0, p1;
          if (pair_on_fma<kPoly>(i)) exp2_poly2(fmaxf(x0, -126.f), fmaxf(x1, -126.f), p0, p1);   // (x - m can be -inf: clamp first)
          else { p0 = ex2(x0); p1 = ex2(x1); }
          l2 = add_f2(l2, pack_f2(p0, p1));
          sv[i] = pack_h2(p0, p1);
        }
        if (!waited) { mbar_wait(bar_pvdone, pv_ph); pv_ph ^= 1; }
        HY3D_TMEM_ST32(tp_, sv);
        tmem_wait_st();
        fence_before_sync();
        __syncwarp();
        if (lane0) mbar_arrive(bar_pfull);
      }
      // ---- finalize: row sums of the two halves through shared memory, O / l -> fp16 tile (q-tile, head) ----
      float* ls = lsum + a * 256;
      { float l0, l1; unpack_f2(l2, l0, l1); ls[hh * 128 + r] = l0 + l1; }
      asm volatile("bar.sync %0, 256;" ::"r"(1 + a) : "memory");
      const float inv = 1.f / (ls[r] + ls[128 + r]);
      mbar_wait(bar_pvdone, pv_ph); pv_ph ^= 1;
      fence_after_sync();
      uint8_t* tile = g.O + ((size_t)qt * (g.split_out ? 3 : 1) * g.H + h) * TILE_BYTES;
      {
        uint32_t ov[32];
        HY3D_TMEM_LD32(to_, ov);
        tmem_wait_ld();
        float x[32];
#pragma unroll
        for (int i = 0; i < 32; ++i) x[i] = __uint_as_float(ov[i]) * inv;
        if (!wi.store) {
        } else if (g.split_out) {
#pragma unroll
          for (int c16 = 0; c16 < 4; ++c16)
            store_t16_split(tile, tile + (size_t)g.H * TILE_BYTES, tile + (size_t)2 * g.H * TILE_BYTES, r, hh * 4 + c16, x + 8 * c16);
        } else {
#pragma unroll
          for (int c16 = 0; c16 < 4; ++c16) store_t16_chunk(tile, r, hh * 4 + c16, x + 8 * c16);
        }
      }
      fence_before_sync();
      asm volatile("bar.sync %0, 256;" ::"r"(1 + a) : "memory");   // ls[] / mxs[] are reused by the next item
    }
  }
  fence_before_sync();
  __syncthreads();
  if (warp == 2) tmem_dealloc(tmem, 512);
}
