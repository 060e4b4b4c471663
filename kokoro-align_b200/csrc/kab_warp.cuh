// kab_warp.cuh -- one WARP per lattice, for the silence-split short segments of BASELINE
// config 2 (S = 2L+1 <= 248, window never clips: lo_i = 0, hi_i = S for every frame,
// max_move = 4, labels in 1..V-1, V <= 512).
//
//   * state row lives in registers: lane l >= 1 owns states K*(l-1) .. K*l-1 (K = 2,4,6,8 even,
//     so even register index == blank state; lane 0 is an all -inf dummy that feeds lane 1's
//     halo); the three halo scores come from lane l-1 by warp shuffle -- no shared-memory round
//     trip and no block barrier on the recurrence.  Hence S <= 31*K <= 248.
//   * emission rows (V floats per frame) are staged a few frames ahead into a per-warp
//     shared-memory ring with 1-D bulk copies (cp.async.bulk + mbarrier complete_tx); the
//     per-state emission is a conflict-free LDS gather row[col[v]] (V = 39 spans 1.2 bank rows).
//     V = 39 (the reference's vocabulary, encoder.py:11) is a compile-time constant of the
//     fast instantiation so that the gathers of a frame group use immediate offsets.
//   * the finiteness check of the log-probs runs once per staged chunk with LDS.128.
//   * Kokoro-Align recurrence, K = 6 and 8: the forward pass computes VALUES ONLY (maximum before the add,
//     DESIGN.md 2) and every KAB_CKPT_C frames stores the score row as a checkpoint row
//     (kab_ckpt_stride floats, state order).  The backtrack then walks blocks of C frames from the
//     last one back: the block's moves depend only on the 3C+1 checkpoint states below the path
//     state at its last frame (one state per lane), so the warp restages the block's emission rows,
//     recomputes its C frames on that window with the post-add selects (2-bit codes in a register)
//     and walks them by shuffle.  best_scores comes from the restaged rows.
//   * CTC forced alignment (torchaudio's select is not a maximum) and Kokoro-Align K = 2 and 4
//     (their forward pass is cheap, the checkpoint backtrack would cost more): frames are processed in groups
//     of FPW = 32/BPF frames, one 32-bit word of 2-bit backpointers per lane and group, stored as
//     one coalesced 128-byte row per warp (word (i / FPW) * 32 + lane), and the same warp walks
//     them back, fetching the owner lane's word with a shuffle.
//   * warps pull lattices from a global queue sorted by decreasing cost (LPT order).
#pragma once
#include "kab_common.cuh"

#define KAB_WARP_STAGES 3
#define KAB_WARPS_PER_CTA 4
#ifndef KAB_WARP_MINBLOCKS
#define KAB_WARP_MINBLOCKS 6  // resident CTAs per SM (24 warps, <= 80 registers): the checkpoint backtrack
                              // is a one-state-per-lane chain of shuffles, and the sixth CTA hides its
                              // latency (DESIGN.md 3.1); the backpointer kernel measured best at 5
#endif

#define KAB_CKPT_C 8  // frames per checkpoint block: the backtrack's window of 3C+1 states must fit one warp
                     // (C <= 10); 8 divides every stage size (8, 16, 32 frames), so blocks never straddle stages

// Floats per checkpoint row: every lane that owns a state < S stores all K of its states.
__host__ __device__ inline int kab_ckpt_stride(int S, int K) { return (K * ((S + K - 1) / K) + 3) & ~3; }

template <int K>
struct KabWarpCfg {  // (backpointer scheme)
  static constexpr int BPF = K <= 2 ? 4 : (K <= 4 ? 8 : 16);  // backpointer bits per lane per frame
  static constexpr int FPW = 32 / BPF;                        // frames per 32-bit word
};

// One values-only frame for this lane's K states: s[] holds frame i-1 on entry and frame i on return.
// Each state takes the maximum of its masked predecessors and then ONE add (fl(max_j x_j + e) ==
// max_j fl(x_j + e), DESIGN.md 2); blank and label state of a pair share one packed add.
// Lane 0 is a dummy whose states are permanently -inf ("states -K..-1"), so the halo of lane 1
// (state 0's lower neighbours) is -inf without any select.
template <int K, bool MM>
__device__ __forceinline__ void kab_warp_frame(float (&s)[K], const float eb, const float (&el)[K / 2],
                                               const bool lane1, const float mm1, const float mm2, const float mm3) {
  float h1, h2, h3;  // previous-frame scores of states K*(lane-1)-1, -2, -3
  if (K >= 4) {
    h1 = __shfl_up_sync(KAB_FULL_MASK, s[K - 1], 1);
    h2 = __shfl_up_sync(KAB_FULL_MASK, s[K - 2], 1);
    h3 = __shfl_up_sync(KAB_FULL_MASK, s[K >= 4 ? K - 3 : 0], 1);
  } else {
    h1 = __shfl_up_sync(KAB_FULL_MASK, s[1], 1);
    h2 = __shfl_up_sync(KAB_FULL_MASK, s[0], 1);
    h3 = __shfl_up_sync(KAB_FULL_MASK, s[1], 2);
    h3 = lane1 ? kab_neg_inf() : h3;  // lane 1: two lanes up is out of range
  }
  float n[K];
#pragma unroll
  for (int q = 0; q < K / 2; ++q) {
    const int kb = 2 * q, kl = 2 * q + 1;
    // blank state kb: moves 0, 1, 3
    const float b1 = kb >= 1 ? s[kb >= 1 ? kb - 1 : 0] : h1;
    const float b3 = kb >= 3 ? s[kb >= 3 ? kb - 3 : 0] : (kb == 2 ? h1 : h3);
    const float mb = kab_max3(s[kb], kab_mm<MM>(b1, mm1), kab_mm<MM>(b3, mm3));
    // label state kl: moves 0..3
    const float l2 = q >= 1 ? s[q >= 1 ? kl - 2 : 0] : h1;
    const float l3 = q >= 1 ? s[q >= 1 ? kl - 3 : 0] : h2;
    const float ml = kab_max3(kab_max2(s[kl], kab_mm<MM>(s[kl - 1], mm1)), kab_mm<MM>(l2, mm2), kab_mm<MM>(l3, mm3));
    kab_add2v(mb, ml, eb, el[q], n[kb], n[kl]);
  }
#pragma unroll
  for (int k = 0; k < K; ++k) s[k] = n[k];
}

// Backpointer frame (K <= 4 lattices, see kab_warp_align): one frame for this lane's K states;
// the frame's 2K backpointer bits are OR-ed into w at
// bits [shift, shift + 2K).  s[] holds frame i-1 on entry and frame i on return.
// Lane 0 is a dummy whose states are permanently -inf ("states -K..-1"), so the halo of lane 1
// (state 0's lower neighbours) is -inf without any select.
template <int K, bool MM>
__device__ __forceinline__ void kab_warp_frame_bp(float (&s)[K], const float eb, const float (&el)[K / 2],
                                               const bool lane1, uint32_t &w, const int shift,
                                                  const uint32_t one, const float mm1, const float mm2, const float mm3) {
  float h1, h2, h3;  // previous-frame scores of states K*(lane-1)-1, -2, -3
  if (K >= 4) {
    h1 = __shfl_up_sync(KAB_FULL_MASK, s[K - 1], 1);
    h2 = __shfl_up_sync(KAB_FULL_MASK, s[K - 2], 1);
    h3 = __shfl_up_sync(KAB_FULL_MASK, s[K >= 4 ? K - 3 : 0], 1);
  } else {
    h1 = __shfl_up_sync(KAB_FULL_MASK, s[1], 1);
    h2 = __shfl_up_sync(KAB_FULL_MASK, s[0], 1);
    h3 = __shfl_up_sync(KAB_FULL_MASK, s[1], 2);
    h3 = lane1 ? kab_neg_inf() : h3;  // lane 1: two lanes up is out of range
  }
  // blank candidates: t[j] = s[j] + eb for every state (even, odd) pair, plus the halo
  float t[K];
#pragma unroll
  for (int m = 0; m < K / 2; ++m) kab_add2(s[2 * m], s[2 * m + 1], eb, t[2 * m], t[2 * m + 1]);
  const float th1 = __fadd_rn(h1, eb), th3 = __fadd_rn(h3, eb);
  float n[K];
#pragma unroll
  for (int q = 0; q < K / 2; ++q) {
    const int kb = 2 * q, kl = 2 * q + 1;
    // blank state kb: moves 0, 1, 3
    const float b1 = kb >= 1 ? t[kb >= 1 ? kb - 1 : 0] : th1;
    const float b3 = kb >= 3 ? t[kb >= 3 ? kb - 3 : 0] : (kb == 2 ? th1 : th3);
    n[kb] = kab_blank_sel(t[kb], kab_mm<MM>(b1, mm1), kab_mm<MM>(b3, mm3), w, 1u << (shift + 2 * kb), 2u << (shift + 2 * kb), one);
    // label state kl: moves 0..3 = states (kl, kl-1) and (kl-2, kl-3), both (even, odd) pairs
    float a0, a1, a2, a3;
    kab_add2(s[kl - 1], s[kl], el[q], a1, a0);
    if (q >= 1) kab_add2(s[q >= 1 ? kl - 3 : 0], s[q >= 1 ? kl - 2 : 0], el[q], a3, a2);
    else kab_add2(h2, h1, el[q], a3, a2);
    n[kl] = kab_label_sel(a0, kab_mm<MM>(a1, mm1), kab_mm<MM>(a2, mm2), kab_mm<MM>(a3, mm3), w, 1u << (shift + 2 * kl), 2u << (shift + 2 * kl), one);
  }
#pragma unroll
  for (int k = 0; k < K; ++k) s[k] = n[k];
}

// This lane's K states of one checkpoint row (lanes >= 1 whose first state is < S).
template <int K>
__device__ __forceinline__ void kab_ckpt_store(float *row, const float (&s)[K]) {
  if (K % 4 == 0) {
#pragma unroll
    for (int k = 0; k < K; k += 4)
      __stcg(reinterpret_cast<float4 *>(row + k), make_float4(s[k], s[k + 1], s[k + 2], s[k + 3]));
  } else {
#pragma unroll
    for (int k = 0; k < K; k += 2) __stcg(reinterpret_cast<float2 *>(row + k), make_float2(s[k], s[k + 1]));
  }
}

// CTC forced alignment (kab_common.cuh): lane l >= 1 owns the same K states; the only halo is state
// K*(l-1)-1 (moves reach two states down, and state v-2 of a label state v is inside the lane for
// v >= 3 of the lane).  rep bit q = move 2 is forbidden into the lane's label state 2q+1.
// FREE (free-ends plans): lane 1's halo is the virtual state -1, score 0 in every frame.
template <int K, bool FREE>
__device__ __forceinline__ void kab_warp_frame_ctc(float (&s)[K], const float eb, const float (&el)[K / 2],
                                                   const uint32_t rep, uint32_t &w, const int shift, const bool lane1) {
  float h1 = __shfl_up_sync(KAB_FULL_MASK, s[K - 1], 1);
  if (FREE && lane1) h1 = 0.0f;
  float n[K];
#pragma unroll
  for (int q = 0; q < K / 2; ++q) {
    const int kb = 2 * q, kl = 2 * q + 1;
    n[kb] = __fadd_rn(kab_ctc_blank_sel(s[kb], kb >= 1 ? s[kb >= 1 ? kb - 1 : 0] : h1, w, shift + 2 * kb), eb);
    const float x2 = (rep >> q) & 1u ? kab_neg_inf() : (kl >= 3 ? s[kl >= 3 ? kl - 2 : 0] : h1);
    n[kl] = __fadd_rn(kab_ctc_label_sel(s[kl], s[kl - 1], x2, w, shift + 2 * kl), el[q]);
  }
#pragma unroll
  for (int k = 0; k < K; ++k) s[k] = n[k];
}

// VCT: compile-time vocabulary (39) or 0 = runtime p.V.  CTC: the CTC forced-alignment recurrence.
// FREE: CTC with free ends (kab_plan_create_ctc_free): a virtual state -1 of score 0 below state 0 in every
// frame, running (score, frame) maxima of the end states S-1 and S-2 (>=: the later frame), the walk starts
// at the chosen end (t1, v) and stops at state -1; frames outside [t0, t1] get state -1 and the blank.
template <int K, int VCT, bool MM, bool CTC, bool FREE = false>
__device__ void kab_warp_align(const KabLattice &lat, const KabParams &p, float *stage_base, uint64_t *bars,
                               uint16_t *labtab, const uint64_t policy, uint32_t &chunk_counter, const int lane,
                               const int blank) {
  using Cfg = KabWarpCfg<K>;
  constexpr int BPF = Cfg::BPF, FPW = Cfg::FPW;
  constexpr int C = KAB_CKPT_C;
  // Backpointer scheme for CTC (its select is not a maximum) and for K <= 4, whose forward pass is
  // cheap enough that the checkpoint backtrack costs more than it saves (DESIGN.md 3.1).
  constexpr bool BP = CTC || K <= 4;
  const int T = lat.T, S = 2 * lat.L + 1;
  const int V = VCT ? VCT : p.V;
  const int F = p.stage_frames;  // multiple of 8 (host guarantees), so groups and blocks never straddle chunks
  const uint32_t stage_words = p.stage_bytes >> 2;
  const int n_chunks = (T + F - 1) / F;
  const uint16_t *col16 = p.col16 + lat.col_off;
  uint32_t *bpw = reinterpret_cast<uint32_t *>(p.bp + lat.bp_off);   // BP: backpointer words
  float *ck = reinterpret_cast<float *>(p.bp + lat.bp_off);          // !BP: checkpoint rows
  const int RS = kab_ckpt_stride(S, K);
  const bool lane0 = lane == 0, lane1 = lane == 1;
  const uint32_t one = p.one;  // runtime 1 (see kab_blank_sel)
  const float mm1 = p.mm1, mm2 = p.mm2, mm3 = p.mm3;
  const int sbase = K * (lane - 1);  // first state of this lane (lane 0: dummy, all -inf)

  // byte offsets (col * 4) of this lane's K/2 label states inside an emission row
  uint32_t coff[K / 2];
  uint32_t rep = 0;  // CTC: bit q = move 2 forbidden into label state sbase + 2q + 1 (v == 1, or a repeated label)
#pragma unroll
  for (int q = 0; q < K / 2; ++q) {
    const int v = sbase + 2 * q + 1;
    const uint32_t col = (v > 0 && v < S) ? col16[(v - 1) >> 1] : 0u;
    coff[q] = 4u * col;
    if (v > 0 && v < S) labtab[(v - 1) >> 1] = (uint16_t)col;  // per-warp copy for the backtrack's output rows
    // (FREE: state 1 takes move 2 from the virtual state -1, and has no label below to repeat)
    if (CTC && (FREE ? v < 1 || v >= S || (v >= 3 && col == col16[(v - 3) >> 1])
                     : v < 3 || v >= S || col == col16[(v - 3) >> 1])) rep |= 1u << q;
  }
  const uint32_t boff = CTC ? 4u * (uint32_t)blank : 0u;  // byte offset of the blank's column

  float s[K];
#pragma unroll
  for (int k = 0; k < K; ++k) s[k] = kab_neg_inf();
  if (lane1 && !FREE) s[0] = 0.0f;  // virtual start state 0, score 0 (align.py:57-58)
  // FREE: running maxima (score, frame) of the end states in their owner lanes: register k1e holds state
  // S-1 there (an even state, so an even register), k2e state S-2 (odd)
  const int k1e = (S - 1) % K, k2e = (S - 2) % K;
  float m1 = kab_neg_inf(), m2 = kab_neg_inf();
  int f1 = T - 1, f2 = T - 1;
  auto track_end = [&](const int t) {
    float e1 = s[0], e2 = s[1];
#pragma unroll
    for (int k = 2; k < K; k += 2) if (k == k1e) e1 = s[k];
#pragma unroll
    for (int k = 3; k < K; k += 2) if (k == k2e) e2 = s[k];
    if (e1 >= m1) { m1 = e1; f1 = t; }
    if (e2 >= m2) { m2 = e2; f2 = t; }
  };

  // -- emission pipeline: the k-th chunk issued uses stage (chunk_counter + k) % STAGES.  F * V * 4 is a multiple
  // of 16, so every chunk of the lattice has the same 16-byte skew and all but the last one are
  // plain aligned copies of `full_bytes`; only the last chunk goes through the clamping descriptor.
  const uint32_t cc0 = chunk_counter;
  const int64_t lat_b0 = lat.t_off * (int64_t)V * 4;
  const char *lp_base = reinterpret_cast<const char *>(p.lp) + (lat_b0 & ~(int64_t)15);
  const int w0 = (int)((lat_b0 & 15) >> 2);  // word index of a chunk's first value inside its stage
  const uint32_t chunk_stride = (uint32_t)(F * V * 4);
  const uint32_t full_bytes = (chunk_stride + (uint32_t)w0 * 4u + 15u) & ~15u;
  uint32_t ist = cc0 % KAB_WARP_STAGES;  // stage of the next chunk to issue
  auto issue = [&](int c) {
    float *dst = stage_base + ist * stage_words;
    if (c + 1 < n_chunks) {
      if (lane0) {
        kab_mbar_expect_tx(&bars[ist], full_bytes);
        kab_bulk_g2s_hint(dst, lp_base + (size_t)c * chunk_stride, full_bytes, &bars[ist], policy);
      }
    } else {
      const int f0 = c * F;
      const KabStageDesc d = kab_stage_desc(p, lat.t_off, f0, T - f0);
      if (lane0) {
        kab_mbar_expect_tx(&bars[ist], d.bytes);
        if (d.bytes) kab_bulk_g2s_hint(dst, d.src, d.bytes, &bars[ist], policy);
      }
      if (lane < (int)d.tail_n)  // last (< 16 B) words of the whole log_probs buffer
        dst[d.tail_word + lane] = __ldg(reinterpret_cast<const float *>(d.src) + d.tail_word + lane);
    }
    ist = ist + 1 == KAB_WARP_STAGES ? 0 : ist + 1;
  };
  const int pre = min(n_chunks, KAB_WARP_STAGES - 1);
  for (int c = 0; c < pre; ++c) issue(c);

  float poison = kab_poison_init<CTC>();  // NaN once a rejected log-prob was staged (kab_poison_t)
  uint32_t *bprow = bpw + lane;  // BP: this lane's slot in the current word-row
  float *ckrow = ck;             // !BP: the next checkpoint row
  uint32_t st = cc0 % KAB_WARP_STAGES, ph = (cc0 / KAB_WARP_STAGES) & 1u;  // stage / phase of the chunk being read
  for (int c = 0; c < n_chunks; ++c) {
    // the stage consumed in iteration c-1 is free again: refill it with chunk c + STAGES - 1
    __syncwarp();
    // (every LDS of that stage has completed: its values were consumed by the frame updates
    // this warp has already issued, so the bulk copy cannot overtake a pending read)
    if (c + KAB_WARP_STAGES - 1 < n_chunks) issue(c + KAB_WARP_STAGES - 1);
    kab_mbar_wait(&bars[st], ph);
    __syncwarp();
    const int nf = min(F, T - c * F);
    const float *stage = stage_base + st * stage_words;
    if (++st == KAB_WARP_STAGES) { st = 0; ph ^= 1u; }
    const int w1 = w0 + nf * V;
    {  // finiteness of exactly this lattice's words [w0, w1) of the stage
      const int v0 = (w0 + 3) >> 2, v1 = w1 >> 2;
      const float4 *s4 = reinterpret_cast<const float4 *>(stage);
      for (int j = v0 + lane; j < v1; j += 32) {
        const float4 x = s4[j];
        poison = kab_poison_t<CTC>(kab_poison_t<CTC>(kab_poison_t<CTC>(kab_poison_t<CTC>(poison, x.x), x.y), x.z), x.w);
      }
      if (lane < 4 * v0 - w0 && w0 + lane < w1) poison = kab_poison_t<CTC>(poison, stage[w0 + lane]);
      if (4 * v1 >= w0 && lane < w1 - 4 * v1) poison = kab_poison_t<CTC>(poison, stage[4 * v1 + lane]);
    }
    const char *rowb = reinterpret_cast<const char *>(stage + w0);
    if constexpr (BP) {  // groups of FPW frames, one word of 2-bit codes per lane and group
      const int n_groups = nf / FPW;
      for (int gi = 0; gi < n_groups; ++gi, rowb += FPW * V * 4) {
        uint32_t word = 0;
#pragma unroll
        for (int f = 0; f < FPW; ++f) {
          const char *rb = rowb + f * V * 4;
          const float eb = *reinterpret_cast<const float *>(rb + boff);
          float el[K / 2];
#pragma unroll
          for (int q = 0; q < K / 2; ++q) el[q] = *reinterpret_cast<const float *>(rb + coff[q]);
          if (CTC) kab_warp_frame_ctc<K, FREE>(s, eb, el, rep, word, f * BPF, lane1);
          else kab_warp_frame_bp<K, MM>(s, eb, el, lane1, word, f * BPF, one, mm1, mm2, mm3);
          if (FREE) track_end(c * F + gi * FPW + f);
        }
        *bprow = word;
        bprow += 32;
      }
      const int rem = nf - n_groups * FPW;  // only in the last chunk
      if (rem) {
        uint32_t word = 0;
#pragma unroll 1
        for (int f = 0; f < rem; ++f, rowb += V * 4) {
          const float eb = *reinterpret_cast<const float *>(rowb + boff);
          float el[K / 2];
#pragma unroll
          for (int q = 0; q < K / 2; ++q) el[q] = *reinterpret_cast<const float *>(rowb + coff[q]);
          uint32_t fw = 0;
          if (CTC) kab_warp_frame_ctc<K, FREE>(s, eb, el, rep, fw, 0, lane1);
          else kab_warp_frame_bp<K, MM>(s, eb, el, lane1, fw, 0, one, mm1, mm2, mm3);
          if (FREE) track_end(c * F + n_groups * FPW + f);
          word |= fw << (f * BPF);
        }
        *bprow = word;
      }
    } else {  // groups of C frames, values only, one checkpoint row per group
      const int n_groups = nf / C;
      for (int gi = 0; gi < n_groups; ++gi, rowb += C * V * 4) {
#pragma unroll
        for (int f = 0; f < C; ++f) {
          const char *rb = rowb + f * V * 4;
          const float eb = *reinterpret_cast<const float *>(rb);
          float el[K / 2];
#pragma unroll
          for (int q = 0; q < K / 2; ++q) el[q] = *reinterpret_cast<const float *>(rb + coff[q]);
          kab_warp_frame<K, MM>(s, eb, el, lane1, mm1, mm2, mm3);
        }
        if (!lane0 && sbase < S) kab_ckpt_store<K>(ckrow + sbase, s);  // scores after frame (row + 1) * C - 1
        ckrow += RS;
      }
      const int rem = nf - n_groups * C;  // only in the last chunk
#pragma unroll 1
      for (int f = 0; f < rem; ++f, rowb += V * 4) {
        const float eb = *reinterpret_cast<const float *>(rowb);
        float el[K / 2];
#pragma unroll
        for (int q = 0; q < K / 2; ++q) el[q] = *reinterpret_cast<const float *>(rowb + coff[q]);
        kab_warp_frame<K, MM>(s, eb, el, lane1, mm1, mm2, mm3);
      }
    }
  }
  chunk_counter = cc0 + n_chunks;
  __syncwarp();

  // score of state u of frame T-1 (from its owner lane)
  auto score_of = [&](int u) {
    float mine = s[0];
#pragma unroll
    for (int k = 1; k < K; ++k) if (k == u % K) mine = s[k];
    return __shfl_sync(KAB_FULL_MASK, mine, u / K + 1);
  };
  int v, t1 = T - 1;
  float fs_free = 0.0f;
  if (FREE) {  // free end: the larger maximum, on a tie the later frame, then S-2 (L = 0: no frame is inside)
    const int o1 = (S - 1) / K + 1, o2 = (S - 2) / K + 1;
    const float a1 = __shfl_sync(KAB_FULL_MASK, m1, o1), a2 = __shfl_sync(KAB_FULL_MASK, m2, o2);
    const int g1 = __shfl_sync(KAB_FULL_MASK, f1, o1), g2 = __shfl_sync(KAB_FULL_MASK, f2, o2);
    const bool top = a1 > a2 || (a1 == a2 && g1 > g2);
    v = top ? S - 1 : S - 2;
    t1 = top ? g1 : g2;
    fs_free = top ? a1 : a2;
    if (S == 1) { v = -1; t1 = -1; fs_free = 0.0f; }
  } else if (CTC) {  // CTC end rule: the better of the last two states, S-2 on a tie (kab_common.cuh)
    v = S - 1;
    if (S >= 2) {
      const float a1 = score_of(S - 1), a2 = score_of(S - 2);
      if (!(a1 > a2)) v = S - 2;
    }
  } else {  // -- forced end state: highest active state of frame T-1 (align.py:99-101)
    int cand = -1;
#pragma unroll
    for (int k = 0; k < K; ++k) {
      const int v = sbase + k;
      if (v >= 0 && v < S && s[k] > kab_neg_inf()) cand = v;
    }
    v = __reduce_max_sync(KAB_FULL_MASK, cand);
  }
  const bool any_bad = __any_sync(KAB_FULL_MASK, poison != poison);
  const int status = any_bad ? 3 : (v < 0 && !FREE ? 1 : 0);
  {
    float fs = __int_as_float(0x7fc00000);
    if (FREE) {
      if (status == 0) fs = fs_free;
    } else if (status == 0) {
      float mine = s[0];
#pragma unroll
      for (int k = 1; k < K; ++k) if (k == v % K) mine = s[k];
      fs = __shfl_sync(KAB_FULL_MASK, mine, v / K + 1);
    }
    if (lane0) {
      p.status[lat.index] = status;
      if (p.final_score) p.final_score[lat.index] = fs;
    }
  }
  if (status != 0) return;
  if constexpr (!BP) {
    // -- backtrack over checkpoint blocks (DESIGN.md 3.1).  Block b = frames [bC, bC + n), n = C except
    // for the last block.  ve = path state at the block's last frame; every path state of the block
    // and of frame bC - 1 is >= ve - 3n >= base = ve - 3C, so lane j recomputes state base + j from
    // checkpoint row b - 1 (frame -1: the virtual start).  Lanes j < 3 take their own value as halo
    // and states above ve are never read: a wrong value climbs at most 3 states per frame, the
    // cone of states the walk reads shrinks by 3 per frame, and the two never meet.
    int32_t *out_path = p.best_path + lat.t_off;
    int32_t *out_lab = p.best_labels + lat.t_off;
    float *out_sc = p.best_scores + lat.t_off;
    int ve = v;
    // states sb + lane (r0) and sb + 32 + lane (r1) of a checkpoint row, sb = ve - 63: a superset of
    // the next block's window, loaded one block ahead (its base is only known after the walk).  The
    // loads are unconditional (row and state clamped to 0, inside the slice); states < 0 and the
    // virtual start are applied where the window is taken, so nothing waits for the loads here.
    auto win_load = [&](int row, int sb, float &r0, float &r1) {
      const float *rp = ck + (size_t)max(row, 0) * RS;
      r0 = __ldcg(rp + max(sb + lane, 0));
      r1 = __ldcg(rp + max(sb + 32 + lane, 0));
    };
    int sb = ve - 63;
    float r0, r1;
    win_load((T - 1) / C - 1, sb, r0, r1);
    for (int k = 0; k < pre; ++k) issue(n_chunks - 1 - k);  // emission rows again, last chunk first
    for (int k = 0; k < n_chunks; ++k) {
      const int c = n_chunks - 1 - k;
      __syncwarp();
      if (k + KAB_WARP_STAGES - 1 < n_chunks) issue(c - (KAB_WARP_STAGES - 1));
      kab_mbar_wait(&bars[st], ph);
      __syncwarp();
      const int nf = min(F, T - c * F);
      const char *rows = reinterpret_cast<const char *>(stage_base + st * stage_words + w0);
      if (++st == KAB_WARP_STAGES) { st = 0; ph ^= 1u; }
      for (int bi = (nf - 1) / C; bi >= 0; --bi) {
        const int f0 = c * F + bi * C, n = min(C, nf - bi * C);
        const char *rb = rows + bi * C * V * 4;
        const int base = ve - 3 * C;
        const int wi = base + lane - sb;  // in [0, 64) for every lane <= 3C
        const float x0 = __shfl_sync(KAB_FULL_MASK, r0, wi & 31), x1 = __shfl_sync(KAB_FULL_MASK, r1, wi & 31);
        const int u = base + lane;
        float x = u < 0 ? kab_neg_inf() : (wi >= 32 ? x1 : x0);
        if (f0 == 0) x = u == 0 ? 0.0f : kab_neg_inf();  // frame -1: the virtual start (align.py:57-58)
        sb = ve - 63;
        win_load(f0 / C - 2, sb, r0, r1);
        const bool blank_lane = (u & 1) == 0;
        const uint32_t uoff = (u > 0 && u < S && !blank_lane) ? 4u * labtab[(u - 1) >> 1] : 0u;
        // recompute: one state per lane, today's post-add select (a blank state is a label state
        // whose move-2 candidate is -inf: same value, same code 0 / 1 / 3)
        uint32_t cw = 0;
#pragma unroll
        for (int j = 0; j < C; ++j) {
          const float e = *reinterpret_cast<const float *>(rb + j * V * 4 + uoff);
          const float h1 = __shfl_up_sync(KAB_FULL_MASK, x, 1);
          const float h2 = __shfl_up_sync(KAB_FULL_MASK, x, 2);
          const float h3 = __shfl_up_sync(KAB_FULL_MASK, x, 3);
          float a0, a1, a2, a3;
          kab_add2(x, h1, e, a0, a1);
          kab_add2(h2, h3, e, a2, a3);
          a2 = blank_lane ? kab_neg_inf() : kab_mm<MM>(a2, mm2);
          x = kab_label_sel(a0, kab_mm<MM>(a1, mm1), a2, kab_mm<MM>(a3, mm3), cw, 1u << (2 * j), 2u << (2 * j), one);
        }
        if (n < C) cw &= (1u << (2 * n)) - 1u;  // frames >= T (rows past the lattice): move 0
        // walk: frame j's code comes from the lane of the path state (wl = its offset from base) and
        // goes into mw, two bits per frame, from which every lane sums the moves above its own frame
        int wl = 3 * C;
        uint32_t mw = 0;
#pragma unroll
        for (int j = C - 1; j >= 0; --j) {
          const uint32_t w = __shfl_sync(KAB_FULL_MASK, cw, wl);
          mw |= w & (3u << (2 * j));
          wl -= (int)((w >> (2 * j)) & 3u);
        }
        const uint32_t above = mw >> min(2 * lane + 2, 2 * C);
        const int myv = ve - (__popc(above & 0x55555555u) + 2 * __popc(above & 0xaaaaaaaau));
        ve = base + wl;  // path state at frame f0 - 1
        if (lane < n) {  // frame f0 + lane: align.py:105-107
          const int lab = (myv & 1) ? (int)labtab[(myv - 1) >> 1] : 0;
          out_path[f0 + lane] = myv;
          out_lab[f0 + lane] = lab;
          out_sc[f0 + lane] = *reinterpret_cast<const float *>(rb + lane * V * 4 + lab * 4);
        }
      }
    }
    chunk_counter += n_chunks;
  } else {
    // -- backtrack (== flush_determined_path, align.py:21-40).  Word-rows are fetched four at a
    // time, one block ahead of the walk (coalesced 128-byte rows, from L2 when they are recent enough), the walk reads the owner lane's word by shuffle, and
    // every 32 frames the lanes flush one coalesced row of each output array.  The score gather
    // of a row is issued at its flush and stored at the next one, so its DRAM latency is hidden.
    constexpr int RB = 4;  // word-rows per block
    int32_t *out_path = p.best_path + lat.t_off;
    int32_t *out_lab = p.best_labels + lat.t_off;
    float *out_sc = p.best_scores + lat.t_off;
    const float *lp = p.lp + lat.t_off * (int64_t)V;
    const int n_rows = (T + FPW - 1) / FPW;
    auto fetch = [&](int rb, uint32_t (&w)[RB]) {
#pragma unroll
      for (int r = 0; r < RB; ++r)
        w[r] = (rb >= 0 && (rb + r) < n_rows) ? __ldcg(&bpw[(size_t)(rb + r) * 32 + lane]) : 0u;
    };
    // The walk keeps the state as (own1, k2) = (owner lane, 2 * index inside the lane) next to v,
    // so a frame costs one shuffle, one shift/mask and a few adds: the 2-bit code IS the move
    // (kab_decode_move).  Frames >= T of the last block have all-zero codes (moves 0), so the
    // block bodies need no bounds checks.
    // FREE: the walk is at state -1 (lane 0's register K-1, whose codes are all 0) until frame t1
    const int vend = v;
    if (FREE) v = -1;
    int myv = FREE ? -1 : 0, pend_t = -1;
    float pend_s = 0.0f;
    int own1 = FREE ? 0 : v / K + 1, k2 = FREE ? 2 * K - 2 : 2 * (v - (v / K) * K);
    uint32_t wr[RB], wn[RB];
    const int rb_last = ((n_rows - 1) / RB) * RB;
    fetch(rb_last, wr);
    for (int rb = rb_last; rb >= 0; rb -= RB) {
      fetch(rb - RB, wn);
      const int fb = rb * FPW;            // first frame of the block (a multiple of RB * FPW, which divides 32)
      const int lb = lane - (fb & 31);    // lane records frame fb + off iff lb == off
#pragma unroll
      for (int r = RB - 1; r >= 0; --r) {
#pragma unroll
        for (int f = FPW - 1; f >= 0; --f) {
          if (FREE && fb + r * FPW + f == t1) { v = vend; own1 = vend / K + 1; k2 = 2 * (vend % K); }
          const uint32_t w = __shfl_sync(KAB_FULL_MASK, wr[r], own1);
          if (lb == r * FPW + f) myv = v;
          const int mv = (int)((w >> (f * BPF + k2)) & 3u);
          v -= mv;
          k2 -= 2 * mv;
          if (k2 < 0) { k2 += 2 * K; --own1; }
          if (K == 2 && k2 < 0) { k2 += 2 * K; --own1; }  // a move of 3 can cross two 2-state lanes
        }
      }
      if ((fb & 31) == 0) {
        if (pend_t >= 0) out_sc[pend_t] = pend_s;  // gather issued one flush ago
        const int t = fb + lane;
        pend_t = -1;
        if (t < T) {
          const bool is_lab = FREE ? (myv & 1) && myv > 0 : (myv & 1);  // (FREE: -1 outside [t0, t1])
          const int lab = is_lab ? (int)labtab[(myv - 1) >> 1] : (CTC ? blank : 0);
          out_path[t] = myv;
          out_lab[t] = lab;                           // align.py:106
          pend_s = __ldg(&lp[(int64_t)t * V + lab]);  // align.py:107
          pend_t = t;
        }
      }
#pragma unroll
      for (int r = 0; r < RB; ++r) wr[r] = wn[r];
    }
    if (pend_t >= 0) out_sc[pend_t] = pend_s;
  }
}

template <int VCT, bool MM, bool CTC, bool FREE = false>
__device__ __forceinline__ void kab_warp_body(const KabLattice *__restrict__ lats, int n_lat, const KabParams &p,
                                              const int blank) {
  extern __shared__ __align__(128) unsigned char kab_smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  uint64_t *bars = reinterpret_cast<uint64_t *>(kab_smem) + warp * KAB_WARP_STAGES;
  float *stage_base = reinterpret_cast<float *>(kab_smem + 128 +
                                                (size_t)warp * KAB_WARP_STAGES * p.stage_bytes);
  uint16_t *labtab = reinterpret_cast<uint16_t *>(kab_smem + 128 +
                                                  (size_t)KAB_WARPS_PER_CTA * KAB_WARP_STAGES * p.stage_bytes) +
                     warp * 128;  // labels of the warp's current lattice (<= 124)
  // L2 policy of the emission loads: evict_normal.  The backtrack re-reads the rows right after the
  // forward pass, most recent rows first (restaged for the recomputation; CTC: one sector of every
  // row for best_scores), so a part of them is still in L2 (measured with the backpointer walk against
  // evict_first: DRAM reads 1.54 -> 1.46 GB, 0.518 -> 0.514 ms).
  uint64_t policy;
  asm volatile("createpolicy.fractional.L2::evict_normal.b64 %0, 1.0;" : "=l"(policy));
  if (lane == 0) {
    for (int s = 0; s < KAB_WARP_STAGES; ++s) kab_mbar_init(&bars[s], 1);
    kab_fence_mbar_init();
  }
  __syncwarp();
  uint32_t chunk_counter = 0;
  for (;;) {
    unsigned int item = 0;
    if (lane == 0) item = atomicAdd(p.queue, 1u);
    item = __shfl_sync(KAB_FULL_MASK, item, 0);
    if (item >= (unsigned int)n_lat) break;
    const KabLattice lat = lats[item];
    switch (lat.k) {
      case 2: kab_warp_align<2, VCT, MM, CTC, FREE>(lat, p, stage_base, bars, labtab, policy, chunk_counter, lane, blank); break;
      case 4: kab_warp_align<4, VCT, MM, CTC, FREE>(lat, p, stage_base, bars, labtab, policy, chunk_counter, lane, blank); break;
      case 6: kab_warp_align<6, VCT, MM, CTC, FREE>(lat, p, stage_base, bars, labtab, policy, chunk_counter, lane, blank); break;
      default: kab_warp_align<8, VCT, MM, CTC, FREE>(lat, p, stage_base, bars, labtab, policy, chunk_counter, lane, blank); break;
    }
    __syncwarp();
  }
}

template <int VCT, bool MM>
__global__ void __launch_bounds__(KAB_WARPS_PER_CTA * 32, KAB_WARP_MINBLOCKS)
    kab_warp_kernel(const KabLattice *__restrict__ lats, int n_lat, KabParams p) {
  kab_warp_body<VCT, MM, false>(lats, n_lat, p, 0);
}

// CTC forced alignment (runtime vocabulary; `blank` = the blank's column -- a kernel argument, not a
// KabParams field, whose growth would move the parameters of every kernel that takes more after it)
__global__ void __launch_bounds__(KAB_WARPS_PER_CTA * 32, KAB_WARP_MINBLOCKS)
    kab_warp_ctc_kernel(const KabLattice *__restrict__ lats, int n_lat, KabParams p, int blank) {
  kab_warp_body<0, false, true>(lats, n_lat, p, blank);
}

// CTC forced alignment with free ends (kab_plan_create_ctc_free)
__global__ void __launch_bounds__(KAB_WARPS_PER_CTA * 32, KAB_WARP_MINBLOCKS)
    kab_warp_ctc_free_kernel(const KabLattice *__restrict__ lats, int n_lat, KabParams p, int blank) {
  kab_warp_body<0, false, true, true>(lats, n_lat, p, blank);
}
