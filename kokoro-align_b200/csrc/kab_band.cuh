// kab_band.cuh -- one CTA per lattice, for chapter-length lattices with the reference's
// diagonal band (align.py:64-65): max_move = 4, labels in 1..V-1, V <= 512, S <= 3T,
// min(beam_size, S) + 32 <= R where R = 104 * NW ring slots (NW warps, NW <= 32).
//
//   * state v lives in ring slot v mod R.  Warp w OWNS slots 104w .. 104w+103: lanes 6..31 hold
//     four consecutive states each IN REGISTERS (even register == blank state).  As the window
//     [lo_i, hi_i) slides up, a lane whose chunk has fallen more than 6 states below lo_i
//     recycles it (between groups) to the next alias (v + R); registers outside the window
//     always hold -inf, so a recycled chunk starts inactive (needs lo_i - lo_{i-1} <= 3, i.e.
//     S <= 3T, and 32 spare ring slots).
//   * the 3-state halo below a lane comes from lane l-1 by SHFL.UP -- no shared memory and NO
//     BARRIER on the per-frame recurrence.  Lanes 0..5 of every warp are GHOST lanes: they hold
//     a copy of the previous warp's top 24 states and recompute them redundantly.  The junk that
//     enters at lane 0 (its lower neighbour is unknown) climbs at most 3 states per frame, so
//     after G = 8 frames it has consumed exactly the 24 ghost states and every owned state is
//     still exact.  Once per group the owners publish their top six lanes through shared memory
//     (one STS.128, one CTA barrier, one LDS.128) and the ghosts start over.
//     tools/emulate_band_v3.py checks this scheme, with adversarial junk, against the CPU restatement.
//   * frames run in groups of 8.  A warp whose cells all stay inside the window for the whole
//     group (the common case) runs a body with no window arithmetic; edge warps run the same
//     body plus the exact incremental window (S*i = q*T + r, no divisions) and -inf masks.
//   * emission rows are staged ahead with 1-D bulk copies (cp.async.bulk + mbarrier; thread 0
//     waits two groups ahead, the group barrier publishes); the gather for the next frame is
//     issued one frame early.
//   * backpointers: one byte (4 cells x 2 bits) per owned lane and frame at
//     i * NBP + (slot >> 2); staged in shared memory, leaving as bulk stores
//     (cp.async.bulk shared -> global), double-buffered.
//   * backtrack in the same CTA: backpointer blocks come back with bulk copies
//     (double-buffered) and one thread walks them at shared-memory latency; the block's outputs
//     are then written coalesced by all threads.
#pragma once
#include "kab_common.cuh"

struct KabTrue { static constexpr bool value = true; };
struct KabFalse { static constexpr bool value = false; };

#define KAB_BAND_STAGES 3
#define KAB_BAND_G 8        // frames per group (between two CTA barriers)
#define KAB_BAND_GHOST 6    // ghost lanes per warp = 3 * G / 4
#define KAB_BAND_OW 104     // ring slots owned by a warp = (32 - GHOST) * 4

// Host + device: geometry of a band launch with NW warps.
struct KabBandGeom {
  int nw, nbp, fb;
  size_t xchg_off, bp_off, path_off, stage_off, smem_bytes;
};
__host__ __device__ inline KabBandGeom kab_band_geom(int nw, int stage_bytes) {
  KabBandGeom g;
  g.nw = nw;
  g.nbp = (26 * nw + 15) & ~15;                       // backpointer row bytes (16-byte multiple)
  g.fb = (16384 / g.nbp) & ~(KAB_BAND_G - 1);         // frames per backpointer block
  g.xchg_off = 128;                                   // after the mbarriers
  g.bp_off = g.xchg_off + 2 * (size_t)nw * KAB_BAND_GHOST * 16;
  g.path_off = g.bp_off + 2 * (size_t)g.fb * g.nbp;
  g.stage_off = (g.path_off + 2 * (size_t)g.fb * 4 + 15) & ~(size_t)15;  // two path buffers
  g.smem_bytes = g.stage_off + (size_t)KAB_BAND_STAGES * stage_bytes;
  return g;
}

// Backtrack of ONE full group (8 frames, descending) from registers, in the backpointer words of the
// cluster and wide kernels (kab_bandp.cuh, kab_wide.cuh: a lane of four states keeps one byte per
// frame, 8 frames per 64-bit word): w0 holds the 8 backpointer bytes of the walker's byte column, w1
// those of the column below (have1: it is available).
// No load sits on the dependent chain (shift -> mask -> subtract -> compare).  Stops before the
// frame that would need a third column; returns the next frame to process (-1: group done) and
// the number of column steps taken (0..2, the last one not yet served when it stopped early).
__device__ __forceinline__ int kab_walk_group8(const uint2 w0, const uint2 w1, const bool have1, int &v, int &k2,
                                               int *pg, int &nchg) {
  // Branch-free on purpose (selects only): with one active thread every taken branch costs a
  // convergence-barrier round trip (~40 cycles, measured), several times the chain itself.  Frames
  // after the stop point are computed and discarded (the caller overwrites their path entries).
  uint32_t cx = w0.x, cy = w0.y;
  int n = 0, f_next = -1, v_s = 0, k2_s = 0, n_s = 0;
  bool stopped = false;
#pragma unroll
  for (int f = 7; f >= 0; --f) {
    const uint32_t word = (f >= 4 ? cy : cx) >> (8 * (f & 3));
    const int mv = (int)((word >> k2) & 3u);
    pg[f] = v;
    v -= mv;
    k2 -= 2 * mv;
    const bool neg = k2 < 0;  // left the byte column
    k2 += neg ? 8 : 0;
    n += neg ? 1 : 0;
    const bool stop_now = neg && !stopped && (n == 2 || !have1);
    f_next = stop_now ? f - 1 : f_next;
    v_s = stop_now ? v : v_s;
    k2_s = stop_now ? k2 : k2_s;
    n_s = stop_now ? n : n_s;
    stopped = stopped || stop_now;
    cx = neg ? w1.x : cx;
    cy = neg ? w1.y : cy;
  }
  if (stopped) { v = v_s; k2 = k2_s; n = n_s; }
  nchg = n;
  return stopped ? f_next : -1;
}

// CTC: the CTC forced-alignment recurrence (kab_common.cuh) in the same window.  Default and long-form
// plans set W so wide that the window is [0, S) in every frame (S + 32 <= R: no chunk is ever recycled);
// banded plans (kab_plan_create_ctc_band) pass beam_size, and a recycled chunk recomputes its repeat bits
// for its new states.  A lattice whose window clips somewhere and whose two end states are both -inf has
// no path inside the band: status 1.  Junk from lane 0 climbs at most two states per frame (16 in a
// group), so the 24 ghost states still cover it; the window advances <= 3 states per frame (S <= 2T + 1).
template <int MAXT, bool MM, bool CTC>
__device__ __forceinline__ void kab_band_body(const KabLattice *__restrict__ lats, int n_lat, const KabParams &p,
                                              const int blank) {
  constexpr int G = KAB_BAND_G, GH = KAB_BAND_GHOST, OW = KAB_BAND_OW;
  const KabBandGeom geo = kab_band_geom(p.band_nw, p.stage_bytes);
  const int NW = geo.nw, NT = NW * 32, R = OW * NW, NBP = geo.nbp, FB = geo.fb;
  const size_t BPB = (size_t)FB * NBP;  // bytes of one backpointer block
  extern __shared__ __align__(128) unsigned char kab_smem[];
  uint64_t *ebars = reinterpret_cast<uint64_t *>(kab_smem);
  uint64_t *bbars = ebars + KAB_BAND_STAGES;
  float4 *xchg = reinterpret_cast<float4 *>(kab_smem + geo.xchg_off);  // [2][NW][GHOST]
  unsigned char *bpblk = kab_smem + geo.bp_off;                        // [2][FB][NBP]
  int *pathbuf = reinterpret_cast<int *>(kab_smem + geo.path_off);
  float *stage_base = reinterpret_cast<float *>(kab_smem + geo.stage_off);
  __shared__ unsigned int s_item;
  __shared__ int s_vmax;
  __shared__ float s_final;
  __shared__ float s_end[2];  // CTC: scores of states S-1, S-2 of the last frame

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const bool owned = lane >= GH;
  // ring slot of this lane's register 0: owned lanes tile the warp's 104 slots, ghost lanes
  // mirror the previous warp's lanes 26..31
  const int slot0 = owned ? OW * warp + 4 * (lane - GH) : (OW * warp - 4 * GH + 4 * lane + R) % R;
  const int prev_warp = warp == 0 ? NW - 1 : warp - 1;
  const float ninf = kab_neg_inf();
  if (tid == 0) {
    for (int s = 0; s < KAB_BAND_STAGES; ++s) kab_mbar_init(&ebars[s], 1);
    kab_mbar_init(&bbars[0], 1);
    kab_mbar_init(&bbars[1], 1);
    kab_fence_mbar_init();
  }
  __syncthreads();
  uint32_t echunks = 0;  // emission chunks issued so far by this CTA (mbarrier phase tracking)
  uint32_t bblocks = 0;  // backpointer blocks fetched so far
  uint32_t xbuf = 0;     // exchange buffer parity

  for (;;) {
    if (tid == 0) {
      s_item = atomicAdd(p.queue, 1u);
      s_vmax = -1;
      if (CTC) s_end[0] = s_end[1] = kab_neg_inf();  // (an end state outside the last window has no owner)
    }
    __syncthreads();
    const unsigned int item = s_item;
    if (item >= (unsigned int)n_lat) break;
    const KabLattice lat = lats[item];
    const int T = lat.T, S = 2 * lat.L + 1, V = p.V, W = p.W;
    const int F = p.stage_frames;
    const uint32_t stage_words = p.stage_bytes >> 2;
    const int n_chunks = (T + F - 1) / F;
    const uint16_t *col16 = p.col16 + lat.col_off;
    unsigned char *bp = p.bp + lat.bp_off;
    const uint32_t one = p.one;  // runtime 1 (see kab_blank_sel)

    // ---- emission pipeline.  Chunk g (counted over the CTA's lifetime) lives in stage
    // g % STAGES and completes phase (g / STAGES) & 1 of that stage's mbarrier.
    const uint32_t ec0 = echunks;
    // F*V*4 is a multiple of 16, so every chunk of this lattice has the same 16-byte skew
    const uint32_t skew = (uint32_t)(((lat.t_off * (int64_t)V * 4) & 15) >> 2);
    // Chunks are F*V*4 bytes apart (a multiple of 16), so all but the last one are plain
    // aligned copies of `full_bytes`; the last chunk goes through the clamping descriptor.
    const char *lp_base = reinterpret_cast<const char *>(p.lp) + ((lat.t_off * (int64_t)V * 4) & ~(int64_t)15);
    const uint32_t chunk_stride = (uint32_t)(F * V * 4);
    const uint32_t full_bytes = (chunk_stride + skew * 4 + 15) & ~15u;
    auto issue = [&](int c, uint32_t stg) {
      float *dst = stage_base + stg * stage_words;
      if (c + 1 < n_chunks) {
        if (tid == 0) {
          kab_mbar_expect_tx(&ebars[stg], full_bytes);
          kab_bulk_g2s(dst, lp_base + (size_t)c * chunk_stride, full_bytes, &ebars[stg]);
        }
      } else {
        const int f0 = c * F, nf = T - f0;
        const KabStageDesc d = kab_stage_desc(p, lat.t_off, f0, nf);
        if (tid == 0) {
          kab_mbar_expect_tx(&ebars[stg], d.bytes);
          if (d.bytes) kab_bulk_g2s(dst, d.src, d.bytes, &ebars[stg]);
        }
        if (tid < (int)d.tail_n)
          dst[d.tail_word + tid] = __ldg(reinterpret_cast<const float *>(d.src) + d.tail_word + tid);
      }
    };
    uint32_t st = ec0 % KAB_BAND_STAGES, ph = (ec0 / KAB_BAND_STAGES) & 1u;  // of the chunk being read
    for (int c = 0; c < min(n_chunks, KAB_BAND_STAGES); ++c) issue(c, (st + c) % KAB_BAND_STAGES);

    // ---- register state: everything inactive except the virtual start state 0 (align.py:57-58)
    float s0 = (owned && slot0 == 0) ? 0.0f : ninf, s1 = ninf, s2 = ninf, s3 = ninf;
    int vb = slot0;  // first state of this lane's chunk (alias level 0)
    auto load_cols = [&](int base, uint32_t &ca, uint32_t &cb) {
      ca = base + 1 < S ? 4u * col16[base >> 1] : 0u;
      cb = base + 3 < S ? 4u * col16[(base >> 1) + 1] : 0u;
    };
    uint32_t c1, c3, nc1, nc3;  // byte offsets of the two label columns; next alias prefetched
    load_cols(vb, c1, c3);
    load_cols(vb + R, nc1, nc3);
    const int half = W / 2;
    const uint32_t boff = CTC ? 4u * (uint32_t)blank : 0u;  // byte offset of the blank's column
    // CTC: bit 0 / 1 = move 2 forbidden into label state vb+1 / vb+3 (state 1, or a repeated label)
    uint32_t rep = 0;
    // CTC, next alias: byte offset of the label column of state vb+R-1 (the one below vb+R+1), prefetched
    // with nc1 / nc3 so that recycling a chunk recomputes its repeat bits without waiting for a load
    uint32_t ncm = 0;
    auto load_below = [&](int base) { return base + 1 < S ? 4u * col16[(base >> 1) - 1] : 0u; };
    if (CTC) {
      const int l1 = vb >> 1;  // label index of state vb+1
      if (vb + 1 < 3 || vb + 1 >= S || col16[l1] == col16[l1 - 1]) rep |= 1u;
      if (vb + 3 >= S || col16[l1 + 1] == col16[l1]) rep |= 2u;
      ncm = load_below(vb + R);
    }

    float poison = kab_poison_init<CTC>();  // NaN once a rejected log-prob was staged (kab_poison_t)
    if (tid == 0) {
      kab_mbar_wait(&ebars[st], ph);
      if (F < 2 * G && n_chunks > 1) {  // F == G: chunk 1 opens at group 1, before the look-ahead wait
        const uint32_t sn = st + 1 == KAB_BAND_STAGES ? 0 : st + 1;
        kab_mbar_wait(&ebars[sn], sn == 0 ? ph ^ 1u : ph);
      }
    }
    __syncthreads();  // tail words and the first chunk(s) visible to everybody
    // rowc: staged row whose emissions are in (eb, e1, e3); cn: chunk being read
    const char *rowc = reinterpret_cast<const char *>(stage_base + st * stage_words + skew);
    int cn = 0;
    auto check_chunk = [&](int c) {  // finiteness of chunk c's words (all threads, strided)
      const float *w = stage_base + st * stage_words + skew;
      const int nw = min(F, T - c * F) * V;
      for (int j = tid; j < nw; j += NT) poison = kab_poison_t<CTC>(poison, w[j]);
    };
    check_chunk(0);
    float eb = *reinterpret_cast<const float *>(rowc + boff);
    float e1 = *reinterpret_cast<const float *>(rowc + c1);
    float e3 = *reinterpret_cast<const float *>(rowc + c3);

    // ---- window state.  S*i = q*T + r is tracked per GROUP of G frames (step S*G) and, inside
    // a group that needs it, per frame (step S): exact floor(S*i/T) without divisions.
    const int qd = S / T, rd = S % T;                                    // per-frame step
    const int qdg = (int)(((int64_t)S * G) / T), rdg = (int)(((int64_t)S * G) % T);  // per-group step
    int qg = 0, rg = 0;  // q, r at the first frame of the current group
    int q = 0, r = 0;    // per-frame window of a SLOW group

    unsigned char *bpst = bpblk + (slot0 >> 2);  // this lane's byte of the group's first staging row

    // One frame.  No barrier: everything a lane needs from other lanes comes by shuffle.
    auto frame = [&](auto slow_tag, unsigned char *bpdst, const char *rownext, const bool has_next) {
      constexpr bool SLOW = decltype(slow_tag)::value;
      int lo = 0, hi = 0;
      if (SLOW) {
        lo = max(0, q - half);   // align.py:64
        hi = min(lo + W, S);     // align.py:65
        q += qd; r += rd;
        if (r >= T) { r -= T; ++q; }
      }
      // previous-frame scores of the three states below this lane's chunk (lane 0: junk, see top)
      const float h1 = __shfl_up_sync(KAB_FULL_MASK, s3, 1);
      const float h2 = __shfl_up_sync(KAB_FULL_MASK, s2, 1);
      const float h3 = __shfl_up_sync(KAB_FULL_MASK, s1, 1);
      // candidates: (even, odd) state pairs share one packed add
      float t0, t1, t2, t3;
      kab_add2(s0, s1, eb, t0, t1);
      kab_add2(s2, s3, eb, t2, t3);
      const float th1 = __fadd_rn(h1, eb), th3 = __fadd_rn(h3, eb);
      float a0, a1, a2, a3, b0, b1, b2, b3;
      kab_add2(s0, s1, e1, a1, a0);
      kab_add2(h2, h1, e1, a3, a2);
      kab_add2(s2, s3, e3, b1, b0);
      kab_add2(s0, s1, e3, b3, b2);
      (void)t3;
      uint32_t m = 0;
      float n0 = kab_blank_sel(t0, kab_mm<MM>(th1, p.mm1), kab_mm<MM>(th3, p.mm3), m, 1u << 0, 2u << 0, one);
      float n1 = kab_label_sel(a0, kab_mm<MM>(a1, p.mm1), kab_mm<MM>(a2, p.mm2), kab_mm<MM>(a3, p.mm3), m, 1u << 2, 2u << 2, one);
      float n2 = kab_blank_sel(t2, kab_mm<MM>(t1, p.mm1), kab_mm<MM>(th1, p.mm3), m, 1u << 4, 2u << 4, one);
      float n3 = kab_label_sel(b0, kab_mm<MM>(b1, p.mm1), kab_mm<MM>(b2, p.mm2), kab_mm<MM>(b3, p.mm3), m, 1u << 6, 2u << 6, one);
      if (CTC) {  // (replaces all of the above but h1, which is the one state below the lane's chunk)
        m = 0;
        n0 = __fadd_rn(kab_ctc_blank_sel(s0, h1, m, 0), eb);
        n1 = __fadd_rn(kab_ctc_label_sel(s1, s0, rep & 1u ? ninf : h1, m, 2), e1);
        n2 = __fadd_rn(kab_ctc_blank_sel(s2, s1, m, 4), eb);
        n3 = __fadd_rn(kab_ctc_label_sel(s3, s2, rep & 2u ? ninf : s1, m, 6), e3);
      }
      if (SLOW) {  // cells outside [lo, hi) are inactive: state vb+k is inside iff 0 <= vb+k-lo < hi-lo
        const unsigned a = (unsigned)(vb - lo), wd = (unsigned)(hi - lo);
        n0 = (a + 0u < wd) ? n0 : ninf;
        n1 = (a + 1u < wd) ? n1 : ninf;
        n2 = (a + 2u < wd) ? n2 : ninf;
        n3 = (a + 3u < wd) ? n3 : ninf;
      }
      s0 = n0; s1 = n1; s2 = n2; s3 = n3;
      if (owned) *bpdst = (unsigned char)m;
      if (has_next) {  // emissions of frame i+1 (its chunk was published by an earlier barrier)
        rowc = rownext;
        eb = *reinterpret_cast<const float *>(rownext + boff);
        e1 = *reinterpret_cast<const float *>(rownext + c1);
        e3 = *reinterpret_cast<const float *>(rownext + c3);
      }
    };

    const int n_groups = (T + G - 1) / G;
    const int VB = V * 4;  // bytes per emission row
#ifdef KAB_BAND_TIMING
    long long tm_fast = 0, tm_slow = 0, tm_epi = 0, tm_bar = 0, tm_post = 0; int n_fast = 0, n_slow = 0;
    const long long tm_start = clock64();
#endif
    int fic = 0;           // frame offset of the current group inside its emission chunk (no divisions
    int fib = 0, blk = 0;  // ... inside its backpointer block; index of that block    in the loop)
    for (int g = 0; g < n_groups; ++g) {
      const int i0 = g * G, nfr = min(G, T - i0);
      // row of the first frame of the NEXT group: same chunk, or the start of the next stage
      const bool next_crosses = fic + G == F;
      const uint32_t nst = st + 1 == KAB_BAND_STAGES ? 0 : st + 1;
      const char *row0 = rowc;  // frame i0 (its emissions are already in eb/e1/e3)
      const char *rowng = next_crosses ? reinterpret_cast<const char *>(stage_base + nst * stage_words + skew)
                                       : row0 + G * VB;
      // window at the first frame of this group and (conservatively) at its last frame
      const int lo0 = max(0, qg - half), hi0 = min(lo0 + W, S);
      int qn = qg + qdg, rn = rg + rdg;
      if (rn >= T) { rn -= T; ++qn; }
      const int lo1 = max(0, qn - half);  // lo of the next group's first frame >= lo of every frame here
      // recycle a chunk that lies entirely more than 3 states below the window.  Done between
      // groups only: the ring has >= 32 spare slots, so the alias cannot reach the top edge
      // before the next group boundary (the window advances <= 3 states per frame)
      while (vb + 3 < lo0 - 3) {
        vb += R;
        if (CTC) {  // the repeat bits of the new states, as at lattice start (vb >= R: state vb+1 is not state 1)
          rep = (vb + 1 >= S || nc1 == ncm ? 1u : 0u) | (vb + 3 >= S || nc3 == nc1 ? 2u : 0u);
          ncm = load_below(vb + R);
        }
        c1 = nc1; c3 = nc3;
        load_cols(vb + R, nc1, nc3);
        e1 = *reinterpret_cast<const float *>(rowc + c1);  // the prefetched emissions belonged
        e3 = *reinterpret_cast<const float *>(rowc + c3);  // to the old alias
      }
      // warp-uniform choice of the group body
      const bool safe = __all_sync(KAB_FULL_MASK, nfr == G && vb >= lo1 && vb + 4 <= hi0);
#ifdef KAB_BAND_TIMING
      const long long tm0 = clock64();
#endif
      if (safe) {
#pragma unroll
        for (int f = 0; f < G; ++f)
          frame(KabFalse{}, bpst + f * NBP, f + 1 < G ? row0 + (f + 1) * VB : rowng, f + 1 < G || i0 + G < T);
      } else if (nfr == G) {
        q = qg; r = rg;
#pragma unroll
        for (int f = 0; f < G; ++f)
          frame(KabTrue{}, bpst + f * NBP, f + 1 < G ? row0 + (f + 1) * VB : rowng, f + 1 < G || i0 + G < T);
      } else {
        q = qg; r = rg;
        for (int f = 0; f < nfr; ++f) frame(KabTrue{}, bpst + f * NBP, row0 + (f + 1) * VB, f + 1 < nfr);
      }
      qg = qn; rg = rn;
      bpst += G * NBP;
#ifdef KAB_BAND_TIMING
      const long long tm1 = clock64();
      if (safe) { tm_fast += tm1 - tm0; ++n_fast; } else { tm_slow += tm1 - tm0; ++n_slow; }
#endif

      // ---- between groups: publish the top six lanes, one CTA barrier, reload the ghosts
      const bool more = i0 + G < T;
      const bool block_done = fib + G == FB || !more;  // backpointer block complete
      if (more && lane >= 32 - GH) xchg[(xbuf * NW + warp) * GH + (lane - (32 - GH))] = make_float4(s0, s1, s2, s3);
      if (block_done) kab_fence_proxy_async();  // staged backpointer bytes -> visible to the bulk store
      if (tid == 0) {
        // the chunk that opens two groups ahead (always the one after the next group's chunk):
        // wait now, this group's barrier publishes it
        if ((F == G || fic == 0) && i0 + 2 * G < T) {
          const bool adv = next_crosses && more;  // the next group already reads chunk cn + 1
          uint32_t s2s = adv ? nst : st, p2 = (adv && nst == 0) ? ph ^ 1u : ph;
          if (++s2s == KAB_BAND_STAGES) { s2s = 0; p2 ^= 1u; }
          kab_mbar_wait(&ebars[s2s], p2);
        }
        if (block_done) kab_bulk_wait_read0();  // the previous bulk store no longer reads its buffer
      }
#ifdef KAB_BAND_TIMING
      const long long tm2 = clock64();
#endif
      __syncthreads();
#ifdef KAB_BAND_TIMING
      const long long tm3 = clock64();
      tm_epi += tm2 - tm1; tm_bar += tm3 - tm2;
#endif
      if (more && !owned) {
        const float4 x = xchg[(xbuf * NW + prev_warp) * GH + lane];
        s0 = x.x; s1 = x.y; s2 = x.z; s3 = x.w;
      }
      xbuf ^= 1u;
      if (next_crosses && more) {  // the next group opens chunk cn+1
        ++cn;
        st = nst;
        if (st == 0) ph ^= 1u;
        check_chunk(cn);
        // everybody has finished with chunk cn-1: refill its stage with chunk cn + STAGES - 1
        if (cn + KAB_BAND_STAGES - 1 < n_chunks)
          issue(cn + KAB_BAND_STAGES - 1, (st + KAB_BAND_STAGES - 1) % KAB_BAND_STAGES);
      }
      if (block_done) {
        const int nb = fib + nfr;  // frames in this block
        if (tid == 0)
          kab_bulk_s2g(bp + (size_t)blk * BPB, bpblk + (size_t)(blk & 1) * BPB, (uint32_t)nb * NBP);
        ++blk; fib = 0;
        bpst = bpblk + (size_t)(blk & 1) * BPB + (slot0 >> 2);
      } else {
        fib += G;
      }
      fic = next_crosses ? 0 : fic + G;
#ifdef KAB_BAND_TIMING
      tm_post += clock64() - tm3;
#endif
    }
#ifdef KAB_BAND_TIMING
    if (lane == 0 && p.debug) {
      long long *d = p.debug + warp * 8;
      d[0] = tm_fast; d[1] = n_fast; d[2] = tm_slow; d[3] = n_slow; d[4] = tm_epi; d[5] = tm_bar; d[6] = tm_post;
      d[7] = clock64() - tm_start;
    }
#endif
    echunks = ec0 + n_chunks;

    if (CTC) {  // CTC end rule: the better of the last two states, S-2 on a tie (kab_common.cuh)
      if (owned) {
        if (vb + 0 == S - 1) s_end[0] = s0;
        if (vb + 1 == S - 1) s_end[0] = s1;
        if (vb + 2 == S - 1) s_end[0] = s2;
        if (vb + 3 == S - 1) s_end[0] = s3;
        if (vb + 0 == S - 2) s_end[1] = s0;
        if (vb + 1 == S - 2) s_end[1] = s1;
        if (vb + 2 == S - 2) s_end[1] = s2;
        if (vb + 3 == S - 2) s_end[1] = s3;
      }
    } else {  // ---- forced end state: highest active state of frame T-1 (align.py:99-101)
      int cand = -1;
      if (owned) {
        if (vb + 0 < S && s0 > ninf) cand = vb + 0;
        if (vb + 1 < S && s1 > ninf) cand = vb + 1;
        if (vb + 2 < S && s2 > ninf) cand = vb + 2;
        if (vb + 3 < S && s3 > ninf) cand = vb + 3;
      }
      cand = __reduce_max_sync(KAB_FULL_MASK, cand);
      if (lane == 0 && cand >= 0) atomicMax(&s_vmax, cand);
    }
    if (tid == 0) kab_bulk_wait0();  // all backpointer blocks are in global memory
    const int any_bad = __syncthreads_or(poison != poison ? 1 : 0);
    int v = s_vmax;
    if (CTC) {
      v = (S >= 2 && !(s_end[0] > s_end[1])) ? S - 2 : S - 1;
      // no path stays inside a window that clips (a covering window follows the recurrence instead)
      const bool clips = W < S || (int)(((int64_t)S * (T - 1)) / T) > half;
      if (clips && !(s_end[0] > ninf) && !(s_end[1] > ninf)) v = -1;
    }
    const int status = any_bad ? 3 : (v < 0 ? 1 : 0);
    if (owned && status == 0) {
      if (vb + 0 == v) s_final = s0;
      if (vb + 1 == v) s_final = s1;
      if (vb + 2 == v) s_final = s2;
      if (vb + 3 == v) s_final = s3;
    }
    __syncthreads();
    if (tid == 0) {
      p.status[lat.index] = status;
      if (p.final_score) p.final_score[lat.index] = status == 0 ? s_final : __int_as_float(0x7fc00000);
    }
    if (status == 0) {
      // ---- backtrack (== flush_determined_path, align.py:21-40)
      const int n_blocks = (T + FB - 1) / FB;
      const uint32_t bb0 = bblocks;
      auto fetch = [&](int blk) {  // thread 0 only
        const uint32_t gi = bb0 + (uint32_t)(n_blocks - 1 - blk), bs = gi & 1u;
        const int nfrm = min(FB, T - blk * FB);
        const uint32_t bytes = (uint32_t)nfrm * NBP;
        kab_mbar_expect_tx(&bbars[bs], bytes);
        kab_bulk_g2s(bpblk + (size_t)bs * BPB, bp + (size_t)blk * BPB, bytes, &bbars[bs]);
      };
      if (tid == 0) fetch(n_blocks - 1);
      int32_t *out_path = p.best_path + lat.t_off;
      int32_t *out_lab = p.best_labels + lat.t_off;
      float *out_sc = p.best_scores + lat.t_off;
      const float *lp = p.lp + lat.t_off * (int64_t)V;
      // Warp 0 walks a block while the other warps write the previous block's outputs.
      int slot = v % R;  // ring slot of the walker's state
      auto flush_block = [&](int blk, int first_thread, int n_threads) {
        const int i0 = blk * FB, i1 = min(T, i0 + FB);
        const int *pbuf = pathbuf + (blk & 1) * FB;
        for (int i = i0 + (tid - first_thread); i < i1; i += n_threads) {
          const int pv = pbuf[i - i0];
          const int lab = (pv & 1) ? (int)col16[(pv - 1) >> 1] : (CTC ? blank : 0);
          out_path[i] = pv;
          out_lab[i] = lab;                              // align.py:106
          out_sc[i] = __ldg(&lp[(int64_t)i * V + lab]);  // align.py:107
        }
      };
      for (int blk = n_blocks - 1; blk >= 0; --blk) {
        const uint32_t gi = bb0 + (uint32_t)(n_blocks - 1 - blk), bs = gi & 1u;
        const int i0 = blk * FB, i1 = min(T, i0 + FB);
        if (warp == 0) {
          if (lane == 0 && blk > 0) fetch(blk - 1);  // other buffer: its previous contents were consumed
          kab_mbar_wait(&bbars[bs], (gi >> 1) & 1u);
          const unsigned char *blkp = bpblk + (size_t)bs * BPB;
          int *pbuf = pathbuf + (blk & 1) * FB;
          if (lane == 0) {  // the walk itself is a dependent chain: one lane, shared-memory latency
            const unsigned char *rowp = blkp + (size_t)(i1 - 1 - i0) * NBP;
            for (int i = i1 - 1; i >= i0; --i, rowp -= NBP) {
              const unsigned char byte = rowp[slot >> 2];
              pbuf[i - i0] = v;
              const int mv = kab_decode_move((byte >> (2 * (slot & 3))) & 3u);
              v -= mv;
              slot -= mv;
              if (slot < 0) slot += R;
            }
          }
          v = __shfl_sync(KAB_FULL_MASK, v, 0);
          slot = __shfl_sync(KAB_FULL_MASK, slot, 0);
          if (NW == 1 && blk + 1 < n_blocks) { __syncwarp(); flush_block(blk + 1, 0, 32); }
        } else if (blk + 1 < n_blocks) {
          flush_block(blk + 1, 32, NT - 32);
        }
        __syncthreads();
      }
      flush_block(0, 0, NT);
      bblocks = bb0 + n_blocks;
    }
    __syncthreads();
  }
}

// MAXT: upper bound of the block size (512 -> up to 128 registers per thread, 1024 -> 64).
template <int MAXT, bool MM>
__global__ void __launch_bounds__(MAXT, 1) kab_band_kernel(const KabLattice *__restrict__ lats, int n_lat,
                                                           KabParams p) {
  kab_band_body<MAXT, MM, false>(lats, n_lat, p, 0);
}

// CTC forced alignment (whole-lattice window; blank column: see kab_warp_ctc_kernel)
template <int MAXT>
__global__ void __launch_bounds__(MAXT, 1) kab_band_ctc_kernel(const KabLattice *__restrict__ lats, int n_lat,
                                                               KabParams p, int blank) {
  kab_band_body<MAXT, false, true>(lats, n_lat, p, blank);
}
