// kab_wide.cuh -- UNBANDED lattices too wide for one CTA (BASELINE config 4(ii): a book-length
// lattice aligned without the diagonal band, S up to ~10^5 states): max_move = 4, labels in
// 1..V-1, V <= 512, the window of align.py:64-65 covers the whole lattice (beam_size >= S and
// S(T-1)/T <= beam_size/2), S > what the band kernel holds.
//
// The state axis is cut into chunks of 104 states, one WARP each (4 states per lane in lanes
// 6..31, lanes 0..5 are ghost lanes that recompute the lower neighbour's top 24 states for 8
// frames -- the scheme of kab_band.cuh), and the warps are spread over the WHOLE GPU: four compute
// warps and one producer warp per CTA, as many CTAs as the lattice needs (S = 10^5 -> 962 warps
// -> 241 CTAs), all resident.  There is no barrier of any kind on the recurrence:
//   * the lattice is a CHAIN: warp w only needs warp w-1's top 24 states after that warp's previous
//     8-frame group.  They travel through a FIFO in global memory (L2): every score is written
//     together with the message's sequence number as ONE 8-byte store, which is single-copy
//     atomic, so the consumer needs no fence and no flag -- it polls the four (score, seq)
//     pairs of its lane, and it issues those loads one group early so that their L2 latency
//     hides behind the frames.  The chain skews by itself into a wavefront (warp w runs two to
//     three groups behind warp w-1); the FIFO is 64 messages deep and the producer reads the
//     consumer's progress counter only when it is about to lap it;
//   * emission rows are staged per CTA by the producer warp (bulk copies + full / empty
//     mbarriers, 16 stages); every CTA reads every row, a few microseconds apart, so all but
//     the first read hit L2; the producer warp also checks the rows for non-finite values;
//   * backpointers: 64-bit words per lane and group (8 frames x 4 cells x 2 bits), staged per
//     warp and written with bulk stores to the warp's region [warp][group][32 lanes][8 B]:
//     2 bits per cell, 25 GB for T = 10^6, S = 10^5 -- no checkpointing needed in 180 GB;
//   * one extra CTA backtracks: it waits until every warp of the lattice has published its
//     highest active state (align.py:99-101) and flushed its backpointers, then walks exactly
//     like kab_bandp.cuh (blocks of 128 frames of the current warp region and the two below it
//     by bulk copies) while the other CTAs are already running the next lattice.
#pragma once
#include "kab_band.cuh"  // KAB_BAND_G / GHOST / OW: the lanes of kab_band.cuh; kab_walk_group8
#include "kab_common.cuh"

// Group timestamps of the KAB_WIDE_TIMING build.  The KAB_BANDP_TIMING build takes them as well (the
// two kernels shared one timing macro), so that build keeps compiling this kernel as it always did.
#if defined(KAB_WIDE_TIMING) || defined(KAB_BANDP_TIMING)
#define KAB_WTM(var) const long long var = clock64()
#else
#define KAB_WTM(var)
#endif

#define KAB_WD_CW 4      // compute warps per CTA
#ifndef KAB_WD_NS
#define KAB_WD_NS 16     // emission stages per CTA: the four warps of a CTA are up to ~10 groups apart
#endif
#ifndef KAB_WD_D
#define KAB_WD_D 64      // neighbour FIFO depth (messages).  Deep on purpose: a consumer that has fallen two
#endif                  // groups behind finds every message prefetched and never blocks again; with 8 slots the
                        // credits keep pulling it back into blocking polls (measured: 55 ms -> 24 ms at D = 64)
#ifndef KAB_WD_LAG
#define KAB_WD_LAG 2     // a warp starts once its lower neighbour has finished this many groups, so that
#endif                   // every later message is already there when it is prefetched (a group early)
#ifndef KAB_WD_FBW
#define KAB_WD_FBW 128   // frames per per-warp backpointer block (256 would cost the second resident CTA per SM)
#endif
#define KAB_WD_FBK 128   // frames per backtrack block
#define KAB_WD_NREG 3    // warp regions staged per backtrack block
#define KAB_WD_THREADS ((KAB_WD_CW + 1) * 32)
#define KAB_WD_MSG_BYTES (KAB_BAND_GHOST * 32)  // 6 lanes x 4 (score, seq) pairs

// Global scratch of one wide lattice (zeroed before every run), at wide_ws + lat.scr_off * 4:
//   [0] vmax + 1 (0 = no active state)   [1] non-finite flag   [2] warps finished   [3] unused
//   (CTC: [0] score bits of state S-2, [3] score bits of state S-1)
//   then cand[nww] (state, score bits), cons[nww] (messages consumed by warp w), fifo[nww][D][192 B]
__host__ __device__ inline size_t kab_wide_cand_off() { return 16; }
__host__ __device__ inline size_t kab_wide_cons_off(int nww) { return 16 + (size_t)nww * 8; }
__host__ __device__ inline size_t kab_wide_fifo_off(int nww) { return (16 + (size_t)nww * 12 + 255) & ~(size_t)255; }
__host__ __device__ inline size_t kab_wide_ws_bytes(int nww) {
  return kab_wide_fifo_off(nww) + (size_t)nww * KAB_WD_D * KAB_WD_MSG_BYTES;
}

struct KabWideGeom {
  size_t bpst_off, bt_off, path_off, stage_off, smem_bytes;
};
__host__ __device__ inline KabWideGeom kab_wide_geom(int stage_bytes) {
  KabWideGeom g;
  // after the mbarriers efull[NS], eempty[NS], btbar[2] (272 bytes at NS = 16; an offset of 256 put warp 0's
  // staged backpointers of states 0..7, frames 0..7 on btbar)
  g.bpst_off = ((size_t)(2 * KAB_WD_NS + 2) * 8 + 127) & ~(size_t)127;
  g.bt_off = g.bpst_off + (size_t)KAB_WD_CW * 2 * KAB_WD_FBW * 32;
  g.path_off = g.bt_off + (size_t)2 * KAB_WD_NREG * KAB_WD_FBK * 32;
  g.stage_off = g.path_off + (size_t)2 * KAB_WD_FBK * 4;
  g.smem_bytes = g.stage_off + (size_t)KAB_WD_NS * stage_bytes;
  return g;
}

// Grid: n_fwd forward CTAs + 1 backtrack CTA (the last one), all resident.  Every CTA runs over the
// wide lattices in the same order.
// CTC: the CTC forced-alignment recurrence (kab_common.cuh, DESIGN.md 3.9) over the whole lattice, blank
// column `blank`.  Junk enters lane 0 of a warp only through h1 (state vb by move 1, vb+1 by move 2) and
// climbs at most two states per frame, so at most 16 states in a group of 8 frames: the 24 ghost states
// still absorb it.  The end states S-1 and S-2 may sit in different warps (S = 1 mod 104: S-1 is the
// first state of the top warp), so their owners publish both scores to the lattice's scratch and the
// backtrack CTA applies the end rule.
template <bool CTC>
__device__ __forceinline__ void kab_wide_body(const KabLattice *__restrict__ lats, int n_lat, const KabParams &p,
                                              unsigned char *wide_ws, const int blank) {
  constexpr int G = KAB_BAND_G, GH = KAB_BAND_GHOST, OW = KAB_BAND_OW;
  constexpr int CW = KAB_WD_CW, NS = KAB_WD_NS, D = KAB_WD_D, FBW = KAB_WD_FBW, FBK = KAB_WD_FBK, NREG = KAB_WD_NREG;
  static_assert(G == 8, "a group of 8 frames is one 64-bit backpointer word per lane");
  const KabWideGeom geo = kab_wide_geom(p.stage_bytes);
  extern __shared__ __align__(128) unsigned char kab_smem[];
  uint64_t *efull = reinterpret_cast<uint64_t *>(kab_smem);  // [NS]
  uint64_t *eempty = efull + NS;                             // [NS]
  uint64_t *btbar = eempty + NS;                             // [2]
  unsigned char *btbuf = kab_smem + geo.bt_off;
  int *pathbuf = reinterpret_cast<int *>(kab_smem + geo.path_off);
  float *stage_base = reinterpret_cast<float *>(kab_smem + geo.stage_off);
  __shared__ int s_v;
  __shared__ int s_status;

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const bool is_bt = blockIdx.x == gridDim.x - 1;
  const bool is_prod = warp == CW;
  const int gw = (int)blockIdx.x * CW + warp;  // global compute-warp index
  const bool owned = lane >= GH;
  const float ninf = kab_neg_inf();
  const int V = p.V, F = p.stage_frames;
  const uint32_t stage_words = p.stage_bytes >> 2;
  const int VB = V * 4;

  if (tid == 0) {
    for (int s = 0; s < NS; ++s) {
      kab_mbar_init(&efull[s], 1);
      kab_mbar_init(&eempty[s], CW);
    }
    kab_mbar_init(&btbar[0], 1);
    kab_mbar_init(&btbar[1], 1);
    kab_fence_mbar_init();
  }
  __syncthreads();

  if (!is_bt) {
    // =========================================================== forward CTAs
    uint32_t echunks = 0;  // emission chunks staged so far by this CTA
    for (int li = 0; li < n_lat; ++li) {
      const KabLattice lat = lats[li];
      const int nww = lat.k;
      if ((int)blockIdx.x * CW >= nww) continue;  // this CTA holds no states of the lattice
      const int T = lat.T, S = 2 * lat.L + 1;
      const int n_chunks = (T + F - 1) / F, n_groups = (T + G - 1) / G;
      unsigned char *ws = wide_ws + (size_t)lat.scr_off * 4;
      unsigned int *ctl = reinterpret_cast<unsigned int *>(ws);
      const uint32_t ec0 = echunks;
      const uint32_t skew = (uint32_t)(((lat.t_off * (int64_t)V * 4) & 15) >> 2);

      if (is_prod) {
        // ------------------------------------------------ producer warp
        const char *lp_base = reinterpret_cast<const char *>(p.lp) + ((lat.t_off * (int64_t)V * 4) & ~(int64_t)15);
        const uint32_t chunk_stride = (uint32_t)(F * V * 4);
        const uint32_t full_bytes = (chunk_stride + skew * 4 + 15) & ~15u;
        float poison = kab_poison_init<CTC>();  // NaN once a rejected log-prob was staged (kab_poison_t)
        auto check_chunk = [&](int c) {
          const uint32_t gc = ec0 + (uint32_t)c, stg = gc % NS;
          kab_mbar_wait(&efull[stg], (gc / NS) & 1u);
          const float *w = stage_base + stg * stage_words + skew;
          const int nw = min(F, T - c * F) * V;
          for (int j = lane; j < nw; j += 32) poison = kab_poison_t<CTC>(poison, w[j]);
        };
        for (int c = 0; c < n_chunks; ++c) {
          const uint32_t gc = ec0 + (uint32_t)c, stg = gc % NS, use = gc / NS;
          if (c >= NS) check_chunk(c - NS);
          if (use > 0) kab_mbar_wait(&eempty[stg], (use - 1u) & 1u);
          float *dst = stage_base + stg * stage_words;
          if (c + 1 < n_chunks) {
            if (lane == 0) {
              kab_mbar_expect_tx(&efull[stg], full_bytes);
              kab_bulk_g2s(dst, lp_base + (size_t)c * chunk_stride, full_bytes, &efull[stg]);
            }
          } else {
            const int f0 = c * F, nf = T - f0;
            const KabStageDesc d = kab_stage_desc(p, lat.t_off, f0, nf);
            if (lane < (int)d.tail_n)
              dst[d.tail_word + lane] = __ldg(reinterpret_cast<const float *>(d.src) + d.tail_word + lane);
            __syncwarp();
            if (lane == 0) {
              kab_mbar_expect_tx(&efull[stg], d.bytes);
              if (d.bytes) kab_bulk_g2s(dst, d.src, d.bytes, &efull[stg]);
            }
          }
          __syncwarp();
        }
        for (int c = max(0, n_chunks - NS); c < n_chunks; ++c) check_chunk(c);
        if (blockIdx.x == 0 && __any_sync(KAB_FULL_MASK, poison != poison) && lane == 0) atomicOr(&ctl[1], 1u);
      } else if (gw >= nww) {
        // ------------------------------------------------ spare compute warp of the last CTA: only
        // keeps the emission ring's accounting (every chunk needs CW releases)
        for (int c = 0; c < n_chunks; ++c) {
          const uint32_t gc = ec0 + (uint32_t)c, stg = gc % NS;
          kab_mbar_spin(&efull[stg], (gc / NS) & 1u);
          __syncwarp();
          if (lane == 0) kab_mbar_arrive(&eempty[stg]);
        }
      } else {
        // ------------------------------------------------ compute warp gw: states 104 gw .. 104 gw + 103
        const uint16_t *col16 = p.col16 + lat.col_off;
        const uint32_t one = p.one;
        const int vb = OW * gw + 4 * (lane - GH);  // first state of this lane (ghost lanes: the 24 below)
        float s0 = (vb == 0) ? 0.0f : ninf, s1 = ninf, s2 = ninf, s3 = ninf;  // start state 0 (align.py:57-58)
        const uint32_t c1 = (vb + 1 > 0 && vb + 1 < S) ? 4u * col16[vb >> 1] : 0u;
        const uint32_t c3 = (vb + 3 > 0 && vb + 3 < S) ? 4u * col16[(vb >> 1) + 1] : 0u;
        const uint32_t boff = CTC ? 4u * (uint32_t)blank : 0u;  // byte offset of the blank's column
        // CTC: bit 0 / 1 = move 2 forbidden into label state vb+1 / vb+3 (state 1, outside the lattice
        // -- the ghost lanes of warp 0 hold states below 0 --, or a repeated label)
        uint32_t rep = 0;
        if (CTC) {
          const int l1 = vb >> 1;  // label index of state vb+1
          if (vb + 1 < 3 || vb + 1 >= S || col16[l1] == col16[l1 - 1]) rep |= 1u;
          if (vb + 3 < 3 || vb + 3 >= S || col16[l1 + 1] == col16[l1]) rep |= 2u;
        }
        uint32_t st = ec0 % NS, ph = (ec0 / NS) & 1u;
        auto chunk_ptr = [&](uint32_t stg) { return reinterpret_cast<const char *>(stage_base + stg * stage_words + skew); };
        float eb[G], e1[G], e3[G], nb[G], n1[G], n3[G];
        auto load_group = [&](const char *row, float (&xb)[G], float (&x1)[G], float (&x3)[G]) {
#pragma unroll
          for (int f = 0; f < G; ++f) {
            xb[f] = *reinterpret_cast<const float *>(row + f * VB + boff);
            x1[f] = *reinterpret_cast<const float *>(row + f * VB + c1);
            x3[f] = *reinterpret_cast<const float *>(row + f * VB + c3);
          }
        };
        kab_mbar_spin(&efull[st], ph);
        const char *rowc = chunk_ptr(st);
        load_group(rowc, eb, e1, e3);

        unsigned char *bpbuf = kab_smem + geo.bpst_off + (size_t)warp * 2 * FBW * 32;
        unsigned char *bpg = p.bp + lat.bp_off + (size_t)gw * n_groups * 256;
        int fib = 0, blk = 0, fic = 0;
        // FIFO: my inbox (messages of warp gw-1) and the inbox of warp gw+1
        unsigned char *fifo = ws + kab_wide_fifo_off(nww);
        const unsigned char *inbox = fifo + (size_t)gw * D * KAB_WD_MSG_BYTES + lane * 32;             // ghost lanes
        unsigned char *outbox = fifo + (size_t)(gw + 1) * D * KAB_WD_MSG_BYTES + (lane - (32 - GH)) * 32;  // top lanes
        unsigned int *cons = reinterpret_cast<unsigned int *>(ws + kab_wide_cons_off(nww));
        const bool has_below = gw > 0, has_above = gw + 1 < nww;
        uint32_t cons_seen = 0;  // messages the warp above is known to have consumed
        uint2 pf0 = make_uint2(0, 0), pf1 = pf0, pf2 = pf0, pf3 = pf0;  // message g-1, loaded a group early

        auto frame = [&](const float xb, const float x1, const float x3, uint32_t &w, const int sh) {
          const float h1 = __shfl_up_sync(KAB_FULL_MASK, s3, 1);
          const float h2 = __shfl_up_sync(KAB_FULL_MASK, s2, 1);
          const float h3 = __shfl_up_sync(KAB_FULL_MASK, s1, 1);
          float t0, t1, t2, t3;
          kab_add2(s0, s1, xb, t0, t1);
          kab_add2(s2, s3, xb, t2, t3);
          const float th1 = __fadd_rn(h1, xb), th3 = __fadd_rn(h3, xb);
          float a0, a1, a2, a3, b0, b1, b2, b3;
          kab_add2(s0, s1, x1, a1, a0);
          kab_add2(h2, h1, x1, a3, a2);
          kab_add2(s2, s3, x3, b1, b0);
          kab_add2(s0, s1, x3, b3, b2);
          (void)t3;
          const float n0 = kab_blank_sel(t0, th1, th3, w, 1u << (sh + 0), 2u << (sh + 0), one);
          const float m1 = kab_label_sel(a0, a1, a2, a3, w, 1u << (sh + 2), 2u << (sh + 2), one);
          const float m2 = kab_blank_sel(t2, t1, th1, w, 1u << (sh + 4), 2u << (sh + 4), one);
          const float m3 = kab_label_sel(b0, b1, b2, b3, w, 1u << (sh + 6), 2u << (sh + 6), one);
          s0 = n0; s1 = m1; s2 = m2; s3 = m3;
        };
        // CTC: select on the previous scores, then one add; only h1 comes from the lane below
        auto frame_ctc = [&](const float xb, const float x1, const float x3, uint32_t &w, const int sh) {
          const float h1 = __shfl_up_sync(KAB_FULL_MASK, s3, 1);
          const float n0 = __fadd_rn(kab_ctc_blank_sel(s0, h1, w, sh + 0), xb);
          const float n1 = __fadd_rn(kab_ctc_label_sel(s1, s0, rep & 1u ? ninf : h1, w, sh + 2), x1);
          const float n2 = __fadd_rn(kab_ctc_blank_sel(s2, s1, w, sh + 4), xb);
          const float n3 = __fadd_rn(kab_ctc_label_sel(s3, s2, rep & 2u ? ninf : s1, w, sh + 6), x3);
          s0 = n0; s1 = n1; s2 = n2; s3 = n3;
        };

        // ---- build the wavefront: wait until the warp below is KAB_WD_LAG groups ahead (its message
        // KAB_WD_LAG - 1 has landed); both then run at the same pace and the lag stays
        if (has_below && n_groups - 1 >= KAB_WD_LAG && !owned) {
          const unsigned char *slot = inbox + (size_t)((KAB_WD_LAG - 1) % D) * KAB_WD_MSG_BYTES;
          while (kab_ld_volatile_b64(slot + 24).y != (uint32_t)KAB_WD_LAG) __nanosleep(64);
        }
        __syncwarp();
#ifdef KAB_WIDE_TIMING
        long long tm_ghost = 0, tm_emis = 0, tm_comp = 0, tm_pub = 0, tm_rest = 0, n_miss = 0;
        const long long tm_start = clock64();
#endif
        for (int g = 0; g < n_groups; ++g) {
          const int i0 = g * G, nfr = min(G, T - i0);
          const bool more = i0 + G < T;
          KAB_WTM(ta);
          // ---- ghost lanes: message g-1 of the warp below (its top 24 states after its group g-1)
          if (g > 0 && !owned) {
            if (has_below) {
              const unsigned char *slot = inbox + (size_t)((g - 1) % D) * KAB_WD_MSG_BYTES;
              const uint32_t seq = (uint32_t)g;
#ifdef KAB_WIDE_TIMING
              if (lane == 0 && (pf0.y != seq || pf1.y != seq || pf2.y != seq || pf3.y != seq)) ++n_miss;
#endif
              while (pf0.y != seq || pf1.y != seq || pf2.y != seq || pf3.y != seq) {
                pf0 = kab_ld_volatile_b64(slot);
                pf1 = kab_ld_volatile_b64(slot + 8);
                pf2 = kab_ld_volatile_b64(slot + 16);
                pf3 = kab_ld_volatile_b64(slot + 24);
              }
              s0 = __uint_as_float(pf0.x); s1 = __uint_as_float(pf1.x);
              s2 = __uint_as_float(pf2.x); s3 = __uint_as_float(pf3.x);
            } else {
              s0 = ninf; s1 = ninf; s2 = ninf; s3 = ninf;  // below state 0
            }
          }
          __syncwarp();
          if (has_below && g > 0 && lane == 0) kab_st_volatile_u32(&cons[gw], (uint32_t)g);  // g messages consumed
          // message g (needed at the next group) may already be there: load it now, check it then
          if (has_below && more && !owned) {
            const unsigned char *slot = inbox + (size_t)(g % D) * KAB_WD_MSG_BYTES;
            pf0 = kab_ld_volatile_b64(slot);
            pf1 = kab_ld_volatile_b64(slot + 8);
            pf2 = kab_ld_volatile_b64(slot + 16);
            pf3 = kab_ld_volatile_b64(slot + 24);
          }
          KAB_WTM(tb);
          const bool next_crosses = fic + G == F;
          const uint32_t nst = st + 1 == NS ? 0 : st + 1;
          const uint32_t nph = nst == 0 ? ph ^ 1u : ph;
          if (next_crosses && more) kab_mbar_spin(&efull[nst], nph);
          KAB_WTM(tc);
          const char *rowng = next_crosses ? chunk_ptr(nst) : rowc + G * VB;
          if (more) load_group(rowng, nb, n1, n3);
          uint32_t wlo = 0, whi = 0;
          if (nfr == G) {
#pragma unroll
            for (int f = 0; f < G; ++f) {
              if (CTC) frame_ctc(eb[f], e1[f], e3[f], f < 4 ? wlo : whi, 8 * (f & 3));
              else frame(eb[f], e1[f], e3[f], f < 4 ? wlo : whi, 8 * (f & 3));
            }
          } else {
#pragma unroll
            for (int f = 0; f < G; ++f)
              if (f < nfr) {
                if (CTC) frame_ctc(eb[f], e1[f], e3[f], f < 4 ? wlo : whi, 8 * (f & 3));
                else frame(eb[f], e1[f], e3[f], f < 4 ? wlo : whi, 8 * (f & 3));
              }
          }
          KAB_WTM(td);
          // ---- message g for the warp above: (score, seq) pairs, one 8-byte store each
          if (more && has_above) {
            if (g >= D && (uint32_t)(g - D) >= cons_seen) {  // about to lap the consumer: read its progress
              do {
                cons_seen = kab_ld_volatile_u32(&cons[gw + 1]);
              } while ((uint32_t)(g - D) >= cons_seen);
            }
            if (lane >= 32 - GH) {
              unsigned char *slot = outbox + (size_t)(g % D) * KAB_WD_MSG_BYTES;
              const uint32_t seq = (uint32_t)(g + 1);
              kab_st_volatile_b64(slot, __float_as_uint(s0), seq);
              kab_st_volatile_b64(slot + 8, __float_as_uint(s1), seq);
              kab_st_volatile_b64(slot + 16, __float_as_uint(s2), seq);
              kab_st_volatile_b64(slot + 24, __float_as_uint(s3), seq);
            }
          }
          KAB_WTM(te);
          // ---- backpointer word of this group -> staging; block finished?
          if (owned) *reinterpret_cast<uint2 *>(bpbuf + ((blk & 1) * FBW + fib) * 32 + (lane - GH) * 8) = make_uint2(wlo, whi);
          fib += G;
          if (fib >= FBW || !more) {
            __syncwarp();
            if (lane == 0) {
              kab_fence_proxy_async();
              kab_bulk_s2g(bpg + (size_t)blk * FBW * 32, bpbuf + (size_t)(blk & 1) * FBW * 32, (uint32_t)fib * 32u);
              kab_bulk_wait_read1();
            }
            __syncwarp();
            ++blk;
            fib = 0;
          }
#pragma unroll
          for (int f = 0; f < G; ++f) { eb[f] = nb[f]; e1[f] = n1[f]; e3[f] = n3[f]; }
          rowc = rowng;
          if (next_crosses || !more) {
            __syncwarp();
            if (lane == 0) kab_mbar_arrive(&eempty[st]);
            st = nst; ph = nph;
            fic = 0;
          } else {
            fic += G;
          }
#ifdef KAB_WIDE_TIMING
          {
            const long long tf = clock64();
            tm_ghost += tb - ta; tm_emis += tc - tb; tm_comp += td - tc; tm_pub += te - td; tm_rest += tf - te;
          }
#endif
        }
#ifdef KAB_WIDE_TIMING
        if (lane == 0 && p.debug && (gw < 4 || gw == nww / 2 || gw == nww - 1)) {
          long long *d = p.debug + (gw < 4 ? gw : (gw == nww / 2 ? 4 : 5)) * 8;
          d[0] = tm_ghost; d[1] = tm_emis; d[2] = tm_comp; d[3] = tm_pub; d[4] = tm_rest; d[5] = n_miss;
          d[6] = clock64() - tm_start; d[7] = n_groups;
        }
#endif
        // ---- this warp's highest active state and its score (align.py:99-101), then "finished"
        int cand = -1;
        float cs = 0.0f;
        if (CTC) {  // the scores of the two end states S-1 -> ctl[3], S-2 -> ctl[0] (end rule: backtrack CTA)
          if (owned) {
            if (vb + 0 == S - 1) ctl[3] = __float_as_uint(s0);
            if (vb + 2 == S - 1) ctl[3] = __float_as_uint(s2);
            if (vb + 1 == S - 2) ctl[0] = __float_as_uint(s1);
            if (vb + 3 == S - 2) ctl[0] = __float_as_uint(s3);
          }
        } else if (owned) {
          if (vb + 0 < S && s0 > ninf) { cand = vb + 0; cs = s0; }
          if (vb + 1 < S && s1 > ninf) { cand = vb + 1; cs = s1; }
          if (vb + 2 < S && s2 > ninf) { cand = vb + 2; cs = s2; }
          if (vb + 3 < S && s3 > ninf) { cand = vb + 3; cs = s3; }
        }
        const int wcand = __reduce_max_sync(KAB_FULL_MASK, cand);  // (CTC: -1)
        if (cand >= 0 && cand == wcand) {
          int2 *cp = reinterpret_cast<int2 *>(ws + kab_wide_cand_off()) + gw;
          *cp = make_int2(cand, __float_as_int(cs));
        }
        __syncwarp();
        if (lane == 0) {
          if (wcand >= 0) atomicMax(&ctl[0], (unsigned int)(wcand + 1));
          kab_bulk_wait0();  // this warp's backpointer blocks are in global memory
          __threadfence();
          atomicAdd(&ctl[2], 1u);
        }
      }
      echunks = ec0 + (uint32_t)n_chunks;
      __syncwarp();
    }
    return;
  }

  // =========================================================== backtrack CTA
  uint32_t bt_use0 = 0, bt_use1 = 0;  // completed phases of the two block barriers (thread 0)
  for (int li = 0; li < n_lat; ++li) {
    const KabLattice lat = lats[li];
    const int nww = lat.k, T = lat.T;
    const int n_groups = (T + G - 1) / G;
    unsigned char *ws = wide_ws + (size_t)lat.scr_off * 4;
    unsigned int *ctl = reinterpret_cast<unsigned int *>(ws);
    if (tid == 0) {
      unsigned int done;
      for (;;) {
        asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(done) : "l"(&ctl[2]) : "memory");
        if (done >= (unsigned int)nww) break;
        __nanosleep(500);
      }
      if (CTC) {  // end rule: S-1 if a[S-1] > a[S-2], else S-2 (a tie, and two -inf, pick S-2)
        const int S = 2 * lat.L + 1;
        const float a1 = __uint_as_float(kab_ld_volatile_u32(&ctl[3])), a2 = __uint_as_float(kab_ld_volatile_u32(&ctl[0]));
        const int v = a1 > a2 ? S - 1 : S - 2;
        const int status = kab_ld_volatile_u32(&ctl[1]) ? 3 : 0;
        s_v = v;
        s_status = status;
        p.status[lat.index] = status;
        if (p.final_score) p.final_score[lat.index] = status == 0 ? (a1 > a2 ? a1 : a2) : __int_as_float(0x7fc00000);
      } else {
        const int v = (int)kab_ld_volatile_u32(&ctl[0]) - 1;
        const int status = kab_ld_volatile_u32(&ctl[1]) ? 3 : (v < 0 ? 1 : 0);
        s_v = v;
        s_status = status;
        p.status[lat.index] = status;
        if (p.final_score) {
          float fs = __int_as_float(0x7fc00000);
          if (status == 0) fs = __int_as_float(reinterpret_cast<const int2 *>(ws + kab_wide_cand_off())[v / OW].y);
          p.final_score[lat.index] = fs;
        }
      }
    }
    __syncthreads();
    int v = s_v;
    if (s_status == 0) {
      const int NT = KAB_WD_THREADS;
      const uint16_t *col16 = p.col16 + lat.col_off;
      const unsigned char *bp = p.bp + lat.bp_off;
      const int n_blocks = (T + FBK - 1) / FBK;
      int32_t *out_path = p.best_path + lat.t_off;
      int32_t *out_lab = p.best_labels + lat.t_off;
      float *out_sc = p.best_scores + lat.t_off;
      const float *lp = p.lp + lat.t_off * (int64_t)V;
      constexpr int RSZ = FBK * 32;
      // block `b` of warp regions wtop, wtop-1, wtop-2 (clamped at region 0) -> buffer `buf` (thread 0)
      auto fetch = [&](int b, int wtop, int buf) {
        const int ng = (min(FBK, T - b * FBK) + G - 1) / G;
        const uint32_t bytes = (uint32_t)ng * 256u;
        kab_mbar_expect_tx(&btbar[buf], bytes * NREG);
        for (int j = 0; j < NREG; ++j) {
          const int reg = max(wtop - j, 0);
          kab_bulk_g2s(btbuf + ((size_t)buf * NREG + j) * RSZ, bp + ((size_t)reg * n_groups + (size_t)b * (FBK / G)) * 256,
                       bytes, &btbar[buf]);
        }
      };
      auto flush_block = [&](int b, int first_thread, int n_threads) {
        const int i0 = b * FBK, i1 = min(T, i0 + FBK);
        const int *pbuf = pathbuf + (b & 1) * FBK;
        for (int i = i0 + (tid - first_thread); i < i1; i += n_threads) {
          const int pv = pbuf[i - i0];
          const int lab = (pv & 1) ? (int)col16[(pv - 1) >> 1] : (CTC ? blank : 0);
          out_path[i] = pv;
          out_lab[i] = lab;                              // align.py:106
          out_sc[i] = __ldg(&lp[(int64_t)i * V + lab]);  // align.py:107
        }
      };
      int wreg = v / OW;               // warp region of the walker's state
      int wtop0 = wreg, wtop1 = wreg;  // top region staged in buffer 0 / 1
      if (tid == 0) fetch(n_blocks - 1, wreg, (n_blocks - 1) & 1);
      for (int b = n_blocks - 1; b >= 0; --b) {
        const int buf = b & 1;
        const int i0 = b * FBK, i1 = min(T, i0 + FBK);
        if (tid == 0) {
          if (b > 0) {
            if (buf) wtop0 = wreg; else wtop1 = wreg;
            fetch(b - 1, wreg, buf ^ 1);
          }
          kab_mbar_wait(&btbar[buf], (buf ? bt_use1 : bt_use0) & 1u);
          if (buf) ++bt_use1; else ++bt_use0;
          int jreg = (buf ? wtop1 : wtop0) - wreg;
          auto restage = [&]() {
            if (buf) wtop1 = wreg; else wtop0 = wreg;
            fetch(b, wreg, buf);
            kab_mbar_wait(&btbar[buf], (buf ? bt_use1 : bt_use0) & 1u);
            if (buf) ++bt_use1; else ++bt_use0;
            jreg = 0;
          };
          if (jreg >= NREG) restage();
          int *pbuf = pathbuf + buf * FBK;
          const unsigned char *rows = btbuf + ((size_t)buf * NREG + jreg) * RSZ;
          int col = (v - wreg * OW) >> 2, k2 = 2 * (v & 3);  // byte column of the walker, bit offset in it
          // Full groups are walked from registers (kab_walk_group8 in kab_band.cuh: two 64-bit loads
          // per group, loaded a group early, and a branch-free 8-frame body); what it leaves takes the
          // generic step, which also handles the step into the warp region below.
          auto step_column = [&]() {
            if (--col < 0) {
              --wreg;
              if (++jreg == NREG) restage();
              rows = btbuf + ((size_t)buf * NREG + jreg) * RSZ;
              col = (OW >> 2) - 1;
            }
          };
          uint2 pw0 = make_uint2(0u, 0u), pw1 = pw0;
          const unsigned char *pfrom = nullptr;
          for (int gq = (i1 - 1 - i0) >> 3; gq >= 0; --gq) {
            int f = min(7, i1 - 1 - i0 - gq * 8);
            int *pg = pbuf + gq * 8;
            if (f == 7) {
              const unsigned char *grow = rows + gq * 256;
              const bool have1 = col > 0 || (jreg + 1 < NREG && wreg > 0);
              const unsigned char *c0 = grow + col * 8;
              const unsigned char *below = col > 0 ? c0 - 8 : grow + RSZ + ((OW >> 2) - 1) * 8;
              uint2 w0, w1;
              if (pfrom == c0) {
                w0 = pw0; w1 = pw1;
              } else {
                w0 = *reinterpret_cast<const uint2 *>(c0);
                w1 = have1 ? *reinterpret_cast<const uint2 *>(below) : make_uint2(0u, 0u);
              }
              if (gq > 0) {
                pw0 = *reinterpret_cast<const uint2 *>(c0 - 256);
                pw1 = have1 ? *reinterpret_cast<const uint2 *>(below - 256) : make_uint2(0u, 0u);
                pfrom = c0 - 256;
              }
              int nchg;
              f = kab_walk_group8(w0, w1, have1, v, k2, pg, nchg);
              for (int c = 0; c < nchg; ++c) step_column();
            }
            for (; f >= 0; --f) {  // generic step
              const unsigned int byte = rows[gq * 256 + col * 8 + f];
              pg[f] = v;
              const int mv = (int)((byte >> k2) & 3u);
              v -= mv;
              k2 -= 2 * mv;
              if (k2 < 0) {
                k2 += 8;
                step_column();
              }
            }
          }
        } else if (tid >= 32 && b + 1 < n_blocks) {
          flush_block(b + 1, 32, NT - 32);
        }
        __syncthreads();
      }
      flush_block(0, 0, NT);
    }
    __syncthreads();
  }
}

__global__ void __launch_bounds__(KAB_WD_THREADS, 1)
    kab_wide_kernel(const KabLattice *__restrict__ lats, int n_lat, KabParams p, unsigned char *wide_ws) {
  kab_wide_body<false>(lats, n_lat, p, wide_ws, 0);
}

// CTC forced alignment (blank column: see kab_warp_ctc_kernel)
__global__ void __launch_bounds__(KAB_WD_THREADS, 1)
    kab_wide_ctc_kernel(const KabLattice *__restrict__ lats, int n_lat, KabParams p, unsigned char *wide_ws, int blank) {
  kab_wide_body<true>(lats, n_lat, p, wide_ws, blank);
}
