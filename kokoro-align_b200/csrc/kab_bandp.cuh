// kab_bandp.cuh -- chapter-length lattices with the reference's diagonal band (align.py:64-65),
// one thread-block CLUSTER per lattice, every warp on its own SM sub-partition, no barrier on
// the recurrence.  Same shapes as kab_band.cuh (max_move = 4, labels in 1..V-1, V <= 512,
// S <= 3T) with min(beam_size, S) + 32 <= R = 104 * NWT ring slots, NWT = 4 * NC compute warps
// in a cluster of NC <= 8 CTAs.
//
// The single-CTA kernel (kab_band.cuh) is issue-bound: ten warps share four schedulers and
// meet at a CTA barrier every 8 frames.  Here
//   * a CTA runs FOUR compute warps (one per scheduler) and one producer warp; a lattice with
//     the 1000-wide band spreads over 3 SMs.  State v lives in ring slot v mod R; warp gw owns
//     slots 104 gw .. 104 gw + 103 in registers (4 states per lane, lanes 6..31), lanes 0..5 are
//     ghost lanes that recompute the lower neighbour's top 24 states for 8 frames (same scheme
//     and same exactness argument as kab_band.cuh);
//   * there is NO group barrier.  After each 8-frame group a warp hands its top six lanes to
//     the warp above through a FIFO in GLOBAL memory (L2): every score is stored together with
//     the message's sequence number as one 8-byte store (single-copy atomic), so there is no
//     fence, no flag and no mbarrier on the recurrence; the consumer's ghost lanes load message
//     g at the start of group g and check it at the start of group g+1 (kab_wide.cuh uses the
//     same scheme).  The first version used st.async + mbarriers over DSMEM: every mbarrier
//     round trip costs a lone warp 100-250 cycles and the ring ran in lockstep (DESIGN.md 3.3).
//     A warp whose 24 ghost states are outside the window does not look at its messages at all,
//     so the ring is a chain whose head runs free, and a warp that (re)joins the chain first
//     waits until its neighbour is two groups ahead: the wavefront that hides the L2 latency;
//   * emission rows are staged per CTA by the producer warp: an 8-stage ring of 1-D bulk
//     copies with full (complete_tx) / empty (4 arrivals) mbarriers, so the four compute warps
//     may be several groups apart;
//   * the emissions of a whole group (3 per frame and lane) are loaded into registers one
//     group ahead, so no shared-memory load sits on the recurrence; the finiteness check of the
//     staged rows is done by the otherwise idle producer warp;
//   * backpointers: one byte (4 cells x 2 bits) per owned lane and frame, accumulated in two
//     registers per group and staged per WARP as [group][lane][8 frames] (one STS.64 per group),
//     written with bulk stores to the warp's own region [gw][group][32 lanes][8 B] of the
//     workspace: the walker finds the 8 frames of a group in one 64-bit word;
//   * the forced end state is a cluster-wide max (remote shared-memory reductions), then CTA 0
//     backtracks: the walk follows one warp region for hundreds of frames, so a block of 128
//     frames of the current region and the two below it is staged by bulk copies (double
//     buffered); the other warps write the previous block's outputs.
#pragma once
#include "kab_band.cuh"  // KAB_BAND_G / GHOST / OW: the lanes of kab_band.cuh; kab_walk_group8
#include "kab_common.cuh"

#define KAB_BP_CW 4      // compute warps per CTA
#define KAB_BP_NS 16     // emission stages per CTA (the four warps of a CTA may be ~12 groups apart)
#define KAB_BP_D 64      // neighbour FIFO depth (messages, global memory)
#define KAB_BP_LAG 2     // a warp joining the chain waits until its lower neighbour is this many groups ahead
#define KAB_BP_FBW 256   // frames per per-warp backpointer block
#define KAB_BP_FBK 128   // frames per backtrack block
#define KAB_BP_NREG 3    // warp regions staged per backtrack block
#define KAB_BP_MSG_BYTES (KAB_BAND_GHOST * 32)  // 6 lanes x 4 (score, seq) pairs
#define KAB_BP_THREADS ((KAB_BP_CW + 1) * 32)

struct KabBandpGeom {
  size_t bpst_off, bt_off, path_off, stage_off, smem_bytes;
};
__host__ __device__ inline KabBandpGeom kab_bandp_geom(int stage_bytes) {
  KabBandpGeom g;
  g.bpst_off = 384;  // after the mbarriers (2 * NS + 2) and the CTA scalars
  g.bt_off = g.bpst_off + (size_t)KAB_BP_CW * 2 * KAB_BP_FBW * 32;
  g.path_off = g.bt_off + (size_t)2 * KAB_BP_NREG * KAB_BP_FBK * 32;
  g.stage_off = g.path_off + (size_t)2 * KAB_BP_FBK * 4;
  g.smem_bytes = g.stage_off + (size_t)KAB_BP_NS * stage_bytes;
  return g;
}

// Bytes of the global scratch of one lattice (layout: kab_cluster_fifo_off)
__host__ __device__ inline size_t kab_bandp_ws_bytes(int nwt) {
  return kab_cluster_fifo_off(nwt) + (size_t)nwt * KAB_BP_D * KAB_BP_MSG_BYTES;
}

#ifdef KAB_BANDP_TIMING
#define KAB_TM(var) const long long var = clock64()
#define KAB_TM_ADD(acc, a, b) acc += (b) - (a)
#else
#define KAB_TM(var)
#define KAB_TM_ADD(acc, a, b)
#endif

__global__ void __launch_bounds__(KAB_BP_THREADS, 1)
    kab_bandp_kernel(const KabLattice *__restrict__ lats, int n_lat, KabParams p) {
  constexpr int G = KAB_BAND_G, GH = KAB_BAND_GHOST, OW = KAB_BAND_OW;
  constexpr int CW = KAB_BP_CW, NS = KAB_BP_NS, D = KAB_BP_D, FBW = KAB_BP_FBW, FBK = KAB_BP_FBK,
                NREG = KAB_BP_NREG;
  static_assert(G == 8, "a group of 8 frames is one 64-bit backpointer word per lane");
  const KabBandpGeom geo = kab_bandp_geom(p.stage_bytes);
  extern __shared__ __align__(128) unsigned char kab_smem[];
  uint64_t *efull = reinterpret_cast<uint64_t *>(kab_smem);        // [NS]
  uint64_t *eempty = efull + NS;                                   // [NS]
  uint64_t *btbar = eempty + NS;                                   // [2]
  unsigned int *s_item = reinterpret_cast<unsigned int *>(btbar + 2);
  int *s_vmax = reinterpret_cast<int *>(s_item + 1);
  unsigned int *s_bad = s_item + 2;
  unsigned char *btbuf = kab_smem + geo.bt_off;                     // [2][NREG][FBK * 32]
  int *pathbuf = reinterpret_cast<int *>(kab_smem + geo.path_off);  // [2][FBK]
  float *stage_base = reinterpret_cast<float *>(kab_smem + geo.stage_off);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t rank = kab_cluster_rank(), NC = kab_cluster_size();
  const int NWT = CW * (int)NC, R = OW * NWT;
  const bool is_prod = warp == CW;
  const int gw = (int)rank * CW + warp;  // global compute-warp index (meaningless for the producer)
  const int ngw = (gw + 1) % NWT;
  const bool owned = lane >= GH;
  const int slot0 = owned ? OW * gw + 4 * (lane - GH) : (OW * gw - 4 * GH + 4 * lane + R) % R;
  const float ninf = kab_neg_inf();

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
  uint32_t echunks = 0;          // emission chunks staged so far by this CTA (same count in every warp)
  uint32_t bt_uses[2] = {0, 0};  // completed phases of the two backtrack barriers (thread 0)

  for (;;) {
    // ---- the cluster agrees on the next work item
    if (tid == 0) {
      *s_vmax = -1;
      *s_bad = 0u;
    }
    if (rank == 0 && tid == 0) {
      const unsigned int it = atomicAdd(p.queue, 1u);
      for (uint32_t r = 0; r < NC; ++r) kab_st_cluster_u32(kab_mapa(kab_smem_u32(s_item), r), it);
    }
    __syncwarp();
    kab_cluster_sync();
    const unsigned int item = *s_item;
    if (item >= (unsigned int)n_lat) break;
    const KabLattice lat = lats[item];
    const int T = lat.T, S = 2 * lat.L + 1, V = p.V, W = p.W;
    const int F = p.stage_frames;
    const uint32_t stage_words = p.stage_bytes >> 2;
    const int n_chunks = (T + F - 1) / F;
    const int n_groups = (T + G - 1) / G;
    const uint32_t ec0 = echunks;
    const uint32_t skew = (uint32_t)(((lat.t_off * (int64_t)V * 4) & 15) >> 2);
    float s0 = ninf, s1 = ninf, s2 = ninf, s3 = ninf;
    int vb = slot0;

    if (is_prod) {
      // ================= producer warp: emission ring + finiteness of the staged rows
      const char *lp_base = reinterpret_cast<const char *>(p.lp) + ((lat.t_off * (int64_t)V * 4) & ~(int64_t)15);
      const uint32_t chunk_stride = (uint32_t)(F * V * 4);
      const uint32_t full_bytes = (chunk_stride + skew * 4 + 15) & ~15u;
      float poison = 0.0f;
      auto check_chunk = [&](int c) {  // waits for chunk c, then scans it (the compute warps may be reading it too)
        const uint32_t gc = ec0 + (uint32_t)c, stg = gc % NS;
        kab_mbar_wait(&efull[stg], (gc / NS) & 1u);
        const float *w = stage_base + stg * stage_words + skew;
        const int nw = min(F, T - c * F) * V;
        for (int j = lane; j < nw; j += 32) poison = kab_poison(poison, w[j]);
      };
      for (int c = 0; c < n_chunks; ++c) {
        const uint32_t gc = ec0 + (uint32_t)c, stg = gc % NS, use = gc / NS;
        // the chunk that used this stage was scanned (below) before the stage is given away
        if (c >= NS) check_chunk(c - NS);
        if (use > 0) kab_mbar_wait(&eempty[stg], (use - 1u) & 1u);  // all four compute warps released it
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
            kab_mbar_expect_tx(&efull[stg], d.bytes);  // (release: the tail words above are ordered before it)
            if (d.bytes) kab_bulk_g2s(dst, d.src, d.bytes, &efull[stg]);
          }
        }
        __syncwarp();
      }
      for (int c = max(0, n_chunks - NS); c < n_chunks; ++c) check_chunk(c);
      if (__any_sync(KAB_FULL_MASK, poison != poison) && lane == 0)
        for (uint32_t rr = 0; rr < NC; ++rr) kab_red_or_cluster_u32(kab_mapa(kab_smem_u32(s_bad), rr), 1u);
    } else {
      // ================= compute warp
      const uint16_t *col16 = p.col16 + lat.col_off;
      const uint32_t one = p.one;
      if (owned && slot0 == 0) s0 = 0.0f;  // virtual start state 0, score 0 (align.py:57-58)
      auto load_cols = [&](int base, uint32_t &ca, uint32_t &cb) {
        ca = base + 1 < S ? 4u * col16[base >> 1] : 0u;
        cb = base + 3 < S ? 4u * col16[(base >> 1) + 1] : 0u;
      };
      uint32_t c1, c3, nc1, nc3;
      load_cols(vb, c1, c3);
      load_cols(vb + R, nc1, nc3);
      const int half = W / 2;
      const int VB = V * 4;

      uint32_t st = ec0 % NS, ph = (ec0 / NS) & 1u;  // stage / phase of the chunk being read
      auto chunk_ptr = [&](uint32_t stg) { return reinterpret_cast<const char *>(stage_base + stg * stage_words + skew); };
      // emissions of a whole group, in registers: blank, first label, second label of this lane
      float eb[G], e1[G], e3[G], nb[G], n1[G], n3[G];
      auto load_group = [&](const char *row, float (&xb)[G], float (&x1)[G], float (&x3)[G]) {
#pragma unroll
        for (int f = 0; f < G; ++f) {
          xb[f] = *reinterpret_cast<const float *>(row + f * VB);
          x1[f] = *reinterpret_cast<const float *>(row + f * VB + c1);
          x3[f] = *reinterpret_cast<const float *>(row + f * VB + c3);
        }
      };
      kab_mbar_spin(&efull[st], ph);
      const char *rowc = chunk_ptr(st);  // first row of the current group
      load_group(rowc, eb, e1, e3);

      const int qd = S / T, rd = S % T;
      const int qdg = (int)(((int64_t)S * G) / T), rdg = (int)(((int64_t)S * G) % T);
      int qg = 0, rg = 0, q = 0, r = 0;

      // backpointers: per-warp staging [2][FBW / 8 groups][32 lanes][8 B]
      unsigned char *bpbuf = kab_smem + geo.bpst_off + (size_t)warp * 2 * FBW * 32;
      unsigned char *bpg = p.bp + lat.bp_off + (size_t)gw * n_groups * 256;  // this warp's region of the workspace
      int fib = 0, blk = 0;
      uint32_t wlo = 0, whi = 0;  // backpointer bytes of frames 0..3 / 4..7 of the current group

      // One frame; sh = bit offset of this frame's byte in the backpointer word w.  The window of
      // align.py:64-65 never appears here: a cell outside [lo, hi) is made inactive through its
      // EMISSION (-inf: every candidate is -inf, so the maximum is), and the masked emissions of an
      // edge warp are prepared per group, off the recurrence chain.  xb0 / xb2 are the blank
      // emissions of this lane's states 0 / 2 (the same value inside the window).
      auto frame = [&](const float xb0, const float xb2, const float x1, const float x3, uint32_t &w, const int sh) {
        const float h1 = __shfl_up_sync(KAB_FULL_MASK, s3, 1);
        const float h2 = __shfl_up_sync(KAB_FULL_MASK, s2, 1);
        const float h3 = __shfl_up_sync(KAB_FULL_MASK, s1, 1);
        float t0, t1;
        kab_add2v(s0, s1, xb0, xb2, t0, t1);  // state 0 <- 0 (move 0), state 2 <- 1 (move 1)
        const float t2 = __fadd_rn(s2, xb2);
        const float th1a = __fadd_rn(h1, xb0), th1b = __fadd_rn(h1, xb2), th3 = __fadd_rn(h3, xb0);
        float a0, a1, a2, a3, b0, b1, b2, b3;
        kab_add2(s0, s1, x1, a1, a0);
        kab_add2(h2, h1, x1, a3, a2);
        kab_add2(s2, s3, x3, b1, b0);
        kab_add2(s0, s1, x3, b3, b2);
        const float n0 = kab_blank_sel(t0, th1a, th3, w, 1u << (sh + 0), 2u << (sh + 0), one);
        const float m1 = kab_label_sel(a0, a1, a2, a3, w, 1u << (sh + 2), 2u << (sh + 2), one);
        const float m2 = kab_blank_sel(t2, t1, th1b, w, 1u << (sh + 4), 2u << (sh + 4), one);
        const float m3 = kab_label_sel(b0, b1, b2, b3, w, 1u << (sh + 6), 2u << (sh + 6), one);
        s0 = n0; s1 = m1; s2 = m2; s3 = m3;
      };

      int fic = 0;  // frame offset of the current group inside its emission chunk
      int lo_prev = 0;            // lo of the first frame of the previous group (<= lo of every later frame)
      // neighbour FIFO in global memory: my inbox (messages of warp pgw) and the inbox of warp ngw
      unsigned char *gws = p.fifo + (size_t)lat.scr_off * 4;
      unsigned int *cons = reinterpret_cast<unsigned int *>(gws);
      unsigned char *gfifo = gws + kab_cluster_fifo_off(NWT);
      const unsigned char *inbox = gfifo + (size_t)gw * D * KAB_BP_MSG_BYTES + (lane < GH ? lane : 0) * 32;
      unsigned char *outbox = gfifo + (size_t)ngw * D * KAB_BP_MSG_BYTES + (lane >= 32 - GH ? lane - (32 - GH) : 0) * 32;
      uint32_t cons_seen = 0;      // messages the warp above is known to be done with
      bool was_needed = false;     // the previous group read its message (the warp is inside the chain)
      uint2 pf0 = make_uint2(0, 0), pf1 = pf0, pf2 = pf0, pf3 = pf0;  // message g-1, loaded a group early
#ifdef KAB_BANDP_TIMING
      long long tm_ghost = 0, tm_emis = 0, tm_comp = 0, tm_pub = 0, tm_rel = 0, tm_bp = 0, tm_guard = 0, n_need = 0, n_safe = 0, tm_wait = 0, n_first = 0, tm_slow = 0;
      const long long tm_start = clock64();
#endif
      for (int g = 0; g < n_groups; ++g) {
        const int i0 = g * G, nfr = min(G, T - i0);
        const bool more = i0 + G < T;
        KAB_TM(ta);
        // ---- ghost lanes: the lower neighbour's top 24 states after its group g-1 (message g-1).
        // Every message is armed (its phase must complete) and its slot returned, but the warp only
        // WAITS for it when the ghost states can matter: if all 24 were outside the window at frame
        // 8g-1 and stay outside during this group they are inactive (-inf) by definition.  At least
        // one warp boundary of the ring is always in that situation, so the ring is a chain whose
        // head never waits and the others find their messages already delivered.
        if (g > 0) {
          int qn2 = qg + qdg;
          if (rg + rdg >= T) ++qn2;
          const int hi1g = min(max(0, qn2 - half) + W, S);  // >= hi of every frame of this group
          const bool outside = owned || vb + 3 < lo_prev || vb >= hi1g;
          const bool need = !__all_sync(KAB_FULL_MASK, outside);
#ifdef KAB_BANDP_TIMING
          n_need += need;
          const long long tw0 = clock64();
#endif
          if (need) {
            if (!owned) {
              if (!was_needed) {  // (re)joining the chain: let the warp below get KAB_BP_LAG groups ahead
                const int mt = min(g - 1 + KAB_BP_LAG - 1, n_groups - 2);
                const unsigned char *ls = inbox + (size_t)(mt % D) * KAB_BP_MSG_BYTES;
                while (kab_ld_volatile_b64(ls + 24).y != (uint32_t)(mt + 1)) __nanosleep(64);
              }
              const unsigned char *slot = inbox + (size_t)((g - 1) % D) * KAB_BP_MSG_BYTES;
              const uint32_t seq = (uint32_t)g;
              while (pf0.y != seq || pf1.y != seq || pf2.y != seq || pf3.y != seq) {
                pf0 = kab_ld_volatile_b64(slot);
                pf1 = kab_ld_volatile_b64(slot + 8);
                pf2 = kab_ld_volatile_b64(slot + 16);
                pf3 = kab_ld_volatile_b64(slot + 24);
              }
              s0 = __uint_as_float(pf0.x); s1 = __uint_as_float(pf1.x);
              s2 = __uint_as_float(pf2.x); s3 = __uint_as_float(pf3.x);
            }
          } else if (!owned) {
            s0 = ninf; s1 = ninf; s2 = ninf; s3 = ninf;
          }
          was_needed = need;
          __syncwarp();
          if (lane == 0) kab_st_volatile_u32(&cons[gw], (uint32_t)g);  // done with messages 0 .. g-1
#ifdef KAB_BANDP_TIMING
          tm_wait += clock64() - tw0;
#endif
        }
        // message g (for the next group) may already be there: load it now, check it then
        if (more && !owned) {
          const unsigned char *slot = inbox + (size_t)(g % D) * KAB_BP_MSG_BYTES;
          pf0 = kab_ld_volatile_b64(slot);
          pf1 = kab_ld_volatile_b64(slot + 8);
          pf2 = kab_ld_volatile_b64(slot + 16);
          pf3 = kab_ld_volatile_b64(slot + 24);
        }
        lo_prev = max(0, qg - half);
        KAB_TM(tb);
        KAB_TM_ADD(tm_ghost, ta, tb);
        const bool next_crosses = fic + G == F;
        const uint32_t nst = st + 1 == NS ? 0 : st + 1;
        const uint32_t nph = nst == 0 ? ph ^ 1u : ph;
        // the next group's emissions are loaded during this group
        if (next_crosses && more) kab_mbar_spin(&efull[nst], nph);
        KAB_TM(tc);
        KAB_TM_ADD(tm_emis, tb, tc);
        const char *rowng = next_crosses ? chunk_ptr(nst) : rowc + G * VB;
        const int lo0 = max(0, qg - half), hi0 = min(lo0 + W, S);
        int qn = qg + qdg, rn = rg + rdg;
        if (rn >= T) { rn -= T; ++qn; }
        const int lo1 = max(0, qn - half);
        if (vb + 3 < lo0 - 3) {  // recycle a chunk that fell below the window (between groups only)
          do {
            vb += R;
            c1 = nc1; c3 = nc3;
            load_cols(vb + R, nc1, nc3);
          } while (vb + 3 < lo0 - 3);
          load_group(rowc, eb, e1, e3);  // the prefetched emissions belonged to the old alias
        }
        if (more) load_group(rowng, nb, n1, n3);
        const bool safe = __all_sync(KAB_FULL_MASK, nfr == G && vb >= lo1 && vb + 4 <= hi0);
        wlo = 0; whi = 0;
#ifdef KAB_BANDP_TIMING
        n_safe += safe;
#endif
        if (safe) {
#pragma unroll
          for (int f = 0; f < G; ++f) frame(eb[f], eb[f], e1[f], e3[f], f < 4 ? wlo : whi, 8 * (f & 3));
        } else {
          // edge warp (or the last, partial group): the exact per-frame window (S*i = q*T + r, no
          // divisions) turned into masked emissions for the whole group
          q = qg; r = rg;
          float mb0[G], mb2[G], mm1[G], mm3[G];
#pragma unroll
          for (int f = 0; f < G; ++f) {
            const int lo = max(0, q - half);   // align.py:64
            const int hi = min(lo + W, S);     // align.py:65
            q += qd; r += rd;
            if (r >= T) { r -= T; ++q; }
            const unsigned a = (unsigned)(vb - lo), wd = (unsigned)(hi - lo);
            mb0[f] = (a + 0u < wd) ? eb[f] : ninf;
            mm1[f] = (a + 1u < wd) ? e1[f] : ninf;
            mb2[f] = (a + 2u < wd) ? eb[f] : ninf;
            mm3[f] = (a + 3u < wd) ? e3[f] : ninf;
          }
          if (nfr == G) {
#pragma unroll
            for (int f = 0; f < G; ++f) frame(mb0[f], mb2[f], mm1[f], mm3[f], f < 4 ? wlo : whi, 8 * (f & 3));
          } else {
#pragma unroll
            for (int f = 0; f < G; ++f)
              if (f < nfr) frame(mb0[f], mb2[f], mm1[f], mm3[f], f < 4 ? wlo : whi, 8 * (f & 3));
          }
        }
        qg = qn; rg = rn;
        KAB_TM(td);
        KAB_TM_ADD(tm_comp, tc, td);
#ifdef KAB_BANDP_TIMING
        if (!safe) tm_slow += td - tc;
#endif

        // ---- hand the top six lanes to the warp above (message g)
        if (more) {
          if (g >= D && (uint32_t)(g - D) >= cons_seen) {  // about to lap the consumer: read its progress
            do {
              cons_seen = kab_ld_volatile_u32(&cons[ngw]);
            } while ((uint32_t)(g - D) >= cons_seen);
          }
          if (lane >= 32 - GH) {
            unsigned char *slot = outbox + (size_t)(g % D) * KAB_BP_MSG_BYTES;
            const uint32_t seq = (uint32_t)(g + 1);
            kab_st_volatile_b64(slot, __float_as_uint(s0), seq);
            kab_st_volatile_b64(slot + 8, __float_as_uint(s1), seq);
            kab_st_volatile_b64(slot + 16, __float_as_uint(s2), seq);
            kab_st_volatile_b64(slot + 24, __float_as_uint(s3), seq);
          }
        }
        KAB_TM(te);
        KAB_TM_ADD(tm_pub, td, te);
        // ---- backpointer word of this group -> staging; block finished?
        if (owned) *reinterpret_cast<uint2 *>(bpbuf + ((blk & 1) * FBW + fib) * 32 + (lane - GH) * 8) = make_uint2(wlo, whi);
        fib += G;
        if (fib >= FBW || !more) {
          __syncwarp();
          if (lane == 0) {
            kab_fence_proxy_async();
            kab_bulk_s2g(bpg + (size_t)blk * FBW * 32, bpbuf + (size_t)(blk & 1) * FBW * 32, (uint32_t)fib * 32u);
            kab_bulk_wait_read1();  // the block before this one has left its buffer
          }
          __syncwarp();
          ++blk;
          fib = 0;
        }
        KAB_TM(tf);
        KAB_TM_ADD(tm_bp, te, tf);
        // ---- next group's emissions become current; emission chunk finished?
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
        KAB_TM(tg);
        KAB_TM_ADD(tm_rel, tf, tg);
      }
#ifdef KAB_BANDP_TIMING
      if (lane == 0 && p.debug) {
        long long *d = p.debug + gw * 16;
        d[0] = tm_ghost; d[1] = tm_emis; d[2] = tm_comp; d[3] = tm_pub; d[4] = tm_rel; d[5] = tm_bp;
        d[6] = clock64() - tm_start; d[7] = n_groups; d[8] = tm_guard; d[9] = n_need; d[10] = n_safe; d[11] = tm_wait; d[12] = n_first; d[13] = tm_slow;
      }
#endif
      // ---- end of the forward pass: cluster-wide forced end state (align.py:99-101)
      int cand = -1;
      if (owned) {
        if (vb + 0 < S && s0 > ninf) cand = vb + 0;
        if (vb + 1 < S && s1 > ninf) cand = vb + 1;
        if (vb + 2 < S && s2 > ninf) cand = vb + 2;
        if (vb + 3 < S && s3 > ninf) cand = vb + 3;
      }
      cand = __reduce_max_sync(KAB_FULL_MASK, cand);
      if (lane == 0) {
        if (cand >= 0)
          for (uint32_t rr = 0; rr < NC; ++rr) kab_red_max_cluster_s32(kab_mapa(kab_smem_u32(s_vmax), rr), cand);
        kab_bulk_wait0();  // this warp's backpointer blocks are in global memory
      }
    }
    echunks = ec0 + (uint32_t)n_chunks;
    __syncwarp();
    kab_cluster_sync();

    int v = *s_vmax;
    const int status = *s_bad ? 3 : (v < 0 ? 1 : 0);
    if (!is_prod && owned && status == 0 && p.final_score) {
      if (vb + 0 == v) p.final_score[lat.index] = s0;
      if (vb + 1 == v) p.final_score[lat.index] = s1;
      if (vb + 2 == v) p.final_score[lat.index] = s2;
      if (vb + 3 == v) p.final_score[lat.index] = s3;
    }
    __syncthreads();  // everybody has read s_vmax / s_bad before thread 0 resets them for the next lattice
    if (rank == 0) {
      if (tid == 0) {
        p.status[lat.index] = status;
        if (status != 0 && p.final_score) p.final_score[lat.index] = __int_as_float(0x7fc00000);
      }
#ifdef KAB_BANDP_TIMING
      const long long tm_bt0 = clock64();
#endif
      if (status == 0 && p.end_state) {
        if (tid == 0) p.end_state[lat.index] = v;  // traceback by kab_bt_maps_kernel / kab_bt_stitch_kernel
      } else if (status == 0) {
        // ---- backtrack (== flush_determined_path, align.py:21-40), CTA 0 only.  Blocks of FBK frames
        // = FBK / 8 groups of 256 bytes per region; the walker (one thread) reads the 8 frames of a
        // group for its byte column and the column below as two 64-bit words and then runs on
        // registers.
        const int NT = KAB_BP_THREADS;
        const uint16_t *col16 = p.col16 + lat.col_off;
        const unsigned char *bp = p.bp + lat.bp_off;
        const int n_blocks = (T + FBK - 1) / FBK;
        int32_t *out_path = p.best_path + lat.t_off;
        int32_t *out_lab = p.best_labels + lat.t_off;
        float *out_sc = p.best_scores + lat.t_off;
        const float *lp = p.lp + lat.t_off * (int64_t)V;
        constexpr int RSZ = FBK * 32;  // bytes of one region of one block
        // fetch block `b` of regions wtop, wtop-1, wtop-2 (mod NWT) into buffer `buf` (thread 0)
        auto fetch = [&](int b, int wtop, int buf) {
          const int ng = (min(FBK, T - b * FBK) + G - 1) / G;
          const uint32_t bytes = (uint32_t)ng * 256u;
          kab_mbar_expect_tx(&btbar[buf], bytes * NREG);
          for (int j = 0; j < NREG; ++j) {
            const int reg = (wtop - j + NWT) % NWT;
            kab_bulk_g2s(btbuf + ((size_t)buf * NREG + j) * RSZ, bp + ((size_t)reg * n_groups + (size_t)b * (FBK / G)) * 256,
                         bytes, &btbar[buf]);
          }
        };
        auto flush_block = [&](int b, int first_thread, int n_threads) {
          const int i0 = b * FBK, i1 = min(T, i0 + FBK);
          const int *pbuf = pathbuf + (b & 1) * FBK;
          for (int i = i0 + (tid - first_thread); i < i1; i += n_threads) {
            const int pv = pbuf[i - i0];
            const int lab = (pv & 1) ? (int)col16[(pv - 1) >> 1] : 0;
            out_path[i] = pv;
            out_lab[i] = lab;                              // align.py:106
            out_sc[i] = __ldg(&lp[(int64_t)i * V + lab]);  // align.py:107
          }
        };
        // walker state (thread 0): v, its ring slot, the region that owns the slot and its first slot
        int slot = v % R, wreg = slot / OW, base = wreg * OW;
        int wtop0 = wreg, wtop1 = wreg;  // top region staged in buffer 0 / 1
        if (tid == 0) fetch(n_blocks - 1, wreg, (n_blocks - 1) & 1);
        for (int b = n_blocks - 1; b >= 0; --b) {
          const int buf = b & 1;
          const int i0 = b * FBK, i1 = min(T, i0 + FBK);
          if (tid == 0) {
            if (b > 0) {  // the block below, predicted from the region the walk is in now
              if (buf) wtop0 = wreg; else wtop1 = wreg;
              fetch(b - 1, wreg, buf ^ 1);
            }
            kab_mbar_wait(&btbar[buf], bt_uses[buf] & 1u);
            ++bt_uses[buf];
            int jreg = ((buf ? wtop1 : wtop0) - wreg + NWT) % NWT;
            auto restage = [&]() {  // the staged regions do not cover the walk: stage again around wreg
              if (buf) wtop1 = wreg; else wtop0 = wreg;
              fetch(b, wreg, buf);
              kab_mbar_wait(&btbar[buf], bt_uses[buf] & 1u);
              ++bt_uses[buf];
              jreg = 0;
            };
            if (jreg >= NREG) restage();
            int *pbuf = pathbuf + buf * FBK;
            const unsigned char *rows = btbuf + ((size_t)buf * NREG + jreg) * RSZ;
            int col = (slot - base) >> 2, k2 = 2 * (slot & 3);  // byte column of the walker, bit offset in it
            // Full groups are walked from registers (kab_walk_group8: two 64-bit loads per group, off
            // the dependent chain); the frames it leaves (a second column step inside a group, a
            // partial group) take the generic step below, which also handles the step into the
            // warp region below (every ~370 frames).
            auto step_column = [&]() {  // the walker's byte column drops by one
              if (--col < 0) {          // ... into the region below (a move crosses at most one boundary)
                wreg = wreg == 0 ? NWT - 1 : wreg - 1;
                base = wreg * OW;
                if (++jreg == NREG) restage();
                rows = btbuf + ((size_t)buf * NREG + jreg) * RSZ;
                col = (OW >> 2) - 1;
              }
            };
            uint2 pw0 = make_uint2(0u, 0u), pw1 = pw0;  // words of the group below, loaded a group early
            const unsigned char *pfrom = nullptr;       // ... from this column address (nullptr: nothing loaded)
            for (int gq = (i1 - 1 - i0) >> 3; gq >= 0; --gq) {
              int f = min(7, i1 - 1 - i0 - gq * 8);
              int *pg = pbuf + gq * 8;
              if (f == 7) {
                const unsigned char *grow = rows + gq * 256;
                const bool have1 = col > 0 || jreg + 1 < NREG;
                const unsigned char *c0 = grow + col * 8;
                const unsigned char *below = col > 0 ? c0 - 8 : grow + RSZ + ((OW >> 2) - 1) * 8;
                uint2 w0, w1;
                if (pfrom == c0) {
                  w0 = pw0; w1 = pw1;
                } else {
                  w0 = *reinterpret_cast<const uint2 *>(c0);
                  w1 = have1 ? *reinterpret_cast<const uint2 *>(below) : make_uint2(0u, 0u);
                }
                if (gq > 0) {  // same column one group down: right unless the walk changes column now
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
            slot = v % R;
          } else if (tid >= 32 && b + 1 < n_blocks) {
            flush_block(b + 1, 32, NT - 32);
          }
          __syncthreads();
        }
        flush_block(0, 0, NT);
      }
      __syncthreads();
#ifdef KAB_BANDP_TIMING
      if (tid == 0 && p.debug) p.debug[32 * 16] = clock64() - tm_bt0;
#endif
    }
  }
}
