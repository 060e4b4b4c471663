// kab_bandq.cuh -- the cluster band kernel with TWO warps per scheduler (the default for chapter
// lattices with the reference's diagonal band, align.py:64-65, when every lattice of the plan gets
// its own cluster).  Same shapes as kab_bandp.cuh: max_move = 4, labels in 1..V-1, V <= 512,
// S <= 3T, min(beam_size, S) + 32 <= R = 40 * NWT ring slots, NWT = 8 * NC compute warps in a
// cluster of NC <= 8 CTAs (the 1000-wide band: 4 CTAs, 32 warps, R = 1280).
//
// Why: kab_bandp.cuh runs ONE warp of four states per lane on every scheduler.  Its timing build
// shows ~270 cycles per frame against a ~40-cycle dependent chain: a lone warp issues the ~45
// instructions of a frame at ~2 cycles each (the ALU and FMA pipes are half rate and the chain
// SHFL -> FADD2 -> FMNMX3 -> FSETP -> IMAD leaves no second instruction to interleave), and all
// of the per-group bookkeeping (neighbour message, emission loads, window masks, backpointer
// staging: more than half of a group) sits on the same single instruction stream.  Here
//   * a lane holds TWO states (one blank + one label): half the instructions on every warp's
//     chain (19 per frame: 3 SHFL, 3 FADD2 + 1 FADD, 1 FMNMX + 2 FMNMX3 + 4 FSETP + 1 FSEL, 4 IMAD);
//   * a CTA runs EIGHT compute warps, two per scheduler, so one warp's bookkeeping and ALU phase
//     overlap the other's frames and FMA phase -- the schedulers finally have a second stream;
//   * the price: 12 of 32 lanes are ghosts (the junk entering at lanes 0 / 1 climbs <= 3 states =
//     1.5 lanes per frame, so 8 frames consume exactly 12 lanes), 40 owned ring slots per warp,
//     26 warps instead of 10 for the 1000-wide band, one more SM per lattice.
//     tools/emulate_band_v4.py checks the scheme (with adversarial junk) against the CPU restatement.
// Everything else is the design of kab_bandp.cuh: no barrier on the recurrence, neighbour
// messages as (score, seq) 8-byte words through a FIFO in L2 loaded one group early, a chain whose
// head runs free, emissions of a whole group in registers one group ahead (staged per CTA by a
// producer warp that also checks finiteness), the window only as masked emissions of edge warps.
// Backpointers: 4 bits per lane and frame = ONE 32-bit word per lane and 8-frame group,
// [warp][group][32 lanes][4 B] (ghost lanes write words nobody reads), staged per warp and
// written with bulk stores.  The traceback is always the parallel map composition of
// kab_btpar.cuh (KabBtLayoutQ); this kernel publishes the forced end state.
#pragma once
#include "kab_band.cuh"  // KAB_BAND_G: frames per group
#include "kab_common.cuh"

#define KAB_BQ_CW 8      // compute warps per CTA
#define KAB_BQ_GH 12     // ghost lanes per warp = 3 * G / 2
#define KAB_BQ_OW 40     // ring slots owned by a warp = (32 - GH) * 2
#define KAB_BQ_NS 48     // emission stages per CTA.  The ring of 8 * NC warps is a CHAIN in time: every warp trails its
                         // lower neighbour by 2-3 groups, and head and tail of the chain can sit in the same
                         // CTA (the ring wraps), ~31 links = ~80 groups = ~40 stages of 16 frames apart.  With
                         // fewer stages the head is throttled to the minimal lag and every link polls.
#define KAB_BQ_D 64      // neighbour FIFO depth (messages, global memory)
#define KAB_BQ_LAG 2     // a warp joining the chain waits until its lower neighbour is this many groups ahead
#define KAB_BQ_FBW 128   // frames per per-warp backpointer block
#define KAB_BQ_MSG_BYTES (KAB_BQ_GH * 16)  // 12 lanes x 2 (score, seq) pairs
#define KAB_BQ_THREADS ((KAB_BQ_CW + 1) * 32)

struct KabBandqGeom {
  size_t bpst_off, stage_off, smem_bytes;
};
__host__ __device__ inline KabBandqGeom kab_bandq_geom(int stage_bytes) {
  KabBandqGeom g;
  g.bpst_off = ((size_t)2 * KAB_BQ_NS * 8 + 64 + 127) & ~(size_t)127;  // after the mbarriers (2 * NS) and the CTA scalars
  g.stage_off = g.bpst_off + (size_t)KAB_BQ_CW * 2 * (KAB_BQ_FBW / 8) * 128;
  g.smem_bytes = g.stage_off + (size_t)KAB_BQ_NS * stage_bytes;
  return g;
}
// Bytes of the global scratch of one lattice (layout: kab_cluster_fifo_off)
__host__ __device__ inline size_t kab_bandq_ws_bytes(int nwt) {
  return kab_cluster_fifo_off(nwt) + (size_t)nwt * KAB_BQ_D * KAB_BQ_MSG_BYTES;
}

#ifdef KAB_BANDQ_TIMING
#define KAB_QTM(var) const long long var = clock64()
#define KAB_QTM_ADD(acc, a, b) acc += (b) - (a)
#else
#define KAB_QTM(var)
#define KAB_QTM_ADD(acc, a, b)
#endif

__global__ void __launch_bounds__(KAB_BQ_THREADS, 1)
    kab_bandq_kernel(const KabLattice *__restrict__ lats, int n_lat, KabParams p) {
  constexpr int G = KAB_BAND_G, GH = KAB_BQ_GH, OW = KAB_BQ_OW;
  constexpr int CW = KAB_BQ_CW, NS = KAB_BQ_NS, D = KAB_BQ_D, FBW = KAB_BQ_FBW;
  static_assert(G == 8, "a group of 8 frames is one 32-bit backpointer word per lane");
  const KabBandqGeom geo = kab_bandq_geom(p.stage_bytes);
  extern __shared__ __align__(128) unsigned char kab_smem[];
  uint64_t *efull = reinterpret_cast<uint64_t *>(kab_smem);  // [NS]
  uint64_t *eempty = efull + NS;                             // [NS]
  unsigned int *s_item = reinterpret_cast<unsigned int *>(eempty + NS);
  int *s_vmax = reinterpret_cast<int *>(s_item + 1);
  unsigned int *s_bad = s_item + 2;
  float *stage_base = reinterpret_cast<float *>(kab_smem + geo.stage_off);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t rank = kab_cluster_rank(), NC = kab_cluster_size();
  const int NWT = CW * (int)NC, R = OW * NWT;
  const bool is_prod = warp == CW;
  const int gw = (int)rank * CW + warp;  // global compute-warp index (meaningless for the producer)
  const int ngw = (gw + 1) % NWT;
  const bool owned = lane >= GH;
  // ring slot of this lane's blank state: owned lanes tile the warp's 40 slots, ghost lanes mirror
  // the previous warp's lanes 20..31
  const int slot0 = owned ? OW * gw + 2 * (lane - GH) : (OW * gw - 2 * GH + 2 * lane + R) % R;
  const float ninf = kab_neg_inf();

  if (tid == 0) {
    for (int s = 0; s < NS; ++s) {
      kab_mbar_init(&efull[s], 1);
      kab_mbar_init(&eempty[s], CW);
    }
    kab_fence_mbar_init();
  }
  __syncthreads();
  uint32_t echunks = 0;  // emission chunks staged so far by this CTA (same count in every warp)

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
    float s0 = ninf, s1 = ninf;  // blank state vb, label state vb + 1
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
        if (use > 0) kab_mbar_wait(&eempty[stg], (use - 1u) & 1u);  // all compute warps released it
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
      auto load_col = [&](int base) -> uint32_t { return base + 1 < S ? 4u * col16[base >> 1] : 0u; };
      uint32_t c1 = load_col(vb), nc1 = load_col(vb + R);  // byte offset of the label column; next alias prefetched
      const int half = W / 2;
      const int VB = V * 4;

      uint32_t st = ec0 % NS, ph = (ec0 / NS) & 1u;  // stage / phase of the chunk being read
      auto chunk_ptr = [&](uint32_t stg) { return reinterpret_cast<const char *>(stage_base + stg * stage_words + skew); };
      // emissions of a whole group, in registers: blank and label of this lane
      float eb[G], e1[G], nb[G], n1[G];
      auto load_group = [&](const char *row, float (&xb)[G], float (&x1)[G]) {
#pragma unroll
        for (int f = 0; f < G; ++f) {
          xb[f] = *reinterpret_cast<const float *>(row + f * VB);
          x1[f] = *reinterpret_cast<const float *>(row + f * VB + c1);
        }
      };
      kab_mbar_spin(&efull[st], ph);
      const char *rowc = chunk_ptr(st);  // first row of the current group
      load_group(rowc, eb, e1);

      const int qd = S / T, rd = S % T;
      const int qdg = (int)(((int64_t)S * G) / T), rdg = (int)(((int64_t)S * G) % T);
      int qg = 0, rg = 0, q = 0, r = 0;

      // backpointers: per-warp staging [2][FBW / 8 groups][32 lanes][4 B]
      unsigned char *bpbuf = kab_smem + geo.bpst_off + (size_t)warp * 2 * (FBW / 8) * 128;
      unsigned char *bpg = p.bp + lat.bp_off + (size_t)gw * n_groups * 128;  // this warp's region of the workspace
      int gib = 0, blk = 0;  // group inside the current block, block index
      uint32_t bw = 0;       // backpointer nibbles of the current group

      // One frame; sh = bit offset of this frame's nibble in bw.  The window of align.py:64-65 never
      // appears here: a cell outside [lo, hi) is made inactive through its EMISSION (-inf: every
      // candidate is -inf, so the maximum is), and the masked emissions of an edge warp are prepared
      // per group, off the recurrence chain.
      auto frame = [&](const float xb, const float x1, const int sh) {
        const float h1 = __shfl_up_sync(KAB_FULL_MASK, s1, 1);  // state vb - 1
        const float h2 = __shfl_up_sync(KAB_FULL_MASK, s0, 1);  // state vb - 2
        const float h3 = __shfl_up_sync(KAB_FULL_MASK, s1, 2);  // state vb - 3
        float t0, th1, a0, a1, a2, a3;
        kab_add2(s0, h1, xb, t0, th1);  // blank <- vb (move 0), vb - 1 (move 1)
        const float th3 = __fadd_rn(h3, xb);  // vb - 3 (move 3)
        kab_add2(s0, s1, x1, a1, a0);   // label <- vb + 1 (move 0), vb (move 1)
        kab_add2(h2, h1, x1, a3, a2);   //       <- vb - 1 (move 2), vb - 2 (move 3)
        const float m0 = kab_blank_sel(t0, th1, th3, bw, 1u << (sh + 0), 2u << (sh + 0), one);
        const float m1 = kab_label_sel(a0, a1, a2, a3, bw, 1u << (sh + 2), 2u << (sh + 2), one);
        s0 = m0; s1 = m1;
      };

      int fic = 0;       // frame offset of the current group inside its emission chunk
      int lo_prev = 0;   // lo of the first frame of the previous group (<= lo of every later frame)
      // neighbour FIFO in global memory: my inbox (messages of the warp below) and the inbox of warp ngw
      unsigned char *gws = p.fifo + (size_t)lat.scr_off * 4;
      unsigned int *cons = reinterpret_cast<unsigned int *>(gws);
      unsigned char *gfifo = gws + kab_cluster_fifo_off(NWT);
      const unsigned char *inbox = gfifo + (size_t)gw * D * KAB_BQ_MSG_BYTES + (lane < GH ? lane : 0) * 16;
      unsigned char *outbox = gfifo + (size_t)ngw * D * KAB_BQ_MSG_BYTES + (lane >= 32 - GH ? lane - (32 - GH) : 0) * 16;
      uint32_t cons_seen = 0;   // messages the warp above is known to be done with
      bool was_needed = false;  // the previous group read its message (the warp is inside the chain)
      uint2 pf0 = make_uint2(0, 0), pf1 = pf0;  // message g-1, loaded a group early
#ifdef KAB_BANDQ_TIMING
      long long tm_ghost = 0, tm_emis = 0, tm_comp = 0, tm_pub = 0, tm_rel = 0, tm_bp = 0, n_need = 0, n_safe = 0, tm_wait = 0, tm_slow = 0;
      long long cat_t[4] = {0, 0, 0, 0}, cat_n[4] = {0, 0, 0, 0}, cat_w[4] = {0, 0, 0, 0};  // by (need, safe)
      bool cur_need = false;
      long long cur_wait = 0;
      const long long tm_start = clock64();
#endif
      for (int g = 0; g < n_groups; ++g) {
        const int i0 = g * G, nfr = min(G, T - i0);
        const bool more = i0 + G < T;
        KAB_QTM(ta);
        // ---- ghost lanes: the lower neighbour's top 24 states after its group g-1 (message g-1).
        // The warp only WAITS for the message when the ghost states can matter: if all 24 were
        // outside the window at frame 8g-1 and stay outside during this group they are inactive
        // (-inf) by definition.  At least one warp boundary of the ring is always in that situation,
        // so the ring is a chain whose head never waits.
        if (g > 0) {
          int qn2 = qg + qdg;
          if (rg + rdg >= T) ++qn2;
          const int hi1g = min(max(0, qn2 - half) + W, S);  // >= hi of every frame of this group
          const bool outside = owned || vb + 1 < lo_prev || vb >= hi1g;
          const bool need = !__all_sync(KAB_FULL_MASK, outside);
#ifdef KAB_BANDQ_TIMING
          n_need += need;
          const long long tw0 = clock64();
#endif
          if (need) {
            if (!owned) {
              if (!was_needed) {  // (re)joining the chain: let the warp below get KAB_BQ_LAG groups ahead
                const int mt = min(g - 1 + KAB_BQ_LAG - 1, n_groups - 2);
                const unsigned char *ls = inbox + (size_t)(mt % D) * KAB_BQ_MSG_BYTES;
                while (kab_ld_volatile_b64(ls + 8).y != (uint32_t)(mt + 1)) __nanosleep(64);
              }
              const unsigned char *slot = inbox + (size_t)((g - 1) % D) * KAB_BQ_MSG_BYTES;
              const uint32_t seq = (uint32_t)g;
              while (pf0.y != seq || pf1.y != seq) {
                pf0 = kab_ld_volatile_b64(slot);
                pf1 = kab_ld_volatile_b64(slot + 8);
              }
              s0 = __uint_as_float(pf0.x);
              s1 = __uint_as_float(pf1.x);
            }
          } else if (!owned) {
            s0 = ninf; s1 = ninf;
          }
          was_needed = need;
          __syncwarp();
          if (lane == 0) kab_st_volatile_u32(&cons[gw], (uint32_t)g);  // done with messages 0 .. g-1
#ifdef KAB_BANDQ_TIMING
          cur_wait = clock64() - tw0;
          cur_need = need;
          tm_wait += cur_wait;
#endif
        }
        // message g (for the next group) may already be there: load it now, check it then
        if (more && !owned) {
          const unsigned char *slot = inbox + (size_t)(g % D) * KAB_BQ_MSG_BYTES;
          pf0 = kab_ld_volatile_b64(slot);
          pf1 = kab_ld_volatile_b64(slot + 8);
        }
        lo_prev = max(0, qg - half);
        KAB_QTM(tb);
        KAB_QTM_ADD(tm_ghost, ta, tb);
        const bool next_crosses = fic + G == F;
        const uint32_t nst = st + 1 == NS ? 0 : st + 1;
        const uint32_t nph = nst == 0 ? ph ^ 1u : ph;
        // the next group's emissions are loaded during this group
        if (next_crosses && more) kab_mbar_spin(&efull[nst], nph);
        KAB_QTM(tc);
        KAB_QTM_ADD(tm_emis, tb, tc);
        const char *rowng = next_crosses ? chunk_ptr(nst) : rowc + G * VB;
        const int lo0 = max(0, qg - half), hi0 = min(lo0 + W, S);
        int qn = qg + qdg, rn = rg + rdg;
        if (rn >= T) { rn -= T; ++qn; }
        const int lo1 = max(0, qn - half);
        if (vb + 1 < lo0 - 3) {  // recycle a chunk that fell below the window (between groups only)
          do {
            vb += R;
            c1 = nc1;
            nc1 = load_col(vb + R);
          } while (vb + 1 < lo0 - 3);
          load_group(rowc, eb, e1);  // the prefetched emissions belonged to the old alias
        }
        if (more) load_group(rowng, nb, n1);
        const bool safe = __all_sync(KAB_FULL_MASK, nfr == G && vb >= lo1 && vb + 2 <= hi0);
        bw = 0;
#ifdef KAB_BANDQ_TIMING
        n_safe += safe;
#endif
        if (safe) {
#pragma unroll
          for (int f = 0; f < G; ++f) frame(eb[f], e1[f], 4 * f);
        } else {
          // edge warp (or the last, partial group): the exact per-frame window (S*i = q*T + r, no
          // divisions) turned into masked emissions for the whole group
          q = qg; r = rg;
          float mb[G], mm[G];
#pragma unroll
          for (int f = 0; f < G; ++f) {
            const int lo = max(0, q - half);   // align.py:64
            const int hi = min(lo + W, S);     // align.py:65
            q += qd; r += rd;
            if (r >= T) { r -= T; ++q; }
            const unsigned a = (unsigned)(vb - lo), wd = (unsigned)(hi - lo);
            mb[f] = (a + 0u < wd) ? eb[f] : ninf;
            mm[f] = (a + 1u < wd) ? e1[f] : ninf;
          }
          if (nfr == G) {
#pragma unroll
            for (int f = 0; f < G; ++f) frame(mb[f], mm[f], 4 * f);
          } else {
#pragma unroll
            for (int f = 0; f < G; ++f)
              if (f < nfr) frame(mb[f], mm[f], 4 * f);
          }
        }
        qg = qn; rg = rn;
        KAB_QTM(td);
        KAB_QTM_ADD(tm_comp, tc, td);
#ifdef KAB_BANDQ_TIMING
        if (!safe) tm_slow += td - tc;
#endif

        // ---- hand the top twelve lanes to the warp above (message g)
        if (more) {
          if (g >= D && (uint32_t)(g - D) >= cons_seen) {  // about to lap the consumer: read its progress
            do {
              cons_seen = kab_ld_volatile_u32(&cons[ngw]);
            } while ((uint32_t)(g - D) >= cons_seen);
          }
          if (lane >= 32 - GH) {
            unsigned char *slot = outbox + (size_t)(g % D) * KAB_BQ_MSG_BYTES;
            const uint32_t seq = (uint32_t)(g + 1);
            kab_st_volatile_b64(slot, __float_as_uint(s0), seq);
            kab_st_volatile_b64(slot + 8, __float_as_uint(s1), seq);
          }
        }
        KAB_QTM(te);
        KAB_QTM_ADD(tm_pub, td, te);
        // ---- backpointer word of this group -> staging; block finished?
        *reinterpret_cast<uint32_t *>(bpbuf + ((blk & 1) * (FBW / 8) + gib) * 128 + lane * 4) = bw;
        ++gib;
        if (gib == FBW / 8 || !more) {
          kab_fence_proxy_async_smem();  // every lane's words -> visible to the bulk store
          __syncwarp();
          if (lane == 0) {
            kab_bulk_s2g(bpg + (size_t)blk * (FBW / 8) * 128, bpbuf + (size_t)(blk & 1) * (FBW / 8) * 128, (uint32_t)gib * 128u);
            kab_bulk_wait_read1();  // the block before this one has left its buffer
          }
          __syncwarp();
          ++blk;
          gib = 0;
        }
        KAB_QTM(tf);
        KAB_QTM_ADD(tm_bp, te, tf);
        // ---- next group's emissions become current; emission chunk finished?
#pragma unroll
        for (int f = 0; f < G; ++f) { eb[f] = nb[f]; e1[f] = n1[f]; }
        rowc = rowng;
        if (next_crosses || !more) {
          __syncwarp();
          if (lane == 0) kab_mbar_arrive(&eempty[st]);
          st = nst; ph = nph;
          fic = 0;
        } else {
          fic += G;
        }
        KAB_QTM(tg);
        KAB_QTM_ADD(tm_rel, tf, tg);
#ifdef KAB_BANDQ_TIMING
        {
          const int cat = (cur_need ? 2 : 0) + (safe ? 1 : 0);
          cat_t[cat] += tg - ta; cat_n[cat] += 1; cat_w[cat] += cur_wait;
          cur_need = false; cur_wait = 0;
        }
#endif
      }
#ifdef KAB_BANDQ_TIMING
      if (lane == 0 && p.debug) {
        long long *d = p.debug + gw * 16;
        d[0] = tm_ghost; d[1] = tm_emis; d[2] = tm_comp; d[3] = tm_pub; d[4] = tm_rel; d[5] = tm_bp;
        d[6] = clock64() - tm_start; d[7] = n_groups; d[9] = n_need; d[10] = n_safe; d[11] = tm_wait; d[13] = tm_slow;
        long long *c = p.debug + 64 * 16 + 8 + gw * 12;
        for (int k = 0; k < 4; ++k) { c[k] = cat_t[k]; c[4 + k] = cat_n[k]; c[8 + k] = cat_w[k]; }
      }
#endif
      // ---- end of the forward pass: cluster-wide forced end state (align.py:99-101)
      int cand = -1;
      if (owned) {
        if (vb + 0 < S && s0 > ninf) cand = vb + 0;
        if (vb + 1 < S && s1 > ninf) cand = vb + 1;
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

    const int v = *s_vmax;
    const int status = *s_bad ? 3 : (v < 0 ? 1 : 0);
    if (!is_prod && owned && status == 0 && p.final_score) {
      if (vb + 0 == v) p.final_score[lat.index] = s0;
      if (vb + 1 == v) p.final_score[lat.index] = s1;
    }
    if (rank == 0 && tid == 0) {
      p.status[lat.index] = status;
      if (status != 0 && p.final_score) p.final_score[lat.index] = __int_as_float(0x7fc00000);
      if (status == 0) p.end_state[lat.index] = v;  // traceback by kab_bt_maps_kernel / kab_bt_stitch_kernel
    }
    __syncthreads();  // everybody has read s_vmax / s_bad before thread 0 resets them for the next lattice
  }
}
