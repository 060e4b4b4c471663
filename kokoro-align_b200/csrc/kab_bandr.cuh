// kab_bandr.cuh -- warp-specialised cluster band kernel: the recurrence warps do NOTHING but the
// recurrence.  Same shapes, ring, lanes and backpointer words as kab_bandq.cuh (two states per
// lane, 12 ghost lanes, 40 owned ring slots per warp; KAB_BR_CW = 4 compute warps per CTA, one per
// scheduler, clusters of NC <= 8 CTAs; KabBtLayoutQ for the traceback).
//
// Why (measured with the KAB_BANDQ_TIMING build and tools/ubench/chain.cu on B200): the frame of
// the two-states-per-lane update is a dependent chain SHFL.UP (24.9 cycles) -> FADD2 (4.7) ->
// FMNMX3 (4.3); the whole value update runs at 43-46 cycles per frame, alone or with two warps
// per scheduler.  kab_bandq.cuh spends ~2 230 cycles per 8-frame group and warp, i.e. 280 per
// frame: the warps of a lattice form a chain in time whose pace is the SERIAL work of its slowest
// member per group, and only ~400 of those cycles are frames -- the rest is the warp's own
// bookkeeping on the same instruction stream: emission gathers for the next group (16 LDS +
// addresses), the exact window turned into masks (edge warps: +270), recycling, mbarrier waits,
// neighbour messages through L2 (loads / polls of 300-700 cycles), credit checks, backpointer
// staging and bulk stores.  Two warps per scheduler do not help a chain: its links are serial.
//
// Here every compute warp has a PREP warp that runs up to KAB_BR_TD groups ahead and hands it
// finished emission tiles in shared memory -- gathered, with the window of align.py:64-65
// already applied as -inf -- so the compute warp's group is: check the neighbour's message (a
// shared-memory word), 8 x (one LDS.64 + the 19-instruction frame), publish its top 12 lanes to
// the warp above (shared memory, or distributed shared memory across the CTA boundary: one
// st.shared::cluster per (score, seq) word, no mbarrier, no L2 round trip), one STS of the
// backpointer word.  The prep warp also owns the ring bookkeeping (aliases, recycling, label
// columns), releases the emission stages, and issues the bulk stores of its compute warp's
// backpointer blocks.  A producer warp stages emission rows by bulk copies and writes the window
// table of every chunk (finiteness is checked by kab_finite_rows_kernel behind this kernel).
//
// What the chain's period turned out to be (DESIGN.md section 3.3b): (1) a warp whose ring slots
// are recycled above the window rejoins the chain every 18 groups -- any start-up lag it is given
// there is paid on the whole lattice, so it joins at once, through the common path; (2) after
// that the chain runs at its minimal lag and its period is ONE warp's own work per group, hence
// the common path of the compute warp: two groups per pass in a compact loop of its own, inline
// polls, predicated end-of-group stores, addresses precomputed, two shared register pairs for the
// three packed adds of a frame.
// GA (template parameter): gather mode for wide vocabularies -- the prep warps read the emissions
// from global memory, the producer warp prefetches the rows into L2.
#pragma once
#include "kab_band.cuh"   // KAB_BAND_G: frames per group
#include "kab_bandq.cuh"  // KAB_BQ_GH / KAB_BQ_OW: the lanes of kab_bandq.cuh
#include "kab_common.cuh"

#define KAB_BR_CW 4           // compute warps per CTA (and as many prep warps): ONE compute warp per scheduler.  The
                              // SM sub-partition issues ~1 instruction per cycle and a warp at most every other
                              // cycle; with two compute + two prep warps per scheduler the compute warps got a
                              // quarter of the slots each (measured: 940 cycles for the 230 instructions of a group)
#define KAB_BR_GH KAB_BQ_GH   // ghost lanes
#define KAB_BR_OW KAB_BQ_OW   // owned ring slots per warp
#define KAB_BR_NS 40          // emission stages per CTA (head and tail of the chain can sit in one CTA)
#define KAB_BR_F 16           // frames per emission stage this kernel is built for (two groups; the plan checks it)
#define KAB_BR_TD 8           // emission tiles per compute warp (groups the prep warps may run ahead)
#define KAB_BR_MD 16          // mailbox depth (messages)
#define KAB_BR_GA_AHEAD 12    // gather mode: chunks (of 16 frames) the L2 prefetch runs ahead of the producer
#define KAB_BR_BG 16          // groups per backpointer block (2 KB)
#define KAB_BR_NBB 4          // backpointer staging buffers per compute warp
#define KAB_BR_THREADS ((3 * KAB_BR_CW + 1) * 32)

struct KabBandrGeom {
  size_t ctrl_off, tile_off, mbox_off, bp_off, vbf_off, wtab_off, stage_off, smem_bytes;
};
__host__ __device__ inline KabBandrGeom kab_bandr_geom(int stage_bytes) {
  KabBandrGeom g;
  g.ctrl_off = ((size_t)(2 * KAB_BR_NS + KAB_BR_CW * KAB_BR_TD) * 8 + 64 + 127) & ~(size_t)127;  // after the mbarriers and CTA scalars
  g.tile_off = g.ctrl_off + (size_t)KAB_BR_CW * 128;                       // one 128-byte control block per compute warp
  g.mbox_off = g.tile_off + (size_t)KAB_BR_CW * KAB_BR_TD * 8 * 32 * 8;    // tiles [w][TD][8 frames][32 lanes] float2
  g.bp_off = g.mbox_off + (size_t)KAB_BR_CW * KAB_BR_MD * KAB_BR_GH * 16;  // mailboxes [w][MD][12 lanes][2] (score, seq)
  g.vbf_off = g.bp_off + (size_t)KAB_BR_CW * KAB_BR_NBB * KAB_BR_BG * 128;  // backpointer staging [w][NBB][BG][32] u32
  g.wtab_off = g.vbf_off + (size_t)KAB_BR_CW * 32 * 4;                     // final alias of every lane
  g.stage_off = g.wtab_off + (size_t)KAB_BR_NS * 32 * 4;                   // window starts [NS][frames of the stage + 1] (<= 32 ints)
  g.smem_bytes = g.stage_off + (size_t)KAB_BR_NS * stage_bytes;
  return g;
}

// control block of compute warp w (u32 words, shared memory)
#define KAB_BR_C_TILESEQ 0    // [TD] tile t holds group g  <=>  low 31 bits == g + 1; bit 31: the ghost lanes need
                              //      the neighbour's message for that group                (prep -> compute)
#define KAB_BR_C_COMPDONE 16  // groups finished: tiles 0 .. n-1 read, messages 0 .. n-2 consumed
                              //                                  (compute -> prep, compute -> lower neighbour)
#define KAB_BR_C_BPREADY 17   // backpointer blocks staged                                 (compute -> prep)
#define KAB_BR_C_BPFREE 18    // backpointer blocks whose staging buffer is free again     (prep -> compute)
#define KAB_BR_C_UPDONE 19    // last warp of a CTA: copy of the COMPDONE word of the warp above, which lives in the
                              // next CTA and PUSHES its progress here (a remote load per group stalled this warp
                              // for ~1 200 cycles and made it the slowest link of the chain)

#ifdef KAB_BANDR_TIMING
#define KAB_RTM(var) const long long var = clock64()
#define KAB_RTM_ADD(acc, a, b) acc += (b) - (a)
#else
#define KAB_RTM(var)
#define KAB_RTM_ADD(acc, a, b)
#endif

// GA ("gather"): the prep warps read the emissions straight from the log-probs in global memory
// (L2) instead of staged rows -- for vocabularies whose rows do not fit a stage (V > 512) and
// lattices with any number of distinct labels: no compact copy, no limit on V; the producer warp
// then only writes the window table.
template <bool MM, bool GA = false>
__global__ void __launch_bounds__(KAB_BR_THREADS, 1)
    kab_bandr_kernel(const KabLattice *__restrict__ lats, int n_lat, KabParams p) {
  constexpr int G = KAB_BAND_G, GH = KAB_BR_GH, OW = KAB_BR_OW;
  constexpr int CW = KAB_BR_CW, NS = KAB_BR_NS, TD = KAB_BR_TD, MD = KAB_BR_MD, BG = KAB_BR_BG;
  static_assert(G == 8, "a group of 8 frames is one 32-bit backpointer word per lane");
  const KabBandrGeom geo = kab_bandr_geom(p.stage_bytes);
  extern __shared__ __align__(128) unsigned char kab_smem[];
  uint64_t *efull = reinterpret_cast<uint64_t *>(kab_smem);  // [NS]
  uint64_t *eempty = efull + NS;                             // [NS]
  uint64_t *slotfree = eempty + NS;                          // [CW][TD] tile slot t of compute warp w has been read
  unsigned int *s_item = reinterpret_cast<unsigned int *>(slotfree + CW * TD);
  int *s_vmax = reinterpret_cast<int *>(s_item + 1);
  unsigned int *s_bad = s_item + 2;
  float *stage_base = reinterpret_cast<float *>(kab_smem + geo.stage_off);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  if (p.started && tid == 0) atomicAdd(p.started, 1u);  // (this CTA holds its SM: KabParams::started)
  const uint32_t rank = kab_cluster_rank(), NC = kab_cluster_size();
  const int NWT = CW * (int)NC, R = OW * NWT;
  // Warp roles by warp id: the scheduler's arbiter prefers the HIGHEST warp id among eligible warps
  // (B300_MICROARCH.md), so the compute warps -- the only ones on the critical path -- take the top
  // ids and the helpers, which poll while they wait, the low ones: warp 0 producer, 1 .. 2 CW prep
  // (two per compute warp: one builds the tiles of the even groups, the other those of the odd
  // ones), 2 CW + 1 .. 3 CW compute -- one compute warp and two prep warps per scheduler.
  const bool is_prod = warp == 0, is_prep = warp >= 1 && warp <= 2 * CW;
  const int pp = is_prep ? (warp - 1) & 1 : 0;                                        // parity a prep warp builds
  const int cw = is_prep ? (warp - 1) >> 1 : (warp > 2 * CW ? warp - 1 - 2 * CW : 0);  // the compute warp this warp is / serves
  const int gw = (int)rank * CW + cw;         // its global index in the ring
  const bool owned = lane >= GH;
  // ring slot of this lane's blank state: owned lanes tile the warp's 40 slots, ghost lanes mirror
  // the previous warp's lanes 20..31
  const int slot0 = owned ? OW * gw + 2 * (lane - GH) : (OW * gw - 2 * GH + 2 * lane + R) % R;
  const float ninf = kab_neg_inf();
  const uint32_t smem0 = kab_smem_u32(kab_smem);
  const uint32_t ctrl = smem0 + (uint32_t)geo.ctrl_off + (uint32_t)cw * 128u;       // this pair's control block
  const uint32_t mbox = smem0 + (uint32_t)geo.mbox_off + (uint32_t)cw * (MD * GH * 16u);
  const uint32_t bpst = smem0 + (uint32_t)geo.bp_off + (uint32_t)cw * (KAB_BR_NBB * BG * 128u);
  int *vbf = reinterpret_cast<int *>(kab_smem + geo.vbf_off) + cw * 32;

  if (tid == 0) {
    for (int s = 0; s < NS; ++s) {
      kab_mbar_init(&efull[s], 1);
      kab_mbar_init(&eempty[s], CW);  // the owner among the two prep warps of every compute warp releases a stage
    }
    kab_fence_mbar_init();
  }
  __syncthreads();
  uint32_t echunks = 0;  // emission chunks staged so far by this CTA (same count in every warp)

  for (;;) {
    // ---- reset the per-lattice words (sequence numbers restart at 1), then the cluster agrees on
    // the next work item; the cluster barrier also keeps remote mailbox stores of the new lattice
    // behind every CTA's reset
    for (uint32_t o = geo.ctrl_off + tid * 4; o < geo.tile_off; o += KAB_BR_THREADS * 4)
      *reinterpret_cast<uint32_t *>(kab_smem + o) = 0u;
    for (uint32_t o = geo.mbox_off + tid * 4; o < geo.bp_off; o += KAB_BR_THREADS * 4)
      *reinterpret_cast<uint32_t *>(kab_smem + o) = 0u;
    if (tid == 0) {
      *s_vmax = -1;
      *s_bad = 0u;
      for (int k = 0; k < CW * TD; ++k) kab_mbar_init(&slotfree[k], 1);  // (everybody left them at the barrier below)
      kab_fence_mbar_init();
    }
    if (rank == 0 && tid == 0) {
      const unsigned int it = atomicAdd(p.queue, 1u);
      for (uint32_t r = 0; r < NC; ++r) kab_st_cluster_u32(kab_mapa(kab_smem_u32(s_item), r), it);
    }
    __syncthreads();
    kab_cluster_sync();
    const unsigned int item = *s_item;
    if (item >= (unsigned int)n_lat) break;
    const KabLattice lat = lats[item];
    const int T = lat.T, S = 2 * lat.L + 1, V = p.V, W = p.W;
    const int F = p.stage_frames;
    const uint32_t stage_words = p.stage_bytes >> 2;
    const int n_chunks = (T + F - 1) / F;
    const int n_groups = (T + G - 1) / G;
    const int n_blocks = (n_groups + BG - 1) / BG;
    const uint32_t ec0 = echunks;
    const uint32_t skew = (uint32_t)(((lat.t_off * (int64_t)V * 4) & 15) >> 2);
    float s0 = ninf, s1 = ninf;  // compute warps: blank state vb, label state vb + 1
    int vb = slot0;              // prep warps track the alias; compute warps read the final one from vbf

    if (is_prod) {
      // ================= producer warp: emission ring and window table.  (The finiteness of the rows is
      // checked by kab_finite_rows_kernel after this kernel: the scan here -- 20 LDS + FMA per lane and
      // chunk -- made the compute warp that shares this warp's scheduler the slowest link of the chain.)
      const char *lp_base = reinterpret_cast<const char *>(p.lp) + ((lat.t_off * (int64_t)V * 4) & ~(int64_t)15);
      const uint32_t chunk_stride = (uint32_t)(F * V * 4);
      const uint32_t full_bytes = (chunk_stride + skew * 4 + 15) & ~15u;
      // window starts: lane l follows frame i = c * F + l with S * i = q * T + r kept exactly (one 64-bit
      // division per lattice, then three integer instructions per chunk)
      int wq = (int)(((long long)S * lane) / T), wr = (int)(((long long)S * lane) % T);
      const int wqF = (int)(((long long)S * F) / T), wrF = (int)(((long long)S * F) % T);
      for (int c = 0; c < n_chunks; ++c) {
        const uint32_t gc = ec0 + (uint32_t)c, stg = gc % NS, use = gc / NS;
        if (use > 0) kab_mbar_wait(&eempty[stg], (use - 1u) & 1u);  // all prep warps released it
        float *dst = stage_base + stg * stage_words;
        // the window of align.py:64 for the frames of this chunk (and the first frame behind it): lo_i =
        // max(0, S*i // T - W // 2) -- here, where nobody waits for it, instead of an incremental
        // (q, r) chain in every prep warp
        if (lane <= F) reinterpret_cast<int *>(kab_smem + geo.wtab_off)[stg * 32 + lane] = max(0, wq - p.W / 2);
        wq += wqF; wr += wrF;          // S * (i + F) = (q + qF) * T + (r + rF), carried
        if (wr >= T) { wr -= T; ++wq; }
        __syncwarp();  // (the arming arrive below releases these words together with the rows)
        if (GA) {
          // The rows themselves go to L2 ahead of the prep warps' gathers: the first warp to reach a chunk
          // would otherwise pay the DRAM latency once per tile.  Each CTA of the cluster prefetches its
          // 1 / NC of the chunk that is KAB_BR_GA_AHEAD chunks ahead (one bulk-prefetch instruction).
          if (lane == 0) {
            const int c_first = c == 0 ? 0 : c + KAB_BR_GA_AHEAD, c_last = min(n_chunks - 1, c + KAB_BR_GA_AHEAD);
            for (int cp = c_first; cp <= c_last; ++cp) {
              const int64_t row0 = lat.t_off + (int64_t)cp * F;
              const uint64_t base = reinterpret_cast<uint64_t>(p.lp);  // (absolute addresses: 16-byte alignment is the instruction's)
              const uint64_t b0 = base + (uint64_t)(row0 * V * 4), b1 = base + (uint64_t)((row0 + min(F, T - cp * F)) * V * 4);
              const uint64_t part = (((b1 - b0 + NC - 1) / NC) + 15) & ~(uint64_t)15;
              const uint64_t a0 = (b0 + (uint64_t)rank * part) & ~(uint64_t)15;
              const uint64_t a1 = min(min(a0 + part + 16, b1), base + (uint64_t)p.lp_bytes) & ~(uint64_t)15;
              if (a1 > a0) kab_bulk_prefetch_l2(reinterpret_cast<const void *>(a0), (uint32_t)(a1 - a0));
            }
            kab_mbar_arrive(&efull[stg]);  // the window table of this chunk is ready
          }
        } else if (c + 1 < n_chunks) {
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
    } else if (is_prep) {
      // ================= prep warp of compute warp cw: emission tiles, ring bookkeeping, backpointer stores.
      // The two prep warps of a compute warp OWN alternate emission chunks (16 frames = two groups):
      // the owner waits for the chunk and the two tile slots once, builds both tiles and releases the
      // chunk; for the other warp's chunks a prep warp only keeps its aliases in step (the window
      // start of a group from an exact incremental S * 8g = q * T + r: four instructions, no shared
      // memory).  Measured: with per-group ownership both warps paid the slot poll, two votes, the
      // mbarrier round trip and the service call for EVERY group -- 660 cycles per group each, the
      // floor of the whole pipeline.
      const uint16_t *col16 = p.col16 + lat.col_off;
      auto load_col = [&](int base) -> uint32_t { return base + 1 < S ? 4u * col16[base >> 1] : 0u; };
      uint32_t c1 = load_col(vb), nc1 = load_col(vb + R);  // byte offset of the label column; next alias prefetched
      const int half = W / 2;
      const int VB = V * 4;
      const int *wtab = reinterpret_cast<const int *>(kab_smem + geo.wtab_off);  // per-frame window starts, written by the producer
      const int qdg = (int)(((int64_t)S * G) / T), rdg = (int)(((int64_t)S * G) % T);
      int qg = 0, rg = 0;  // S * (8 g) = qg * T + rg for the group being tracked
      int lo_prev = 0;     // lo of the first frame of the previous group (<= lo of every later frame)
      unsigned char *bpg = p.bp + lat.bp_off + (size_t)gw * n_groups * 128;  // the compute warp's region of the workspace
      int bp_issued = 0;  // backpointer blocks handed to the bulk-copy engine
      // backpointer blocks the compute warp has staged -> bulk stores (the even prep warp; every lane
      // reads the same word, so the branch is warp-uniform without a shuffle)
      auto service_bp = [&]() {
        const int ready = (int)kab_lds_relaxed_u32(ctrl + 4 * KAB_BR_C_BPREADY);
        if (ready > bp_issued) {  // (at most one new block per visit: a block is 16 groups long)
          kab_fence_cta();
          const int b = bp_issued;
          const int ng = min(BG, n_groups - b * BG);
          if (lane == 0) {
            kab_bulk_s2g(bpg + (size_t)b * BG * 128, kab_smem + geo.bp_off + (size_t)cw * (KAB_BR_NBB * BG * 128) + (size_t)(b & (KAB_BR_NBB - 1)) * BG * 128,
                         (uint32_t)ng * 128u);
            kab_bulk_wait_read1();  // the block before this one has left its buffer
            kab_sts_relaxed_u32(ctrl + 4 * KAB_BR_C_BPFREE, (uint32_t)b);  // blocks 0 .. b-1 are free
          }
          bp_issued = b + 1;
          __syncwarp();
        }
      };
#ifdef KAB_BANDR_TIMING
      long long pm_wait = 0, pm_tile = 0, pm_rest = 0, pm_safe = 0;
      const long long pm_start = clock64();
#endif
      uint32_t flags = 0;  // does the compute warp need its neighbour's message for the group being built?
      for (int c = 0; c < n_chunks; ++c) {
        const bool own = (c & 1) == pp;
        const uint32_t gc = ec0 + (uint32_t)c, st = gc % NS, ph = (gc / NS) & 1u;
        const int g0 = c * (KAB_BR_F / G);  // first group of the chunk
        KAB_RTM(pa);
        if (own) {
          // the slots of both tiles are free once the compute warp has finished groups g0 - TD and
          // g0 + 1 - TD: it arrives on the slot's mbarrier after every group, and this warp sleeps in
          // mbarrier.try_wait (hardware) instead of polling shared memory -- the polling loops of the
          // helpers were most of the instructions the SM executed
          if (pp == 0) service_bp();
#pragma unroll
          for (int gi = 0; gi < KAB_BR_F / G; ++gi) {
            const int g = g0 + gi;
            if (g >= TD && g < n_groups) kab_mbar_wait(&slotfree[cw * TD + (g & (TD - 1))], (uint32_t)(g / TD - 1) & 1u);
          }
          kab_mbar_wait(&efull[st], ph);
        }
        KAB_RTM(pb);
        KAB_RTM_ADD(pm_wait, pa, pb);
        const char *rowc = GA ? reinterpret_cast<const char *>(p.lp + (lat.t_off + (int64_t)c * F) * V)
                              : reinterpret_cast<const char *>(stage_base + st * stage_words + skew);
        auto emission = [&](const char *a) -> float {
          return GA ? __ldg(reinterpret_cast<const float *>(a)) : *reinterpret_cast<const float *>(a);
        };
#pragma unroll
        for (int gi = 0; gi < KAB_BR_F / G; ++gi, rowc += G * VB) {
          const int g = g0 + gi;
          if (g >= n_groups) break;
          const int i0 = g * G, nfr = min(G, T - i0);
          const bool more = i0 + G < T;
          const int t = g & (TD - 1);
          const int lo0 = max(0, qg - half);
          qg += qdg; rg += rdg;
          if (rg >= T) { rg -= T; ++qg; }
          const int lo1 = max(0, qg - half);  // lo of the next group's first frame >= lo of every frame here
          // does the compute warp need its neighbour's message for this group?  (same test as
          // kab_bandq.cuh: not if all 24 ghost states are outside the window for the whole group;
          // evaluated with the aliases of the previous group, before recycling)
          const uint32_t flags_first = gi == 1 ? flags : 0u;  // (the chunk's first group)
          flags = 0;
          if (own) {
            const int hi1g = min(lo1 + W, S);  // >= hi of every frame of this group
            const bool outside = owned || vb + 1 < lo_prev || vb >= hi1g;
            flags = (g > 0 && !__all_sync(KAB_FULL_MASK, outside)) ? 1u : 0u;
          }
          lo_prev = lo0;
          if (vb + 1 < lo0 - 3) {  // recycle a chunk that fell below the window (between groups only)
            do {
              vb += R;
              c1 = nc1;
              nc1 = load_col(vb + R);
            } while (vb + 1 < lo0 - 3);
          }
          if (!own) continue;
          const int hi0 = min(lo0 + W, S);
          const bool safe = __all_sync(KAB_FULL_MASK, nfr == G && vb >= lo1 && vb + 2 <= hi0);
          float2 *tile = reinterpret_cast<float2 *>(kab_smem + geo.tile_off + (size_t)cw * (TD * 2048) + (size_t)t * 2048) + lane;
          if (safe) {
#pragma unroll
            for (int f = 0; f < G; ++f)
              tile[f * 32] = make_float2(emission(rowc + f * VB), emission(rowc + f * VB + c1));
          } else {
            // edge warp (or the last, partial group): the exact per-frame window turned into masked emissions
            const int *wl = wtab + st * 32 + gi * G;
#pragma unroll
            for (int f = 0; f < G; ++f) {
              const int lo = wl[f];              // align.py:64
              const int hi = min(lo + W, S);     // align.py:65
              const unsigned a = (unsigned)(vb - lo), wd = (unsigned)(hi - lo);
              float xb = ninf, x1 = ninf;
              if (f < nfr) {
                xb = emission(rowc + f * VB);
                x1 = emission(rowc + f * VB + c1);
              }
              tile[f * 32] = make_float2((a + 0u < wd) ? xb : ninf, (a + 1u < wd) ? x1 : ninf);
            }
          }
          if (!more) vbf[lane] = vb;  // final alias of this lane (the compute warp's forced end state)
          __syncwarp();  // (the tile's STS were issued before this warp's next STS: shared memory keeps a warp's stores in order)
          // (the chunk's second word carries the first group's flag too: the compute warp reads one word per pair)
          if (lane == 0) kab_sts_relaxed_u32(ctrl + 4 * (KAB_BR_C_TILESEQ + t), (uint32_t)(g + 1) | (flags << 31) | (flags_first << 30));
#ifdef KAB_BANDR_TIMING
          pm_safe += safe;
#endif
        }
        KAB_RTM(pc);
        KAB_RTM_ADD(pm_tile, pb, pc);
        if (own) {  // the chunk's rows are in the tiles: give the stage back
          __syncwarp();
          if (lane == 0) kab_mbar_arrive(&eempty[st]);
        }
        if (pp == 0) service_bp();
        KAB_RTM(pd);
        KAB_RTM_ADD(pm_rest, pc, pd);
      }
#ifdef KAB_BANDR_TIMING
      if (lane == 0 && p.debug && pp == 0) {
        long long *d = p.debug + 64 * 16 + gw * 8;
        d[0] = pm_wait; d[1] = pm_tile; d[2] = pm_rest; d[3] = clock64() - pm_start; d[4] = pm_safe; d[5] = n_groups;
      }
#endif
      if (pp == 0) {
        while (bp_issued < n_blocks) service_bp();
        if (lane == 0) kab_bulk_wait0();  // the compute warp's backpointer blocks are in global memory
      }
    } else {
      // ================= compute warp: the recurrence
      // Nothing here waits on a fence: every hand-over is a word that carries its own sequence
      // number, polled in shared memory (the LSU of an SM executes a warp's shared-memory accesses in
      // order, the writers fence on their side), and the words are loaded one group early.
      const uint32_t one = p.one;
      if (owned && slot0 == 0) s0 = 0.0f;  // virtual start state 0, score 0 (align.py:57-58)
      uint32_t bw = 0;  // backpointer nibbles of the current group
      auto frame = [&](const float xb, const float x1, const int sh) {
        const float h1 = __shfl_up_sync(KAB_FULL_MASK, s1, 1);  // state vb - 1
        const float h2 = __shfl_up_sync(KAB_FULL_MASK, s0, 1);  // state vb - 2
        const float h3 = __shfl_up_sync(KAB_FULL_MASK, s1, 2);  // state vb - 3
        float t0, th1, a0, a1, a2, a3;
        // two register pairs feed the three packed adds: (vb, vb - 1) gets both emissions, (vb + 1, vb - 2)
        // the label's -- with the pairs (vb, vb - 1), (vb, vb + 1), (vb - 2, vb - 1) ptxas needed three
        // copies per frame, and a lone warp's frame is issue bound (one instruction every other cycle)
        const unsigned long long pu = kab_pack2(s0, h1), pv = kab_pack2(s1, h2);
        kab_add2p(pu, xb, t0, th1);           // blank <- vb (move 0), vb - 1 (move 1)
        const float th3 = __fadd_rn(h3, xb);  // vb - 3 (move 3)
        kab_add2p(pu, x1, a1, a2);            // label <- vb (move 1), vb - 1 (move 2)
        kab_add2p(pv, x1, a0, a3);            //       <- vb + 1 (move 0), vb - 2 (move 3)
        const float m0 = kab_blank_sel(t0, kab_mm<MM>(th1, p.mm1), kab_mm<MM>(th3, p.mm3), bw, 1u << (sh + 0), 2u << (sh + 0), one);
        const float m1 = kab_label_sel(a0, kab_mm<MM>(a1, p.mm1), kab_mm<MM>(a2, p.mm2), kab_mm<MM>(a3, p.mm3), bw, 1u << (sh + 2), 2u << (sh + 2), one);
        s0 = m0; s1 = m1;
      };
      // mailboxes: mine (messages of the warp below), and the one of the warp above -- in this CTA,
      // or in the next CTA of the cluster (distributed shared memory)
      const bool remote_up = cw == CW - 1;
      const uint32_t up_rank = remote_up ? (rank + 1 == NC ? 0u : rank + 1u) : rank;
      const int up_cw = remote_up ? 0 : cw + 1;
      const uint32_t up_mbox_local = smem0 + (uint32_t)geo.mbox_off + (uint32_t)up_cw * (MD * GH * 16u);
      const uint32_t up_ctrl_local = smem0 + (uint32_t)geo.ctrl_off + (uint32_t)up_cw * 128u;
      // (st.shared::cluster compiles to a generic ST through the shared window -- hundreds of cycles even
      // when the target is this CTA -- so the seven links inside a CTA use plain STS / LDS)
      const uint32_t up_lane_off = (uint32_t)(lane >= 32 - GH ? lane - (32 - GH) : 0) * 16u;
      const uint32_t up_mbox = (remote_up ? kab_mapa(up_mbox_local, up_rank) : up_mbox_local) + up_lane_off;
      const uint32_t up_done = remote_up ? ctrl + 4 * KAB_BR_C_UPDONE : up_ctrl_local + 4 * KAB_BR_C_COMPDONE;
      auto read_up_done = [&]() { return kab_lds_relaxed_u32(up_done); };
      // first warp of a CTA: its progress also goes to the warp below, in the previous CTA of the cluster
      const bool remote_down = cw == 0;
      const uint32_t down_done = kab_mapa(smem0 + (uint32_t)geo.ctrl_off + (uint32_t)(CW - 1) * 128u + 4 * KAB_BR_C_UPDONE,
                                          rank == 0 ? NC - 1 : rank - 1);
      auto publish = [&](uint32_t slot, uint32_t seq) {  // lanes 20..31: the two (score, seq) words of message seq - 1
        if (remote_up) {
          kab_st_cluster_b64(slot, __float_as_uint(s0), seq);
          kab_st_cluster_b64(slot + 8, __float_as_uint(s1), seq);
        } else {
          kab_sts_b64(slot, __float_as_uint(s0), seq);
          kab_sts_b64(slot + 8, __float_as_uint(s1), seq);
        }
      };
      const uint32_t inbox = mbox + (uint32_t)(lane < GH ? lane : 0) * 16u;
      uint32_t up_done_seen = 0;  // groups the warp above is known to have finished
      uint2 pf0 = make_uint2(0, 0), pf1 = pf0;  // message g-1, loaded a group early
      uint32_t tw = kab_lds_relaxed_u32(ctrl + 4 * KAB_BR_C_TILESEQ);  // tile word of group 0
      uint32_t bp_free = 0;       // backpointer blocks whose staging buffer is known to be free
#ifdef KAB_BANDR_TIMING
      long long tm_tile = 0, tm_msg = 0, tm_frames = 0, tm_pub = 0, tm_bp = 0, n_need = 0, tm_wait = 0, tm_fast = 0, n_fast = 0;
      const long long tm_start = clock64();
#endif
      static_assert((TD & (TD - 1)) == 0 && (MD & (MD - 1)) == 0 && (BG & (BG - 1)) == 0 && (KAB_BR_NBB & (KAB_BR_NBB - 1)) == 0,
                    "ring indices are masks");
      // (32-bit shared-window addresses computed once: a generic-to-shared conversion inside the loop
      // costs an S2UR + ULEA on the path to the first frame)
      const uint32_t tiles_lane = smem0 + (uint32_t)geo.tile_off + (uint32_t)cw * (TD * 2048u) + (uint32_t)lane * 8u;
      const uint32_t slotfree_u32 = smem0 + (uint32_t)((2 * NS + cw * TD) * 8);  // &slotfree[cw * TD]
      const uint32_t bpst_lane = bpst + (uint32_t)lane * 4u;  // group g's word: + (g mod (NBB * BG)) * 128
      // end-of-group stores as predicated instructions (no divergent blocks): per-lane flags
      const uint32_t f_l0 = lane == 0, f_dn = lane == 0 && remote_down;
      const uint32_t f_pl = lane >= 32 - GH && !remote_up, f_pr = lane >= 32 - GH && remote_up;
      const int last_common = n_groups - 2;  // the groups 1 .. n_groups - 2 can take the common path
      int room_until = MD - 2;               // ... while the mailbox above is known to have room: g <= room_until
      // ghost lanes <- message g-1 (loaded a group ago, polled until it is there), then message g is
      // loaded for the next group
      auto take_message = [&](int g, bool need) {
        const uint32_t seq = (uint32_t)g;
        const uint32_t slot = inbox + (uint32_t)((g - 1) & (MD - 1)) * (GH * 16u);
        while (!__all_sync(KAB_FULL_MASK, owned || !need || (pf0.y == seq && pf1.y == seq))) {
          pf0 = kab_lds_relaxed_b64(slot);
          pf1 = kab_lds_relaxed_b64(slot + 8);
        }
        if (!owned) {
          s0 = need ? __uint_as_float(pf0.x) : ninf;
          s1 = need ? __uint_as_float(pf1.x) : ninf;
        }
        const uint32_t nslot = inbox + (uint32_t)(g & (MD - 1)) * (GH * 16u);
        pf0 = kab_lds_relaxed_b64(nslot);
        pf1 = kab_lds_relaxed_b64(nslot + 8);
      };
      for (int g = 0; g < n_groups;) {
        // ---- COMMON PATH: two groups (one emission chunk) per pass -- all of them but the first two,
        // the last ones and the rare wait for mailbox room.  Straight-line code: a lone warp pays ~15
        // cycles per conditional block and 4-5 per dependent instruction, and in a chain that runs at
        // its minimal lag EVERY group of every follower arrives just before its message, so the polls
        // (tile word once per pair, neighbour's message per group) are inline, the end-of-group stores
        // are predicated, and the per-pass bookkeeping (loop test, tile word, progress counters, slot
        // hand-back, block test) is paid once per 16 frames.  A warp (re)joining the chain -- its ring
        // slots recycled above the window -- comes through here too and simply waits for its first
        // message: any start-up lag it were given is paid again at EVERY change of the head, i.e.
        // every 18 groups ((18 + lag) / 18 on the whole lattice; measured with a trace of group start
        // times: two groups of intended lag plus the slow general body cost 6 groups per change,
        // 8.4 -> 6.6 ms).  g is even here (the general body below takes two groups per pass).
        while (g >= 2 && g + 1 <= min(last_common, room_until)) {  // (its own compact loop: one backward branch)
          const int t = g & (TD - 1);
          KAB_RTM(fa);
          // the chunk's second tile word (published last) carries both need flags
          while ((tw & 0x3fffffffu) != (uint32_t)g + 2u) tw = kab_lds_relaxed_u32(ctrl + 4 * (KAB_BR_C_TILESEQ + t + 1));
          const bool need0 = (tw & 0x40000000u) != 0u, need1 = (tw >> 31) != 0u;
          const uint32_t tl = tiles_lane + (uint32_t)t * 2048u;
          float2 e[G], e2[G];
#pragma unroll
          for (int f = 0; f < G; ++f)
            asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(e[f].x), "=f"(e[f].y) : "r"(tl + f * 256) : "memory");
          KAB_RTM(fw0);
          take_message(g, need0);
          KAB_RTM(fw1);
#pragma unroll
          for (int f = 0; f < G; ++f)
            asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(e2[f].x), "=f"(e2[f].y) : "r"(tl + 2048 + f * 256) : "memory");
          tw = kab_lds_relaxed_u32(ctrl + 4 * (KAB_BR_C_TILESEQ + ((t + 3) & (TD - 1))));  // next pair's
          const uint32_t up_done_now = read_up_done();  // (used after the frames: mailbox room without a wait)
          bw = 0;
          KAB_RTM(ff0);
#pragma unroll
          for (int f = 0; f < G; ++f) frame(e[f].x, e[f].y, 4 * f);
          KAB_RTM(ff1);
          // message g at once: the warp above is waiting for it
          asm volatile(
              "{\n\t.reg .pred p2, p3;\n\t.reg .b64 q0, q1;\n\t"
              "setp.ne.u32 p2, %0, 0;\n\t"
              "setp.ne.u32 p3, %1, 0;\n\t"
              "mov.b64 q0, {%4, %3};\n\t"
              "mov.b64 q1, {%5, %3};\n\t"
              "@p2 st.shared.v2.b32 [%2], {%4, %3};\n\t"
              "@p2 st.shared.v2.b32 [%2+8], {%5, %3};\n\t"
              "@p3 st.relaxed.cluster.shared::cluster.b64 [%2], q0;\n\t"
              "@p3 st.relaxed.cluster.shared::cluster.b64 [%2+8], q1;\n\t}" ::"r"(f_pl),
              "r"(f_pr), "r"(up_mbox + (uint32_t)(g & (MD - 1)) * (GH * 16u)), "r"((uint32_t)g + 1u), "r"(__float_as_uint(s0)), "r"(__float_as_uint(s1))
              : "memory");
          const uint32_t bw0 = bw;
          KAB_RTM(fx0);
          take_message(g + 1, need1);
          KAB_RTM(fx1);
          bw = 0;
#pragma unroll
          for (int f = 0; f < G; ++f) frame(e2[f].x, e2[f].y, 4 * f);
          KAB_RTM(fx2);
          // message g + 1, then: both groups are finished, their tiles have been read (the prep warps
          // may reuse the slots), progress for the warp below
          asm volatile(
              "{\n\t.reg .pred p0, p1, p2, p3;\n\t.reg .b64 q0, q1;\n\t"
              "setp.ne.u32 p2, %2, 0;\n\t"
              "setp.ne.u32 p3, %3, 0;\n\t"
              "setp.ne.u32 p0, %0, 0;\n\t"
              "setp.ne.u32 p1, %1, 0;\n\t"
              "mov.b64 q0, {%9, %5};\n\t"
              "mov.b64 q1, {%10, %5};\n\t"
              "@p2 st.shared.v2.b32 [%8], {%9, %5};\n\t"
              "@p2 st.shared.v2.b32 [%8+8], {%10, %5};\n\t"
              "@p3 st.relaxed.cluster.shared::cluster.b64 [%8], q0;\n\t"
              "@p3 st.relaxed.cluster.shared::cluster.b64 [%8+8], q1;\n\t"
              "@p0 st.relaxed.cluster.shared::cta.u32 [%4], %5;\n\t"
              "@p0 mbarrier.arrive.shared::cta.b64 _, [%6];\n\t"
              "@p0 mbarrier.arrive.shared::cta.b64 _, [%6+8];\n\t"
              "@p1 st.shared::cluster.u32 [%7], %5;\n\t}" ::"r"(f_l0),
              "r"(f_dn), "r"(f_pl), "r"(f_pr), "r"(ctrl + 4 * KAB_BR_C_COMPDONE), "r"((uint32_t)g + 2u), "r"(slotfree_u32 + (uint32_t)t * 8u),
              "r"(down_done), "r"(up_mbox + (uint32_t)((g + 1) & (MD - 1)) * (GH * 16u)), "r"(__float_as_uint(s0)), "r"(__float_as_uint(s1))
              : "memory");
          {
            const uint32_t ba = bpst_lane + (uint32_t)(g & (KAB_BR_NBB * BG - 1)) * 128u;
            asm volatile("st.shared.u32 [%0], %1;\n\tst.shared.u32 [%0+128], %2;" ::"r"(ba), "r"(bw0), "r"(bw) : "memory");
          }
          up_done_seen = max(up_done_seen, up_done_now);
          room_until = (int)up_done_seen + MD - 2;
          if ((g & (BG - 1)) == BG - 2) {  // the block is complete: hand it to the prep warp's bulk store
            kab_fence_proxy_async_smem();
            kab_fence_cta();
            __syncwarp();
            const int blk = (g >> 4) + 1;  // blocks finished
            static_assert(BG == 16, "g >> 4");
            if (lane == 0) kab_sts_relaxed_u32(ctrl + 4 * KAB_BR_C_BPREADY, (uint32_t)blk);
            // the next block's buffer (that of block blk - NBB) must have left shared memory: the
            // prep warp issued that store 48 groups ago, so this does not wait
            if (blk >= KAB_BR_NBB)
              while (bp_free < (uint32_t)(blk - KAB_BR_NBB + 1)) bp_free = kab_lds_relaxed_u32(ctrl + 4 * KAB_BR_C_BPFREE);
          }
#ifdef KAB_BANDR_TIMING
          { const long long fb = clock64(); tm_fast += fb - fa; n_fast += 2; n_need += need0 + need1; tm_wait += fw1 - fw0 + fx1 - fx0;
            tm_frames += ff1 - ff0 + fx2 - fx1; tm_tile += fw0 - fa;
            if (lane == 0 && p.debug && g < 16384) {  // per-pass trace: start (SM clock), tile wait, both message waits, frames, flags
              long long *d = p.debug + 64 * 26 + ((size_t)gw * 16384 + g) * 2;
              d[0] = fa;
              d[1] = (fw0 - fa) | ((fw1 - fw0) << 12) | ((fx1 - fx0) << 24) | ((ff1 - ff0 + fx2 - fx1) << 36) | ((long long)need0 << 50) | ((long long)need1 << 51);
              d[2] = fb; d[3] = 0;
            } }
#endif
          g += 2;
        }
        if (g >= n_groups) break;
        // ---- GENERAL BODY: one group, every wait spelled out; two per pass so that g stays even
        for (int rep = 0; rep < 2 && g < n_groups; ++rep, ++g) {
        const int gib = g & (BG - 1), blk = g / BG;  // group inside its backpointer block, block index
        const int i0 = g * G, nfr = min(G, T - i0);
        const bool more = i0 + G < T;
        const int t = g % TD;
        KAB_RTM(ta);
#ifdef KAB_BANDR_TIMING
        if (lane == 0 && p.debug && g < 16384) {
          unsigned long long gt;
          asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(gt));
          p.debug[64 * 26 + ((size_t)gw * 16384 + g) * 2] = (long long)gt;
          p.debug[64 * 26 + ((size_t)gw * 16384 + g) * 2 + 1] = 2;
        }
#endif
        // ---- this group's tile (its word was loaded during the previous group)
        while ((tw & 0x3fffffffu) != (uint32_t)(g + 1)) tw = kab_lds_relaxed_u32(ctrl + 4 * (KAB_BR_C_TILESEQ + t));
        const bool need = (tw >> 31) != 0u;
        const float2 *tile = reinterpret_cast<const float2 *>(kab_smem + geo.tile_off + (size_t)cw * (TD * 2048) + (size_t)t * 2048) + lane;
        float2 e[G];
#pragma unroll
        for (int f = 0; f < G; ++f) {  // (volatile: after the poll above, before the hand-back below)
          asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(e[f].x), "=f"(e[f].y) : "r"(kab_smem_u32(tile + f * 32)) : "memory");
        }
        if (more) tw = kab_lds_relaxed_u32(ctrl + 4 * (KAB_BR_C_TILESEQ + (t + 1 == TD ? 0 : t + 1)));
        KAB_RTM(tb);
        KAB_RTM_ADD(tm_tile, ta, tb);
        // ---- ghost lanes: the lower neighbour's top 24 states after its group g-1 (message g-1)
        if (g > 0) {
#ifdef KAB_BANDR_TIMING
          const long long tw0 = clock64();
#endif
          if (need) {
            if (!owned) {
              const uint32_t slot = inbox + (uint32_t)((g - 1) % MD) * (GH * 16u);
              const uint32_t seq = (uint32_t)g;
              while (pf0.y != seq || pf1.y != seq) {
                pf0 = kab_lds_relaxed_b64(slot);
                pf1 = kab_lds_relaxed_b64(slot + 8);
              }
              s0 = __uint_as_float(pf0.x);
              s1 = __uint_as_float(pf1.x);
            }
          } else if (!owned) {
            s0 = ninf; s1 = ninf;
          }
#ifdef KAB_BANDR_TIMING
          tm_wait += clock64() - tw0; n_need += need;
#endif
        }
        // message g (for the next group) may already be there: load it now, check it then
        if (more && !owned) {
          const uint32_t slot = inbox + (uint32_t)(g % MD) * (GH * 16u);
          pf0 = kab_lds_relaxed_b64(slot);
          pf1 = kab_lds_relaxed_b64(slot + 8);
        }
        KAB_RTM(tc);
        KAB_RTM_ADD(tm_msg, tb, tc);
        // ---- the frames
        bw = 0;
        if (nfr == G) {
#pragma unroll
          for (int f = 0; f < G; ++f) frame(e[f].x, e[f].y, 4 * f);
        } else {
#pragma unroll
          for (int f = 0; f < G; ++f)
            if (f < nfr) frame(e[f].x, e[f].y, 4 * f);
        }
        // group g is finished: its tile has been read (the values are in the scores), message g-1 consumed
        __syncwarp();
        if (lane == 0) {
          kab_sts_relaxed_u32(ctrl + 4 * KAB_BR_C_COMPDONE, (uint32_t)(g + 1));
          kab_mbar_arrive(&slotfree[cw * TD + t]);
          if (remote_down) kab_st_cluster_u32(down_done, (uint32_t)(g + 1));
        }
        KAB_RTM(td);
        KAB_RTM_ADD(tm_frames, tc, td);
        // ---- hand the top twelve lanes to the warp above (message g).  Slot g % MD held message
        // g - MD, which the warp above consumed at the start of its group g - MD + 1.
        if (more) {
          if (g >= MD && up_done_seen < (uint32_t)(g - MD + 2)) {  // about to lap the consumer: read its progress
            for (;;) {
              up_done_seen = read_up_done();
              if (up_done_seen >= (uint32_t)(g - MD + 2)) break;
              __nanosleep(100);  // (a free-running warp far ahead of the window: nobody waits for it)
            }
          }
          if (lane >= 32 - GH) publish(up_mbox + (uint32_t)(g % MD) * (GH * 16u), (uint32_t)(g + 1));
        }
        // (the common path's room test reads room_until: without this refresh a warp that once ran
        // into the limit -- every warp does, free-running while its ring slots are outside the window --
        // stayed in this body for the rest of the lattice: 68 % of all groups, found in the ncu source page)
        up_done_seen = max(up_done_seen, read_up_done());
        room_until = (int)up_done_seen + MD - 2;
        KAB_RTM(te);
        KAB_RTM_ADD(tm_pub, td, te);
        // ---- backpointer word of this group -> staging; block finished?
        if (gib == 0 && blk >= KAB_BR_NBB)  // the buffer of block blk - NBB must have left shared memory
          while (bp_free < (uint32_t)(blk - KAB_BR_NBB + 1)) bp_free = kab_lds_relaxed_u32(ctrl + 4 * KAB_BR_C_BPFREE);
        asm volatile("st.shared.u32 [%0], %1;" ::"r"(bpst_lane + (uint32_t)(g & (KAB_BR_NBB * BG - 1)) * 128u), "r"(bw) : "memory");
        if (gib == BG - 1 || !more) {
          kab_fence_proxy_async_smem();  // every lane's words -> visible to the bulk store
          kab_fence_cta();
          __syncwarp();
          if (lane == 0) kab_sts_relaxed_u32(ctrl + 4 * KAB_BR_C_BPREADY, (uint32_t)(blk + 1));
        }
        KAB_RTM(tf);
        KAB_RTM_ADD(tm_bp, te, tf);
        }
      }
#ifdef KAB_BANDR_TIMING
      if (lane == 0 && p.debug) {
        long long *d = p.debug + gw * 16;
        d[0] = tm_tile; d[1] = tm_msg; d[2] = tm_frames; d[3] = tm_pub; d[4] = tm_bp; d[5] = clock64() - tm_start;
        d[6] = n_groups; d[7] = n_need; d[8] = tm_wait;
        p.debug[64 * 16 + 64 * 8 + gw * 2] = tm_fast; p.debug[64 * 16 + 64 * 8 + gw * 2 + 1] = n_fast;
        if (gw < 4) printf("warp %2d (cw %d): common path %lld groups, %lld cycles each: tile wait + loads %lld, message poll %lld, frames %lld\n", gw, cw,
               n_fast, n_fast ? tm_fast / n_fast : 0, n_fast ? tm_tile / n_fast : 0, n_fast ? tm_wait / n_fast : 0, n_fast ? tm_frames / n_fast : 0);
      }
#endif
      // ---- end of the forward pass: cluster-wide forced end state (align.py:99-101)
      kab_fence_cta();
      vb = vbf[lane];  // (written by the prep warp before it published the last tile)
      int cand = -1;
      if (owned) {
        if (vb + 0 < S && s0 > ninf) cand = vb + 0;
        if (vb + 1 < S && s1 > ninf) cand = vb + 1;
      }
      cand = __reduce_max_sync(KAB_FULL_MASK, cand);
      if (lane == 0 && cand >= 0)
        for (uint32_t rr = 0; rr < NC; ++rr) kab_red_max_cluster_s32(kab_mapa(kab_smem_u32(s_vmax), rr), cand);
    }
    echunks = ec0 + (uint32_t)n_chunks;
    __syncthreads();
    kab_cluster_sync();

    const int v = *s_vmax;
    const int status = *s_bad ? 3 : (v < 0 ? 1 : 0);
    if (!is_prod && !is_prep && owned && status == 0 && p.final_score) {  // (compute warps)
      if (vb + 0 == v) p.final_score[lat.index] = s0;
      if (vb + 1 == v) p.final_score[lat.index] = s1;
    }
    if (rank == 0 && tid == 0) {
      p.status[lat.index] = status;
      if (status != 0 && p.final_score) p.final_score[lat.index] = __int_as_float(0x7fc00000);
      if (status == 0) p.end_state[lat.index] = v;  // traceback by kab_bt_maps_kernel / kab_bt_stitch_kernel
    }
    __syncthreads();  // everybody has read s_vmax / s_bad before they are reset for the next lattice
  }
}

// Finiteness of the log-probs of the band lattices (status 3, as everywhere): a streaming pass over
// the rows kab_bandr_kernel has just read (L2-resident for a chapter, 70 us of HBM time for a book),
// launched between the forward pass and the traceback kernels, which skip lattices whose status is
// not 0.  grid (lattices, slabs of KAB_FIN_ROWS rows).
#define KAB_FIN_ROWS 2048
__global__ void __launch_bounds__(256)
kab_finite_rows_kernel(const KabLattice *__restrict__ lats, const float *__restrict__ lp, int V, int32_t *status,
                       float *final_score) {
  const KabLattice lat = lats[blockIdx.x];
  const int64_t r0 = (int64_t)blockIdx.y * KAB_FIN_ROWS;
  if (r0 >= lat.T) return;
  const int64_t n = (min((int64_t)lat.T, r0 + KAB_FIN_ROWS) - r0) * V;
  const float *x = lp + (lat.t_off + r0) * V;
  float poison = 0.0f;
  int64_t i = threadIdx.x;
  const int64_t head = min(n, (int64_t)((4 - ((reinterpret_cast<uintptr_t>(x) >> 2) & 3)) & 3));  // words before a 16-byte boundary
  if (i < head) poison = kab_poison(poison, __ldg(x + i));
  const float4 *x4 = reinterpret_cast<const float4 *>(x + head);
  const int64_t n4 = (n - head) >> 2;
  for (int64_t j = threadIdx.x; j < n4; j += 256) {
    const float4 v = __ldg(x4 + j);
    poison = kab_poison(kab_poison(kab_poison(kab_poison(poison, v.x), v.y), v.z), v.w);
  }
  for (int64_t j = head + (n4 << 2) + threadIdx.x; j < n; j += 256) poison = kab_poison(poison, __ldg(x + j));
  if (__syncthreads_or(poison != poison) && threadIdx.x == 0) {
    status[lat.index] = 3;
    if (final_score) final_score[lat.index] = __int_as_float(0x7fc00000);
  }
}
