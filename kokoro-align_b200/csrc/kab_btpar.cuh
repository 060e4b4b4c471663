// kab_btpar.cuh -- parallel backtrack for the cluster band kernel (kab_bandp.cuh).
//
// The traceback of align.py:21-40 / :99-102 is a chain of T dependent steps
//     v_{t-1} = v_t - move[t][v_t]
// and the in-kernel walker of kab_bandp.cuh spends ~78 cycles on each: a quarter of the time of a
// long lattice, on ONE thread, while the rest of the GPU idles (a plan that uses this kernel has
// at most a few dozen lattices).  The steps are function compositions, so they parallelise
// exactly -- no speculation:
//   1. kab_bt_maps_kernel: the frames are cut into blocks of KAB_BT_BLOCK frames.  For every block and
//      EVERY state of the window at the block's last frame, one thread walks the block backwards
//      and records where it leaves it: maps[block][0][v - lo] = state at the frame before the block
//      (and, in passing, where it stands after every KAB_BT_SUB frames: maps[block][q][v - lo], q > 0,
//      is its state at the frame before sub-block q).
//      T x W steps in total (as many as the forward pass has cells), spread over the whole GPU.
//      Walkers that start in inactive states produce values nobody looks up (their addresses are
//      derived from the ring position, which always stays inside the workspace).
//   2. kab_bt_stitch_kernel (one CTA per lattice): thread 0 composes the maps from the forced end
//      state down -- T / KAB_BT_BLOCK dependent table look-ups -- which yields the true entry
//      state of every block; then the threads re-walk the blocks from their entry states, all
//      blocks at once and every block as KAB_BT_NSUB sub-blocks whose entry states are one look-up in
//      the same maps (best_path): a lone walker costs ~330 cycles per frame, so the re-walk is the
//      length of ONE sub-block;
//   3. kab_bt_gather_kernel: best_labels and best_scores of the path (align.py:105-107), coalesced
//      over the frames.
// Backpointer layouts (template parameter of the kernels):
//   KabBtLayoutP (kab_bandp_kernel): byte of (frame t, state v) at
//     bp[((reg * n_groups + t / 8) * 32 + col) * 8 + t % 8],   slot = v mod R, reg = slot / 104,
//     col = (slot % 104) / 4, move = (byte >> 2 * (slot & 3)) & 3;
//   KabBtLayoutQ (kab_bandq_kernel): 32-bit word of (group t / 8, lane) at
//     bp[((reg * n_groups + t / 8) * 32 + 12 + (slot % 40) / 2) * 4],   reg = slot / 40,
//     move = (word >> (4 * (t % 8) + 2 * (slot & 1))) & 3.
#pragma once
#include "kab_band.cuh"   // KAB_BAND_OW: KabBtLayoutP
#include "kab_bandq.cuh"  // KAB_BQ_GH / KAB_BQ_OW: KabBtLayoutQ
#include "kab_common.cuh"

struct KabBtLayoutP {
  static constexpr int OW = KAB_BAND_OW;  // ring slots per warp region
  static constexpr int GROW = 256;        // bytes per region and 8-frame group
  static __device__ __forceinline__ int move(const unsigned char *gp, int rs, int f) {
    const unsigned int byte = __ldg(gp + ((rs >> 2) << 3) + f);  // (read-only here: the forward kernel wrote it)
    return (int)((byte >> (2 * (rs & 3))) & 3u);
  }
  static __device__ __forceinline__ int byte_off(int rs) { return (rs >> 2) << 3; }  // of the state's codes inside a group's row
};
struct KabBtLayoutQ {
  static constexpr int OW = KAB_BQ_OW;
  static constexpr int GROW = 128;
  static __device__ __forceinline__ int move(const unsigned char *gp, int rs, int f) {
    const uint32_t word = __ldg(reinterpret_cast<const uint32_t *>(gp + (KAB_BQ_GH + (rs >> 1)) * 4));
    return (int)((word >> (4 * f + 2 * (rs & 1))) & 3u);
  }
  static __device__ __forceinline__ int byte_off(int rs) { return (KAB_BQ_GH + (rs >> 1)) * 4; }
};

#define KAB_BT_BLOCK 1024   // frames per block
#define KAB_BT_SUB 256      // frames per sub-block of the re-walk (128: 138 -> 126 us on Gon gitsune, twice the maps)
#define KAB_BT_NSUB (KAB_BT_BLOCK / KAB_BT_SUB)
#define KAB_BT_THREADS 128  // threads per CTA of the map kernel (= entry states per CTA)
#define KAB_BT_PF_AHEAD 6    // groups a lone walker prefetches ahead

struct KabBtMeta {       // one per lattice of the band list (same order)
  int64_t map_off;       // first int32 of this lattice's maps ([n_blocks][KAB_BT_NSUB][wl])
  int32_t first_block;   // prefix sum of n_blocks over the list
  int32_t n_blocks;
  int32_t wl;            // map row length: min(W, S) rounded up to 32
  int32_t pad;
};

// walker: state v, its position rs inside ring region reg, and gp = the backpointer rows of that
// region for the CURRENT 8-frame group (the caller moves it down by 256 bytes per group)
template <class LY>
struct KabBtWalker {
  int v, rs, reg;
  const unsigned char *gp;
  __device__ __forceinline__ void init(int v0, int R, const unsigned char *bp, int64_t stride, int g) {
    v = v0;
    const int slot = v0 % R;
    reg = slot / LY::OW;
    rs = slot - reg * LY::OW;
    gp = bp + reg * stride + (size_t)g * LY::GROW;
  }
  // one frame back (frame f of the current group); returns the state AT that frame (before the move).
  // The region change (once per ~370 frames of a walker) is a real branch into a non-inlined helper:
  // predicated inline it was 9 of the 21 instructions of every step.
  struct Wrap { int reg; long long delta; };
  static __device__ __noinline__ Wrap wrap_region(int reg, int NWT, long long stride) {
    Wrap w;
    const bool first = reg == 0;
    w.reg = first ? NWT - 1 : reg - 1;
    w.delta = first ? (long long)(NWT - 1) * stride : -stride;
    return w;
  }
  __device__ __forceinline__ int step(int f, int NWT, int64_t stride) {
    const int at = v;
    const int mv = LY::move(gp, rs, f);
    v -= mv;  // (a walker that started in an inactive state may run below 0: its value is never used,
    rs -= mv;  //  and the addresses come from rs / reg, which stay inside the workspace)
    if (rs < 0) {  // into the region below (a move crosses at most one boundary)
      rs += LY::OW;
      const Wrap w = wrap_region(reg, NWT, stride);
      reg = w.reg;
      gp += w.delta;
    }
    return at;
  }
  // frames te .. t0 (t0 a multiple of 8), descending; f(t, state at t) for every frame.
  // PF: a LONE walker (the stitch kernel's re-walk: one thread per block, nothing to hide the latency
  // behind) prefetches the rows of the groups it will reach -- a group's row of this region is one
  // 128 / 256-byte line whatever the state, so the address is known ahead -- and then pays L1 hits
  // instead of one L2 round trip per group (measured: 345 -> see DESIGN.md section 3.4).
  template <bool PF = false, class F>
  __device__ __forceinline__ void walk(int te, int t0, int NWT, int64_t stride, F f) {
    int g = te >> 3;
    const int g0 = t0 >> 3;
    // (the sector the walker is heading for and the one below it: a path climbs ~2 states per group,
    // 24 at most, and a state is 2 bytes of a row in both layouts)
    auto prefetch_row = [&](int ahead) {
      const unsigned char *a = gp - (size_t)ahead * LY::GROW + (LY::byte_off(rs) & ~31);
      asm volatile("prefetch.global.L1 [%0];" ::"l"(a));
      if (LY::byte_off(rs) >= 32) asm volatile("prefetch.global.L1 [%0];" ::"l"(a - 32));
    };
    if (PF) {
#pragma unroll
      for (int a = 1; a < KAB_BT_PF_AHEAD; ++a)
        if (g - a >= g0) prefetch_row(a);
    }
    if ((te & 7) != 7) {  // partial group at the top (the last frames of the lattice)
      for (int k = te & 7; k >= 0; --k) f(g * 8 + k, step(k, NWT, stride));
      --g;
      gp -= LY::GROW;
    }
    for (; g >= g0; --g, gp -= LY::GROW) {
      if (PF && g - KAB_BT_PF_AHEAD >= g0) prefetch_row(KAB_BT_PF_AHEAD);
#pragma unroll
      for (int k = 7; k >= 0; --k) f(g * 8 + k, step(k, NWT, stride));
    }
  }
};

__device__ __forceinline__ int kab_bt_lo(int64_t S, int64_t t, int64_t T, int W) {  // align.py:64
  const int64_t lo = S * t / T - W / 2;
  return lo < 0 ? 0 : (int)lo;
}

// grid.x = total blocks of all lattices, grid.y = chunks of KAB_BT_THREADS entry states
template <class LY>
__global__ void __launch_bounds__(KAB_BT_THREADS)
kab_bt_maps_kernel(const KabLattice *__restrict__ lats, const KabBtMeta *__restrict__ meta, int n_lat,
                   const unsigned char *__restrict__ bpw, const int32_t *__restrict__ status, int32_t *__restrict__ maps,
                   int W, int NWT) {
  int li = 0;
  while (li + 1 < n_lat && (int)blockIdx.x >= meta[li + 1].first_block) ++li;
  const KabLattice lat = lats[li];
  const KabBtMeta m = meta[li];
  if (status[lat.index] != 0) return;
  const int b = (int)blockIdx.x - m.first_block;
  const int T = lat.T, S = 2 * lat.L + 1, R = LY::OW * NWT, n_groups = (T + 7) / 8;
  const int t0 = b * KAB_BT_BLOCK, te = min(T, t0 + KAB_BT_BLOCK) - 1;
  const int lo = kab_bt_lo(S, te, T, W), hi = min(lo + W, S);
  const int j = blockIdx.y * KAB_BT_THREADS + threadIdx.x;
  if (lo + j >= hi) return;
  const unsigned char *bp = bpw + lat.bp_off;
  const int64_t stride = (int64_t)n_groups * LY::GROW;
  KabBtWalker<LY> w;
  w.init(lo + j, R, bp, stride, te >> 3);
  int32_t *row = maps + m.map_off + (int64_t)b * KAB_BT_NSUB * m.wl + j;
#pragma unroll 1
  for (int q = KAB_BT_NSUB - 1; q >= 0; --q) {  // (the walker carries on where the sub-block above ended)
    const int s0 = t0 + q * KAB_BT_SUB;
    if (s0 > te) continue;
    w.walk(min(te, s0 + KAB_BT_SUB - 1), s0, NWT, stride, [](int, int) {});
    row[(int64_t)q * m.wl] = w.v;
  }
}

// one CTA per lattice
template <class LY>
__global__ void __launch_bounds__(1024)
kab_bt_stitch_kernel(const KabLattice *__restrict__ lats, const KabBtMeta *__restrict__ meta, KabParams p,
                     const int32_t *__restrict__ end_state, const int32_t *__restrict__ maps,
                     int32_t *__restrict__ entry, int NWT) {
  const KabLattice lat = lats[blockIdx.x];
  const KabBtMeta m = meta[blockIdx.x];
  if (p.status[lat.index] != 0) return;
  const int T = lat.T, S = 2 * lat.L + 1, W = p.W, R = LY::OW * NWT, n_groups = (T + 7) / 8;
  int32_t *ent = entry + m.first_block;
  // window start of every block's last frame (64-bit divisions): all threads, off the chain below
  for (int b = threadIdx.x; b < m.n_blocks; b += blockDim.x)
    ent[b] = kab_bt_lo(S, min(T, (b + 1) * KAB_BT_BLOCK) - 1, T, W);
  __syncthreads();
#ifdef KAB_BT_TIMING
  const long long tt0 = clock64();
#endif
  if (threadIdx.x == 0) {  // compose the block maps from the forced end state down: one L2 load per block
    int v = end_state[lat.index];
    for (int b = m.n_blocks - 1; b >= 0; --b) {
      const int lo = ent[b];
      ent[b] = v;
      v = __ldcg(&maps[m.map_off + (int64_t)b * KAB_BT_NSUB * m.wl + (v - lo)]);
    }
  }
  __syncthreads();
#ifdef KAB_BT_TIMING
  const long long tt1 = clock64();
#endif
  // every block re-walked from its entry state, one thread each: only the backpointer bytes are on
  // the dependent chain (eight frames share a sector)
  const unsigned char *bp = p.bp + lat.bp_off;
  const int64_t stride = (int64_t)n_groups * LY::GROW;
  int32_t *out_path = p.best_path + lat.t_off;
  for (int k = threadIdx.x; k < m.n_blocks * KAB_BT_NSUB; k += blockDim.x) {
    const int b = k / KAB_BT_NSUB, q = k % KAB_BT_NSUB;
    const int t0 = b * KAB_BT_BLOCK, te = min(T, t0 + KAB_BT_BLOCK) - 1;
    const int s0 = t0 + q * KAB_BT_SUB;
    if (s0 > te) continue;
    const int se = min(te, s0 + KAB_BT_SUB - 1);
    int v0 = ent[b];  // the block's entry state; a lower sub-block starts where the walker from there left the one above
    if (se != te) v0 = __ldcg(&maps[m.map_off + ((int64_t)b * KAB_BT_NSUB + q + 1) * m.wl + (v0 - kab_bt_lo(S, te, T, W))]);
    KabBtWalker<LY> w;
    w.init(v0, R, bp, stride, se >> 3);
    w.template walk<true>(se, s0, NWT, stride, [&](int t, int at) { out_path[t] = at; });
  }
#ifdef KAB_BT_TIMING
  if (threadIdx.x < 3 || threadIdx.x == 79) printf("stitch thread %d: compose %lld cycles, walk %lld cycles (%d blocks)\n", threadIdx.x, tt1 - tt0, clock64() - tt1, m.n_blocks);
#endif
}

// labels and scores of the path (align.py:105-107): grid (lattices, chunks of 4096 frames), coalesced
#define KAB_BT_GATHER_FRAMES 4096
__global__ void __launch_bounds__(256)
kab_bt_gather_kernel(const KabLattice *__restrict__ lats, KabParams p) {
  const KabLattice lat = lats[blockIdx.x];
  const int f0 = blockIdx.y * KAB_BT_GATHER_FRAMES;
  if (f0 >= lat.T || p.status[lat.index] != 0) return;
  const int f1 = min(lat.T, f0 + KAB_BT_GATHER_FRAMES), V = p.V;
  const uint16_t *col16 = p.col16 + lat.col_off;
  const int32_t *path = p.best_path + lat.t_off;
  int32_t *out_lab = p.best_labels + lat.t_off;
  float *out_sc = p.best_scores + lat.t_off;
  const float *lp = p.lp + lat.t_off * (int64_t)V;
  for (int t = f0 + threadIdx.x; t < f1; t += blockDim.x) {
    const int pv = path[t];
    const int lab = (pv & 1) ? (int)col16[(pv - 1) >> 1] : 0;
    out_lab[t] = lab;                              // align.py:106
    out_sc[t] = __ldg(&lp[(int64_t)t * V + lab]);  // align.py:107
  }
}
