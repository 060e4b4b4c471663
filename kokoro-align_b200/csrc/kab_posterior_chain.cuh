// kab_posterior_chain.cuh -- forward-backward posteriors of unbanded long-form lattices too wide for one CTA
// (kab_plan_ctc_posteriors_device, DESIGN.md 3.9g), sm_100a.
//
// The recurrence, the outputs and their scratch are those of kab_posterior.cuh (the fwd / bwd value rows of
// KabPostParams, then kab_ctc_posterior_combine_kernel); only the layout differs.  The lattice's L + 1 pairs
// (forward: blank 2k, label 2k+1; backward: label 2k-1, blank 2k) are cut into slices of KAB_PC_K pairs per
// lane, 32 K pairs per WARP, and the warps are spread over the whole GPU (cooperative launch: all resident):
//   * a CHAIN per direction: a lane needs one state of the previous frame from below (forward: the label
//     state 2k-1 under its first pair) or from above (backward: y = beta + e of the label state 2k+1 over its
//     last pair).  Inside a warp that is one shuffle; across warps it travels through a FIFO in global
//     memory (L2), one message per group of KAB_PC_G frames: the boundary value of each frame and the
//     sender's offset, every word together with the message's sequence number as ONE 8-byte single-copy-
//     atomic store -- no fence, no flag (the wide kernel's protocol, kab_wide.cuh).  The receiver loads the
//     next message a group early, publishes how many it has consumed, and the sender reads that count only
//     when it is about to lap it.  A warp starts once its neighbour has finished KAB_PC_LAG groups, so the
//     chain runs as a wavefront and the messages are there when they are read;
//   * normalisation without communication: every warp keeps its own offset (double).  Every frame it subtracts
//     its drift c, the mean change of its maximum per frame (folded into the emissions: one FFMA), and at the
//     end of every group it subtracts what is left of its maximum (one redux) and adds that / G to c, so the
//     values stay within a few units of 0 (the precision of the single-CTA pass's per-frame renormalisation).
//     A message carries the sender's offset (as a hi / lo float pair) and drift, and the receiver moves the
//     boundary values onto its own offset; a warp that holds no finite value yet adopts the sender's offset
//     and drift, so values that enter a warp are never rounded against an offset far from them;
//   * emissions are read by label from global memory (L2: every warp reads the same rows within a few
//     microseconds), one group ahead, by asynchronous copies into the lane's column of two shared-memory
//     stages; any vocab_size works.  Path entries are loaded a group ahead as well;
//   * the owner of the path state p_t writes alpha_t(p_t) (beta_t(p_t)) + its offset, natural log, in double;
//     the owner of state S-1 also writes log Z.  Both directions run side by side when the grid fits, else
//     every warp runs the forward pass and then the backward pass.
#pragma once
#include <climits>
#include "kab_posterior.cuh"

#define KAB_PC_K 4       // pairs per lane (8 states, 16 MUFU operations per frame)
#define KAB_PC_G 8       // frames per group: one message, one renormalisation
#define KAB_PC_D 32      // FIFO depth (messages)
#define KAB_PC_LAG 2     // groups the neighbour is ahead when a warp starts
#define KAB_PC_CW 4      // warps per CTA
#define KAB_PC_MSG 128   // bytes per message: G (value, seq) words, then the offset's (hi, seq), (lo, seq) and
                         // the drift's (c, seq)
#define KAB_PC_PAIRS (32 * KAB_PC_K)

// One lattice of the chain pass
struct KabPostChainLat {
  int64_t t_off, l_off;  // first row / first label
  int64_t ws_off;        // byte offset of its workspace: cons[2][nw] (messages consumed), fifo[2][nw][D][MSG]
  int32_t T, S;
  int32_t index;         // position in the batch
  int32_t nw;            // warps per direction: ceil((L + 1) / (32 K))
};

__host__ __device__ inline size_t kab_pc_fifo_off(int nw) { return ((size_t)2 * nw * 4 + 127) & ~(size_t)127; }
__host__ __device__ inline size_t kab_pc_ws_bytes(int nw) {
  return kab_pc_fifo_off(nw) + (size_t)2 * nw * KAB_PC_D * KAB_PC_MSG;
}

// 4-byte asynchronous global -> shared copies (LDGSTS), waited for by the issuing thread
__device__ __forceinline__ void kab_cp_async4(float *dst, const float *src) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(kab_smem_u32(dst)), "l"(src) : "memory");
}
__device__ __forceinline__ void kab_cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void kab_cp_async_wait0() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void kab_cp_async_wait1() { asm volatile("cp.async.wait_group 1;" ::: "memory"); }

// maximum over the warp (every lane gets it): floats ordered as ints, one redux
__device__ __forceinline__ float kab_pc_warp_max(float x) {
  const int i = __float_as_int(x);
  const int k = __reduce_max_sync(KAB_FULL_MASK, i >= 0 ? i : i ^ 0x7fffffff);
  return __int_as_float(k >= 0 ? k : k ^ 0x7fffffff);
}

// x[d] for d < 8 by a tree of selects on the bits of d (an indexed register array would go to local memory)
__device__ __forceinline__ float kab_pc_pick(const float (&x)[2 * KAB_PC_K], const unsigned d) {
  static_assert(2 * KAB_PC_K == 8, "three levels of selects");
  const bool b0 = d & 1u, b1 = d & 2u, b2 = d & 4u;
  const float a0 = b0 ? x[1] : x[0], a1 = b0 ? x[3] : x[2], a2 = b0 ? x[5] : x[4], a3 = b0 ? x[7] : x[6];
  const float c0 = b1 ? a1 : a0, c1 = b1 ? a3 : a2;
  return b2 ? c1 : c0;
}

template <bool BACK>
__device__ __forceinline__ void kab_pc_run(const KabPostChainLat &lat, const KabPostParams &p, unsigned char *ws,
                                           float *estage, const int w, const int lane) {
  constexpr int K = KAB_PC_K, G = KAB_PC_G, D = KAB_PC_D, MSG = KAB_PC_MSG;
  const float ninf = kab_neg_inf();
  const float LOG2E = 1.4426950408889634f;
  const double LN2 = 0.6931471805599453;
  const int T = lat.T, S = lat.S, L = (S - 1) / 2, nw = lat.nw;
  if (p.status[lat.index] != 0 || T <= 0) {
    if (!BACK && w == 0 && lane == 0)
      p.log_likelihood[lat.index] = T <= 0 ? (double)ninf : __longlong_as_double(0x7ff8000000000000ll);
    return;
  }
  const int n_groups = (T + G - 1) / G;
  const int k0 = (w * 32 + lane) * K;            // first pair of this lane
  const int base = BACK ? 2 * k0 - 1 : 2 * k0;   // first state of this lane
  const bool has_end = k0 <= L && L < k0 + K;    // owns pair L (state S-1)
  // the path states this lane answers for: its own, plus those below 0 (first lane) and from S up (has_end)
  const int own_lo = k0 == 0 ? INT_MIN : base, own_hi = has_end ? INT_MAX : base + 2 * K;
  const int32_t *labs = p.labs + lat.l_off;
  const float *rows = p.lp + lat.t_off * (int64_t)p.V;
  const int32_t *path = p.path + p.path_skew + lat.t_off;
  double *out = (BACK ? p.bwd : p.fwd) + lat.t_off;

  // pair j: the label's column, and bit j of: label state inside the lattice / blank state inside / move 2
  // allowed (forward: into the label 2k+1; backward: out of the label 2k-1)
  int col[K];
  uint32_t lval = 0, bval = 0, allow = 0;
#pragma unroll
  for (int j = 0; j < K; ++j) {
    const int k = k0 + j, li = BACK ? k - 1 : k;
    const bool lv = li >= 0 && li < L;
    const int32_t lw = lv ? __ldg(labs + li) : 0;
    col[j] = lv ? (lw & 0xffff) : p.blank;
    lval |= (uint32_t)lv << j;
    bval |= (uint32_t)(k <= L) << j;
    allow |= (uint32_t)(lv && (((uint32_t)lw >> (BACK ? 30 : 31)) & 1u)) << j;
  }

  // the chain: forward values climb (warp w-1 -> w), backward values descend (w+1 -> w)
  const int src = BACK ? w + 1 : w - 1, dst = BACK ? w - 1 : w + 1;
  const bool has_src = src >= 0 && src < nw, has_dst = dst >= 0 && dst < nw;
  const int edge = BACK ? 31 : 0;       // the lane whose neighbour state lives in warp src
  const int send_lane = BACK ? 0 : 31;  // the lane whose boundary state warp dst needs
  unsigned int *cons = reinterpret_cast<unsigned int *>(ws) + (BACK ? nw : 0);
  unsigned char *fifo = ws + kab_pc_fifo_off(nw) + (size_t)(BACK ? nw : 0) * D * MSG;
  const unsigned char *inbox = fifo + (size_t)w * D * MSG + lane * 8;  // lanes 0 .. G+1: one word each
  unsigned char *outbox = fifo + (size_t)(has_dst ? dst : 0) * D * MSG;
  constexpr int NWORDS = G + 3;
  uint2 pf = make_uint2(0u, 0u);
  auto poll = [&](int g) {
    if (lane < NWORDS) pf = kab_ld_volatile_b64(inbox + (size_t)(g % D) * MSG);
  };
  // message g is complete when the words of its frames and of the offset carry seq g + 1 (the words of frames
  // past T are never written)
  auto arrived = [&](int g) {
    const bool mine = lane < min(G, T - g * G) || (lane >= G && lane < NWORDS);
    return __all_sync(KAB_FULL_MASK, !mine || pf.y == (uint32_t)(g + 1));
  };

  // emissions of a group's frames, copied asynchronously into this lane's column of the warp's two stages
  // ([stage][f][0] the blank, [f][1 + j] pair j's label); the path entry of frame f in lane f
  float *stg = estage + lane;
  int pc = 0, pn = 0;
  auto load_group = [&](int g, int &pth) {
    float *dst = stg + (g & 1) * G * (K + 1) * 32;
#pragma unroll
    for (int f = 0; f < G; ++f) {
      const int s = min(g * G + f, T - 1), t = BACK ? T - 1 - s : s;
      const float *r = rows + (int64_t)t * p.V;
      kab_cp_async4(dst + (f * (K + 1)) * 32, r + p.blank);
#pragma unroll
      for (int j = 0; j < K; ++j) kab_cp_async4(dst + (f * (K + 1) + j + 1) * 32, r + col[j]);
    }
    kab_cp_async_commit();
    const int s = min(g * G + (lane & (G - 1)), T - 1);
    pth = __ldg(path + (BACK ? T - 1 - s : s));
  };
  load_group(0, pc);

  // ---- the wavefront: start once warp src has finished KAB_PC_LAG groups (or all of them)
  if (has_src) {
    const int g0 = min(KAB_PC_LAG, n_groups) - 1;
    poll(g0);
    while (!arrived(g0)) {
      __nanosleep(64);
      poll(g0);
    }
    poll(0);
  }

  float v[2 * K];  // forward: alpha (blank 2k, label 2k+1); backward: y = beta + e (label 2k-1, blank 2k)
#pragma unroll
  for (int i = 0; i < 2 * K; ++i) v[i] = ninf;
  // this warp's offset (base 2) at the start of the group, and its drift: after frame f of the group the true
  // value of a state is v + off + (f + 1) c
  double off = 0.0;
  float c = 0.0f;
  bool dead = true;       // no finite value in the warp: adopt the sender's offset and drift
  float hraw = ninf;      // warp src's boundary value of the last frame of the previous group, its offset osp
  double osp = 0.0;
  float mv = ninf;        // lane f < G: warp src's boundary value after frame f of this group, on this warp's
                          // offset after frame f
  uint32_t cons_seen = 0;

  for (int g = 0; g < n_groups; ++g) {
    const int nfr = min(G, T - g * G);
    const bool more = g + 1 < n_groups;
    float hfirst = ninf;  // (edge lane) the neighbour value for the group's first frame
    if (has_src) {
      while (!arrived(g)) poll(g);
      const float ohi = __uint_as_float(__shfl_sync(KAB_FULL_MASK, pf.x, G));
      const float olo = __uint_as_float(__shfl_sync(KAB_FULL_MASK, pf.x, G + 1));
      const float cs = __uint_as_float(__shfl_sync(KAB_FULL_MASK, pf.x, G + 2));
      const double os = (double)ohi + (double)olo;
      if (dead) { off = os; c = cs; }
      mv = __uint_as_float(pf.x) + ((float)(os - off) + (float)(lane + 1) * (cs - c));
      if (g > 0) hfirst = hraw + (float)(osp - off);
      hraw = __uint_as_float(__shfl_sync(KAB_FULL_MASK, pf.x, G - 1));
      osp = os + (double)cs * G;  // (the sender's offset after the group's last frame)
      if (lane == 0) kab_st_volatile_u32(&cons[w], (uint32_t)(g + 1));  // g + 1 messages consumed
      if (more) poll(g + 1);  // checked at the next group
    }
    if (more) load_group(g + 1, pn);
    if (more) kab_cp_async_wait1(); else kab_cp_async_wait0();  // this group's stage has landed
    const float *ec = stg + (g & 1) * G * (K + 1) * 32;
    unsigned char *slot = outbox + (size_t)(g % D) * MSG;
    if (has_dst) {
      if (g >= D && (uint32_t)(g - D) >= cons_seen) {  // about to lap the receiver: read its progress
        do {
          cons_seen = kab_ld_volatile_u32(&cons[dst]);
        } while ((uint32_t)(g - D) >= cons_seen);
      }
      if (lane == send_lane) {
        const float ohi = (float)off;
        kab_st_volatile_b64(slot + G * 8, __float_as_uint(ohi), (uint32_t)(g + 1));
        kab_st_volatile_b64(slot + G * 8 + 8, __float_as_uint((float)(off - (double)ohi)), (uint32_t)(g + 1));
        kab_st_volatile_b64(slot + G * 8 + 16, __float_as_uint(c), (uint32_t)(g + 1));
      }
    }
#pragma unroll
    for (int f = 0; f < G; ++f) {
      if (f < nfr) {
        const int s = g * G + f, t = BACK ? T - 1 - s : s;
        const bool init = s == 0;
        const float hin = BACK ? __shfl_down_sync(KAB_FULL_MASK, v[0], 1) : __shfl_up_sync(KAB_FULL_MASK, v[2 * K - 1], 1);
        const float hm = f == 0 ? hfirst : __shfl_sync(KAB_FULL_MASK, mv, f - 1);
        const float h = lane == edge ? (has_src ? hm : ninf) : hin;
        float nv[2 * K], o[2 * K];  // new values; the values at frame t (forward: alpha; backward: beta)
#pragma unroll
        for (int j = 0; j < K; ++j) {
          const float eb = fmaf(ec[(f * (K + 1)) * 32], LOG2E, -c), el = fmaf(ec[(f * (K + 1) + j + 1) * 32], LOG2E, -c);
          if (!BACK) {
            const float x1 = j == 0 ? h : v[2 * j - 1], x0 = v[2 * j], xn = v[2 * j + 1];
            float xb, xl;
            if (init) {
              xb = k0 + j == 0 ? 0.0f : ninf;
              xl = xb;
            } else {
              xb = kab_lse2(x0, x1);
              xl = kab_lse2(xn, (allow >> j) & 1u ? xb : x0);
            }
            nv[2 * j] = (bval >> j) & 1u ? xb + eb : ninf;
            nv[2 * j + 1] = (lval >> j) & 1u ? xl + el : ninf;
            o[2 * j] = nv[2 * j];
            o[2 * j + 1] = nv[2 * j + 1];
          } else {
            const float yl = v[2 * j], yb = v[2 * j + 1], yn = j == K - 1 ? h : v[2 * j + 2];
            float bb, bl;
            if (init) {
              bb = k0 + j == L ? 0.0f : ninf;
              bl = bb;
            } else {
              bb = kab_lse2(yb, yn);
              bl = kab_lse2(yl, (allow >> j) & 1u ? bb : yb);
            }
            bb = (bval >> j) & 1u ? bb : ninf;
            bl = (lval >> j) & 1u ? bl : ninf;
            o[2 * j] = bl;
            o[2 * j + 1] = bb;
            nv[2 * j] = bl + el;
            nv[2 * j + 1] = bb + eb;
          }
        }
#pragma unroll
        for (int i = 0; i < 2 * K; ++i) v[i] = nv[i];
        // the value at the path state, by the lane that answers for it
        const int pt = __shfl_sync(KAB_FULL_MASK, pc, f);
        if (pt >= own_lo && pt < own_hi) {
          const unsigned d = (unsigned)(pt - base);
          const float x = pt >= 0 && pt < S && d < 2 * K ? kab_pc_pick(o, d) : ninf;
          // (forward: alpha after this frame's drift; backward: beta, before it)
          out[t] = kab_finite(x) ? ((double)x + off + (double)c * (BACK ? f : f + 1)) * LN2 : (double)ninf;
        }
        if (has_dst && lane == send_lane)
          kab_st_volatile_b64(slot + f * 8, __float_as_uint(BACK ? v[0] : v[2 * K - 1]), (uint32_t)(g + 1));
      }
    }
    off += (double)c * nfr;
    if (more) {  // renormalise by what is left of the warp's maximum, and correct the drift by it
      float m = v[0];
#pragma unroll
      for (int i = 1; i < 2 * K; ++i) m = fmaxf(m, v[i]);
      m = kab_pc_warp_max(m);
      dead = m == ninf;
      if (!dead) {
#pragma unroll
        for (int i = 0; i < 2 * K; ++i) v[i] -= m;
        off += (double)m;
        c += m * (1.0f / G);
      }
      pc = pn;
    }
  }
  if (!BACK) {  // log Z = lse(alpha_{T-1}(S-1), alpha_{T-1}(S-2)) by the owner of S-1
    const int nfl = T - (n_groups - 1) * G;
    const float hin = __shfl_up_sync(KAB_FULL_MASK, v[2 * K - 1], 1);
    const float hm = __shfl_sync(KAB_FULL_MASK, mv, nfl - 1);
    const float h = lane == 0 ? (has_src ? hm : ninf) : hin;  // alpha_{T-1} of the state under the lane
    if (has_end) {
      const int j = L - k0;  // S-1 is state 2 j of the lane, S-2 state 2 j - 1 (j = 0: the state under it)
      const float a1 = kab_pc_pick(v, 2 * j), a2 = j > 0 ? kab_pc_pick(v, 2 * j - 1) : h;
      const float z = kab_lse2(a1, a2);
      p.log_likelihood[lat.index] = z == ninf ? (double)ninf : ((double)z + off) * LN2;
    }
  }
}

// Grid: CTAs of KAB_PC_CW warps, all resident.  split > 0: warps [0, split) run the forward pass and warps
// [split, 2 split) the backward pass, side by side; split == 0: every warp runs both, forward first.  Every
// warp walks the lattices in the same order (a lattice uses its first nw warps of each direction).
__global__ void __launch_bounds__(KAB_PC_CW * 32, 4)
    kab_ctc_posterior_chain_kernel(const KabPostChainLat *__restrict__ lats, int n_lat, KabPostParams p,
                                   unsigned char *ws, int split) {
  __shared__ float s_stage[KAB_PC_CW][2 * KAB_PC_G * (KAB_PC_K + 1) * 32];
  const int lane = threadIdx.x & 31;
  float *estage = s_stage[threadIdx.x >> 5];
  const int gw = (int)blockIdx.x * KAB_PC_CW + (threadIdx.x >> 5);
  const int w = split > 0 && gw >= split ? gw - split : gw;
  const bool fwd = split == 0 || gw < split, bwd = split == 0 || gw >= split;
  for (int li = 0; li < n_lat; ++li) {
    const KabPostChainLat lat = lats[li];
    if (w >= lat.nw) continue;
    unsigned char *lws = ws + lat.ws_off;
    if (fwd) kab_pc_run<false>(lat, p, lws, estage, w, lane);
    if (bwd) kab_pc_run<true>(lat, p, lws, estage, w, lane);
  }
}
