// kab_posterior.cuh -- forward-backward posteriors of a CTC state path and the lattice log-likelihood
// (kab_plan_ctc_posteriors_device, DESIGN.md 3.9f), sm_100a.
//
// The sum-product recurrence over the lattice of a CTC plan (torchaudio's CTC lattice: blank-interleaved
// states, move 2 into an odd state whose label differs from the one two states down), in the plan's window
// [lo_t, hi_t) of every frame.  Only ONE value per frame leaves each pass: the log forward (or backward)
// value at the path state p_t, so nothing of size T x S is stored.
//
//   kab_ctc_posterior_kernel<NT>: one CTA per (lattice, direction); blockIdx.x = 2 * i + (backward).  The
//     window's states live in two shared-memory buffers (one barrier per frame).  Emission rows and path
//     states are staged ahead in a ring of KAB_POST_NST chunks of F frames by 1-D bulk copies.  Values are
//     base 2 (log-probs scaled by log2(e) as they are read) and renormalised every frame by the previous
//     frame's value at the path state; thread 0 adds those offsets up in double.
//   kab_ctc_posterior_combine_kernel: gamma_t = exp(fwd_t + bwd_t - log Z) in double, per frame.
#pragma once
#include "kab_common.cuh"

#define KAB_POST_NST 4    // ring chunks in flight
#define KAB_POST_PAD 8    // -inf slots below the window's first pair (the backward pass reads up to 7 below)
#define KAB_POST_TAIL 8   // -inf slots above the last pair (the forward pass reads up to 7 above)

// One lattice of a posterior launch (a list per block size, longest first)
struct KabPostLat {
  int64_t t_off, l_off;  // first row / first label
  int32_t T, S;          // frames, states (2L + 1)
  int32_t index;         // position in the batch (status, log-likelihood)
  int32_t np;            // pair slots per frame: min(W, S) / 2 + 2
  int32_t banded;        // the window moves (the plan's W clips it somewhere); else [0, S) in every frame
};

struct KabPostParams {
  const float *lp;          // the caller's [sum T, V] log-probs (16-byte aligned)
  int64_t lp_bytes;
  const int32_t *path;      // best_path rounded down to 16 bytes; entry t_off + path_skew is row t_off
  int64_t path_bytes;       // bytes from `path` to the end of best_path
  int32_t path_skew;
  const int32_t *labs;      // [sum L]: label | bit 31: move 2 into it allowed | bit 30: move 2 out of it allowed
  const int32_t *status;    // [B] the alignment's statuses
  double *fwd, *bwd;        // [sum T] log forward / backward value at the path state (natural log)
  double *log_likelihood;   // [B]
  int64_t W;                // the plan's beam (CTC_W: the whole lattice)
  int32_t V, blank;
  int32_t F;                // frames per ring chunk
  int32_t e_words, p_words; // words of a chunk's emission rows (0: rows are read from global) and path entries
  int32_t bufcap;           // words of one state buffer
};

__device__ __forceinline__ float kab_ex2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float kab_lg2(float x) {
  float y;
  asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
// log2(2^a + 2^b): two MUFU operations; both -inf gives -inf (not the NaN of -inf - -inf)
__device__ __forceinline__ float kab_lse2(float a, float b) {
  const float m = fmaxf(a, b);
  const float r = m + kab_lg2(1.0f + kab_ex2(fminf(a, b) - m));
  return m == kab_neg_inf() ? m : r;
}

// floor(S * t / T) for consecutive t, without a 64-bit division per frame (S < 3 T + 1 in every lattice that
// reaches the kernel: T >= L + R, so the quotient moves by at most 3 per frame)
struct KabDiag {
  int64_t q, r, S, T;
  __device__ void init(int64_t S_, int64_t T_, int64_t t) { S = S_; T = T_; q = S * t / T; r = S * t - q * T; }
  __device__ void up() { r += S; while (r >= T) { r -= T; ++q; } }
  __device__ void down() { r -= S; while (r < 0) { r += T; --q; } }
};

template <int NT>
__global__ void __launch_bounds__(NT) kab_ctc_posterior_kernel(const KabPostLat *__restrict__ lats, KabPostParams p) {
  extern __shared__ __align__(16) unsigned char smem[];
  uint64_t *bars = reinterpret_cast<uint64_t *>(smem);
  float *s_pv = reinterpret_cast<float *>(smem + 8 * KAB_POST_NST);  // [2] value at the path state, by step parity
  float *ring = reinterpret_cast<float *>(smem + 8 * KAB_POST_NST + 16);
  const int stage_words = p.e_words + p.p_words;
  float *bufa = ring + KAB_POST_NST * stage_words;
  float *bufb = bufa + p.bufcap;

  const KabPostLat lat = lats[blockIdx.x >> 1];
  const bool back = blockIdx.x & 1;
  const int tid = threadIdx.x;
  const float ninf = kab_neg_inf();
  if (p.status[lat.index] != 0) {
    if (!back && tid == 0) p.log_likelihood[lat.index] = __longlong_as_double(0x7ff8000000000000ll);
    return;
  }
  const int T = lat.T, S = lat.S, L = (S - 1) / 2, np = lat.np, F = p.F;
  const int n_chunks = (T + F - 1) / F;
  const bool staged = p.e_words > 0;
  const float LOG2E = 1.4426950408889634f;
  const double LN2 = 0.6931471805599453;

  if (tid == 0) {
    for (int s = 0; s < KAB_POST_NST; ++s) kab_mbar_init(&bars[s], 1);
    kab_fence_mbar_init();
  }
  for (int i = tid; i < 2 * p.bufcap; i += NT) bufa[i] = ninf;
  __syncthreads();

  // chunk c holds steps [c F, c F + F): frames [f0, f0 + nf), ascending (forward) or descending (backward)
  auto chunk_frames = [&](int c, int &f0, int &nf) {
    if (!back) { f0 = c * F; nf = min(F, T - f0); }
    else { const int f1 = T - c * F; f0 = max(0, f1 - F); nf = f1 - f0; }
  };
  KabParams qe{}, qp{};
  qe.lp = p.lp; qe.lp_bytes = p.lp_bytes; qe.V = p.V;
  qp.lp = reinterpret_cast<const float *>(p.path); qp.lp_bytes = p.path_bytes; qp.V = 1;
  const int64_t path_row0 = lat.t_off + p.path_skew;
  auto issue = [&](int c) {
    int f0, nf;
    chunk_frames(c, f0, nf);
    float *dst = ring + (c % KAB_POST_NST) * stage_words;
    KabStageDesc de{};
    if (staged) de = kab_stage_desc(qe, lat.t_off, f0, nf);
    const KabStageDesc dp = kab_stage_desc(qp, path_row0, f0, nf);
    uint64_t *bar = &bars[c % KAB_POST_NST];
    if (tid == 0) {
      kab_mbar_expect_tx(bar, de.bytes + dp.bytes);
      if (de.bytes) kab_bulk_g2s(dst, de.src, de.bytes, bar);
      if (dp.bytes) kab_bulk_g2s(dst + p.e_words, dp.src, dp.bytes, bar);
    }
    if (tid < (int)de.tail_n) dst[de.tail_word + tid] = __ldg(reinterpret_cast<const float *>(de.src) + de.tail_word + tid);
    if (tid < (int)dp.tail_n)
      dst[p.e_words + dp.tail_word + tid] = __ldg(reinterpret_cast<const float *>(dp.src) + dp.tail_word + tid);
  };
  // the reader's view of chunk c: its first frame and the word offsets of row 0 / path entry 0
  int cf0 = 0, e_skew = 0, p_skew = 0;
  const float *ce = nullptr, *cp = nullptr;
  auto open = [&](int c) {
    int nf;
    chunk_frames(c, cf0, nf);
    const float *base = ring + (c % KAB_POST_NST) * stage_words;
    if (staged) e_skew = (int)kab_stage_desc(qe, lat.t_off, cf0, nf).skew;
    p_skew = (int)kab_stage_desc(qp, path_row0, cf0, nf).skew;
    ce = base + e_skew;
    cp = base + p.e_words + p_skew;
  };
  for (int c = 0; c < min(KAB_POST_NST, n_chunks); ++c) issue(c);
  if (tid == 0) kab_mbar_wait(&bars[0], 0);
  __syncthreads();
  open(0);

  const int64_t W = p.W, half = W / 2;
  KabDiag dg;
  dg.init(S, T, back ? T - 1 : 0);
  const int32_t *labs = p.labs + lat.l_off;
  const float *lp_rows = p.lp + lat.t_off * (int64_t)p.V;
  double *out = (back ? p.bwd : p.fwd) + lat.t_off;
  double off = 0.0;  // (thread 0) the offsets subtracted so far, base 2
  float *prev = bufa, *cur = bufb;
  int pplo = 0, plo = 0, lo = 0, hi = S, tprev = 0;
  bool inwin_prev = false;

  for (int s = 0; s < T; ++s) {
    const int t = back ? T - 1 - s : s;
    if (lat.banded) {
      if (s > 0) { if (back) dg.down(); else dg.up(); }
      const int64_t l = max((int64_t)0, dg.q - half);
      lo = (int)l;
      hi = (int)min(l + W, (int64_t)S);
    }
    pplo = plo;
    plo = lo >> 1;
    const int row = t - cf0;
    const int pt = __float_as_int(cp[row]);
    // the previous frame's value at its path state: the offset of this frame (0 where it is -inf or the path
    // left the window); thread 0 turns it into that frame's output
    float c = 0.0f;
    if (s > 0) {
      const float cr = inwin_prev ? s_pv[(s - 1) & 1] : ninf;
      const bool fin = kab_finite(cr);
      c = fin ? cr : 0.0f;
      if (tid == 0) {
        out[tprev] = fin ? ((double)cr + off) * LN2 : (double)ninf;
        off += (double)c;
      }
    }
    const float eb = (staged ? ce[row * p.V + p.blank] : __ldg(lp_rows + (int64_t)t * p.V + p.blank)) * LOG2E;
    const int d = 2 * (plo - pplo);  // slot of state u in prev: u - 2 pplo + PAD
    float *pv = &s_pv[s & 1];
    for (int q = tid; q < np; q += NT) {
      const int k = plo + q;
      const int vb = 2 * k;
      if (!back) {  // pair (blank 2k, label 2k+1), label index k
        const int32_t lw = k < L ? __ldg(labs + k) : 0;
        const int lab = lw & 0xffff;
        const float el = (staged ? ce[row * p.V + lab] : __ldg(lp_rows + (int64_t)t * p.V + lab)) * LOG2E;
        float xb, xl;
        if (s == 0) {
          xb = vb == 0 ? 0.0f : ninf;
          xl = vb == 0 ? 0.0f : ninf;
        } else {
          const int j = 2 * q + d + KAB_POST_PAD;
          const float x1 = prev[j - 1], x0 = prev[j], xn = prev[j + 1];
          xb = kab_lse2(x0, x1);
          xl = kab_lse2(xn, lw < 0 ? xb : x0);
        }
        const float nb = (vb >= lo && vb < hi) ? xb - c + eb : ninf;
        const float nl = (vb + 1 >= lo && vb + 1 < hi) ? xl - c + el : ninf;
        cur[2 * q + KAB_POST_PAD] = nb;
        cur[2 * q + KAB_POST_PAD + 1] = nl;
        if (vb == pt) *pv = nb;
        if (vb + 1 == pt) *pv = nl;
      } else {  // pair (label 2k-1, blank 2k), label index k-1; the buffers hold y = beta + emission
        const int32_t lw = (k >= 1 && k <= L) ? __ldg(labs + k - 1) : 0;
        const int lab = lw & 0xffff;
        const float el = (staged ? ce[row * p.V + lab] : __ldg(lp_rows + (int64_t)t * p.V + lab)) * LOG2E;
        float bb, bl;
        if (s == 0) {
          bb = (vb == S - 1 || vb == S - 2) ? 0.0f : ninf;
          bl = (vb - 1 == S - 1 || vb - 1 == S - 2) ? 0.0f : ninf;
        } else {
          const int j = 2 * q + d + KAB_POST_PAD;  // (d <= 0 here: the window only moves down)
          const float yl = prev[j - 1], yb = prev[j], yn = prev[j + 1];
          bb = kab_lse2(yb, yn);
          bl = kab_lse2(yl, (lw >> 30) & 1 ? bb : yb);
        }
        bb = (vb >= lo && vb < hi) ? bb - c : ninf;
        bl = (k >= 1 && vb - 1 >= lo && vb - 1 < hi) ? bl - c : ninf;
        cur[2 * q + KAB_POST_PAD] = bb + eb;
        cur[2 * q + KAB_POST_PAD - 1] = bl + el;
        if (vb == pt) *pv = bb;
        if (vb - 1 == pt) *pv = bl;
      }
    }
    inwin_prev = pt >= lo && pt < hi;
    tprev = t;
    const bool chunk_end = (s + 1) % F == 0 && s + 1 < T;
    if (chunk_end && tid == 0) {
      const int cn = (s + 1) / F;
      kab_mbar_wait(&bars[cn % KAB_POST_NST], (uint32_t)(cn / KAB_POST_NST) & 1u);
    }
    __syncthreads();
    if (chunk_end) {  // chunk s / F is consumed: its stage takes chunk s / F + NST
      const int cd = s / F;
      if (cd + KAB_POST_NST < n_chunks) issue(cd + KAB_POST_NST);
      open(cd + 1);
    }
    float *tmp = prev; prev = cur; cur = tmp;
  }
  if (tid == 0) {
    const float cr = inwin_prev ? s_pv[(T - 1) & 1] : ninf;
    out[tprev] = kab_finite(cr) ? ((double)cr + off) * LN2 : (double)ninf;
    if (!back) {  // log Z: the end states S-1, S-2 inside the last window (prev holds frame T-1)
      const float a1 = (S - 1 >= lo && S - 1 < hi) ? prev[S - 1 - 2 * plo + KAB_POST_PAD] : ninf;
      const float a2 = (S - 2 >= 0 && S - 2 >= lo && S - 2 < hi) ? prev[S - 2 - 2 * plo + KAB_POST_PAD] : ninf;
      const float z = kab_lse2(a1, a2);
      p.log_likelihood[lat.index] = z == ninf ? (double)ninf : ((double)z + off) * LN2;
    }
  }
}

// gamma_t = exp(fwd_t + bwd_t - log Z) in double, rounded to float32 and clamped to [0, 1]; 0 for a lattice whose
// status is not 0 or whose log Z is -inf, and for rows before the first lattice
__global__ void kab_ctc_posterior_combine_kernel(const int64_t *__restrict__ t_off, int64_t B, int64_t total_T,
                                                 const int32_t *__restrict__ status, const double *__restrict__ fwd,
                                                 const double *__restrict__ bwd, const double *__restrict__ ll,
                                                 float *__restrict__ post) {
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < total_T; i += (int64_t)gridDim.x * blockDim.x) {
    float g = 0.0f;
    if (i >= t_off[0]) {
      int64_t a = 0, b = B;  // the lattice b with t_off[b] <= i < t_off[b + 1]
      while (b - a > 1) {
        const int64_t m = (a + b) >> 1;
        if (__ldg(t_off + m) <= i) a = m; else b = m;
      }
      const double z = ll[a];
      if (status[a] == 0 && z > -INFINITY) {
        const double x = exp(fwd[i] + bwd[i] - z);
        g = (float)fmin(fmax(x, 0.0), 1.0);
      }
    }
    post[i] = g;
  }
}
