// kab_generic.cuh -- the catch-all kernel: any beam_size, any max_move (1..16), any label values
// (label 0 inside the transcript, negative numpy-style labels), S > 3T, vocabularies too wide
// for the staged kernels.  One CTA per lattice, score rows in global memory (L2-resident),
// one byte of backpointer per evaluated cell.  Correctness first: this is the path the
// reference's non-default keyword arguments (align.py:43) take; the default configuration is
// served by kab_warp.cuh / kab_band.cuh.
#pragma once
#include "kab_common.cuh"

// CTC: the CTC forced-alignment recurrence (kab_common.cuh) in the same window (value-independent blank
// test: the state's parity), blank column `blank`.  Default and long-form plans pass a W so wide that the
// window is [0, S) in every frame; banded plans (kab_plan_create_ctc_band) pass beam_size.  A window that
// clips somewhere and leaves both end states -inf: no path inside the band, status 1.
// FREE: CTC with free ends (kab_plan_create_ctc_free; always unbanded): a virtual state -1 of score 0 in
// every frame is state 0's move-1 and state 1's move-2 predecessor, thread 0 keeps running (score, frame)
// maxima of the end states (>=: the later frame), and the walk starts at the chosen end (t1, v) and stops
// at state -1; frames outside [t0, t1] get state -1 and the blank.
template <int NT, bool CTC, bool FREE = false>
__device__ __forceinline__ void kab_generic_body(const KabLattice *__restrict__ lats, int n_lat, const KabParams &p,
                                                 const int blank) {
  __shared__ unsigned int s_item;
  __shared__ long long s_vmax;
  const int tid = threadIdx.x;

  for (;;) {
    if (tid == 0) {
      s_item = atomicAdd(p.queue, 1u);
      s_vmax = -1;
    }
    __syncthreads();
    const unsigned int item = s_item;
    if (item >= (unsigned int)n_lat) break;
    const KabLattice lat = lats[item];
    const int64_t T = lat.T, S = 2 * (int64_t)lat.L + 1, W = p.W, M = p.M, V = p.V;
    const int64_t Wc = max((int64_t)1, min(W, S));
    const int32_t *raw = p.raw + lat.lab_off;
    const float *lp = p.lp + lat.t_off * V;
    uint8_t *bp = p.bp + lat.bp_off;
    float *prev = p.scratch + lat.scr_off;
    float *cur = prev + (S + 16);

    if (tid == 0 && !FREE) __stcg(&prev[0], 0.0f);  // virtual start, align.py:57-58
    __syncthreads();

    int64_t plo = 0, phi = FREE ? 0 : 1;
    float m1 = kab_neg_inf(), m2 = kab_neg_inf();  // FREE (thread 0): end maxima of S-1, S-2 and their frames
    int64_t f1 = T - 1, f2 = T - 1;
    bool bad = false;
    for (int64_t i = 0; i < T; ++i) {
      int64_t lo = (S * i) / T - W / 2;  // align.py:64 (64-bit: S*i reaches 1e11)
      if (lo < 0) lo = 0;
      int64_t hi = min(lo + W, S);  // align.py:65
      if (hi < lo) hi = lo;
      const float *row = lp + i * V;
      for (int64_t c = tid; c < V; c += NT) {
        const float x = __ldg(&row[c]);
        bad |= CTC ? !(x < __int_as_float(0x7f800000)) : !kab_finite(x);  // CTC: -inf is accepted
      }
      if (CTC) {
        for (int64_t v = lo + tid; v < hi; v += NT) {
          const bool lab = (v & 1) != 0;
          const int32_t ext = lab ? raw[(v - 1) >> 1] : blank;
          const float e = __ldg(&row[ext]);
          // predecessors outside the previous window are -inf
          const float x0 = v >= plo && v < phi ? __ldcg(&prev[v]) : kab_neg_inf();
          float x1 = v - 1 >= plo && v - 1 < phi ? __ldcg(&prev[v - 1]) : kab_neg_inf();
          float x2 = lab && v >= 3 && v - 2 >= plo && v - 2 < phi && ext != raw[(v - 3) >> 1] ? __ldcg(&prev[v - 2]) : kab_neg_inf();
          if constexpr (FREE) if (v == 0) x1 = 0.0f;  // the virtual state -1
          if constexpr (FREE) if (v == 1) x2 = 0.0f;
          uint32_t code = 0;
          const float best = lab ? kab_ctc_label_sel(x0, x1, x2, code, 0) : kab_ctc_blank_sel(x0, x1, code, 0);
          __stcg(&cur[v], __fadd_rn(best, e));
          bp[i * Wc + (v - lo)] = (uint8_t)code;
        }
      } else
      for (int64_t v = lo + tid; v < hi; v += NT) {
        const int32_t ext = (v & 1) ? raw[(v - 1) >> 1] : 0;
        const int32_t col = ext < 0 ? ext + (int32_t)V : ext;
        const float e = __ldg(&row[col]);
        float best = kab_neg_inf();
        int bj = 0;
        for (int64_t j = 0; j < M; ++j) {
          const int64_t u = v - j;
          if (u < plo || u >= phi) continue;                 // not a state of the previous window
          if (j > 0 && (j & 1) == 0 && ext == 0) continue;   // align.py:80-81 (value test)
          const float val = __fadd_rn(__ldcg(&prev[u]), e);  // align.py:77
          if (val > best) { best = val; bj = (int)j; }       // first max wins, align.py:83
        }
        __stcg(&cur[v], best);
        bp[i * Wc + (v - lo)] = (uint8_t)bj;
      }
      __syncthreads();
      float *t = prev; prev = cur; cur = t;
      plo = lo; phi = hi;
      if constexpr (FREE) if (tid == 0 && S >= 3) {
        const float a1 = __ldcg(&prev[S - 1]), a2 = __ldcg(&prev[S - 2]);
        if (a1 >= m1) { m1 = a1; f1 = i; }
        if (a2 >= m2) { m2 = a2; f2 = i; }
      }
    }

    // forced end state: highest active state of the last frame, align.py:99-101
    long long vmax = -1;
    if (!CTC)
      for (int64_t v = plo + tid; v < phi; v += NT)
        if (__ldcg(&prev[v]) > kab_neg_inf()) vmax = v;
    if (vmax >= 0) atomicMax(&s_vmax, vmax);
    const int any_bad = __syncthreads_or(bad ? 1 : 0);
    int64_t v = s_vmax;
    // CTC end rule: the better of the last two states, S-2 on a tie (a state outside the last window: -inf);
    // none of them finite in a window that clips: no path inside the band
    int64_t t1 = T - 1;
    float fs_free = 0.0f;
    if constexpr (FREE) {  // free end (thread 0's maxima): the larger one, on a tie the later frame, then S-2
      const bool top = m1 > m2 || (m1 == m2 && f1 > f2);
      v = top ? S - 1 : S - 2;
      t1 = top ? f1 : f2;
      fs_free = top ? m1 : m2;
      if (S == 1) { v = -1; t1 = -1; fs_free = 0.0f; }  // L = 0: no frame is inside
    } else if (CTC) {
      const float e1 = S - 1 >= plo && S - 1 < phi ? __ldcg(&prev[S - 1]) : kab_neg_inf();
      const float e2 = S >= 2 && S - 2 >= plo && S - 2 < phi ? __ldcg(&prev[S - 2]) : kab_neg_inf();
      v = (S >= 2 && !(e1 > e2)) ? S - 2 : S - 1;
      const bool clips = W < S || (S * (T - 1)) / T > W / 2;
      if (clips && !(e1 > kab_neg_inf()) && !(e2 > kab_neg_inf())) v = -1;
    }

    if (tid == 0) {
      int st = 0;
      if (any_bad) st = 3;
      else if (v < 0 && !FREE) st = 1;
      p.status[lat.index] = st;
      if (p.final_score) p.final_score[lat.index] = st == 0 ? (FREE ? fs_free : __ldcg(&prev[v])) : __int_as_float(0x7fc00000);
      if (st == 0) {
        int32_t *out_path = p.best_path + lat.t_off;
        int32_t *out_lab = p.best_labels + lat.t_off;
        float *out_sc = p.best_scores + lat.t_off;
        const int64_t vend = v;
        if constexpr (FREE) v = -1;
        for (int64_t i = T - 1; i >= 0; --i) {  // == flush_determined_path, align.py:21-40
          int64_t lo = (S * i) / T - W / 2;
          if (lo < 0) lo = 0;
          if constexpr (FREE) if (i == t1) v = vend;
          if constexpr (FREE) if (v < 0) {  // outside [t0, t1]
            out_path[i] = -1;
            out_lab[i] = blank;
            out_sc[i] = __ldg(&lp[i * V + blank]);
            continue;
          }
          const int32_t ext = (v & 1) ? raw[(v - 1) >> 1] : (CTC ? blank : 0);
          const int32_t col = ext < 0 ? ext + (int32_t)V : ext;
          out_path[i] = (int32_t)v;
          out_lab[i] = ext;                      // align.py:106
          out_sc[i] = __ldg(&lp[i * V + col]);   // align.py:107
          v -= bp[i * Wc + (v - lo)];
        }
      }
    }
    __syncthreads();
  }
}

template <int NT>
__global__ void __launch_bounds__(NT) kab_generic_kernel(const KabLattice *__restrict__ lats, int n_lat,
                                                         KabParams p) {
  kab_generic_body<NT, false>(lats, n_lat, p, 0);
}

template <int NT>
__global__ void __launch_bounds__(NT) kab_generic_ctc_kernel(const KabLattice *__restrict__ lats, int n_lat,
                                                             KabParams p, int blank) {
  kab_generic_body<NT, true>(lats, n_lat, p, blank);
}

// CTC forced alignment with free ends (kab_plan_create_ctc_free)
template <int NT>
__global__ void __launch_bounds__(NT) kab_generic_ctc_free_kernel(const KabLattice *__restrict__ lats, int n_lat,
                                                                  KabParams p, int blank) {
  kab_generic_body<NT, true, true>(lats, n_lat, p, blank);
}
