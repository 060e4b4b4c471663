// kab_spans.cuh -- token spans and word spans of a per-frame token sequence on the device
// (torchaudio.functional.merge_tokens semantics, and the word grouping of torchaudio's forced-
// alignment tutorial), for a flat batch of items.  DESIGN.md 3.10.
//
// Spans.  A run is a maximal stretch of equal tokens; frame 0 always starts one.  Every run whose
// token is not the blank is a span (token, start, end), end exclusive, in item-relative frames.
// Its score is the mean of scores[start:end] with one fixed order of operations, so that a CPU
// restatement reproduces it bit for bit: the values are converted to double and added in frame
// order starting from the first (__dadd_rn: no contraction), the sum is divided by end - start in
// double (__ddiv_rn) and rounded once to float32.  -inf and NaN propagate.
//
// Words.  Word w of an item covers word_len[w] consecutive spans from span first_token: start =
// the first span's start, end = the last span's end, score =
// fl32(sum_j double(score_j) * len_j / sum_j len_j), the numerator summed from +0.0 in span order
// (__dmul_rn then __dadd_rn), one __ddiv_rn -- Python's `sum(s.score * len(s) for s in spans) /
// sum(len(s) for s in spans)` evaluated on these spans, rounded once.
//
// Layout: one CTA per item (grid-stride over the batch).  The merge kernel walks the item in
// chunks of KAB_SPAN_THREADS * KAB_SPAN_FRAMES frames; each thread flags the span starts among
// its KAB_SPAN_FRAMES consecutive frames, a block scan of the flag counts gives every start its
// span index, and the thread that owns a start walks forward to the end of the run, summing as it
// goes (one dependent double add per frame).  The word kernel first reduces the item's word
// lengths (status), then scans them in chunks of KAB_WORD_THREADS words for each word's first
// span, and one thread per word sums its spans.
#pragma once
#include "kab_common.cuh"

#define KAB_SPAN_THREADS 256
#define KAB_SPAN_FRAMES 4   // consecutive frames per thread and chunk
#define KAB_WORD_THREADS 128

// mirror kab_token_span / kab_word_span (include/kokoro_align_b200.h), 16 bytes each
struct KabTokenSpan {
  int32_t token, start, end;
  float score;
};
struct KabWordSpan {
  int32_t start, end, first_token;
  float score;
};

// Exclusive block scan of one int per thread; *total receives the block's sum.  warp_tot: shared
// [NT / 32].  Ends with a barrier, so warp_tot can be reused by the next call.
template <int NT>
__device__ __forceinline__ int kab_block_excl_scan(int v, int *warp_tot, int *total) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int x = v;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const int y = __shfl_up_sync(KAB_FULL_MASK, x, d);
    if (lane >= d) x += y;
  }
  if (lane == 31) warp_tot[warp] = x;
  __syncthreads();
  if (warp == 0) {
    int w = lane < NT / 32 ? warp_tot[lane] : 0;
#pragma unroll
    for (int d = 1; d < NT / 32; d <<= 1) {
      const int y = __shfl_up_sync(KAB_FULL_MASK, w, d);
      if (lane >= d) w += y;
    }
    if (lane < NT / 32) warp_tot[lane] = w;  // inclusive
  }
  __syncthreads();
  const int base = warp ? warp_tot[warp - 1] : 0;
  *total = warp_tot[NT / 32 - 1];
  __syncthreads();
  return base + x - v;
}

__device__ __forceinline__ void kab_store16(void *dst, int32_t a, int32_t b, int32_t c, float d, bool vec) {
  if (vec) {
    *reinterpret_cast<int4 *>(dst) = make_int4(a, b, c, __float_as_int(d));
  } else {
    int32_t *p = reinterpret_cast<int32_t *>(dst);
    p[0] = a; p[1] = b; p[2] = c; p[3] = __float_as_int(d);
  }
}

__device__ __forceinline__ int4 kab_load16(const void *src, bool vec) {
  if (vec) return __ldg(reinterpret_cast<const int4 *>(src));
  const int32_t *p = reinterpret_cast<const int32_t *>(src);
  return make_int4(__ldg(p), __ldg(p + 1), __ldg(p + 2), __ldg(p + 3));
}

// grid-stride over items; vec: d_spans is 16-byte aligned (one vector store per span)
__global__ void __launch_bounds__(KAB_SPAN_THREADS) kab_merge_tokens_kernel(
    int64_t n_items, const int64_t *__restrict__ t_off, const int32_t *__restrict__ tokens,
    const float *__restrict__ scores, int32_t blank, KabTokenSpan *__restrict__ spans,
    int32_t *__restrict__ n_spans, int vec) {
  __shared__ int warp_tot[KAB_SPAN_THREADS / 32];
  constexpr int CHUNK = KAB_SPAN_THREADS * KAB_SPAN_FRAMES;
  for (int64_t b = blockIdx.x; b < n_items; b += gridDim.x) {
    const int64_t off = t_off[b];
    const int T = (int)(t_off[b + 1] - off);
    const int32_t *tok = tokens + off;
    const float *sc = scores + off;
    KabTokenSpan *out = spans + off;
    int base = 0;  // spans before this chunk
    for (int c0 = 0; c0 < T; c0 += CHUNK) {
      const int f0 = c0 + (int)threadIdx.x * KAB_SPAN_FRAMES;
      int prev = f0 > 0 && f0 < T ? __ldg(tok + f0 - 1) : 0;
      int tk[KAB_SPAN_FRAMES];
      unsigned starts = 0;
#pragma unroll
      for (int j = 0; j < KAB_SPAN_FRAMES; ++j) {
        const int t = f0 + j;
        tk[j] = t < T ? __ldg(tok + t) : blank;
        if (t < T && tk[j] != blank && (t == 0 || tk[j] != prev)) starts |= 1u << j;
        prev = tk[j];
      }
      int total;
      int k = base + kab_block_excl_scan<KAB_SPAN_THREADS>(__popc(starts), warp_tot, &total);
#pragma unroll
      for (int j = 0; j < KAB_SPAN_FRAMES; ++j) {
        if (!(starts >> j & 1)) continue;
        const int s = f0 + j, c = tk[j];
        double acc = (double)__ldg(sc + s);
        int e = s + 1;
        for (; e < T && __ldg(tok + e) == c; ++e) acc = __dadd_rn(acc, (double)__ldg(sc + e));
        const float mean = __double2float_rn(__ddiv_rn(acc, (double)(e - s)));
        kab_store16(out + k, c, s, e, mean, vec);
        ++k;
      }
      base += total;
    }
    if (threadIdx.x == 0) n_spans[b] = base;
  }
}

// Block sum of one int64 per thread (every thread gets it).  red: shared [NT / 32].
template <int NT>
__device__ __forceinline__ long long kab_block_sum(long long v, long long *red) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) v += __shfl_xor_sync(KAB_FULL_MASK, v, d);
  if (lane == 0) red[warp] = v;
  __syncthreads();
  long long s = 0;
#pragma unroll
  for (int w = 0; w < NT / 32; ++w) s += red[w];
  __syncthreads();
  return s;
}

// grid-stride over items; vec bit 0: d_spans, bit 1: d_words is 16-byte aligned
__global__ void __launch_bounds__(KAB_WORD_THREADS) kab_word_spans_kernel(
    int64_t n_items, const int64_t *__restrict__ t_off, const KabTokenSpan *__restrict__ spans,
    const int32_t *__restrict__ n_spans, const int64_t *__restrict__ word_off,
    const int32_t *__restrict__ word_len, KabWordSpan *__restrict__ words,
    int32_t *__restrict__ word_status, int vec) {
  __shared__ int warp_tot[KAB_WORD_THREADS / 32];
  __shared__ long long red[KAB_WORD_THREADS / 32];
  for (int64_t b = blockIdx.x; b < n_items; b += gridDim.x) {
    const int64_t w0 = word_off[b], nw = word_off[b + 1] - w0;
    const int ns = n_spans[b];
    // the lengths must be >= 1 and sum to the item's span count; otherwise status 1, no words
    long long sum = 0;
    int bad = 0;
    for (int64_t i = threadIdx.x; i < nw; i += KAB_WORD_THREADS) {
      const int l = __ldg(word_len + w0 + i);
      sum += l;
      bad |= l < 1;
    }
    bad = __syncthreads_or(bad);
    sum = kab_block_sum<KAB_WORD_THREADS>(sum, red);
    bad = bad || nw < 0 || sum != (long long)ns;
    if (threadIdx.x == 0) word_status[b] = bad;
    if (bad) continue;
    const KabTokenSpan *sp = spans + t_off[b];
    int base = 0;  // spans of the words before this chunk
    for (int64_t c0 = 0; c0 < nw; c0 += KAB_WORD_THREADS) {
      const int64_t i = c0 + threadIdx.x;
      const int l = i < nw ? __ldg(word_len + w0 + i) : 0;
      int total;
      const int k = base + kab_block_excl_scan<KAB_WORD_THREADS>(l, warp_tot, &total);
      if (i < nw) {
        double num = 0.0;
        long long den = 0;
        int start = 0, end = 0;
        for (int j = 0; j < l; ++j) {
          const int4 r = kab_load16(sp + k + j, vec & 1);
          const int len = r.z - r.y;
          num = __dadd_rn(num, __dmul_rn((double)__int_as_float(r.w), (double)len));
          den += len;
          if (j == 0) start = r.y;
          end = r.z;
        }
        kab_store16(words + w0 + i, start, end, k, __double2float_rn(__ddiv_rn(num, (double)den)), vec & 2);
      }
      base += total;
    }
  }
}
