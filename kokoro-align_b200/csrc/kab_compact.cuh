// kab_compact.cuh -- wide vocabularies (V > 512, BASELINE config 5's V = 4096) for the staged
// kernels.  A lattice only ever reads the columns of its own labels and the blank
// (align.py:77: log_probs[i, ext[v]]), so when no lattice of the plan uses more than 511 distinct
// labels the plan works on a COMPACT copy of the log-probs: row t of lattice b keeps
// log_probs[t, gather[b][j]], j < Vc, with gather[b][0] = 0 (blank) and gather[b][1..] the
// lattice's distinct label columns in ascending order.  The staged kernels then run unchanged
// with V = Vc and labels renumbered to compact indices; best_labels is mapped back afterwards
// (a label value IS its column), best_scores are the same floats.  The non-finite contract is the
// same as everywhere else (status 3 for a non-finite value ANYWHERE in the lattice's [T, V] rows,
// as every other kernel has it): the gather kernel streams the whole rows once
// (coalesced; 4 V bytes per frame, a fraction of what the recurrence moves) and flags the lattice,
// and the label expansion that runs after the staged kernels turns the flag into the status.
// CTC forced-alignment plans (kab_plan_create_ctc, V > 512) use the same copy with gather[b][0] = the
// plan's blank id; their staged kernels then take blank column 0, and a lattice with more than 511
// distinct labels goes to the generic kernel on its own (not the whole plan).  The whole-row check is the CTC one
// there (kab_poison_t<true>): NaN and +inf flag the lattice, -inf (masking) does not -- what
// kab_generic_ctc_kernel checks over the same rows.
#pragma once
#include "kab_common.cuh"

#define KAB_COMPACT_FRAMES 64  // frames per CTA of the two helper kernels

// grid (lattices of one work list, frame chunks); block 256 = 8 warps, a warp per frame
template <bool CTC>
__device__ __forceinline__ void kab_compact_body(const KabLattice *__restrict__ lats, const float *__restrict__ lp,
                                                 float *__restrict__ lpc, const int32_t *__restrict__ gather, int V,
                                                 int Vc, int32_t *__restrict__ nonfinite) {
  const KabLattice lat = lats[blockIdx.x];
  const int f0 = blockIdx.y * KAB_COMPACT_FRAMES;
  if (f0 >= lat.T) return;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int32_t *g = gather + (size_t)lat.index * Vc;
  const int f1 = min(lat.T, f0 + KAB_COMPACT_FRAMES);
  float poison = kab_poison_init<CTC>();
  for (int f = f0 + warp; f < f1; f += 8) {
    const float *src = lp + (size_t)(lat.t_off + f) * V;
    float *dst = lpc + (size_t)(lat.t_off + f) * Vc;
    for (int j = lane; j < V; j += 32) poison = kab_poison_t<CTC>(poison, __ldg(src + j));  // the whole row, once
    for (int j = lane; j < Vc; j += 32) dst[j] = __ldg(src + g[j]);                         // (now L1 / L2 hits)
  }
  if (__any_sync(KAB_FULL_MASK, poison != poison) && lane == 0) nonfinite[lat.index] = 1;
}

__global__ void kab_compact_kernel(const KabLattice *__restrict__ lats, const float *__restrict__ lp,
                                   float *__restrict__ lpc, const int32_t *__restrict__ gather, int V, int Vc,
                                   int32_t *__restrict__ nonfinite) {
  kab_compact_body<false>(lats, lp, lpc, gather, V, Vc, nonfinite);
}

// CTC forced alignment: gather[b][0] is the blank's column; NaN / +inf anywhere in the rows flag the lattice
__global__ void kab_compact_ctc_kernel(const KabLattice *__restrict__ lats, const float *__restrict__ lp,
                                       float *__restrict__ lpc, const int32_t *__restrict__ gather, int V, int Vc,
                                       int32_t *__restrict__ nonfinite) {
  kab_compact_body<true>(lats, lp, lpc, gather, V, Vc, nonfinite);
}

// best_labels: compact index -> label value, for the lattices that were aligned (status 0)
__global__ void kab_expand_labels_kernel(const KabLattice *__restrict__ lats, int32_t *__restrict__ best_labels,
                                         int32_t *status, float *final_score, const int32_t *__restrict__ gather,
                                         int Vc, const int32_t *__restrict__ nonfinite) {
  const KabLattice lat = lats[blockIdx.x];
  const int f0 = blockIdx.y * KAB_COMPACT_FRAMES;
  if (nonfinite[lat.index]) {  // KAB_ST_NONFINITE wins over whatever the staged kernel reported
    if (blockIdx.y == 0 && threadIdx.x == 0) {
      status[lat.index] = 3;
      if (final_score) final_score[lat.index] = __int_as_float(0x7fc00000);
    }
    return;
  }
  if (f0 >= lat.T || status[lat.index] != 0) return;
  const int32_t *g = gather + (size_t)lat.index * Vc;
  const int f1 = min(lat.T, f0 + KAB_COMPACT_FRAMES);
  for (int f = f0 + threadIdx.x; f < f1; f += blockDim.x) {
    int32_t *p = best_labels + lat.t_off + f;
    const int32_t c = *p;
    if ((unsigned)c < (unsigned)Vc) *p = g[c];
  }
}
