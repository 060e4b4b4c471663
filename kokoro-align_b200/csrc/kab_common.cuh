// kab_common.cuh -- shared device helpers for the CTC best-path kernels (sm_100a).
//
// The recurrence implemented by every kernel is the reference's
// kokoro_align/align.py:43-109 (see SURVEY.md section 8a for the per-cell restatement):
//   cand_j = fl32(score_{i-1}[v-j] + lp[i, ext[v]]),  j = 0..M-1, strict '>' scan in j order,
//   even j > 0 forbidden into states with ext[v] == 0, window [lo_i, hi_i) per frame,
//   virtual start state 0 with score 0, forced end at the highest active state.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#define KAB_FULL_MASK 0xffffffffu

// Per-lattice work descriptor (device array, one list per kernel class, sorted by cost).
struct KabLattice {
  int64_t t_off;    // first row of this lattice in log_probs / the output arrays
  int64_t col_off;  // first entry in the padded uint16 column table (fast kernels)
  int64_t lab_off;  // first entry in the raw int32 label table (generic kernel)
  int64_t bp_off;   // byte offset of this lattice's backpointers in the workspace
  int64_t scr_off;  // float offset of the generic kernel's two score rows
  int32_t T;        // frames
  int32_t L;        // labels; S = 2L+1 extended states
  int32_t index;    // position in the caller's batch (final_score / status slot)
  int32_t k;        // class parameter: states per lane (warp kernel)
};

struct KabParams {
  const float *lp;          // [sum T, V]
  int64_t lp_bytes;         // total bytes of lp (bulk copies never read past it)
  const uint16_t *col16;    // numpy-style column index of every label, padded per lattice
  const int32_t *raw;       // raw label values (generic kernel: value-based blank test)
  uint8_t *bp;              // backpointer workspace
  float *scratch;           // generic kernel score rows
  unsigned char *fifo;      // cluster band kernel: per-lattice progress counters and neighbour FIFOs
  int32_t *best_path;       // [sum T]
  int32_t *best_labels;     // [sum T]
  float *best_scores;       // [sum T]
  float *final_score;       // [B] or nullptr
  int32_t *status;          // [B]
  unsigned int *queue;      // this kernel class's work-queue counter
  int32_t V, W, M;
  int32_t stage_frames;     // emission frames per bulk-copy stage
  int32_t stage_bytes;      // bytes of one stage buffer (multiple of 16)
  int32_t band_nw;          // warps per CTA of the band kernel
  int32_t *end_state;       // cluster band kernel: not nullptr = write the forced end state of every lattice
                            // here ([B]) and leave the traceback to kab_btpar.cuh
  long long *debug;         // development only (KAB_BAND_TIMING builds)
  uint32_t one;             // the value 1, opaque to the compiler (kab_blank_sel / kab_label_sel)
  float mm1, mm2, mm3;      // max_move < 4 (the MM instantiations of the staged kernels): 0 or -inf, added to the
                            // candidates of moves 1 / 2 / 3 -- a candidate that max_move excludes (align.py:70)
                            // becomes -inf, which is what "no candidate" is everywhere else
  unsigned int *started;    // kab_bandr_kernel: not nullptr = every CTA counts itself here when it starts (hybrid
                            // band plans: the single-CTA kernel is launched behind kab_gate_kernel, which waits
                            // until the clusters hold their SMs)
};

// Waits until *counter has reached target (a count that only grows): see KabParams::started.
__global__ void kab_gate_kernel(const unsigned int *counter, unsigned int target) {
  if (threadIdx.x == 0) {
    unsigned int v;
    for (;;) {
      asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(counter) : "memory");
      if ((int)(v - target) >= 0) break;
      __nanosleep(500);
    }
  }
}

// max_move < 4 in the kernels written for four moves: x + 0.0f == x for every candidate (finite or
// -inf, never -0), x + -inf == -inf.  MM == false (max_move 4): nothing is emitted.
template <bool MM>
__device__ __forceinline__ float kab_mm(const float cand, const float mask) {
  return MM ? __fadd_rn(cand, mask) : cand;
}

__device__ __forceinline__ float kab_neg_inf() { return __int_as_float(0xff800000); }
__device__ __forceinline__ bool kab_finite(float x) { return fabsf(x) < __int_as_float(0x7f800000); }
// Finiteness accumulator on the FMA pipe (the ALU pipe is the busy one): x * 0 is 0 for a finite x
// and NaN for +-inf / NaN, so `acc` turns NaN, and stays NaN, once a non-finite value was seen.
__device__ __forceinline__ float kab_poison(float acc, float x) { return fmaf(x, 0.0f, acc); }

// ---------------------------------------------------------------- CTC forced alignment (the CTC
// instantiations; torchaudio.functional.forced_align's recurrence, DESIGN.md 3.9)
//   x0 = a[v], x1 = a[v-1], x2 = a[v-2] (label states only, -inf into a repeated label and for v == 1);
//   j = 2 if x2 > x1 and x2 > x0, else 1 if x1 > x0 and x1 > x2, else 0 -- so x1 == x2 > x0 keeps x0;
//   a'[v] = fl32(x_j + lp[t, ext[v]]): the select is on the previous scores, then ONE add.
// The 2-bit backpointer code is the move, as in the Kokoro kernels, so their walks apply unchanged.
// -inf log-probs are accepted (masking); only NaN and +inf are rejected.  Accumulator that starts at
// -inf: acc + x stays -inf for a finite or -inf x and turns NaN, for good, at the first NaN or +inf.
__device__ __forceinline__ float kab_poison_ctc(float acc, float x) { return __fadd_rn(acc, x); }
template <bool CTC>
__device__ __forceinline__ float kab_poison_t(float acc, float x) {
  return CTC ? kab_poison_ctc(acc, x) : kab_poison(acc, x);
}
template <bool CTC>
__device__ __forceinline__ float kab_poison_init() { return CTC ? kab_neg_inf() : 0.0f; }
// Blank state: moves 0, 1.  The code's bits are OR-ed into w at bit pos.
__device__ __forceinline__ float kab_ctc_blank_sel(float x0, float x1, uint32_t &w, const int pos) {
  const bool p1 = x1 > x0;
  w |= (uint32_t)p1 << pos;
  return p1 ? x1 : x0;
}
// Label state: moves 0, 1, 2 (x2 already -inf where move 2 is forbidden).
__device__ __forceinline__ float kab_ctc_label_sel(float x0, float x1, float x2, uint32_t &w, const int pos) {
  const bool p2 = x2 > x1 && x2 > x0;
  const bool p1 = x1 > x0 && x1 > x2;  // (excludes p2)
  w |= ((uint32_t)p2 << 1 | (uint32_t)p1) << pos;
  return p2 ? x2 : (p1 ? x1 : x0);
}

// ---------------------------------------------------------------- inline-PTX memory and synchronisation wrappers
// (mbarriers, 1-D bulk copies, fences, clusters / distributed shared memory, relaxed accesses)
__device__ __forceinline__ uint32_t kab_smem_u32(const void *p) {
  return (uint32_t)__cvta_generic_to_shared(p);
}

// ---- mbarriers
__device__ __forceinline__ void kab_mbar_init(uint64_t *bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(kab_smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void kab_fence_mbar_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void kab_mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(kab_smem_u32(bar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void kab_mbar_arrive(uint64_t *bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(kab_smem_u32(bar)) : "memory");
}
// Two ways to wait for a phase: try_wait may suspend the warp (kab_mbar_wait), test_wait never does
// (kab_mbar_spin: try_wait may suspend the warp for ~800 cycles (measured) when it races with the
// arming arrive).
__device__ __forceinline__ bool kab_mbar_try_wait(uint64_t *bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(kab_smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void kab_mbar_wait(uint64_t *bar, uint32_t parity) {
  while (!kab_mbar_try_wait(bar, parity)) {
  }
}
__device__ __forceinline__ bool kab_mbar_test_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void kab_mbar_spin(uint64_t *bar, uint32_t parity) {
  const uint32_t a = kab_smem_u32(bar);
  while (!kab_mbar_test_wait(a, parity)) {
  }
}

// ---- 1-D bulk copies (TMA)
// global -> shared bulk copy; completion is signalled on `bar` (complete_tx::bytes).
__device__ __forceinline__ void kab_bulk_g2s(void *dst, const void *src, uint32_t bytes, uint64_t *bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   kab_smem_u32(dst)),
               "l"(src), "r"(bytes), "r"(kab_smem_u32(bar))
               : "memory");
}
// Same, with an L2 eviction-priority hint (createpolicy); the warp kernel passes evict_normal.
__device__ __forceinline__ void kab_bulk_g2s_hint(void *dst, const void *src, uint32_t bytes, uint64_t *bar,
                                                  uint64_t policy) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::"r"(
          kab_smem_u32(dst)),
      "l"(src), "r"(bytes), "r"(kab_smem_u32(bar)), "l"(policy)
      : "memory");
}
// Bulk prefetch of a global range into L2 (no destination): address 16-byte aligned, size a multiple of 16.
__device__ __forceinline__ void kab_bulk_prefetch_l2(const void *src, uint32_t bytes) {
  asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(src), "r"(bytes) : "memory");
}
// shared -> global bulk copy, committed as its own bulk group
__device__ __forceinline__ void kab_bulk_s2g(void *dst, const void *src, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst), "r"(kab_smem_u32(src)),
               "r"(bytes)
               : "memory");
  asm volatile("cp.async.bulk.commit_group;" ::: "memory");
}
// wait until at most 0 / 1 bulk groups still read their source; until all bulk groups are complete
__device__ __forceinline__ void kab_bulk_wait_read0() {
  asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
}
__device__ __forceinline__ void kab_bulk_wait_read1() {
  asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
}
__device__ __forceinline__ void kab_bulk_wait0() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }

// ---- fences
__device__ __forceinline__ void kab_fence_proxy_async() { asm volatile("fence.proxy.async;" ::: "memory"); }
// shared-memory-only form: SASS FENCE.VIEW.ASYNC.S without the MEMBAR.ALL.GPU of the generic one
__device__ __forceinline__ void kab_fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void kab_fence_cta() { asm volatile("fence.acq_rel.cta;" ::: "memory"); }

// ---- clusters and distributed shared memory
__device__ __forceinline__ uint32_t kab_cluster_rank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ uint32_t kab_cluster_size() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_nctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void kab_cluster_sync() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// shared::cta address -> shared::cluster address of the same variable in CTA `rank`
__device__ __forceinline__ uint32_t kab_mapa(uint32_t addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
  return r;
}
__device__ __forceinline__ void kab_st_cluster_u32(uint32_t addr, uint32_t v) {
  asm volatile("st.shared::cluster.u32 [%0], %1;" ::"r"(addr), "r"(v) : "memory");
}
// (score, seq) as ONE 64-bit store into the shared memory of any CTA of the cluster (addr from mapa)
__device__ __forceinline__ void kab_st_cluster_b64(uint32_t addr, uint32_t lo, uint32_t hi) {
  asm volatile(
      "{\n\t.reg .b64 q;\n\t"
      "mov.b64 q, {%1, %2};\n\t"
      "st.relaxed.cluster.shared::cluster.b64 [%0], q;\n\t}" ::"r"(addr), "r"(lo), "r"(hi)
      : "memory");
}
__device__ __forceinline__ void kab_red_max_cluster_s32(uint32_t addr, int v) {
  asm volatile("red.relaxed.cluster.shared::cluster.max.s32 [%0], %1;" ::"r"(addr), "r"(v) : "memory");
}
__device__ __forceinline__ void kab_red_or_cluster_u32(uint32_t addr, uint32_t v) {
  asm volatile("red.relaxed.cluster.shared::cluster.or.b32 [%0], %1;" ::"r"(addr), "r"(v) : "memory");
}
// Global scratch of one lattice of the cluster band kernels kab_bandp / kab_bandq (zeroed before every
// run), at p.fifo + lat.scr_off * 4: cons[nwt] (messages warp w is done with), then fifo[nwt][D][192 B]
__host__ __device__ inline size_t kab_cluster_fifo_off(int nwt) { return ((size_t)nwt * 4 + 255) & ~(size_t)255; }

// ---- relaxed accesses
// Global memory, .gpu scope.  (score, seq) travel as ONE 64-bit access: PTX guarantees single-copy
// atomicity for a naturally aligned .b64 access, not for a .v2.b32 vector (which the memory model
// treats as two accesses).
__device__ __forceinline__ void kab_st_volatile_b64(void *p, uint32_t lo, uint32_t hi) {
  asm volatile(
      "{\n\t.reg .b64 q;\n\t"
      "mov.b64 q, {%1, %2};\n\t"
      "st.relaxed.gpu.global.b64 [%0], q;\n\t}" ::"l"(p), "r"(lo), "r"(hi)
      : "memory");
}
__device__ __forceinline__ uint2 kab_ld_volatile_b64(const void *p) {
  uint2 v;
  asm volatile(
      "{\n\t.reg .b64 q;\n\t"
      "ld.relaxed.gpu.global.b64 q, [%2];\n\t"
      "mov.b64 {%0, %1}, q;\n\t}"
      : "=r"(v.x), "=r"(v.y)
      : "l"(p)
      : "memory");
  return v;
}
__device__ __forceinline__ uint32_t kab_ld_volatile_u32(const void *p) {
  uint32_t v;
  asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ void kab_st_volatile_u32(void *p, uint32_t v) {
  asm volatile("st.relaxed.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
// The own CTA's shared memory (32-bit shared::cta addresses), .cluster scope.
__device__ __forceinline__ uint32_t kab_lds_relaxed_u32(uint32_t addr) {
  uint32_t v;
  asm volatile("ld.relaxed.cluster.shared::cta.u32 %0, [%1];" : "=r"(v) : "r"(addr) : "memory");
  return v;
}
__device__ __forceinline__ void kab_sts_relaxed_u32(uint32_t addr, uint32_t v) {
  asm volatile("st.relaxed.cluster.shared::cta.u32 [%0], %1;" ::"r"(addr), "r"(v) : "memory");
}
__device__ __forceinline__ uint2 kab_lds_relaxed_b64(uint32_t addr) {
  uint2 v;
  asm volatile(
      "{\n\t.reg .b64 q;\n\t"
      "ld.relaxed.cluster.shared::cta.b64 q, [%2];\n\t"
      "mov.b64 {%0, %1}, q;\n\t}"
      : "=r"(v.x), "=r"(v.y)
      : "r"(addr)
      : "memory");
  return v;
}
__device__ __forceinline__ void kab_sts_b64(uint32_t addr, uint32_t lo, uint32_t hi) {  // own CTA: a plain STS.64
  asm volatile("st.shared.v2.b32 [%0], {%1, %2};" ::"r"(addr), "r"(lo), "r"(hi) : "memory");
}

// ---------------------------------------------------------------- emission staging
// Frames [f0, f0+nf) of a lattice are rows of V floats starting at byte b0 of lp.  Rows are only
// 4-byte aligned (V = 39 -> 156 B), bulk copies need 16-byte alignment, so a stage fetches the
// enclosing 16-byte aligned span and readers add `skew` words.  A span end that would run
// past the end of lp is clamped and the (< 16 B) remainder is fetched with plain loads.
struct KabStageDesc {
  const char *src;     // 16-byte aligned global address
  uint32_t bytes;      // multiple of 16 (may be 0)
  uint32_t skew;       // word index of frame f0 column 0 inside the stage buffer
  uint32_t tail_word;  // first word index not covered by the bulk copy
  uint32_t tail_n;     // number of trailing words to copy with plain loads (0..3)
};

__device__ __forceinline__ KabStageDesc kab_stage_desc(const KabParams &p, int64_t t_off, int32_t f0,
                                                       int32_t nf) {
  KabStageDesc d;
  const int64_t b0 = (t_off + f0) * (int64_t)p.V * 4;
  const int64_t b1 = b0 + (int64_t)nf * p.V * 4;
  const int64_t a0 = b0 & ~(int64_t)15;
  int64_t a1 = (b1 + 15) & ~(int64_t)15;
  if (a1 > p.lp_bytes) a1 = b1 & ~(int64_t)15;
  if (a1 < a0) a1 = a0;
  d.src = reinterpret_cast<const char *>(p.lp) + a0;
  d.bytes = (uint32_t)(a1 - a0);
  d.skew = (uint32_t)((b0 - a0) >> 2);
  d.tail_word = d.bytes >> 2;
  d.tail_n = a1 < b1 ? (uint32_t)((b1 - a1) >> 2) : 0u;
  return d;
}

// ---------------------------------------------------------------- the two cell updates (M = 4)
// Blank state (ext[v] == 0): moves 0, 1, 3 (move 2 = blank -> blank is forbidden, align.py:80-81).
// Label state: moves 0, 1, 2, 3.  Every candidate is one IEEE fp32 add (align.py:77); the scan
// is strict '>' in j order (np.argmax returns the first maximum, align.py:83), so the smallest
// move wins ties.  Written in PTX:
//   * the candidate sums come from packed fp32x2 adds (FADD2 on sm_100a: two IEEE-rn fp32 adds,
//     second operand broadcast), so adjacent states (s[2m], s[2m+1]) share one instruction;
//   * winners are taken with max.f32 (the candidates are never NaN and never -0, so max returns
//     exactly the value the reference's first-max argmax selects);
//   * the 2-bit move goes into the backpointer word with two predicated ORs.
//     bit1 / bit2 are the constants 1 << pos, 2 << pos.
__device__ __forceinline__ void kab_add2(float lo, float hi, float e, float &olo, float &ohi) {
  asm("{\n\t"
      ".reg .b64 u, v, w;\n\t"
      "mov.b64 u, {%2, %3};\n\t"
      "mov.b64 v, {%4, %4};\n\t"
      "add.rn.f32x2 w, u, v;\n\t"
      "mov.b64 {%0, %1}, w;\n\t"
      "}"
      : "=f"(olo), "=f"(ohi)
      : "f"(lo), "f"(hi), "f"(e));
}
// The same with the pair already packed (one register pair feeding two packed adds needs no copies):
// kab_pack2(lo, hi) once, kab_add2p(pair, e, ...) per addend.
__device__ __forceinline__ unsigned long long kab_pack2(float lo, float hi) {
  unsigned long long u;
  asm("mov.b64 %0, {%1, %2};" : "=l"(u) : "f"(lo), "f"(hi));
  return u;
}
__device__ __forceinline__ void kab_add2p(unsigned long long u, float e, float &olo, float &ohi) {
  asm("{\n\t"
      ".reg .b64 v, w;\n\t"
      "mov.b64 v, {%3, %3};\n\t"
      "add.rn.f32x2 w, %2, v;\n\t"
      "mov.b64 {%0, %1}, w;\n\t"
      "}"
      : "=f"(olo), "=f"(ohi)
      : "l"(u), "f"(e));
}
// Packed add with two different addends: olo = lo + elo, ohi = hi + ehi (two IEEE-rn fp32 adds).
__device__ __forceinline__ void kab_add2v(float lo, float hi, float elo, float ehi, float &olo, float &ohi) {
  asm("{\n\t"
      ".reg .b64 u, v, w;\n\t"
      "mov.b64 u, {%2, %3};\n\t"
      "mov.b64 v, {%4, %5};\n\t"
      "add.rn.f32x2 w, u, v;\n\t"
      "mov.b64 {%0, %1}, w;\n\t"
      "}"
      : "=f"(olo), "=f"(ohi)
      : "f"(lo), "f"(hi), "f"(elo), "f"(ehi));
}
// max.f32 of two / three values (FMNMX / FMNMX3).  The values-only warp forward pass takes the
// maximum BEFORE the add: rounding is monotone, so max_j fl(x_j + e) == fl(max_j x_j + e).
__device__ __forceinline__ float kab_max2(float a, float b) {
  float m;
  asm("max.f32 %0, %1, %2;" : "=f"(m) : "f"(a), "f"(b));
  return m;
}
__device__ __forceinline__ float kab_max3(float a, float b, float c) {
  float m;
  asm("max.f32 %0, %1, %2, %3;" : "=f"(m) : "f"(a), "f"(b), "f"(c));
  return m;
}
// Blank state: candidates a0 (move 0), a1 (move 1), a3 (move 3); ascending strict-'>' scan.
// The predicated "OR" is issued as mad.lo (w = one * bit + w, `one` is a register holding 1 that
// ptxas cannot fold): IMAD runs on the FMA pipe, the compares/max/selects on the ALU pipe, and
// both pipes issue at half rate on sm_100 -- this keeps them balanced.  The bits touched by one
// frame are disjoint, so the adds never carry.
// Backpointer codes: a label state stores its move (0..3); a blank state stores 0, 1 or 3 (bit 0 =
// move != 0, bit 1 = move 3), so the 2-bit code is the move for both.
__device__ __forceinline__ int kab_decode_move(uint32_t code) { return (int)code; }
__device__ __forceinline__ float kab_blank_sel(float a0, float a1, float a3, uint32_t &w, const uint32_t bit1,
                                               const uint32_t bit2, const uint32_t one) {
  float best;
  // The first maximum is the smallest move whose candidate EQUALS the 3-input maximum (FMNMX3):
  // bit 0 = (move != 0), bit 1 = (move != 0 and move != 1), i.e. codes 0, 1, 3.
  asm("{\n\t"
      ".reg .pred p1, p3;\n\t"
      "max.f32 %0, %2, %3, %4;\n\t"
      "setp.neu.f32 p1, %2, %0;\n\t"
      "setp.neu.and.f32 p3, %3, %0, p1;\n\t"
      "@p1 mad.lo.u32 %1, %7, %5, %1;\n\t"
      "@p3 mad.lo.u32 %1, %7, %6, %1;\n\t"
      "}"
      : "=f"(best), "+r"(w)
      : "f"(a0), "f"(a1), "f"(a3), "r"(bit1), "r"(bit2), "r"(one));
  return best;
}
// Label state: candidates a0..a3; tournament form of the ascending strict-'>' scan: the winner
// of (0,1) against the winner of (2,3), the upper pair wins only if strictly greater.
__device__ __forceinline__ float kab_label_sel(float a0, float a1, float a2, float a3, uint32_t &w,
                                               const uint32_t bit1, const uint32_t bit2, const uint32_t one) {
  float best;
  // m01 = max(a0, a1); best = max3(m01, a2, a3); the upper pair won iff best != m01 (strictly
  // greater); the odd candidate of the winning pair won iff its even candidate != best.
  asm("{\n\t"
      ".reg .f32 m01, z;\n\t"
      ".reg .pred ph, pl;\n\t"
      "max.f32 m01, %2, %3;\n\t"
      "max.f32 %0, m01, %4, %5;\n\t"
      "setp.neu.f32 ph, m01, %0;\n\t"
      "selp.f32 z, %4, %2, ph;\n\t"
      "setp.neu.f32 pl, z, %0;\n\t"
      "@pl mad.lo.u32 %1, %8, %6, %1;\n\t"
      "@ph mad.lo.u32 %1, %8, %7, %1;\n\t"
      "}"
      : "=f"(best), "+r"(w)
      : "f"(a0), "f"(a1), "f"(a2), "f"(a3), "r"(bit1), "r"(bit2), "r"(one));
  return best;
}
