// kab_softmax.cuh -- the normalisation in front of the alignment, align.py:116-117, on the device
// (SURVEY.md 8(f) rank 2):
//     logits -= np.mean(logits, axis=-1, keepdims=True)
//     log_probs = logits - np.log(np.sum(np.exp(logits), axis=-1, keepdims=True))
// Every step is the same IEEE fp32 operation numpy performs, in numpy's order: the two row sums
// follow numpy's pairwise summation (0 + eight strided accumulators combined as a balanced
// tree, then the tail one by one -- checked against np.sum for V = 5 ... 128), the mean is one
// fp32 division, the subtractions are single fp32 operations.  What is NOT reproducible is
// numpy's exp / log: its SIMD float32 exp differs from the correctly rounded value in ~40 % of
// the arguments and depends on the host CPU's instruction set.  The device uses CUDA's expf /
// logf (<= 2 / 1 ulp), so log_probs agree with numpy's to a few ulp (tests: 4e-6 absolute), not
// bit for bit; the alignment of those log_probs is then exact.  Opt-in for that reason: the
// default host path keeps numpy's normalisation and is bit-identical to the reference.
//
// In place (in == out) is allowed.  HBM-bound streaming kernel: a CTA copies a tile of KAB_SM_ROWS rows to shared memory with
// coalesced (16-byte when aligned) loads, one thread normalises one row (row stride odd: no
// bank conflicts), the tile is written back the same way.  Algorithmic bytes 8·V per row.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "kab_common.cuh"  // mbarrier + bulk-copy helpers

#define KAB_SM_ROWS 256     // rows per tile = threads per CTA
#define KAB_SM_MAX_V 128    // widest row of the thread-per-row kernel

// numpy's float32 pairwise sum of n <= 128 values produced in ascending order by f(i)
template <class F>
__device__ __forceinline__ float kab_np_rowsum(int n, F f) {
  if (n < 8) {
    float r = 0.f;
    for (int i = 0; i < n; ++i) r = __fadd_rn(r, f(i));
    return r;
  }
  float r[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) r[j] = f(j);
  int i = 8;
  for (; i + 8 <= n; i += 8) {
#pragma unroll
    for (int j = 0; j < 8; ++j) r[j] = __fadd_rn(r[j], f(i + j));
  }
  float res = __fadd_rn(__fadd_rn(__fadd_rn(r[0], r[1]), __fadd_rn(r[2], r[3])),
                        __fadd_rn(__fadd_rn(r[4], r[5]), __fadd_rn(r[6], r[7])));
  for (; i < n; ++i) res = __fadd_rn(res, f(i));
  return res;
}

// the same with a compile-time length (fully unrolled: f's operands stay in registers)
template <int N, class F>
__device__ __forceinline__ float kab_np_rowsum_ct(F f) {
  static_assert(N >= 8 && N <= 128, "");
  float r[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) r[j] = f(j);
#pragma unroll
  for (int i = 8; i + 8 <= N; i += 8) {
#pragma unroll
    for (int j = 0; j < 8; ++j) r[j] = __fadd_rn(r[j], f(i + j));
  }
  float res = __fadd_rn(__fadd_rn(__fadd_rn(r[0], r[1]), __fadd_rn(r[2], r[3])),
                        __fadd_rn(__fadd_rn(r[4], r[5]), __fadd_rn(r[6], r[7])));
#pragma unroll
  for (int i = N - N % 8; i < N; ++i) res = __fadd_rn(res, f(i));
  return res;
}

// ---- V = 39 (the reference's vocabulary, encoder.py:11) and 16-byte aligned buffers: persistent
// CTAs, one per SM, over full tiles of KAB_SM_ROWS rows (39 936 B, contiguous in HBM) in a ring of
// KAB_SMT_BUFS shared-memory buffers.  Thread 0 keeps two tile loads in flight (1-D bulk copies
// completing on an mbarrier), every thread normalises one row in registers and writes it back to
// the same buffer, and the tile leaves by a bulk store; a buffer is reloaded two iterations after
// its store was issued (cp.async.bulk.wait_group.read 1), so neither direction ever waits for
// the other.  The rows behind the last full tile go through kab_log_softmax_kernel.
#define KAB_SMT_BUFS 4
template <int V>
__global__ void __launch_bounds__(KAB_SM_ROWS, 1)
kab_log_softmax_tma_kernel(const float *in, float *out, int64_t n_tiles) {
  extern __shared__ __align__(128) unsigned char kab_smt_raw[];
  uint64_t *bars = reinterpret_cast<uint64_t *>(kab_smt_raw);
  float *tiles = reinterpret_cast<float *>(kab_smt_raw + 128);
  constexpr uint32_t TILE_EL = KAB_SM_ROWS * V, TILE_BYTES = TILE_EL * 4;
  static_assert(TILE_BYTES % 16 == 0 && (V & 1), "");
  if ((int64_t)blockIdx.x >= n_tiles) return;
  const int nk = (int)((n_tiles - blockIdx.x + gridDim.x - 1) / gridDim.x);
  uint64_t policy;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(policy));
  if (threadIdx.x == 0) {
    for (int b = 0; b < KAB_SMT_BUFS; ++b) kab_mbar_init(&bars[b], 1);
    kab_fence_mbar_init();
  }
  __syncthreads();
  auto issue = [&](int k) {  // thread 0 only
    const int64_t tile = blockIdx.x + (int64_t)k * gridDim.x;
    const int b = k % KAB_SMT_BUFS;
    kab_mbar_expect_tx(&bars[b], TILE_BYTES);
    kab_bulk_g2s_hint(tiles + (size_t)b * TILE_EL, in + tile * TILE_EL, TILE_BYTES, &bars[b], policy);
  };
  if (threadIdx.x == 0) {
    issue(0);
    if (nk > 1) issue(1);
  }
  for (int k = 0; k < nk; ++k) {
    const int b = k % KAB_SMT_BUFS;
    if (threadIdx.x == 0 && k + 2 < nk) {
      if (k >= 2) kab_bulk_wait_read1();  // the store of tile k-2 has left buffer (k+2) % BUFS
      issue(k + 2);
    }
    kab_mbar_wait(&bars[b], (uint32_t)(k / KAB_SMT_BUFS) & 1u);
    float *row = tiles + (size_t)b * TILE_EL + threadIdx.x * V;
    float x[V];
#pragma unroll
    for (int i = 0; i < V; ++i) x[i] = row[i];
    const float mean = __fdiv_rn(kab_np_rowsum_ct<V>([&](int i) { return x[i]; }), (float)V);
    const float se = kab_np_rowsum_ct<V>([&](int i) {
      x[i] = __fsub_rn(x[i], mean);
      return expf(x[i]);
    });
    const float lse = logf(se);
#pragma unroll
    for (int i = 0; i < V; ++i) row[i] = __fsub_rn(x[i], lse);
    kab_fence_proxy_async_smem();  // the rows -> visible to the bulk store
    __syncthreads();
    if (threadIdx.x == 0) {
      const int64_t tile = blockIdx.x + (int64_t)k * gridDim.x;
      kab_bulk_s2g(out + tile * TILE_EL, tiles + (size_t)b * TILE_EL, TILE_BYTES);
    }
  }
  if (threadIdx.x == 0) kab_bulk_wait_read0();  // shared memory must outlive the last stores' reads
}

// VT > 0: compile-time vocabulary (39: the reference's), 0: runtime V <= KAB_SM_MAX_V
template <int VT>
__global__ void __launch_bounds__(KAB_SM_ROWS)
kab_log_softmax_kernel(const float *in, float *out, int64_t n_rows, int V_rt, int vec_ok) {
  extern __shared__ __align__(16) float kab_sm_tile[];
  const int V = VT > 0 ? VT : V_rt;
  const int VS = V | 1;  // odd row stride in shared memory
  const int64_t n_tiles = (n_rows + KAB_SM_ROWS - 1) / KAB_SM_ROWS;
  for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const int64_t r0 = tile * KAB_SM_ROWS;
    const int rows = (int)min((int64_t)KAB_SM_ROWS, n_rows - r0);
    const int n_el = rows * V;
    const float *src = in + r0 * V;
    float *dst = out + r0 * V;
    // ---- tile in (flat copy; smem index = row * VS + col)
    if ((V & 1) && vec_ok) {
      const float4 *s4 = reinterpret_cast<const float4 *>(src);
      float4 *t4 = reinterpret_cast<float4 *>(kab_sm_tile);
      const int n4 = n_el >> 2;
      for (int e = threadIdx.x; e < n4; e += KAB_SM_ROWS) t4[e] = __ldcs(s4 + e);
      for (int e = (n4 << 2) + threadIdx.x; e < n_el; e += KAB_SM_ROWS) kab_sm_tile[e] = __ldcs(src + e);
    } else if (V & 1) {
      for (int e = threadIdx.x; e < n_el; e += KAB_SM_ROWS) kab_sm_tile[e] = __ldcs(src + e);
    } else {
      for (int e = threadIdx.x; e < n_el; e += KAB_SM_ROWS) kab_sm_tile[(e / V) * VS + e % V] = __ldcs(src + e);
    }
    __syncthreads();
    // ---- one row per thread
    if ((int)threadIdx.x < rows) {
      float *x = kab_sm_tile + threadIdx.x * VS;
      const float mean = __fdiv_rn(kab_np_rowsum(V, [&](int i) { return x[i]; }), (float)V);
      const float se = kab_np_rowsum(V, [&](int i) {
        const float y = __fsub_rn(x[i], mean);
        x[i] = y;
        return expf(y);
      });
      const float lse = logf(se);
      for (int i = 0; i < V; ++i) x[i] = __fsub_rn(x[i], lse);
    }
    __syncthreads();
    // ---- tile out
    if ((V & 1) && vec_ok) {
      float4 *d4 = reinterpret_cast<float4 *>(dst);
      const float4 *t4 = reinterpret_cast<const float4 *>(kab_sm_tile);
      const int n4 = n_el >> 2;
      for (int e = threadIdx.x; e < n4; e += KAB_SM_ROWS) d4[e] = t4[e];
      for (int e = (n4 << 2) + threadIdx.x; e < n_el; e += KAB_SM_ROWS) dst[e] = kab_sm_tile[e];
    } else if (V & 1) {
      for (int e = threadIdx.x; e < n_el; e += KAB_SM_ROWS) dst[e] = kab_sm_tile[e];
    } else {
      for (int e = threadIdx.x; e < n_el; e += KAB_SM_ROWS) dst[e] = kab_sm_tile[(e / V) * VS + e % V];
    }
    __syncthreads();
  }
}

// The hand-off from the acoustic model (SURVEY.md 8(f) rank 4): predict() (train.py:215-229) gets a
// padded, time-major batch `logits [T_max, B, V]` + `lens [B]` from the encoder and appends
// logits[:len_j, j, :] of every segment j to the chapter's *.logits.npz.  This kernel does that
// append and align.py:116-117 in one pass, device to device: output row out_off[j] + t (the packed
// chapter rows) = log_softmax(logits[t, j, :]).  Same arithmetic as kab_log_softmax_kernel; a CTA
// takes a tile of KAB_SM_ROWS OUTPUT rows (contiguous stores), the loads are whole 4 V-byte rows.
template <int VT>
__global__ void __launch_bounds__(KAB_SM_ROWS)
kab_log_softmax_pack_kernel(const float *__restrict__ in, int64_t B, const int64_t *__restrict__ out_off,
                            float *__restrict__ out, int64_t n_rows, int V_rt) {
  extern __shared__ __align__(16) float kab_sm_tile[];
  __shared__ const float *srow[KAB_SM_ROWS];
  const int V = VT > 0 ? VT : V_rt;
  const int VS = V | 1;
  const int64_t n_tiles = (n_rows + KAB_SM_ROWS - 1) / KAB_SM_ROWS;
  for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const int64_t r0 = tile * KAB_SM_ROWS;
    const int rows = (int)min((int64_t)KAB_SM_ROWS, n_rows - r0);
    if ((int)threadIdx.x < rows) {  // source row of output row r: segment j = last one with out_off[j] <= r
      const int64_t r = r0 + threadIdx.x;
      int64_t lo = 0, hi = B;
      while (hi - lo > 1) {
        const int64_t mid = (lo + hi) >> 1;
        if (out_off[mid] <= r) lo = mid; else hi = mid;
      }
      srow[threadIdx.x] = in + ((r - out_off[lo]) * B + lo) * V;
    }
    __syncthreads();
    const int n_el = rows * V;
    for (int e = threadIdx.x; e < n_el; e += KAB_SM_ROWS) {
      const int rr = e / V, c = e - rr * V;
      kab_sm_tile[rr * VS + c] = __ldcs(srow[rr] + c);
    }
    __syncthreads();
    if ((int)threadIdx.x < rows) {
      float *x = kab_sm_tile + threadIdx.x * VS;
      const float mean = __fdiv_rn(kab_np_rowsum(V, [&](int i) { return x[i]; }), (float)V);
      const float se = kab_np_rowsum(V, [&](int i) {
        const float y = __fsub_rn(x[i], mean);
        x[i] = y;
        return expf(y);
      });
      const float lse = logf(se);
      for (int i = 0; i < V; ++i) x[i] = __fsub_rn(x[i], lse);
    }
    __syncthreads();
    float *dst = out + r0 * V;
    for (int e = threadIdx.x; e < n_el; e += KAB_SM_ROWS) dst[e] = kab_sm_tile[(e / V) * VS + e % V];
    __syncthreads();
  }
}

// V > KAB_SM_MAX_V: a warp per row, lane-strided partial sums combined by a butterfly (the sums
// are then NOT in numpy's order -- the same few-ulp tolerance applies)
__global__ void __launch_bounds__(256)
kab_log_softmax_wide_kernel(const float *in, float *out, int64_t n_rows, int V) {
  const int lane = threadIdx.x & 31;
  const int64_t warp0 = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5), n_warps = (int64_t)gridDim.x * 8;
  for (int64_t r = warp0; r < n_rows; r += n_warps) {
    const float *x = in + r * V;
    float *y = out + r * V;
    float s = 0.f;
    for (int i = lane; i < V; i += 32) s += x[i];
#pragma unroll
    for (int d = 16; d; d >>= 1) s += __shfl_xor_sync(0xffffffffu, s, d);
    const float mean = __fdiv_rn(s, (float)V);
    float se = 0.f;
    for (int i = lane; i < V; i += 32) se += expf(__fsub_rn(x[i], mean));
#pragma unroll
    for (int d = 16; d; d >>= 1) se += __shfl_xor_sync(0xffffffffu, se, d);
    const float lse = logf(se);
    for (int i = lane; i < V; i += 32) y[i] = __fsub_rn(__fsub_rn(x[i], mean), lse);
  }
}
