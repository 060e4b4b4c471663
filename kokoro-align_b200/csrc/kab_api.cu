// kab_api.cu -- C ABI (include/kokoro_align_b200.h) over the sm_100a CTC best-path kernels.
//
// Host side of the drop-in boundary for kokoro_align/align.py:43-109: lattice
// classification, label tables (align.py:46-48), backpointer workspace, launches.
// No CPU fallback: every compute entry needs a CUDA device.
#include "../../include/kokoro_align_b200.h"

#include <algorithm>
#include <atomic>
#include <chrono>
#include <map>
#include <mutex>
#include <thread>
#include <unordered_map>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <limits>
#include <new>
#include <optional>
#include <vector>

#include "kab_band.cuh"
#include "kab_bandp.cuh"
#include "kab_bandr.cuh"
#include "kab_btpar.cuh"
#include "kab_wide.cuh"
#include "kab_common.cuh"
#include "kab_compact.cuh"
#include "kab_debug.h"
#include "kab_generic.cuh"
#include "kab_posterior.cuh"
#include "kab_posterior_chain.cuh"
#include "kab_softmax.cuh"
#include "kab_segstats.cuh"
#include "kab_spans.cuh"
#include "kab_warp.cuh"
#include "kab_pool.h"  // pool_malloc / pool_free / pool_trim_device

namespace {

thread_local char g_cuda_err[512] = "";

int cuda_fail(cudaError_t e, const char *what) {
  snprintf(g_cuda_err, sizeof(g_cuda_err), "%s: %s", what, cudaGetErrorString(e));
  return KAB_E_CUDA;
}
#define KAB_CUDA(call)                                    \
  do {                                                    \
    cudaError_t e_ = (call);                              \
    if (e_ != cudaSuccess) return cuda_fail(e_, #call);   \
  } while (0)

int sm_count_of(int device, int *out) {  // (cudaGetDeviceProperties takes milliseconds; this is cached)
  static std::atomic<int> cache[POOL_MAX_DEV];
  if (device >= 0 && device < POOL_MAX_DEV) {
    const int c = cache[device].load(std::memory_order_relaxed);
    if (c) { *out = c; return KAB_OK; }
  }
  int n = 0;
  KAB_CUDA(cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, device));
  if (device >= 0 && device < POOL_MAX_DEV) cache[device].store(n, std::memory_order_relaxed);
  *out = n;
  return KAB_OK;
}

// cudaFuncAttributeMaxDynamicSharedMemorySize is per-function, per-device GLOBAL state, while the
// size a launch needs depends on the plan (vocabulary, beam).  Several plans may be alive at once
// (best_path_files runs two side by side), so the attribute only ever GROWS: the largest size any
// plan of this process has asked for, kept under a mutex.  A launch may use any size up to it.
cudaError_t ensure_dyn_smem(const void *fn, int device, size_t bytes) {
  static std::mutex mu;
  static std::map<std::pair<const void *, int>, size_t> have;
  std::lock_guard<std::mutex> lk(mu);
  size_t &cur = have[{fn, device}];
  if (bytes <= cur) return cudaSuccess;
  const cudaError_t e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
  if (e == cudaSuccess) cur = bytes;
  return e;
}

// The ABI entry points run on the plan's device and give the caller's current device back.
struct DeviceGuard {
  int prev = -1;
  bool switched = false;
  cudaError_t enter(int device) {
    cudaError_t e = cudaGetDevice(&prev);
    if (e != cudaSuccess) return e;
    if (prev != device) {
      e = cudaSetDevice(device);
      switched = e == cudaSuccess;
    }
    return e;
  }
  ~DeviceGuard() { if (switched) cudaSetDevice(prev); }
};
// KAB_TRACE=1: wall time of the host-side phases of every call, to stderr (development)
struct Trace {
  bool on;
  const char *what;
  std::chrono::steady_clock::time_point t0;
  explicit Trace(const char *w) : on(getenv("KAB_TRACE") != nullptr), what(w), t0(std::chrono::steady_clock::now()) {}
  void mark(const char *phase) {
    if (!on) return;
    const auto t1 = std::chrono::steady_clock::now();
    fprintf(stderr, "[kab] %s: %s %.3f ms\n", what, phase, std::chrono::duration<double, std::milli>(t1 - t0).count());
    t0 = t1;
  }
};

// kernel classes (one work queue each)
constexpr int N_QUEUES = 4;
constexpr int Q_WARP = 0, Q_BAND = 1, Q_GENERIC = 2, Q_WIDE = 3;
constexpr int BAND_MAX_WARPS = 32;
constexpr int GENERIC_NT = 256;
constexpr int MAX_STAGE_V = 512;  // widest vocabulary the staged (warp / band) kernels take: whole rows
                                  // are staged, 8 frames x 2 KB x 3 stages x 4 warps = 197 KB per CTA at V = 512

inline int64_t align_up(int64_t x, int64_t a) { return (x + a - 1) / a * a; }

// the window of align.py:64-65 never clips: every frame sees the whole lattice
inline bool unbanded(int64_t T, int64_t S, int64_t W) { return W >= S && (S * (T - 1)) / T <= W / 2; }

// a lattice the band kernels take (not the warp class, and its window fits a CTA's ring)
inline bool band_shaped(int64_t T, int64_t S, int64_t W) {
  if (unbanded(T, S, W) && S <= 248) return false;  // warp class
  return W >= 1 && S <= 3 * T && std::min<int64_t>(W, S) + 32 <= (int64_t)KAB_BAND_OW * BAND_MAX_WARPS;
}

// forward CTAs of the wide kernel's chain of warps over S states (the backtrack CTA comes on top)
inline int64_t wide_ctas(int64_t S) { return ((S + KAB_BAND_OW - 1) / KAB_BAND_OW + KAB_WD_CW - 1) / KAB_WD_CW; }

int64_t cells_eval_of(int64_t T, int64_t S, int64_t W) {
  // sum_i (hi_i - lo_i), align.py:64-65.  Closed form when the window never clips.
  if (unbanded(T, S, W)) return T * S;
  int64_t cells = 0;
  for (int64_t i = 0; i < T; ++i) {
    int64_t lo = std::max<int64_t>(0, (S * i) / T - W / 2);
    int64_t hi = std::min(lo + W, S);
    if (hi > lo) cells += hi - lo;
  }
  return cells;
}

}  // namespace

// What a plan computes.  Child plans (segments, book pipes, the hybrid sub-plan) take their parent's.
struct PlanSpec {
  int32_t V = 0, W = 0, M = 0;  // (CTC: W is CTC_W, or beam_size of a banded plan, kab_plan_create_ctc_band)
  bool ctc = false;       // CTC forced-alignment plan (kab_plan_create_ctc)
  int32_t blank = 0;      // ... and its blank id
  bool ctc_long = false;  // ... whose lattices too wide for the band kernel go to the wide kernel (kab_plan_create_ctc_long)
  bool free_ends = false; // ... with free ends: the transcript may cover any window of frames (kab_plan_create_ctc_free)
};

// The kernel of a plan's band list.  CTA: kab_band.cuh (two lattices per SM).  The cluster kernels: P kab_bandp.cuh
// (KabBtLayoutP, has its own backtrack walker), Q kab_bandq.cuh (two states per lane, KabBtLayoutQ), R kab_bandr.cuh
// (Q's lanes, warp-specialised: prep warps, shared-memory mailboxes), R_GATHER kab_bandr.cuh in its gather mode
// (V > 512: emissions straight from the caller's log-probs, any number of distinct labels, no compact copy).
enum class BandKernel { CTA, P, Q, R, R_GATHER };

// How a warp, band or wide list is launched; resolved once at plan creation
struct Launch {
  const void *fn = nullptr;
  dim3 grid, block;
  size_t smem = 0;
  unsigned cluster = 0;                       // > 0: cluster dimension (cluster band kernels)
  bool cooperative = false;                   // the whole grid must be resident (wide kernel)
  int32_t stage_frames = 0, stage_bytes = 0;  // band list: the emission staging of its KabParams
};

struct kab_plan {
  int device = 0;
  int64_t B = 0, total_T = 0, total_L = 0;
  PlanSpec spec;
  int32_t Vc = 0;              // > 0: the staged kernels work on compact log-probs of Vc columns (kab_compact.cuh)
  int32_t *d_gather = nullptr;  // [B][Vc] compact column -> column of log_probs (= label value)
  float *d_lpc = nullptr;       // [sum T][Vc] compact log-probs
  int32_t *d_nonfinite = nullptr;  // [B] compact path: a non-finite value anywhere in the lattice's rows
  int max_T[4] = {0, 0, 0, 0};  // longest lattice of every work list (grid of the compaction kernels)
  int sm_count = 0;
  int32_t stage_frames = 0, stage_bytes = 0;
  int32_t band_nw = 0;  // warps per CTA of the band kernel (ring of 104 * band_nw states)
  BandKernel band_kernel = BandKernel::CTA;
  int32_t band_nc = 0, band_cw = 0;  // cluster band kernels: CTAs per cluster, compute warps per CTA
  // Hybrid band plan: the longest band lattices run in a sub-plan (kab_bandr.cuh, whole clusters: the
  // shortest frame) on a side stream while this plan's single-CTA kernel (kab_band.cuh: the highest
  // throughput) takes the others on the SMs that are left.
  kab_plan *sub = nullptr;
  cudaStream_t s_sub = nullptr;
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
  int32_t band_sm_reserved = 0;  // SMs left to the sub-plan's clusters
  unsigned int *d_started = nullptr;  // sub-plan: CTAs of kab_bandr_kernel that have started, over all runs
  unsigned int gate_target = 0;       // ... and the count the current run will bring it to
  kab_plan_info info{};
  std::vector<KabLattice> lists[N_QUEUES];
  bool any_bad_label = false;  // some lattices have a status decided here (bad label; CTC: T < L + R too)
  // device memory
  KabLattice *d_lists[N_QUEUES] = {};
  uint16_t *d_col16 = nullptr;
  int32_t *d_raw = nullptr;
  uint8_t *d_bp = nullptr;
  float *d_scratch = nullptr;
  unsigned int *d_queue = nullptr;
  int32_t *d_status_init = nullptr;
  unsigned char *d_wide_ws = nullptr;  // wide kernel: per-lattice control words and neighbour FIFOs
  int64_t wide_ws_bytes = 0;
  // parallel backtrack of the cluster band kernel (kab_btpar.cuh)
  std::vector<KabBtMeta> bt_meta;
  KabBtMeta *d_bt_meta = nullptr;
  int32_t *d_bt_maps = nullptr, *d_bt_entry = nullptr, *d_end_state = nullptr;
  int64_t bt_map_ints = 0;
  int32_t bt_blocks = 0, bt_max_wl = 0;
  unsigned char *d_band_fifo = nullptr;  // cluster band kernel: per-lattice progress counters and FIFOs
  int64_t band_fifo_bytes = 0;
  Launch launch[N_QUEUES];  // (the generic list: its grid only)
  // host copies (used to build the pipelined segments of kab_plan_run_host)
  std::vector<int64_t> h_t_off, h_l_off;
  std::vector<int32_t> h_labels;
  // kab_plan_run_host: the batch is cut into contiguous segments (child plans) so that the
  // H2D copy of segment k+1, the kernels of segment k and the D2H copy of segment k-1 overlap
  std::vector<kab_plan *> segs;
  std::vector<int64_t> seg_b0;
  // ... or, for a book (a few dozen chapter lattices, bound by the longest one): two sub-plans over the
  // same arrays -- pipe[0] the longest chapters, whose rows are copied first and whose clusters start
  // while the rest (pipe[1]) is still on its way
  static constexpr int NPIPE = 3;  // the longest chapter | the next ones, up to a third of the frames | the rest
  kab_plan *pipe[NPIPE] = {nullptr, nullptr, nullptr};
  std::vector<std::pair<int64_t, int64_t>> pipe_rows[NPIPE];  // (first row, rows) of the copies, in order
  cudaStream_t s_pipe[NPIPE] = {nullptr, nullptr, nullptr};   // ([0] unused: pipe[0] runs on `stream`)
  cudaEvent_t ev_pipe_in[NPIPE] = {nullptr, nullptr, nullptr}, ev_pipe_done[NPIPE] = {nullptr, nullptr, nullptr};
  cudaStream_t s_in = nullptr, s_out = nullptr;
  std::vector<cudaEvent_t> ev_in, ev_cmp;
  bool is_child = false;
  // streams kab_plan_run_device was last called on, each with an event recorded behind the plan's
  // kernels: kab_plan_destroy waits for THESE, not for the whole device
  std::vector<std::pair<cudaStream_t, cudaEvent_t>> run_events;
  // buffers of kab_plan_run_host (host_ready: streams, buffers and segment plans all exist)
  bool host_ready = false;
  cudaStream_t stream = nullptr;
  float *d_lp = nullptr;
  int32_t *d_path = nullptr, *d_lab = nullptr, *d_st = nullptr;
  float *d_sc = nullptr, *d_fs = nullptr;
  // segment statistics (kab_segstats.cuh)
  int64_t *d_t_off = nullptr;      // [B+1] first row of every lattice
  float *d_seg_scratch = nullptr;  // [sum T] compacted voiced scores
  int64_t *d_seg_off = nullptr;    // kab_plan_run_host_segments: [B+1] + [n_segments] boundaries on the device
  KabSegmentRecord *d_seg_rec = nullptr;
  uint8_t *d_lab8 = nullptr;
  int64_t seg_cap = 0;
  // CTC posteriors (kab_posterior.cuh), built at the first kab_plan_ctc_posteriors_device: a lattice list and
  // launch per block size, the labels with their move-2 bits, the two [sum T] value rows
  struct PostList { KabPostLat *d_lats = nullptr; int n = 0; Launch launch; int32_t bufcap = 0, e_words = 0; };
  bool post_ready = false;
  PostList post[3];
  int32_t post_F = 0, post_p_words = 0;
  int32_t *d_post_labs = nullptr;
  double *d_post_scr = nullptr;
  // ... and the chain pass (kab_posterior_chain.cuh) of unbanded long-form lattices above
  // KAB_POSTERIOR_MAX_STATES: its lattice list, launch (split: kab_ctc_posterior_chain_kernel's argument) and
  // workspace (control words and FIFOs, zeroed before every call)
  int64_t post_chain_min = KAB_POSTERIOR_MAX_STATES;  // lattices with more states take the chain pass
  KabPostChainLat *d_post_chain = nullptr;
  int post_chain_n = 0, post_chain_split = 0;
  Launch post_chain;
  unsigned char *d_post_chain_ws = nullptr;
  int64_t post_chain_ws_bytes = 0;
};

namespace {

int plan_free(kab_plan *pl);

// kab_plan_destroy waits for the plan's launches (an event behind the last one on every stream it
// was run on), not for the whole device
int record_run_event(kab_plan *pl, cudaStream_t stream) {
  if (pl->is_child) return KAB_OK;  // (the parent's streams are synchronised by the parent)
  cudaEvent_t ev = nullptr;
  for (auto &se : pl->run_events)
    if (se.first == stream) ev = se.second;
  if (!ev) {
    KAB_CUDA(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
    pl->run_events.emplace_back(stream, ev);
  }
  KAB_CUDA(cudaEventRecord(ev, stream));
  return KAB_OK;
}

// Streams, buffers and child plans of kab_plan_run_host (also the undo of a failed set-up).
void host_teardown(kab_plan *pl) {
  for (kab_plan *c : pl->segs) plan_free(c);
  pl->segs.clear();
  pl->seg_b0.clear();
  for (int k = 0; k < kab_plan::NPIPE; ++k) {
    if (pl->pipe[k]) plan_free(pl->pipe[k]);
    pl->pipe[k] = nullptr;
    pl->pipe_rows[k].clear();
    if (pl->ev_pipe_in[k]) cudaEventDestroy(pl->ev_pipe_in[k]);
    if (pl->ev_pipe_done[k]) cudaEventDestroy(pl->ev_pipe_done[k]);
    if (pl->s_pipe[k]) cudaStreamDestroy(pl->s_pipe[k]);
    pl->ev_pipe_in[k] = nullptr; pl->ev_pipe_done[k] = nullptr; pl->s_pipe[k] = nullptr;
  }
  for (cudaEvent_t e : pl->ev_in) cudaEventDestroy(e);
  for (cudaEvent_t e : pl->ev_cmp) cudaEventDestroy(e);
  pl->ev_in.clear();
  pl->ev_cmp.clear();
  pool_free(pl->d_lp); pool_free(pl->d_path); pool_free(pl->d_lab); pool_free(pl->d_st);
  pool_free(pl->d_sc); pool_free(pl->d_fs); pool_free(pl->d_seg_off); pool_free(pl->d_seg_rec); pool_free(pl->d_lab8);
  pl->d_lp = nullptr; pl->d_path = nullptr; pl->d_lab = nullptr; pl->d_st = nullptr;
  pl->d_sc = nullptr; pl->d_fs = nullptr; pl->d_seg_off = nullptr; pl->d_seg_rec = nullptr; pl->d_lab8 = nullptr;
  pl->seg_cap = 0;
  if (pl->stream) cudaStreamDestroy(pl->stream);
  if (pl->s_in) cudaStreamDestroy(pl->s_in);
  if (pl->s_out) cudaStreamDestroy(pl->s_out);
  pl->stream = nullptr; pl->s_in = nullptr; pl->s_out = nullptr;
  pl->host_ready = false;
}

// the posterior pass's device state (kab_plan_ctc_posteriors_device; also the undo of a failed set-up)
void cleanup_post(kab_plan *pl) {
  for (auto &l : pl->post) { pool_free(l.d_lats); l = kab_plan::PostList{}; }
  pool_free(pl->d_post_labs); pool_free(pl->d_post_scr); pool_free(pl->d_post_chain); pool_free(pl->d_post_chain_ws);
  pl->d_post_labs = nullptr; pl->d_post_scr = nullptr; pl->d_post_chain = nullptr; pl->d_post_chain_ws = nullptr;
  pl->post_chain_n = 0; pl->post_chain_split = 0; pl->post_chain = Launch{}; pl->post_chain_ws_bytes = 0;
  pl->post_ready = false;
}

int plan_free(kab_plan *pl) {
  if (!pl) return KAB_OK;
  Trace tr("kab_plan_destroy");
  DeviceGuard guard;
  guard.enter(pl->device);
  // pooled blocks may be handed to another plan at once, so nothing of this one may still be in
  // flight (kab_plan_run_device is asynchronous): wait for the plan's own launches -- the events
  // recorded behind them -- not for the device, which would stall the caller's unrelated streams
  for (auto &se : pl->run_events) {
    cudaEventSynchronize(se.second);
    cudaEventDestroy(se.second);
  }
  pl->run_events.clear();
  if (pl->stream) cudaStreamSynchronize(pl->stream);
  if (pl->s_out) cudaStreamSynchronize(pl->s_out);
  host_teardown(pl);
  if (pl->s_sub) cudaStreamSynchronize(pl->s_sub);
  if (pl->sub) plan_free(pl->sub);
  if (pl->ev_fork) cudaEventDestroy(pl->ev_fork);
  if (pl->ev_join) cudaEventDestroy(pl->ev_join);
  if (pl->s_sub) cudaStreamDestroy(pl->s_sub);
  for (int q = 0; q < N_QUEUES; ++q) pool_free(pl->d_lists[q]);
  pool_free(pl->d_col16); pool_free(pl->d_raw); pool_free(pl->d_bp); pool_free(pl->d_scratch);
  pool_free(pl->d_queue); pool_free(pl->d_status_init); pool_free(pl->d_wide_ws); pool_free(pl->d_band_fifo); pool_free(pl->d_bt_meta); pool_free(pl->d_bt_maps); pool_free(pl->d_bt_entry); pool_free(pl->d_end_state); pool_free(pl->d_gather); pool_free(pl->d_lpc); pool_free(pl->d_nonfinite); pool_free(pl->d_t_off); pool_free(pl->d_seg_scratch); pool_free(pl->d_started);

  cleanup_post(pl);
  delete pl;
  tr.mark("free");
  return KAB_OK;
}

}  // namespace

extern "C" {

int kab_version(void) { return KAB_VERSION; }

const char *kab_error_string(int code) {
  switch (code) {
    case KAB_OK: return "ok";
    case KAB_E_CUDA: return "CUDA error (see kab_last_cuda_error)";
    case KAB_E_BAD_ARG: return "bad argument";
    case KAB_E_NOMEM: return "out of host memory";
    case KAB_E_UNSUPPORTED: return "unsupported shape";
    default: return "unknown error";
  }
}

const char *kab_last_cuda_error(void) { return g_cuda_err; }

int kab_device_count(int *count) {
  if (!count) return KAB_E_BAD_ARG;
  KAB_CUDA(cudaGetDeviceCount(count));
  return KAB_OK;
}

namespace {
// mask: only the lattices with mask[b] != 0 belong to this plan (nullptr: all); band_mode: -1 the
// plan chooses (and may go hybrid), 0 the single-CTA band kernel, 1 kab_bandr.cuh
int plan_create_impl(kab_plan **out, int device, const PlanSpec &s, int64_t B, const int64_t *t_off,
                     const int32_t *labels, const int64_t *l_off, const uint8_t *mask, int band_mode);
// CTC plans: three moves; default and long-form plans leave every lattice unbanded -- a window this wide
// is [0, S) in every frame of the band kernel (S <= 3296 there)
constexpr int32_t CTC_W = 0x3fffffff, CTC_M = 3;
// banded CTC plans: a lattice whose window clips runs on the single-CTA band kernel while min(W, S) is at
// most this, otherwise on the generic kernel (the NW = 32 ring holds 3328 states: 64 to spare, where
// band_shaped asks for 32)
constexpr int64_t CTC_BAND_MAX_W = 3264;
}  // namespace

int kab_plan_create(kab_plan **out, int device, int64_t B, const int64_t *t_off, const int32_t *labels,
                    const int64_t *l_off, int32_t V, int32_t W, int32_t M) {
  return plan_create_impl(out, device, PlanSpec{V, W, M}, B, t_off, labels, l_off, nullptr, -1);
}

int kab_plan_create_ctc(kab_plan **out, int device, int64_t B, const int64_t *t_off, const int32_t *labels,
                        const int64_t *l_off, int32_t V, int32_t blank) {
  if (blank < 0 || blank >= V) return KAB_E_BAD_ARG;
  // (only the single-CTA band kernel has a CTC mode)
  return plan_create_impl(out, device, PlanSpec{V, CTC_W, CTC_M, true, blank}, B, t_off, labels, l_off, nullptr, 0);
}

int kab_plan_create_ctc_long(kab_plan **out, int device, int64_t B, const int64_t *t_off, const int32_t *labels,
                             const int64_t *l_off, int32_t V, int32_t blank) {
  if (blank < 0 || blank >= V) return KAB_E_BAD_ARG;
  // (the single-CTA band kernel below S = 3297, the wide kernel above it where it fits)
  return plan_create_impl(out, device, PlanSpec{V, CTC_W, CTC_M, true, blank, true}, B, t_off, labels, l_off, nullptr, 0);
}

int kab_plan_create_ctc_free(kab_plan **out, int device, int64_t B, const int64_t *t_off, const int32_t *labels,
                             const int64_t *l_off, int32_t V, int32_t blank) {
  if (blank < 0 || blank >= V) return KAB_E_BAD_ARG;
  // (routed as by kab_plan_create_ctc_long: every lattice is unbanded)
  return plan_create_impl(out, device, PlanSpec{V, CTC_W, CTC_M, true, blank, true, true}, B, t_off, labels, l_off, nullptr, 0);
}

int kab_plan_create_ctc_band(kab_plan **out, int device, int64_t B, const int64_t *t_off, const int32_t *labels,
                             const int64_t *l_off, int32_t V, int32_t blank, int32_t beam_size) {
  if (blank < 0 || blank >= V || beam_size < 1) return KAB_E_BAD_ARG;
  // (lattices the window covers are routed as by kab_plan_create_ctc_long)
  return plan_create_impl(out, device, PlanSpec{V, beam_size, CTC_M, true, blank, true}, B, t_off, labels, l_off, nullptr, 0);
}

namespace {

// The development / test knobs KAB_<NAME> of INTEGRATION.md section 6 (-1: not set), read at every plan
// creation: tests change them between plans.  serial_bt: KAB_BAND_SERIAL_BT != 0.
struct Knobs {
  int stage_frames, band_cluster, band_q, band_r, band_hybrid, serial_bt, warp_ctas_per_sm;
  bool band_gather, ctc_compact, serial_setup;
  static int get(const char *name) { const char *v = getenv(name); return v ? atoi(v) : -1; }
  static Knobs read() {
    const char *sb = getenv("KAB_BAND_SERIAL_BT");
    return Knobs{get("KAB_STAGE_FRAMES"), get("KAB_BAND_CLUSTER"), get("KAB_BAND_Q"), get("KAB_BAND_R"), get("KAB_BAND_HYBRID"),
                 sb ? (atoi(sb) != 0) : -1, get("KAB_WARP_CTAS_PER_SM"), get("KAB_BAND_GATHER") != 0, get("KAB_CTC_COMPACT") != 0,
                 getenv("KAB_SERIAL_SETUP") != nullptr};
  }
};

// what the label scan finds out about one lattice (repeats: adjacent equal labels)
struct LatFacts { uint8_t bad, special, compact; int32_t distinct, repeats; int64_t col_off; };

// The working state of one plan creation, handed from stage to stage
struct Setup {
  kab_plan *pl;
  const PlanSpec &s;
  const Knobs knob;
  int64_t B;
  const int64_t *t_off, *l_off;
  const int32_t *labels;
  const uint8_t *mask;
  bool gather = false;  // band-shaped lattices run kab_bandr.cuh's gather mode (BandKernel::R_GATHER)
  int32_t Veff = 0;     // vocabulary the staged kernels see
  std::vector<LatFacts> facts;
  std::vector<int32_t> gather_rows;  // [B][Vc] compact column -> column of log_probs
  std::vector<uint16_t> col16;
  std::vector<int32_t> status_init;
  int64_t bp_bytes = 0, scr_floats = 0, max_band_weff = 0;
  int wide_capacity = 0, wide_max_ctas = 0;
  std::vector<uint8_t> hyb_mask;  // hybrid band plan: the lattices of the sub-plan
  int hyb_k = 0;                  // ... and its clusters
  bool in(int64_t b) const { return !mask || mask[b]; }
  int64_t frames(int64_t b) const { return t_off[b + 1] - t_off[b]; }
  int64_t len(int64_t b) const { return l_off[b + 1] - l_off[b]; }
  void for_lattices(const std::function<void(int64_t, int64_t *)> &fn) const;
  void scan_labels(), compact_vocabulary(), classify(), choose_band_kernel(int band_mode), lay_out_band();
  int allocate(), finish();
};

// The label scans (range check, distinct labels, column table) are independent per lattice and are
// most of plan creation for a batch of 10 000 segments (4.5 of 5 ms): several host threads do them
// ahead of the (cheap, sequential) classification.  fn(b, scratch bit words) over the plan's lattices.
void Setup::for_lattices(const std::function<void(int64_t, int64_t *)> &fn) const {
  const int n_mask = (s.V + 63) / 64;
  const unsigned hw = std::thread::hardware_concurrency();
  const int nt = (B >= 2048 && pl->total_L >= 65536 && hw >= 4 && !knob.serial_setup) ? (int)std::min<unsigned>(8, hw / 2) : 1;
  auto work = [&](int t) {
    std::vector<int64_t> words((size_t)std::max(n_mask, 1), 0);
    const int64_t b0 = B * t / nt, b1 = B * (t + 1) / nt;
    for (int64_t b = b0; b < b1; ++b)
      if (in(b)) fn(b, words.data());
  };
  std::vector<std::thread> th;
  for (int t = 1; t < nt; ++t) th.emplace_back(work, t);
  work(0);
  for (auto &w : th) w.join();
}

void Setup::scan_labels() {
  const int n_mask = (s.V + 63) / 64;
  facts.assign((size_t)B, LatFacts{});
  for_lattices([&](int64_t b, int64_t *seen) {
    const int64_t L = len(b);
    const int32_t *lab = labels + l_off[b];
    LatFacts f{};
    std::fill(seen, seen + n_mask, (int64_t)0);
    for (int64_t l = 0; l < L; ++l) {
      if (s.ctc ? (lab[l] < 0 || lab[l] >= s.V || lab[l] == s.blank) : (lab[l] < -s.V || lab[l] >= s.V)) { f.bad = 1; break; }
      if (!s.ctc && lab[l] <= 0) f.special = 1;  // (CTC: the blank test is the state's parity, any label is fast)
      if (l > 0 && lab[l] == lab[l - 1]) ++f.repeats;
      const int32_t c = lab[l] < 0 ? lab[l] + s.V : lab[l];
      if (!(seen[c >> 6] >> (c & 63) & 1)) { seen[c >> 6] |= (int64_t)1 << (c & 63); ++f.distinct; }
    }
    facts[(size_t)b] = f;
  });
}

// ---- stage 2: wide vocabularies -- can the staged kernels work on a compact copy of the log-probs?  Then
// the emission staging and the padded column table (numpy-style wrap of negative labels).
void Setup::compact_vocabulary() {
  // Band-shaped lattices of a wide vocabulary do not need the compact copy at all: kab_bandr.cuh's
  // gather mode reads log_probs[t, label] itself (VERDICT round 1, item 8: a chapter with more than
  // 511 distinct BPE tokens sent the whole plan to the generic kernel).  It is used when every
  // band-shaped lattice of the plan fits that kernel's ring (beam + 32 <= 1280 states).
  const int64_t ga_max_weff = (int64_t)KAB_BQ_OW * KAB_BR_CW * 8 - 32;
  bool ok = !s.ctc && s.V > MAX_STAGE_V && s.M <= 4 && knob.band_gather && kab_bandr_geom(64).smem_bytes <= 227 * 1024, any_band = false;
  for (int64_t b = 0; b < B && ok; ++b) {
    const int64_t S = 2 * len(b) + 1;
    if (in(b) && band_shaped(frames(b), S, s.W)) { any_band = true; ok = std::min<int64_t>(s.W, S) <= ga_max_weff; }
  }
  gather = ok && any_band;
  // Vc: the blank's column and the most distinct labels of a lattice that goes through the copy.  CTC plans
  // (kab_compact_ctc_kernel): one with more than MAX_STAGE_V - 1 distinct labels goes to the generic kernel on
  // its own instead of taking the whole plan there; KAB_CTC_COMPACT=0 (the reference arm of the tests and
  // tools/forced_align_vocab_bench.py) sends every lattice there.
  int64_t dmax = -1, off = 0;
  for (int64_t b = 0; b < B; ++b) {
    if (!in(b)) continue;
    LatFacts &f = facts[(size_t)b];
    f.col_off = off;  // in the padded column table (a bad-label lattice has no columns)
    if (f.bad) continue;
    off += align_up(len(b), 8) + 8;
    if (f.special || (gather && band_shaped(frames(b), 2 * len(b) + 1, s.W))) continue;
    if (!s.ctc || f.distinct + 1 <= MAX_STAGE_V) dmax = std::max<int64_t>(dmax, f.distinct);
  }
  if (s.V > MAX_STAGE_V && (s.ctc ? knob.ctc_compact : s.M <= 4) && dmax >= 0 && dmax + 1 <= MAX_STAGE_V) {
    pl->Vc = (int32_t)std::max<int64_t>(8, align_up(dmax + 1, 4));
    gather_rows.assign((size_t)B * pl->Vc, 0);
  }
  Veff = pl->Vc ? pl->Vc : s.V;

  // emission staging geometry: ~4 KB stages, at most 16 frames each
  pl->stage_frames = Veff <= 64 ? 16 : 8;  // multiple of 8: frame groups never straddle stages
  if (knob.stage_frames == 8 || knob.stage_frames == 16 || knob.stage_frames == 32) pl->stage_frames = knob.stage_frames;
  pl->stage_bytes = (int32_t)align_up((int64_t)pl->stage_frames * Veff * 4 + 24, 16);

  col16.assign((size_t)off, 0);
  const int n_mask = (s.V + 63) / 64;
  for_lattices([&](int64_t b, int64_t *seen) {  // the compact numbering's gather rows, the column table
    LatFacts &f = facts[(size_t)b];
    if (f.bad) return;
    const int64_t L = len(b);
    const int32_t *lab = labels + l_off[b];
    uint16_t *c = col16.data() + f.col_off;
    const bool ga = gather && !f.special && band_shaped(frames(b), 2 * L + 1, s.W);
    if (pl->Vc && !f.special && !ga && f.distinct + 1 <= pl->Vc) {
      // compact numbering: the blank's column (0, or the CTC blank id), then the lattice's distinct label
      // columns in ascending order
      f.compact = 1;
      std::fill(seen, seen + n_mask, (int64_t)0);
      for (int64_t l = 0; l < L; ++l) seen[lab[l] >> 6] |= (int64_t)1 << (lab[l] & 63);
      int32_t *g = gather_rows.data() + (size_t)b * pl->Vc;
      g[0] = s.ctc ? s.blank : 0;
      int32_t n = 1;
      for (int w = 0; w < n_mask; ++w)
        for (int64_t m = seen[w]; m; m &= m - 1) g[n++] = w * 64 + __builtin_ctzll((unsigned long long)m);
      for (int64_t l = 0; l < L; ++l) c[l] = (uint16_t)(std::lower_bound(g + 1, g + n, lab[l]) - g);
    } else {
      for (int64_t l = 0; l < L; ++l) c[l] = (uint16_t)(lab[l] < 0 ? lab[l] + s.V : lab[l]);
    }
  });
}

// ---- stage 3: the work lists (warp, band, wide, generic); the offsets of all but the band list
void Setup::classify() {
  const int64_t W = s.W, M = s.M;
  // resident CTAs of the wide kernel (its warps spin on each other: the whole grid must be resident)
  Launch &lw = pl->launch[Q_WIDE];
  lw = Launch{s.free_ends ? (const void *)kab_wide_ctc_free_kernel
              : s.ctc ? (const void *)kab_wide_ctc_kernel : (const void *)kab_wide_kernel, dim3(), dim3(KAB_WD_THREADS),
              kab_wide_geom(pl->stage_bytes).smem_bytes, 0, true};
  {
    int occ = 0;
    if (lw.smem <= 227 * 1024 && ensure_dyn_smem(lw.fn, pl->device, lw.smem) == cudaSuccess &&
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, lw.fn, KAB_WD_THREADS, lw.smem) == cudaSuccess)
      wide_capacity = occ * pl->sm_count;
    (void)cudaGetLastError();
  }
  // CTC long-form plans: the wide kernel runs its lattices one after another, each on the whole GPU; the
  // generic kernel runs them side by side, one CTA each.  A makespan estimate from measured costs (B200, V = 32,
  // tools/forced_align_long_bench.py, DESIGN.md 3.9) gives all lattices that both kernels could take to one of
  // them: wide ~102 ns per frame of a sequence of lattices; generic 0.68 Gcells/s for a lone lattice (its
  // longest one bounds it) and 79 Gcells/s for 256 lattices side by side.  256 utterances of 2-5 minutes:
  // 276 ms wide, 230 ms generic; one 10-minute utterance: 5.2 ms wide, 796 ms generic.  (Compact plans, V > 512:
  // 177 ns per frame wide at Vc = 272 and 0.58 Gcells/s for a lone generic lattice at V = 1025; the constants
  // stay, DESIGN.md 3.9c.)
  bool ctc_wide = false;
  if (s.ctc && s.ctc_long) {
    double sum_t = 0.0, cells = 0.0, max_cells = 0.0;
    for (int64_t b = 0; b < B; ++b) {
      if (!in(b) || facts[(size_t)b].bad) continue;
      if (pl->Vc && !facts[(size_t)b].compact) continue;  // (too many distinct labels for the compact copy: generic)
      const int64_t T = frames(b), S = 2 * len(b) + 1;
      if (!unbanded(T, S, W)) continue;                      // (banded plans: band or generic class)
      if (S + 32 <= KAB_BAND_OW * BAND_MAX_WARPS) continue;  // warp or band class
      if (wide_ctas(S) + 1 > wide_capacity) continue;
      sum_t += (double)T;
      cells += (double)T * (double)S;
      max_cells = std::max(max_cells, (double)T * (double)S);
    }
    ctc_wide = sum_t * 102.0 <= std::max(max_cells / 0.68, cells / 79.0);  // (ns)
  }
  kab_plan_info &info = pl->info;
  status_init.assign((size_t)B, 0);
  for (int64_t b = 0; b < B; ++b) {
    if (!in(b)) continue;
    const int64_t T = frames(b), L = len(b), S = 2 * L + 1;
    const LatFacts &f = facts[(size_t)b];
    // reference: IndexError at align.py:77; CTC: no path fits when T < L + R (R = adjacent equal labels,
    // which need a blank between)
    if (f.bad || (s.ctc && T < L + f.repeats)) {
      status_init[(size_t)b] = f.bad ? KAB_ST_BAD_LABEL : KAB_ST_DEAD_BAND;
      pl->any_bad_label = true;
      continue;
    }
    KabLattice d{};
    d.t_off = t_off[b];
    d.lab_off = l_off[b];
    d.T = (int32_t)T; d.L = (int32_t)L; d.index = (int32_t)b;
    d.col_off = f.col_off;
    const bool ga = gather && !f.special && band_shaped(T, S, W);  // gather mode: the labels stay column numbers

    // max_move 1 .. 3 run in the same kernels (their MM instantiations turn the excluded moves'
    // candidates into -inf); more than four moves only exist in the generic kernel
    const bool fast = M <= 4 && !f.special && (ga || (Veff <= MAX_STAGE_V && (!pl->Vc || f.distinct + 1 <= pl->Vc)));
    const bool full = unbanded(T, S, W);
    const int64_t weff = std::min<int64_t>(W, S);
    int q;
    if (fast && !ga && full && S <= 248) {
      q = Q_WARP;
      d.k = S <= 62 ? 2 : (S <= 124 ? 4 : (S <= 186 ? 6 : 8));  // 31 lanes x K states
      d.bp_off = bp_bytes;
      if (s.ctc || d.k <= 4) {  // backpointer word-rows (kab_warp_align: the BP scheme)
        const int fpw = d.k <= 2 ? 8 : (d.k <= 4 ? 4 : 2);
        bp_bytes += align_up((T + fpw - 1) / fpw * 128, 256);
      } else {  // score checkpoint rows, one per KAB_CKPT_C frames
        bp_bytes += align_up((T + KAB_CKPT_C - 1) / KAB_CKPT_C * kab_ckpt_stride((int)S, d.k) * 4, 256);
      }
    } else if (fast && band_shaped(T, S, W) && (!s.ctc || full || weff <= CTC_BAND_MAX_W)) {
      q = Q_BAND;  // backpointer offsets are assigned by lay_out_band, once the kernel is known
      max_band_weff = std::max(max_band_weff, weff);
    } else if (fast && !ga && (s.ctc ? ctc_wide : M == 4) && full && wide_ctas(S) + 1 <= wide_capacity) {
      q = Q_WIDE;  // unbanded and wider than a CTA: a chain of warps over the whole GPU
      const int nww = (int)((S + KAB_BAND_OW - 1) / KAB_BAND_OW);
      d.k = nww;
      wide_max_ctas = std::max(wide_max_ctas, (int)wide_ctas(S));
      d.bp_off = bp_bytes;
      bp_bytes += (int64_t)nww * ((T + 7) / 8) * 256;  // [warp][group][32 lanes][8 B]
      d.scr_off = pl->wide_ws_bytes / 4;
      pl->wide_ws_bytes += (int64_t)align_up((int64_t)kab_wide_ws_bytes(nww), 256);
    } else {
      q = Q_GENERIC;
      d.bp_off = bp_bytes;
      bp_bytes += align_up(T * std::max<int64_t>(1, weff), 256);
      d.scr_off = scr_floats;
      scr_floats += align_up(2 * (S + 16), 64);
    }
    pl->lists[q].push_back(d);
    pl->max_T[q] = std::max(pl->max_T[q], (int)T);
    info.n_class[q == Q_WARP ? KAB_CLASS_WARP : (q == Q_GENERIC ? KAB_CLASS_GENERIC : (q == Q_WIDE ? KAB_CLASS_WIDE : KAB_CLASS_BAND))]++;
    const int64_t cells = cells_eval_of(T, S, W);
    info.cells_eval += cells;
    info.cells_nominal += T * S;
    int bbits = 0;
    while ((1 << bbits) < M) ++bbits;
    const int64_t dcols = std::min<int64_t>(s.V, f.distinct + 1);
    info.algorithmic_bytes += 4 * dcols * T + (cells * bbits + 7) / 8 + (T * bbits + 7) / 8 + 12 * T;
  }
}

// ---- stage 4: the band list's kernel, from makespan estimates and the knobs; maybe a hybrid split
void Setup::choose_band_kernel(int band_mode) {
  std::vector<KabLattice> &bl = pl->lists[Q_BAND];
  if (bl.empty()) return;
  pl->band_nw = (int32_t)((max_band_weff + 32 + KAB_BAND_OW - 1) / KAB_BAND_OW);
  // Two band kernels.  The pipelined cluster kernel (kab_bandp.cuh: rings of 4 * NC warps over a
  // cluster of NC <= 8 CTAs, one warp per scheduler) has the shorter frame (Gon gitsune 14.2 vs
  // 15.4 ms, config 4(i) 168 vs 188 ms) but takes NC whole SMs per lattice; the single-CTA kernel
  // (kab_band.cuh) runs two lattices per SM.  So: the cluster kernel when every band lattice of
  // the plan gets its own cluster at once, the single-CTA kernel for larger batches.
  // KAB_BAND_CLUSTER=0 forces the single-CTA kernel, =N (>= 1) the cluster kernel with >= N CTAs.
  const int nc = (pl->band_nw + KAB_BP_CW - 1) / KAB_BP_CW;
  int want_nc = knob.band_cluster;
  if (band_mode >= 0) want_nc = band_mode == 0 ? 0 : -1;  // (sub-plans of a hybrid plan: the kernel is given)
  const bool cluster_ok = nc <= 8 && kab_bandp_geom(pl->stage_bytes).smem_bytes <= 227 * 1024;
  // kab_bandq.cuh (two warps per scheduler, two states per lane: the shorter frame) when its ring
  // of 40-slot warps fits a cluster of <= 8 CTAs and every lattice gets its own cluster at once;
  // KAB_BAND_Q=0 keeps kab_bandp.cuh, =1 forces kab_bandq.cuh whenever its geometry allows
  const int nwq = (int)((max_band_weff + 32 + KAB_BQ_OW - 1) / KAB_BQ_OW);
  const int ncq = (nwq + KAB_BQ_CW - 1) / KAB_BQ_CW;
  const bool q_ok = ncq <= 8 && kab_bandq_geom(pl->stage_bytes).smem_bytes <= 227 * 1024;
  // kab_bandr.cuh: the same lanes with ONE compute warp per scheduler and the bookkeeping on helper
  // warps -- by far the shortest frame, at 4 compute warps per CTA (7 CTAs for the 1000-wide band).
  // Its clusters take lattices from the work queue, so a plan may hold more lattices than clusters.
  // KAB_BAND_R=0 disables it, =1 forces it whenever its geometry allows.
  const int ncr = (nwq + KAB_BR_CW - 1) / KAB_BR_CW;
  const bool r_ok = gather || (ncr <= 8 && pl->stage_frames == KAB_BR_F && kab_bandr_geom(pl->stage_bytes).smem_bytes <= 227 * 1024);
  const int want_q = band_mode >= 0 ? (band_mode == 0 ? 0 : -1) : knob.band_q;
  const int want_r = band_mode >= 0 ? band_mode : knob.band_r;
  int64_t n_band = (int64_t)bl.size();
  // Which kernel for this plan?  A makespan estimate from measured per-frame costs (B200, 1000-wide
  // band): kab_bandr.cuh ~70 ns per frame on one of sm_count / ncr clusters that pull lattices from
  // the work queue, kab_band.cuh ~190 ns per frame with two lattices per SM.  A book (36 chapters)
  // is bound by its longest chapter -> bandr; hundreds of chapters at once -> the single-CTA kernel.
  double sum_t = 0.0, max_t = 0.0, bt_steps = 0.0;
  for (const KabLattice &d : bl) {
    sum_t += d.T; max_t = std::max(max_t, (double)d.T);
    bt_steps += (double)d.T * (double)std::min<int64_t>(s.W, 2 * (int64_t)d.L + 1);
  }
  // (bandr: 70 ns per frame for the longest lattice; with every cluster of the GPU busy on a queue of
  // lattices ~90 ns per frame of a cluster's share, plus the map walkers of the parallel traceback at
  // 1.85e12 steps/s -- 162 chapters on one GPU: 60.6 ms measured, 59 estimated; the first version of
  // this estimate (70 ns, no traceback) said 41 and took the plan away from the single-CTA kernel's 49)
  const double est_r = std::max(max_t * 70.0, sum_t / std::max(1, pl->sm_count / std::max(1, ncr)) * 90.0) + bt_steps * 0.55e-3;
  // (190 ns per frame is a lone lattice's latency in the single-CTA kernel; with every SM holding two of
  // them a CTA slot's frames cost ~330 ns each -- 18 books on one GPU: 49 M frames / 296 slots, 54.5 ms.
  // The estimates keep the one figure: with 330 in the throughput terms the split below was chosen
  // less often and measured worse, 36.9 instead of 34.9 ms for 18 books on two GPUs.)
  const double est_b = std::max(max_t, sum_t / (double)(pl->sm_count * (pl->band_nw <= 16 ? 2 : 1))) * 190.0;
  const bool use_r = gather || (r_ok && want_r != 0 && want_nc != 0 && want_q != 0 && (want_r >= 1 || want_nc >= 1 || est_r <= est_b));
  const bool use_q = !use_r && s.M == 4 && q_ok && want_q != 0 && want_nc != 0 && (want_q >= 1 || n_band <= pl->sm_count / ncq);
  // Hybrid: a plan of hundreds of chapters takes the single-CTA kernel (throughput), but its makespan
  // is then the LONGEST chapter at that kernel's 190 ns per frame.  Give the longest ones to
  // kab_bandr.cuh (70 ns per frame) on k clusters and the rest to the single-CTA kernel on the other
  // SMs, side by side: the split (k clusters, the m longest lattices) with the smallest estimated
  // makespan, taken when it beats the single kernel by 15 %.  KAB_BAND_HYBRID=0 / 1 disables / forces it.
  const int want_h = knob.band_hybrid;
  if (band_mode < 0 && !mask && !use_r && !use_q && r_ok && !gather && !pl->Vc && s.V <= MAX_STAGE_V && want_h != 0 &&
      want_r < 0 && want_q < 0 && want_nc < 0 && n_band >= 2) {
    std::stable_sort(bl.begin(), bl.end(), [](const KabLattice &a, const KabLattice &b2) { return a.T > b2.T; });
    std::vector<double> pre((size_t)n_band + 1, 0.0);
    for (int64_t i = 0; i < n_band; ++i) pre[(size_t)i + 1] = pre[(size_t)i] + bl[(size_t)i].T;
    const int per_sm = pl->band_nw <= 16 ? 2 : 1;
    double best = est_b;
    int best_k = 0;
    int64_t best_m = 0;
    for (int k = 1; k <= pl->sm_count / ncr / 2; ++k) {
      const double sm_left = (double)(pl->sm_count - k * ncr) * per_sm;
      for (int64_t m = k; m < n_band && m <= 16 * (int64_t)k; ++m) {
        const double tr_ = std::max((double)bl[0].T, pre[(size_t)m] / k) * 70.0;
        const double tb_ = std::max((double)bl[(size_t)m].T, (sum_t - pre[(size_t)m]) / sm_left) * 190.0;
        const double ms = std::max(tr_, tb_);
        if (ms < best) { best = ms; best_k = k; best_m = m; }
      }
    }
    if (want_h >= 1 && best_k == 0) { best_k = 1; best_m = 1; }
    if (best_k > 0 && (want_h >= 1 || best < 0.85 * est_b)) {
      hyb_mask.assign((size_t)B, 0);
      for (int64_t i = 0; i < best_m; ++i) hyb_mask[(size_t)bl[(size_t)i].index] = 1;
      bl.erase(bl.begin(), bl.begin() + best_m);
      hyb_k = best_k;
      want_nc = 0;  // (the rest: the single-CTA kernel, whatever its number)
      pl->band_sm_reserved = best_k * ncr;
      pl->max_T[Q_BAND] = bl.empty() ? 0 : bl[0].T;
    }
  }
  if (use_r || use_q) {
    pl->band_kernel = use_q ? BandKernel::Q : (gather ? BandKernel::R_GATHER : BandKernel::R);
    pl->band_cw = use_r ? KAB_BR_CW : KAB_BQ_CW; pl->band_nc = use_r ? ncr : ncq;
    return;
  }
  if (want_nc < 0 && cluster_ok) {
    // resident clusters of this size: every SM holds one CTA of the cluster kernel
    const int64_t resident = pl->sm_count / nc;
    want_nc = (int64_t)bl.size() <= resident ? nc : 0;
  }
  if (s.M == 4 && cluster_ok && want_nc >= 1) {
    pl->band_kernel = BandKernel::P;
    pl->band_cw = KAB_BP_CW; pl->band_nc = std::min(8, std::max(nc, want_nc));
  }
}

bool band_layout_q(BandKernel k) { return k == BandKernel::Q || k == BandKernel::R || k == BandKernel::R_GATHER; }

// ---- stage 5: band backpointers and workspaces, longest-first order, the parallel backtrack's maps
void Setup::lay_out_band() {
  const BandKernel bk = pl->band_kernel;
  const int nwt = pl->band_cw * pl->band_nc;
  const int nbp = pl->band_nw ? kab_band_geom(pl->band_nw, pl->stage_bytes).nbp : 0;  // (single-CTA kernel)
  for (KabLattice &d : pl->lists[Q_BAND]) {
    d.bp_off = bp_bytes;
    if (bk == BandKernel::CTA) {
      bp_bytes += align_up((int64_t)d.T * nbp, 256);
      continue;
    }
    // [warp][group][32 lanes][4 B] (KabBtLayoutQ) or [8 B] (KabBtLayoutP)
    bp_bytes += (int64_t)((d.T + 7) / 8) * (band_layout_q(bk) ? 128 : 256) * nwt;
    d.scr_off = pl->band_fifo_bytes / 4;
    pl->band_fifo_bytes += (int64_t)align_up((int64_t)(band_layout_q(bk) ? kab_bandq_ws_bytes(nwt) : kab_bandp_ws_bytes(nwt)), 256);
  }
  // longest-processing-time-first order inside every queue
  for (int q = 0; q < N_QUEUES; ++q)
    std::stable_sort(pl->lists[q].begin(), pl->lists[q].end(), [&](const KabLattice &a, const KabLattice &b2) {
      // warp class: K-major (warps resident on one SM then run the same code variant, which
      // keeps the instruction cache warm), longest first inside each K and the cheap K = 2
      // lattices last, where they fill the tail
      if (q == Q_WARP && a.k != b2.k) return a.k > b2.k;
      return a.T > b2.T;
    });

  // parallel backtrack of the cluster band kernels: per-lattice block maps.  kab_bandq.cuh and kab_bandr.cuh
  // have no walker of their own; kab_bandp.cuh has one (KAB_BAND_SERIAL_BT=1 keeps it: development /
  // comparison).  The maps kernel walks sum T * min(W, S) steps at ~1.85e12 steps/s (measured: the
  // 36-chapter book, 2.7e9 steps, 1.46 ms); the in-kernel walkers run side by side, 40 ns per frame of the
  // longest lattice.  So the parallel traceback is used when the plan is a few lattices or very unequal
  // ones (a book), not for dozens of equal ones.  KAB_BAND_SERIAL_BT=0 forces it.
  if (pl->lists[Q_BAND].empty() || bk == BandKernel::CTA) return;
  if (bk == BandKernel::P) {
    double steps = 0.0, tmax = 0.0;
    for (const KabLattice &d : pl->lists[Q_BAND]) {
      steps += (double)d.T * (double)std::min<int64_t>(s.W, 2 * (int64_t)d.L + 1);
      tmax = std::max(tmax, (double)d.T);
    }
    if (knob.serial_bt >= 0 ? knob.serial_bt != 0 : steps * 0.55e-12 > 0.6 * tmax * 40e-9) return;
  }
  for (const KabLattice &d : pl->lists[Q_BAND]) {
    KabBtMeta m{};
    m.map_off = pl->bt_map_ints;
    m.first_block = pl->bt_blocks;
    m.n_blocks = (d.T + KAB_BT_BLOCK - 1) / KAB_BT_BLOCK;
    m.wl = (int32_t)align_up(std::min<int64_t>(s.W, 2 * (int64_t)d.L + 1), 32);
    pl->bt_map_ints += (int64_t)m.n_blocks * KAB_BT_NSUB * m.wl;
    pl->bt_blocks += m.n_blocks;
    pl->bt_max_wl = std::max(pl->bt_max_wl, m.wl);
    pl->bt_meta.push_back(m);
  }
}

// pool_malloc (nothing for 0 bytes) and, given `src`, the upload of its bytes; a failure is cuda_fail(e, what)
int alloc(void **dst, size_t bytes, const char *what, const void *src = nullptr) {
  cudaError_t e = bytes ? pool_malloc(dst, bytes) : cudaSuccess;
  if (e == cudaSuccess && bytes && src) e = cudaMemcpy(*dst, src, bytes, cudaMemcpyHostToDevice);
  return e == cudaSuccess ? KAB_OK : cuda_fail(e, what);
}

cudaLaunchConfig_t launch_config(const Launch &k, cudaLaunchAttribute *at, cudaStream_t stream) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = k.grid; cfg.blockDim = k.block; cfg.dynamicSmemBytes = k.smem; cfg.stream = stream;
  cfg.attrs = at;
  cfg.numAttrs = k.cluster || k.cooperative ? 1 : 0;
  at[0].id = k.cluster ? cudaLaunchAttributeClusterDimension : cudaLaunchAttributeCooperative;
  if (k.cluster) at[0].val.clusterDim = {k.cluster, 1, 1};
  else at[0].val.cooperative = 1;
  return cfg;
}

// Launches a warp, band or wide list from its record.  The arguments are the kernel's parameters:
// (lattices, count, KabParams[, workspace: the wide kernel][, blank column: the CTC kernels]).
cudaError_t launch_list(const Launch &k, const KabLattice *lats, int n, KabParams p, unsigned char *const *wide_ws,
                        const int *blank, cudaStream_t stream) {
  void *args[5] = {&lats, &n, &p};
  int na = 3;
  if (wide_ws) args[na++] = (void *)wide_ws;
  if (blank) args[na++] = (void *)blank;
  cudaLaunchAttribute at[1];
  const cudaLaunchConfig_t cfg = launch_config(k, at, stream);
  return cudaLaunchKernelExC(&cfg, k.fn, args);
}

// ---- stage 6: device allocations and uploads; the launch records (kernel attributes and occupancy queries
// on the functions launched)
int Setup::allocate() {
  int rc = KAB_OK;
  cudaError_t e;
  for (int q = 0; q < N_QUEUES; ++q)
    if ((rc = alloc((void **)&pl->d_lists[q], pl->lists[q].size() * sizeof(KabLattice), "work list", pl->lists[q].data()))) return rc;
  if ((rc = alloc((void **)&pl->d_col16, col16.size() * sizeof(uint16_t), "column table", col16.data()))) return rc;
  if ((rc = alloc((void **)&pl->d_t_off, B > 0 ? (size_t)(B + 1) * sizeof(int64_t) : 0, "frame offsets", t_off))) return rc;
  if (pl->Vc) {
    if ((rc = alloc((void **)&pl->d_nonfinite, (size_t)B * sizeof(int32_t), "pool_malloc(non-finite flags)"))) return rc;
    if ((rc = alloc((void **)&pl->d_gather, gather_rows.size() * sizeof(int32_t), "gather rows", gather_rows.data()))) return rc;
    if ((rc = alloc((void **)&pl->d_lpc, (size_t)pl->total_T * pl->Vc * sizeof(float), "pool_malloc(compact log-probs)"))) return rc;
  }
  if (!pl->lists[Q_GENERIC].empty() && (rc = alloc((void **)&pl->d_raw, (size_t)pl->total_L * sizeof(int32_t), "labels", labels))) return rc;
  if (pl->any_bad_label && (rc = alloc((void **)&pl->d_status_init, (size_t)B * sizeof(int32_t), "statuses", status_init.data()))) return rc;
  if ((rc = alloc((void **)&pl->d_bp, (size_t)bp_bytes, "pool_malloc(backpointers)"))) return rc;
  if ((rc = alloc((void **)&pl->d_scratch, (size_t)scr_floats * 4, "pool_malloc(scratch)"))) return rc;
  if ((rc = alloc((void **)&pl->d_queue, N_QUEUES * sizeof(unsigned int), "pool_malloc(queue)"))) return rc;
  if (!pl->bt_meta.empty()) {
    if ((rc = alloc((void **)&pl->d_bt_meta, pl->bt_meta.size() * sizeof(KabBtMeta), "backtrack metadata", pl->bt_meta.data()))) return rc;
    if ((rc = alloc((void **)&pl->d_bt_maps, (size_t)pl->bt_map_ints * 4, "pool_malloc(backtrack maps)"))) return rc;
    if ((rc = alloc((void **)&pl->d_bt_entry, (size_t)pl->bt_blocks * 4, "pool_malloc(backtrack entries)"))) return rc;
    if ((rc = alloc((void **)&pl->d_end_state, (size_t)B * 4, "pool_malloc(end states)"))) return rc;
  }
  if ((rc = alloc((void **)&pl->d_band_fifo, (size_t)pl->band_fifo_bytes, "pool_malloc(band FIFOs)"))) return rc;
  if ((rc = alloc((void **)&pl->d_wide_ws, (size_t)pl->wide_ws_bytes, "pool_malloc(wide workspace)"))) return rc;
  if (!pl->lists[Q_WARP].empty()) {
    Launch &l = pl->launch[Q_WARP];
    l.fn = s.free_ends ? (const void *)kab_warp_ctc_free_kernel
         : s.ctc ? (const void *)kab_warp_ctc_kernel
         : s.M == 4 ? (Veff == 39 ? (const void *)kab_warp_kernel<39, false> : (const void *)kab_warp_kernel<0, false>)
                    : (Veff == 39 ? (const void *)kab_warp_kernel<39, true> : (const void *)kab_warp_kernel<0, true>);
    l.block = dim3(KAB_WARPS_PER_CTA * 32);
    l.smem = 128 + (size_t)KAB_WARPS_PER_CTA * (KAB_WARP_STAGES * pl->stage_bytes + 256);  // + label tables
    if ((e = ensure_dyn_smem(l.fn, pl->device, l.smem)) != cudaSuccess) return cuda_fail(e, "cudaFuncSetAttribute(warp)");
    int occ = 0;
    if ((e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, l.fn, l.block.x, l.smem)) != cudaSuccess) return cuda_fail(e, "occupancy(warp)");
    const int64_t ctas = ((int64_t)pl->lists[Q_WARP].size() + KAB_WARPS_PER_CTA - 1) / KAB_WARPS_PER_CTA;
    occ = std::min(occ, KAB_WARP_MINBLOCKS);
    if (knob.warp_ctas_per_sm >= 1) occ = std::min(occ, knob.warp_ctas_per_sm);
    l.grid = dim3((unsigned)std::min<int64_t>(ctas, (int64_t)pl->sm_count * std::max(occ, 1)));
  }
  if (!pl->lists[Q_BAND].empty()) {
    Launch &l = pl->launch[Q_BAND];
    const BandKernel bk = pl->band_kernel;
    const int64_t n_band = (int64_t)pl->lists[Q_BAND].size();
    const bool mm = s.M != 4, small = pl->band_nw <= 16;
    l.fn = bk == BandKernel::P ? (const void *)kab_bandp_kernel
         : bk == BandKernel::Q ? (const void *)kab_bandq_kernel
         : bk == BandKernel::R ? (mm ? (const void *)kab_bandr_kernel<true> : (const void *)kab_bandr_kernel<false>)
         : bk == BandKernel::R_GATHER ? (mm ? (const void *)kab_bandr_kernel<true, true> : (const void *)kab_bandr_kernel<false, true>)
         : s.free_ends ? (small ? (const void *)kab_band_ctc_free_kernel<512> : (const void *)kab_band_ctc_free_kernel<1024>)
         : s.ctc ? (small ? (const void *)kab_band_ctc_kernel<512> : (const void *)kab_band_ctc_kernel<1024>)
         : small ? (mm ? (const void *)kab_band_kernel<512, true> : (const void *)kab_band_kernel<512, false>)
                 : (mm ? (const void *)kab_band_kernel<1024, true> : (const void *)kab_band_kernel<1024, false>);
    const bool ga = bk == BandKernel::R_GATHER;  // (no emission stages: the geometry's minimum)
    l.stage_frames = ga ? KAB_BR_F : pl->stage_frames;
    l.stage_bytes = ga ? 64 : pl->stage_bytes;
    if (bk == BandKernel::CTA) {
      l.block = dim3(pl->band_nw * 32);
      l.smem = kab_band_geom(pl->band_nw, pl->stage_bytes).smem_bytes;
      int occ = 0;
      if ((e = ensure_dyn_smem(l.fn, pl->device, l.smem)) != cudaSuccess) return cuda_fail(e, "cudaFuncSetAttribute(band)");
      if ((e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, l.fn, l.block.x, l.smem)) != cudaSuccess) return cuda_fail(e, "occupancy(band)");
      l.grid = dim3((unsigned)std::min<int64_t>(n_band, (int64_t)(pl->sm_count - pl->band_sm_reserved) * std::max(occ, 1)));
    } else {
      const bool r = bk == BandKernel::R || bk == BandKernel::R_GATHER;
      l.block = dim3(r ? KAB_BR_THREADS : (bk == BandKernel::Q ? KAB_BQ_THREADS : KAB_BP_THREADS));
      l.smem = r ? kab_bandr_geom(l.stage_bytes).smem_bytes
                 : (bk == BandKernel::Q ? kab_bandq_geom(l.stage_bytes).smem_bytes : kab_bandp_geom(l.stage_bytes).smem_bytes);
      l.cluster = (unsigned)pl->band_nc;
      if ((e = ensure_dyn_smem(l.fn, pl->device, l.smem)) != cudaSuccess) return cuda_fail(e, "cudaFuncSetAttribute(cluster band)");
      l.grid = dim3((unsigned)(pl->band_nc * pl->sm_count));
      cudaLaunchAttribute at[1];
      const cudaLaunchConfig_t cfg = launch_config(l, at, nullptr);
      int ncl = 0;
      if ((e = cudaOccupancyMaxActiveClusters(&ncl, l.fn, &cfg)) != cudaSuccess) return cuda_fail(e, "cudaOccupancyMaxActiveClusters(cluster band)");
      l.grid = dim3((unsigned)(std::min<int64_t>(std::max(ncl, 1), n_band) * pl->band_nc));
    }
  }
  if (!pl->lists[Q_WIDE].empty()) pl->launch[Q_WIDE].grid = dim3((unsigned)(wide_max_ctas + 1));  // forward CTAs + the backtrack CTA
  if (!pl->lists[Q_GENERIC].empty())
    pl->launch[Q_GENERIC].grid = dim3((unsigned)std::min<int64_t>((int64_t)pl->lists[Q_GENERIC].size(), (int64_t)pl->sm_count * 4));
  return KAB_OK;
}

// ---- stage 7: the plan's info, and the sub-plan of a hybrid band plan
int Setup::finish() {
  kab_plan_info &info = pl->info;
  info.backptr_bytes = bp_bytes;
  info.workspace_bytes = bp_bytes + scr_floats * 4 + pl->wide_ws_bytes + pl->band_fifo_bytes + (int64_t)col16.size() * 2 +
                         (pl->d_raw ? pl->total_L * 4 : 0) + B * (int64_t)sizeof(KabLattice);
  info.kernel_launches = 0;
  for (int q = 0; q < N_QUEUES; ++q) info.kernel_launches += pl->lists[q].empty() ? 0 : 1;
  const BandKernel bk = pl->band_kernel;
  if (!pl->lists[Q_BAND].empty()) {
    const int32_t code[] = {KAB_BAND_KERNEL_CTA, KAB_BAND_KERNEL_CLUSTER, KAB_BAND_KERNEL_CLUSTER2, KAB_BAND_KERNEL_SPEC, KAB_BAND_KERNEL_SPEC};
    info.band_kernel = code[(int)bk];  // (in BandKernel's order)
    info.band_cluster = pl->band_nc > 0 ? pl->band_nc : 1;
  }
  if (!pl->bt_meta.empty()) info.kernel_launches += 3;                      // kab_bt_maps_kernel, kab_bt_stitch_kernel, kab_bt_gather_kernel
  if (bk == BandKernel::R || bk == BandKernel::R_GATHER) info.kernel_launches += 1;  // kab_finite_rows_kernel
  if (pl->Vc)                                                               // kab_compact_kernel (CTC: _ctc_), kab_expand_labels_kernel
    for (int q : {Q_WARP, Q_BAND, Q_WIDE}) info.kernel_launches += pl->lists[q].empty() ? 0 : 2;
  if (hyb_k == 0) return KAB_OK;
  // the sub-plan of a hybrid band plan: same arrays, its own lattices, workspaces and stream
  if (int rc = plan_create_impl(&pl->sub, pl->device, s, B, t_off, labels, l_off, hyb_mask.data(), 1)) return rc;
  pl->sub->is_child = true;
  pl->sub->launch[Q_BAND].grid.x = std::min(pl->sub->launch[Q_BAND].grid.x, (unsigned)(hyb_k * pl->sub->band_nc));
  cudaError_t e = pool_malloc((void **)&pl->sub->d_started, sizeof(unsigned int));
  if (e == cudaSuccess) e = cudaMemset(pl->sub->d_started, 0, sizeof(unsigned int));
  if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&pl->s_sub, cudaStreamNonBlocking);
  if (e == cudaSuccess) e = cudaEventCreateWithFlags(&pl->ev_fork, cudaEventDisableTiming);
  if (e == cudaSuccess) e = cudaEventCreateWithFlags(&pl->ev_join, cudaEventDisableTiming);
  if (e != cudaSuccess) return cuda_fail(e, "stream / events of the hybrid band plan");
  info.band_kernel = KAB_BAND_KERNEL_HYBRID;
  info.band_cluster = pl->sub->band_nc;
  info.backptr_bytes += pl->sub->info.backptr_bytes;
  info.workspace_bytes += pl->sub->info.workspace_bytes;
  info.kernel_launches += pl->sub->info.kernel_launches;
  return KAB_OK;
}

int plan_create_impl(kab_plan **out, int device, const PlanSpec &s, int64_t B, const int64_t *t_off,
                     const int32_t *labels, const int64_t *l_off, const uint8_t *mask, int band_mode) {
  if (!out || B < 0 || !t_off || !l_off || s.V < 1 || s.V > 65535 || s.W < 0 || s.M < 1 || s.M > 255) return KAB_E_BAD_ARG;
  if (B > 0 && (t_off[0] < 0 || l_off[0] < 0)) return KAB_E_BAD_ARG;
  if (B > 0 && l_off[B] > l_off[0] && !labels) return KAB_E_BAD_ARG;
  for (int64_t b = 0; b < B; ++b) {
    const int64_t T = t_off[b + 1] - t_off[b], L = l_off[b + 1] - l_off[b];
    if (T < 1 || T > 0x3fffffff || L < 0 || L > 0x3ffffff0) return KAB_E_BAD_ARG;
  }
  DeviceGuard guard;
  KAB_CUDA(guard.enter(device));
  kab_plan *pl = new (std::nothrow) kab_plan();
  if (!pl) return KAB_E_NOMEM;
  pl->device = device; pl->B = B; pl->spec = s;
  pl->total_T = B ? t_off[B] : 0;  // offsets are absolute rows / entries of the caller's arrays
  pl->total_L = B ? l_off[B] : 0;
  if (B > 0) {
    pl->h_t_off.assign(t_off, t_off + B + 1);
    pl->h_l_off.assign(l_off, l_off + B + 1);
    if (pl->total_L > 0) pl->h_labels.assign(labels, labels + pl->total_L);
  }
  Trace tr("kab_plan_create");
  if (int rcs = sm_count_of(device, &pl->sm_count)) { delete pl; return rcs; }
  pl->info.n_lattices = B; pl->info.device = device; pl->info.total_frames = pl->total_T;

  Setup x{pl, s, Knobs::read(), B, t_off, l_off, labels, mask};
  x.scan_labels();
  x.compact_vocabulary();
  x.classify();
  x.choose_band_kernel(band_mode);
  x.lay_out_band();
  tr.mark("classify");
  int rc = x.allocate();
  tr.mark("allocate, upload, kernel attributes");
  if (rc == KAB_OK) rc = x.finish();
  if (rc != KAB_OK) { plan_free(pl); return rc; }
  *out = pl;
  return KAB_OK;
}
}  // namespace

int kab_plan_get_info(const kab_plan *pl, kab_plan_info *info) {
  if (!pl || !info) return KAB_E_BAD_ARG;
  *info = pl->info;
  return KAB_OK;
}

int kab_plan_destroy(kab_plan *pl) { return plan_free(pl); }

int kab_plan_run_device(kab_plan *pl, const float *d_log_probs, int32_t *d_best_path, int32_t *d_best_labels,
                        float *d_best_scores, float *d_final_score, int32_t *d_status, void *stream_) {
  if (!pl) return KAB_E_BAD_ARG;
  if (pl->B == 0) return KAB_OK;
  if (!d_log_probs || !d_best_path || !d_best_labels || !d_best_scores || !d_status) return KAB_E_BAD_ARG;
  if (reinterpret_cast<uintptr_t>(d_log_probs) & 15) return KAB_E_BAD_ARG;  // bulk copies need 16-byte alignment
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  DeviceGuard guard;
  KAB_CUDA(guard.enter(pl->device));
  const PlanSpec &s = pl->spec;
  KabParams p{};
  p.lp = d_log_probs;
  p.lp_bytes = pl->total_T * (int64_t)s.V * 4;
  p.col16 = pl->d_col16; p.raw = pl->d_raw; p.bp = pl->d_bp; p.scratch = pl->d_scratch;
  p.best_path = d_best_path; p.best_labels = d_best_labels; p.best_scores = d_best_scores;
  p.final_score = d_final_score; p.status = d_status;
  p.V = s.V; p.W = s.W; p.M = s.M;
  p.stage_frames = pl->stage_frames; p.stage_bytes = pl->stage_bytes;
  p.one = 1u;
  p.started = pl->d_started;
  {  // max_move < 4: the excluded moves' candidates become -inf (kab_mm)
    const float ninf = -std::numeric_limits<float>::infinity();
    p.mm1 = s.M >= 2 ? 0.0f : ninf; p.mm2 = s.M >= 3 ? 0.0f : ninf; p.mm3 = s.M >= 4 ? 0.0f : ninf;
  }
  p.band_nw = pl->band_nw;

  // the staged kernels' view of the log-probs: the caller's array, or its compact copy (not the gather mode's)
  KabParams pf = p;
  const BandKernel bk = pl->band_kernel;
  auto on_copy = [&](int q) { return !pl->lists[q].empty() && !(q == Q_BAND && bk == BandKernel::R_GATHER); };
  if (pl->Vc) {
    KAB_CUDA(cudaMemsetAsync(pl->d_nonfinite, 0, (size_t)pl->B * sizeof(int32_t), stream));
    for (int q : {Q_WARP, Q_BAND, Q_WIDE})
      if (on_copy(q)) {
        const dim3 grid((unsigned)pl->lists[q].size(), (unsigned)((pl->max_T[q] + KAB_COMPACT_FRAMES - 1) / KAB_COMPACT_FRAMES));
        (s.ctc ? kab_compact_ctc_kernel : kab_compact_kernel)<<<grid, 256, 0, stream>>>(pl->d_lists[q], d_log_probs, pl->d_lpc,
                                                                                          pl->d_gather, s.V, pl->Vc, pl->d_nonfinite);
      }
    pf.lp = pl->d_lpc; pf.V = pl->Vc; pf.lp_bytes = pl->total_T * (int64_t)pl->Vc * 4;
  }
  // CTC: the blank's column in the staged kernels' view (compact column 0 of the copy); the generic kernel
  // reads the caller's array and keeps the blank id
  const int sblank = pl->Vc ? 0 : s.blank;
  const int *blank_arg = s.ctc ? &sblank : nullptr;

  if (pl->sub) {  // hybrid band plan: the long lattices first (their clusters need whole SMs), on the side stream
    KAB_CUDA(cudaEventRecord(pl->ev_fork, stream));
    KAB_CUDA(cudaStreamWaitEvent(pl->s_sub, pl->ev_fork, 0));
    if (int rcs = kab_plan_run_device(pl->sub, d_log_probs, d_best_path, d_best_labels, d_best_scores, d_final_score, d_status, pl->s_sub))
      return rcs;
    KAB_CUDA(cudaEventRecord(pl->ev_join, pl->s_sub));
    // the single-CTA kernel below would otherwise spread one CTA over every SM before the clusters
    // (which need whole SMs) are placed, and the two kernels would run one after the other
    pl->sub->gate_target += pl->sub->launch[Q_BAND].grid.x;
    if (!pl->lists[Q_BAND].empty()) kab_gate_kernel<<<1, 32, 0, stream>>>(pl->sub->d_started, pl->sub->gate_target);
  }
  KAB_CUDA(cudaMemsetAsync(pl->d_queue, 0, N_QUEUES * sizeof(unsigned int), stream));
  if (pl->any_bad_label)
    KAB_CUDA(cudaMemcpyAsync(d_status, pl->d_status_init, (size_t)pl->B * sizeof(int32_t), cudaMemcpyDeviceToDevice, stream));

  if (!pl->lists[Q_WARP].empty()) {
    KabParams pw = pf; pw.queue = pl->d_queue + Q_WARP;
    KAB_CUDA(launch_list(pl->launch[Q_WARP], pl->d_lists[Q_WARP], (int)pl->lists[Q_WARP].size(), pw, nullptr, blank_arg, stream));
  }
  if (!pl->lists[Q_BAND].empty()) {
    const Launch &lb = pl->launch[Q_BAND];
    KabParams pb = bk == BandKernel::R_GATHER ? p : pf;
    pb.queue = pl->d_queue + Q_BAND; pb.stage_frames = lb.stage_frames; pb.stage_bytes = lb.stage_bytes;
    pb.fifo = pl->d_band_fifo; pb.end_state = pl->d_end_state;  // (end_state nullptr: the kernel walks back itself)
    const int n_band = (int)pl->lists[Q_BAND].size(), nwt = pl->band_cw * pl->band_nc;
    std::optional<KabBandTiming> t_cta; std::optional<KabBandpTiming> t_p; std::optional<KabBandqTiming> t_q; std::optional<KabBandrTiming> t_r;
    if (bk == BandKernel::CTA) t_cta.emplace(pb, stream, pl->band_nw);  // (development builds only: kab_debug.h)
    else if (bk == BandKernel::P) t_p.emplace(pb, stream, nwt);
    else if (bk == BandKernel::Q) t_q.emplace(pb, stream, nwt);
    else t_r.emplace(pb, stream, nwt);
    if (bk == BandKernel::P || bk == BandKernel::Q)  // (bandr: mailboxes in shared memory)
      KAB_CUDA(cudaMemsetAsync(pl->d_band_fifo, 0, (size_t)pl->band_fifo_bytes, stream));
    KAB_CUDA(launch_list(lb, pl->d_lists[Q_BAND], n_band, pb, nullptr, blank_arg, stream));
    if (bk == BandKernel::R || bk == BandKernel::R_GATHER) {
      const dim3 fg((unsigned)n_band, (unsigned)((pl->max_T[Q_BAND] + KAB_FIN_ROWS - 1) / KAB_FIN_ROWS));
      kab_finite_rows_kernel<<<fg, 256, 0, stream>>>(pl->d_lists[Q_BAND], pb.lp, pb.V, d_status, d_final_score);
    }
    if (pl->d_end_state) {  // the parallel backtrack (kab_btpar.cuh)
      const dim3 mg((unsigned)pl->bt_blocks, (unsigned)((pl->bt_max_wl + KAB_BT_THREADS - 1) / KAB_BT_THREADS));
      auto maps_stitch = [&](auto layout) {
        using Layout = decltype(layout);
        kab_bt_maps_kernel<Layout><<<mg, KAB_BT_THREADS, 0, stream>>>(pl->d_lists[Q_BAND], pl->d_bt_meta, n_band, pl->d_bp, d_status,
                                                                      pl->d_bt_maps, s.W, nwt);
        kab_bt_stitch_kernel<Layout><<<n_band, 1024, 0, stream>>>(pl->d_lists[Q_BAND], pl->d_bt_meta, pb, pl->d_end_state,
                                                                  pl->d_bt_maps, pl->d_bt_entry, nwt);
      };
      if (band_layout_q(bk)) maps_stitch(KabBtLayoutQ{}); else maps_stitch(KabBtLayoutP{});
      const dim3 gg((unsigned)n_band, (unsigned)((pl->max_T[Q_BAND] + KAB_BT_GATHER_FRAMES - 1) / KAB_BT_GATHER_FRAMES));
      kab_bt_gather_kernel<<<gg, 256, 0, stream>>>(pl->d_lists[Q_BAND], pb);
    }
  }
  if (!pl->lists[Q_WIDE].empty()) {
    KAB_CUDA(cudaMemsetAsync(pl->d_wide_ws, 0, (size_t)pl->wide_ws_bytes, stream));
    KabWideTiming wide_timing(pf, stream);
    // cooperative launch: the warps of the chain spin on each other, so the whole grid has to be
    // resident -- the runtime checks that instead of letting the kernel hang
    KAB_CUDA(launch_list(pl->launch[Q_WIDE], pl->d_lists[Q_WIDE], (int)pl->lists[Q_WIDE].size(), pf, &pl->d_wide_ws, blank_arg, stream));
  }
  if (pl->Vc)  // best_labels of the staged kernels: compact index -> label value
    for (int q : {Q_WARP, Q_BAND, Q_WIDE})
      if (on_copy(q)) {
        const dim3 grid((unsigned)pl->lists[q].size(), (unsigned)((pl->max_T[q] + KAB_COMPACT_FRAMES - 1) / KAB_COMPACT_FRAMES));
        kab_expand_labels_kernel<<<grid, 64, 0, stream>>>(pl->d_lists[q], d_best_labels, d_status, d_final_score,
                                                          pl->d_gather, pl->Vc, pl->d_nonfinite);
      }
  if (!pl->lists[Q_GENERIC].empty()) {
    KabParams pg = p; pg.queue = pl->d_queue + Q_GENERIC;
    if (s.free_ends)
      kab_generic_ctc_free_kernel<GENERIC_NT><<<pl->launch[Q_GENERIC].grid, GENERIC_NT, 0, stream>>>(
          pl->d_lists[Q_GENERIC], (int)pl->lists[Q_GENERIC].size(), pg, s.blank);
    else if (s.ctc)
      kab_generic_ctc_kernel<GENERIC_NT><<<pl->launch[Q_GENERIC].grid, GENERIC_NT, 0, stream>>>(
          pl->d_lists[Q_GENERIC], (int)pl->lists[Q_GENERIC].size(), pg, s.blank);
    else
      kab_generic_kernel<GENERIC_NT><<<pl->launch[Q_GENERIC].grid, GENERIC_NT, 0, stream>>>(
          pl->d_lists[Q_GENERIC], (int)pl->lists[Q_GENERIC].size(), pg);
  }
  KAB_CUDA(cudaGetLastError());
  if (pl->sub) KAB_CUDA(cudaStreamWaitEvent(stream, pl->ev_join, 0));
  return record_run_event(pl, stream);
}

int kab_log_softmax_device(const float *d_logits, float *d_log_probs, int64_t n_rows, int32_t V, void *stream_) {
  if (n_rows < 0 || V < 1) return KAB_E_BAD_ARG;
  if (n_rows == 0) return KAB_OK;
  if (!d_logits || !d_log_probs) return KAB_E_BAD_ARG;
  cudaStream_t stream = (cudaStream_t)stream_;
  int dev = 0, sms = 0;
  KAB_CUDA(cudaGetDevice(&dev));
  KAB_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  if (V <= KAB_SM_MAX_V) {
    const size_t smem = (size_t)KAB_SM_ROWS * (V | 1) * sizeof(float);
    const int64_t n_tiles = (n_rows + KAB_SM_ROWS - 1) / KAB_SM_ROWS;
    const int per_sm = (int)std::max<size_t>(1, std::min<size_t>(8, (200 * 1024) / (smem + 1024)));
    const unsigned grid = (unsigned)std::min<int64_t>(n_tiles, (int64_t)sms * per_sm);
    const int vec_ok = ((uintptr_t)d_logits % 16 == 0 && (uintptr_t)d_log_probs % 16 == 0) ? 1 : 0;
    static const bool no_tma = getenv("KAB_SOFTMAX_NO_TMA") != nullptr;  // development knob
    if (V == 39 && vec_ok && !no_tma) {
      // full tiles through the bulk-copy pipeline (one persistent CTA per SM), the tail below
      const int64_t n_full = n_rows / KAB_SM_ROWS;
      if (n_full > 0) {
        const size_t smem_t = 128 + (size_t)KAB_SMT_BUFS * KAB_SM_ROWS * 39 * sizeof(float);
        KAB_CUDA(ensure_dyn_smem((const void *)kab_log_softmax_tma_kernel<39>, dev, smem_t));
        kab_log_softmax_tma_kernel<39><<<(unsigned)std::min<int64_t>(n_full, sms), KAB_SM_ROWS, smem_t, stream>>>(
            d_logits, d_log_probs, n_full);
      }
      const int64_t tail = n_rows - n_full * KAB_SM_ROWS;
      if (tail > 0) {
        KAB_CUDA(ensure_dyn_smem((const void *)kab_log_softmax_kernel<39>, dev, smem));
        kab_log_softmax_kernel<39><<<1, KAB_SM_ROWS, smem, stream>>>(d_logits + n_full * KAB_SM_ROWS * 39,
                                                                      d_log_probs + n_full * KAB_SM_ROWS * 39, tail, V, 1);
      }
    } else if (V == 39) {
      KAB_CUDA(ensure_dyn_smem((const void *)kab_log_softmax_kernel<39>, dev, smem));
      kab_log_softmax_kernel<39><<<grid, KAB_SM_ROWS, smem, stream>>>(d_logits, d_log_probs, n_rows, V, vec_ok);
    } else {
      KAB_CUDA(ensure_dyn_smem((const void *)kab_log_softmax_kernel<0>, dev, smem));
      kab_log_softmax_kernel<0><<<grid, KAB_SM_ROWS, smem, stream>>>(d_logits, d_log_probs, n_rows, V, vec_ok);
    }
  } else {
    const unsigned grid = (unsigned)std::min<int64_t>((n_rows + 7) / 8, (int64_t)sms * 8);
    kab_log_softmax_wide_kernel<<<grid, 256, 0, stream>>>(d_logits, d_log_probs, n_rows, V);
  }
  KAB_CUDA(cudaGetLastError());
  return KAB_OK;
}

namespace {
// ---- CTC posteriors (kab_posterior.cuh): three block sizes, chosen per lattice by its pair slots per frame
constexpr int POST_NT[3] = {64, 256, 1024};
inline int post_class(int64_t np) { return np <= 128 ? 0 : np <= 1024 ? 1 : 2; }
inline int64_t post_window(const kab_plan *pl, int64_t b) {
  return std::min<int64_t>(pl->spec.W, 2 * (pl->h_l_off[b + 1] - pl->h_l_off[b]) + 1);
}
// an unbanded lattice of a long-form plan (not free ends) above the single-CTA limit: the chain pass
inline bool post_chained(const kab_plan *pl, int64_t b) {
  const PlanSpec &s = pl->spec;
  return s.ctc_long && !s.free_ends && s.W == CTC_W && 2 * (pl->h_l_off[b + 1] - pl->h_l_off[b]) + 1 > pl->post_chain_min;
}
inline size_t post_smem(int32_t e_words, int32_t p_words, int32_t bufcap) {
  return 8 * KAB_POST_NST + 16 + (size_t)KAB_POST_NST * (e_words + p_words) * 4 + (size_t)2 * bufcap * 4;
}

// The first kab_plan_ctc_posteriors_device of a plan: the labels with their move-2 bits, the lattice lists and
// their launches, the value rows.  Emission rows are staged while the ring fits next to the state buffers.
int post_setup(kab_plan *pl) {
  const int64_t B = pl->B, V = pl->spec.V;
  const std::vector<int64_t> &to = pl->h_t_off, &lo = pl->h_l_off;
  const std::vector<int32_t> &lab = pl->h_labels;
  std::vector<int32_t> labs((size_t)pl->total_L, 0);
  for (int64_t b = 0; b < B; ++b)
    for (int64_t l = lo[b]; l < lo[b + 1]; ++l) {
      const bool in = l > lo[b] && lab[l] != lab[l - 1], out = l + 1 < lo[b + 1] && lab[l + 1] != lab[l];
      labs[l] = (int32_t)((uint32_t)(lab[l] & 0xffff) | (uint32_t)in << 31 | (uint32_t)out << 30);
    }
  std::vector<KabPostLat> lists[3];
  std::vector<KabPostChainLat> chain;
  int nw_max = 0;
  for (int64_t b = 0; b < B; ++b) {
    const int64_t T = to[b + 1] - to[b], S = 2 * (lo[b + 1] - lo[b]) + 1;
    if (post_chained(pl, b)) {
      const int nw = (int)((S + 1) / 2 + KAB_PC_PAIRS - 1) / KAB_PC_PAIRS;
      chain.push_back(KabPostChainLat{to[b], lo[b], pl->post_chain_ws_bytes, (int32_t)T, (int32_t)S, (int32_t)b, nw});
      pl->post_chain_ws_bytes += (int64_t)align_up((int64_t)kab_pc_ws_bytes(nw), 256);
      nw_max = std::max(nw_max, nw);
      continue;
    }
    const int64_t np = post_window(pl, b) / 2 + 2;
    lists[post_class(np)].push_back(KabPostLat{to[b], lo[b], (int32_t)T, (int32_t)S, (int32_t)b, (int32_t)np,
                                               unbanded(T, S, pl->spec.W) ? 0 : 1});
  }
  pl->post_F = (int32_t)std::max<int64_t>(1, std::min<int64_t>(16, 1024 / (4 * V)));
  pl->post_p_words = (int32_t)(align_up(pl->post_F * 4, 16) + 32) / 4;
  const int32_t e_words = (int32_t)((align_up(pl->post_F * V * 4, 16) + 32) / 4);
  int rc;
  for (int c = 0; c < 3; ++c) {
    std::vector<KabPostLat> &v = lists[c];
    kab_plan::PostList &pc = pl->post[c];
    pc.n = (int)v.size();
    if (v.empty()) continue;
    std::sort(v.begin(), v.end(), [](const KabPostLat &x, const KabPostLat &y) {
      return (int64_t)x.T * x.np > (int64_t)y.T * y.np;
    });
    int64_t np_max = 0;
    for (const KabPostLat &x : v) np_max = std::max<int64_t>(np_max, x.np);
    pc.bufcap = (int32_t)align_up(KAB_POST_PAD + 2 * np_max + KAB_POST_TAIL, 4);
    pc.e_words = post_smem(e_words, pl->post_p_words, pc.bufcap) <= 227 * 1024 ? e_words : 0;
    Launch &l = pc.launch;
    l.fn = c == 0 ? (const void *)kab_ctc_posterior_kernel<POST_NT[0]>
         : c == 1 ? (const void *)kab_ctc_posterior_kernel<POST_NT[1]> : (const void *)kab_ctc_posterior_kernel<POST_NT[2]>;
    l.grid = dim3((unsigned)(2 * v.size()));
    l.block = dim3(POST_NT[c]);
    l.smem = post_smem(pc.e_words, pl->post_p_words, pc.bufcap);
    cudaError_t e = ensure_dyn_smem(l.fn, pl->device, l.smem);
    if (e != cudaSuccess) return cuda_fail(e, "cudaFuncSetAttribute(posteriors)");
    if ((rc = alloc((void **)&pc.d_lats, v.size() * sizeof(KabPostLat), "posterior lattices", v.data()))) return rc;
  }
  if (!chain.empty()) {
    // every warp of the chain spins on its neighbours: the whole grid must be resident (a cooperative launch
    // refuses rather than hangs); both directions side by side when they fit, else one after the other
    Launch &l = pl->post_chain;
    l.fn = (const void *)kab_ctc_posterior_chain_kernel;
    l.block = dim3(KAB_PC_CW * 32);
    l.cooperative = true;
    int occ = 0;
    cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, l.fn, KAB_PC_CW * 32, 0);
    if (e != cudaSuccess) return cuda_fail(e, "occupancy(posterior chain)");
    const int64_t capacity = (int64_t)occ * pl->sm_count, ctas = (nw_max + KAB_PC_CW - 1) / KAB_PC_CW;
    const bool serial = getenv("KAB_POSTERIOR_CHAIN_SERIAL") != nullptr;  // test knob: one direction at a time
    if (ctas > capacity) return KAB_E_UNSUPPORTED;
    const bool side = 2 * ctas <= capacity && !serial;
    pl->post_chain_split = side ? (int)ctas * KAB_PC_CW : 0;
    l.grid = dim3((unsigned)(side ? 2 * ctas : ctas));
    pl->post_chain_n = (int)chain.size();
    if ((rc = alloc((void **)&pl->d_post_chain, chain.size() * sizeof(KabPostChainLat), "posterior chain lattices", chain.data())))
      return rc;
    if ((rc = alloc((void **)&pl->d_post_chain_ws, (size_t)pl->post_chain_ws_bytes, "pool_malloc(posterior chain workspace)")))
      return rc;
  }
  if ((rc = alloc((void **)&pl->d_post_labs, labs.size() * sizeof(int32_t), "posterior labels", labs.data()))) return rc;
  if ((rc = alloc((void **)&pl->d_post_scr, (size_t)2 * std::max<int64_t>(pl->total_T, 1) * sizeof(double), "pool_malloc(posterior values)")))
    return rc;
  pl->post_ready = true;
  return KAB_OK;
}
}  // namespace

int kab_plan_ctc_posteriors_device(kab_plan *pl, const float *d_log_probs, const int32_t *d_best_path,
                                   const int32_t *d_status, double *d_log_likelihood, float *d_posteriors,
                                   void *stream_) {
  if (!pl) return KAB_E_BAD_ARG;
  if (!pl->spec.ctc || pl->spec.free_ends) return KAB_E_UNSUPPORTED;
  if (!pl->post_ready) {  // test knob: move lattices with more states than this to the chain pass
    const char *knob = getenv("KAB_POSTERIOR_CHAIN_MIN_STATES");
    pl->post_chain_min = knob ? std::min<int64_t>(atoll(knob), KAB_POSTERIOR_MAX_STATES) : KAB_POSTERIOR_MAX_STATES;
  }
  for (int64_t b = 0; b < pl->B; ++b)
    if (post_chained(pl, b) ? 2 * (pl->h_l_off[b + 1] - pl->h_l_off[b]) + 1 > KAB_POSTERIOR_LONG_MAX_STATES
                            : post_window(pl, b) > KAB_POSTERIOR_MAX_STATES)
      return KAB_E_UNSUPPORTED;
  if (pl->B == 0) return KAB_OK;
  if (!d_log_probs || !d_best_path || !d_status || !d_log_likelihood || !d_posteriors) return KAB_E_BAD_ARG;
  if ((reinterpret_cast<uintptr_t>(d_log_probs) & 15) || (reinterpret_cast<uintptr_t>(d_best_path) & 3)) return KAB_E_BAD_ARG;
  cudaStream_t stream = reinterpret_cast<cudaStream_t>(stream_);
  DeviceGuard guard;
  KAB_CUDA(guard.enter(pl->device));
  if (!pl->post_ready)
    if (int rc = post_setup(pl)) { cleanup_post(pl); return rc; }
  const uintptr_t pa = reinterpret_cast<uintptr_t>(d_best_path);
  KabPostParams p{};
  p.lp = d_log_probs; p.lp_bytes = pl->total_T * (int64_t)pl->spec.V * 4;
  p.path_skew = (int32_t)((pa & 15) >> 2);
  p.path = reinterpret_cast<const int32_t *>(pa & ~(uintptr_t)15);
  p.path_bytes = (pl->total_T + p.path_skew) * 4;
  p.labs = pl->d_post_labs; p.status = d_status;
  p.fwd = pl->d_post_scr; p.bwd = pl->d_post_scr + std::max<int64_t>(pl->total_T, 1);
  p.log_likelihood = d_log_likelihood;
  p.W = pl->spec.W; p.V = pl->spec.V; p.blank = pl->spec.blank;
  p.F = pl->post_F; p.p_words = pl->post_p_words;
  for (const kab_plan::PostList &pc : pl->post) {
    if (!pc.n) continue;
    KabPostParams q = p;
    q.e_words = pc.e_words; q.bufcap = pc.bufcap;
    const KabPostLat *lats = pc.d_lats;
    void *args[2] = {&lats, &q};
    KAB_CUDA(cudaLaunchKernel(pc.launch.fn, pc.launch.grid, pc.launch.block, args, pc.launch.smem, stream));
  }
  if (pl->post_chain_n) {
    KAB_CUDA(cudaMemsetAsync(pl->d_post_chain_ws, 0, (size_t)pl->post_chain_ws_bytes, stream));
    const KabPostChainLat *lats = pl->d_post_chain;
    int n = pl->post_chain_n, split = pl->post_chain_split;
    unsigned char *ws = pl->d_post_chain_ws;
    void *args[5] = {&lats, &n, &p, &ws, &split};
    cudaLaunchAttribute at[1];
    const cudaLaunchConfig_t cfg = launch_config(pl->post_chain, at, stream);
    KAB_CUDA(cudaLaunchKernelExC(&cfg, pl->post_chain.fn, args));
  }
  const unsigned grid = (unsigned)std::min<int64_t>((pl->total_T + 255) / 256, (int64_t)pl->sm_count * 8);
  if (grid > 0)
    kab_ctc_posterior_combine_kernel<<<grid, 256, 0, stream>>>(pl->d_t_off, pl->B, pl->total_T, d_status, p.fwd, p.bwd,
                                                               d_log_likelihood, d_posteriors);
  KAB_CUDA(cudaGetLastError());
  return record_run_event(pl, stream);
}

namespace {
// one CTA per item, at most this many CTAs per SM in the grid (the kernels grid-stride over the rest)
int span_grid(int64_t n_items, int *grid) {
  int dev = 0, sms = 0;
  KAB_CUDA(cudaGetDevice(&dev));
  KAB_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  *grid = (int)std::min<int64_t>(n_items, (int64_t)sms * 32);
  return KAB_OK;
}
}  // namespace

int kab_merge_tokens_device(int64_t n_items, const int64_t *d_t_off, const int32_t *d_tokens, const float *d_scores,
                            int32_t blank, kab_token_span *d_spans, int32_t *d_n_spans, void *stream) {
  if (n_items < 0 || !d_t_off || !d_tokens || !d_scores || !d_spans || !d_n_spans) return KAB_E_BAD_ARG;
  int grid = 0, rc;
  if ((rc = span_grid(n_items, &grid)) != KAB_OK || n_items == 0) return rc;
  const int vec = (uintptr_t)d_spans % 16 == 0;
  kab_merge_tokens_kernel<<<grid, KAB_SPAN_THREADS, 0, (cudaStream_t)stream>>>(
      n_items, d_t_off, d_tokens, d_scores, blank, reinterpret_cast<KabTokenSpan *>(d_spans), d_n_spans, vec);
  KAB_CUDA(cudaGetLastError());
  return KAB_OK;
}

int kab_word_spans_device(int64_t n_items, const int64_t *d_t_off, const kab_token_span *d_spans,
                          const int32_t *d_n_spans, const int64_t *d_word_off, const int32_t *d_word_len,
                          kab_word_span *d_words, int32_t *d_word_status, void *stream) {
  if (n_items < 0 || !d_t_off || !d_spans || !d_n_spans || !d_word_off || !d_word_len || !d_words || !d_word_status)
    return KAB_E_BAD_ARG;
  int grid = 0, rc;
  if ((rc = span_grid(n_items, &grid)) != KAB_OK || n_items == 0) return rc;
  const int vec = ((uintptr_t)d_spans % 16 == 0 ? 1 : 0) | ((uintptr_t)d_words % 16 == 0 ? 2 : 0);
  kab_word_spans_kernel<<<grid, KAB_WORD_THREADS, 0, (cudaStream_t)stream>>>(
      n_items, d_t_off, reinterpret_cast<const KabTokenSpan *>(d_spans), d_n_spans, d_word_off, d_word_len,
      reinterpret_cast<KabWordSpan *>(d_words), d_word_status, vec);
  KAB_CUDA(cudaGetLastError());
  return KAB_OK;
}

int kab_log_softmax_pack_device(const float *d_logits_tbv, int64_t t_max, int64_t n_seq, int32_t V,
                                const int64_t *d_out_off, float *d_log_probs, int64_t n_rows, void *stream_) {
  if (t_max < 0 || n_seq < 0 || n_rows < 0 || V < 1 || V > KAB_SM_MAX_V) return KAB_E_BAD_ARG;
  if (n_rows == 0) return KAB_OK;
  if (!d_logits_tbv || !d_out_off || !d_log_probs || n_seq == 0) return KAB_E_BAD_ARG;
  cudaStream_t stream = (cudaStream_t)stream_;
  int dev = 0, sms = 0;
  KAB_CUDA(cudaGetDevice(&dev));
  KAB_CUDA(sm_count_of(dev, &sms) == KAB_OK ? cudaSuccess : cudaErrorUnknown);
  const size_t smem = (size_t)KAB_SM_ROWS * (V | 1) * sizeof(float);
  const int64_t n_tiles = (n_rows + KAB_SM_ROWS - 1) / KAB_SM_ROWS;
  const int per_sm = (int)std::max<size_t>(1, std::min<size_t>(8, (200 * 1024) / (smem + 4096)));
  const unsigned grid = (unsigned)std::min<int64_t>(n_tiles, (int64_t)sms * per_sm);
  if (V == 39) {
    KAB_CUDA(ensure_dyn_smem((const void *)kab_log_softmax_pack_kernel<39>, dev, smem));
    kab_log_softmax_pack_kernel<39><<<grid, KAB_SM_ROWS, smem, stream>>>(d_logits_tbv, n_seq, d_out_off, d_log_probs, n_rows, V);
  } else {
    KAB_CUDA(ensure_dyn_smem((const void *)kab_log_softmax_pack_kernel<0>, dev, smem));
    kab_log_softmax_pack_kernel<0><<<grid, KAB_SM_ROWS, smem, stream>>>(d_logits_tbv, n_seq, d_out_off, d_log_probs, n_rows, V);
  }
  KAB_CUDA(cudaGetLastError());
  return KAB_OK;
}

// segment statistics of arrays already on the device (kab_segstats.cuh); asynchronous on `stream`
static int segment_stats_launch(kab_plan *pl, const int32_t *d_path, const int32_t *d_lab, const float *d_sc,
                                const int32_t *d_st, int64_t n_seg, const int64_t *d_seg_lat_off,
                                const int64_t *d_seg_end, KabSegmentRecord *d_rec, uint8_t *d_lab8,
                                cudaStream_t stream) {
  if (n_seg > 0) {
    if (!pl->d_seg_scratch) KAB_CUDA(pool_malloc((void **)&pl->d_seg_scratch, (size_t)std::max<int64_t>(pl->total_T, 1) * 4));
    const unsigned grid = (unsigned)std::min<int64_t>((n_seg + KAB_SEG_WARPS - 1) / KAB_SEG_WARPS, (int64_t)pl->sm_count * 3);
    KAB_CUDA(ensure_dyn_smem((const void *)kab_segment_stats_kernel, pl->device, KAB_SEG_SMEM));
    kab_segment_stats_kernel<<<grid, KAB_SEG_WARPS * 32, KAB_SEG_SMEM, stream>>>(n_seg, pl->B, d_seg_lat_off, d_seg_end, pl->d_t_off,
                                                                      d_path, d_lab, d_sc, d_st, pl->d_seg_scratch, d_rec);
  }
  if (d_lab8 && pl->total_T > 0) {
    const unsigned grid = (unsigned)std::min<int64_t>((pl->total_T + 1023) / 1024, (int64_t)pl->sm_count * 8);
    kab_labels_u8_kernel<<<grid, 256, 0, stream>>>(d_lab, d_lab8, pl->total_T);
  }
  KAB_CUDA(cudaGetLastError());
  return record_run_event(pl, stream);
}

int kab_plan_segment_stats_device(kab_plan *pl, const int32_t *d_best_path, const int32_t *d_best_labels,
                                  const float *d_best_scores, const int32_t *d_status, int64_t n_segments,
                                  const int64_t *d_seg_lat_off, const int64_t *d_seg_end,
                                  kab_segment_record *d_records, uint8_t *d_labels_u8, void *stream_) {
  if (!pl || n_segments < 0) return KAB_E_BAD_ARG;
  if (pl->spec.ctc) return KAB_E_UNSUPPORTED;  // (the records are those of Kokoro-Align's align())
  if (pl->B == 0) return n_segments == 0 ? KAB_OK : KAB_E_BAD_ARG;
  if (!d_best_path || !d_best_labels || !d_best_scores || !d_status) return KAB_E_BAD_ARG;
  if (n_segments > 0 && (!d_seg_lat_off || !d_seg_end || !d_records)) return KAB_E_BAD_ARG;
  static_assert(sizeof(kab_segment_record) == sizeof(KabSegmentRecord), "record layout");
  DeviceGuard guard;
  KAB_CUDA(guard.enter(pl->device));
  return segment_stats_launch(pl, d_best_path, d_best_labels, d_best_scores, d_status, n_segments, d_seg_lat_off,
                              d_seg_end, reinterpret_cast<KabSegmentRecord *>(d_records), d_labels_u8,
                              reinterpret_cast<cudaStream_t>(stream_));
}

namespace {

struct HostRun {  // what one kab_plan_run_host* call asks for
  const float *h_in = nullptr;  // log-probs, or raw logits when `logits`
  bool logits = false;
  float *h_lp_out = nullptr;
  int32_t *h_path = nullptr, *h_lab = nullptr, *h_status = nullptr;
  float *h_sc = nullptr, *h_fs = nullptr;
  // segment records (optional)
  int64_t n_seg = 0;
  const int64_t *h_seg_lat_off = nullptr, *h_seg_end = nullptr;
  kab_segment_record *h_rec = nullptr;
  uint8_t *h_lab8 = nullptr;
};

// Streams, device buffers and -- for large batches -- the child plans of the pipelined path.  Built
// into the plan only as a whole: any failure tears everything down again (host_teardown), so a later
// call starts from scratch instead of running over a half-built set of segments.
int host_setup(kab_plan *pl) {
  if (pl->host_ready) return KAB_OK;
  const size_t n = (size_t)pl->total_T, B = (size_t)pl->B;
  const int64_t V = pl->spec.V;
  auto fail = [&](int rc) { host_teardown(pl); return rc; };
#define KAB_SETUP(call)                                                  \
  do {                                                                   \
    cudaError_t e_ = (call);                                             \
    if (e_ != cudaSuccess) return fail(cuda_fail(e_, #call));            \
  } while (0)
  KAB_SETUP(cudaStreamCreateWithFlags(&pl->stream, cudaStreamNonBlocking));
  KAB_SETUP(cudaStreamCreateWithFlags(&pl->s_in, cudaStreamNonBlocking));
  KAB_SETUP(cudaStreamCreateWithFlags(&pl->s_out, cudaStreamNonBlocking));
  KAB_SETUP(pool_malloc((void **)&pl->d_lp, n * V * 4));
  KAB_SETUP(pool_malloc((void **)&pl->d_path, n * 4));
  KAB_SETUP(pool_malloc((void **)&pl->d_lab, n * 4));
  KAB_SETUP(pool_malloc((void **)&pl->d_sc, n * 4));
  KAB_SETUP(pool_malloc((void **)&pl->d_fs, B * 4));
  KAB_SETUP(pool_malloc((void **)&pl->d_st, B * 4));
  // ---- cut the batch into segments of >= 32 MB of log-probs, at lattice boundaries whose
  // first row is 16-byte aligned (bulk copies), at most 12 segments
  const int64_t bytes_total = (int64_t)n * V * 4;
  // (only worthwhile when every segment still holds enough lattices to fill the GPU: a few
  // long chapters are better off in one launch, where they run side by side)
  int want = (int)std::min<int64_t>(std::min<int64_t>(12, bytes_total / (32ll << 20)), (int64_t)B / 512);
  if (const char *fs = getenv("KAB_HOST_SEGMENTS")) want = atoi(fs);  // development / tests
  if (want >= 2 && pl->h_t_off[0] == 0) {
    std::vector<int64_t> cuts{0};
    for (int k = 1; k < want; ++k) {
      const int64_t target = (int64_t)n * k / want;
      int64_t b = std::lower_bound(pl->h_t_off.begin(), pl->h_t_off.end(), target) - pl->h_t_off.begin();
      while (b < (int64_t)B && (pl->h_t_off[b] * V) % 4 != 0) ++b;
      if (b > cuts.back() && b < (int64_t)B) cuts.push_back(b);
    }
    if (cuts.size() >= 2) {
      cuts.push_back((int64_t)B);
      const char *inject = getenv("KAB_TEST_FAIL_CHILD");  // tests: make the k-th child plan fail
      // The child plans are independent (classification of their lattices on the host, a few pool
      // allocations and uploads): one host thread each -- created one after the other they were
      // 6.6 of the 7.2 ms of this function for the 12 segments of config 2.
      const size_t nseg = cuts.size() - 1;
      std::vector<kab_plan *> child(nseg, nullptr);
      std::vector<int> child_rc(nseg, KAB_OK);
      auto make_child = [&](size_t k) {
        const int64_t b0 = cuts[k], b1 = cuts[k + 1];
        std::vector<int64_t> to(pl->h_t_off.begin() + b0, pl->h_t_off.begin() + b1 + 1);
        std::vector<int64_t> lo(pl->h_l_off.begin() + b0, pl->h_l_off.begin() + b1 + 1);
        const int64_t t0 = to[0], l0 = lo[0];
        for (auto &x : to) x -= t0;
        for (auto &x : lo) x -= l0;
        const int32_t *lab = pl->h_labels.empty() ? nullptr : pl->h_labels.data() + l0;
        child_rc[k] = (inject && atoi(inject) == (int)k) ? KAB_E_NOMEM
                                                        : plan_create_impl(&child[k], pl->device, pl->spec, b1 - b0, to.data(), lab, lo.data(), nullptr,
                                                                           pl->spec.ctc ? 0 : -1);
      };
      if (std::thread::hardware_concurrency() >= 4 && !getenv("KAB_SERIAL_SETUP")) {
        std::vector<std::thread> th;
        for (size_t k = 1; k < nseg; ++k) th.emplace_back(make_child, k);
        make_child(0);
        for (auto &t : th) t.join();
      } else {
        for (size_t k = 0; k < nseg; ++k) make_child(k);
      }
      int first_rc = KAB_OK;
      for (size_t k = 0; k < nseg; ++k) {
        if (child_rc[k] != KAB_OK) { if (first_rc == KAB_OK) first_rc = child_rc[k]; continue; }
        child[k]->is_child = true;
        if (first_rc == KAB_OK) {
          pl->segs.push_back(child[k]);
          pl->seg_b0.push_back(cuts[k]);
        } else {
          kab_plan_destroy(child[k]);  // (behind a failed one: not part of the pipeline)
        }
      }
      if (first_rc != KAB_OK) return fail(first_rc);
      for (size_t k = 0; k < nseg; ++k) {
        cudaEvent_t e1 = nullptr, e2 = nullptr;
        KAB_SETUP(cudaEventCreateWithFlags(&e1, cudaEventDisableTiming));
        pl->ev_in.push_back(e1);
        KAB_SETUP(cudaEventCreateWithFlags(&e2, cudaEventDisableTiming));
        pl->ev_cmp.push_back(e2);
      }
    }
  }
  // ---- a book: few lattices, the time of the longest.  Its rows go first and its clusters start at once.
  {
    const char *be = getenv("KAB_HOST_BOOK");
    const std::vector<KabLattice> &bl = pl->lists[Q_BAND];  // (longest first)
    if (pl->segs.empty() && !pl->sub && !pl->is_child && pl->band_kernel == BandKernel::R && !pl->Vc && !pl->any_bad_label &&
        pl->h_t_off[0] == 0 && bl.size() >= 4 && !(be && atoi(be) == 0) && (bytes_total >= (48ll << 20) || (be && atoi(be) >= 1))) {
      double band_t = 0.0;
      for (const KabLattice &d : bl) band_t += d.T;
      constexpr int NP = kab_plan::NPIPE;
      std::vector<uint8_t> m[NP];
      for (int k = 0; k < NP; ++k) m[k].assign(B, k == NP - 1 ? 1 : 0);
      // pipe 0: the longest chapter; pipe 1: the next ones while they stay within a third of the frames
      size_t taken = 0, cnt[NP] = {0, 0, 0};
      double acc = 0.0;
      for (int k = 0; k + 1 < NP; ++k) {
        while (taken + 1 < bl.size() && (k == 0 ? cnt[0] < 1 : (cnt[1] < 5 && acc + bl[taken].T <= 0.34 * band_t))) {
          const KabLattice &d = bl[taken++];
          acc += d.T;
          m[k][(size_t)d.index] = 1; m[NP - 1][(size_t)d.index] = 0;
          pl->pipe_rows[k].emplace_back(pl->h_t_off[(size_t)d.index], (int64_t)d.T);
          ++cnt[k];
        }
      }
      for (size_t b = 0; b < B;) {  // the other lattices: contiguous runs of rows
        if (!m[NP - 1][b]) { ++b; continue; }
        size_t e = b;
        while (e < B && m[NP - 1][e]) ++e;
        pl->pipe_rows[NP - 1].emplace_back(pl->h_t_off[b], pl->h_t_off[e] - pl->h_t_off[b]);
        b = e;
      }
      const int32_t *lab = pl->h_labels.empty() ? nullptr : pl->h_labels.data();
      int rcs[NP] = {KAB_OK, KAB_OK, KAB_OK};
      auto make = [&](int k) {
        if (k + 1 < NP && cnt[k] == 0) return;
        rcs[k] = plan_create_impl(&pl->pipe[k], pl->device, pl->spec, (int64_t)B, pl->h_t_off.data(), lab, pl->h_l_off.data(),
                                  m[k].data(), k + 1 < NP ? 1 : -1);
      };
      {
        std::vector<std::thread> th;
        for (int k = 1; k < NP; ++k) th.emplace_back(make, k);
        make(0);
        for (auto &t : th) t.join();
      }
      for (int k = 0; k < NP; ++k)
        if (rcs[k] != KAB_OK) return fail(rcs[k]);
      // the clusters of the GPU: one per lattice of pipes 0 and 1, the others for the rest
      int ncl_left = pl->band_nc > 0 ? pl->sm_count / pl->band_nc : 0;
      for (int k = 0; k < NP; ++k) {
        if (!pl->pipe[k]) continue;
        pl->pipe[k]->is_child = true;
        if (pl->pipe[k]->band_nc > 0 && !pl->pipe[k]->lists[Q_BAND].empty()) {
          const int want_cl = k + 1 < NP ? (int)cnt[k] : std::max(1, ncl_left);
          unsigned &grid = pl->pipe[k]->launch[Q_BAND].grid.x;
          grid = std::min(grid, (unsigned)(want_cl * pl->pipe[k]->band_nc));
          ncl_left -= want_cl;
        }
        if (k > 0) KAB_SETUP(cudaStreamCreateWithFlags(&pl->s_pipe[k], cudaStreamNonBlocking));
        KAB_SETUP(cudaEventCreateWithFlags(&pl->ev_pipe_in[k], cudaEventDisableTiming));
        KAB_SETUP(cudaEventCreateWithFlags(&pl->ev_pipe_done[k], cudaEventDisableTiming));
      }
    }
  }
#undef KAB_SETUP
  pl->host_ready = true;
  return KAB_OK;
}

int run_host_impl(kab_plan *pl, const HostRun &r) {
  if (!pl) return KAB_E_BAD_ARG;
  if (pl->B == 0) return r.n_seg == 0 ? KAB_OK : KAB_E_BAD_ARG;
  if (!r.h_in || !r.h_status) return KAB_E_BAD_ARG;
  const bool arrays = r.h_path || r.h_lab || r.h_sc;
  if (arrays && (!r.h_path || !r.h_lab || !r.h_sc)) return KAB_E_BAD_ARG;
  if (!arrays && !r.h_rec && !r.h_lab8) return KAB_E_BAD_ARG;  // nothing requested
  if (r.n_seg < 0 || (r.n_seg > 0 && (!r.h_seg_lat_off || !r.h_seg_end || !r.h_rec))) return KAB_E_BAD_ARG;
  if (r.n_seg > 0) {  // the reference's `indices`: cumulative ends per lattice, non-decreasing, >= 0
    if (r.h_seg_lat_off[0] != 0 || r.h_seg_lat_off[pl->B] != r.n_seg) return KAB_E_BAD_ARG;
    for (int64_t b = 0; b < pl->B; ++b) {
      if (r.h_seg_lat_off[b + 1] < r.h_seg_lat_off[b]) return KAB_E_BAD_ARG;
      int64_t prev = 0;
      for (int64_t k = r.h_seg_lat_off[b]; k < r.h_seg_lat_off[b + 1]; ++k) {
        if (r.h_seg_end[k] < prev) return KAB_E_BAD_ARG;
        prev = r.h_seg_end[k];
      }
    }
  }
  DeviceGuard guard;
  KAB_CUDA(guard.enter(pl->device));
  Trace tr("kab_plan_run_host");
  const size_t n = (size_t)pl->total_T, B = (size_t)pl->B;
  const int64_t V = pl->spec.V;
  if (int rc = host_setup(pl)) return rc;
  const bool want_stats = r.n_seg > 0 || r.h_lab8;
  if (want_stats) {
    const int64_t need = (int64_t)B + 1 + r.n_seg;
    if (need > pl->seg_cap) {
      pool_free(pl->d_seg_off); pool_free(pl->d_seg_rec);
      pl->d_seg_off = nullptr; pl->d_seg_rec = nullptr; pl->seg_cap = 0;
      KAB_CUDA(pool_malloc((void **)&pl->d_seg_off, (size_t)need * 8));
      KAB_CUDA(pool_malloc((void **)&pl->d_seg_rec, (size_t)std::max<int64_t>(r.n_seg, 1) * sizeof(KabSegmentRecord)));
      pl->seg_cap = need;
    }
    if (r.h_lab8 && !pl->d_lab8) KAB_CUDA(pool_malloc((void **)&pl->d_lab8, std::max<size_t>(n, 1)));
    if (r.n_seg > 0) {  // (on the compute stream, where the statistics kernel runs)
      KAB_CUDA(cudaMemcpyAsync(pl->d_seg_off, r.h_seg_lat_off, (B + 1) * 8, cudaMemcpyHostToDevice, pl->stream));
      KAB_CUDA(cudaMemcpyAsync(pl->d_seg_off + B + 1, r.h_seg_end, (size_t)r.n_seg * 8, cudaMemcpyHostToDevice, pl->stream));
    }
  }
  tr.mark("streams, buffers, segments");
  // results that leave after the alignment of the whole batch (stream s): segment records, byte labels
  auto finish = [&](cudaStream_t s) -> int {
    if (!want_stats) return KAB_OK;
    int rc = segment_stats_launch(pl, pl->d_path, pl->d_lab, pl->d_sc, pl->d_st, r.n_seg, pl->d_seg_off,
                                  pl->d_seg_off + B + 1, pl->d_seg_rec, r.h_lab8 ? pl->d_lab8 : nullptr, s);
    if (rc != KAB_OK) return rc;
    if (r.n_seg > 0)
      KAB_CUDA(cudaMemcpyAsync(r.h_rec, pl->d_seg_rec, (size_t)r.n_seg * sizeof(KabSegmentRecord), cudaMemcpyDeviceToHost, s));
    if (r.h_lab8) KAB_CUDA(cudaMemcpyAsync(r.h_lab8, pl->d_lab8, n, cudaMemcpyDeviceToHost, s));
    return KAB_OK;
  };
  if (pl->segs.empty()) {  // small batch: one copy in, one run, one copy out
    cudaStream_t s = pl->stream;
    int rc = KAB_OK;
    if (pl->pipe[0]) {
      // a book: the longest chapters' rows first, their clusters start while the others' rows arrive
      constexpr int NP = kab_plan::NPIPE;
      for (int k = 0; k < NP; ++k) {
        if (!pl->pipe[k]) continue;
        for (const auto &rr : pl->pipe_rows[k])
          KAB_CUDA(cudaMemcpyAsync(pl->d_lp + rr.first * V, r.h_in + rr.first * V, (size_t)rr.second * V * 4, cudaMemcpyHostToDevice, pl->s_in));
        KAB_CUDA(cudaEventRecord(pl->ev_pipe_in[k], pl->s_in));
      }
      for (int k = 0; k < NP; ++k) {
        if (!pl->pipe[k]) continue;
        cudaStream_t ck = k == 0 ? s : pl->s_pipe[k];
        KAB_CUDA(cudaStreamWaitEvent(ck, pl->ev_pipe_in[k], 0));
        if (r.logits)
          for (const auto &rr : pl->pipe_rows[k])
            if ((rc = kab_log_softmax_device(pl->d_lp + rr.first * V, pl->d_lp + rr.first * V, rr.second, pl->spec.V, ck)) != KAB_OK) return rc;
        rc = kab_plan_run_device(pl->pipe[k], pl->d_lp, pl->d_path, pl->d_lab, pl->d_sc, pl->d_fs, pl->d_st, ck);
        if (rc != KAB_OK) return rc;
        if (k > 0) {
          KAB_CUDA(cudaEventRecord(pl->ev_pipe_done[k], ck));
          KAB_CUDA(cudaStreamWaitEvent(s, pl->ev_pipe_done[k], 0));
        }
      }
    } else {
      KAB_CUDA(cudaMemcpyAsync(pl->d_lp, r.h_in, n * V * 4, cudaMemcpyHostToDevice, s));
      if (r.logits && (rc = kab_log_softmax_device(pl->d_lp, pl->d_lp, (int64_t)n, pl->spec.V, s)) != KAB_OK) return rc;
      rc = kab_plan_run_device(pl, pl->d_lp, pl->d_path, pl->d_lab, pl->d_sc, pl->d_fs, pl->d_st, s);
      if (rc != KAB_OK) return rc;
    }
    if (r.h_lp_out) KAB_CUDA(cudaMemcpyAsync(r.h_lp_out, pl->d_lp, n * V * 4, cudaMemcpyDeviceToHost, s));
    if (arrays) {
      KAB_CUDA(cudaMemcpyAsync(r.h_path, pl->d_path, n * 4, cudaMemcpyDeviceToHost, s));
      KAB_CUDA(cudaMemcpyAsync(r.h_lab, pl->d_lab, n * 4, cudaMemcpyDeviceToHost, s));
      KAB_CUDA(cudaMemcpyAsync(r.h_sc, pl->d_sc, n * 4, cudaMemcpyDeviceToHost, s));
    }
    if (r.h_fs) KAB_CUDA(cudaMemcpyAsync(r.h_fs, pl->d_fs, B * 4, cudaMemcpyDeviceToHost, s));
    KAB_CUDA(cudaMemcpyAsync(r.h_status, pl->d_st, B * 4, cudaMemcpyDeviceToHost, s));
    if ((rc = finish(s)) != KAB_OK) return rc;
    tr.mark("enqueue");
    KAB_CUDA(cudaStreamSynchronize(s));
    tr.mark("synchronize");
    return KAB_OK;
  }
  // ---- pipelined: three streams (copy in / kernels / copy out), one event pair per segment
  for (size_t k = 0; k < pl->segs.size(); ++k) {
    kab_plan *c = pl->segs[k];
    const size_t b0 = (size_t)pl->seg_b0[k], t0 = (size_t)pl->h_t_off[b0];
    const size_t nk = (size_t)c->total_T, bk = (size_t)c->B;
    KAB_CUDA(cudaMemcpyAsync(pl->d_lp + t0 * V, r.h_in + t0 * V, nk * V * 4, cudaMemcpyHostToDevice, pl->s_in));
    KAB_CUDA(cudaEventRecord(pl->ev_in[k], pl->s_in));
    KAB_CUDA(cudaStreamWaitEvent(pl->stream, pl->ev_in[k], 0));
    int rc = KAB_OK;
    if (r.logits && (rc = kab_log_softmax_device(pl->d_lp + t0 * V, pl->d_lp + t0 * V, (int64_t)nk, pl->spec.V, pl->stream)) != KAB_OK)
      return rc;
    rc = kab_plan_run_device(c, pl->d_lp + t0 * V, pl->d_path + t0, pl->d_lab + t0, pl->d_sc + t0,
                             pl->d_fs + b0, pl->d_st + b0, pl->stream);
    if (rc != KAB_OK) return rc;
    KAB_CUDA(cudaEventRecord(pl->ev_cmp[k], pl->stream));
    KAB_CUDA(cudaStreamWaitEvent(pl->s_out, pl->ev_cmp[k], 0));
    if (r.h_lp_out)
      KAB_CUDA(cudaMemcpyAsync(r.h_lp_out + t0 * V, pl->d_lp + t0 * V, nk * V * 4, cudaMemcpyDeviceToHost, pl->s_out));
    if (arrays) {
      KAB_CUDA(cudaMemcpyAsync(r.h_path + t0, pl->d_path + t0, nk * 4, cudaMemcpyDeviceToHost, pl->s_out));
      KAB_CUDA(cudaMemcpyAsync(r.h_lab + t0, pl->d_lab + t0, nk * 4, cudaMemcpyDeviceToHost, pl->s_out));
      KAB_CUDA(cudaMemcpyAsync(r.h_sc + t0, pl->d_sc + t0, nk * 4, cudaMemcpyDeviceToHost, pl->s_out));
    }
    if (r.h_fs)
      KAB_CUDA(cudaMemcpyAsync(r.h_fs + b0, pl->d_fs + b0, bk * 4, cudaMemcpyDeviceToHost, pl->s_out));
    KAB_CUDA(cudaMemcpyAsync(r.h_status + b0, pl->d_st + b0, bk * 4, cudaMemcpyDeviceToHost, pl->s_out));
  }
  if (int rc = finish(pl->stream)) return rc;
  KAB_CUDA(cudaStreamSynchronize(pl->s_out));
  KAB_CUDA(cudaStreamSynchronize(pl->stream));
  return KAB_OK;
}

}  // namespace

int kab_plan_run_host(kab_plan *pl, const float *h_log_probs, int32_t *h_best_path, int32_t *h_best_labels,
                      float *h_best_scores, float *h_final_score, int32_t *h_status) {
  if (!h_best_path || !h_best_labels || !h_best_scores) return pl && pl->B == 0 ? KAB_OK : KAB_E_BAD_ARG;
  HostRun r;
  r.h_in = h_log_probs; r.h_path = h_best_path; r.h_lab = h_best_labels; r.h_sc = h_best_scores;
  r.h_fs = h_final_score; r.h_status = h_status;
  return run_host_impl(pl, r);
}

int kab_plan_run_host_logits(kab_plan *pl, const float *h_logits, int32_t *h_best_path, int32_t *h_best_labels,
                             float *h_best_scores, float *h_final_score, int32_t *h_status, float *h_log_probs) {
  if (!h_best_path || !h_best_labels || !h_best_scores) return pl && pl->B == 0 ? KAB_OK : KAB_E_BAD_ARG;
  HostRun r;
  r.h_in = h_logits; r.logits = true; r.h_lp_out = h_log_probs;
  r.h_path = h_best_path; r.h_lab = h_best_labels; r.h_sc = h_best_scores;
  r.h_fs = h_final_score; r.h_status = h_status;
  return run_host_impl(pl, r);
}

int kab_plan_run_host_segments(kab_plan *pl, const float *h_in, int32_t is_logits, int64_t n_segments,
                               const int64_t *h_seg_lat_off, const int64_t *h_seg_end,
                               kab_segment_record *h_records, uint8_t *h_labels_u8, int32_t *h_best_path,
                               int32_t *h_best_labels, float *h_best_scores, float *h_final_score,
                               int32_t *h_status) {
  if (pl && pl->spec.ctc) return KAB_E_UNSUPPORTED;  // (the records are those of Kokoro-Align's align())
  HostRun r;
  r.h_in = h_in; r.logits = is_logits != 0;
  r.n_seg = n_segments; r.h_seg_lat_off = h_seg_lat_off; r.h_seg_end = h_seg_end; r.h_rec = h_records;
  r.h_lab8 = h_labels_u8;
  r.h_path = h_best_path; r.h_lab = h_best_labels; r.h_sc = h_best_scores;
  r.h_fs = h_final_score; r.h_status = h_status;
  return run_host_impl(pl, r);
}

int kab_ctc_best_path(const float *log_probs, int64_t T, int32_t V, const int32_t *labels, int64_t L,
                      int32_t beam_size, int32_t max_move, int32_t *best_path, int32_t *best_labels,
                      float *best_scores, float *final_score, int32_t *status) {
  if (!status) return KAB_E_BAD_ARG;
  const int64_t t_off[2] = {0, T}, l_off[2] = {0, L};
  int dev = 0;
  KAB_CUDA(cudaGetDevice(&dev));
  kab_plan *pl = nullptr;
  int rc = kab_plan_create(&pl, dev, 1, t_off, labels, l_off, V, beam_size, max_move);
  if (rc != KAB_OK) return rc;
  rc = kab_plan_run_host(pl, log_probs, best_path, best_labels, best_scores, final_score, status);
  kab_plan_destroy(pl);
  return rc;
}

int kab_pool_trim(void) {
  DevPool &P = pool();
  std::lock_guard<std::mutex> lk(P.mu);
  for (int d = 0; d < POOL_MAX_DEV; ++d) pool_trim_device(P, d, 0);
  return KAB_OK;
}

int kab_host_alloc(void **ptr, size_t bytes) {
  if (!ptr) return KAB_E_BAD_ARG;
  KAB_CUDA(cudaHostAlloc(ptr, bytes, cudaHostAllocDefault));
  return KAB_OK;
}

int kab_host_free(void *ptr) {
  KAB_CUDA(cudaFreeHost(ptr));
  return KAB_OK;
}

}  // extern "C"

#include "kab_text.h"  // kab_encode_transcript, kab_merge_repeated (host-only text helpers)
