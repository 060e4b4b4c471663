/*
 * kokoro_align_b200.h -- C ABI of the B200-native CTC best-path aligner.
 *
 * Drop-in boundary for ONE path of kaiidams/Kokoro-Align: the banded, max_move-transition
 * CTC best-path alignment
 *     kokoro_align/align.py:43-109   ctc_best_path(log_probs, labels, beam_size=1000, max_move=4)
 *     kokoro_align/align.py:21-40    flush_determined_path  (the traceback)
 * called once per chapter from kokoro_align/align.py:112-124 (best_path) by
 * run_example.py:247-254.  The reference has no FFI of its own (it is pure Python/numpy);
 * these entry points are what a ctypes binding in align.py would call -- see INTEGRATION.md.
 *
 * Plain pointers and sizes only; no torch / C++ types.  All functions return 0 on success or
 * a negative KAB_E_* code (kab_error_string() gives text; CUDA errors are reported as
 * KAB_E_CUDA and the CUDA message is available from kab_last_cuda_error()).
 * There is no CPU fallback: without a CUDA device every compute entry fails with KAB_E_CUDA.
 *
 * Batch layout ("flat batch"):  B independent lattices.
 *   log_probs  float32 [sum_b T_b, V] row-major, lattice b = rows t_off[b] .. t_off[b+1]
 *   labels     int32   [sum_b L_b],            lattice b = l_off[b] .. l_off[b+1]
 *   outputs    best_path int32 [sum T], best_labels int32 [sum T], best_scores float32 [sum T]
 *              (align.py:105-109), final_score float32 [B] (DP score of the end state,
 *              internal to the reference), status int32 [B] (KAB_ST_*).
 * Outputs of a lattice whose status != 0 are unspecified.
 */
#ifndef KOKORO_ALIGN_B200_H
#define KOKORO_ALIGN_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define KAB_VERSION 200 /* 0.2.0 */

/* return codes */
#define KAB_OK 0
#define KAB_E_CUDA (-1)        /* CUDA runtime error, or no device */
#define KAB_E_BAD_ARG (-2)     /* NULL pointer, negative size, max_move outside 1..255, T_b < 1 */
#define KAB_E_NOMEM (-3)       /* host allocation failed */
#define KAB_E_UNSUPPORTED (-4) /* shape outside what the kernels handle (documented per call) */

/* per-lattice status, written to status[b] */
#define KAB_ST_OK 0
#define KAB_ST_DEAD_BAND 1 /* no active state in the last frame: reference raises ValueError, align.py:101 */
#define KAB_ST_BAD_LABEL 2 /* label outside [-V, V): reference raises IndexError, align.py:77 */
#define KAB_ST_NONFINITE 3 /* a log-prob of the lattice is not finite (rejected, see DESIGN.md) */

/* kernel classes a lattice can be routed to (kab_plan_info) */
#define KAB_CLASS_WARP 0    /* one warp per lattice, full window, S <= 248, max_move 4 */
#define KAB_CLASS_BAND 1    /* one CTA per lattice, ring of >= beam_size+12 states in registers, max_move 4 */
#define KAB_CLASS_GENERIC 2 /* any beam_size / max_move / label values */
#define KAB_CLASS_WIDE 3    /* unbanded lattice too wide for one CTA: a chain of warps over the whole GPU */

typedef struct kab_plan kab_plan; /* opaque */

typedef struct kab_plan_info {
  int64_t n_lattices;
  int64_t n_class[4];       /* lattices per KAB_CLASS_* */
  int64_t total_frames;     /* sum_b T_b */
  int64_t cells_eval;       /* sum_b sum_i (hi_i - lo_i): cells the recurrence evaluates */
  int64_t cells_nominal;    /* sum_b T_b * S_b */
  int64_t workspace_bytes;  /* device memory held by the plan (backpointers, labels, queues) */
  int64_t backptr_bytes;    /* of which packed backpointers; for KAB_CLASS_WARP lattices of a best-path
                               plan with more than 124 states: the score checkpoint rows that replace them
                               (one row per 8 frames) */
  int64_t algorithmic_bytes;/* SURVEY.md 8(d): 4*min(V,D+1)*T + cells*b/8 + T*b/8 + 12*T, summed */
  int32_t kernel_launches;  /* kernels launched by one kab_plan_run_* */
  int32_t device;
  int32_t band_kernel;      /* which kernel takes the KAB_CLASS_BAND lattices: KAB_BAND_KERNEL_* (0: none) */
  int32_t band_cluster;     /* CTAs per cluster of that kernel (1 for the single-CTA kernel) */
} kab_plan_info;

#define KAB_BAND_KERNEL_CTA 1      /* kab_band_kernel: one CTA per lattice, two lattices per SM */
#define KAB_BAND_KERNEL_CLUSTER 2  /* kab_bandp_kernel: cluster, four states per lane */
#define KAB_BAND_KERNEL_CLUSTER2 3 /* kab_bandq_kernel: cluster, two states per lane */
#define KAB_BAND_KERNEL_SPEC 4     /* kab_bandr_kernel: cluster, warp-specialised (prep warps, shared-memory mailboxes) */
#define KAB_BAND_KERNEL_HYBRID 5   /* the longest lattices in kab_bandr_kernel clusters (band_cluster CTAs each), the others in
                                      kab_band_kernel on the remaining SMs, side by side */

int kab_version(void);
const char *kab_error_string(int code);
const char *kab_last_cuda_error(void);
int kab_device_count(int *count);

/*
 * Build a plan for a fixed batch of transcripts and frame counts (host pointers; copied).
 * Replaces the label expansion of align.py:46-48 and the per-frame window arithmetic of
 * align.py:64-65; classifies every lattice, uploads the label tables and allocates the
 * backpointer workspace on `device`.  beam_size / max_move are align.py:43's keywords.
 */
int kab_plan_create(kab_plan **plan, int device, int64_t n_lattices, const int64_t *t_off,
                    const int32_t *labels, const int64_t *l_off, int32_t vocab_size,
                    int32_t beam_size, int32_t max_move);
/*
 * A plan in CTC forced-alignment mode: the recurrence of torchaudio.functional.forced_align (three
 * moves, +2 forbidden into a blank and between equal labels, select on the previous frame's scores
 * with its tie rule, the better of the last two states at the end; DESIGN.md 3.9), for a batch.
 * `blank` in [0, vocab_size) is the blank id; labels are token ids in [0, vocab_size) other than it.
 * Every kab_plan_run_* entry takes such a plan: best_path = extended-state index, best_labels =
 * token id per frame (`blank` on even states), best_scores = log_probs[t, best_labels[t]],
 * final_score = DP score of the chosen end state.  Statuses: KAB_ST_DEAD_BAND when T_b < L_b + R_b
 * (R_b = adjacent equal labels; decided here), KAB_ST_BAD_LABEL for a label outside [0, V) or equal
 * to the blank, KAB_ST_NONFINITE for a NaN or +inf log-prob (-inf is accepted: masking).
 * kab_plan_segment_stats_device and kab_plan_run_host_segments return KAB_E_UNSUPPORTED.
 * KAB_E_BAD_ARG for a blank outside [0, vocab_size).
 * Classes: S <= 248 KAB_CLASS_WARP, S <= 3296 KAB_CLASS_BAND, longer lattices KAB_CLASS_GENERIC.  A
 * vocabulary above 512 reaches the warp and band classes through a compact copy of each lattice's own
 * columns (the blank first, then its distinct labels; DESIGN.md 3.9c); a lattice with more than 511
 * distinct labels goes to KAB_CLASS_GENERIC on its own.  The outputs are the same on every class.
 */
int kab_plan_create_ctc(kab_plan **plan, int device, int64_t n_lattices, const int64_t *t_off,
                        const int32_t *labels, const int64_t *l_off, int32_t vocab_size, int32_t blank);
/*
 * kab_plan_create_ctc for long-form alignment (a chapter or any long recording against its text in
 * one lattice): the same arguments, outputs, statuses and errors, but lattices with more than 3296
 * states go to KAB_CLASS_WIDE (a chain of warps over the whole GPU, 2 bits of backpointer per cell)
 * instead of KAB_CLASS_GENERIC (1 byte per cell) where they fit -- vocab_size <= 338 (the wide
 * kernel's emission stages; above 512, the compact width Vc <= 336, i.e. at most 335 distinct labels
 * in the plan's largest compact lattice) and ceil(S/104)/4 + 1 CTAs resident at once -- and where a makespan
 * estimate says so: wide lattices run one after another, each on the whole GPU, generic ones side by
 * side, so a batch of many shorter lattices may stay generic (DESIGN.md 3.9).  Warp and band
 * lattices are routed as by kab_plan_create_ctc.
 */
int kab_plan_create_ctc_long(kab_plan **plan, int device, int64_t n_lattices, const int64_t *t_off,
                             const int32_t *labels, const int64_t *l_off, int32_t vocab_size,
                             int32_t blank);
/*
 * CTC forced alignment with free ends (recordings with untranscribed speech before or after the
 * transcript, a passage inside a longer recording): kab_plan_create_ctc_long's recurrence with
 *   - a virtual state -1 of score 0 in EVERY frame, state 0's move-1 and state 1's move-2 predecessor
 *     (torchaudio's select and tie rules unchanged; frame 0 gets the usual initialisation); the walk
 *     stops there, at the window's first frame t0;
 *   - the end at the maximum of a_t[v] over every frame t and v in {S-1, S-2}: a tie between frames
 *     picks the later frame, within a frame S-2; every candidate -inf: (T-1, S-2).  That frame is t1.
 * Frames outside [t0, t1] get best_path -1, best_labels = blank, best_scores = log_probs[t, blank];
 * final_score = a_t1[v_end], the path score over [t0, t1].  The statuses are kab_plan_create_ctc's;
 * a lattice with L = 0 has every frame outside, final_score 0 and status 0.  Routed as by
 * kab_plan_create_ctc_long (every lattice unbanded); there is no banded free-ends plan.
 * KAB_E_BAD_ARG for a blank outside [0, vocab_size).
 */
int kab_plan_create_ctc_free(kab_plan **plan, int device, int64_t n_lattices, const int64_t *t_off,
                             const int32_t *labels, const int64_t *l_off, int32_t vocab_size,
                             int32_t blank);
/*
 * Banded CTC forced alignment (long recordings, long batches): kab_plan_create_ctc with the
 * recurrence limited to a window of beam_size = W >= 1 states around the diagonal, the window of
 * kab_plan_create (align.py:64-65).  Lattice b (T frames, S = 2L+1 states) at frame i:
 *     lo_i = max(0, floor(S*i/T) - floor(W/2)),   hi_i = min(lo_i + W, S)
 * Every frame applies the CTC recurrence unchanged and then sets every state outside [lo_i, hi_i)
 * to -inf.  The result is the best path INSIDE the band: it equals the unbanded one when that path
 * lies inside the band.
 *   - Covering lattices (W >= S and floor(S*(T-1)/T) <= floor(W/2): the window never clips) are
 *     routed and computed as by kab_plan_create_ctc_long; their outputs are byte-identical to it,
 *     including its "both end states -inf: follow the recurrence" case.
 *   - Any other lattice ends in S-1 if a[S-1] > a[S-2], else S-2; when both are -inf no path stays
 *     inside the band: KAB_ST_DEAD_BAND with a NaN final_score (outputs unspecified).
 *   - The other statuses are those of kab_plan_create_ctc.
 * Routing of a lattice whose window clips: KAB_CLASS_BAND (single-CTA band kernel, T * NBP bytes of
 * backpointers, NBP = (26 * NW + 15) & ~15, NW = ceil((min(W, S) + 32) / 104) warps) when
 * min(W, S) <= 3264 and its columns are staged (vocab_size <= 512, or at most 511 distinct labels
 * through the compact copy); otherwise KAB_CLASS_GENERIC, T * min(W, S) bytes.  kab_plan_info's
 * cells_eval and algorithmic_bytes count the windowed cells.
 * KAB_E_BAD_ARG for a blank outside [0, vocab_size) or beam_size < 1.
 */
int kab_plan_create_ctc_band(kab_plan **plan, int device, int64_t n_lattices, const int64_t *t_off,
                             const int32_t *labels, const int64_t *l_off, int32_t vocab_size,
                             int32_t blank, int32_t beam_size);
int kab_plan_get_info(const kab_plan *plan, kab_plan_info *info);
int kab_plan_destroy(kab_plan *plan);

/*
 * Run the alignment with every buffer already on the plan's device (align.py:57-107 for all
 * lattices of the batch).  `stream` is a cudaStream_t (NULL = default stream); the call is
 * asynchronous with respect to the host.  d_final_score may be NULL.
 */
int kab_plan_run_device(kab_plan *plan, const float *d_log_probs, int32_t *d_best_path,
                        int32_t *d_best_labels, float *d_best_scores, float *d_final_score,
                        int32_t *d_status, void *stream);

/*
 * Same, host buffers (pageable or pinned): copies log_probs to the device, runs, copies the
 * three output arrays, final_score and status back, and returns after everything is complete.
 */
int kab_plan_run_host(kab_plan *plan, const float *h_log_probs, int32_t *h_best_path,
                      int32_t *h_best_labels, float *h_best_scores, float *h_final_score,
                      int32_t *h_status);

/*
 * align.py:116-117 on the device (SURVEY.md 8(f) rank 2): rows of raw encoder logits ->
 * log-probabilities, `x -= mean(x); x - log(sum(exp(x)))`, every fp32 operation and both row
 * sums in numpy's order; exp / log are CUDA's expf / logf, so the result agrees with numpy's to
 * a few ulp (4e-6 absolute in the tests), NOT bit for bit -- numpy's own SIMD exp is
 * CPU-dependent.  d_log_probs may equal d_logits (in place).  Asynchronous on `stream`.
 */
int kab_log_softmax_device(const float *d_logits, float *d_log_probs, int64_t n_rows,
                           int32_t vocab_size, void *stream);

/*
 * The hand-off from the acoustic model (SURVEY.md 8(f) rank 4).  predict() (train.py:215-229)
 * receives a padded, time-major batch logits [t_max, n_seq, V] with lens [n_seq] from the encoder
 * and appends logits[:len_j, j, :] of every sequence j to the chapter's *.logits.npz.  This does
 * the same append plus align.py:116-117 on the device: row d_out_off[j] + t of d_log_probs =
 * log_softmax(logits[t, j, :]), d_out_off int64 [n_seq + 1] on the device (packed row offsets of
 * this batch inside the chapter buffer; d_out_off[0] is the first row written, n_rows =
 * d_out_off[n_seq] - d_out_off[0] -- pass d_log_probs already offset so that d_out_off[0] == 0).
 * vocab_size <= 128.  Asynchronous on `stream`.
 */
int kab_log_softmax_pack_device(const float *d_logits_tbv, int64_t t_max, int64_t n_seq,
                                int32_t vocab_size, const int64_t *d_out_off, float *d_log_probs,
                                int64_t n_rows, void *stream);

/*
 * kab_plan_run_host for RAW LOGITS (the `*.logits.npz` rows of align.py:113-114): copies them to
 * the device, normalises them there (kab_log_softmax_device, in place) and aligns.  Opt-in: the
 * alignment is exact for the device's log-probs, which differ from numpy's by a few ulp.
 * h_log_probs, if not NULL, receives the [sum T, V] log-probs the alignment used.
 */
int kab_plan_run_host_logits(kab_plan *plan, const float *h_logits, int32_t *h_best_path,
                             int32_t *h_best_labels, float *h_best_scores, float *h_final_score,
                             int32_t *h_status, float *h_log_probs);

/*
 * Per-segment statistics of an alignment -- everything the reference's align() (align.py:127-169)
 * reads from the three T-length arrays -- computed on the device (SURVEY.md 8(f) rank 1):
 *   text_start       best_path[audio_start] // 2                          align.py:131,151
 *   text_end         best_path[audio_end] // 2, or -1 when audio_end >= T ("len(aligner)", align.py:152)
 *   non_blanks       np.sum(best_labels[a:b] != 0)                        align.py:160
 *   non_blanks_score np.sum(best_scores[a:b][best_labels[a:b] != 0])      align.py:161
 *   all_score        np.sum(best_scores[a:b])                             align.py:162
 * both sums in numpy's float32 pairwise order, bit for bit.  status = the lattice's KAB_ST_*, or -1
 * when audio_start lies outside the lattice (the reference raises IndexError there).
 */
typedef struct kab_segment_record {
  int32_t text_start, text_end, non_blanks;
  float non_blanks_score, all_score;
  int32_t status;
} kab_segment_record;

/*
 * Segments are given the way the reference stores them (`indices` of *.mfcc.npz, preprocess.py:12-35:
 * cumulative segment ENDS in frames, relative to their lattice), concatenated over the batch:
 * seg_lat_off int64 [B+1] (segments of lattice b = seg_lat_off[b] .. seg_lat_off[b+1]-1), seg_end
 * int64 [n_segments] (non-decreasing inside a lattice).  Device pointers; the arrays are the outputs
 * of kab_plan_run_device on the same plan; d_labels_u8 (may be NULL) receives best_labels as bytes
 * [sum T] (the `decoded` column of align() needs the per-frame labels; vocab_size <= 256).
 * Asynchronous on `stream`.
 */
int kab_plan_segment_stats_device(kab_plan *plan, const int32_t *d_best_path, const int32_t *d_best_labels,
                                  const float *d_best_scores, const int32_t *d_status, int64_t n_segments,
                                  const int64_t *d_seg_lat_off, const int64_t *d_seg_end,
                                  kab_segment_record *d_records, uint8_t *d_labels_u8, void *stream);

/*
 * Forward-backward posteriors of a CTC alignment (DESIGN.md 3.9f), a second device pass over a CTC plan's
 * outputs.  For lattice b (ext = the blank-interleaved states, S = 2L + 1, move 2 into an odd v >= 3 iff
 * ext[v] != ext[v-2]) and the plan's window [lo_t, hi_t) of frame t ([0, S) for kab_plan_create_ctc and
 * kab_plan_create_ctc_long plans, kab_plan_create_ctc_band's band otherwise), in natural log:
 *   alpha_0 = lp[0, blank] at state 0 and lp[0, ext[1]] at state 1; alpha_t(v) = logsumexp of alpha_{t-1} over
 *   v, v-1 and v-2 where allowed, + lp[t, ext[v]]; beta_{T-1} = 0 at S-1 and S-2; beta_t(v) = logsumexp over
 *   the successors v' of beta_{t+1}(v') + lp[t+1, ext[v']]; every state outside its frame's window is -inf.
 *   d_log_likelihood[b] (double) = log Z = logsumexp(alpha_{T-1}(S-1), alpha_{T-1}(S-2)): -ctc_loss of an
 *     unbanded lattice; for a banded one, the log of the probability of the paths inside the band.
 *   d_posteriors[t] (float32, [sum T]) = exp(alpha_t(p_t) + beta_t(p_t) - log Z), clamped to [0, 1], for the
 *     state path p = d_best_path (usually what kab_plan_run_device wrote; any path is accepted, a p_t outside
 *     the window gives 0).
 * A lattice whose d_status is not 0 gets posteriors 0 and log-likelihood NaN; log Z = -inf gives
 * posteriors 0.  d_log_probs are the caller's [sum T, V] rows (16-byte aligned), read by label: any
 * vocab_size works.  A window of up to KAB_POSTERIOR_MAX_STATES states runs in one CTA.  The lattices of a
 * kab_plan_create_ctc_long plan with more states (S up to KAB_POSTERIOR_LONG_MAX_STATES) run on a chain of
 * warps over the whole GPU (DESIGN.md 3.9g), the same quantities with the same tolerances; such a plan's
 * first call checks that the chain's grid can be resident.  KAB_E_UNSUPPORTED for a plan that is not a CTC
 * plan, a free-ends plan, a lattice of a kab_plan_create_ctc or kab_plan_create_ctc_band plan whose window
 * min(beam_size, S) exceeds KAB_POSTERIOR_MAX_STATES (use kab_plan_create_ctc_band or _long), a long-form
 * lattice above KAB_POSTERIOR_LONG_MAX_STATES, or a chain grid the device cannot hold.  The first call
 * builds and uploads what the pass needs (labels, lattice lists, 16 bytes per frame of values, and 8 KB per
 * 256 states of a long-form lattice above the limit for the chain's FIFOs); kab_plan_get_info does not count
 * it.  Asynchronous on `stream`; kab_plan_destroy waits for it.
 */
#define KAB_POSTERIOR_MAX_STATES 28000 /* the states of two float buffers in one CTA's shared memory */
#define KAB_POSTERIOR_LONG_MAX_STATES 324001 /* long-form plans: a three-hour lattice on a B200's resident warps */
int kab_plan_ctc_posteriors_device(kab_plan *plan, const float *d_log_probs, const int32_t *d_best_path,
                                   const int32_t *d_status, double *d_log_likelihood, float *d_posteriors,
                                   void *stream);

/*
 * kab_plan_run_host (is_logits = 0) / kab_plan_run_host_logits (is_logits != 0) that also -- or
 * only -- returns the segment records: h_best_path / h_best_labels / h_best_scores may be NULL
 * (all three), and then 24 bytes per segment come back instead of 12 bytes per frame;
 * h_labels_u8 (may be NULL) as above.  KAB_E_BAD_ARG for segment ends that decrease.
 */
int kab_plan_run_host_segments(kab_plan *plan, const float *h_log_probs_or_logits, int32_t is_logits,
                               int64_t n_segments, const int64_t *h_seg_lat_off, const int64_t *h_seg_end,
                               kab_segment_record *h_records, uint8_t *h_labels_u8, int32_t *h_best_path,
                               int32_t *h_best_labels, float *h_best_scores, float *h_final_score,
                               int32_t *h_status);

/*
 * Token spans of per-frame token sequences (torchaudio.functional.merge_tokens), on the device, for a
 * flat batch: item b = frames d_t_off[b] .. d_t_off[b+1] of d_tokens int32 / d_scores float32
 * (d_t_off int64 [n_items + 1], T_b < 2^31).  A run is a maximal stretch of equal tokens (frame 0
 * always starts one); every run whose token is not `blank` is a span {token, start, end (exclusive),
 * score} in item-relative frames.  score = the mean of scores[start:end]: the values converted to
 * double and added in frame order from the first, divided by end - start in double, rounded once to
 * float32 (DESIGN.md 3.10; -inf and NaN propagate).  Any token values are accepted.
 * The spans of item b go to d_spans[d_t_off[b] .. d_t_off[b] + d_n_spans[b]) (capacity sum T: an
 * item has at most as many spans as frames).  Device pointers on the caller's current device;
 * asynchronous on `stream` (a cudaStream_t, NULL = default stream): the call only launches
 * kab_merge_tokens_kernel.  KAB_E_BAD_ARG for a NULL pointer or n_items < 0.
 */
typedef struct kab_token_span { int32_t token, start, end; float score; } kab_token_span;      /* 16 B */
typedef struct kab_word_span  { int32_t start, end, first_token; float score; } kab_word_span;  /* 16 B */

int kab_merge_tokens_device(int64_t n_items, const int64_t *d_t_off, const int32_t *d_tokens,
                            const float *d_scores, int32_t blank, kab_token_span *d_spans,
                            int32_t *d_n_spans, void *stream);
/*
 * Word spans of those token spans (the word grouping of torchaudio's forced-alignment tutorial):
 * word w of item b groups d_word_len[d_word_off[b] + w] consecutive spans (d_word_off int64
 * [n_items + 1]) and goes to d_words[d_word_off[b] + w]: start = its first span's start, end = its
 * last span's end, first_token = the item-relative index of its first span, score =
 * float32(sum_j double(score_j) * len_j / sum_j len_j), the numerator summed in span order from 0.
 * d_spans / d_n_spans / d_t_off as kab_merge_tokens_device left them.  d_word_status[b] = 1 when
 * the item's word lengths do not sum to d_n_spans[b] or one is < 1 (its words are then not
 * written), else 0.  Asynchronous like kab_merge_tokens_device (kab_word_spans_kernel).
 */
int kab_word_spans_device(int64_t n_items, const int64_t *d_t_off, const kab_token_span *d_spans,
                          const int32_t *d_n_spans, const int64_t *d_word_off, const int32_t *d_word_len,
                          kab_word_span *d_words, int32_t *d_word_status, void *stream);

/*
 * One-shot single lattice with host buffers == kokoro_align/align.py:43
 * ctc_best_path(log_probs[T,V], labels[L], beam_size, max_move) -> (best_path, best_labels,
 * best_scores); *status receives KAB_ST_*; final_score may be NULL.
 */
int kab_ctc_best_path(const float *log_probs, int64_t T, int32_t vocab_size, const int32_t *labels,
                      int64_t L, int32_t beam_size, int32_t max_move, int32_t *best_path,
                      int32_t *best_labels, float *best_scores, float *final_score,
                      int32_t *status);

/*
 * Labels of a `text|voca` transcript file, transcript.py:60-67 + encoder.py:5-19: the second
 * '|'-separated field of every line, split at spaces, tokens looked up in the vocabulary and
 * unknown ones dropped.  `text` = the file's bytes; token_ids[b0 | b1 << 8] = id of the 1- or
 * 2-byte token (b1 = 0 for one byte) or -1; `labels` needs room for n_bytes / 2 + 1 ids.
 * Host-only (no CUDA).  Returns KAB_E_UNSUPPORTED when the bytes leave the plain case the
 * byte-level scan reproduces exactly (a line without '|', a lone '\r', control or non-ASCII
 * bytes inside a voca field); the Python caller then runs the reference's own text code.
 */
int kab_encode_transcript(const uint8_t *text, int64_t n_bytes, const int16_t *token_ids,
                          int8_t *labels, int64_t *n_labels);

/*
 * encoder.py:28, the regular expression of merge_repeated -- re.sub(r'(.+)( \1)+', r'\1', text)
 * -- which align() (align.py:159) runs on the decoded labels of every segment and which costs the
 * backtracking engine ~30 ms per segment (90 s per book).  Same leftmost / greedy semantics, byte
 * for byte, for ASCII text without newlines; KAB_E_UNSUPPORTED otherwise (the Python mirror then
 * uses `re`).  `out` needs room for n bytes.  Host-only.
 */
int kab_merge_repeated(const uint8_t *text, int64_t n_bytes, uint8_t *out, int64_t *n_out);

/*
 * Device memory of destroyed plans is kept in a per-device pool and reused by later plans (the
 * drop-in ctc_best_path() builds one plan per call; cudaFree synchronises the device).  This
 * returns every cached block to the driver.
 */
int kab_pool_trim(void);

/* Pinned host memory for kab_plan_run_host callers (cudaHostAlloc / cudaFreeHost). */
int kab_host_alloc(void **ptr, size_t bytes);
int kab_host_free(void *ptr);

#ifdef __cplusplus
}
#endif
#endif /* KOKORO_ALIGN_B200_H */
