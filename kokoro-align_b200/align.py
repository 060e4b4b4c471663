"""Host-side mirror of the reference's best-path interface (kokoro_align/align.py).

Same names, arguments, return values and exception types as the reference:

    ctc_best_path(log_probs, labels, beam_size=1000, max_move=4)      align.py:43-109
    best_path(input_file, voca_file, output_file)                     align.py:112-124

backed by the sm_100a kernels through the C ABI (include/kokoro_align_b200.h).  The batched
form (``AlignPlan``) is what a B200 pipeline uses: many independent chapter / segment
lattices per launch, inputs optionally already resident in HBM.
"""
import ctypes
import itertools
from dataclasses import dataclass
from typing import NamedTuple

import numpy as np

from . import _lib
from ._lib import ST_BAD_LABEL, ST_DEAD_BAND, ST_NONFINITE, ST_OK, KabError, PlanInfo  # noqa: F401


# kab_segment_record (include/kokoro_align_b200.h): what align() (align.py:127-169) needs per segment
SEGMENT_RECORD = np.dtype([("text_start", "<i4"), ("text_end", "<i4"), ("non_blanks", "<i4"),
                           ("non_blanks_score", "<f4"), ("all_score", "<f4"), ("status", "<i4")])


def flat_segments(indices_list):
    """The reference's per-chapter ``indices`` arrays (cumulative segment ends, preprocess.py:12-35)
    -> the C-ABI layout (seg_lat_off int64 [B+1], seg_end int64 [n_segments]).  A tuple is taken
    to be that layout already (callers that run the same segmentation many times build it once)."""
    if isinstance(indices_list, tuple):
        seg_lat_off, seg_end = indices_list
        return (np.ascontiguousarray(seg_lat_off, dtype=np.int64), np.ascontiguousarray(seg_end, dtype=np.int64))
    seg_lat_off = np.concatenate([[0], np.cumsum([len(x) for x in indices_list])]).astype(np.int64)
    seg_end = (np.concatenate([np.asarray(x, dtype=np.int64) for x in indices_list])
               if len(indices_list) else np.zeros(0, np.int64))
    return seg_lat_off, np.ascontiguousarray(seg_end, dtype=np.int64)


def raise_for_status(status, V=None):
    """Turn a per-lattice status into the exception the reference raises (SURVEY.md 8b)."""
    if status == ST_OK:
        return
    if status == ST_DEAD_BAND:   # np.argmax of an empty array, align.py:101
        raise ValueError("attempt to get argmax of an empty sequence")
    if status == ST_BAD_LABEL:   # log_probs[i, labels[v]], align.py:77
        raise IndexError(f"index out of bounds for axis 1 with size {V}")
    if status == ST_NONFINITE:
        raise ValueError("log_probs must be finite")
    raise KabError(f"unknown lattice status {status}")


def _ptr(a):
    return ctypes.c_void_p(a.ctypes.data) if a is not None else ctypes.c_void_p(0)


class AlignPlan:
    """A fixed batch of transcripts + frame counts, classified and resident on one GPU.

    t_off / l_off are int64 [B+1] row / label offsets into the flat ``log_probs [sum T, V]``
    and ``labels [sum L]`` arrays (the C-ABI "flat batch" layout).
    """

    def __init__(self, t_off, labels, l_off, vocab_size, beam_size=1000, max_move=4, device=0):
        self._setup(t_off, labels, l_off, vocab_size, device)
        self._create(_lib.lib().kab_plan_create, int(beam_size), int(max_move))

    @classmethod
    def ctc(cls, t_off, labels, l_off, vocab_size, blank=0, device=0, long_form=False, beam_size=None, *,
            free_ends=False):
        """A plan in CTC forced-alignment mode (kab_plan_create_ctc): torchaudio's forced_align
        recurrence for every lattice of the batch; labels are token ids in [0, vocab_size) other
        than ``blank``.  best_labels are then token ids per frame (``blank`` on even states).
        long_form=True (kab_plan_create_ctc_long): lattices with more than 3296 states run on the
        wide kernel where it fits and is estimated faster (a whole chapter in one lattice), with the
        same outputs.  Wide vocabularies (vocab_size > 512, e.g. NeMo's 1025) reach the warp, band
        and wide kernels through a compact copy of every lattice's own columns; a lattice with more
        than 511 distinct labels runs on the generic kernel on its own, and the wide kernel takes
        long lattices while no compact lattice of the plan has more than 335 distinct labels.
        beam_size=W (kab_plan_create_ctc_band; long_form makes no difference): the recurrence is limited to
        the window of W states around the diagonal of the Kokoro plans (align.py:64-65), so a lattice costs
        T * W cells instead of T * S.  A lattice the window never clips is computed as by long_form=True;
        for any other the result is the best path INSIDE the band, which equals torchaudio's only when the
        unbanded best path lies inside it, and status 1 (ST_DEAD_BAND) says no path stays inside.
        free_ends=True (kab_plan_create_ctc_free; routed as long_form=True): the transcript may cover any
        window of frames [t0, t1] of its lattice, for recordings with untranscribed speech at the edges.
        The path is the best one over every window of at least L + R frames (ties: the later end, the
        earlier start); frames outside the window get state -1, the blank and its log-prob, so
        merge_tokens_batch's spans give where the text starts and ends, and final_score is the score over
        the window.  Not combined with beam_size (ValueError)."""
        _check_free_ends(free_ends, beam_size)
        plan = cls.__new__(cls)
        plan._setup(t_off, labels, l_off, vocab_size, device)
        L = _lib.lib()
        if free_ends:
            plan._create(L.kab_plan_create_ctc_free, int(blank))
        elif beam_size is not None:
            plan._create(L.kab_plan_create_ctc_band, int(blank), int(beam_size))
        else:
            plan._create(L.kab_plan_create_ctc_long if long_form else L.kab_plan_create_ctc, int(blank))
        return plan

    def _setup(self, t_off, labels, l_off, vocab_size, device):
        self.t_off = np.ascontiguousarray(t_off, dtype=np.int64)
        self.l_off = np.ascontiguousarray(l_off, dtype=np.int64)
        self.labels = np.ascontiguousarray(labels).astype(np.int32, copy=False)
        self.labels = np.ascontiguousarray(self.labels)
        self.B = int(self.t_off.shape[0] - 1)
        self.V = int(vocab_size)
        self.total_T = int(self.t_off[-1]) if self.B else 0
        self.device = int(device)
        self._h = ctypes.c_void_p(0)

    def _create(self, create, *mode_args):
        L = _lib.lib()
        _lib.check(create(ctypes.byref(self._h), self.device, self.B, _ptr(self.t_off), _ptr(self.labels),
                          _ptr(self.l_off), self.V, *mode_args))
        info = PlanInfo()
        _lib.check(L.kab_plan_get_info(self._h, ctypes.byref(info)))
        self.info = info

    def close(self):
        h, self._h = getattr(self, "_h", None), None
        if h and _lib is not None and _lib._lib is not None:   # (module globals vanish at exit)
            _lib._lib.kab_plan_destroy(h)

    __del__ = close

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    # -- host buffers in, host buffers out (H2D + kernels + D2H inside the call)
    def run_host(self, log_probs, out=None, logits=False, log_probs_out=None):
        """logits=True: ``log_probs`` holds RAW LOGITS and align.py:116-117 runs on the device
        (kab_softmax.cuh; a few ulp from numpy's values, so opt-in); ``log_probs_out`` (float32
        [sum T, V]) then receives the log-probs that were aligned."""
        lp = np.ascontiguousarray(log_probs, dtype=np.float32)
        if lp.shape != (self.total_T, self.V):
            raise ValueError(f"log_probs must have shape {(self.total_T, self.V)}, got {lp.shape}")
        if out is None:
            out = (np.empty(self.total_T, np.int32), np.empty(self.total_T, np.int32),
                   np.empty(self.total_T, np.float32), np.empty(self.B, np.float32),
                   np.empty(self.B, np.int32))
        path, labs, scores, final, status = out
        if logits:
            if log_probs_out is not None:
                assert log_probs_out.dtype == np.float32 and log_probs_out.flags.c_contiguous \
                    and log_probs_out.shape == lp.shape
            _lib.check(_lib.lib().kab_plan_run_host_logits(self._h, _ptr(lp), _ptr(path), _ptr(labs),
                                                           _ptr(scores), _ptr(final), _ptr(status),
                                                           _ptr(log_probs_out)))
        else:
            _lib.check(_lib.lib().kab_plan_run_host(self._h, _ptr(lp), _ptr(path), _ptr(labs),
                                                    _ptr(scores), _ptr(final), _ptr(status)))
        return path, labs, scores, final, status

    def run_host_segments(self, log_probs, indices_list, logits=False, arrays=False, labels_u8=False):
        """Align and return the per-segment records of align() (align.py:151-162) computed on the
        device: ``indices_list[b]`` = the reference's ``indices`` (cumulative segment ends) of
        lattice b.  Only 24 bytes per SEGMENT cross PCIe unless ``arrays`` (the three T-length
        arrays as well) or ``labels_u8`` (best_labels as bytes, for the ``decoded`` column) is set.
        Returns (records [n_segments] SEGMENT_RECORD, final_score, status, extras) with
        extras = {"best_path", "best_labels", "best_scores", "labels_u8"} as requested."""
        lp = np.ascontiguousarray(log_probs, dtype=np.float32)
        if lp.shape != (self.total_T, self.V):
            raise ValueError(f"log_probs must have shape {(self.total_T, self.V)}, got {lp.shape}")
        seg_lat_off, seg_end = flat_segments(indices_list)
        if seg_lat_off.shape[0] != self.B + 1:
            raise ValueError(f"indices_list must hold one array per lattice ({self.B}), got {seg_lat_off.shape[0] - 1}")
        n_seg = int(seg_end.shape[0])
        rec = np.zeros(n_seg, SEGMENT_RECORD)
        final, status = np.empty(self.B, np.float32), np.empty(self.B, np.int32)
        extras = {}
        if arrays:
            extras.update(best_path=np.empty(self.total_T, np.int32), best_labels=np.empty(self.total_T, np.int32),
                          best_scores=np.empty(self.total_T, np.float32))
        if labels_u8:
            if self.V > 256:
                raise ValueError("labels_u8 needs vocab_size <= 256")
            extras["labels_u8"] = np.empty(self.total_T, np.uint8)
        _lib.check(_lib.lib().kab_plan_run_host_segments(
            self._h, _ptr(lp), int(bool(logits)), n_seg, _ptr(seg_lat_off), _ptr(seg_end), _ptr(rec),
            _ptr(extras.get("labels_u8")), _ptr(extras.get("best_path")), _ptr(extras.get("best_labels")),
            _ptr(extras.get("best_scores")), _ptr(final), _ptr(status)))
        return rec, final, status, extras

    def segment_stats_torch(self, best_path, best_labels, best_scores, status, indices_list, labels_u8=False,
                            stream=None):
        """Segment records from the CUDA tensors run_torch returned (nothing leaves the device).
        Returns (records: CUDA uint8 tensor [n_segments, 24] -- view it with SEGMENT_RECORD after
        .cpu().numpy() --, labels_u8 CUDA tensor or None); asynchronous."""
        import torch
        dev = best_path.device
        seg_lat_off, seg_end = flat_segments(indices_list)
        n_seg = int(seg_end.shape[0])
        d_off = torch.from_numpy(seg_lat_off).to(dev)
        d_end = torch.from_numpy(seg_end).to(dev)
        rec = torch.zeros((n_seg, SEGMENT_RECORD.itemsize), dtype=torch.uint8, device=dev)
        lab8 = torch.empty(self.total_T, dtype=torch.uint8, device=dev) if labels_u8 else None
        s = torch.cuda.current_stream(dev) if stream is None else stream
        _lib.check(_lib.lib().kab_plan_segment_stats_device(
            self._h, ctypes.c_void_p(best_path.data_ptr()), ctypes.c_void_p(best_labels.data_ptr()),
            ctypes.c_void_p(best_scores.data_ptr()), ctypes.c_void_p(status.data_ptr()), n_seg,
            ctypes.c_void_p(d_off.data_ptr()), ctypes.c_void_p(d_end.data_ptr()), ctypes.c_void_p(rec.data_ptr()),
            ctypes.c_void_p(lab8.data_ptr() if lab8 is not None else 0), ctypes.c_void_p(s.cuda_stream)))
        rec._kab_keep = (d_off, d_end)   # the kernel reads them asynchronously
        return rec, lab8

    # -- device pointers (e.g. torch tensors' data_ptr()), asynchronous on `stream`
    def run_device(self, d_log_probs, d_best_path, d_best_labels, d_best_scores, d_final_score,
                   d_status, stream=0):
        _lib.check(_lib.lib().kab_plan_run_device(self._h, ctypes.c_void_p(d_log_probs),
                                                  ctypes.c_void_p(d_best_path),
                                                  ctypes.c_void_p(d_best_labels),
                                                  ctypes.c_void_p(d_best_scores),
                                                  ctypes.c_void_p(d_final_score),
                                                  ctypes.c_void_p(d_status), ctypes.c_void_p(stream)))

    def run_torch(self, log_probs, stream=None, logits=False):
        """log_probs: CUDA float32 tensor [sum T, V] on this plan's device.  Returns CUDA tensors
        (best_path, best_labels, best_scores, final_score, status); asynchronous.
        logits=True: the tensor holds RAW LOGITS (the encoder's output, train.py:215-229) and is
        normalised IN PLACE first (align.py:116-117 on the device, kab_log_softmax_device)."""
        import torch
        assert log_probs.is_cuda and log_probs.dtype == torch.float32 and log_probs.is_contiguous()
        assert tuple(log_probs.shape) == (self.total_T, self.V), (tuple(log_probs.shape), self.total_T, self.V)
        dev = log_probs.device
        n = self.total_T
        if logits:
            log_softmax_torch(log_probs, out=log_probs, stream=stream)
        path = torch.empty(n, dtype=torch.int32, device=dev)
        labs = torch.empty(n, dtype=torch.int32, device=dev)
        scores = torch.empty(n, dtype=torch.float32, device=dev)
        final = torch.empty(self.B, dtype=torch.float32, device=dev)
        status = torch.empty(self.B, dtype=torch.int32, device=dev)
        s = torch.cuda.current_stream(dev) if stream is None else stream
        self.run_device(log_probs.data_ptr(), path.data_ptr(), labs.data_ptr(), scores.data_ptr(),
                        final.data_ptr(), status.data_ptr(), s.cuda_stream)
        return path, labs, scores, final, status

    def ctc_posteriors_torch(self, log_probs, best_path, status, stream=None):
        """Forward-backward posteriors of a CTC plan's state paths (kab_plan_ctc_posteriors_device, DESIGN.md
        3.9f), on the device: log_probs CUDA float32 [sum T, V] (the rows that were aligned), best_path int32
        [sum T] (run_torch's state path, or any other state path), status int32 [B] (run_torch's).  Returns
        (posteriors float32 [sum T], log_likelihood float64 [B]): posteriors[t] = exp(alpha_t(p_t) + beta_t(p_t) -
        log Z), the probability that the lattice's paths pass through state p_t at frame t (0 where p_t is outside
        the window), and log Z, the log of the total probability of the transcript (-ctc_loss; a banded plan: of
        the paths inside the band).  A lattice whose status is not 0 gets 0 and NaN.  Asynchronous.  KabError for
        a Kokoro or free-ends plan and for a window min(beam_size, S) above POSTERIOR_MAX_STATES, except in a
        long_form plan without beam_size: there lattices up to POSTERIOR_LONG_MAX_STATES run on a chain of warps
        over the whole GPU (DESIGN.md 3.9g)."""
        import torch
        assert log_probs.is_cuda and log_probs.dtype == torch.float32 and log_probs.is_contiguous()
        assert tuple(log_probs.shape) == (self.total_T, self.V), (tuple(log_probs.shape), self.total_T, self.V)
        assert best_path.dtype == torch.int32 and best_path.is_contiguous() and best_path.numel() == self.total_T
        assert status.dtype == torch.int32 and status.is_contiguous() and status.numel() == self.B
        dev = log_probs.device
        post = torch.empty(self.total_T, dtype=torch.float32, device=dev)
        ll = torch.empty(self.B, dtype=torch.float64, device=dev)
        s = torch.cuda.current_stream(dev) if stream is None else stream
        _lib.check(_lib.lib().kab_plan_ctc_posteriors_device(
            self._h, _vp(log_probs), _vp(best_path), _vp(status), _vp(ll), _vp(post), ctypes.c_void_p(s.cuda_stream)))
        return post, ll


def ctc_best_path(log_probs, labels, beam_size=1000, max_move=4, return_final_score=False):
    """Drop-in for kokoro_align.align.ctc_best_path (align.py:43-109).

    log_probs: [T, V] float32 (other float dtypes are cast to float32 first -- the reference's
    own path is float32 end to end, align.py:113-117); labels: [L] any integer dtype (int8 from
    encoder.encode_text).  Returns (best_path int32 [T], best_labels int32 [T],
    best_scores float32 [T]).  Raises ValueError when no state is active in the last frame and
    IndexError for a label outside [-V, V), as the reference does.
    """
    lp = np.ascontiguousarray(log_probs, dtype=np.float32)
    if lp.ndim != 2:
        raise ValueError("log_probs must be [T, V]")
    labels = np.ascontiguousarray(labels)
    T, V = lp.shape
    if T == 0:   # beams[-1] on an empty list, align.py:100
        raise IndexError("list index out of range")
    if max_move < 1 or beam_size < 0:   # argmax over an empty move axis / negative dimensions
        raise ValueError("attempt to get argmax of an empty sequence")
    with AlignPlan([0, T], labels, [0, labels.shape[0]], V, beam_size, max_move,
                   device=_current_device()) as plan:
        path, labs, scores, final, status = plan.run_host(lp)
    raise_for_status(int(status[0]), V)
    if return_final_score:
        return path, labs, scores, final[0]
    return path, labs, scores


# ---------------------------------------------------------------- CTC forced alignment
# torchaudio.functional.forced_align's recurrence (three moves, its tie rule, the better of the last
# two states at the end; DESIGN.md 3.9) on the CTC plans of the C ABI (kab_plan_create_ctc).

def _ctc_item_checks(tg, V, blank, where=""):
    """torchaudio's checks of one item, in its order and with its exception types.  tg: int64
    numpy [L].  Returns R, the number of adjacent equal targets."""
    if (tg == blank).any():
        raise ValueError(f"{where}targets Tensor shouldn't contain blank index. Found {tg}.")
    if tg.size == 0:
        raise RuntimeError(f"{where}targets must not be empty")
    if tg.max() >= V:
        raise ValueError(f"{where}targets values must be less than the CTC dimension")
    if tg.min() < 0:
        raise ValueError(f"{where}targets values must be non-negative")
    return int((tg[1:] == tg[:-1]).sum())


def _ctc_tensor_checks(log_probs, targets, blank):
    import torch
    if log_probs.dim() != 3:
        raise RuntimeError("log_probs must be 3-D (batch_size, input length, num classes)")
    if targets.dim() != 2:
        raise RuntimeError("targets must be 2-D (batch_size, target length,)")
    if log_probs.dtype != torch.float32:
        raise RuntimeError(f"log_probs must be float32 (the kernels align in fp32), got {log_probs.dtype}")
    if targets.dtype not in (torch.int32, torch.int64):
        raise RuntimeError(f"targets must be int32 or int64, got {targets.dtype}")
    if targets.device != log_probs.device:
        raise RuntimeError("log_probs and targets must be on the same device")
    if not 0 <= blank < log_probs.shape[-1]:
        raise RuntimeError("blank must be within [0, num classes)")


def _ctc_lengths(lengths, B, full, what):
    """input_lengths / target_lengths -> int64 numpy [B] (None: every item is `full` long)."""
    if lengths is None:
        return np.full(B, full, np.int64)
    n = np.asarray(lengths.cpu() if hasattr(lengths, "cpu") else lengths, dtype=np.int64)
    if n.ndim != 1 or n.shape[0] != B:
        raise RuntimeError(f"{what} must be 1-D (batch_size,)")
    if B and (n.min() < 0 or n.max() > full):
        raise RuntimeError(f"{what} must lie in [0, {full}]")
    return n


def _check_beam(beam_size):
    if beam_size is not None and int(beam_size) < 1:
        raise ValueError(f"beam_size must be >= 1, got {beam_size}")


def _check_free_ends(free_ends, beam_size):
    if free_ends and beam_size is not None:
        raise ValueError("free_ends=True does not combine with beam_size: the band assumes that the transcript "
                         "spans the whole recording")


def _check_posteriors(free_ends, beam_size, S, where=lambda b: "", long_form=False):
    """posteriors=True: no free ends, and every item's window min(beam_size, S) within the posterior pass's limit
    (long_form=True without beam_size: S within POSTERIOR_LONG_MAX_STATES, the chain pass of DESIGN.md 3.9g).
    S: int64 numpy [B] states per item."""
    if free_ends:
        raise ValueError("posteriors=True does not combine with free_ends=True")
    if long_form and beam_size is None:
        over = np.flatnonzero(S > _lib.POSTERIOR_LONG_MAX_STATES)
        if over.size:
            b = int(over[0])
            raise ValueError(f"{where(b)}long-form posteriors need at most {_lib.POSTERIOR_LONG_MAX_STATES} states, the "
                             f"item has S = {int(S[b])} (2 L + 1); pass beam_size <= {_lib.POSTERIOR_MAX_STATES} for "
                             f"banded posteriors")
        return
    w = S if beam_size is None else np.minimum(S, int(beam_size))
    over = np.flatnonzero(w > _lib.POSTERIOR_MAX_STATES)
    if over.size:
        b = int(over[0])
        raise ValueError(f"{where(b)}posteriors need at most {_lib.POSTERIOR_MAX_STATES} states per frame, the item has "
                         f"S = {int(S[b])} (2 L + 1) states in a window of {int(w[b])}; pass beam_size <= "
                         f"{_lib.POSTERIOR_MAX_STATES} for banded posteriors")


def _band_lost(beam_size, where=""):
    return ValueError(f"{where}no CTC path stays within beam_size={beam_size}; widen the beam")


def forced_align(log_probs, targets, input_lengths=None, target_lengths=None, blank=0, *, long_form=False,
                 beam_size=None, free_ends=False, posteriors=False):
    """Drop-in for torchaudio.functional.forced_align (same arguments, output shapes and dtypes,
    exception types): log_probs float32 [1, T, V], targets int32 / int64 [1, L] on the same device
    (CPU or CUDA).  Returns (paths [1, T] of the targets' dtype: the token id of every frame,
    scores float32 [1, T]: log_probs[0, t, paths[0, t]]) on the input's device; the output is what
    torchaudio.functional.merge_tokens takes.  Bit-exact with torchaudio's CPU implementation
    whenever the chosen end state has a finite score (where both end states are -inf, torchaudio's
    traceback is undefined; this one follows the recurrence, DESIGN.md 3.9).  NaN or +inf
    log-probs raise ValueError (-inf, for masking, is accepted), in any column of the row.
    long_form=True: a lattice of more than 3296 states (2 L + 1) runs on the wide kernel, with the
    same outputs.  Any vocabulary size up to 65535 reaches the staged kernels while the target has at
    most 511 distinct ids (AlignPlan.ctc).
    beam_size=W: banded alignment for long recordings (AlignPlan.ctc): only the W states of the window
    around the diagonal S*t/T are kept in frame t, which takes T * W cells of work and backpointers instead
    of T * S.  The result is the best path INSIDE the band; it equals torchaudio's only when the unbanded
    best path lies inside the band.  ValueError when no path stays inside it (widen the beam) and for
    beam_size < 1.
    free_ends=True: the targets are aligned to the best window [t0, t1] of the recording rather than to all
    of it (speech before or after the transcript, a passage inside a longer recording; AlignPlan.ctc).
    Frames outside the window hold the blank and its log-prob, so merge_tokens gives the spans of the
    text.  For a gap in the middle of the transcript, append a zero log-prob column as a <star> token
    (the MMS recipe) and put it in the targets.  Not combined with beam_size (ValueError).
    posteriors=True: also returns the forward-backward posterior of the aligned state in every frame and the log
    of the total probability of the targets (AlignPlan.ctc_posteriors_torch), computed on the device from the
    same plan and rows: (paths, scores, posteriors float32 [1, T], log_likelihood float64 [1]).  The paths and
    scores are those of posteriors=False; CPU tensors run on the current CUDA device.  exp(sum(scores) -
    log_likelihood) is the posterior of the whole path, a confidence for the utterance.  ValueError with
    free_ends=True and when the window min(beam_size, 2 L + 1) exceeds POSTERIOR_MAX_STATES (pass beam_size).
    With long_form=True and no beam_size the limit is POSTERIOR_LONG_MAX_STATES (324 001 states, a three-hour
    recording): lattices above POSTERIOR_MAX_STATES run on a chain of warps over the whole GPU (DESIGN.md 3.9g),
    exact, unbanded, log_likelihood = -ctc_loss."""
    import torch
    _check_beam(beam_size)
    _check_free_ends(free_ends, beam_size)
    _ctc_tensor_checks(log_probs, targets, blank)
    if log_probs.size(0) != 1 or targets.size(0) != 1:
        raise RuntimeError("The batch dimension for log_probs and targets must be 1 (forced_align_batch takes batches)")
    T, V = int(log_probs.shape[1]), int(log_probs.shape[2])
    if int(_ctc_lengths(input_lengths, 1, T, "input_lengths").max()) != T:
        raise RuntimeError("input length mismatch")
    L = int(targets.shape[1])
    if target_lengths is not None and int(_ctc_lengths(target_lengths, 1, L, "target_lengths").max()) != L:
        raise RuntimeError("target length mismatch")
    tg = targets[0].cpu().numpy().astype(np.int64)
    R = _ctc_item_checks(tg, V, blank)
    if T < L + R:
        raise RuntimeError(f"targets length is too long for CTC. Found log_probs length: {T}, targets length: {L}, "
                           f"and number of repeats: {R}")
    if posteriors:
        _check_posteriors(free_ends, beam_size, np.array([2 * L + 1]), long_form=long_form)
    dev = log_probs.device
    with AlignPlan.ctc([0, T], tg, [0, L], V, blank, device=dev.index if dev.type == "cuda" else _current_device(),
                       long_form=long_form, beam_size=beam_size, free_ends=free_ends) as plan:
        if posteriors:
            gdev = _span_device(log_probs)
            with torch.cuda.device(gdev):
                lp = log_probs[0].contiguous().to(gdev)
                path, labs, scores, _, st = plan.run_torch(lp)
                post, ll = plan.ctc_posteriors_torch(lp, path, st)
                status = int(st[0])   # (synchronises: the plan is destroyed below)
            labs, scores, post, ll = labs.to(dev), scores.to(dev), post.to(dev), ll.to(dev)
        elif dev.type == "cuda":
            with torch.cuda.device(dev):
                _, labs, scores, _, status = plan.run_torch(log_probs[0].contiguous())
                status = int(status[0])   # (synchronises: the plan is destroyed below)
        else:
            _, labs, scores, _, st = plan.run_host(log_probs[0].contiguous().numpy())
            labs, scores, status = torch.from_numpy(labs), torch.from_numpy(scores), int(st[0])
    if status == ST_NONFINITE:
        raise ValueError("log_probs must not contain NaN or +inf")
    if status == ST_DEAD_BAND and beam_size is not None:
        raise _band_lost(beam_size)
    raise_for_status(status, V)
    if posteriors:
        return labs.to(targets.dtype).view(1, T), scores.view(1, T), post.view(1, T), ll
    return labs.to(targets.dtype).view(1, T), scores.view(1, T)


def forced_align_batch(log_probs, targets, input_lengths=None, target_lengths=None, blank=0, *, long_form=False,
                       beam_size=None, free_ends=False, posteriors=False):
    """forced_align for a padded batch, in one plan: log_probs float32 [B, T_max, V], targets
    int32 / int64 [B, L_max], input_lengths / target_lengths [B] (None: all full length).  Item b
    is aligned over its first input_lengths[b] frames and target_lengths[b] targets.  Returns
    (paths [B, T_max] of the targets' dtype, scores float32 [B, T_max]) on the input's device;
    frames past an item's length hold the blank and score 0.  Raises, like forced_align, for the
    first item that fails, naming its index.  On CUDA the valid rows are packed on the device.
    long_form: as in forced_align.  With more than 512 classes, the items with at most 511 distinct
    target ids run on the staged kernels and the others on the generic kernel (AlignPlan.ctc).
    beam_size: as in forced_align (each item's band follows its own T and S; the results are the best
    paths inside the bands); an item with no path inside its band raises ValueError naming it.
    free_ends: as in forced_align, per item (each item's best window of its own frames).
    posteriors=True: as in forced_align, per item: (paths, scores, posteriors float32 [B, T_max] with 0 past an
    item's length, log_likelihood float64 [B]); merge_tokens_batch(paths, posteriors, input_lengths) then gives
    span scores that are mean posteriors.  ValueError naming the first item whose window is too wide (long_form:
    whose S exceeds POSTERIOR_LONG_MAX_STATES)."""
    import torch
    _check_beam(beam_size)
    _check_free_ends(free_ends, beam_size)
    _ctc_tensor_checks(log_probs, targets, blank)
    B, T_max, V = (int(x) for x in log_probs.shape)
    if targets.size(0) != B:
        raise RuntimeError(f"log_probs and targets hold {B} and {targets.size(0)} items")
    L_max = int(targets.shape[1])
    tl = _ctc_lengths(input_lengths, B, T_max, "input_lengths")
    ll = _ctc_lengths(target_lengths, B, L_max, "target_lengths")
    tg_all = targets.cpu().numpy().astype(np.int64)
    for b in range(B):
        where = f"item {b}: "
        R = _ctc_item_checks(tg_all[b, :ll[b]], V, blank, where)
        if tl[b] < 1:
            raise RuntimeError(f"{where}input length must be >= 1")
        if tl[b] < ll[b] + R:
            raise RuntimeError(f"{where}targets length is too long for CTC. Found log_probs length: {tl[b]}, "
                               f"targets length: {ll[b]}, and number of repeats: {R}")
    if posteriors:
        _check_posteriors(free_ends, beam_size, 2 * ll + 1, lambda b: f"item {b}: ", long_form)
    t_off = np.concatenate([[0], np.cumsum(tl)]).astype(np.int64)
    l_off = np.concatenate([[0], np.cumsum(ll)]).astype(np.int64)
    labels = (np.concatenate([tg_all[b, :ll[b]] for b in range(B)]) if B else np.zeros(0, np.int64)).astype(np.int32)
    dev = log_probs.device
    valid = torch.arange(T_max, device=dev)[None, :] < torch.from_numpy(tl).to(dev)[:, None]   # [B, T_max]
    paths = torch.full((B, T_max), blank, dtype=targets.dtype, device=dev)
    scores = torch.zeros((B, T_max), dtype=torch.float32, device=dev)
    if posteriors:
        post_pad = torch.zeros((B, T_max), dtype=torch.float32, device=dev)
        loglik = torch.zeros(B, dtype=torch.float64, device=dev)
    if B == 0:
        return (paths, scores, post_pad, loglik) if posteriors else (paths, scores)
    with AlignPlan.ctc(t_off, labels, l_off, V, blank, device=dev.index if dev.type == "cuda" else _current_device(),
                       long_form=long_form, beam_size=beam_size, free_ends=free_ends) as plan:
        if posteriors:
            gdev = _span_device(log_probs)
            with torch.cuda.device(gdev):
                lp = log_probs[valid].contiguous().to(gdev)   # rows packed on the input's device
                path, labs, sc, _, st = plan.run_torch(lp)
                post, loglik = plan.ctc_posteriors_torch(lp, path, st)
                status = st.cpu().numpy()
            labs, sc, post, loglik = labs.to(dev), sc.to(dev), post.to(dev), loglik.to(dev)
        elif dev.type == "cuda":
            with torch.cuda.device(dev):
                _, labs, sc, _, status = plan.run_torch(log_probs[valid].contiguous())   # rows packed on the device
                status = status.cpu().numpy()
        else:
            _, labs, sc, _, status = plan.run_host(log_probs[valid].numpy())
            labs, sc = torch.from_numpy(labs), torch.from_numpy(sc)
    for b in np.flatnonzero(status != ST_OK):
        if status[b] == ST_NONFINITE:
            raise ValueError(f"item {b}: log_probs must not contain NaN or +inf")
        if status[b] == ST_DEAD_BAND and beam_size is not None:
            raise _band_lost(beam_size, f"item {b}: ")
        raise_for_status(int(status[b]), V)
    paths[valid] = labs.to(targets.dtype)
    scores[valid] = sc
    if posteriors:
        post_pad[valid] = post
        return paths, scores, post_pad, loglik
    return paths, scores


# ---------------------------------------------------------------- token and word spans
# torchaudio.functional.merge_tokens and the word grouping of torchaudio's forced-alignment tutorial,
# batched on the device (kab_merge_tokens_device / kab_word_spans_device, DESIGN.md 3.10).

@dataclass
class TokenSpan:
    """A span of one token (torchaudio.functional.TokenSpan's fields): frames [start, end)."""
    token: int
    start: int
    end: int
    score: float

    def __len__(self):
        return self.end - self.start


class TokenSpans(NamedTuple):
    """Padded token spans of a batch: [B, N_max] tensors (token: the tokens' dtype, start / end:
    int64, score: float32; padding -1 / -1 / -1 / 0) and count int64 [B]."""
    token: "torch.Tensor"
    start: "torch.Tensor"
    end: "torch.Tensor"
    score: "torch.Tensor"
    count: "torch.Tensor"


class WordSpans(NamedTuple):
    """Padded word spans of a batch: [B, W_max] tensors (start / end / first_token: int64, score:
    float32; padding -1 and 0) and count int64 [B] (words per item)."""
    start: "torch.Tensor"
    end: "torch.Tensor"
    score: "torch.Tensor"
    first_token: "torch.Tensor"
    count: "torch.Tensor"


def _span_device(t):
    """The CUDA device the span kernels run on for tensor t (CPU tensors: the current one)."""
    import torch
    if t.is_cuda:
        return t.device
    if not torch.cuda.is_available():
        raise KabError("no CUDA device: the span kernels have no CPU fallback")
    return torch.device("cuda", torch.cuda.current_device())


def _vp(t):
    return ctypes.c_void_p(t.data_ptr())


def _unpad(flat, off, count, n_max, fill):
    """Rows off[b] + j (j < count[b]) of a flat [n, 4] int32 record tensor -> [B, n_max, 4], padded
    with the row `fill`."""
    import torch
    j = torch.arange(n_max, device=flat.device)
    rows = off[:, None] + j[None, :]
    valid = j[None, :] < count[:, None]
    out = flat[rows.clamp_(max=max(flat.shape[0] - 1, 0))] if flat.shape[0] else flat.new_zeros(rows.shape + (4,))
    return torch.where(valid[..., None], out, torch.tensor(fill, dtype=torch.int32, device=flat.device))


def merge_tokens_batch(tokens, scores, lengths=None, blank=0):
    """torchaudio.functional.merge_tokens for a padded batch, on the device: tokens int32 / int64
    [B, T_max] (e.g. forced_align_batch's paths, or greedy CTC decodes), scores float32 [B, T_max]
    (what a span's score averages: forced_align's log-probs or their exp()), lengths [B] (None: every
    item is T_max frames long).  Returns TokenSpans of padded [B, N_max] tensors, N_max =
    count.max(), on the input's device (CPU tensors run on the current CUDA device).  Span scores are
    float32 means computed in double in frame order (DESIGN.md 3.10), within 2.4e-7 relative of
    torchaudio's float32 mean().  ValueError for negative tokens, non-float32 scores or mismatched
    shapes."""
    import torch
    if tokens.dim() != 2 or scores.dim() != 2 or tuple(tokens.shape) != tuple(scores.shape):
        raise ValueError(f"tokens and scores must both be [B, T_max], got {tuple(tokens.shape)} and {tuple(scores.shape)}")
    if tokens.dtype not in (torch.int32, torch.int64):
        raise ValueError(f"tokens must be int32 or int64, got {tokens.dtype}")
    if scores.dtype != torch.float32:
        raise ValueError(f"scores must be float32, got {scores.dtype}")
    B, T_max = (int(x) for x in tokens.shape)
    if lengths is None:
        tl = np.full(B, T_max, np.int64)
    else:
        tl = np.asarray(lengths.cpu() if hasattr(lengths, "cpu") else lengths, dtype=np.int64)
        if tl.ndim != 1 or tl.shape[0] != B:
            raise ValueError(f"lengths must be [B] = [{B}], got shape {tl.shape}")
        if B and (tl.min() < 0 or tl.max() > T_max):
            raise ValueError(f"lengths must lie in [0, {T_max}]")
    if lengths is None:
        tok_f, sc_f = tokens.reshape(-1), scores.reshape(-1)
    else:   # the valid frames, packed on the input's device
        valid = torch.arange(T_max, device=tokens.device)[None, :] < torch.from_numpy(tl).to(tokens.device)[:, None]
        tok_f, sc_f = tokens[valid], scores[valid]
    if tok_f.numel():
        lo, hi = torch.stack(list(torch.aminmax(tok_f))).tolist()
        if lo < 0:
            raise ValueError("tokens must be non-negative")
        if hi > 0x7fffffff:
            raise ValueError("tokens must fit in int32")
    out_dev = tokens.device
    dev = _span_device(tokens)
    with torch.cuda.device(dev):
        tok_f = tok_f.to(dev, torch.int32).contiguous()
        sc_f = sc_f.to(dev).contiguous()
        n = int(tl.sum())
        t_off_h = np.concatenate([[0], np.cumsum(tl)]).astype(np.int64)
        t_off = torch.from_numpy(t_off_h).to(dev)
        recs = torch.empty((max(n, 1), 4), dtype=torch.int32, device=dev)
        cnt = torch.empty(max(B, 1), dtype=torch.int32, device=dev)
        if n == 0:   # (C entry points take no NULL buffers)
            tok_f = torch.zeros(1, dtype=torch.int32, device=dev)
            sc_f = torch.zeros(1, dtype=torch.float32, device=dev)
        s = torch.cuda.current_stream(dev)
        _lib.check(_lib.lib().kab_merge_tokens_device(B, _vp(t_off), _vp(tok_f), _vp(sc_f), int(blank), _vp(recs),
                                                      _vp(cnt), ctypes.c_void_p(s.cuda_stream)))
        count = cnt[:B].to(torch.int64)
        n_max = int(count.max()) if B else 0
        pad = _unpad(recs, t_off[:-1], count, n_max, [-1, -1, -1, 0])
        res = TokenSpans(pad[..., 0].to(tokens.dtype), pad[..., 1].to(torch.int64), pad[..., 2].to(torch.int64),
                         pad[..., 3].contiguous().view(torch.float32), count)
    if out_dev != dev:
        res = TokenSpans(*(x.to(out_dev) for x in res))
    return res


def merge_tokens(tokens, scores, blank=0):
    """Drop-in for torchaudio.functional.merge_tokens (one item): tokens int32 / int64 [T], scores
    float32 [T] -> List[TokenSpan], computed on the device (merge_tokens_batch)."""
    if tokens.ndim != 1 or scores.ndim != 1:
        raise ValueError("`tokens` and `scores` must be 1D Tensor.")
    if len(tokens) != len(scores):
        raise ValueError("`tokens` and `scores` must be the same length.")
    r = merge_tokens_batch(tokens[None], scores[None], None, blank)
    n = int(r.count[0])
    tok, st, en = (x[0, :n].tolist() for x in r[:3])
    sc = r.score[0, :n].tolist()
    return [TokenSpan(token=a, start=b, end=c, score=d) for a, b, c, d in zip(tok, st, en, sc)]


def word_spans(token_spans, word_lengths):
    """Word spans from the TokenSpans of merge_tokens_batch, on their device: word_lengths[b] lists
    the number of tokens (spans) of each word of item b (each >= 1, summing to the item's span
    count).  Returns WordSpans: start = the first span's start, end = the last span's end,
    first_token = the index of the first span, score = float32(sum(score * len) / sum(len)) over
    the word's spans -- the tutorial's `_score`, bit for bit.  ValueError naming the first item
    whose lengths do not fit."""
    import torch
    token, start, end, score, count = token_spans
    B = int(count.shape[0])
    if len(word_lengths) != B:
        raise ValueError(f"word_lengths must hold one sequence per item ({B}), got {len(word_lengths)}")
    cnt_h = count.cpu().numpy().astype(np.int64)
    n_words = np.fromiter((len(w) for w in word_lengths), np.int64, B)
    w_off_h = np.concatenate([[0], np.cumsum(n_words)]).astype(np.int64)
    flat = np.fromiter(itertools.chain.from_iterable(word_lengths), np.int64, int(w_off_h[-1]))
    csum = np.concatenate([[0], np.cumsum(flat)])
    zero = np.searchsorted(w_off_h, np.flatnonzero(flat < 1), "right") - 1   # items with a word of length < 1
    short = np.flatnonzero(csum[w_off_h[1:]] - csum[w_off_h[:-1]] != cnt_h)
    if zero.size or short.size:
        b = int(min(zero.min() if zero.size else B, short.min() if short.size else B))
        if zero.size and b == zero.min():
            raise ValueError(f"item {b}: every word must have at least one token")
        total = int(csum[w_off_h[b + 1]] - csum[w_off_h[b]])
        raise ValueError(f"item {b}: word lengths sum to {total}, the item has {int(cnt_h[b])} token spans")
    out_dev = count.device
    dev = _span_device(count)
    with torch.cuda.device(dev):
        n_max = int(token.shape[1]) if token.dim() == 2 else 0
        valid = torch.arange(n_max, device=dev)[None, :] < count.to(dev)[:, None]
        recs = torch.stack([token.to(dev).to(torch.int32), start.to(dev).to(torch.int32), end.to(dev).to(torch.int32),
                            score.to(dev).to(torch.float32).view(torch.int32)], -1)[valid].contiguous()
        s_off = torch.from_numpy(np.concatenate([[0], np.cumsum(cnt_h)]).astype(np.int64)).to(dev)
        n_w = int(w_off_h[-1])
        w_off = torch.from_numpy(w_off_h).to(dev)
        w_len = torch.from_numpy(flat.astype(np.int32)).to(dev)
        words = torch.empty((max(n_w, 1), 4), dtype=torch.int32, device=dev)
        status = torch.empty(max(B, 1), dtype=torch.int32, device=dev)
        if recs.shape[0] == 0:
            recs = torch.zeros((1, 4), dtype=torch.int32, device=dev)
        if w_len.numel() == 0:
            w_len = torch.zeros(1, dtype=torch.int32, device=dev)
        cnt32 = count.to(dev).to(torch.int32)
        s = torch.cuda.current_stream(dev)
        _lib.check(_lib.lib().kab_word_spans_device(B, _vp(s_off), _vp(recs), _vp(cnt32),
                                                    _vp(w_off), _vp(w_len), _vp(words), _vp(status),
                                                    ctypes.c_void_p(s.cuda_stream)))
        wc = torch.from_numpy(n_words).to(dev)
        pad = _unpad(words, w_off[:-1], wc, int(n_words.max()) if B else 0, [-1, -1, -1, 0])
        res = WordSpans(pad[..., 0].to(torch.int64), pad[..., 1].to(torch.int64), pad[..., 3].contiguous().view(torch.float32),
                        pad[..., 2].to(torch.int64), wc)
    if out_dev != dev:
        res = WordSpans(*(x.to(out_dev) for x in res))
    return res


def trim_pool():
    """Return the device memory cached from destroyed plans to the driver (kab_pool_trim)."""
    _lib.check(_lib.lib().kab_pool_trim())


def _current_device():
    try:
        import torch
        if torch.cuda.is_available():
            return torch.cuda.current_device()
    except ImportError:
        pass
    return 0


def log_softmax(logits):
    """The reference's normalisation, align.py:116-117, kept on the host in fp32 numpy so that
    the parity boundary (the log_probs array) is bit-identical (SURVEY.md 8c)."""
    logits = logits - np.mean(logits, axis=-1, keepdims=True)
    return logits - np.log(np.sum(np.exp(logits), axis=-1, keepdims=True))


def log_softmax_torch(logits, out=None, stream=None):
    """align.py:116-117 on the device: CUDA float32 tensor [rows, V] of raw logits -> log-probs
    (``out`` may be ``logits`` itself: in place).  See kab_softmax.cuh for the parity statement."""
    import torch
    assert logits.is_cuda and logits.dtype == torch.float32 and logits.is_contiguous() and logits.dim() == 2
    if out is None:
        out = torch.empty_like(logits)
    assert out.is_cuda and out.dtype == torch.float32 and out.is_contiguous() and out.shape == logits.shape
    s = torch.cuda.current_stream(logits.device) if stream is None else stream
    with torch.cuda.device(logits.device):
        _lib.check(_lib.lib().kab_log_softmax_device(ctypes.c_void_p(logits.data_ptr()),
                                                     ctypes.c_void_p(out.data_ptr()), logits.shape[0],
                                                     logits.shape[1], ctypes.c_void_p(s.cuda_stream)))
    return out


def _read_transcript_labels_text(voca_file):
    """transcript.py:60-67 + encoder.py:18-19, line by line (the reference's own control flow)."""
    from .encoder import encode_text
    res = []
    with open(voca_file) as f:
        for line in f:
            parts = line.rstrip('\r\n').split('|')
            res.append(parts[1])
    return encode_text(' '.join(res))


_TOKEN_IDS = None


def read_transcript_labels(voca_file):
    """Labels of a ``text|voca`` transcript: transcript.py:60-67 + encoder.py:5-19 (tokens
    outside the 39-symbol vocabulary are dropped, int8 ids).  The plain case (ASCII phonemes
    separated by spaces) is scanned by kab_encode_transcript in the C library -- a book's
    transcripts hold ~4e5 tokens and the per-token Python loop was a third of the files-to-files
    time; anything else takes the reference's own text code path."""
    global _TOKEN_IDS
    if _TOKEN_IDS is None:
        from .encoder import VOCAB
        table = np.full(65536, -1, np.int16)
        for n, tok in enumerate(VOCAB):
            b = tok.encode()
            assert 1 <= len(b) <= 2
            table[b[0] | ((b[1] << 8) if len(b) > 1 else 0)] = n
        _TOKEN_IDS = table
    with open(voca_file, 'rb') as f:
        raw = f.read()
    out = np.empty(len(raw) // 2 + 1, np.int8)
    n = ctypes.c_int64(0)
    rc = _lib.lib().kab_encode_transcript(raw, len(raw), _ptr(_TOKEN_IDS), _ptr(out), ctypes.byref(n))
    if rc == _lib.KAB_E_UNSUPPORTED:
        return _read_transcript_labels_text(voca_file)
    _lib.check(rc)
    return out[:n.value].copy()


def best_path(input_file, voca_file, output_file, device_log_softmax=False):
    """Drop-in for kokoro_align.align.best_path (align.py:112-124): raw logits npz + voca.txt
    -> best_path.npz {best_path, best_labels, best_scores}.

    device_log_softmax=True (opt-in, SURVEY.md 8(f) rank 2) normalises the logits on the GPU
    instead of in numpy: the log-probs then differ from numpy's by a few ulp (kab_softmax.cuh)."""
    with np.load(input_file) as f:
        logits = f['data']
    labels = read_transcript_labels(voca_file)
    if device_log_softmax:
        logits = np.ascontiguousarray(logits, dtype=np.float32)
        T, V = logits.shape
        if T == 0:
            raise IndexError("list index out of range")
        with AlignPlan([0, T], labels, [0, len(labels)], V, device=_current_device()) as plan:
            path, labs, scores, _, status = plan.run_host(logits, logits=True)
        raise_for_status(int(status[0]), V)
    else:
        path, labs, scores = ctc_best_path(log_softmax(logits), labels)
    np.savez(output_file, best_path=path, best_labels=labs, best_scores=scores)


# ----- npz wire format (SURVEY.md 8(f) rank 3): {data, indices} written by preprocess.py:12-35 /
# train.py:228 with np.savez, i.e. a ZIP archive of STORED .npy members.  The rows of a stored
# member are one contiguous byte range of the file, so they are read straight into (pinned)
# batch memory -- no intermediate array, no concatenation.

def npz_member_info(path, key='data'):
    """(shape, dtype, byte offset of the array data or None when the member is compressed)."""
    import struct
    import zipfile
    from numpy.lib import format as npf
    with zipfile.ZipFile(path) as z:
        zi = z.getinfo(key + '.npy')
        with z.open(zi) as m:
            version = npf.read_magic(m)
            if version == (1, 0):
                shape, fortran, dtype = npf.read_array_header_1_0(m)
            else:
                shape, fortran, dtype = npf.read_array_header_2_0(m)
            header_len = m.tell()
        if fortran and len(shape) > 1:
            return shape, dtype, None
        if zi.compress_type != zipfile.ZIP_STORED:
            return shape, dtype, None
        with open(path, 'rb') as f:
            f.seek(zi.header_offset)
            local = f.read(30)
        if local[:4] != b'PK\x03\x04':
            return shape, dtype, None
        n_name, n_extra = struct.unpack('<HH', local[26:30])
        return shape, dtype, zi.header_offset + 30 + n_name + n_extra + header_len


def npz_read_into(path, dst, key='data', info=None):
    """Read member ``key`` of an npz into the C-contiguous array ``dst`` (same shape and dtype):
    one readinto() from the file for stored members, np.load otherwise."""
    shape, dtype, offset = info or npz_member_info(path, key)
    if tuple(shape) != dst.shape:
        raise ValueError(f"{path}:{key} has shape {shape}, expected {dst.shape}")
    if offset is None or dtype != dst.dtype:
        with np.load(path) as f:
            dst[...] = f[key]
        return dst
    view = memoryview(dst.reshape(-1).view(np.uint8))
    with open(path, 'rb', buffering=0) as f:
        f.seek(offset)
        got = 0
        while got < len(view):
            n = f.readinto(view[got:])
            if not n:
                raise OSError(f"{path}: truncated member {key}")
            got += n
    return dst


class _PinnedPool:
    """One grow-only pinned host buffer per process (cudaHostAlloc is slow: ~0.2 ms / MB), reused
    by consecutive best_path_files calls."""
    ptr, size = None, 0

    @classmethod
    def array(cls, shape, dtype=np.float32):
        n = int(np.prod(shape)) * np.dtype(dtype).itemsize
        if n > cls.size:
            L = _lib.lib()
            if cls.ptr:
                _lib.check(L.kab_host_free(cls.ptr))
                cls.ptr, cls.size = None, 0
            p = ctypes.c_void_p(0)
            want = max(n, 1 << 20)
            _lib.check(L.kab_host_alloc(ctypes.byref(p), want))
            cls.ptr, cls.size = p, want
        buf = (ctypes.c_uint8 * max(n, 1)).from_address(cls.ptr.value)
        return np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)


def best_path_files(logits_files, voca_files, best_path_files, skip_existing=True, beam_size=1000,
                    max_move=4, verbose=True, device_log_softmax=False, io_threads=8, timings=None,
                    align_fn=None, pipeline=True):
    """The per-book loop of run_example.py:247-254 as ONE batch: every chapter whose output does
    not exist yet is read straight into one pinned batch buffer (npz_read_into), normalised
    (align.py:116-117: numpy on the host by default -- bit-identical to the reference -- or on the
    GPU with device_log_softmax=True), and all of them are aligned in a single plan: the chapters
    are independent lattices, so they run side by side on the GPU (36 chapters of a 9-hour book
    take the time of the longest one).  Writes the same best_path.npz files, prints the
    reference's two messages, and raises the reference's exception for the first chapter that
    fails (after the other chapters have been written).  Returns the written paths.

    Under torch.distributed (one process per GPU) every rank reads and aligns its own LPT shard
    of the chapters (parallel.shard_batch: no collective on the data path) and writes its own
    output files; the written paths are gathered on rank 0 (other ranks return []).
    ``timings``: optional dict that receives the wall seconds of every phase (per phase the
    slower of the two groups).  ``pipeline=False`` aligns all chapters in one plan."""
    import os
    import time
    from concurrent.futures import ThreadPoolExecutor
    from . import parallel
    t_start = time.perf_counter()
    try:
        import torch.distributed as dist
        world = dist.get_world_size() if dist.is_initialized() else 1
        rank = dist.get_rank() if dist.is_initialized() else 0
    except ImportError:
        dist, world, rank = None, 1, 0

    def scan():
        """What is to be done, decided ONCE (rank 0 under torch.distributed): the chapters whose
        output does not exist yet, their shapes and -- for the LPT shards -- their labels."""
        todo, skipped = [], []
        for lf, vf, bf in zip(logits_files, voca_files, best_path_files):
            if skip_existing and os.path.exists(bf):
                skipped.append(bf)
            else:
                todo.append((lf, vf, bf))
        infos = [npz_member_info(lf) for lf, _, _ in todo]
        for (shape, _, _), (lf, _, _) in zip(infos, todo):
            if len(shape) != 2 or shape[1] != infos[0][0][1]:
                raise ValueError(f"{lf}: logits must be [T, {infos[0][0][1]}], got {shape}")
        labs = None
        if world > 1:   # the LPT shards need the label counts of every chapter
            labs = [np.asarray(read_transcript_labels(vf), dtype=np.int32) for _, vf, _ in todo]
        return todo, skipped, infos, labs

    if world > 1:
        # Every rank must see the SAME list: a rank that starts late would otherwise find outputs the
        # faster ranks have already written, compute a different partition, and chapters would be
        # aligned twice or never.  Rank 0 scans, everybody receives its answer (or its exception).
        box = [None]
        if rank == 0:
            try:
                box[0] = ("ok", scan())
            except Exception as e:   # noqa: BLE001  (re-raised on every rank below)
                box[0] = ("error", e)
        dist.broadcast_object_list(box, src=0)
        if box[0][0] == "error":
            raise box[0][1]
        todo, skipped, infos, labs = box[0][1]
    else:
        todo, skipped, infos, labs = scan()
    if verbose and rank == 0:
        for bf in skipped:
            print(f'Skip writing {bf}')
    if not todo:
        return []
    V = int(infos[0][0][1])
    T_all = [int(i[0][0]) for i in infos]
    if world > 1:
        mine = [int(i) for i in parallel.shard_batch(T_all, [len(x) for x in labs], rank, world, beam_size)]
    else:
        mine = list(range(len(todo)))
    written, first_bad = [], ST_OK
    group_times = []
    groups, local_exc = [], None
    try:
        if mine:
            if any(T_all[i] == 0 for i in mine):   # beams[-1] on an empty list, align.py:100
                raise IndexError("list index out of range")
            # Two groups, each with its own plan and host thread: the chapters on the critical path
            # (at least half as long as the longest) and the rest.  The long group is read, copied and
            # launched first, so its forward passes -- which bound the book -- start while the many
            # short chapters are still being read and their transcripts parsed; both plans then run
            # side by side on the GPU (every chapter lattice has its own cluster of SMs).
            t_max = max(T_all[i] for i in mine)
            long_group = [i for i in mine if 2 * T_all[i] >= t_max]
            short_group = [i for i in mine if 2 * T_all[i] < t_max]
            groups = [long_group, short_group] if (pipeline and align_fn is None and long_group and short_group
                                                   and len(mine) >= 4) else [mine]
            rows = int(sum(T_all[i] for i in mine))
            # (align_fn: the multi-rank CPU tests replace the CUDA plan; then no pinned memory either)
            batch = _PinnedPool.array((rows, V)) if align_fn is None else np.empty((rows, V), np.float32)
            device = _current_device()
            io = ThreadPoolExecutor(max(1, io_threads))

            def run_group(members, row0):
                tm = {}
                t0 = time.perf_counter()
                t_off = np.concatenate([[0], np.cumsum([T_all[i] for i in members])]).astype(np.int64)
                view = batch[row0:row0 + int(t_off[-1])]

                def load(n):
                    dst = view[int(t_off[n]):int(t_off[n + 1])]
                    npz_read_into(todo[members[n]][0], dst, info=infos[members[n]])
                    if not device_log_softmax:   # row blocks: numpy's temporaries stay in cache (same bits)
                        for a in range(0, dst.shape[0], 2048):
                            dst[a:a + 2048] = log_softmax(dst[a:a + 2048])
                # the logits stream into the batch buffer (readinto releases the GIL) while this
                # thread parses the transcripts
                loads = [io.submit(load, n) for n in range(len(members))]
                glabs = [labs[i] if labs is not None else
                         np.asarray(read_transcript_labels(todo[i][1]), dtype=np.int32) for i in members]
                for f in loads:
                    f.result()
                l_off = np.concatenate([[0], np.cumsum([len(x) for x in glabs])]).astype(np.int64)
                labels = np.concatenate(glabs) if glabs else np.zeros(0, np.int32)
                tm["read_normalise_and_labels_s"] = time.perf_counter() - t0
                t0 = time.perf_counter()
                plan = None
                try:
                    if align_fn is not None:
                        path, lab, sc, _, status = align_fn(view, t_off, labels, l_off, V, beam_size, max_move, 0)
                    else:
                        plan = AlignPlan(t_off, labels, l_off, V, beam_size, max_move, device=device)
                        path, lab, sc, _, status = plan.run_host(view, logits=device_log_softmax)
                    tm["plan_and_align_s"] = time.perf_counter() - t0
                    t0 = time.perf_counter()

                    def save(n):
                        a, b = int(t_off[n]), int(t_off[n + 1])
                        np.savez(todo[members[n]][2], best_path=path[a:b], best_labels=lab[a:b], best_scores=sc[a:b])
                    good = [n for n in range(len(members)) if status[n] == ST_OK]
                    for f in [io.submit(save, n) for n in good]:
                        f.result()
                    tm["write_s"] = time.perf_counter() - t0
                finally:
                    if plan is not None:   # (destroying a plan waits for the device: after the outputs are written)
                        plan.close()
                return [(members[n], int(status[n])) for n in range(len(members))], tm

            try:
                row0, jobs = 0, []
                with ThreadPoolExecutor(len(groups)) as gex:
                    for members in groups:
                        jobs.append(gex.submit(run_group, members, row0))
                        row0 += int(sum(T_all[i] for i in members))
                    results = [j.result() for j in jobs]
            finally:
                io.shutdown()
            status_of = {}
            for res, tm in results:
                status_of.update(res)
                group_times.append(tm)
            for i in mine:   # messages and return value in the order of the call
                if status_of[i] != ST_OK:
                    first_bad = first_bad or status_of[i]
                else:
                    if verbose:
                        print(f'Writing {todo[i][2]}')
                    written.append(todo[i][2])
    except Exception as e:   # noqa: BLE001  (under torch.distributed: raised after the collective)
        if world == 1:
            raise
        local_exc = e
    if timings is not None:
        for key in ("read_normalise_and_labels_s", "plan_and_align_s", "write_s"):
            timings[key] = max((tm.get(key, 0.0) for tm in group_times), default=0.0)
        timings.update(total_s=time.perf_counter() - t_start, frames=int(sum(T_all[i] for i in mine)),
                       chapters=len(mine), groups=[len(g) for g in groups])
    if world > 1:
        # No rank returns or raises before this collective (the others would wait for it forever);
        # failures travel with the results and are raised on EVERY rank afterwards.
        parts = [None] * world
        dist.all_gather_object(parts, (written, first_bad, local_exc))
        for _, _, exc in parts:
            if exc is not None:
                raise exc
        first_bad = next((b for _, b, _ in parts if b != ST_OK), ST_OK)
        raise_for_status(first_bad, V)
        if rank != 0:
            return []
        order = {bf: k for k, (_, _, bf) in enumerate(todo)}
        return sorted((bf for w, _, _ in parts for bf in w), key=order.get)
    if local_exc is not None:
        raise local_exc
    raise_for_status(first_bad, V)
    return written


# --------------------------------------------------------------------------- the consumer
# SURVEY.md 8(f) rank 1: the step that reads best_path.npz (align.py:127-169).  Host-side text
# work; it defines the output contract of the kernels (best_path // 2 at the segment
# boundaries, per-segment sums of best_scores), so it lives beside them.

_PUNCT = (',', '.', '!', '?')


class TokenTable:
    """label index -> token index table of a ``text|voca`` transcript (the behaviour of
    transcript.py:13-57): a token owns the labels from the middle of the previous voiced token
    to its own middle; punctuation-only tokens move the boundary without owning labels."""

    def __init__(self, voca_file):
        from .encoder import encode_text
        self.texts, self.vocas, self.table = [], [], []
        labels_seen, boundary = 0, 0
        with open(voca_file) as f:
            for n, line in enumerate(f):
                text, voca = line.rstrip('\r\n').split('|')
                self.texts.append(text)
                self.vocas.append(voca)
                k = len(encode_text(voca))
                if k:
                    labels_seen += k
                    upto = labels_seen - k // 2
                    self.table.extend([boundary] * (upto - len(self.table)))
                    boundary = n + 1
                elif voca in _PUNCT:
                    boundary = n + 1

    def __len__(self):
        return len(self.table)

    def get_token(self, start, end, remove_wordsep=True):
        import re
        lo = self.table[start] if start < len(self.table) else len(self.texts)
        hi = self.table[end] if end < len(self.table) else len(self.texts)
        text = ' '.join(t for t in self.texts[lo:hi] if t)
        parts = [t for t in self.vocas[lo:hi] if t]
        if remove_wordsep:
            voca = ' '.join(parts)
        else:
            voca = ' _ '.join(parts)
            voca = re.sub(r'_ ([.,!?])', r'\1', voca)
            voca = re.sub(r'([.,!?]) _', r'\1', voca)
        return text.strip(), voca.strip()


def _write_align_file(align_file, ends, table, seg, remove_wordsep):
    """The output loop of align.py:146-166.  seg(i, a, b) -> (text_start, text_end or None,
    labels[a:b], non_blanks, non_blanks_score, all_score); text_end None = "len(aligner)"."""
    import os
    from .encoder import decode_text, merge_repeated
    try:
        with open(align_file, 'wt') as out:
            for i in range(len(ends)):
                a = ends[i - 1] if i > 0 else 0
                b = ends[i]
                ts, te, labels, nb, nbs, alls = seg(i, int(a), int(b))
                t0 = min(ts, len(table))
                t1 = min(len(table) if te is None else te, len(table))
                decoded = merge_repeated(decode_text(labels))
                text, voca = table.get_token(t0, t1, remove_wordsep=remove_wordsep)
                out.write(f'{b}|{text}|{voca}|{decoded}|{nb}|{nbs}|{alls}\n')
    except BaseException:
        os.unlink(align_file)
        raise


def align(best_path_file, mfcc_file, voca_file, align_file, remove_wordsep):
    """Drop-in for kokoro_align.align.align (align.py:127-169): one line per silence-split
    segment, ``audio_end|text|voca|decoded|non_blanks|non_blanks_score|all_score``."""
    with np.load(best_path_file) as f:
        label_idx = f['best_path'] // 2            # extended-state index -> label index
        best_labels = f['best_labels']
        best_scores = f['best_scores']
    with np.load(mfcc_file) as f:
        ends = f['indices']
    table = TokenTable(voca_file)
    n_frames = len(label_idx)

    def seg(i, a, b):
        labels = best_labels[a:b]
        scores = best_scores[a:b]
        voiced = labels != 0
        return (int(label_idx[a]), int(label_idx[b]) if b < n_frames else None, labels,
                np.sum(voiced).item(), np.sum(scores[voiced]).item(), np.sum(scores).item())
    _write_align_file(align_file, ends, table, seg, remove_wordsep)


def align_from_records(records, labels_u8, ends, voca_file, align_file, remove_wordsep):
    """align() (align.py:127-169) from the per-segment records the DEVICE computed
    (kab_segstats.cuh: boundaries, counts and both np.sum's in numpy's pairwise order) and the
    per-frame labels as bytes -- text-identical to align() on the same alignment."""
    table = TokenTable(voca_file)

    def seg(i, a, b):
        r = records[i]
        if r["status"] == -1:   # best_path[audio_start] past the end, align.py:151
            raise IndexError(f"index {a} is out of bounds for axis 0 with size {len(labels_u8)}")
        raise_for_status(int(r["status"]))
        te = int(r["text_end"])
        return (int(r["text_start"]), None if te < 0 else te, labels_u8[a:b], int(r["non_blanks"]),
                r["non_blanks_score"].item(), r["all_score"].item())
    _write_align_file(align_file, ends, table, seg, remove_wordsep)


def best_path_and_align(logits_file, mfcc_file, voca_file, align_file, remove_wordsep, best_path_file=None,
                        device_log_softmax=False):
    """best_path() (align.py:112-124) + align() (align.py:127-169) of one chapter in one device
    round trip: the logits go up, 24 bytes per segment and one byte per frame come back (the
    three T-length arrays only when ``best_path_file`` is given, which is then written exactly as
    best_path() writes it).  Same align.txt as the two reference steps."""
    with np.load(logits_file) as f:
        logits = np.ascontiguousarray(f['data'], dtype=np.float32)
    with np.load(mfcc_file) as f:
        ends = f['indices']
    labels = read_transcript_labels(voca_file)
    T, V = logits.shape
    if T == 0:
        raise IndexError("list index out of range")
    lp = logits if device_log_softmax else log_softmax(logits)
    with AlignPlan([0, T], labels, [0, len(labels)], V, device=_current_device()) as plan:
        rec, _, status, ex = plan.run_host_segments(lp, [ends], logits=device_log_softmax,
                                                    arrays=best_path_file is not None, labels_u8=True)
    raise_for_status(int(status[0]), V)
    if best_path_file is not None:
        np.savez(best_path_file, best_path=ex["best_path"], best_labels=ex["best_labels"],
                 best_scores=ex["best_scores"])
    align_from_records(rec, ex["labels_u8"], ends, voca_file, align_file, remove_wordsep)


# --------------------------------------------------------------------------- the producer
# SURVEY.md 8(f) rank 4: predict() (train.py:201-231) runs the encoder on the GPU, copies every
# batch of logits to the host and writes them to *.logits.npz; best_path() reads them back,
# normalises them in numpy and aligns.  On one device none of that has to leave HBM.

class ChapterLogits:
    """The chapter's packed log-probs [T, V] in HBM, filled batch by batch from the encoder's
    padded time-major output (the rows predict() appends to *.logits.npz, train.py:222-228),
    normalised on the way (align.py:116-117, kab_log_softmax_pack_device)."""

    def __init__(self, total_frames, vocab_size, device=None):
        import torch
        self.dev = torch.device("cuda", _current_device()) if device is None else torch.device(device)
        self.log_probs = torch.empty((int(total_frames), int(vocab_size)), dtype=torch.float32, device=self.dev)
        self.rows = 0
        self.indices = []          # cumulative segment ends == the `indices` of the npz container

    def append(self, logits, lens, stream=None):
        """logits: CUDA float32 [T_max, B, V] (AudioToChar.forward, train.py:62-65); lens: the B
        valid lengths (CPU tensor / list, as pad_packed_sequence returns them)."""
        import torch
        assert logits.is_cuda and logits.dtype == torch.float32 and logits.dim() == 3
        logits = logits.contiguous()
        t_max, B, V = logits.shape
        lens = [int(x) for x in lens]
        assert len(lens) == B and all(0 <= x <= t_max for x in lens) and V == self.log_probs.shape[1]
        off = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
        n = int(off[-1])
        assert self.rows + n <= self.log_probs.shape[0], "more frames than the chapter was sized for"
        d_off = torch.from_numpy(off).to(self.dev, non_blocking=False)
        s = torch.cuda.current_stream(self.dev) if stream is None else stream
        dst = self.log_probs[self.rows:self.rows + n]
        with torch.cuda.device(self.dev):
            _lib.check(_lib.lib().kab_log_softmax_pack_device(
                ctypes.c_void_p(logits.data_ptr()), t_max, B, V, ctypes.c_void_p(d_off.data_ptr()),
                ctypes.c_void_p(dst.data_ptr()), n, ctypes.c_void_p(s.cuda_stream)))
        self._keep = (logits, d_off)   # asynchronous readers
        for x in lens:
            self.rows += x
            self.indices.append(self.rows)
        return self


def best_path_from_logits_tensor(logits, labels, indices=None, beam_size=1000, max_move=4, normalised=False,
                                 stream=None):
    """The encoder -> aligner hand-off without the PCIe round trip of predict() + best_path()
    (train.py:215-229, align.py:113-117).  ``logits``: CUDA float32 [T, V] -- the chapter's raw
    logits (normalised in place here) or, with ``normalised=True``, log-probs already (e.g.
    ChapterLogits.log_probs).  ``indices``: the chapter's cumulative segment ends; when given the
    per-segment records of align() are computed on the device as well.
    Returns a dict of CUDA tensors {best_path, best_labels, best_scores, final_score, status
    [, records, labels_u8]}; raises the reference's exceptions (this synchronises on status)."""
    import torch
    assert logits.is_cuda and logits.dim() == 2
    T, V = logits.shape
    if T == 0:
        raise IndexError("list index out of range")
    labels = np.ascontiguousarray(labels)
    with torch.cuda.device(logits.device):
        with AlignPlan([0, T], labels, [0, labels.shape[0]], V, beam_size, max_move,
                       device=logits.device.index) as plan:
            path, labs, scores, final, status = plan.run_torch(logits, stream=stream, logits=not normalised)
            out = dict(best_path=path, best_labels=labs, best_scores=scores, final_score=final, status=status)
            if indices is not None:
                out["records"], out["labels_u8"] = plan.segment_stats_torch(path, labs, scores, status, [indices],
                                                                            labels_u8=V <= 256, stream=stream)
            raise_for_status(int(status.cpu()[0]), V)     # (synchronises; the plan may go afterwards)
    return out
