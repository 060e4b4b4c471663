"""Token spans and word spans on the B200 (kab_merge_tokens_device / kab_word_spans_device) against
torchaudio's per-item merge_tokens loop, on the paths of a CTC forced alignment.

    python tools/merge_tokens_bench.py --out profiles/r03_merge_tokens_bench.json

Workload: the "utterances" workload of tools/forced_align_bench.py (4 096 utterances, T ~ U[250,
1 500], V = 32, same seeds), aligned by a CTC plan; span scores average exp(log-prob) (the chain
INTEGRATION.md section 7 shows); words are seeded groupings of 1 to 8 tokens.
Ours: CUDA events around each C entry over --reps runs, inputs resident, L2 flushed (a 512 MB write)
before every run; the host-clock time of merge_tokens_batch + word_spans from padded CUDA tensors to
a device synchronise; the alignment's own time (CUDA events, same protocol), for scale.
Baseline: torchaudio.functional.merge_tokens once per item, on CPU tensors over all items, and on
CUDA tensors over a seeded 256-item sample, extrapolated to the batch (each span's .item()
synchronises the device).  Every output is compared: ours against the restatement
(oracle/merge_tokens_np.py) bit for bit, against torchaudio's CPU spans (token / start / end exact,
score within 1e-6 relative), the words against the tutorial's formula bit for bit.  One JSON line,
with the card's name and power limit read in the same run.
"""
import argparse
import ctypes
import json
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from tools.forced_align_bench import card, workload  # noqa: E402


def tutorial_word_scores(tok, st, en, sc, wl):
    """The forced-alignment tutorial's `_score` over `unflatten(spans, wl)`, in Python floats."""
    out, i = [], 0
    for n in wl:
        spans = list(zip(st[i:i + n].tolist(), en[i:i + n].tolist(), sc[i:i + n].tolist()))
        out.append(np.float32(sum(s * (e - a) for a, e, s in spans) / sum(e - a for a, e, _ in spans)))
        i += n
    return np.array(out, np.float32)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--ta-cuda-sample", type=int, default=256)
    args = ap.parse_args()
    import torch
    import torchaudio.functional as F
    from kokoro_align_b200 import _lib, align
    from oracle.merge_tokens_np import merge_tokens_np
    assert torch.cuda.is_available(), "needs a CUDA device"
    dev = torch.device("cuda", 0)
    name, power = card()
    flush = torch.empty(128 << 20, dtype=torch.float32, device=dev)
    s = torch.cuda.current_stream(dev)
    L = _lib.lib()

    def timed(fn, reps):
        fn()   # warm-up
        torch.cuda.synchronize()
        times = []
        for _ in range(reps):
            flush.fill_(1.0)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(s)
            fn()
            e1.record(s)
            e1.synchronize()
            times.append(e0.elapsed_time(e1))
        return times

    T, tgs = workload("utterances", 1234)
    V, B = 32, len(T)
    t_off_h = np.concatenate([[0], np.cumsum(T)]).astype(np.int64)
    l_off = np.concatenate([[0], np.cumsum([len(x) for x in tgs])]).astype(np.int64)
    g = torch.Generator(device=dev).manual_seed(99)
    lp = torch.log_softmax(2.0 * torch.randn(int(t_off_h[-1]), V, device=dev, generator=g), dim=-1).contiguous()
    n = int(t_off_h[-1])
    plan = align.AlignPlan.ctc(t_off_h, np.concatenate(tgs), l_off, V, 0)
    labs = torch.empty(n, dtype=torch.int32, device=dev)
    path, sc = torch.empty_like(labs), torch.empty(n, dtype=torch.float32, device=dev)
    fs, st = torch.empty(B, dtype=torch.float32, device=dev), torch.empty(B, dtype=torch.int32, device=dev)
    align_times = timed(lambda: plan.run_device(lp.data_ptr(), path.data_ptr(), labs.data_ptr(), sc.data_ptr(),
                                                fs.data_ptr(), st.data_ptr(), s.cuda_stream), 5)
    assert (st.cpu().numpy() == 0).all()
    plan.close()
    prob = sc.exp()

    # the two C entries, flat layout
    vp = lambda t: ctypes.c_void_p(t.data_ptr())  # noqa: E731
    t_off = torch.from_numpy(t_off_h).to(dev)
    recs = torch.empty((n, 4), dtype=torch.int32, device=dev)
    cnt = torch.empty(B, dtype=torch.int32, device=dev)

    def merge():
        _lib.check(L.kab_merge_tokens_device(B, vp(t_off), vp(labs), vp(prob), 0, vp(recs), vp(cnt),
                                             ctypes.c_void_p(s.cuda_stream)))
    merge_times = timed(merge, args.reps)
    count = cnt.cpu().numpy().astype(np.int64)
    rng = np.random.default_rng(4321)
    wl = []
    for c in count:
        w = []
        while sum(w) < c:
            w.append(int(min(rng.integers(1, 9), c - sum(w))))
        wl.append(w)
    n_words = np.array([len(w) for w in wl], np.int64)
    w_off = torch.from_numpy(np.concatenate([[0], np.cumsum(n_words)]).astype(np.int64)).to(dev)
    w_len = torch.from_numpy(np.concatenate(wl).astype(np.int32)).to(dev)
    words = torch.empty((int(n_words.sum()), 4), dtype=torch.int32, device=dev)
    wst = torch.empty(B, dtype=torch.int32, device=dev)

    def word():
        _lib.check(L.kab_word_spans_device(B, vp(t_off), vp(recs), vp(cnt), vp(w_off), vp(w_len), vp(words),
                                           vp(wst), ctypes.c_void_p(s.cuda_stream)))
    word_times = timed(word, args.reps)
    assert (wst.cpu().numpy() == 0).all()

    # the Python chain from padded CUDA tensors
    T_max = int(T.max())
    lengths = torch.from_numpy(T)
    valid = torch.arange(T_max, device=dev)[None, :] < lengths.to(dev)[:, None]
    paths_p = torch.zeros((B, T_max), dtype=torch.int32, device=dev)
    prob_p = torch.zeros((B, T_max), dtype=torch.float32, device=dev)
    paths_p[valid] = labs
    prob_p[valid] = prob
    chain_ms = []
    for _ in range(6):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        res = align.merge_tokens_batch(paths_p, prob_p, lengths)
        wres = align.word_spans(res, wl)
        torch.cuda.synchronize()
        chain_ms.append((time.perf_counter() - t0) * 1e3)
    chain_ms = chain_ms[1:]

    # outputs: C entries vs the Python chain vs the restatement vs torchaudio
    r_tok, r_st, r_en, r_sc, r_cnt = (x.cpu().numpy() for x in res)
    flat = recs.cpu().numpy()
    labs_h, prob_h = labs.cpu().numpy(), prob.cpu().numpy()
    eq_c_python, eq_oracle, ta_equal_idx, max_rel = True, True, True, 0.0
    for b in range(B):
        a, e, k = int(t_off_h[b]), int(t_off_h[b + 1]), int(count[b])
        o = merge_tokens_np(labs_h[a:e], prob_h[a:e], 0)
        f = flat[a:a + k]
        eq_c_python &= (k == r_cnt[b] and np.array_equal(f[:, 0], r_tok[b, :k]) and np.array_equal(f[:, 1], r_st[b, :k])
                        and np.array_equal(f[:, 2], r_en[b, :k]) and f[:, 3].tobytes() == r_sc[b, :k].tobytes())
        eq_oracle &= (len(o[0]) == k and np.array_equal(o[0], r_tok[b, :k]) and np.array_equal(o[1], r_st[b, :k])
                      and np.array_equal(o[2], r_en[b, :k]) and o[3].tobytes() == r_sc[b, :k].tobytes())
    counts_equal_targets = bool(np.array_equal(count, [len(x) for x in tgs]))
    w_sc, w_c = wres.score.cpu().numpy(), wres.count.cpu().numpy()
    eq_words = bool(np.array_equal(w_c, n_words))
    for b in range(B):
        k = len(wl[b])
        k_s = int(count[b])
        ref = tutorial_word_scores(r_tok[b, :k_s], r_st[b, :k_s], r_en[b, :k_s], r_sc[b, :k_s], wl[b])
        eq_words &= w_sc[b, :k].tobytes() == ref.tobytes()
    wflat = words.cpu().numpy()
    eq_words_c = bool(all(wflat[int(w_off[b]):int(w_off[b]) + len(wl[b]), 3].tobytes() == w_sc[b, :len(wl[b])].tobytes()
                          for b in range(B)))

    # torchaudio, one call per item: CPU over all items, CUDA over a sample
    lab_cpu, prob_cpu = torch.from_numpy(labs_h), torch.from_numpy(prob_h)
    t0 = time.perf_counter()
    ta = [F.merge_tokens(lab_cpu[int(t_off_h[b]):int(t_off_h[b + 1])], prob_cpu[int(t_off_h[b]):int(t_off_h[b + 1])])
          for b in range(B)]
    ta_cpu_ms = (time.perf_counter() - t0) * 1e3
    for b in range(B):
        k = int(count[b])
        spans = ta[b]
        ta_equal_idx &= (len(spans) == k and [x.token for x in spans] == r_tok[b, :k].tolist()
                         and [x.start for x in spans] == r_st[b, :k].tolist() and [x.end for x in spans] == r_en[b, :k].tolist())
        if k:
            ref = np.array([x.score for x in spans], np.float32)
            d = np.abs(r_sc[b, :k].astype(np.float64) - ref)
            max_rel = max(max_rel, float(np.max(np.where(ref != 0, d / np.maximum(np.abs(ref), 1e-300), d))))
    sample = np.sort(np.random.default_rng(7).choice(B, args.ta_cuda_sample, replace=False))
    F.merge_tokens(labs[:int(T[0])], prob[:int(T[0])])   # warm-up
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for b in sample:
        F.merge_tokens(labs[int(t_off_h[b]):int(t_off_h[b + 1])], prob[int(t_off_h[b]):int(t_off_h[b + 1])])
    torch.cuda.synchronize()
    ta_cuda_sample_ms = (time.perf_counter() - t0) * 1e3

    n_spans, n_w = int(count.sum()), int(n_words.sum())
    merge_ms, word_ms = float(np.median(merge_times)), float(np.median(word_times))
    line = {
        "bench": "merge_tokens", "workload": "utterances", "utterances": B, "frames": n, "spans": n_spans, "words": n_w,
        "merge_tokens_kernel_ms_median": merge_ms, "merge_tokens_kernel_ms_all": merge_times,
        "word_spans_kernel_ms_median": word_ms, "word_spans_kernel_ms_all": word_times,
        "kernels_ms_total": merge_ms + word_ms,
        "bytes_merge": 8 * n + 8 * (B + 1) + 16 * n_spans + 4 * B,
        "bytes_words": 16 * n_spans + 4 * B + 8 * (B + 1) * 2 + 4 * n_w + 16 * n_w + 4 * B,
        "python_chain_ms_median": float(np.median(chain_ms)), "python_chain_ms_all": chain_ms,
        "python_chain_timing": "host clock, merge_tokens_batch + word_spans from padded CUDA tensors to a synchronise",
        "align_ms_median": float(np.median(align_times)), "align_ms_all": align_times,
        "kernels_fraction_of_align": (merge_ms + word_ms) / float(np.median(align_times)),
        "torchaudio_cpu_loop_ms": ta_cpu_ms,
        "torchaudio_cuda_loop_ms_sample": ta_cuda_sample_ms, "torchaudio_cuda_sample_items": int(len(sample)),
        "torchaudio_cuda_loop_ms_extrapolated": ta_cuda_sample_ms * B / len(sample),
        "speedup_kernels_vs_torchaudio_cpu": ta_cpu_ms / (merge_ms + word_ms),
        "speedup_chain_vs_torchaudio_cpu": ta_cpu_ms / float(np.median(chain_ms)),
        "equal_c_entry_python": bool(eq_c_python), "equal_oracle": bool(eq_oracle),
        "equal_torchaudio_cpu_token_start_end": bool(ta_equal_idx),
        "max_rel_score_diff_vs_torchaudio_cpu": max_rel, "scores_within_1e-6_of_torchaudio_cpu": bool(max_rel <= 1e-6),
        "counts_equal_target_lengths": counts_equal_targets,
        "equal_word_formula": bool(eq_words), "equal_word_c_entry_python": eq_words_c,
        "l2_flushed": True, "timing": "CUDA events around each C entry, inputs resident",
        "gpu": name, "power_limit": power, "torch": torch.__version__,
    }
    print(json.dumps(line), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
