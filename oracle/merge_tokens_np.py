"""CPU restatement of token spans (torchaudio.functional.merge_tokens) and word spans (the word
grouping of torchaudio's forced-alignment tutorial) with the order of operations the span kernels
use (kab_spans.cuh, DESIGN.md 3.10), so that they are reproduced bit for bit.

    runs:   maximal stretches of equal tokens; frame 0 always starts one
    spans:  every run whose token is not the blank -> (token, start, end), end exclusive
    score:  fl32( (s[start] + s[start+1] + ... + s[end-1]) / (end - start) ), every value converted
            to float64, the sum sequential from the first value (np.add.accumulate), one float64
            division, one rounding to float32
    words:  word w = word_lengths[w] consecutive spans; start = first span's start, end = last span's
            end, first_token = index of the first span, score = fl32( sum_j f64(score_j) * len_j /
            sum_j len_j ), the numerator summed sequentially from +0.0 (the tutorial's Python `sum`)

torchaudio's own float32 mean() sums in a CPU-dependent vectorised order; this mean lies within a
few 1e-7 (relative) of it.
"""
import numpy as np

_SHORT = 64   # spans up to this long are summed column by column across spans, longer ones one by one


def _seq_sums(x, starts, lens):
    """Sequential float64 sums x[s] + x[s+1] + ... + x[s+n-1] (from the first value) for every span."""
    acc = np.empty(starts.shape[0], np.float64)
    short = lens <= _SHORT
    for chunk in np.array_split(np.flatnonzero(short), max(1, int(short.sum()) // 65536 + 1)):
        if chunk.size == 0:
            continue
        w = int(lens[chunk].max())
        cols = np.arange(w)
        idx = starts[chunk, None] + cols[None, :]
        inside = cols[None, :] < lens[chunk, None]
        P = np.where(inside, x[np.where(inside, idx, 0)], 0.0)
        # row-wise accumulate is sequential; the padding lies after each span's last value
        acc[chunk] = np.add.accumulate(P, axis=1)[np.arange(chunk.size), lens[chunk] - 1]
    for k in np.flatnonzero(~short):
        acc[k] = np.add.accumulate(x[starts[k]:starts[k] + lens[k]])[-1]
    return acc


def merge_tokens_np(tokens, scores, blank=0):
    """tokens int [T], scores float32 [T] -> (token int64 [N], start int64 [N], end int64 [N],
    score float32 [N])."""
    tok = np.asarray(tokens, dtype=np.int64).reshape(-1)
    x = np.asarray(scores, dtype=np.float32).reshape(-1).astype(np.float64)
    T = tok.shape[0]
    if T == 0:
        z = np.zeros(0, np.int64)
        return z, z.copy(), z.copy(), np.zeros(0, np.float32)
    run_start = np.concatenate([[0], np.flatnonzero(tok[1:] != tok[:-1]) + 1])
    run_end = np.append(run_start[1:], T)
    keep = tok[run_start] != blank
    start, end = run_start[keep], run_end[keep]
    lens = end - start
    with np.errstate(invalid="ignore"):
        mean = _seq_sums(x, start, lens) / lens.astype(np.float64)
    return tok[start], start, end, mean.astype(np.float32)


def merge_tokens_batch_np(tokens, scores, lengths, blank=0):
    """Padded [B, T_max] -> list of B tuples of merge_tokens_np."""
    return [merge_tokens_np(np.asarray(tokens[b])[:int(lengths[b])], np.asarray(scores[b])[:int(lengths[b])], blank)
            for b in range(len(lengths))]


def word_spans_np(start, end, score, word_lengths):
    """One item's spans (start, end, score float32 [N]) grouped by word_lengths (each >= 1, summing
    to N) -> (start int64 [W], end int64 [W], first_token int64 [W], score float32 [W])."""
    wl = np.asarray(word_lengths, dtype=np.int64).reshape(-1)
    assert (wl >= 1).all() and int(wl.sum()) == len(start)
    first = np.concatenate([[0], np.cumsum(wl)[:-1]]).astype(np.int64) if wl.size else np.zeros(0, np.int64)
    last = first + wl - 1
    lens = (np.asarray(end, np.int64) - np.asarray(start, np.int64)).astype(np.float64)
    term = np.asarray(score, np.float32).astype(np.float64) * lens   # one rounding per product
    num = np.zeros(wl.shape[0], np.float64)
    den = np.zeros(wl.shape[0], np.int64)
    for j in range(int(wl.max()) if wl.size else 0):
        m = wl > j
        num[m] = num[m] + term[first[m] + j]
        den[m] += lens[first[m] + j].astype(np.int64)
    with np.errstate(invalid="ignore"):
        ws = (num / den.astype(np.float64)).astype(np.float32)
    return np.asarray(start, np.int64)[first], np.asarray(end, np.int64)[last], first, ws
