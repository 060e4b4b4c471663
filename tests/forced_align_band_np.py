"""CPU restatement of BANDED CTC forced alignment (kab_plan_create_ctc_band, beam_size): the recurrence of
oracle/forced_align_np.py -- torchaudio's forced_align -- limited to the window of the Kokoro plans
(align.py:64-65).  For lattice (T frames, S = 2L+1 states) and beam_size = W, at frame t only the states of

    lo_t = max(0, floor(S*t/T) - floor(W/2)),   hi_t = min(lo_t + W, S)

keep their scores: each frame applies the recurrence unchanged, then every state outside [lo_t, hi_t) is
-inf.  End: S-1 if a[S-1] > a[S-2], else S-2.  When the window clips somewhere (not W >= S and
floor(S*(T-1)/T) <= floor(W/2)) and both end states are -inf, no path stays inside the band: status 1.
A window that never clips gives oracle/forced_align_np.py's results, its "both end states -inf: follow
the recurrence" case included; beam_size=None is that unbanded restatement.  Each frame is sliced to its
window, so a lattice costs O(T*W) time and memory and lattices of hundreds of thousands of frames check.
"""
import numpy as np

NEG_INF = np.float32(-np.inf)


def windows(T, S, beam_size=None):
    """(lo, hi) int64 [T] of the band of beam_size around the diagonal (None: [0, S) in every frame), and
    whether it clips in some frame."""
    if beam_size is None:
        return np.zeros(T, np.int64), np.full(T, S, np.int64), False
    W = int(beam_size)
    lo = np.maximum(0, S * np.arange(T, dtype=np.int64) // T - W // 2)
    hi = np.minimum(lo + W, S)
    return lo, hi, not (W >= S and S * (T - 1) // T <= W // 2)


def forced_align_band_np(lp, targets, blank=0, beam_size=None):
    """lp float32 [T, V], targets int [L] (no blank, T >= L + repeats).  Returns (state path int32 [T],
    paths int32 [T], scores float32 [T], final score float32, status); status 1 (outputs zero, final NaN)
    when no path stays inside a band that clips."""
    lp = np.ascontiguousarray(lp, dtype=np.float32)
    tg = np.asarray(targets, dtype=np.int64)
    T = lp.shape[0]
    S = 2 * tg.shape[0] + 1
    ext = np.full(S, blank, np.int64)
    ext[1::2] = tg
    # move 2 is allowed into an odd state v >= 3 whose label differs from the one two states down
    allow2 = np.zeros(S, bool)
    allow2[3::2] = ext[3::2] != ext[1:-2:2]
    lo_t, hi_t, clips = windows(T, S, beam_size)
    bp = np.zeros((T, int((hi_t - lo_t).max())), np.int8)   # bp[t, v - lo_t]
    # virtual start state 0 with score 0: frame 0 is an ordinary frame after it.  prev holds the scores of
    # the previous window [plo, phi); every state outside it is -inf
    prev, plo, phi = np.zeros(1, np.float32), 0, 1
    for t in range(T):
        lo, hi = int(lo_t[t]), int(hi_t[t])
        seg = np.full(hi - lo + 2, NEG_INF, np.float32)   # previous scores of the states lo-2 .. hi-1
        a, b = max(lo - 2, plo), min(hi, phi)
        if b > a:
            seg[a - lo + 2:b - lo + 2] = prev[a - plo:b - plo]
        x0 = seg[2:]
        x1 = seg[1:-1]
        x2 = np.where(allow2[lo:hi], seg[:-2], NEG_INF).astype(np.float32)
        j2 = (x2 > x1) & (x2 > x0)
        j1 = (x1 > x0) & (x1 > x2)
        best = np.where(j2, x2, np.where(j1, x1, x0))
        bp[t, :hi - lo] = np.where(j2, 2, np.where(j1, 1, 0))
        prev = (best + lp[t, ext[lo:hi]]).astype(np.float32)
        plo, phi = lo, hi

    def score(v):
        return prev[v - plo] if plo <= v < phi else NEG_INF
    e1, e2 = score(S - 1), score(S - 2)
    if clips and not e1 > NEG_INF and not e2 > NEG_INF:
        return np.zeros(T, np.int32), np.zeros(T, np.int32), np.zeros(T, np.float32), np.float32(np.nan), 1
    v = S - 1 if (S == 1 or e1 > e2) else S - 2
    final = score(v)
    states = np.empty(T, np.int32)
    for t in range(T - 1, -1, -1):
        states[t] = v
        v -= int(bp[t, v - lo_t[t]])
    paths = ext[states].astype(np.int32)
    scores = lp[np.arange(T), paths]
    return states, paths, scores, np.float32(final), 0


def forced_align_band_batch_np(lp, t_off, labels, l_off, blank=0, beam_size=None):
    """Flat batch (the C-ABI layout) -> (states, paths, scores, final [B], status [B]); status 2 for a label
    outside [0, V) or equal to the blank, 1 for T_b < L_b + R_b or no path inside the band, 3 for a NaN or
    +inf log-prob (the kernels' statuses).  Outputs of a lattice with a non-zero status stay 0 (final NaN)."""
    B = len(t_off) - 1
    n = int(t_off[-1])
    states = np.zeros(n, np.int32)
    paths = np.zeros(n, np.int32)
    scores = np.zeros(n, np.float32)
    final = np.full(B, np.nan, np.float32)
    status = np.zeros(B, np.int32)
    for b in range(B):
        a, e = int(t_off[b]), int(t_off[b + 1])
        tg = np.asarray(labels[int(l_off[b]):int(l_off[b + 1])], dtype=np.int64)
        R = int((tg[1:] == tg[:-1]).sum())
        x = lp[a:e]
        if ((tg < 0) | (tg >= lp.shape[1]) | (tg == blank)).any():
            status[b] = 2
            continue
        if e - a < tg.shape[0] + R:
            status[b] = 1
            continue
        if np.isnan(x).any() or np.isposinf(x).any():
            status[b] = 3
            continue
        st, pa, sc, f, status[b] = forced_align_band_np(x, tg, blank, beam_size)
        if status[b] == 0:
            states[a:e], paths[a:e], scores[a:e], final[b] = st, pa, sc, f
    return states, paths, scores, final, status
