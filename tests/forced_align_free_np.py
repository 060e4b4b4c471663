"""CPU restatement of CTC forced alignment with free ends (kab_plan_create_ctc_free), in float32 numpy,
O(T*S).  The recurrence of oracle/forced_align_np.py (torchaudio's) with two changes:

    free start: a virtual state -1 with score 0 in EVERY frame is state 0's x1 and state 1's x2; the
                select and tie rules are unchanged (state 0 takes it iff 0 > a[0], state 1 iff 0 > a[1]
                and 0 > a[0]).  Frame 0 gets today's initialisation.  The walk stops at state -1: the
                frame where it gets there is t0.
    free end:   the maximum of a_t[v] over every frame t and v in {S-1, S-2}; a tie between frames picks
                the later frame, within a frame S-2.  Every candidate -inf: (T-1, S-2).  That frame is t1.

Outputs: frames outside [t0, t1] get state -1, label blank and score lp[t, blank]; final = a_t1[v_end].
L = 0: every frame is outside and final = 0.  The statuses are forced_align_np's.
"""
import numpy as np

NEG_INF = np.float32(-np.inf)


def forced_align_free_np(lp, targets, blank=0):
    """lp float32 [T, V], targets int [L] (no blank, T >= L + repeats).
    Returns (states int32 [T], paths int32 [T], scores float32 [T], final float32, (t0, t1))."""
    lp = np.ascontiguousarray(lp, dtype=np.float32)
    tg = np.asarray(targets, dtype=np.int64)
    T = lp.shape[0]
    L = tg.shape[0]
    S = 2 * L + 1
    rows = np.arange(T)
    if L == 0:
        return (np.full(T, -1, np.int32), np.full(T, blank, np.int32), lp[rows, blank].copy(), np.float32(0.0),
                (T, -1))
    ext = np.full(S, blank, np.int64)
    ext[1::2] = tg
    allow2 = np.zeros(S, bool)
    allow2[3::2] = ext[3::2] != ext[1:-2:2]
    bp = np.zeros((T, S), np.int8)
    prev = np.full(S, NEG_INF, np.float32)
    m = [NEG_INF, NEG_INF]          # running maxima of states S-1, S-2
    f = [T - 1, T - 1]              # ... and their (latest) frames
    zero = np.float32(0.0)
    for t in range(T):
        x0 = prev
        x1 = np.concatenate([[zero], prev[:-1]]).astype(np.float32)          # state 0: the virtual -1
        x2 = np.where(allow2, np.concatenate([[NEG_INF, NEG_INF], prev[:-2]])[:S], NEG_INF).astype(np.float32)
        x2[1] = zero                                                           # state 1: the virtual -1
        j2 = (x2 > x1) & (x2 > x0)
        j1 = (x1 > x0) & (x1 > x2)
        best = np.where(j2, x2, np.where(j1, x1, x0))
        bp[t] = np.where(j2, 2, np.where(j1, 1, 0))
        prev = (best + lp[t, ext]).astype(np.float32)
        for k, v in enumerate((S - 1, S - 2)):
            if prev[v] >= m[k]:
                m[k], f[k] = prev[v], t
    top = m[0] > m[1] or (m[0] == m[1] and f[0] > f[1])
    v = S - 1 if top else S - 2
    t1 = f[0] if top else f[1]
    final = m[0] if top else m[1]
    states = np.full(T, -1, np.int32)
    t0 = 0
    for t in range(t1, -1, -1):
        states[t] = v
        v -= int(bp[t, v])
        if v < 0:
            t0 = t
            break
    inside = states >= 0
    paths = np.where(inside, ext[np.maximum(states, 0)], blank).astype(np.int32)
    scores = lp[rows, paths]
    return states, paths, scores, np.float32(final), (t0, t1)


def forced_align_free_batch_np(lp, t_off, labels, l_off, blank=0):
    """Flat batch (the C-ABI layout) -> (states, paths, scores, final [B], status [B]); the statuses of
    forced_align_batch_np (2 bad label, 1 T_b < L_b + R_b, 3 NaN or +inf)."""
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
        states[a:e], paths[a:e], scores[a:e], final[b], _ = forced_align_free_np(x, tg, blank)
    return states, paths, scores, final, status
