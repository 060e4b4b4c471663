"""CPU restatement of CTC forced alignment as torchaudio.functional.forced_align computes it
(torchaudio 2.x, libtorchaudio/forced_align/cpu/compute.cpp), in float32 numpy.  The reference the
CTC plans (kab_plan_create_ctc) are checked against.

    ext = [blank, t0, blank, t1, ..., blank]          S = 2L+1; the blank id is arbitrary
    frame 0:  a[0] = lp[0, blank], a[1] = lp[0, t0]   (a virtual start state 0 with score 0)
    frame t:  x0 = a[v], x1 = a[v-1],
              x2 = a[v-2] for an odd v >= 3 with ext[v] != ext[v-2], else -inf
              j = 2 if x2 > x1 and x2 > x0, elif x1 > x0 and x1 > x2: 1, else 0
              a'[v] = fl32(x_j + lp[t, ext[v]])       (the select is on the previous scores)
    end:      S-1 if a[S-1] > a[S-2] else S-2          (a tie picks S-2)
    paths[t] = ext[v_t], scores[t] = lp[t, paths[t]]

The tie rule is torchaudio's: x1 == x2 > x0 keeps x0, which is not a maximum.  torchaudio also
prunes the cells that cannot reach the end; those only ever feed each other, so the full lattice
gives the same path whenever the chosen end state has a finite score.  When both end states are
-inf, torchaudio walks back through backpointers it never wrote (its result is undefined); this
restatement, like the kernels, follows the recurrence.
"""
import numpy as np

NEG_INF = np.float32(-np.inf)


def forced_align_np(lp, targets, blank=0):
    """lp float32 [T, V], targets int [L] (no blank, T >= L + repeats).
    Returns (state path int32 [T], paths int32 [T], scores float32 [T], final score float32).
    L = 0 (S = 1, which the C ABI accepts and torchaudio does not): the path is all blank and the
    final score is the float32 running sum of lp[:, blank] from 0, in frame order."""
    lp = np.ascontiguousarray(lp, dtype=np.float32)
    tg = np.asarray(targets, dtype=np.int64)
    T = lp.shape[0]
    S = 2 * tg.shape[0] + 1
    ext = np.full(S, blank, np.int64)
    ext[1::2] = tg
    # move 2 is allowed into an odd state v >= 3 whose label differs from the one two states down
    allow2 = np.zeros(S, bool)
    allow2[3::2] = ext[3::2] != ext[1:-2:2]
    bp = np.zeros((T, S), np.int8)
    # virtual start state 0 with score 0: frame 0 is an ordinary frame after it
    prev = np.full(S, NEG_INF, np.float32)
    prev[0] = np.float32(0.0)
    for t in range(T):
        x0 = prev
        x1 = np.concatenate([[NEG_INF], prev[:-1]]).astype(np.float32)
        x2 = np.where(allow2, np.concatenate([[NEG_INF, NEG_INF], prev[:-2]])[:S], NEG_INF).astype(np.float32)
        j2 = (x2 > x1) & (x2 > x0)
        j1 = (x1 > x0) & (x1 > x2)
        best = np.where(j2, x2, np.where(j1, x1, x0))
        bp[t] = np.where(j2, 2, np.where(j1, 1, 0))
        prev = (best + lp[t, ext]).astype(np.float32)
    v = S - 1 if (S == 1 or prev[S - 1] > prev[S - 2]) else S - 2
    final = prev[v]
    states = np.empty(T, np.int32)
    for t in range(T - 1, -1, -1):
        states[t] = v
        v -= int(bp[t, v])
    paths = ext[states].astype(np.int32)
    scores = lp[np.arange(T), paths]
    return states, paths, scores, np.float32(final)


def forced_align_batch_np(lp, t_off, labels, l_off, blank=0):
    """Flat batch (the C-ABI layout) -> (states, paths, scores, final [B], status [B]); status 2 for
    a label outside [0, V) or equal to the blank, 1 for T_b < L_b + R_b, 3 for a NaN or +inf
    log-prob (the kernels' statuses)."""
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
        states[a:e], paths[a:e], scores[a:e], final[b] = forced_align_np(x, tg, blank)
    return states, paths, scores, final, status
