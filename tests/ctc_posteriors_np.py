"""float64 restatement of the forward-backward posteriors of a CTC state path (kab_plan_ctc_posteriors_device,
DESIGN.md 3.9f).  ext = the blank-interleaved states (S = 2L + 1), move 2 into an odd v >= 3 iff ext[v] !=
ext[v-2], the window [lo_t, hi_t) of tests/forced_align_band_np.py:windows (beam_size=None: [0, S)):

    alpha_0 = lp[0, blank] at 0, lp[0, ext[1]] at 1; alpha_t(v) = lse(alpha_{t-1}(v), alpha_{t-1}(v-1),
    alpha_{t-1}(v-2) if allowed) + lp[t, ext[v]]; beta_{T-1} = 0 at S-1, S-2; beta_t(v) = lse over v' in
    {v, v+1, v+2 if allowed into v'} of beta_{t+1}(v') + lp[t+1, ext[v']]; -inf outside every frame's window.
    log Z = lse(alpha_{T-1}(S-1), alpha_{T-1}(S-2));  gamma_t = exp(alpha_t(p_t) + beta_t(p_t) - log Z).

The passes keep one window of values and store only the value at the path state per frame, so lattices of tens
of thousands of frames check in seconds.  full_alpha_beta keeps everything (small shapes: invariants)."""
import numpy as np

from tests.forced_align_band_np import windows

NEG_INF = -np.inf


def _ext(targets, blank):
    tg = np.asarray(targets, dtype=np.int64)
    S = 2 * tg.shape[0] + 1
    ext = np.full(S, blank, np.int64)
    ext[1::2] = tg
    allow2 = np.zeros(S + 2, bool)   # (two False entries past the end: successors of the last states)
    allow2[3:S:2] = ext[3::2] != ext[1:-2:2]
    return ext, allow2, S


def _lse(*xs):
    r = xs[0]
    for x in xs[1:]:
        r = np.logaddexp(r, x)
    return r


def _slice(vals, vlo, a, b):
    """Values of the states [a, b) from `vals` (states [vlo, vlo + len)), -inf outside."""
    out = np.full(b - a, NEG_INF)
    x, y = max(a, vlo), min(b, vlo + len(vals))
    if y > x:
        out[x - a:y - a] = vals[x - vlo:y - vlo]
    return out


def path_values(lp, targets, path, blank=0, beam_size=None):
    """(fwd [T], bwd [T], log Z): log alpha_t(p_t), log beta_t(p_t) (-inf where p_t is outside the window)."""
    lp = np.asarray(lp, dtype=np.float64)
    T = lp.shape[0]
    ext, allow2, S = _ext(targets, blank)
    lo_t, hi_t, _ = windows(T, S, beam_size)
    path = np.asarray(path, dtype=np.int64)

    def at(vals, vlo, t):
        p = int(path[t])
        return vals[p - vlo] if vlo <= p < vlo + len(vals) else NEG_INF

    fwd, bwd = np.empty(T), np.empty(T)
    lo, hi = int(lo_t[0]), int(hi_t[0])
    a0 = np.full(S, NEG_INF)
    a0[0] = lp[0, blank]
    if S > 1:
        a0[1] = lp[0, ext[1]]
    a = a0[lo:hi].copy()
    fwd[0] = at(a, lo, 0)
    for t in range(1, T):
        plo = lo
        lo, hi = int(lo_t[t]), int(hi_t[t])
        seg = _slice(a, plo, lo - 2, hi)
        a = _lse(seg[2:], seg[1:-1], np.where(allow2[lo:hi], seg[:-2], NEG_INF)) + lp[t, ext[lo:hi]]
        fwd[t] = at(a, lo, t)
    logz = _lse(*_slice(a, lo, S - 2, S)) if S > 1 else a[S - 1 - lo] if lo <= S - 1 < hi else NEG_INF
    lo, hi = int(lo_t[T - 1]), int(hi_t[T - 1])
    b = np.where((np.arange(lo, hi) >= S - 2), 0.0, NEG_INF)
    bwd[T - 1] = at(b, lo, T - 1)
    for t in range(T - 2, -1, -1):
        nlo = lo
        lo, hi = int(lo_t[t]), int(hi_t[t])
        y = b + lp[t + 1, ext[nlo:nlo + len(b)]]
        seg = _slice(y, nlo, lo, hi + 2)
        b = _lse(seg[:-2], seg[1:-1], np.where(allow2[lo + 2:hi + 2], seg[2:], NEG_INF))
        bwd[t] = at(b, lo, t)
    return fwd, bwd, float(logz)


def ctc_posteriors_np(lp, targets, path, blank=0, beam_size=None):
    """(gamma float64 [T], log Z) for the state path `path` (0 where log Z is -inf)."""
    fwd, bwd, logz = path_values(lp, targets, path, blank, beam_size)
    if not logz > NEG_INF:
        return np.zeros(len(fwd)), logz
    return np.exp(fwd + bwd - logz), logz


def ctc_posteriors_batch_np(lp, t_off, labels, l_off, path, status, blank=0, beam_size=None):
    """The flat batch of the C ABI: (posteriors float32 [sum T], rounded and clamped as the device does,
    log_likelihood float64 [B]); a lattice whose status is not 0 gets 0 and NaN."""
    B = len(t_off) - 1
    post = np.zeros(int(t_off[-1]), np.float32)
    ll = np.full(B, np.nan)
    for b in range(B):
        if status[b] != 0:
            continue
        a, e = int(t_off[b]), int(t_off[b + 1])
        g, ll[b] = ctc_posteriors_np(lp[a:e], labels[int(l_off[b]):int(l_off[b + 1])], path[a:e], blank, beam_size)
        post[a:e] = np.clip(g, 0.0, 1.0).astype(np.float32)
    return post, ll


def full_alpha_beta(lp, targets, blank=0, beam_size=None):
    """alpha, beta float64 [T, S] (small shapes), straight from the definitions."""
    lp = np.asarray(lp, dtype=np.float64)
    T = lp.shape[0]
    ext, allow2, S = _ext(targets, blank)
    lo_t, hi_t, _ = windows(T, S, beam_size)
    inwin = (np.arange(S)[None, :] >= lo_t[:, None]) & (np.arange(S)[None, :] < hi_t[:, None])
    al = np.full((T, S), NEG_INF)
    be = np.full((T, S), NEG_INF)
    al[0, 0] = lp[0, blank]
    if S > 1:
        al[0, 1] = lp[0, ext[1]]
    al[0, ~inwin[0]] = NEG_INF
    for t in range(1, T):
        for v in range(S):
            c = [al[t - 1, v]] + ([al[t - 1, v - 1]] if v >= 1 else []) + ([al[t - 1, v - 2]] if allow2[v] else [])
            al[t, v] = _lse(*c) + lp[t, ext[v]] if inwin[t, v] else NEG_INF
    be[T - 1, max(S - 2, 0):] = 0.0
    be[T - 1, ~inwin[T - 1]] = NEG_INF
    for t in range(T - 2, -1, -1):
        for v in range(S):
            c = [be[t + 1, w] + lp[t + 1, ext[w]] for w in (v, v + 1, v + 2)
                 if w < S and (w < v + 2 or allow2[w])]
            be[t, v] = _lse(*c) if inwin[t, v] else NEG_INF
    return al, be
