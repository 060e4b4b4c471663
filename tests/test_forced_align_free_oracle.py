"""The free-ends CTC restatement (tests/forced_align_free_np.py, the reference of kab_plan_create_ctc_free):
on tie-free lattices its final score is the best forced_align_np score over every window of at least L + R
frames, bit for bit, and its path inside the chosen window is that window's forced_align_np path (and
torchaudio's); on tiny lattices a brute force over every free-ends path pins the tie rules."""

import numpy as np
import pytest

from oracle.forced_align_np import forced_align_np
from tests.forced_align_free_np import forced_align_free_batch_np, forced_align_free_np

NEG_INF = np.float32(-np.inf)


def _item(rng, T, L, V, blank, repeat_p=0.3, quant=None, neginf=0.0):
    pool = np.array([x for x in range(V) if x != blank])
    tg = rng.choice(pool, L)
    rep = rng.random(L) < repeat_p
    if L:
        rep[0] = False
    tg[rep] = tg[np.flatnonzero(rep) - 1]
    lp = np.log(rng.dirichlet(np.full(V, 0.5), T)).astype(np.float32)
    if quant:
        lp = (np.round(lp * quant) / quant).astype(np.float32)
    if neginf:
        lp[rng.random(lp.shape) < neginf] = -np.inf
    return lp, tg.astype(np.int32)


def _repeats(tg):
    return int((tg[1:] == tg[:-1]).sum())


def _windows_best(lp, tg, blank):
    """max over windows [t0, t1] (>= L + R frames) of forced_align_np's final score, with its windows."""
    T, need = lp.shape[0], len(tg) + _repeats(tg)
    best, where = NEG_INF, []
    for t0 in range(T):
        for t1 in range(t0 + need - 1, T):
            f = forced_align_np(lp[t0:t1 + 1], tg, blank)[3]
            if f > best:
                best, where = f, [(t0, t1)]
            elif f == best:
                where.append((t0, t1))
    return best, where


def _torchaudio():
    try:
        import torch
        import torchaudio.functional as F
        return torch, F
    except Exception:  # noqa: BLE001 (torchaudio is optional here)
        return None, None


def _check_against_windows(lp, tg, blank):
    T = lp.shape[0]
    states, paths, scores, final, (t0, t1) = forced_align_free_np(lp, tg, blank)
    best, where = _windows_best(lp, tg, blank)
    assert final.tobytes() == np.float32(best).tobytes()
    assert len(where) == 1 and where[0] == (t0, t1)  # tie-free: one best window
    s, p, sc, f = forced_align_np(lp[t0:t1 + 1], tg, blank)
    np.testing.assert_array_equal(states[t0:t1 + 1], s)
    np.testing.assert_array_equal(paths[t0:t1 + 1], p)
    assert scores[t0:t1 + 1].tobytes() == sc.tobytes()
    out = np.r_[0:t0, t1 + 1:T]
    assert (states[out] == -1).all() and (paths[out] == blank).all()
    assert scores[out].tobytes() == lp[out, blank].tobytes()
    torch, F = _torchaudio()
    if torch is not None:
        ta_p, ta_s = F.forced_align(torch.from_numpy(lp[t0:t1 + 1])[None], torch.from_numpy(tg.astype(np.int32))[None],
                                    blank=blank)
        np.testing.assert_array_equal(ta_p[0].numpy(), p)
        assert ta_s[0].numpy().tobytes() == sc.tobytes()
    return t0, t1


@pytest.mark.parametrize("seed", range(12))
def test_free_ends_is_best_window(seed):
    """Tie-free random lattices (continuous log-probs, repeats, blank ids first, last and in the middle)."""
    rng = np.random.default_rng(seed)
    V = 6
    blank = (0, V - 1, 3)[seed % 3]
    L = int(rng.integers(1, 5))
    tg_probe = rng.integers(0, 2, L)
    T = L + int(tg_probe.sum()) + int(rng.integers(0, 9))
    lp, tg = _item(rng, T, L, V, blank)
    _check_against_windows(lp, tg, blank)


def _planted(T, a, b, tg, V, blank, rng):
    """Log-probs that favour the transcript in frames [a, b) and the blank elsewhere."""
    lp = np.log(rng.dirichlet(np.full(V, 0.5), T)).astype(np.float32)
    for r in (slice(0, a), slice(b, T)):  # outside: every label unlikely, the blank likely
        lp[r] = np.float32(-20.0) - rng.random((lp[r].shape[0], V)).astype(np.float32)
        lp[r, blank] = np.float32(-0.01)
    n = b - a
    for k, lab in enumerate(tg):
        t = a + (k * n) // len(tg)
        lp[t, lab] = np.float32(-0.001 * (k + 1))
    return lp


def test_window_edges():
    """t0 = 0 and t1 = T-1, and a window of exactly L + R frames."""
    rng = np.random.default_rng(5)
    V, blank = 7, 0
    tg = np.array([1, 2, 2, 3], np.int32)
    need = len(tg) + _repeats(tg)
    # whole recording: every frame strongly favours its planted label
    T = need
    lp = np.full((T, V), np.float32(-20.0), np.float32)
    for t, lab in enumerate([1, 2, 0, 2, 3]):
        lp[t, lab] = np.float32(-0.01 * (t + 1))
    t0, t1 = _check_against_windows(lp, tg, blank)
    assert (t0, t1) == (0, T - 1)
    # a window of exactly L + R frames in the middle of blank-favouring frames
    T = 14
    lp = np.log(rng.dirichlet(np.full(V, 0.5), T)).astype(np.float32)
    lp[:, blank] = np.float32(-0.05) - np.arange(T, dtype=np.float32) * np.float32(1e-4)
    for t, lab in zip(range(5, 10), [1, 2, 0, 2, 3]):
        lp[t] = np.float32(-30.0)
        lp[t, lab] = np.float32(-0.02)
    t0, t1 = _check_against_windows(lp, tg, blank)
    assert (t0, t1) == (5, 9)


def test_planted_spans():
    rng = np.random.default_rng(11)
    V, blank = 9, 4
    tg = np.array([1, 2, 3, 5, 6, 7], np.int32)
    lp = _planted(40, 12, 27, tg, V, blank, rng)
    t0, t1 = _check_against_windows(lp, tg, blank)
    assert 12 <= t0 and t1 < 27


def test_empty_transcript():
    lp = np.log(np.random.default_rng(0).dirichlet(np.ones(5), 7)).astype(np.float32)
    states, paths, scores, final, _ = forced_align_free_np(lp, np.zeros(0, np.int32), 2)
    assert (states == -1).all() and (paths == 2).all()
    assert scores.tobytes() == lp[:, 2].tobytes() and final == 0.0


# ---------------------------------------------------------------- brute force over every free-ends path

def _all_paths(T, S, allow2):
    """Every free-ends state sequence: (t0, t1, states of frames t0..t1), a CTC path from state 0 or 1
    at t0 to S-1 or S-2 at t1."""
    for t0 in range(T):
        for t1 in range(t0, T):
            n = t1 - t0 + 1

            def rec(seq):
                if len(seq) == n:
                    if seq[-1] >= S - 2:
                        yield tuple(seq)
                    return
                v = seq[-1]
                for mv in (0, 1, 2):
                    u = v + mv
                    if u >= S or (mv == 2 and not allow2[u]):
                        continue
                    yield from rec(seq + [u])
            for s0 in (0, 1):
                if s0 < S:
                    yield from ((t0, t1, p) for p in rec([s0]))


def _path_score(lp, ext, t0, seq):
    acc = np.float32(0.0)
    for k, v in enumerate(seq):
        acc = np.float32(acc + lp[t0 + k, ext[v]])
    return acc


@pytest.mark.parametrize("seed", range(10))
def test_brute_force_ties(seed):
    """Quantised log-probs (many exact ties), -inf masks: the restatement's final score is the best
    path score.  Where that best path is unique, the restatement picks it; where several tie, its pick
    is one of them and follows the rules: the later end frame, S-2 within a frame, and a select that
    keeps the earlier frame (or state) on a tie."""
    rng = np.random.default_rng(100 + seed)
    V, blank = 4, seed % 4
    L = int(rng.integers(1, 3))
    T = int(rng.integers(L + 1, L + 5))
    lp, tg = _item(rng, T, L, V, blank, quant=1, neginf=0.15 if seed % 2 else 0.0)
    if T < L + _repeats(tg):
        return
    S = 2 * L + 1
    ext = np.full(S, blank, np.int64)
    ext[1::2] = tg
    allow2 = np.zeros(S, bool)
    allow2[3::2] = ext[3::2] != ext[1:-2:2]
    allow2[1] = True
    states, paths, scores, final, (t0, t1) = forced_align_free_np(lp, tg, blank)
    cands = [(_path_score(lp, ext, a, p), a, b, p) for a, b, p in _all_paths(T, S, allow2)]
    best = max(c[0] for c in cands)
    assert final.tobytes() == np.float32(best).tobytes()
    if best == NEG_INF:
        return
    winners = [c for c in cands if c[0] == best]
    mine = (t0, t1, tuple(int(x) for x in states[t0:t1 + 1]))
    assert mine in [(a, b, p) for _, a, b, p in winners]
    # end rule: the latest end frame among the winners, then S-2
    assert t1 == max(b for _, _, b, _ in winners)
    ends = {p[-1] for _, _, b, p in winners if b == t1}
    if S - 2 in ends:
        assert states[t1] == S - 2


def test_end_tie_rules_exact():
    """Hand-made ties: the later of two equal end frames; S-2 over S-1 within a frame; the earlier start."""
    blank, tg = 0, np.array([1], np.int32)  # S = 3, end states 2 and 1
    # frame 1 and 3 both give the same best score through label 1; the later frame wins
    lp = np.array([[-9, -1, -9], [-9, -9, -9], [-9, -1, -9]], np.float32)
    lp = np.vstack([np.full((1, 3), -9, np.float32), lp])  # T = 4
    lp[1] = [-9, -1, -9]
    lp[3] = [-9, -1, -9]
    lp[2] = [-9, -9, -9]
    states, paths, scores, final, (t0, t1) = forced_align_free_np(lp, tg, blank)
    assert final == np.float32(-1) and t1 == 3 and states[3] == 1 and t0 == 3
    # within a frame S-1 (blank after the label) equal to S-2: S-2
    lp = np.array([[-1, -1, -9], [0, -9, -9]], np.float32)  # a_1[2] = -1 + 0 = -1 = a_0[1] ... and a_1[1] = -10
    states, paths, scores, final, (t0, t1) = forced_align_free_np(lp, tg, blank)
    assert final == np.float32(-1)
    assert (t1, states[t1]) == (1, 2)  # the later frame beats the earlier S-2
    lp = np.array([[-9, 0, -9]], np.float32)
    states, _, _, final, (t0, t1) = forced_align_free_np(lp, tg, blank)
    assert final == 0 and (t0, t1) == (0, 0) and states[0] == 1


def test_all_end_candidates_neg_inf():
    """Every end candidate -inf: the end is (T-1, S-2), status 0, and the walk follows the recurrence."""
    T, V, blank = 6, 4, 0
    tg = np.array([1, 2], np.int32)
    lp = np.log(np.random.default_rng(3).dirichlet(np.ones(V), T)).astype(np.float32)
    lp[:, 2] = -np.inf
    states, paths, scores, final, (t0, t1) = forced_align_free_np(lp, tg, blank)
    assert final == NEG_INF and t1 == T - 1 and states[T - 1] == 2 * len(tg) - 1
    st, pa, sc, fi, status = forced_align_free_batch_np(lp, np.array([0, T]), tg, np.array([0, 2]), blank)
    assert status[0] == 0 and fi[0] == NEG_INF
    np.testing.assert_array_equal(st, states)


def test_batch_statuses():
    rng = np.random.default_rng(8)
    V, blank = 6, 1
    items = [_item(rng, 9, 3, V, blank), _item(rng, 2, 3, V, blank), _item(rng, 7, 2, V, blank)]
    items[2][0][3, 0] = np.nan
    bad = (np.log(rng.dirichlet(np.ones(V), 5)).astype(np.float32), np.array([blank, 2], np.int32))
    items.append(bad)
    lp = np.concatenate([x for x, _ in items])
    t_off = np.concatenate([[0], np.cumsum([x.shape[0] for x, _ in items])])
    l_off = np.concatenate([[0], np.cumsum([len(t) for _, t in items])])
    labels = np.concatenate([t for _, t in items])
    st, pa, sc, fi, status = forced_align_free_batch_np(lp, t_off, labels, l_off, blank)
    assert list(status) == [0, 1, 3, 2]
    s0 = forced_align_free_np(items[0][0], items[0][1], blank)
    np.testing.assert_array_equal(st[:9], s0[0])
    assert fi[0] == s0[3]
