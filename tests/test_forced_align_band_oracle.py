"""The banded CTC restatement (tests/forced_align_band_np.py, the reference of kab_plan_create_ctc_band):
a window that never clips gives the unbanded restatement byte for byte; on tiny lattices the DP value and
the dead-band status agree with a brute force over every CTC path inside the window; the window's cell
count is parallel.cells_eval's."""
import numpy as np
import pytest

from oracle.forced_align_np import forced_align_batch_np, forced_align_np
from tests.forced_align_band_np import forced_align_band_batch_np, forced_align_band_np, windows
from tests.test_forced_align_oracle import CASES

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


def _covering_beams(T, S):
    """The smallest beam whose window never clips, and a wider one."""
    W = S
    while not (W >= S and S * (T - 1) // T <= W // 2):
        W += 1
    return [W, 2 * W + 7]


@pytest.mark.parametrize("name,case", CASES, ids=[n for n, _ in CASES])
def test_covering_beam_is_unbanded_golden(name, case):
    lp, tg, blank = case["lp"], case["targets"], int(case["blank"])
    T, S = lp.shape[0], 2 * len(tg) + 1
    for W in [None] + _covering_beams(T, S):
        states, paths, scores, final, status = forced_align_band_np(lp, tg, blank, W)
        assert status == 0
        np.testing.assert_array_equal(states, case["states"])
        np.testing.assert_array_equal(paths, case["paths"])
        assert scores.tobytes() == case["scores"].tobytes()
        assert final.tobytes() == case["final"].tobytes()


@pytest.mark.parametrize("seed", range(6))
def test_covering_beam_is_unbanded_random(seed):
    """Random lattices (repeats, ties, -inf masks, both end states -inf): any covering beam gives
    oracle/forced_align_np.py's outputs byte for byte, and the batch forms agree."""
    rng = np.random.default_rng(seed)
    items = []
    for k in range(8):
        L = int(rng.integers(0, 60))
        T = L + int(rng.integers(L // 3 + 1, 80))
        lp, tg = _item(rng, T, L, 12, seed % 12, quant=2 if k % 3 == 0 else None, neginf=0.05 if k % 3 == 1 else 0.0)
        if k == 2 and L:
            lp[-1, seed % 12] = -np.inf
            lp[-1, tg[-1]] = -np.inf
        items.append((lp, tg))
    for lp, tg in items:
        T, S = lp.shape[0], 2 * len(tg) + 1
        want = forced_align_np(lp, tg, seed % 12)
        for W in _covering_beams(T, S):
            got = forced_align_band_np(lp, tg, seed % 12, W)
            assert got[4] == 0
            for a, b in zip(got[:4], want):
                assert np.asarray(a).tobytes() == np.asarray(b).tobytes()
    t_off = np.concatenate([[0], np.cumsum([x[0].shape[0] for x in items])]).astype(np.int64)
    l_off = np.concatenate([[0], np.cumsum([len(x[1]) for x in items])]).astype(np.int64)
    lp = np.concatenate([x[0] for x in items])
    labels = np.concatenate([x[1] for x in items]).astype(np.int32)
    big = 10 * int(lp.shape[0])
    for a, b in zip(forced_align_band_batch_np(lp, t_off, labels, l_off, seed % 12, big),
                    forced_align_batch_np(lp, t_off, labels, l_off, seed % 12)):
        assert a.tobytes() == b.tobytes()


def _brute(lp, tg, blank, W):
    """Best in-band path score ending at S-1 and at S-2 (float32 sums in frame order; -inf: none)."""
    T = lp.shape[0]
    S = 2 * len(tg) + 1
    ext = np.full(S, blank, np.int64)
    ext[1::2] = tg
    lo, hi, _ = windows(T, S, W)
    best = {S - 1: NEG_INF, S - 2: NEG_INF}

    def walk(t, v, acc):
        if not lo[t] <= v < hi[t]:
            return
        acc = np.float32(acc + lp[t, ext[v]])
        if t == T - 1:
            if v in best:
                best[v] = max(best[v], acc)
            return
        for mv in (0, 1, 2):
            u = v + mv
            if u >= S or (mv == 2 and (u % 2 == 0 or u < 3 or ext[u] == ext[u - 2])):
                continue
            walk(t + 1, u, acc)
    for v0 in range(min(S, 2)):   # from the virtual start state 0: stay (blank) or move to the first label
        walk(0, v0, np.float32(0.0))
    return best, ext


@pytest.mark.parametrize("seed", range(40))
def test_brute_force_tiny(seed):
    """S <= 9, T <= 8, every beam 1 .. S + 2: final_score is the best in-band path's float32 sum at the
    chosen end state, the returned path is an in-band CTC path with that sum, and status 1 exactly when the
    window clips and no in-band path ends with a finite score.  The DP value is that maximum because float32
    rounding is monotone -- except at torchaudio's tie x1 == x2 > x0, which keeps x0, so the log-probs here
    are continuous (no finite ties; -inf masks stay).  Ties are checked against the unbanded restatement."""
    rng = np.random.default_rng(100 + seed)
    L = int(rng.integers(1, 5))
    V, blank = 5, seed % 5
    lp, tg = _item(rng, 1, L, V, blank, repeat_p=0.4)
    R = int((tg[1:] == tg[:-1]).sum())
    T = int(rng.integers(L + R, 9))
    lp, _ = _item(rng, T, 0, V, blank, neginf=0.15 if seed % 2 else 0.0)
    S = 2 * L + 1
    for W in range(1, S + 3):
        best, ext = _brute(lp, tg, blank, W)
        states, paths, scores, final, status = forced_align_band_np(lp, tg, blank, W)
        _, _, clips = windows(T, S, W)
        e1, e2 = best[S - 1], best[S - 2]
        if clips and not e1 > NEG_INF and not e2 > NEG_INF:
            assert status == 1, (W, e1, e2)
            continue
        assert status == 0
        v = S - 1 if e1 > e2 else S - 2
        assert states[-1] == v
        assert final.tobytes() == np.float32(best[v]).tobytes(), (W, final, best[v])
        if np.isfinite(final):   # (-inf: a covering window follows the recurrence, as unbanded)
            lo, hi, _ = windows(T, S, W)
            assert ((states >= lo) & (states < hi)).all()
            assert states[0] in (0, 1) and set(np.diff(states).tolist()) <= {0, 1, 2}
            acc = np.float32(0.0)
            for t in range(T):
                acc = np.float32(acc + lp[t, ext[states[t]]])
            assert acc.tobytes() == final.tobytes()
        np.testing.assert_array_equal(paths, ext[states])


@pytest.mark.parametrize("T,L,W", [(1, 0, 1), (5, 2, 1), (50, 20, 7), (300, 120, 40), (1000, 333, 1000),
                                   (997, 400, 73), (4000, 1900, 3264), (12345, 3700, 1000)])
def test_cells_match_parallel_cells_eval(T, L, W):
    from kokoro_align_b200 import parallel
    lo, hi, clips = windows(T, 2 * L + 1, W)
    assert int((hi - lo).sum()) == parallel.cells_eval(T, L, W)
    assert (hi > lo).all()


def test_band_lost_in_batch():
    """A path planted far above the diagonal with every other cell -inf: lost in a narrow band (status 1,
    final NaN), found in a covering one; statuses 2 and 3 are unchanged."""
    V, blank, L = 6, 0, 10
    tg = (np.arange(L) % 5 + 1).astype(np.int32)
    T = 60
    lp = np.full((T, V), -np.inf, np.float32)
    lp[:L, tg] = np.float32(-1.0)        # labels in the first L frames, then blanks
    lp[np.arange(L), tg] = np.float32(-0.5)
    lp[L:, blank] = np.float32(-0.25)
    lp2 = lp.copy()
    lp2[3, 2] = np.nan
    items = [(lp, tg), (lp, tg), (lp2, tg), (lp, np.array([1, 0, 2], np.int32))]
    t_off = np.concatenate([[0], np.cumsum([x[0].shape[0] for x in items])]).astype(np.int64)
    l_off = np.concatenate([[0], np.cumsum([len(x[1]) for x in items])]).astype(np.int64)
    flat = np.concatenate([x[0] for x in items])
    labels = np.concatenate([x[1] for x in items]).astype(np.int32)
    st, pa, sc, f, status = forced_align_band_batch_np(flat, t_off, labels, l_off, blank, 4)
    assert status.tolist() == [1, 1, 3, 2] and np.isnan(f).all()
    st, pa, sc, f, status = forced_align_band_batch_np(flat, t_off, labels, l_off, blank, 100)
    assert status.tolist() == [0, 0, 3, 2]
    want = forced_align_np(lp, tg, blank)
    assert st[:T].tobytes() == want[0].tobytes() and f[0].tobytes() == want[3].tobytes()
