"""Lane-level numpy emulation of the warp kernel's checkpointed best path (DESIGN.md 2 and 3.1):
a values-only forward pass (maximum of the masked predecessors, then one add) that stores the score
row every C frames, and a backtrack that walks blocks of C frames from the last one back.  For each
block the 32 lanes of the warp hold the 3C+1 checkpoint states below the path state at the block's
last frame (one state per lane, superset loaded one block ahead), recompute the block's C frames
with the post-add select of the kernel, keep the 2-bit codes in one word per lane and walk them
with a shuffle of the owner lane's word.  The kernel runs this scheme for its K = 6 and K = 8 lattices
(K = 2 and 4 keep backpointers); the emulation covers every K, since the scheme does not depend on it.

This file checks the SCHEME -- checkpoint row layout, the window arithmetic, the halo of the
bottom lanes (a shuffle-up past lane 0 returns the lane's own value), rows past the lattice read by
a partial last block, the codes of a blank lane (label select with a -inf move-2 candidate) --
against the C oracle, bit for bit.  It also asserts that every value the walk reads is the value of
the full forward pass.  It is a development aid that runs without a GPU; no product code depends
on it.

    python tools/emulate_warp_ckpt.py            # about fifty shapes, max_move 4, 3 and 2, falling paths
"""
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

C = 8          # frames per checkpoint block (KAB_CKPT_C)
NINF = np.float32(-np.inf)
F32 = np.float32


def k_class(S):
    """States per lane of the warp kernel (kab_api.cu)."""
    return 2 if S <= 62 else (4 if S <= 124 else (6 if S <= 186 else 8))


def ckpt_stride(S, K):
    """Floats per checkpoint row (kab_ckpt_stride)."""
    return (K * ((S + K - 1) // K) + 3) & ~3


def _shfl_up(x, d):
    y = x.copy()
    y[d:] = x[:-d]
    return y


def _label_sel(a0, a1, a2, a3):
    """kab_label_sel: value and 2-bit code (the move) per lane."""
    m01 = np.maximum(a0, a1)
    best = np.maximum(np.maximum(m01, a2), a3)
    ph = m01 != best
    pl = np.where(ph, a2, a0) != best
    return best, pl.astype(np.uint32) | (ph.astype(np.uint32) << np.uint32(1))


def emulate(lp, labels, max_move=4, junk_seed=0):
    """(best_path, best_labels, best_scores, final_score, status) of one warp-class lattice with
    labels in 1..V-1; status 1 = no active end state.  Rows past T (read by a partial last block)
    are filled with junk, NaN and infinities included."""
    lp = np.ascontiguousarray(lp, dtype=np.float32)
    T, V = lp.shape
    labels = np.asarray(labels, dtype=np.int64)
    L = len(labels)
    S = 2 * L + 1
    assert S <= 248 and T >= 1 and (L == 0 or (labels.min() >= 1 and labels.max() < V))
    K = k_class(S)
    MM = max_move < 4
    mm = [F32(0.0) if j < max_move else NINF for j in range(4)]
    col = np.zeros(S, np.int64)
    col[1::2] = labels

    # ---- forward, values only; full[i] is kept only to check what the walk reads
    RS = ckpt_stride(S, K)
    nb = (T + C - 1) // C
    ck = np.full((nb, RS), np.nan, np.float32)  # never-written entries are NaN: reading one shows
    full = np.empty((T, S), np.float32)
    s = np.full(S, NINF, np.float32)
    s[0] = 0.0  # frame -1: the virtual start
    mask_mm = (lambda x, j: x + mm[j]) if MM else (lambda x, j: x)
    with np.errstate(invalid="ignore", over="ignore"):
        for i in range(T):
            pad = np.concatenate([np.full(3, NINF, np.float32), s])
            x1, x2, x3 = mask_mm(pad[2:-1], 1), mask_mm(pad[1:-2], 2), mask_mm(pad[:-3], 3)
            m = np.maximum(np.maximum(s, x1), x3)
            m[1::2] = np.maximum(m[1::2], x2[1::2])
            s = (m + lp[i, col]).astype(np.float32)
            full[i] = s
            if (i + 1) % C == 0:
                ck[(i + 1) // C - 1, :S] = s
    active = np.nonzero(s > NINF)[0]
    if len(active) == 0:
        return None, None, None, np.float32(np.nan), 1
    v = int(active[-1])
    final = s[v]

    # ---- backtrack over blocks of C frames, 32 lanes
    rng = np.random.default_rng(junk_seed)
    junk = rng.normal(0, 50, (C, V)).astype(np.float32)
    junk.flat[rng.integers(0, junk.size, 3)] = [np.nan, np.inf, -np.inf]
    rows = np.concatenate([lp, junk])
    lanes = np.arange(32)

    def win_load(row, sb):  # unconditional loads, row and state clamped to 0
        u0, u1 = np.maximum(sb + lanes, 0), np.maximum(sb + 32 + lanes, 0)
        assert (u1 < S).all()  # never past the last state: sb + 63 == ve
        return ck[max(row, 0), u0].copy(), ck[max(row, 0), u1].copy()

    path = np.empty(T, np.int32)
    labs = np.empty(T, np.int32)
    scores = np.empty(T, np.float32)
    ve = v
    sb = ve - 63
    r0, r1 = win_load((T - 1) // C - 1, sb)
    with np.errstate(invalid="ignore", over="ignore"):
        for b in range((T - 1) // C, -1, -1):
            f0, n = b * C, min(C, T - b * C)
            base = ve - 3 * C
            wi = base + lanes - sb
            assert (wi[:3 * C + 1] >= 0).all() and (wi[:3 * C + 1] < 64).all()
            u = base + lanes
            x = np.where(u < 0, NINF, np.where(wi >= 32, r1[wi & 31], r0[wi & 31])).astype(np.float32)
            if f0 == 0:  # frame -1: the virtual start
                x = np.where(u == 0, F32(0), NINF).astype(np.float32)
            sb = ve - 63
            r0, r1 = win_load(b - 2, sb)
            blank = (u & 1) == 0
            ucol = np.where((u > 0) & (u < S) & ~blank, col[np.clip(u, 0, S - 1)], 0)
            cw = np.zeros(32, np.uint32)
            xs = []
            for j in range(C):
                e = rows[f0 + j, ucol]
                h1, h2, h3 = _shfl_up(x, 1), _shfl_up(x, 2), _shfl_up(x, 3)
                a0, a1, a2, a3 = x + e, h1 + e, h2 + e, h3 + e
                a2 = np.where(blank, NINF, mask_mm(a2, 2))
                x, code = _label_sel(a0, mask_mm(a1, 1), a2, mask_mm(a3, 3))
                x = x.astype(np.float32)
                cw |= code << np.uint32(2 * j)
                xs.append(x)
            if n < C:
                cw &= np.uint32((1 << (2 * n)) - 1)
            wl = 3 * C
            mw = 0
            for j in range(C - 1, -1, -1):
                assert 0 <= wl <= 3 * C
                if j < n:  # the cone is exact: what the walk reads is the full forward pass's value
                    assert xs[j][wl].tobytes() == full[f0 + j, base + wl].tobytes(), (f0 + j, base + wl)
                w = int(cw[wl])
                mw |= w & (3 << (2 * j))
                wl -= (w >> (2 * j)) & 3
            for j in range(n):  # lane j: ve minus the moves of the frames above j
                above = mw >> min(2 * j + 2, 2 * C)
                v_j = ve - (bin(above & 0x55555555).count("1") + 2 * bin(above & 0xAAAAAAAA).count("1"))
                path[f0 + j] = v_j
                labs[f0 + j] = col[v_j]
                scores[f0 + j] = rows[f0 + j, col[v_j]]
            ve = base + wl
    assert ve == 0  # frame -1: the virtual start
    return path, labs, scores, final, 0


def check(lp, labels, max_move=4, junk_seed=0):
    """Emulation against the C oracle, bit for bit (path, labels, scores, final score, status)."""
    from oracle import ctc_oracle
    T = lp.shape[0]
    t_off = np.array([0, T], np.int64)
    l_off = np.array([0, len(labels)], np.int64)
    rp, rl, rs, rf, rst = ctc_oracle.ctc_best_path_batch(lp, t_off, np.asarray(labels, np.int32), l_off,
                                                         1000, max_move)
    path, labs, scores, final, status = emulate(lp, labels, max_move, junk_seed)
    assert status == rst[0], (status, rst[0])
    if status:
        return
    np.testing.assert_array_equal(path, rp)
    np.testing.assert_array_equal(labs, rl)
    assert scores.tobytes() == rs.tobytes()
    assert np.float32(final).tobytes() == rf[0].tobytes()


def falling_lattice(T, V=39, seed=0):
    """S = 3T + 1: the only path to the forced end state S - 1 moves 3 in every frame."""
    rng = np.random.default_rng(seed)
    L = (3 * T) // 2
    labels = rng.integers(1, V, L).astype(np.int32)
    lp = -np.abs(rng.normal(0, 3, (T, V))).astype(np.float32)
    return lp, labels


def main():
    from kokoro_align_b200 import synth
    n = 0
    for T in (1, C - 1, C, C + 1, 2 * C + 1, 861):
        for L in (0, 1, 30, 61, 92, 123):
            if 2 * L + 1 > 3 * T + 1:
                continue
            lp, labels = synth.make_lattice_exact(T, L, 39, seed=T * 131 + L, planted=True)
            for mmv in (4, 3, 2):
                check(lp, labels, mmv, junk_seed=n)
                n += 1
    for T in (2, 8, 16, 40, 80):
        lp, labels = falling_lattice(T, seed=T)
        check(lp, labels)
        n += 1
    print(f"{n} lattices: emulation == C oracle, bit for bit")


if __name__ == "__main__":
    main()
