"""Writes tests/golden/forced_align_golden.npz: CTC forced-alignment cases with the outputs of
torchaudio.functional.forced_align (CPU), the reference implementation CTC users run today.

    python tests/golden/make_forced_align_golden.py

Every case holds <name>__lp (float32 [T, V]), <name>__targets (int32 [L]), <name>__blank, and the
expected <name>__paths / __scores (torchaudio's) plus <name>__states (extended-state path) and
<name>__final (DP score of the end state) from oracle/forced_align_np.py, which is asserted to agree
with torchaudio here.  Cases whose end states are both -inf (<name>__torchaudio == 0) hold the
restatement's outputs only: torchaudio's traceback reads backpointers it never wrote there.
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

from oracle.forced_align_np import forced_align_np  # noqa: E402

OUT = os.path.join(HERE, "forced_align_golden.npz")


def _targets(rng, V, blank, L, repeat_p=0.0):
    pool = np.array([x for x in range(V) if x != blank])
    tg = rng.choice(pool, L)
    for i in range(1, L):
        if rng.random() < repeat_p:
            tg[i] = tg[i - 1]
    return tg.astype(np.int32)


def _lp(rng, T, V, quant=None):
    lp = np.log(rng.dirichlet(np.full(V, 0.5), T)).astype(np.float32)
    if quant:
        lp = (np.round(lp * quant) / quant).astype(np.float32)   # many exact ties
    return lp


def cases():
    rng = np.random.default_rng(20261020)
    out = []

    def add(name, lp, tg, blank):
        out.append((name, np.ascontiguousarray(lp, np.float32), np.asarray(tg, np.int32), int(blank)))

    def slack(tg, extra):
        return len(tg) + int((tg[1:] == tg[:-1]).sum()) + extra

    # ties: log-probs on a 1/2 or 1/4 grid, blank at 0, V-1 and in the middle
    for k in range(12):
        V = 5 if k < 6 else 9
        blank = [0, V - 1, V // 2][k % 3]
        tg = _targets(rng, V, blank, int(rng.integers(2, 9)), repeat_p=0.3)
        add(f"ties{k}_V{V}_b{blank}", _lp(rng, slack(tg, int(rng.integers(0, 12))), V, quant=2 if k % 2 else 4), tg, blank)
    # tight lattices: T == L + R, with repeats
    for k in range(4):
        V, blank = 7, [0, 6, 3, 2][k]
        tg = _targets(rng, V, blank, int(rng.integers(3, 20)), repeat_p=0.4)
        add(f"tight{k}_b{blank}", _lp(rng, slack(tg, 0), V, quant=4 if k % 2 else None), tg, blank)
    # label 0 with a blank that is not 0
    for k, blank in enumerate([3, 31]):
        tg = _targets(rng, 32, blank, 12, repeat_p=0.2)
        tg[::3] = 0
        add(f"label0_{k}_b{blank}", _lp(rng, slack(tg, 15), 32), tg, blank)
    # -inf entries (masking), the end still reachable
    for k in range(4):
        V, blank = 32, [0, 31, 16, 5][k]
        tg = _targets(rng, V, blank, 20, repeat_p=0.2)
        lp = _lp(rng, slack(tg, 30), V, quant=2 if k % 2 else None)
        lp[rng.random(lp.shape) < 0.15] = -np.inf
        lp[:, blank] = np.where(rng.random(lp.shape[0]) < 0.05, -np.inf, lp[:, blank])
        add(f"neginf{k}_b{blank}", lp, tg, blank)
    # both end states -inf
    for k in range(3):
        V, blank = 6, [0, 5, 2][k]
        tg = _targets(rng, V, blank, 6, repeat_p=0.3)
        lp = _lp(rng, slack(tg, 5), V)
        if k == 0:
            lp[:] = -np.inf
        else:
            lp[-1, :] = -np.inf
        add(f"deadend{k}_b{blank}", lp, tg, blank)
    # S just under / over the warp (248) and band (3296) limits; V in {5, 32, 512}
    for L, V, extra in [(123, 32, 40), (124, 32, 40), (1647, 5, 60), (1648, 5, 60)]:
        blank = int(rng.integers(0, V))
        tg = _targets(rng, V, blank, L, repeat_p=0.1)
        add(f"S{2 * L + 1}_V{V}_b{blank}", _lp(rng, slack(tg, extra), V, quant=4), tg, blank)
    for k, (L, extra) in enumerate([(20, 30), (124, 10)]):
        blank = [0, 511][k]
        tg = _targets(rng, 512, blank, L, repeat_p=0.1)
        add(f"V512_S{2 * L + 1}_b{blank}", _lp(rng, slack(tg, extra), 512), tg, blank)
    return out


def main():
    import torch
    import torchaudio.functional as F
    arrays = {}
    for name, lp, tg, blank in cases():
        states, paths, scores, final = forced_align_np(lp, tg, blank)
        ta = bool(np.isfinite(final))
        if ta:
            p, s = F.forced_align(torch.from_numpy(lp)[None], torch.from_numpy(tg)[None], blank=blank)
            p, s = p[0].numpy().astype(np.int32), s[0].numpy()
            assert np.array_equal(p, paths) and s.tobytes() == scores.tobytes(), name
        arrays.update({f"{name}__lp": lp, f"{name}__targets": tg, f"{name}__blank": np.int32(blank),
                       f"{name}__paths": paths, f"{name}__scores": scores, f"{name}__states": states,
                       f"{name}__final": np.float32(final), f"{name}__torchaudio": np.int32(ta)})
    np.savez_compressed(OUT, **arrays)
    print(f"{OUT}: {len(arrays) // 8} cases, {os.path.getsize(OUT)} bytes")


if __name__ == "__main__":
    main()
