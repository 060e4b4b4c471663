"""CTC forced alignment of the default plans at the geometry and value edges of their two kernels,
kab_warp_ctc_kernel (S <= 248) and the single-CTA band kernel in CTC mode (249 <= S <= 3296), bit for
bit against the restatement (oracle/forced_align_np.py) and torchaudio's CPU forced_align wherever the
chosen end state is finite.

Geometry.  Warp kernel: lanes of K = 2/4/6/8 states for S <= 62/124/186/248, whose backpointer words
hold fpw = 8/4/2 frames.  Band kernel: a ring of ceil((S + 32) / 104) warps -- 3 at S = 249, 3 -> 4
at 279 | 281, 16 -> 17 at 1631 | 1633 (two lattices per SM -> one), 32 at 3295 -- whose width is the
plan's largest.  Frame counts: tight (T = L + R), tight + 1, T mod fpw, T mod 8 (band frame groups),
T mod 16 (16-frame emission stages, V <= 64) and one long lattice per kernel.
Values: Dirichlet log-probs; ties everywhere (quantised, all-zero and constant rows: the select rule
and the S-2 end rule on the whole path); the climbing path (distinct labels, T = L: move 2 in every
frame, across every warp's 104 slots -- the ghost lanes' worst case); repeated labels everywhere
(T = 2L - 1); -inf masks, a -inf blank column, a -inf row and both end states -inf.
The CPU half (the cases against live torchaudio) is in test_forced_align_oracle.py."""
import functools
import zlib

import numpy as np
import pytest

from oracle.forced_align_np import forced_align_batch_np, forced_align_np
from tests.test_gpu_forced_align import _flat, _torchaudio

pytestmark = pytest.mark.gpu

WARP, BAND, GENERIC, WIDE = 0, 1, 2, 3
KAB_BAND_KERNEL_CTA = 1

# (S, V, blank, T kind, content).  T kind: "tight" (T = L + R), "tight1" (L + R + 1), (res, mod) -- the
# smallest T >= 1.25 (L + R) with T = res mod mod -- or a frame count.
WARP_CASES = [
    # S = 3 (K = 2, fpw = 8), T = 1 among them
    (3, 2, 0, "tight", "zero"), (3, 5, 4, "tight", "dir"), (3, 32, 0, "tight1", "q1"), (3, 65, 64, (7, 8), "const"),
    (3, 129, 7, (0, 16), "q2"), (3, 512, 511, (1, 8), "mask"),
    # S = 61 | 63: K 2 -> 4, fpw 8 -> 4
    (61, 2, 1, "tight", "allrep"), (61, 5, 0, "tight", "climb"), (61, 32, 31, (0, 8), "q2"), (61, 64, 0, (7, 8), "zero"),
    (61, 65, 32, (15, 16), "dir"), (61, 129, 0, (1, 8), "mask"),
    (63, 5, 4, "tight", "allrep"), (63, 32, 0, "tight", "climb"), (63, 64, 63, (0, 4), "q1"), (63, 65, 0, (3, 4), "const"),
    (63, 512, 255, (1, 16), "dir"), (63, 2, 0, "tight1", "zero"),
    # S = 123 | 125: K 4 -> 6, fpw 4 -> 2
    (123, 32, 7, "tight", "blankmask"), (123, 129, 128, (1, 4), "q2"), (123, 5, 2, (0, 16), "mask"),
    (123, 64, 0, "tight1", "end"), (123, 65, 32, (3, 4), "dir"), (123, 2, 0, (3, 4), "const"),
    (125, 65, 64, "tight", "climb"), (125, 32, 0, (0, 2), "zero"), (125, 2, 1, "tight", "allrep"), (125, 512, 0, (15, 16), "row"),
    # S = 185 | 187: K 6 -> 8
    (185, 5, 0, (1, 2), "q1"), (185, 129, 64, "tight", "climb"), (185, 32, 31, "tight1", "const"), (185, 64, 32, (0, 16), "mask"),
    (187, 512, 511, "tight", "blankmask"), (187, 64, 63, (1, 2), "dir"), (187, 5, 4, "tight", "allrep"), (187, 65, 0, (15, 16), "end"),
    # S = 247: the largest warp lattice, one of them long
    (247, 32, 0, "tight", "climb"), (247, 129, 0, (0, 2), "q2"), (247, 2, 0, "tight", "allrep"), (247, 64, 0, 2500, "dir"),
    (247, 5, 2, "tight1", "zero"), (247, 65, 32, (1, 16), "row"),
]
BAND_CASES = [
    # S = 249: the smallest band lattice (3 warps)
    (249, 32, 0, "tight", "climb"), (249, 5, 0, (7, 8), "q1"), (249, 129, 128, (0, 8), "dir"), (249, 2, 1, "tight", "allrep"),
    (249, 512, 255, (1, 16), "mask"),
    # S = 279 | 281: S + 32 crosses 3 * 104 (3 -> 4 warps)
    (279, 65, 0, (1, 8), "zero"), (279, 64, 63, "tight", "blankmask"), (279, 32, 7, (15, 16), "q2"),
    (281, 65, 64, "tight", "climb"), (281, 5, 4, "tight1", "const"), (281, 129, 0, (0, 16), "end"),
    # S = 1631 | 1633: 16 -> 17 warps
    (1631, 32, 0, "tight", "climb"), (1631, 2, 0, "tight", "allrep"), (1631, 512, 511, (7, 8), "q1"), (1631, 64, 32, (0, 8), "row"),
    (1633, 32, 31, "tight", "climb"), (1633, 129, 64, 5000, "dir"), (1633, 5, 2, (1, 16), "zero"), (1633, 65, 0, (7, 8), "mask"),
    # S = 3295: the largest band lattice (32 warps)
    (3295, 32, 0, "tight", "climb"), (3295, 5, 0, "tight", "allrep"), (3295, 64, 63, (15, 16), "q2"),
    (3295, 512, 0, (0, 8), "end"), (3295, 129, 7, "tight", "blankmask"),
]
EDGE_CASES = WARP_CASES + BAND_CASES
# V = 1025: the warp and band kernels on the compact copy of the lattices' columns (DESIGN.md 3.9c)
COMPACT_CASES = [
    (3, 1025, 1024, "tight", "dir"), (61, 1025, 1024, (7, 8), "q2"), (247, 1025, 1024, "tight1", "zero"),
    (3295, 1025, 1024, "tight", "climb"),
    (63, 1025, 0, "tight", "climb"), (187, 1025, 0, (1, 2), "allrep"), (1633, 1025, 0, (0, 8), "q1"),
    (125, 1025, 512, (15, 16), "end"), (249, 1025, 512, "tight", "climb"), (281, 1025, 512, (15, 16), "mask"),
]
CONTENTS = ("dir", "q1", "q2", "zero", "const", "climb", "allrep", "mask", "blankmask", "row", "end")


def case_id(case):
    S, V, blank, t_kind, content = case
    tk = t_kind if isinstance(t_kind, str) else (f"T{t_kind}" if isinstance(t_kind, int) else f"{t_kind[0]}m{t_kind[1]}")
    return f"S{S}-V{V}-b{blank}-{tk}-{content}"


def _targets(rng, L, V, blank, mode):
    """L labels: "rand" (adjacent repeats with p = 0.2), "norep" (no two adjacent equal) or "allrep" (one
    label L times).  With a nonzero blank, label 0 is among them.  V > 512: from 300 ids (0 and V - 1 among
    them), which keeps every lattice on the compact copy."""
    pool = np.delete(np.arange(V), blank)
    if V > 512:
        keep = [x for x in (0, V - 1) if x != blank]
        pool = np.concatenate([keep, rng.choice(np.setdiff1d(pool, keep), 300 - len(keep), replace=False)])
    if len(pool) == 1 or mode == "allrep":
        assert mode != "norep" or L == 1
        return np.full(L, 0 if blank != 0 else pool[0], np.int32)
    if mode == "norep":
        tg = np.empty(L, np.int64)
        for i in range(L):
            tg[i] = rng.choice(pool)
            while i and tg[i] == tg[i - 1]:
                tg[i] = rng.choice(pool)
    else:
        tg = rng.choice(pool, L)
        rep = rng.random(L) < 0.2
        rep[0] = False
        for i in np.flatnonzero(rep):
            tg[i] = tg[i - 1]
    if blank != 0 and not (tg == 0).any():
        tg[L // 2] = 0   # (norep: no neighbour is 0)
    return tg.astype(np.int32)


def make_case(case):
    """(log-probs float32 [T, V], targets int32 [L]) of one case, from a seed derived from the case."""
    S, V, blank, t_kind, content = case
    assert S % 2 == 1 and content in CONTENTS
    rng = np.random.default_rng(zlib.crc32(repr(case).encode()))
    L = (S - 1) // 2
    tg = _targets(rng, L, V, blank, {"climb": "norep", "blankmask": "norep", "allrep": "allrep"}.get(content, "rand"))
    need = L + int((tg[1:] == tg[:-1]).sum())
    if t_kind == "tight":
        T = need
    elif t_kind == "tight1":
        T = need + 1
    elif isinstance(t_kind, int):
        T = t_kind
        assert T >= need
    else:
        res, mod = t_kind
        T = max(need, int(1.25 * need))
        T += (res - T) % mod
    if content == "zero":
        lp = np.zeros((T, V), np.float32)
    elif content == "const":   # one value per row: every path of a frame adds the same numbers, in the same order
        lp = np.repeat(rng.uniform(-4.0, 0.0, (T, 1)).astype(np.float32), V, axis=1)
    else:
        lp = np.log(rng.dirichlet(np.full(V, 0.5), T)).astype(np.float32)
        if content in ("q1", "q2"):
            q = 1 if content == "q1" else 2
            lp = (np.round(lp * q) / q).astype(np.float32)
        elif content == "mask":
            lp[rng.random(lp.shape) < rng.uniform(0.05, 0.1)] = -np.inf
        elif content == "blankmask":
            lp[:, blank] = -np.inf
        elif content == "row":
            lp[T // 2] = -np.inf
        elif content == "end":
            lp[-1, blank] = -np.inf
            lp[-1, tg[-1]] = -np.inf
    return np.ascontiguousarray(lp), tg


@functools.lru_cache(maxsize=None)
def case_data(case):
    """make_case and the restatement's (states, paths, scores, final) of it."""
    lp, tg = make_case(case)
    return lp, tg, forced_align_np(lp, tg, case[2])


def _fpw(S):
    return 8 if S <= 62 else (4 if S <= 124 else 2)


def _band_nw(S):
    return -(-(S + 32) // 104)


def _align256(x):
    return -(-x // 256) * 256


def _backptr_bytes(Ts, Ss):
    """Backpointer bytes of a default CTC plan of warp and band lattices: a 128-byte word-row per fpw frames for
    a warp lattice; for a band lattice one row of (26 NW + 15) & ~15 bytes per frame, NW the plan's widest ring."""
    nw = max((_band_nw(S) for S in Ss if S > 248), default=0)
    nbp = (26 * nw + 15) & ~15
    return sum(_align256(-(-T // _fpw(S)) * 128) if S <= 248 else _align256(T * nbp) for T, S in zip(Ts, Ss))


def _owner(S, v):
    """Which lane or warp computes state v (for a failure message)."""
    if S <= 248:
        K = 2 if S <= 62 else (4 if S <= 124 else (6 if S <= 186 else 8))
        return f"warp kernel K={K}, lane {v // K + 1}"
    return f"band kernel NW={_band_nw(S)}, warp {v // 104}, lane {6 + (v % 104) // 4}"


def _same(got, want, what, S=None, states=None):
    """Byte equality of two 4-byte arrays; the message names the first differing frame (and its state's owner)."""
    got, want = np.ascontiguousarray(got), np.ascontiguousarray(want)
    assert got.shape == want.shape and got.dtype.itemsize == want.dtype.itemsize == 4, (what, got.shape, want.shape)
    if got.tobytes() == want.tobytes():
        return
    i = int(np.flatnonzero(got.view(np.int32) != want.view(np.int32))[0])
    where = f", state {int(states[i])} ({_owner(S, int(states[i]))})" if states is not None else ""
    raise AssertionError(f"{what}: first difference at frame {i} of {len(got)}{where}: {got[i]!r}, expected {want[i]!r}")


def _check_lattice(out, b, a, e, tg, ref, what, S, lp=None, blank=None):
    """Lattice b (frames [a, e)) of a run's outputs against the restatement's ref, and torchaudio's CPU
    forced_align (given lp) where the chosen end state is finite."""
    path, labs, scores, final, status = out
    states, paths, sc, f = ref
    assert status[b] == 0, (what, int(status[b]))
    _same(path[a:e], states, f"{what}: states", S, states)
    _same(labs[a:e], paths, f"{what}: token ids", S, states)
    _same(scores[a:e], sc, f"{what}: scores", S, states)
    assert final[b].tobytes() == f.tobytes(), (what, final[b], f)
    F = _torchaudio() if lp is not None else None
    if F is not None and np.isfinite(f):
        import torch
        p, s = F.forced_align(torch.from_numpy(lp)[None], torch.from_numpy(tg)[None], blank=blank)
        _same(labs[a:e], p[0].numpy(), f"{what}: token ids vs torchaudio", S, states)
        _same(scores[a:e], s[0].numpy(), f"{what}: scores vs torchaudio", S, states)


@pytest.fixture(scope="module")
def kab():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from kokoro_align_b200 import align
    return align


@pytest.fixture(scope="module")
def alone(kab):
    """case -> (outputs, info) of the case's lattice alone in its own plan (computed once)."""
    cache = {}

    def run(case):
        if case not in cache:
            lp, tg, _ = case_data(case)
            T = lp.shape[0]
            with kab.AlignPlan.ctc([0, T], tg, [0, len(tg)], case[1], case[2]) as plan:
                cache[case] = (plan.run_host(lp), plan.info)
        return cache[case]
    return run


@pytest.mark.parametrize("case", EDGE_CASES, ids=[case_id(c) for c in EDGE_CASES])
def test_edge_alone(alone, case):
    """Each edge lattice alone in its plan: routing (class, backpointer bytes, band kernel) and outputs."""
    S, V, blank = case[:3]
    lp, tg, ref = case_data(case)
    T = lp.shape[0]
    out, info = alone(case)
    _check_lattice(out, 0, 0, T, tg, ref, case_id(case), S, lp, blank)
    assert list(info.n_class) == ([1, 0, 0, 0] if S <= 248 else [0, 1, 0, 0]), list(info.n_class)
    if S <= 248:
        assert info.backptr_bytes == _align256(-(-T // _fpw(S)) * 128), (info.backptr_bytes, T, _fpw(S))
    else:
        assert info.band_kernel == KAB_BAND_KERNEL_CTA
        assert info.backptr_bytes == _backptr_bytes([T], [S]), (info.backptr_bytes, T, _band_nw(S))


def _with_fillers(cases, V, blank, rng):
    """The cases' lattices with one or two 1-3-frame filler lattices (L = 1) before each one, chosen so that
    the starts t_off * V * 4 mod 16 of consecutive cases cycle through every value they can take at this V.
    Returns (items, index of every case's item)."""
    skews = sorted({(k * V) % 4 for k in range(4)})
    pool = np.delete(np.arange(V), blank)
    items, where, t = [], [], 0
    for i, case in enumerate(cases):
        want = skews[i % len(skews)]
        n = next(n for n in range(1, 7) if ((t + n) * V) % 4 == want)
        for f in ([n] if n <= 3 else [3, n - 3]):
            items.append((np.log(rng.dirichlet(np.ones(V), f)).astype(np.float32), rng.choice(pool, 1).astype(np.int32)))
        t += n
        lp, tg, _ = case_data(case)
        where.append(len(items))
        items.append((lp, tg))
        t += lp.shape[0]
    return items, where


def _groups(cases):
    g = {}
    for c in cases:
        g.setdefault((c[1], c[2]), []).append(c)
    return g


GROUPS = _groups(EDGE_CASES)


@pytest.mark.parametrize("V,blank", list(GROUPS), ids=[f"V{v}-b{b}" for v, b in GROUPS])
def test_vocabulary_plan(kab, alone, V, blank):
    """All edge lattices of a (vocabulary, blank) in one plan, between filler lattices that move their starts
    through every 16-byte skew: outputs byte-equal to the lattices' own plans.  The band lattices all run in
    the ring of the widest one (the S = 249 lattice of V = 32 in the 32 warps of S = 3295)."""
    cases = GROUPS[(V, blank)]
    rng = np.random.default_rng(V * 1000 + blank)
    items, where = _with_fillers(cases, V, blank, rng)
    lp, t_off, labels, l_off = _flat(items)
    starts = {int(t_off[i]) * V % 4 for i in where}
    assert len(starts) == min(len(cases), len({(k * V) % 4 for k in range(4)})), starts
    with kab.AlignPlan.ctc(t_off, labels, l_off, V, blank) as plan:
        out = plan.run_host(lp)
        info = plan.info
    S = 2 * np.diff(l_off) + 1
    assert list(info.n_class) == [int((S <= 248).sum()), int((S > 248).sum()), 0, 0]
    assert info.backptr_bytes == _backptr_bytes(np.diff(t_off).tolist(), S.tolist())
    if (S > 248).any():
        assert info.band_kernel == KAB_BAND_KERNEL_CTA
    rs, rp, rsc, rf, rst = forced_align_batch_np(lp, t_off, labels, l_off, blank)
    assert (out[4] == 0).all() and (rst == 0).all()
    for b in range(len(items)):
        a, e = int(t_off[b]), int(t_off[b + 1])
        if b in where:
            case = cases[where.index(b)]
            one, _ = alone(case)
            for k, name in enumerate(("states", "token ids", "scores")):
                _same(out[k][a:e], one[k], f"{case_id(case)} at t_off {a}: {name} vs its own plan", int(S[b]), one[0])
            assert out[3][b].tobytes() == one[3][0].tobytes(), case_id(case)
        ref = (rs[a:e], rp[a:e], rsc[a:e], rf[b])
        _check_lattice(out, b, a, e, None, ref, f"lattice {b}", int(S[b]))


SHIFTED = [(63, 5, 4, "tight", "allrep"), (187, 65, 0, (15, 16), "end"), (281, 5, 4, "tight1", "const"),
           (1633, 65, 0, (7, 8), "mask"), (249, 129, 128, (0, 8), "dir")]


@pytest.mark.parametrize("case", SHIFTED, ids=[case_id(c) for c in SHIFTED])
def test_same_lattice_at_every_offset(kab, case):
    """One lattice four times in a batch, at starts of every 16-byte skew: byte-identical outputs."""
    S, V, blank = case[:3]
    lp0, tg0, ref = case_data(case)
    items, where = _with_fillers([case] * 4, V, blank, np.random.default_rng(S))
    lp, t_off, labels, l_off = _flat(items)
    assert len({int(t_off[i]) * V % 4 for i in where}) == 4
    with kab.AlignPlan.ctc(t_off, labels, l_off, V, blank) as plan:
        out = plan.run_host(lp)
    for b in where:
        a, e = int(t_off[b]), int(t_off[b + 1])
        _check_lattice(out, b, a, e, tg0, ref, f"{case_id(case)} at t_off {a}", S)


def test_plan_reuse_host_and_torch(kab):
    """One plan run on log-probs A, B, A through run_host and then run_torch: each run equals its own
    reference, so nothing of a run carries over to the next."""
    import torch
    V, blank = 65, 0
    cases = GROUPS[(V, blank)]
    rng = np.random.default_rng(65)
    items, _ = _with_fillers(cases, V, blank, rng)
    lp_a, t_off, labels, l_off = _flat(items)
    lp_b = np.log(rng.dirichlet(np.full(V, 0.5), lp_a.shape[0])).astype(np.float32)
    refs = {id(x): forced_align_batch_np(x, t_off, labels, l_off, blank) for x in (lp_a, lp_b)}
    S = 2 * np.diff(l_off) + 1
    with kab.AlignPlan.ctc(t_off, labels, l_off, V, blank) as plan:
        assert plan.info.n_class[BAND] == int((S > 248).sum()) > 0
        runs = [("run_host", x, plan.run_host(x)) for x in (lp_a, lp_b, lp_a)]
        for x in (lp_a, lp_b, lp_a):
            runs.append(("run_torch", x, tuple(y.cpu().numpy() for y in plan.run_torch(torch.from_numpy(x).cuda()))))
    for k, (how, x, out) in enumerate(runs):
        rs, rp, rsc, rf, rst = refs[id(x)]
        np.testing.assert_array_equal(out[4], rst)
        for b in range(len(items)):
            a, e = int(t_off[b]), int(t_off[b + 1])
            _check_lattice(out, b, a, e, None, (rs[a:e], rp[a:e], rsc[a:e], rf[b]), f"{how} #{k}: lattice {b}", int(S[b]))


COMPACT_GROUPS = _groups(COMPACT_CASES)


@pytest.mark.parametrize("blank", [b for _, b in COMPACT_GROUPS], ids=[f"b{b}" for _, b in COMPACT_GROUPS])
def test_compact_vocabulary(kab, monkeypatch, blank):
    """V = 1025: edge lattices on the compact copy (warp and band classes) against the restatement,
    torchaudio and the KAB_CTC_COMPACT=0 twin of the plan (every lattice on the generic kernel)."""
    from tests.test_gpu_forced_align_vocab import _check3
    V = 1025
    cases = COMPACT_GROUPS[(V, blank)]
    items, where = _with_fillers(cases, V, blank, np.random.default_rng(blank))
    lp, t_off, labels, l_off = _flat(items)
    info, _ = _check3(kab, monkeypatch, lp, t_off, labels, l_off, V, blank)
    S = 2 * np.diff(l_off) + 1
    assert list(info.n_class) == [int((S <= 248).sum()), int((S > 248).sum()), 0, 0]


def test_empty_transcript(kab):
    """L = 0 (S = 1, accepted by the C ABI): state 0 and the blank in every frame, the blank's log-probs as
    scores, and as final score their float32 running sum from 0 in frame order -- alone and among edge
    lattices, including a -inf blank log-prob (final score -inf)."""
    rng = np.random.default_rng(70)
    V, blank = 65, 32

    def empty(T, neginf_at=None):
        lp = np.log(rng.dirichlet(np.ones(V), T)).astype(np.float32)
        if neginf_at is not None:
            lp[neginf_at, blank] = -np.inf
        return lp, np.zeros(0, np.int32)

    def expect(lp):
        f = np.float32(0.0)
        for t in range(lp.shape[0]):
            f = np.float32(f + lp[t, blank])
        T = lp.shape[0]
        return np.zeros(T, np.int32), np.full(T, blank, np.int32), np.ascontiguousarray(lp[:, blank]), f

    for T in (1, 7, 8, 9, 40):
        lp, tg = empty(T)
        ref = expect(lp)
        assert all(x.tobytes() == y.tobytes() for x, y in zip(forced_align_np(lp, tg, blank), ref))
        with kab.AlignPlan.ctc([0, T], tg, [0, 0], V, blank) as plan:
            out = plan.run_host(lp)
            assert list(plan.info.n_class) == [1, 0, 0, 0]
            assert plan.info.backptr_bytes == _align256(-(-T // 8) * 128)
        _check_lattice(out, 0, 0, T, tg, ref, f"L = 0, T = {T}", 1)
    cases = GROUPS[(V, blank)]
    edges = [case_data(c)[:2] for c in cases]
    items = [empty(3), edges[0], empty(17, neginf_at=5), edges[1], empty(1), edges[2], empty(64)]
    lp, t_off, labels, l_off = _flat(items)
    with kab.AlignPlan.ctc(t_off, labels, l_off, V, blank) as plan:
        out = plan.run_host(lp)
        assert plan.info.n_class[WARP] == len(items)
    for b, (x, tg) in enumerate(items):
        a, e = int(t_off[b]), int(t_off[b + 1])
        ref = expect(x) if len(tg) == 0 else case_data(cases[b // 2])[2]
        _check_lattice(out, b, a, e, tg, ref, f"lattice {b} (L = {len(tg)})", 2 * len(tg) + 1)
    assert np.isneginf(out[3][2])
