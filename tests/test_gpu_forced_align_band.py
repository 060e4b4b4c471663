"""Banded CTC forced alignment on the B200 (kab_plan_create_ctc_band, beam_size): every lattice bit for bit
against the banded restatement (tests/forced_align_band_np.py) -- states, token ids, scores, final score and
status -- across the band kernel's geometry (NW = 1 .. 32 warps, recycled ring chunks), window shapes, label
and value edges, vocabularies, the windowed generic kernel, routing and backpointer sizes, covering beams
(byte-identical to the long-form plans), band-lost statuses, planted paths at real size and the entry points."""
import numpy as np
import pytest

from tests.forced_align_band_np import forced_align_band_batch_np, windows
from tests.test_gpu_forced_align import _flat

pytestmark = pytest.mark.gpu

CLS_WARP, CLS_BAND, CLS_GENERIC, CLS_WIDE = 0, 1, 2, 3


@pytest.fixture(scope="module")
def kab():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from kokoro_align_b200 import align
    return align


def _targets(rng, L, V, blank, repeat_p=0.2, pool=None):
    pool = np.array([x for x in range(V) if x != blank]) if pool is None else np.asarray(pool)
    tg = rng.choice(pool, L)
    rep = rng.random(L) < repeat_p
    rep[0] = False
    tg[rep] = tg[np.flatnonzero(rep) - 1]
    return tg.astype(np.int32)


def _random_lp(rng, T, V, quant=None, neginf=0.0):
    lp = np.log(rng.dirichlet(np.full(V, 0.5), T)).astype(np.float32)
    if quant:
        lp = (np.round(lp * quant) / quant).astype(np.float32)
    if neginf:
        lp[rng.random(lp.shape) < neginf] = -np.inf
    return lp


def _planted_path(T, tg, amp=0.0, cycles=1.0, shift=0):
    """A CTC state path that follows the diagonal S*(t+1)/T plus a drift amp*sin(2 pi cycles t / T) (zero at
    both ends) and `shift` states, as closely as the CTC moves allow.  Returns the states [T]."""
    S = 2 * len(tg) + 1
    ext = np.zeros(S, np.int64)
    ext[1::2] = tg
    t = np.arange(T)
    goal = np.clip(np.floor(S * (t + 1) / T + amp * np.sin(2 * np.pi * cycles * t / T)).astype(np.int64) + shift, 0, S - 1)
    states = np.empty(T, np.int64)
    v = 0
    for i in range(T):
        if goal[i] > v:
            two = v + 2 <= goal[i] and (v + 2) % 2 == 1 and v + 2 >= 3 and ext[v + 2] != ext[v]
            v += 2 if two else 1
        states[i] = v
    assert v >= S - 2, "planted path cannot reach the end (construction)"
    return states


def _planted_lp(rng, states, tg, V, blank, bonus=8.0, mask=False):
    """Emissions that favour the planted path's token in every frame (log_softmax of Gaussian logits plus a
    bonus; mask: every other column -inf, so the planted label sequence is the only finite one)."""
    S = 2 * len(tg) + 1
    ext = np.full(S, blank, np.int64)
    ext[1::2] = tg
    T = len(states)
    tok = ext[states]
    if mask:
        lp = np.full((T, V), -np.inf, np.float32)
        lp[np.arange(T), tok] = -rng.random(T).astype(np.float32)
        return lp
    x = rng.standard_normal((T, V))
    x[np.arange(T), tok] += bonus
    x -= x.max(axis=1, keepdims=True)
    return (x - np.log(np.exp(x).sum(axis=1, keepdims=True))).astype(np.float32)


def _nbp(W, S):
    nw = -(-(min(W, S) + 32) // 104)
    return (26 * nw + 15) & ~15


def _a256(x):
    return -(-x // 256) * 256


def _cells(T, S, W):
    lo, hi, _ = windows(int(T), int(S), W)
    return int((hi - lo).sum())


def _run(kab, lp, t_off, labels, l_off, V, blank, W, torch_run=False):
    with kab.AlignPlan.ctc(t_off, labels, l_off, V, blank, beam_size=W) as plan:
        if torch_run:
            import torch
            out = tuple(x.cpu().numpy() for x in plan.run_torch(torch.from_numpy(lp).cuda()))
        else:
            out = plan.run_host(lp)
        return out, plan.info


def _check(kab, lp, t_off, labels, l_off, V, blank, W, out=None):
    """Plan outputs vs the banded restatement, bit for bit; returns (outputs, info, reference status)."""
    info = None
    if out is None:
        out, info = _run(kab, lp, t_off, labels, l_off, V, blank, W)
    path, labs, scores, final, status = out
    rs, rp, rsc, rf, rst = forced_align_band_batch_np(lp, t_off, labels, l_off, blank, W)
    np.testing.assert_array_equal(status, rst)
    for b in range(len(t_off) - 1):
        if rst[b] != 0:
            assert np.isnan(final[b]), f"lattice {b}"
            continue
        a, e = int(t_off[b]), int(t_off[b + 1])
        np.testing.assert_array_equal(path[a:e], rs[a:e], err_msg=f"lattice {b}")
        np.testing.assert_array_equal(labs[a:e], rp[a:e], err_msg=f"lattice {b}")
        assert scores[a:e].tobytes() == rsc[a:e].tobytes(), f"lattice {b}"
        assert final[b].tobytes() == rf[b].tobytes(), f"lattice {b}"
    return out, info, rst


# ---- band-kernel geometry: NW = 1 (W <= 72) .. 2, 16 -> 17 (two CTAs per SM up to 16), 32; 3265 -> generic
GEOM_W = [1, 2, 5, 6, 7, 72, 73, 1000, 1632, 1633, 3264, 3265]


@pytest.mark.parametrize("W", GEOM_W)
def test_band_geometry(kab, W):
    rng = np.random.default_rng(1000 + W)
    V, blank = 32, 3
    # a lattice wider than the beam whose planted path drifts within the band, and one of random emissions
    L = max(40, int(0.7 * W))
    T = int(L * 3.2) + 7
    tg = _targets(rng, L, V, blank)
    amp = max(0.0, W / 2 - 4) * 0.8
    states = _planted_path(T, tg, amp=min(amp, T / 8), cycles=1.5)
    items = [(_planted_lp(rng, states, tg, V, blank), tg)]
    tg2 = _targets(rng, L, V, blank, repeat_p=0.3)
    items.append((_random_lp(rng, T + 3, V, quant=2), tg2))
    lp, t_off, labels, l_off = _flat(items)
    out, info, rst = _check(kab, lp, t_off, labels, l_off, V, blank, W)
    assert rst[0] == 0 or W < 5
    Ts, Ss = np.diff(t_off), 2 * np.diff(l_off) + 1
    assert all(windows(int(t), int(s), W)[2] for t, s in zip(Ts, Ss))   # every window clips
    if W <= 3264:
        assert info.n_class[CLS_BAND] == 2, list(info.n_class)
        nbp = _nbp(W, int(Ss.max()))
        assert info.backptr_bytes == sum(_a256(int(t) * nbp) for t in Ts)
    else:
        assert info.n_class[CLS_GENERIC] == 2, list(info.n_class)
        assert info.backptr_bytes == sum(_a256(int(t) * min(W, int(s))) for t, s in zip(Ts, Ss))
    assert info.cells_eval == sum(_cells(t, s, W) for t, s in zip(Ts, Ss))


# ---- window shapes and label edges
def test_window_shapes(kab):
    """Windows that clip at the bottom (early frames), at the top (late frames) and at both; S <= 248 with a
    window that clips (band, not warp); S >> R (chunks recycle many times); T mod 8 in {0, 1, 7}; tight
    T = L + R."""
    rng = np.random.default_rng(7)
    V, blank = 32, 0
    items = []
    for L, T, amp in ((100, 330, 10.0), (120, 241, 0.0), (123, 385, 6.0), (2000, 6400, 30.0), (3000, 9601, 20.0),
                      (900, 2999, 25.0), (60, 128, 3.0), (61, 129, 3.0), (50, 135, 4.0)):
        tg = _targets(rng, L, V, blank)
        st = _planted_path(T, tg, amp=amp, cycles=2.0)
        items.append((_planted_lp(rng, st, tg, V, blank), tg))
    tg = _targets(rng, 400, V, blank, repeat_p=0.3)   # tight: T = L + R
    T = 400 + int((tg[1:] == tg[:-1]).sum())
    items.append((_random_lp(rng, T, V), tg))
    lp, t_off, labels, l_off = _flat(items)
    Ts, Ss = np.diff(t_off), 2 * np.diff(l_off) + 1
    for W in (64, 100, 247):
        out, info, rst = _check(kab, lp, t_off, labels, l_off, V, blank, W)
        warp = sum(not windows(int(t), int(s), W)[2] and s <= 248 for t, s in zip(Ts, Ss))
        assert info.n_class[CLS_WARP] == warp and info.n_class[CLS_BAND] == len(items) - warp
        assert (rst[:-1] == 0).all()


def test_repeats_across_recycled_chunks(kab):
    """Runs of repeated labels everywhere (p = 0.5), on lattices much longer than the ring, so that recycled
    chunks start and end inside repeats: a stale repeat bit would allow a forbidden move 2 (or forbid an allowed
    one).  Planted paths and quantised random emissions (ties)."""
    rng = np.random.default_rng(8)
    V, blank = 5, 2
    items = []
    for L, T in ((3000, 8000), (2500, 7001), (4000, 12007)):
        tg = _targets(rng, L, V, blank, repeat_p=0.5)
        st = _planted_path(T, tg, amp=15.0, cycles=3.0)
        items.append((_planted_lp(rng, st, tg, V, blank, bonus=3.0), tg))
        items.append((_random_lp(rng, T, V, quant=1), tg))
    lp, t_off, labels, l_off = _flat(items)
    for W in (73, 200, 1000):
        out, info, rst = _check(kab, lp, t_off, labels, l_off, V, blank, W)
        assert info.n_class[CLS_BAND] == len(items)
        assert (rst[::2] == 0).all()


@pytest.mark.parametrize("blank_pos", ["first", "middle", "last"])
def test_ties_masks_and_blank(kab, blank_pos):
    """Quantised rows (ties everywhere), 5 % -inf masks, the blank first, in the middle and last."""
    rng = np.random.default_rng(9)
    V = 32
    blank = {"first": 0, "middle": 13, "last": V - 1}[blank_pos]
    items = []
    for k in range(6):
        L = int(rng.integers(300, 1500))
        T = int(L * rng.uniform(2.2, 3.5))
        tg = _targets(rng, L, V, blank, repeat_p=0.3)
        if k % 2 == 0:
            st = _planted_path(T, tg, amp=20.0)
            lp = _planted_lp(rng, st, tg, V, blank, bonus=2.0)
            lp = (np.round(lp * 2) / 2).astype(np.float32)
        else:
            lp = _random_lp(rng, T, V, neginf=0.05)
        items.append((lp, tg))
    lp, t_off, labels, l_off = _flat(items)
    _check(kab, lp, t_off, labels, l_off, V, blank, 150)


# ---- vocabularies
@pytest.mark.parametrize("V,blank", [(5, 0), (32, 31), (129, 64), (512, 511)])
def test_vocabularies(kab, V, blank):
    rng = np.random.default_rng(V)
    items = []
    for L, T in ((800, 2600), (1500, 4801), (3000, 9000)):
        tg = _targets(rng, L, V, blank)
        st = _planted_path(T, tg, amp=40.0)
        items.append((_planted_lp(rng, st, tg, V, blank), tg))
        items.append((_random_lp(rng, T, V, quant=2), _targets(rng, L, V, blank)))
    lp, t_off, labels, l_off = _flat(items)
    out, info, rst = _check(kab, lp, t_off, labels, l_off, V, blank, 400)
    assert info.n_class[CLS_BAND] == len(items) and (rst[::2] == 0).all()


def test_vocabulary_1025_compact_and_generic_twin(kab, monkeypatch):
    """V = 1025 (blank 1024, NeMo): lattices of <= 511 distinct ids run on the band kernel through the compact
    copy, one of 1024 distinct ids on the windowed generic kernel; KAB_CTC_COMPACT=0 sends all of them to the
    generic kernel.  Both plans equal the restatement, byte for byte equal to each other."""
    rng = np.random.default_rng(1025)
    V, blank = 1025, 1024
    items = []
    for L, T, n_ids in ((900, 3000, 300), (1500, 5001, 500), (2000, 6400, 40)):
        pool = rng.choice(np.arange(1024), n_ids, replace=False)
        tg = _targets(rng, L, V, blank, pool=pool)
        st = _planted_path(T, tg, amp=30.0)
        items.append((_planted_lp(rng, st, tg, V, blank), tg))
    tg = rng.permutation(np.arange(1024)).astype(np.int32)   # 1024 distinct labels
    st = _planted_path(4500, tg, amp=30.0)
    items.append((_planted_lp(rng, st, tg, V, blank), tg))
    lp, t_off, labels, l_off = _flat(items)
    W = 500
    out, info, rst = _check(kab, lp, t_off, labels, l_off, V, blank, W)
    assert (rst == 0).all()
    assert info.n_class[CLS_BAND] == 3 and info.n_class[CLS_GENERIC] == 1, list(info.n_class)
    monkeypatch.setenv("KAB_CTC_COMPACT", "0")
    out2, info2, _ = _check(kab, lp, t_off, labels, l_off, V, blank, W)
    assert info2.n_class[CLS_GENERIC] == 4
    Ts, Ss = np.diff(t_off), 2 * np.diff(l_off) + 1
    assert info2.backptr_bytes == sum(_a256(int(t) * min(W, int(s))) for t, s in zip(Ts, Ss))
    for a, b in zip(out, out2):
        assert a.tobytes() == b.tobytes()


# ---- covering beams, statuses
def test_covering_beam_equals_long_form(kab):
    """Warp, band and wide lattices with a beam the windows never clip: the classes and the outputs of the
    long-form plan, byte for byte, including a lattice whose two end states are both -inf (status 0)."""
    rng = np.random.default_rng(11)
    V, blank = 32, 7
    items = []
    for L, T in ((40, 150), (100, 300), (900, 2500), (1600, 4000), (4500, 11000), (5000, 12000)):
        tg = _targets(rng, L, V, blank)
        items.append((_random_lp(rng, T, V), tg))
    lp0, tg0 = items[2]
    lp0[-1, blank] = -np.inf
    lp0[-1, tg0[-1]] = -np.inf
    lp, t_off, labels, l_off = _flat(items)
    W = 10 ** 6
    with kab.AlignPlan.ctc(t_off, labels, l_off, V, blank, long_form=True) as plan:
        want = plan.run_host(lp)
        want_cls = list(plan.info.n_class)
    out, info, rst = _check(kab, lp, t_off, labels, l_off, V, blank, W)
    assert list(info.n_class) == want_cls and want_cls[CLS_WIDE] == 2, want_cls
    assert rst[2] == 0 and np.isneginf(out[3][2])
    for a, b in zip(out, want):
        assert a.tobytes() == b.tobytes()


def test_band_lost_status_and_errors(kab, monkeypatch):
    """A path planted far above the diagonal, every other emission -inf: status 1 with a NaN final score in a
    narrow band, on the band kernel (compact copy of V = 1025) and on the windowed generic kernel
    (KAB_CTC_COMPACT=0); status 0 with a beam that covers the lattice.  forced_align_batch names the item."""
    import torch
    rng = np.random.default_rng(12)
    V, blank = 1025, 1024
    pool = np.arange(1, 300)
    good = []
    for L, T in ((700, 2300), (900, 3000)):
        tg = _targets(rng, L, V, blank, pool=pool)
        good.append((_planted_lp(rng, _planted_path(T, tg, amp=10.0), tg, V, blank), tg))
    tg = _targets(rng, 800, V, blank, pool=pool)
    T = 2600
    st = _planted_path(T, tg, amp=300.0, cycles=0.5)   # up to 300 states above the diagonal
    bad = (_planted_lp(rng, st, tg, V, blank, mask=True), tg)
    items = [good[0], bad, good[1]]
    lp, t_off, labels, l_off = _flat(items)
    for W, compact, cls in ((200, "1", CLS_BAND), (200, "0", CLS_GENERIC), (10 ** 5, "1", CLS_BAND)):
        monkeypatch.setenv("KAB_CTC_COMPACT", compact)
        out, info, rst = _check(kab, lp, t_off, labels, l_off, V, blank, W)
        assert info.n_class[cls] == 3, list(info.n_class)
        assert rst.tolist() == ([0, 1, 0] if W == 200 else [0, 0, 0])
        assert np.isnan(out[3][1]) == (W == 200)
    monkeypatch.delenv("KAB_CTC_COMPACT")
    B, T_max, L_max = 3, max(x[0].shape[0] for x in items), max(len(x[1]) for x in items)
    lpp = np.zeros((B, T_max, V), np.float32)
    tgp = np.ones((B, L_max), np.int64)
    for b, (x, t) in enumerate(items):
        lpp[b, :x.shape[0]] = x
        tgp[b, :len(t)] = t
    tl = torch.tensor([x[0].shape[0] for x in items])
    ll = torch.tensor([len(x[1]) for x in items])
    for dev in ("cpu", "cuda"):
        with pytest.raises(ValueError, match=r"item 1: no CTC path stays within beam_size=200; widen the beam"):
            kab.forced_align_batch(torch.from_numpy(lpp).to(dev), torch.from_numpy(tgp).to(dev), tl, ll, blank=blank,
                                   beam_size=200)
        with pytest.raises(ValueError, match=r"no CTC path stays within beam_size=200"):
            kab.forced_align(torch.from_numpy(bad[0])[None].to(dev), torch.from_numpy(bad[1])[None].to(dev), blank=blank,
                             beam_size=200)
    for W in (0, -3):
        with pytest.raises(ValueError, match="beam_size"):
            kab.forced_align(torch.from_numpy(bad[0])[None], torch.from_numpy(bad[1])[None], blank=blank, beam_size=W)
    from kokoro_align_b200 import _lib
    with pytest.raises(_lib.KabError):
        kab.AlignPlan.ctc(t_off, labels, l_off, V, blank, beam_size=0)


# ---- planted paths at real size
def test_ten_minutes_equals_long_form(kab):
    """T = 30 000, L = 9 000, W = 1000, drift bounded by construction: the banded plan (band kernel, 2 % of the
    cells) gives the long-form plan's (wide kernel) outputs byte for byte."""
    rng = np.random.default_rng(13)
    V, blank, T, L = 32, 0, 30000, 9000
    tg = _targets(rng, L, V, blank)
    st = _planted_path(T, tg, amp=300.0, cycles=4.0)
    lp = _planted_lp(rng, st, tg, V, blank, bonus=4.0)
    t_off, l_off = np.array([0, T]), np.array([0, L])
    out, info, rst = _check(kab, lp, t_off, tg, l_off, V, blank, 1000)
    assert rst[0] == 0 and info.n_class[CLS_BAND] == 1
    with kab.AlignPlan.ctc(t_off, tg, l_off, V, blank, long_form=True) as plan:
        assert plan.info.n_class[CLS_WIDE] == 1
        want = plan.run_host(lp)
    for a, b in zip(out, want):
        assert a.tobytes() == b.tobytes()


def test_beyond_wide_capacity(kab):
    """T = 400 000, L = 120 000 (S = 240 001, more states than the wide kernel holds at V = 32): status 0 on the
    band kernel, equal to the restatement."""
    import torch
    rng = np.random.default_rng(14)
    V, blank, T, L = 32, 0, 400000, 120000
    tg = _targets(rng, L, V, blank)
    st = _planted_path(T, tg, amp=300.0, cycles=10.0)
    lp = _planted_lp(rng, st, tg, V, blank, bonus=4.0)
    t_off, l_off = np.array([0, T]), np.array([0, L])
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    assert 2 * L + 1 > (sms - 1) * 2 * 4 * 104   # beyond even two wide CTAs per SM
    out, info, rst = _check(kab, lp, t_off, tg, l_off, V, blank, 1000)
    assert rst[0] == 0 and info.n_class[CLS_BAND] == 1
    assert info.backptr_bytes == _a256(T * _nbp(1000, 2 * L + 1))


# ---- entry points
def test_run_torch_and_run_host_children(kab, monkeypatch):
    """run_torch; run_host cutting the batch into child plans, which inherit the beam (a lattice that only a
    band loses has status 1 in every child)."""
    rng = np.random.default_rng(15)
    V, blank = 32, 4
    items = []
    for k in range(3):
        for L, T in ((300, 1000), (1200, 3900)):
            tg = _targets(rng, L, V, blank)
            items.append((_planted_lp(rng, _planted_path(T, tg, amp=20.0), tg, V, blank), tg))
        tg = _targets(rng, 800, V, blank)
        items.append((_planted_lp(rng, _planted_path(2600, tg, amp=300.0, cycles=0.5), tg, V, blank, mask=True), tg))
    lp, t_off, labels, l_off = _flat(items)
    W = 150
    out, info = _run(kab, lp, t_off, labels, l_off, V, blank, W, torch_run=True)
    _, _, rst = _check(kab, lp, t_off, labels, l_off, V, blank, W, out=out)
    assert rst.tolist() == [0, 0, 1] * 3
    monkeypatch.setenv("KAB_HOST_SEGMENTS", "3")
    out2, _ = _run(kab, lp, t_off, labels, l_off, V, blank, W)
    _check(kab, lp, t_off, labels, l_off, V, blank, W, out=out2)


def test_python_entry_points(kab):
    """forced_align(beam_size=...) and forced_align_batch(beam_size=...) on CPU and CUDA tensors."""
    import torch
    rng = np.random.default_rng(16)
    V, blank = 32, 0
    items = []
    for L, T in ((500, 1700), (1100, 3600), (2000, 6000)):
        tg = _targets(rng, L, V, blank)
        items.append((_planted_lp(rng, _planted_path(T, tg, amp=50.0), tg, V, blank, bonus=3.0), tg))
    W = 300
    lp, t_off, labels, l_off = _flat(items)
    rs, rp, rsc, rf, rst = forced_align_band_batch_np(lp, t_off, labels, l_off, blank, W)
    assert (rst == 0).all()
    lp0, tg0 = items[0]
    n0 = lp0.shape[0]
    for dev in ("cpu", "cuda"):
        p, s = kab.forced_align(torch.from_numpy(lp0)[None].to(dev), torch.from_numpy(tg0)[None].to(dev), blank=blank,
                                beam_size=W)
        assert p.device.type == dev and p.dtype == torch.int32 and p.shape == (1, n0)
        np.testing.assert_array_equal(p[0].cpu().numpy(), rp[:n0])
        assert s[0].cpu().numpy().tobytes() == rsc[:n0].tobytes()
    B, T_max, L_max = len(items), max(x[0].shape[0] for x in items), max(len(x[1]) for x in items)
    lpp = np.zeros((B, T_max, V), np.float32)
    tgp = np.ones((B, L_max), np.int64)
    for b, (x, tg) in enumerate(items):
        lpp[b, :x.shape[0]] = x
        tgp[b, :len(tg)] = tg
    tl = torch.tensor([x[0].shape[0] for x in items])
    ll = torch.tensor([len(x[1]) for x in items])
    for dev in ("cpu", "cuda"):
        p, s = kab.forced_align_batch(torch.from_numpy(lpp).to(dev), torch.from_numpy(tgp).to(dev), tl, ll, blank=blank,
                                      beam_size=W)
        assert p.device.type == dev and p.dtype == torch.int64 and p.shape == (B, T_max)
        for b in range(B):
            a, e = int(t_off[b]), int(t_off[b + 1])
            np.testing.assert_array_equal(p[b, :e - a].cpu().numpy(), rp[a:e])
            assert s[b, :e - a].cpu().numpy().tobytes() == rsc[a:e].tobytes()
            assert (p[b, e - a:] == blank).all() and (s[b, e - a:] == 0).all()
