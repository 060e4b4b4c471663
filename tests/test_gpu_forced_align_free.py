"""CTC forced alignment with free ends on the B200 (kab_plan_create_ctc_free, free_ends=True): every lattice bit
for bit against the free-ends restatement (tests/forced_align_free_np.py) -- states, token ids, scores, final
score and status -- at the edges of the warp (K = 2/4/6/8), band (3 -> 4, 16 -> 17 and 32 warps), wide
(S = 1 mod 104, the end frame at every residue mod 8) and generic kernels, through the compact copy of V = 1025
and its generic twin, with quantised ties and -inf masks; routing, child plans, plan reuse, the entry points
and a one-hour chapter with a preamble and an outro against the long-form plan on its window."""
import numpy as np
import pytest

from tests.forced_align_free_np import forced_align_free_batch_np
from tests.test_gpu_forced_align import _flat

pytestmark = pytest.mark.gpu

CLS_WARP, CLS_BAND, CLS_GENERIC, CLS_WIDE = 0, 1, 2, 3


@pytest.fixture(scope="module")
def kab():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from kokoro_align_b200 import align
    return align


def _targets(rng, L, V, blank, repeat_p=0.2):
    pool = np.array([x for x in range(V) if x != blank])
    tg = rng.choice(pool, L)
    rep = rng.random(L) < repeat_p
    if L:
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


def _planted_states(n, tg):
    """A CTC state path over n >= L + R frames through every label, from state 1 to S-2 (the last label): the
    shortest path (a blank between repeated labels) with the n - L - R extra frames spread evenly as stays."""
    seq = []
    for k, lab in enumerate(tg):
        if k and lab == tg[k - 1]:
            seq.append(2 * k)
        seq.append(2 * k + 1)
    assert n >= len(seq), "window shorter than L + R (construction)"
    stay = np.bincount((np.arange(n - len(seq)) * len(seq)) // max(n - len(seq), 1), minlength=len(seq))
    return np.repeat(np.asarray(seq, np.int64), 1 + stay[:len(seq)])


def _planted_lp(rng, T, a, b, tg, V, blank, mask=False):
    """Frames [a, b) favour a planted path through the transcript (mask: its tokens are the only finite
    ones), every other frame the blank (labels near -20)."""
    S = 2 * len(tg) + 1
    ext = np.full(S, blank, np.int64)
    ext[1::2] = tg
    lp = np.float32(-20.0) - rng.random((T, V)).astype(np.float32)
    lp[:, blank] = np.float32(-0.01) - np.float32(0.001) * rng.random(T).astype(np.float32)
    tok = ext[_planted_states(b - a, tg)]
    rows = np.arange(a, b)
    if mask:
        lp[a:b] = -np.inf
        lp[rows, tok] = -0.5 * rng.random(b - a).astype(np.float32)
    else:
        x = rng.standard_normal((b - a, V))
        x[np.arange(b - a), tok] += 8.0
        x -= x.max(axis=1, keepdims=True)
        lp[a:b] = (x - np.log(np.exp(x).sum(axis=1, keepdims=True))).astype(np.float32)
    return lp


def _run(kab, lp, t_off, labels, l_off, V, blank, torch_run=False):
    with kab.AlignPlan.ctc(t_off, labels, l_off, V, blank, free_ends=True) as plan:
        if torch_run:
            import torch
            out = tuple(x.cpu().numpy() for x in plan.run_torch(torch.from_numpy(lp).cuda()))
        else:
            out = plan.run_host(lp)
        return out, plan.info


def _check(kab, lp, t_off, labels, l_off, V, blank, out=None):
    """Plan outputs vs the free-ends restatement, bit for bit; returns (outputs, info, reference)."""
    info = None
    if out is None:
        out, info = _run(kab, lp, t_off, labels, l_off, V, blank)
    path, labs, scores, final, status = out
    ref = forced_align_free_batch_np(lp, t_off, labels, l_off, blank)
    rs, rp, rsc, rf, rst = ref
    np.testing.assert_array_equal(status, rst)
    for b in range(len(t_off) - 1):
        if rst[b] != 0:  # (statuses 1 and 2 are set at plan creation: final_score unspecified there)
            assert rst[b] != 3 or np.isnan(final[b]), f"lattice {b}"
            continue
        a, e = int(t_off[b]), int(t_off[b + 1])
        np.testing.assert_array_equal(path[a:e], rs[a:e], err_msg=f"lattice {b}")
        np.testing.assert_array_equal(labs[a:e], rp[a:e], err_msg=f"lattice {b}")
        assert scores[a:e].tobytes() == rsc[a:e].tobytes(), f"lattice {b}"
        assert final[b].tobytes() == rf[b].tobytes(), f"lattice {b}"
    return out, info, ref


def _window(states):
    inside = np.flatnonzero(states >= 0)
    return int(inside[0]), int(inside[-1])


# ---- warp kernel: K = 2 / 4 / 6 / 8 at both edges of each (S = 61 | 63, 123 | 125, 185 | 187, 247)
@pytest.mark.parametrize("L", [1, 30, 31, 61, 62, 92, 93, 123])
def test_warp_geometry(kab, L):
    rng = np.random.default_rng(100 + L)
    V, blank = 29, L % 29
    items = []
    for k in range(6):
        tg = _targets(rng, L, V, blank)
        need = L + int((tg[1:] == tg[:-1]).sum())
        T = need + int(rng.integers(0, 3 * L + 40))
        if k < 3:
            a = int(rng.integers(0, T - need + 1))
            b = a + need + int(rng.integers(0, T - a - need + 1))
            items.append((_planted_lp(rng, T, a, b, tg, V, blank, mask=k == 2), tg))
        else:
            items.append((_random_lp(rng, T, V, quant=2 if k == 4 else None, neginf=0.05 if k == 5 else 0.0), tg))
    lp, t_off, labels, l_off = _flat(items)
    _, info, _ = _check(kab, lp, t_off, labels, l_off, V, blank)
    assert info.n_class[CLS_WARP] == len(items)


# ---- band kernel: NW = 3 -> 4 (S = 279 | 281), 16 -> 17 (S = 1631 | 1633), 32 (S = 3295)
@pytest.mark.parametrize("L", [139, 140, 815, 816, 1647])
def test_band_geometry(kab, L):
    rng = np.random.default_rng(200 + L)
    V, blank = 32, 31 if L % 2 else 0
    items = []
    for k in range(3):
        tg = _targets(rng, L, V, blank)
        need = L + int((tg[1:] == tg[:-1]).sum())
        T = need + int(rng.integers(50, L + 100))
        if k == 0:
            items.append((_planted_lp(rng, T, 37, 37 + need + (T - need - 60) // 2, tg, V, blank), tg))
        else:
            items.append((_random_lp(rng, T, V, quant=2 if k == 2 else None), tg))
    lp, t_off, labels, l_off = _flat(items)
    _, info, _ = _check(kab, lp, t_off, labels, l_off, V, blank)
    assert info.n_class[CLS_BAND] == len(items)


# ---- wide kernel: S = 3329 = 1 mod 104 (S-1 opens the top warp, S-2 closes the one below); the end frame
# t1 at every residue mod 8, so the walk starts at every position inside a group of 8 frames
def test_wide_end_frame_residues(kab):
    rng = np.random.default_rng(300)
    V, blank, L = 32, 5, 1664
    assert (2 * L + 1) % 104 == 1
    items = []
    tg = _targets(rng, L, V, blank, repeat_p=0.0)
    n = L + 300
    for r in range(8):
        T = n + 200
        items.append((_planted_lp(rng, T, 40 + r, 40 + r + n, tg, V, blank, mask=r % 2 == 1), tg))
    lp, t_off, labels, l_off = _flat(items)
    _, info, ref = _check(kab, lp, t_off, labels, l_off, V, blank)
    assert info.n_class[CLS_WIDE] == len(items)
    ends = set()
    for b in range(len(items)):
        a, e = int(t_off[b]), int(t_off[b + 1])
        t0, t1 = _window(ref[0][a:e])
        assert 40 + b <= t0 and t1 < 40 + b + n
        ends.add(t1 % 8)
    assert ends == set(range(8))


def test_wide_random_and_ties(kab):
    rng = np.random.default_rng(301)
    V, blank = 16, 0
    items = []
    for k, L in enumerate((1700, 1664)):
        tg = _targets(rng, L, V, blank)
        T = L + int((tg[1:] == tg[:-1]).sum()) + 500
        items.append((_random_lp(rng, T, V, quant=1 if k else None, neginf=0.02 if k else 0.0), tg))
    lp, t_off, labels, l_off = _flat(items)
    _, info, _ = _check(kab, lp, t_off, labels, l_off, V, blank)
    assert info.n_class[CLS_WIDE] == len(items)


# ---- V = 1025: compact copy (warp, band, and a lattice of > 511 distinct ids on the generic kernel) against
# the all-generic twin (KAB_CTC_COMPACT=0)
def test_vocabulary_1025_compact_and_generic_twin(kab, monkeypatch):
    rng = np.random.default_rng(400)
    V, blank = 1025, 1024
    items = []
    for L, T in ((40, 300), (200, 700), (600, 1500)):
        tg = _targets(rng, L, V, blank)
        need = L + int((tg[1:] == tg[:-1]).sum())
        items.append((_planted_lp(rng, T, 20, 20 + need + (T - need - 40) // 2, tg, V, blank), tg))
    tg = rng.permutation(np.arange(1024))[:600].astype(np.int32)  # 600 distinct ids: generic
    items.append((_random_lp(rng, 900, V), tg))
    lp, t_off, labels, l_off = _flat(items)
    out, info, _ = _check(kab, lp, t_off, labels, l_off, V, blank)
    assert info.n_class[CLS_WARP] == 1 and info.n_class[CLS_BAND] == 2 and info.n_class[CLS_GENERIC] == 1
    monkeypatch.setenv("KAB_CTC_COMPACT", "0")
    twin, tinfo = _run(kab, lp, t_off, labels, l_off, V, blank)
    assert tinfo.n_class[CLS_GENERIC] == len(items)
    for x, y in zip(out, twin):
        assert x.tobytes() == y.tobytes()


# ---- quantised ties, -inf masks (every end candidate -inf too), empty transcripts, statuses, mixed classes
def test_ties_masks_statuses_mixed(kab):
    rng = np.random.default_rng(500)
    V, blank = 12, 3
    items = []
    for L, T in ((5, 20), (40, 90), (150, 400), (1000, 1400)):
        tg = _targets(rng, L, V, blank)
        items.append((_random_lp(rng, T, V, quant=1), tg))
        items.append((_random_lp(rng, T, V, quant=2, neginf=0.1), tg))
    tg = _targets(rng, 30, V, blank)
    lp_dead = _random_lp(rng, 80, V)
    lp_dead[:, tg[-1]] = -np.inf  # the last label never fires: every end candidate is -inf
    items.append((lp_dead, tg))
    items.append((_random_lp(rng, 17, V), np.zeros(0, np.int32)))        # L = 0
    items.append((_random_lp(rng, 5, V), _targets(rng, 9, V, blank)))   # T < L + R: status 1
    bad = _random_lp(rng, 60, V)
    bad[7, 0] = np.inf
    items.append((bad, _targets(rng, 20, V, blank)))                      # status 3
    items.append((_random_lp(rng, 30, V), np.array([1, blank, 2], np.int32)))  # status 2
    lp, t_off, labels, l_off = _flat(items)
    out, info, ref = _check(kab, lp, t_off, labels, l_off, V, blank)
    assert ref[4][-4:].tolist() == [0, 1, 3, 2]
    assert info.n_class[CLS_WARP] >= 1 and info.n_class[CLS_BAND] >= 1
    path, labs, scores, final, status = out
    b = len(items) - 5  # every end candidate -inf: (T-1, S-2), status 0
    assert status[b] == 0 and final[b] == -np.inf and path[int(t_off[b + 1]) - 1] == 2 * 30 - 1
    b = len(items) - 4  # L = 0
    a, e = int(t_off[b]), int(t_off[b + 1])
    assert final[b] == 0 and (path[a:e] == -1).all() and (labs[a:e] == blank).all()


# ---- entry points
def test_run_host_children_and_reuse(kab, monkeypatch):
    """run_host cutting the batch into child plans (which inherit free ends), and one plan run on A, B, A."""
    import torch
    rng = np.random.default_rng(600)
    V, blank = 32, 0
    items_a, items_b = [], []
    for L, T in ((20, 200), (100, 500), (400, 1200), (1500, 2500)):
        tg = _targets(rng, L, V, blank)
        need = L + int((tg[1:] == tg[:-1]).sum())
        items_a.append((_planted_lp(rng, T, 11, 11 + need + (T - need) // 2, tg, V, blank), tg))
        items_b.append((_random_lp(rng, T, V), tg))
    lpa, t_off, labels, l_off = _flat(items_a)
    lpb = _flat(items_b)[0]
    with kab.AlignPlan.ctc(t_off, labels, l_off, V, blank, free_ends=True) as plan:
        oa = plan.run_host(lpa)
        ob = plan.run_host(lpb)
        oa2 = tuple(x.cpu().numpy() for x in plan.run_torch(torch.from_numpy(lpa).cuda()))
    _check(kab, lpa, t_off, labels, l_off, V, blank, out=oa)
    _check(kab, lpb, t_off, labels, l_off, V, blank, out=ob)
    for x, y in zip(oa, oa2):
        assert x.tobytes() == y.tobytes()
    monkeypatch.setenv("KAB_HOST_SEGMENTS", "3")
    oc, _ = _run(kab, lpa, t_off, labels, l_off, V, blank)
    for x, y in zip(oa, oc):
        assert x.tobytes() == y.tobytes()


def test_python_entry_points_and_spans(kab):
    """forced_align / forced_align_batch(free_ends=True) on CPU and CUDA tensors; merge_tokens_batch on the
    result gives spans inside the planted frames [a, b); free_ends with beam_size raises ValueError."""
    import torch
    rng = np.random.default_rng(700)
    V, blank = 32, 0
    items, planted = [], []
    for L, T, a in ((30, 400, 120), (200, 900, 300), (900, 2500, 700)):
        tg = _targets(rng, L, V, blank)
        need = L + int((tg[1:] == tg[:-1]).sum())
        b = a + need + 40
        items.append((_planted_lp(rng, T, a, b, tg, V, blank), tg))
        planted.append((a, b))
    lp, t_off, labels, l_off = _flat(items)
    rs, rp, rsc, rf, rst = forced_align_free_batch_np(lp, t_off, labels, l_off, blank)
    assert (rst == 0).all()
    lp0, tg0 = items[0]
    n0 = lp0.shape[0]
    for dev in ("cpu", "cuda"):
        p, s = kab.forced_align(torch.from_numpy(lp0)[None].to(dev), torch.from_numpy(tg0)[None].to(dev), blank=blank,
                                free_ends=True)
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
        p, s = kab.forced_align_batch(torch.from_numpy(lpp).to(dev), torch.from_numpy(tgp).to(dev), tl, ll,
                                      blank=blank, free_ends=True)
        for b in range(B):
            a, e = int(t_off[b]), int(t_off[b + 1])
            np.testing.assert_array_equal(p[b, :e - a].cpu().numpy(), rp[a:e])
            assert s[b, :e - a].cpu().numpy().tobytes() == rsc[a:e].tobytes()
        spans = kab.merge_tokens_batch(p.cuda(), s.cuda(), tl.cuda(), blank=blank)
        for b, (a0, b0) in enumerate(planted):
            c = int(spans.count[b])
            assert c == len(items[b][1])
            np.testing.assert_array_equal(spans.token[b, :c].cpu().numpy(), items[b][1])
            assert int(spans.start[b, 0]) >= a0 and int(spans.end[b, c - 1]) <= b0
    with pytest.raises(ValueError):
        kab.forced_align(torch.from_numpy(lp0)[None], torch.from_numpy(tg0)[None], blank=blank, free_ends=True,
                         beam_size=100)
    with pytest.raises(ValueError):
        kab.AlignPlan.ctc(t_off, labels, l_off, V, blank, beam_size=100, free_ends=True)


# ---- a one-hour chapter (T = 180 000 frames of 20 ms, L = 54 000, V = 32) with a 3 000-frame preamble and a
# 1 500-frame outro, on the wide kernel: its window equals a long-form plan on log_probs[t0:t1+1], byte for byte
def test_chapter_against_long_form_window(kab):
    rng = np.random.default_rng(800)
    V, blank, T, L = 32, 0, 180_000, 54_000
    tg = _targets(rng, L, V, blank, repeat_p=0.05)
    a, b = 3000, T - 1500
    lp = _planted_lp(rng, T, a, b, tg, V, blank)
    t_off, l_off = np.array([0, T], np.int64), np.array([0, L], np.int64)
    (path, labs, scores, final, status), info = _run(kab, lp, t_off, tg, l_off, V, blank)
    assert status[0] == 0 and info.n_class[CLS_WIDE] == 1
    t0, t1 = _window(path)
    assert a <= t0 and t1 < b
    assert (path[:t0] == -1).all() and (path[t1 + 1:] == -1).all()
    assert (labs[:t0] == blank).all() and (labs[t1 + 1:] == blank).all()
    out = np.r_[0:t0, t1 + 1:T]
    assert scores[out].tobytes() == lp[out, blank].tobytes()
    sub = np.ascontiguousarray(lp[t0:t1 + 1])
    with kab.AlignPlan.ctc(np.array([0, t1 + 1 - t0], np.int64), tg, l_off, V, blank, long_form=True) as plan:
        lpath, llabs, lsc, lfin, lst = plan.run_host(sub)
        assert plan.info.n_class[CLS_WIDE] == 1
    assert lst[0] == 0
    assert path[t0:t1 + 1].tobytes() == lpath.tobytes()
    assert labs[t0:t1 + 1].tobytes() == llabs.tobytes()
    assert scores[t0:t1 + 1].tobytes() == lsc.tobytes()
    assert final.tobytes() == lfin.tobytes()
    with kab.AlignPlan.ctc(t_off, tg, l_off, V, blank, long_form=True) as plan:
        whole = plan.run_host(lp)
    assert whole[4][0] == 0 and final[0] >= whole[3][0]
