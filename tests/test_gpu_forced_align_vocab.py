"""CTC forced alignment of wide vocabularies (V > 512) on the staged kernels: the compact copy of the
log-probs (kab_compact_ctc_kernel, blank = compact column 0) feeds the warp, band and wide kernels.  Every
case is checked bit for bit against the restatement, torchaudio's CPU forced_align (where the chosen end
state is finite) and, byte for byte, the same plan built with KAB_CTC_COMPACT=0 (every lattice on the
generic kernel, the routing before the compact copy)."""
import numpy as np
import pytest

from oracle.forced_align_np import forced_align_batch_np, forced_align_np
from tests.test_gpu_forced_align import _flat, _torchaudio

pytestmark = pytest.mark.gpu

WARP, BAND, GENERIC, WIDE = 0, 1, 2, 3


@pytest.fixture(scope="module")
def kab():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from kokoro_align_b200 import align
    return align


def _lp(rng, T, V, quant=None, neginf=0.0):
    """float32 log_softmax of Gaussian logits [T, V]; quant: rounded to 1/quant (ties); neginf: masked share."""
    x = rng.standard_normal((T, V), dtype=np.float32) * np.float32(3.0)
    x -= x.max(axis=1, keepdims=True)
    lp = (x - np.log(np.exp(x).sum(axis=1, keepdims=True))).astype(np.float32)
    if quant:
        lp = (np.round(lp * quant) / quant).astype(np.float32)
    if neginf:
        lp[rng.random(lp.shape) < neginf] = -np.inf
    return lp


def _labels(rng, ids, L, repeat_p=0.2):
    """L targets holding every id of `ids` at least once (exactly len(ids) distinct), with adjacent repeats."""
    ids = [int(x) for x in ids]
    assert L >= len(ids)
    tg = [ids[i] for i in rng.permutation(len(ids))]
    while len(tg) < L:
        i = int(rng.integers(1, len(tg) + 1))
        tg.insert(i, tg[i - 1] if rng.random() < repeat_p else ids[int(rng.integers(len(ids)))])
    return np.array(tg, np.int32)


def _item(rng, V, blank, T, L, n_ids, must=(), pool=None, **lp_kw):
    """One lattice: L targets over n_ids distinct ids (the ids in `must` among them), T >= L + R frames."""
    if pool is None:
        pool = np.delete(np.arange(V), blank)
    must = [m for m in must if m != blank]
    rest = np.setdiff1d(pool, must)
    ids = np.concatenate([must, rng.choice(rest, n_ids - len(must), replace=False)]).astype(np.int64)
    tg = _labels(rng, ids, L, lp_kw.pop("repeat_p", 0.2))
    T = max(T, L + int((tg[1:] == tg[:-1]).sum()))
    return _lp(rng, T, V, **lp_kw), tg


def _run(kab, lp, t_off, labels, l_off, V, blank, long_form):
    with kab.AlignPlan.ctc(t_off, labels, l_off, V, blank, long_form=long_form) as plan:
        return plan.run_host(lp), plan.info


def _check3(kab, monkeypatch, lp, t_off, labels, l_off, V, blank, long_form=False, ta_check=True):
    """The plan against the restatement, torchaudio CPU and its KAB_CTC_COMPACT=0 twin.  Returns the
    plan infos (compact, reference arm)."""
    out, info = _run(kab, lp, t_off, labels, l_off, V, blank, long_form)
    monkeypatch.setenv("KAB_CTC_COMPACT", "0")
    try:
        ref, ref_info = _run(kab, lp, t_off, labels, l_off, V, blank, long_form)
    finally:
        monkeypatch.delenv("KAB_CTC_COMPACT")
    rs, rp, rsc, rf, rst = forced_align_batch_np(lp, t_off, labels, l_off, blank)
    path, labs, scores, final, status = out
    np.testing.assert_array_equal(status, rst)
    np.testing.assert_array_equal(ref[4], rst)
    F = _torchaudio() if ta_check else None
    for b in range(len(t_off) - 1):
        if rst[b] == 3:   # (the NaN final score of a rejected lattice, on both routes)
            assert final[b].tobytes() == ref[3][b].tobytes() == np.float32(np.nan).tobytes(), f"lattice {b}"
        if rst[b] != 0:
            continue
        a, e = int(t_off[b]), int(t_off[b + 1])
        np.testing.assert_array_equal(path[a:e], rs[a:e], err_msg=f"lattice {b}")
        np.testing.assert_array_equal(labs[a:e], rp[a:e], err_msg=f"lattice {b}")
        assert scores[a:e].tobytes() == rsc[a:e].tobytes(), f"lattice {b}"
        assert final[b].tobytes() == rf[b].tobytes(), f"lattice {b}"
        for k in range(3):
            assert out[k][a:e].tobytes() == ref[k][a:e].tobytes(), f"lattice {b} vs KAB_CTC_COMPACT=0"
        assert final[b].tobytes() == ref[3][b].tobytes(), f"lattice {b} vs KAB_CTC_COMPACT=0"
        if F is not None and np.isfinite(rf[b]):
            import torch
            tg = torch.from_numpy(labels[int(l_off[b]):int(l_off[b + 1])])[None]
            p, s = F.forced_align(torch.from_numpy(lp[a:e])[None], tg, blank=blank)
            np.testing.assert_array_equal(labs[a:e], p[0].numpy(), err_msg=f"lattice {b} vs torchaudio")
            assert scores[a:e].tobytes() == s[0].numpy().tobytes(), f"lattice {b} vs torchaudio"
    valid = int((rst != 2).sum() - (rst == 1).sum())
    assert ref_info.n_class[GENERIC] == valid, list(ref_info.n_class)   # (the reference arm: all generic)
    return info, ref_info


def _mixed(rng, V, blank, n_warp, n_band, n_long, must=(), band=((400, 1400), (125, 600))):
    """Warp-shaped (S <= 248), band-shaped (S <= 3296; band = (T range, L range)) and long (S = 3401)
    lattices; `must` ids in the first lattice of every kind; ties, -inf masks and repeats spread over the batch."""
    items, kind = [], []
    for k, (n, t_rng, l_rng, id_cap) in enumerate(((n_warp, (30, 160), (5, 123), 40), (n_band, *band, 300),
                                                   (n_long, (2000, 2600), (1700, 1701), 300))):
        for i in range(n):
            T, L = int(rng.integers(*t_rng)), int(rng.integers(*l_rng))
            L = min(L, T - 2) if k == 0 else L
            n_ids = int(rng.integers(min(len(must) + 1, L), min(L, id_cap) + 1))
            lp_kw = [dict(quant=2, repeat_p=0.4), dict(neginf=0.02), dict(repeat_p=0.1)][i % 3]
            items.append(_item(rng, V, blank, T, L, max(n_ids, len(must) + 1), must=must if i == 0 else (), **lp_kw))
            kind.append(k)
    return items, np.array(kind)


CASES = [(V, b) for V in (513, 1025, 5000, 65535) for b in (0, V - 1, V // 2)]


@pytest.mark.parametrize("V,blank", CASES, ids=[f"V{v}-b{b}" for v, b in CASES])
def test_vocab_classes(kab, monkeypatch, V, blank):
    """Every class at V > 512 with the blank first, last and in the middle: warp and band (default and
    long-form plans), generic (default plan, S > 3296), wide (long-form plan).  The extreme ids (0 with a
    nonzero blank, V - 1) are labels of one lattice of each kind."""
    rng = np.random.default_rng(V * 7 + blank)
    must = [x for x in (0, 1, V - 2, V - 1) if x != blank]
    big = V == 65535   # (a 65535-column row is 256 KB: short lattices only)
    items, kind = (_mixed(rng, V, blank, 4, 1, 0, must=must, band=((260, 320), (125, 140))) if big
                   else _mixed(rng, V, blank, 10, 3, 1, must=must))
    lp, t_off, labels, l_off = _flat(items)
    S = 2 * np.diff(l_off) + 1
    assert ((S <= 248) == (kind == 0)).all() and ((S > 3296) == (kind == 2)).all()
    assert set(must) <= set(labels.tolist())
    info, _ = _check3(kab, monkeypatch, lp, t_off, labels, l_off, V, blank)
    assert list(info.n_class) == [int((kind == 0).sum()), int((kind == 1).sum()), int((kind == 2).sum()), 0]
    if not big:
        info, _ = _check3(kab, monkeypatch, lp, t_off, labels, l_off, V, blank, long_form=True)
        assert list(info.n_class) == [int((kind == 0).sum()), int((kind == 1).sum()), 0, int((kind == 2).sum())]


@pytest.mark.parametrize("long_form", [False, True])
def test_both_end_states_neginf(kab, monkeypatch, long_form):
    """Both end states -inf at the last frame, in every class: the restatement's path on both routes."""
    rng = np.random.default_rng(41)
    V, blank = 1025, 1024
    items, kind = _mixed(rng, V, blank, 4, 2, 1)
    for lp, tg in items:
        lp[-1, blank] = -np.inf
        lp[-1, tg[-1]] = -np.inf
    lp, t_off, labels, l_off = _flat(items)
    rf = forced_align_batch_np(lp, t_off, labels, l_off, blank)[3]
    assert np.isneginf(rf).all()
    info, _ = _check3(kab, monkeypatch, lp, t_off, labels, l_off, V, blank, long_form=long_form, ta_check=False)
    assert info.n_class[WIDE if long_form else GENERIC] == 1 and info.n_class[WARP] == 4 and info.n_class[BAND] == 2


def test_per_lattice_fallback_and_launches(kab, monkeypatch):
    """511 distinct labels stay staged (Vc = 512); 512 go to the generic kernel -- that lattice alone.
    kernel_launches: the compaction and the label expansion for each staged list that has lattices."""
    rng = np.random.default_rng(42)
    V, blank = 1025, 1024
    items = [_item(rng, V, blank, 1000, 700, 511), _item(rng, V, blank, 1000, 700, 512)]
    items += [_item(rng, V, blank, int(rng.integers(40, 150)), 30, 20) for _ in range(5)]
    lp, t_off, labels, l_off = _flat(items)
    info, ref_info = _check3(kab, monkeypatch, lp, t_off, labels, l_off, V, blank)
    assert list(info.n_class) == [5, 1, 1, 0]
    assert info.kernel_launches == 3 + 2 * 2 and ref_info.kernel_launches == 1
    # only the lattice with 512 distinct labels: no staged list, no compaction
    one = _flat(items[1:2])
    info, _ = _check3(kab, monkeypatch, *one, V, blank)
    assert list(info.n_class) == [0, 0, 1, 0] and info.kernel_launches == 1


@pytest.mark.parametrize("n_ids,cls", [(335, WIDE), (339, GENERIC)])
def test_wide_boundary(kab, monkeypatch, n_ids, cls):
    """Long form: Vc = 336 fits the wide kernel's emission ring, Vc = 340 does not (generic)."""
    rng = np.random.default_rng(43 + n_ids)
    V, blank = 1025, 0
    items = [_item(rng, V, blank, 2200, 1700, n_ids), _item(rng, V, blank, 120, 40, 30)]
    lp, t_off, labels, l_off = _flat(items)
    info, _ = _check3(kab, monkeypatch, lp, t_off, labels, l_off, V, blank, long_form=True)
    assert info.n_class[cls] == 1 and info.n_class[WARP] == 1, list(info.n_class)


def test_nonfinite_in_unused_columns(kab, monkeypatch):
    """NaN and +inf in columns no lattice uses: status 3 on both routes (the whole row is checked), in
    every class; -inf there: status 0.  Also a label equal to the blank (2) and T < L + R (1)."""
    import torch
    rng = np.random.default_rng(44)
    V, blank = 1025, 7
    pool = np.delete(np.arange(600), blank)   # columns 600 .. 1024 belong to no lattice
    items, kind = [], []
    for T, L, n_ids, k in [(100, 30, 20, 0)] * 5 + [(800, 200, 100, 1)] * 3 + [(2200, 1700, 250, 2)] * 2:
        items.append(_item(rng, V, blank, T, L, n_ids, pool=pool))
        kind.append(k)
    items[1][0][50, 900] = np.nan
    items[2][0][0, 1000] = np.inf
    items[3][0][-1, 1024] = -np.inf
    items[6][0][400, 800] = np.nan
    items[9][0][1234, 950] = np.inf
    tg4 = items[4][1].copy()
    tg4[3] = blank
    items[4] = (items[4][0], tg4)
    items[7] = (items[7][0][:150], items[7][1])     # 150 frames for 200 targets: no path
    lp, t_off, labels, l_off = _flat(items)
    expect = [0, 3, 3, 0, 2, 0, 3, 1, 0, 3]
    for long_form in (False, True):
        info, _ = _check3(kab, monkeypatch, lp, t_off, labels, l_off, V, blank, long_form=long_form)
        with kab.AlignPlan.ctc(t_off, labels, l_off, V, blank, long_form=long_form) as plan:
            assert plan.run_host(lp)[4].tolist() == expect
        assert list(info.n_class) == [4, 2, 0 if long_form else 2, 2 if long_form else 0]
    for dev in ("cpu", "cuda"):
        for b, raises in ((1, True), (2, True), (3, False), (6, True)):
            x, tg = (torch.from_numpy(a)[None].to(dev) for a in items[b])
            if raises:
                with pytest.raises(ValueError, match="NaN or \\+inf"):
                    kab.forced_align(x, tg, blank=blank)
            else:
                p, s = kab.forced_align(x, tg, blank=blank)
                np.testing.assert_array_equal(p[0].cpu().numpy(), forced_align_np(items[b][0], items[b][1], blank)[1])
    T_max = max(items[b][0].shape[0] for b in (0, 1))
    lpp = np.zeros((2, T_max, V), np.float32)
    tgp = np.zeros((2, 30), np.int64)
    for i, b in enumerate((0, 1)):
        lpp[i, :items[b][0].shape[0]] = items[b][0]
        tgp[i] = items[b][1]
    with pytest.raises(ValueError, match="item 1"):
        kab.forced_align_batch(torch.from_numpy(lpp).cuda(), torch.from_numpy(tgp).cuda(),
                               torch.tensor([items[0][0].shape[0], items[1][0].shape[0]]), blank=blank)


def test_python_entry_points(kab):
    """forced_align on CPU and CUDA tensors (default and long form) and the padded forced_align_batch,
    NeMo's layout: V = 1025, blank = 1024."""
    import torch
    rng = np.random.default_rng(45)
    V, blank = 1025, 1024
    items, kind = _mixed(rng, V, blank, 6, 2, 1, must=(0, 1023))
    for b in (0, int(np.flatnonzero(kind == 1)[0]), int(np.flatnonzero(kind == 2)[0])):
        lp0, tg0 = items[b]
        _, paths, sc, _ = forced_align_np(lp0, tg0, blank)
        for dev in ("cpu", "cuda"):
            for long_form in (False, True):
                p, s = kab.forced_align(torch.from_numpy(lp0)[None].to(dev), torch.from_numpy(tg0)[None].to(dev),
                                        blank=blank, long_form=long_form)
                assert p.device.type == dev and p.dtype == torch.int32 and p.shape == (1, lp0.shape[0])
                np.testing.assert_array_equal(p[0].cpu().numpy(), paths)
                assert s[0].cpu().numpy().tobytes() == sc.tobytes()
    B, T_max, L_max = len(items), max(x[0].shape[0] for x in items), max(len(x[1]) for x in items)
    lpp = np.zeros((B, T_max, V), np.float32)
    tgp = np.zeros((B, L_max), np.int64)
    for b, (x, tg) in enumerate(items):
        lpp[b, :x.shape[0]] = x
        tgp[b, :len(tg)] = tg
    tl = torch.tensor([x[0].shape[0] for x in items])
    ll = torch.tensor([len(x[1]) for x in items])
    for dev in ("cpu", "cuda"):
        p, s = kab.forced_align_batch(torch.from_numpy(lpp).to(dev), torch.from_numpy(tgp).to(dev), tl, ll, blank=blank)
        assert p.device.type == dev and p.dtype == torch.int64 and p.shape == (B, T_max)
        for b, (x, tg) in enumerate(items):
            _, rp, rsc, _ = forced_align_np(x, tg, blank)
            n = x.shape[0]
            np.testing.assert_array_equal(p[b, :n].cpu().numpy(), rp)
            assert s[b, :n].cpu().numpy().tobytes() == rsc.tobytes()
            assert (p[b, n:] == blank).all() and (s[b, n:] == 0).all()


def test_run_torch_and_run_host_children(kab, monkeypatch):
    """run_torch of a compact plan; run_host cutting the batch into three child plans, each with its own
    compact copy (the compaction kernel runs for the warp and band lists of every child, the generic
    kernel never)."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    rng = np.random.default_rng(46)
    V, blank = 1025, 0
    Ts = [4 * int(rng.integers(10, 40)) for _ in range(8)] + [4 * int(rng.integers(150, 300))]
    items = []
    for _ in range(3):   # three equal groups of frames: the cuts fall between them
        for i, T in enumerate(Ts):
            L = T // 4 if i < 8 else 200
            items.append(_item(rng, V, blank, T, L, min(L, 25 + 10 * i), repeat_p=0.0))
    lp, t_off, labels, l_off = _flat(items)
    assert (np.diff(t_off) % 4 == 0).all()
    rs, rp, rsc, rf, rst = forced_align_batch_np(lp, t_off, labels, l_off, blank)
    assert (rst == 0).all()
    with kab.AlignPlan.ctc(t_off, labels, l_off, V, blank) as plan:
        assert list(plan.info.n_class) == [24, 3, 0, 0]
        outs = [tuple(x.cpu().numpy() for x in plan.run_torch(torch.from_numpy(lp).cuda()))]
    monkeypatch.setenv("KAB_HOST_SEGMENTS", "3")
    with kab.AlignPlan.ctc(t_off, labels, l_off, V, blank) as plan:
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            outs.append(plan.run_host(lp))
            torch.cuda.synchronize()
    counts = {e.key: e.count for e in prof.key_averages()}
    n_compact = sum(c for k, c in counts.items() if "kab_compact_ctc_kernel" in k)
    assert n_compact == 6, counts
    assert any("kab_expand_labels_kernel" in k for k in counts), sorted(counts)
    assert not any("kab_generic_ctc_kernel" in k or "kab_compact_kernel" in k for k in counts), sorted(counts)
    for path, labs, scores, final, status in outs:
        np.testing.assert_array_equal(status, rst)
        np.testing.assert_array_equal(path, rs)
        np.testing.assert_array_equal(labs, rp)
        assert scores.tobytes() == rsc.tobytes() and final.tobytes() == rf.tobytes()
