"""Token spans and word spans on the B200 (kab_merge_tokens_device / kab_word_spans_device and the
Python entry points): token / start / end / count bit for bit and scores bit for bit against the
restatement (oracle/merge_tokens_np.py), scores within 1e-6 (relative) of torchaudio's CPU
merge_tokens, word scores bit for bit against the forced-alignment tutorial's formula."""
import ctypes

import numpy as np
import pytest

from oracle.merge_tokens_np import merge_tokens_np, word_spans_np
from tests.test_merge_tokens_oracle import greedy_paths, tutorial_words

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def kab():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from kokoro_align_b200 import align
    return align


def _torchaudio():
    try:
        import torch
        import torchaudio.functional as F
        F.merge_tokens(torch.zeros(2, dtype=torch.int32), torch.zeros(2))
        return F
    except Exception:  # noqa: BLE001
        return None


def same_f32(a, b):
    """Bit-equal float32 arrays, NaN equal to NaN (NaN payloads are not part of the contract)."""
    a, b = np.asarray(a, np.float32), np.asarray(b, np.float32)
    return a.shape == b.shape and bool(((a.view(np.uint32) == b.view(np.uint32)) | (np.isnan(a) & np.isnan(b))).all())


def pad(items, dtype=np.int32, fill=0):
    """[(tokens [T], scores [T])] -> padded tokens [B, T_max], scores [B, T_max], lengths [B]."""
    T = np.array([len(x[0]) for x in items], np.int64)
    tok = np.full((len(items), max(1, int(T.max()) if len(T) else 1)), fill, dtype)
    sc = np.zeros(tok.shape, np.float32)
    for b, (t, s) in enumerate(items):
        tok[b, :len(t)] = t
        sc[b, :len(t)] = s
    return tok, sc, T


def check_spans(res, tokens, scores, lengths, blank, ta_items=None):
    """res: TokenSpans (any device) vs the restatement on every item and torchaudio's CPU
    merge_tokens on the items ta_items (None: all)."""
    import torch
    tok, st, en, sc, cnt = (x.cpu().numpy() for x in res)
    B = len(lengths)
    assert tok.shape[0] == B and cnt.shape == (B,)
    assert tok.shape[1] == (int(cnt.max()) if B else 0)
    F = _torchaudio()
    for b in range(B):
        n, T = int(cnt[b]), int(lengths[b])
        rt, rs, re_, rsc = merge_tokens_np(tokens[b][:T], scores[b][:T], blank)
        assert n == len(rt), f"item {b}"
        np.testing.assert_array_equal(tok[b, :n], rt, err_msg=f"item {b}")
        np.testing.assert_array_equal(st[b, :n], rs, err_msg=f"item {b}")
        np.testing.assert_array_equal(en[b, :n], re_, err_msg=f"item {b}")
        assert same_f32(sc[b, :n], rsc), f"item {b}"
        assert (tok[b, n:] == -1).all() and (st[b, n:] == -1).all() and (en[b, n:] == -1).all() and (sc[b, n:] == 0).all()
        if F is not None and (ta_items is None or b in ta_items):
            ref = F.merge_tokens(torch.from_numpy(np.ascontiguousarray(tokens[b][:T])),
                                 torch.from_numpy(np.ascontiguousarray(scores[b][:T])), blank)
            assert [(s.token, s.start, s.end) for s in ref] == list(zip(rt.tolist(), rs.tolist(), re_.tolist()))
            np.testing.assert_allclose(sc[b, :n], np.array([s.score for s in ref], np.float32), rtol=1e-6, atol=0)


def _forced_align_items(rng, n, V, blank, t_range, l_frac, tight=False, repeat_p=0.3):
    out = []
    pool = np.array([x for x in range(V) if x != blank])
    for _ in range(n):
        T = int(rng.integers(*t_range))
        L = max(1, int(T * rng.uniform(*l_frac)))
        tg = rng.choice(pool, L)
        rep = rng.random(L) < repeat_p
        rep[0] = False
        tg[rep] = tg[np.flatnonzero(rep) - 1]
        R = int((tg[1:] == tg[:-1]).sum())
        T = L + R if tight else max(T, L + R)
        out.append((np.log(rng.dirichlet(np.full(V, 0.5), T)).astype(np.float32), tg.astype(np.int64)))
    return out


@pytest.mark.parametrize("blank", [0, 7])
def test_forced_align_outputs(kab, blank):
    """forced_align_batch of a mixed batch (warp, band and generic lattices, one with S > 3296, tight
    T == L + R items, repeated targets) -> merge_tokens_batch: one span per target."""
    import torch
    rng = np.random.default_rng(40 + blank)
    V = 32
    items = (_forced_align_items(rng, 30, V, blank, (20, 300), (0.1, 0.45))
             + _forced_align_items(rng, 6, V, blank, (20, 200), (0.2, 0.4), tight=True)
             + _forced_align_items(rng, 4, V, blank, (900, 3000), (0.2, 0.35))
             + _forced_align_items(rng, 1, V, blank, (4000, 4001), (0.42, 0.43)))
    B = len(items)
    T = np.array([x[0].shape[0] for x in items])
    L = np.array([len(x[1]) for x in items])
    assert (2 * L + 1 > 3296).any() and ((2 * L + 1 <= 248).any()) and ((2 * L + 1 > 248) & (2 * L + 1 <= 3296)).any()
    lp = np.zeros((B, T.max(), V), np.float32)
    tg = np.zeros((B, L.max()), np.int64)
    for b, (x, t) in enumerate(items):
        lp[b, :len(x)] = x
        tg[b, :len(t)] = t
    dev = "cuda"
    paths, scores = kab.forced_align_batch(torch.from_numpy(lp).to(dev), torch.from_numpy(tg).to(dev),
                                           torch.from_numpy(T), torch.from_numpy(L), blank=blank)
    for sc in (scores, scores.exp()):
        res = kab.merge_tokens_batch(paths, sc, torch.from_numpy(T), blank=blank)
        assert res.token.device.type == "cuda" and res.token.dtype == torch.int64
        check_spans(res, paths.cpu().numpy(), sc.cpu().numpy(), T, blank)
        np.testing.assert_array_equal(res.count.cpu().numpy(), L)
        tok = res.token.cpu().numpy()
        for b in range(B):
            np.testing.assert_array_equal(tok[b, :L[b]], tg[b, :L[b]])


def test_greedy_paths_and_edge_cases(kab):
    """Greedy argmax paths (leading / trailing blanks, long runs), an all-blank item, T = 0, T = 1,
    blank = V - 1, int64 tokens, -inf and NaN scores, runs across the kernel's chunk boundaries."""
    import torch
    rng = np.random.default_rng(5)
    V = 29
    blank = V - 1
    items = greedy_paths(rng, 50, V, blank, (1, 3000))
    items += [(np.full(9, blank, np.int32), np.zeros(9, np.float32)),   # all blank
              (np.zeros(0, np.int32), np.zeros(0, np.float32)),         # T = 0
              (np.array([3], np.int32), np.array([-0.25], np.float32))]  # T = 1
    chunk = np.full(3000, blank, np.int32)   # runs that end / start / cross at multiples of 1024 frames
    chunk[1020:1030] = 4
    chunk[1030:2048] = 5
    chunk[2048:2049] = 6
    chunk[2049:3000] = 6 + (np.arange(951) // 7) % 3
    items.append((chunk, np.log(rng.random(3000)).astype(np.float32)))   # log-probs: no cancellation
    nonfin = items[3][1].copy()
    nonfin[::17] = -np.inf
    nonfin[5::23] = np.nan
    items.append((items[3][0], nonfin))
    tok, sc, T = pad(items, np.int64, fill=blank)
    res = kab.merge_tokens_batch(torch.from_numpy(tok).cuda(), torch.from_numpy(sc).cuda(), torch.from_numpy(T),
                                 blank=blank)
    assert res.token.dtype == torch.int64
    check_spans(res, tok, sc, T, blank)
    # CPU tensors in, CPU tensors out; int32 tokens
    res_cpu = kab.merge_tokens_batch(torch.from_numpy(tok.astype(np.int32)), torch.from_numpy(sc), T, blank=blank)
    assert all(x.device.type == "cpu" for x in res_cpu) and res_cpu.token.dtype == torch.int32
    for a, b in zip(res, res_cpu):
        assert np.array_equal(a.cpu().numpy().view(np.uint32) if a.dtype == torch.float32 else a.cpu().numpy(),
                              b.numpy().view(np.uint32) if b.dtype == torch.float32 else b.numpy())
    # lengths=None: every item is T_max frames (the padding is blank)
    res_full = kab.merge_tokens_batch(torch.from_numpy(tok).cuda(), torch.from_numpy(sc).cuda(), blank=blank)
    check_spans(res_full, tok, sc, np.full(len(T), tok.shape[1]), blank, ta_items={0, 1})


def test_extremes_200k_frames(kab):
    """A single item of 2e5 spans, and a single span of 2e5 frames."""
    import torch
    rng = np.random.default_rng(6)
    n = 200000
    sc = rng.random(n).astype(np.float32)
    alt = (1 + np.arange(n) % 2).astype(np.int32)          # 1 2 1 2 ...: one span per frame
    one = np.full(n, 3, np.int32)
    for tok in (alt, one):
        res = kab.merge_tokens_batch(torch.from_numpy(tok[None]).cuda(), torch.from_numpy(sc[None]).cuda())
        check_spans(res, tok[None], sc[None], [n], 0)
    assert int(res.count[0]) == 1 and int(res.end[0, 0]) == n


def test_kokoro_best_labels(kab):
    """The best_labels of Kokoro-mode plans (blank 0) -> phoneme spans."""
    import torch
    from kokoro_align_b200 import synth
    Ts = np.array([86, 300, 431, 861, 6000])
    Ls = np.array([12, 42, 60, 121, 1700])
    lp, t_off, labels, l_off = synth.make_batch(Ts, Ls, seed=77)
    with kab.AlignPlan(t_off, labels, l_off, 39) as plan:
        _, labs, scores, _, status = plan.run_host(lp)
    assert (status == 0).all()
    items = [(labs[t_off[b]:t_off[b + 1]], scores[t_off[b]:t_off[b + 1]]) for b in range(len(Ts))]
    tok, sc, T = pad(items)
    res = kab.merge_tokens_batch(torch.from_numpy(tok).cuda(), torch.from_numpy(sc).cuda(), torch.from_numpy(T))
    check_spans(res, tok, sc, T, 0)
    assert (res.count.cpu().numpy() > 0).all()


def test_utterance_workload(kab):
    """The 4 096-utterance workload of tools/forced_align_bench.py: CTC-plan paths -> spans, against
    the restatement in full and torchaudio on a seeded sample of 64 items."""
    import torch
    from tools.forced_align_bench import workload
    T, tgs = workload("utterances", 1234)
    V, B = 32, len(T)
    t_off = np.concatenate([[0], np.cumsum(T)]).astype(np.int64)
    l_off = np.concatenate([[0], np.cumsum([len(x) for x in tgs])]).astype(np.int64)
    g = torch.Generator(device="cuda").manual_seed(99)
    lp = torch.log_softmax(2.0 * torch.randn(int(t_off[-1]), V, device="cuda", generator=g), dim=-1).contiguous()
    with kab.AlignPlan.ctc(t_off, np.concatenate(tgs), l_off, V, 0) as plan:
        _, labs, sc, _, st = plan.run_torch(lp)
        assert int(st.abs().sum()) == 0
    T_max = int(T.max())
    valid = torch.arange(T_max, device="cuda")[None, :] < torch.from_numpy(T).cuda()[:, None]
    paths = torch.zeros((B, T_max), dtype=torch.int32, device="cuda")
    scores = torch.zeros((B, T_max), dtype=torch.float32, device="cuda")
    paths[valid] = labs
    scores[valid] = sc.exp()
    res = kab.merge_tokens_batch(paths, scores, torch.from_numpy(T))
    sample = set(np.random.default_rng(0).choice(B, 64, replace=False).tolist())
    check_spans(res, paths.cpu().numpy(), scores.cpu().numpy(), T, 0, ta_items=sample)
    np.testing.assert_array_equal(res.count.cpu().numpy(), [len(x) for x in tgs])


def test_single_item_merge_tokens(kab):
    import torch
    F = _torchaudio()
    rng = np.random.default_rng(8)
    for path, lp in greedy_paths(rng, 6, 12, 0, (1, 2000)) + [(np.zeros(0, np.int32), np.zeros(0, np.float32))]:
        rt, rs, re_, rsc = merge_tokens_np(path, np.exp(lp), 0)
        for dev in ("cpu", "cuda"):
            spans = kab.merge_tokens(torch.from_numpy(path).to(dev), torch.from_numpy(np.exp(lp)).to(dev))
            assert all(isinstance(s, kab.TokenSpan) for s in spans)
            assert [(s.token, s.start, s.end) for s in spans] == list(zip(rt.tolist(), rs.tolist(), re_.tolist()))
            assert same_f32([s.score for s in spans], rsc)
            assert [len(s) for s in spans] == (re_ - rs).tolist()
        if F is not None:
            ref = F.merge_tokens(torch.from_numpy(path), torch.from_numpy(np.exp(lp)))
            assert [(s.token, s.start, s.end) for s in ref] == [(s.token, s.start, s.end) for s in spans]
            np.testing.assert_allclose([s.score for s in spans], [s.score for s in ref], rtol=1e-6, atol=0)


def test_word_spans(kab):
    import torch
    rng = np.random.default_rng(12)
    items = greedy_paths(rng, 40, 20, 0, (1, 1500))
    tok, sc, T = pad(items)
    for dev in ("cuda", "cpu"):
        res = kab.merge_tokens_batch(torch.from_numpy(tok).to(dev), torch.from_numpy(np.exp(sc)).to(dev),
                                     torch.from_numpy(T))
        cnt = res.count.cpu().numpy()
        wl = []
        for b in range(len(T)):
            w = []
            while sum(w) < cnt[b]:
                w.append(int(min(rng.integers(1, 9), cnt[b] - sum(w))))
            wl.append(w)
        words = kab.word_spans(res, wl)
        assert all(x.device.type == dev for x in words)
        ws, we, wsc, wf, wc = (x.cpu().numpy() for x in words)
        rt, rs, re_, rsc = (x.cpu().numpy() for x in res[:4])
        np.testing.assert_array_equal(wc, [len(w) for w in wl])
        for b in range(len(T)):
            n, k = int(cnt[b]), len(wl[b])
            spans = [kab.TokenSpan(int(a), int(s), int(e), float(c))
                     for a, s, e, c in zip(rt[b, :n], rs[b, :n], re_[b, :n], rsc[b, :n])]
            ref = tutorial_words(spans, wl[b]) if k else []
            assert ws[b, :k].tolist() == [r[0] for r in ref] and we[b, :k].tolist() == [r[1] for r in ref]
            assert wsc[b, :k].tobytes() == np.array([r[2] for r in ref], np.float32).tobytes(), f"item {b}"
            if k:
                o = word_spans_np(rs[b, :n], re_[b, :n], rsc[b, :n], wl[b])
                np.testing.assert_array_equal(wf[b, :k], o[2])
                assert wsc[b, :k].tobytes() == o[3].tobytes()
            assert (ws[b, k:] == -1).all() and (wf[b, k:] == -1).all() and (wsc[b, k:] == 0).all()
    bad = [list(w) for w in wl]
    b0 = next(b for b in range(len(bad)) if bad[b])
    bad[b0] = bad[b0] + [1]
    with pytest.raises(ValueError, match=f"item {b0}"):
        kab.word_spans(res, bad)
    bad = [list(w) for w in wl]
    bad[b0] = bad[b0] + [0]
    with pytest.raises(ValueError, match=f"item {b0}"):
        kab.word_spans(res, bad)


def test_c_entry_points_directly():
    """The flat layout: spans of item b at d_spans[t_off[b] ..] (t_off[0] != 0 here), items never
    merge across their boundary, untouched capacity stays untouched; an item whose word lengths do
    not fit gets d_word_status = 1 without a C error, the others their words."""
    import torch
    from kokoro_align_b200 import _lib
    L = _lib.lib()
    vp = lambda t: ctypes.c_void_p(t.data_ptr())  # noqa: E731
    tok = torch.tensor([9, 9, 9, 5, 5, 5, 5, 0, 2, 0, 0, 7], dtype=torch.int32, device="cuda")
    sc = torch.arange(12, dtype=torch.float32, device="cuda") / 4
    t_off = torch.tensor([2, 5, 8, 8, 12], dtype=torch.int64, device="cuda")   # items [2,5) [5,8) [8,8) [8,12)
    recs = torch.full((12, 4), -7, dtype=torch.int32, device="cuda")
    cnt = torch.full((4,), -7, dtype=torch.int32, device="cuda")
    s = torch.cuda.current_stream()
    assert L.kab_merge_tokens_device(4, vp(t_off), vp(tok), vp(sc), 0, vp(recs), vp(cnt), ctypes.c_void_p(s.cuda_stream)) == 0
    torch.cuda.synchronize()
    r = recs.cpu().numpy()
    assert cnt.cpu().tolist() == [2, 1, 0, 2]
    expect = {2: (9, 0, 1), 3: (5, 1, 3), 5: (5, 0, 2), 8: (2, 0, 1), 9: (7, 3, 4)}
    for row in range(12):
        if row in expect:
            assert tuple(r[row, :3]) == expect[row], row
        else:
            assert (r[row] == -7).all(), row
    scores = r[:, 3].copy().view(np.float32)
    x = sc.cpu().numpy()
    assert scores[3] == np.float32((np.float64(x[3]) + np.float64(x[4])) / 2)
    assert scores[5] == np.float32((np.float64(x[5]) + np.float64(x[6])) / 2)
    # words: item 0 [1, 1], item 1 [3] (does not fit: it has 1 span), item 2 [], item 3 [2]
    w_off = torch.tensor([0, 2, 3, 3, 4], dtype=torch.int64, device="cuda")
    w_len = torch.tensor([1, 1, 3, 2], dtype=torch.int32, device="cuda")
    words = torch.full((4, 4), -7, dtype=torch.int32, device="cuda")
    status = torch.full((4,), -7, dtype=torch.int32, device="cuda")
    assert L.kab_word_spans_device(4, vp(t_off), vp(recs), vp(cnt), vp(w_off), vp(w_len), vp(words), vp(status),
                                   ctypes.c_void_p(s.cuda_stream)) == 0
    torch.cuda.synchronize()
    w = words.cpu().numpy()
    assert status.cpu().tolist() == [0, 1, 0, 0]
    assert tuple(w[0, :3]) == (0, 1, 0) and tuple(w[1, :3]) == (1, 3, 1) and (w[2] == -7).all()
    assert tuple(w[3, :3]) == (0, 4, 0)
    ws = w[:, 3].copy().view(np.float32)
    assert ws[0] == scores[2] and ws[1] == scores[3]
    num = np.float64(scores[8]) * 1 + np.float64(scores[9]) * 1
    assert ws[3] == np.float32(num / 2)
    assert L.kab_merge_tokens_device(-1, vp(t_off), vp(tok), vp(sc), 0, vp(recs), vp(cnt), None) == _lib.KAB_E_BAD_ARG
    assert L.kab_merge_tokens_device(4, vp(t_off), None, vp(sc), 0, vp(recs), vp(cnt), None) == _lib.KAB_E_BAD_ARG
    assert L.kab_word_spans_device(4, vp(t_off), vp(recs), vp(cnt), vp(w_off), vp(w_len), None, vp(status),
                                   None) == _lib.KAB_E_BAD_ARG
