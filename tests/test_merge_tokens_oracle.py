"""The CPU restatement of token and word spans (oracle/merge_tokens_np.py) against live
torchaudio.functional.merge_tokens and the forced-alignment tutorial's word score; the C-ABI
struct mirrors; the span entry points fail loudly without a CUDA device."""
import ctypes

import numpy as np
import pytest

from oracle.merge_tokens_np import merge_tokens_batch_np, merge_tokens_np, word_spans_np
from tests.test_forced_align_oracle import CASES


def _merge_tokens():
    try:
        import torch
        import torchaudio.functional as F
        F.merge_tokens(torch.zeros(2, dtype=torch.int32), torch.zeros(2))
        return torch, F
    except Exception:  # noqa: BLE001 -- not installed
        pytest.skip("torchaudio's merge_tokens is not available")


def assert_matches_torchaudio(F, torch, tokens, scores, blank):
    tok, st, en, sc = merge_tokens_np(tokens, scores, blank)
    ref = F.merge_tokens(torch.from_numpy(np.asarray(tokens)), torch.from_numpy(np.asarray(scores, np.float32)), blank)
    assert [s.token for s in ref] == tok.tolist()
    assert [s.start for s in ref] == st.tolist()
    assert [s.end for s in ref] == en.tolist()
    np.testing.assert_allclose(sc, np.array([s.score for s in ref], np.float32), rtol=1e-6, atol=0)


def greedy_paths(rng, n, V, blank, t_range):
    """Argmax decodes of random emissions: leading / trailing blanks, repeats, long and short runs."""
    out = []
    for _ in range(n):
        T = int(rng.integers(*t_range))
        lp = np.log(rng.dirichlet(np.full(V, 0.3), T)).astype(np.float32)
        lp[:, blank] += np.float32(rng.uniform(0, 3))   # blank-heavy, as CTC emissions are
        if rng.random() < 0.3:   # stretch some runs
            lp = np.repeat(lp, rng.integers(1, 6, T), axis=0)[:T]
        path = lp.argmax(1).astype(np.int32)
        out.append((path, lp[np.arange(T), path]))
    return out


def test_oracle_matches_torchaudio_on_forced_alignments():
    torch, F = _merge_tokens()
    n = 0
    for name, c in CASES:
        paths, scores, blank = c["paths"], c["scores"], int(c["blank"])
        for sc in (scores, np.exp(scores)):
            assert_matches_torchaudio(F, torch, paths, sc.astype(np.float32), blank)
        n += 1
    assert n >= 10


@pytest.mark.parametrize("V,blank", [(32, 0), (29, 28), (6, 3)])
def test_oracle_matches_torchaudio_on_greedy_paths(V, blank):
    torch, F = _merge_tokens()
    rng = np.random.default_rng(V * 10 + blank)
    items = greedy_paths(rng, 40, V, blank, (1, 600))
    items += [(np.full(7, blank, np.int32), np.zeros(7, np.float32)),                # all blank
              (np.array([blank ^ 1], np.int32), np.array([-0.5], np.float32)),       # T = 1
              (np.zeros(0, np.int32), np.zeros(0, np.float32))]                      # T = 0
    for path, lp in items:
        for sc in (lp, np.exp(lp)):
            assert_matches_torchaudio(F, torch, path, sc.astype(np.float32), blank)


def test_oracle_long_spans_and_nonfinite():
    """One 30 000-frame span (summed alone) next to short ones; -inf and NaN propagate."""
    torch, F = _merge_tokens()
    rng = np.random.default_rng(2)
    tok = np.concatenate([np.zeros(5), np.full(30000, 3), np.array([0, 1, 1, 2, 0])]).astype(np.int32)
    sc = rng.random(tok.shape[0]).astype(np.float32)
    assert_matches_torchaudio(F, torch, tok, sc, 0)
    sc[30006] = -np.inf
    sc[30008] = np.nan
    t, s, e, m = merge_tokens_np(tok, sc, 0)
    assert e.tolist() == [30005, 30008, 30009] and np.isneginf(m[1]) and np.isnan(m[2])
    # the sequential double sum of the long span, written out
    acc = np.float64(sc[5])
    for v in sc[6:30005]:
        acc = acc + np.float64(v)
    assert m[0] == np.float32(acc / 30000)


def test_batch_restatement_respects_lengths():
    tok = np.array([[1, 1, 0, 2, 2], [3, 0, 3, 3, 9]], np.int32)
    sc = np.arange(10, dtype=np.float32).reshape(2, 5)
    r = merge_tokens_batch_np(tok, sc, [5, 3])
    assert r[0][0].tolist() == [1, 2] and r[0][1].tolist() == [0, 3] and r[0][2].tolist() == [2, 5]
    assert r[1][0].tolist() == [3, 3] and r[1][2].tolist() == [1, 3]


def tutorial_words(spans, word_lengths):
    """torchaudio's forced-alignment tutorial, verbatim: unflatten + _score (Python floats)."""
    def unflatten(list_, lengths):
        assert len(list_) == sum(lengths)
        i = 0
        ret = []
        for length in lengths:
            ret.append(list_[i:i + length])
            i += length
        return ret

    def _score(spans):
        return sum(s.score * len(s) for s in spans) / sum(len(s) for s in spans)
    return [(w[0].start, w[-1].end, np.float32(_score(w))) for w in unflatten(spans, word_lengths)]


def test_word_oracle_equals_tutorial_formula():
    from kokoro_align_b200.align import TokenSpan
    rng = np.random.default_rng(9)
    for path, lp in greedy_paths(rng, 60, 20, 0, (5, 800)):
        for sc in (lp, np.exp(lp)):
            tok, st, en, m = merge_tokens_np(path, sc.astype(np.float32), 0)
            if len(tok) == 0:
                continue
            wl = []
            while sum(wl) < len(tok):
                wl.append(int(min(rng.integers(1, 9), len(tok) - sum(wl))))
            ws, we, wf, wsc = word_spans_np(st, en, m, wl)
            spans = [TokenSpan(int(a), int(b), int(c), float(d)) for a, b, c, d in zip(tok, st, en, m)]
            ref = tutorial_words(spans, wl)
            assert ws.tolist() == [r[0] for r in ref] and we.tolist() == [r[1] for r in ref]
            assert wf.tolist() == np.concatenate([[0], np.cumsum(wl)[:-1]]).tolist()
            assert wsc.tobytes() == np.array([r[2] for r in ref], np.float32).tobytes()


def test_token_span_dataclass():
    from kokoro_align_b200.align import TokenSpan
    s = TokenSpan(token=4, start=3, end=9, score=0.5)
    assert len(s) == 6 and (s.token, s.start, s.end, s.score) == (4, 3, 9, 0.5)


def test_struct_mirrors_are_16_bytes():
    from kokoro_align_b200 import _lib
    assert ctypes.sizeof(_lib.TokenSpanRec) == 16 and ctypes.sizeof(_lib.WordSpanRec) == 16
    assert [f[0] for f in _lib.TokenSpanRec._fields_] == ["token", "start", "end", "score"]
    assert [f[0] for f in _lib.WordSpanRec._fields_] == ["start", "end", "first_token", "score"]


def test_span_entry_points_need_a_device():
    torch = pytest.importorskip("torch")
    if torch.cuda.is_available():
        pytest.skip("CUDA present")
    from kokoro_align_b200 import _lib, align
    L = _lib.lib()
    buf = (ctypes.c_int64 * 16)()
    p = ctypes.cast(buf, ctypes.c_void_p)
    assert L.kab_merge_tokens_device(1, p, p, p, 0, p, p, None) == _lib.KAB_E_CUDA
    assert L.kab_word_spans_device(1, p, p, p, p, p, p, p, None) == _lib.KAB_E_CUDA
    assert L.kab_merge_tokens_device(-1, p, p, p, 0, p, p, None) == _lib.KAB_E_BAD_ARG
    assert L.kab_word_spans_device(1, p, None, p, p, p, p, p, None) == _lib.KAB_E_BAD_ARG
    with pytest.raises(align.KabError):
        align.merge_tokens_batch(torch.zeros(1, 4, dtype=torch.int32), torch.zeros(1, 4))
    with pytest.raises(align.KabError):
        align.merge_tokens(torch.zeros(4, dtype=torch.int32), torch.zeros(4))


@pytest.mark.parametrize("bad", ["ndim", "length", "negative", "float64", "lengths_shape", "lengths_range"])
def test_argument_errors(bad):
    torch = pytest.importorskip("torch")
    from kokoro_align_b200 import align
    tok, sc = torch.zeros(2, 5, dtype=torch.int64), torch.zeros(2, 5)
    with pytest.raises(ValueError):
        if bad == "ndim":
            align.merge_tokens(tok, sc[0])
        elif bad == "length":
            align.merge_tokens(tok[0], sc[0, :4])
        elif bad == "negative":
            tok[1, 2] = -1
            align.merge_tokens_batch(tok, sc)
        elif bad == "float64":
            align.merge_tokens_batch(tok, sc.double())
        elif bad == "lengths_shape":
            align.merge_tokens_batch(tok, sc, torch.tensor([5]))
        else:
            align.merge_tokens_batch(tok, sc, torch.tensor([5, 6]))


def test_word_spans_argument_errors():
    """Checked on the host before any device work: the first item whose word lengths do not sum to
    its span count, or that has a word of length 0, is named."""
    torch = pytest.importorskip("torch")
    from kokoro_align_b200 import align
    z = torch.zeros(3, 4, dtype=torch.int64)
    spans = align.TokenSpans(z, z, z, torch.zeros(3, 4), torch.tensor([4, 2, 0]))
    with pytest.raises(ValueError, match="item 1"):
        align.word_spans(spans, [[1, 3], [1], []])
    with pytest.raises(ValueError, match="item 0"):
        align.word_spans(spans, [[4, 0], [2], [1]])
    with pytest.raises(ValueError, match="item 2"):
        align.word_spans(spans, [[2, 2], [1, 1], [1]])
    with pytest.raises(ValueError):
        align.word_spans(spans, [[4], [2]])
