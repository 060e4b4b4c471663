"""The CPU restatement of CTC forced alignment (oracle/forced_align_np.py) against the goldens
written from torchaudio's forced_align, and against live torchaudio where it can be imported; the
argument checks of forced_align / forced_align_batch that run before any device work."""
import os

import numpy as np
import pytest

from oracle.forced_align_np import forced_align_batch_np, forced_align_np

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "forced_align_golden.npz")


def load_cases():
    z = np.load(GOLDEN)
    names = sorted({k.split("__")[0] for k in z.files})
    return [(n, {k.split("__")[1]: z[k] for k in z.files if k.split("__")[0] == n}) for n in names]


CASES = load_cases()


@pytest.mark.parametrize("name,case", CASES, ids=[n for n, _ in CASES])
def test_restatement_matches_golden(name, case):
    states, paths, scores, final = forced_align_np(case["lp"], case["targets"], int(case["blank"]))
    np.testing.assert_array_equal(states, case["states"])
    np.testing.assert_array_equal(paths, case["paths"])
    assert scores.tobytes() == case["scores"].tobytes()
    assert final.tobytes() == case["final"].tobytes()


def test_golden_covers_the_issue_cases():
    names = [n for n, _ in CASES]
    for prefix in ("ties", "tight", "label0", "neginf", "deadend", "S247", "S249", "S3295", "S3297", "V512"):
        assert any(n.startswith(prefix) for n in names), prefix
    vs = {int(c["lp"].shape[1]) for _, c in CASES}
    assert {5, 32, 512} <= vs
    blanks = {(int(c["blank"]), int(c["lp"].shape[1])) for _, c in CASES}
    assert any(b == 0 for b, _ in blanks) and any(b == v - 1 for b, v in blanks) and any(0 < b < v - 1 for b, v in blanks)
    # end states both -inf: the restatement's outputs (torchaudio's are undefined there)
    assert sum(int(c["torchaudio"]) == 0 for _, c in CASES) >= 1


def _torchaudio():
    try:
        import torch
        import torchaudio.functional as F
        F.forced_align(torch.zeros(1, 2, 3), torch.ones(1, 1, dtype=torch.int32))
        return torch, F
    except Exception:  # noqa: BLE001 -- not installed, or built without the alignment op
        pytest.skip("torchaudio's forced_align is not available")


def test_golden_matches_live_torchaudio():
    torch, F = _torchaudio()
    for name, c in CASES:
        if not int(c["torchaudio"]):
            continue
        p, s = F.forced_align(torch.from_numpy(c["lp"])[None], torch.from_numpy(c["targets"])[None],
                              blank=int(c["blank"]))
        np.testing.assert_array_equal(p[0].numpy(), c["paths"], err_msg=name)
        assert s[0].numpy().tobytes() == c["scores"].tobytes(), name


@pytest.mark.parametrize("seed", range(4))
def test_restatement_matches_live_torchaudio(seed):
    """Random small lattices, half on a 1/2 grid (ties), some with -inf entries and tight lengths."""
    torch, F = _torchaudio()
    rng = np.random.default_rng(1000 + seed)
    for it in range(60):
        V = int(rng.integers(3, 41))
        blank = int(rng.integers(0, V))
        L = int(rng.integers(1, 12))
        tg = rng.choice([x for x in range(V) if x != blank], L)
        if it % 3 == 0:
            tg[1:] = np.where(rng.random(L - 1) < 0.5, tg[:-1], tg[1:])
        R = int((tg[1:] == tg[:-1]).sum())
        T = L + R + int(rng.integers(0, 12))
        lp = np.log(rng.dirichlet(np.ones(V), T)).astype(np.float32)
        if it % 2:
            lp = (np.round(lp * 2) / 2).astype(np.float32)
        if it % 5 == 0:
            lp[rng.random(lp.shape) < 0.2] = -np.inf
        _, paths, scores, final = forced_align_np(lp, tg, blank)
        if not np.isfinite(final):
            continue   # (torchaudio's traceback is undefined there)
        p, s = F.forced_align(torch.from_numpy(lp)[None], torch.from_numpy(tg.astype(np.int32))[None], blank=blank)
        np.testing.assert_array_equal(p[0].numpy(), paths)
        assert s[0].numpy().tobytes() == scores.tobytes()


@pytest.mark.parametrize("blank", [0, 3, 6])
def test_restatement_empty_transcript(blank):
    """L = 0 (S = 1): state 0 and the blank in every frame, scores lp[:, blank], and as final score their
    float32 running sum from 0 in frame order (-inf from a -inf blank log-prob on)."""
    rng = np.random.default_rng(blank)
    for T in (1, 2, 9, 50):
        lp = np.log(rng.dirichlet(np.ones(7), T)).astype(np.float32)
        if T == 50:
            lp[31, blank] = -np.inf
        states, paths, scores, final = forced_align_np(lp, np.zeros(0, np.int32), blank)
        f = np.float32(0.0)
        for t in range(T):
            f = np.float32(f + lp[t, blank])
        assert (states == 0).all() and (paths == blank).all() and states.dtype == paths.dtype == np.int32
        assert scores.tobytes() == np.ascontiguousarray(lp[:, blank]).tobytes()
        assert final.tobytes() == f.tobytes() and (np.isneginf(final) == (T == 50))
    _, _, _, final, status = forced_align_batch_np(lp, np.array([0, 20, 50]), np.array([(blank + 1) % 7], np.int32),
                                                   np.array([0, 0, 1]), blank)
    assert status.tolist() == [0, 0]


def test_edge_case_generator():
    """The cases of test_gpu_forced_align_edges.py are what their names say."""
    from tests.test_gpu_forced_align_edges import COMPACT_CASES, EDGE_CASES, make_case
    for case in EDGE_CASES + COMPACT_CASES:
        S, V, blank, t_kind, content = case
        lp, tg = make_case(case)
        L, T = len(tg), lp.shape[0]
        R = int((tg[1:] == tg[:-1]).sum())
        assert lp.dtype == np.float32 and lp.shape[1] == V and S == 2 * L + 1, case
        assert ((tg >= 0) & (tg < V) & (tg != blank)).all() and T >= L + R, case
        assert blank == 0 or V == 2 or content == "allrep" or (tg == 0).any(), case
        if t_kind in ("tight", "tight1"):
            assert T == L + R + (t_kind == "tight1"), case
        elif isinstance(t_kind, int):
            assert T == t_kind, case
        else:
            assert T % t_kind[1] == t_kind[0], case
        if content in ("climb", "blankmask"):
            assert R == 0
        if content == "climb":
            assert T == L
        if content == "allrep":
            assert (tg == tg[0]).all()
        if content in ("zero", "const"):
            assert (lp == lp[:, :1]).all()
        if V > 512:
            assert len(set(tg.tolist())) <= 300
    S = np.array([c[0] for c in EDGE_CASES])
    for s in (3, 61, 63, 123, 125, 185, 187, 247, 249, 279, 281, 1631, 1633, 3295):
        assert (S == s).any(), s
    assert {2, 5, 32, 64, 65, 129, 512} == {c[1] for c in EDGE_CASES}


def test_edge_cases_match_live_torchaudio():
    """The restatement against torchaudio's CPU forced_align on every case of test_gpu_forced_align_edges.py
    whose chosen end state is finite; the -inf row and -inf end cases end -inf."""
    torch, F = _torchaudio()
    from tests.test_gpu_forced_align_edges import COMPACT_CASES, EDGE_CASES, case_data, case_id
    n = 0
    for case in EDGE_CASES + COMPACT_CASES:
        blank, content = case[2], case[4]
        lp, tg, (_, paths, scores, final) = case_data(case)
        if content in ("row", "end"):
            assert np.isneginf(final), case_id(case)
            continue
        if content != "mask":
            assert np.isfinite(final), case_id(case)
        if not np.isfinite(final):
            continue
        p, s = F.forced_align(torch.from_numpy(lp)[None], torch.from_numpy(tg)[None], blank=blank)
        np.testing.assert_array_equal(p[0].numpy(), paths, err_msg=case_id(case))
        assert s[0].numpy().tobytes() == scores.tobytes(), case_id(case)
        n += 1
    assert n >= 60


def test_batch_restatement_statuses():
    rng = np.random.default_rng(7)
    lp = np.log(rng.dirichlet(np.ones(5), 13)).astype(np.float32)
    lp[9, 2] = np.nan
    t_off = np.array([0, 4, 6, 12])
    labels = np.array([1, 2, 2, 3, 3, 1, 4, 0], np.int32)   # lattice 1: [3, 3] needs 3 frames, has 2
    l_off = np.array([0, 3, 5, 7, 8])
    _, _, _, final, status = forced_align_batch_np(lp, np.append(t_off, 13), labels, l_off, blank=0)
    assert status.tolist() == [0, 1, 3, 2] and np.isfinite(final[0])


# ---- argument checks of the Python entry points (raised before any device work)

def _fa():
    torch = pytest.importorskip("torch")
    from kokoro_align_b200 import align
    return torch, align


@pytest.mark.parametrize("bad,exc", [
    ("blank_in_targets", ValueError), ("target_ge_V", ValueError), ("negative_target", ValueError),
    ("empty_targets", RuntimeError), ("too_short", RuntimeError), ("batch2", RuntimeError),
    ("input_length_mismatch", RuntimeError), ("target_length_mismatch", RuntimeError),
    ("blank_out_of_range", RuntimeError), ("float64", RuntimeError), ("2d", RuntimeError)])
def test_forced_align_argument_errors(bad, exc):
    torch, align = _fa()
    lp = torch.randn(1, 10, 5).log_softmax(-1)
    tg = torch.tensor([[1, 2, 2]], dtype=torch.int32)
    kw = {}
    if bad == "blank_in_targets":
        tg = torch.tensor([[1, 0, 2]], dtype=torch.int32)
    elif bad == "target_ge_V":
        tg = torch.tensor([[1, 5]], dtype=torch.int32)
    elif bad == "negative_target":
        tg = torch.tensor([[1, -2]], dtype=torch.int32)
    elif bad == "empty_targets":
        tg = torch.zeros(1, 0, dtype=torch.int32)
    elif bad == "too_short":
        tg = torch.tensor([[1, 1, 1, 1, 1, 1]], dtype=torch.int32)   # L + R = 11 > 10
    elif bad == "batch2":
        lp, tg = lp.expand(2, -1, -1), tg.expand(2, -1)
    elif bad == "input_length_mismatch":
        kw["input_lengths"] = torch.tensor([9])
    elif bad == "target_length_mismatch":
        kw["target_lengths"] = torch.tensor([2])
    elif bad == "blank_out_of_range":
        kw["blank"] = 7
    elif bad == "float64":
        lp = lp.double()
    elif bad == "2d":
        lp = lp[0]
    with pytest.raises(exc):
        align.forced_align(lp, tg, **kw)


def test_forced_align_batch_names_the_failing_item():
    torch, align = _fa()
    lp = torch.randn(3, 10, 5).log_softmax(-1)
    tg = torch.tensor([[1, 2, 0], [3, 3, 3], [1, 0, 0]], dtype=torch.int64)
    with pytest.raises(RuntimeError, match="item 1"):   # [3, 3, 3] needs 5 frames, item 1 has 4
        align.forced_align_batch(lp, tg, torch.tensor([10, 4, 10]), torch.tensor([2, 3, 1]))
    with pytest.raises(ValueError, match="item 2"):
        align.forced_align_batch(lp, tg, torch.tensor([10, 10, 10]), torch.tensor([2, 3, 2]))
