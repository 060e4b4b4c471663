"""Forward-backward posteriors of CTC alignments on the B200 (kab_plan_ctc_posteriors_device, DESIGN.md 3.9f):
every lattice against the float64 restatement (tests/ctc_posteriors_np.py) -- log-likelihood within
max(1e-3, 2e-6 |ref|), posteriors within 1e-4 (T <= 4000) or 1e-3 -- across the three block sizes and the state
limit, every route of the alignment (warp, band, wide, generic; default, long-form and banded plans), wide
vocabularies, ties, masks and statuses, a long planted chapter, arbitrary state paths and the entry points."""
import numpy as np
import pytest

from tests.ctc_posteriors_np import ctc_posteriors_batch_np
from tests.forced_align_band_np import forced_align_band_batch_np
from tests.test_gpu_forced_align import _flat
from tests.test_gpu_forced_align_band import _planted_lp, _planted_path, _random_lp, _targets

pytestmark = pytest.mark.gpu

MAX_STATES = 28000


@pytest.fixture(scope="module")
def kab():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from kokoro_align_b200 import align
    return align


def _check_values(post, ll, lp, t_off, labels, l_off, path, status, blank, W, what=""):
    rpost, rll = ctc_posteriors_batch_np(lp, t_off, labels, l_off, path, status, blank, W)
    for b in range(len(t_off) - 1):
        a, e = int(t_off[b]), int(t_off[b + 1])
        if status[b] != 0:
            assert np.isnan(ll[b]) and not post[a:e].any(), f"{what}lattice {b}"
            continue
        if rll[b] == -np.inf:
            assert ll[b] == -np.inf and not post[a:e].any(), f"{what}lattice {b}"
            continue
        assert abs(ll[b] - rll[b]) <= max(1e-3, 2e-6 * abs(rll[b])), f"{what}lattice {b}: {ll[b]} vs {rll[b]}"
        tol = 1e-4 if e - a <= 4000 else 1e-3
        err = np.abs(post[a:e].astype(np.float64) - rpost[a:e]).max()
        assert err <= tol, f"{what}lattice {b} (T = {e - a}): posterior error {err}"


def _run(kab, lp, t_off, labels, l_off, V, blank, W=None, long_form=False, path=None, stream=None):
    """Align and take the posteriors of the Viterbi path (or of `path`); returns numpy outputs."""
    import torch
    with kab.AlignPlan.ctc(t_off, labels, l_off, V, blank, long_form=long_form, beam_size=W) as plan:
        d_lp = torch.from_numpy(lp).cuda()
        best, labs, sc, final, st = plan.run_torch(d_lp)
        if path is not None:
            best = torch.from_numpy(np.ascontiguousarray(path, np.int32)).cuda()
        post, ll = plan.ctc_posteriors_torch(d_lp, best, st, stream=stream)
        if stream is not None:
            stream.synchronize()
        return (best.cpu().numpy(), st.cpu().numpy(), post.cpu().numpy(), ll.cpu().numpy(), plan.info)


def _check(kab, lp, t_off, labels, l_off, V, blank, W=None, long_form=False, what="", planted=False):
    """planted: one lattice built around a path that fits (status 0), too large for the alignment restatement."""
    path, st, post, ll, info = _run(kab, lp, t_off, labels, l_off, V, blank, W, long_form)
    rst = np.zeros(len(t_off) - 1, np.int32) if planted else forced_align_band_batch_np(lp, t_off, labels, l_off, blank, W)[4]
    np.testing.assert_array_equal(st, rst)
    _check_values(post, ll, lp, t_off, labels, l_off, path, st, blank, W, what)
    return path, st, post, ll, info


def _items(rng, shapes, V, blank, quant=None, neginf=0.0, pool=None):
    return [(_random_lp(rng, T, V, quant, neginf), _targets(rng, L, V, blank, pool=pool)) for T, L in shapes]


@pytest.mark.parametrize("W,shapes", [
    (None, [(300, 1), (400, 125), (500, 126), (600, 127)]),             # np 3 .. 129: 64 -> 256 threads
    (None, [(2100, 1021), (2100, 1022), (2400, 1023)]),                  # np 512 .. 1025: 256 -> 1024 threads
    (252, [(900, 400)]), (253, [(900, 400)]), (2044, [(3000, 1400)]), (2045, [(3000, 1400)]),
])
def test_block_size_boundaries(kab, W, shapes):
    rng = np.random.default_rng(len(shapes) * 1000 + (W or 0))
    lp, t_off, labels, l_off = _flat(_items(rng, shapes, 32, 0))
    _check(kab, lp, t_off, labels, l_off, 32, 0, W, long_form=True)


def test_state_limit(kab):
    import torch
    rng = np.random.default_rng(28000)
    L = 14500   # S = 29001: the window min(W, S) decides
    tg = _targets(rng, L, 32, 0, repeat_p=0.0)
    states = _planted_path(16000, tg)
    lp = _planted_lp(rng, states, tg, 32, 0)
    lp, t_off, labels, l_off = _flat([(lp, tg)])
    _check(kab, lp, t_off, labels, l_off, 32, 0, MAX_STATES, what="W = limit: ", planted=True)
    with pytest.raises(ValueError, match="beam_size"):
        kab.forced_align(torch.from_numpy(lp)[None], torch.from_numpy(tg)[None].long(), beam_size=MAX_STATES + 1,
                         posteriors=True)
    with kab.AlignPlan.ctc(t_off, labels, l_off, 32, 0, beam_size=MAX_STATES + 1) as plan:
        d_lp = torch.from_numpy(lp).cuda()
        path, _, _, _, st = plan.run_torch(d_lp)
        with pytest.raises(kab.KabError, match="unsupported"):
            plan.ctc_posteriors_torch(d_lp, path, st)


def test_routes_of_default_and_long_form_plans(kab):
    rng = np.random.default_rng(11)
    shapes = [(60, 20), (150, 60), (700, 300), (2000, 900), (8000, 1700)]   # warp, band and generic lattices
    lp, t_off, labels, l_off = _flat(_items(rng, shapes, 32, 0))
    _, _, _, _, info = _check(kab, lp, t_off, labels, l_off, 32, 0)
    assert info.n_class[0] and info.n_class[1] and info.n_class[2]
    # the 10-minute utterance of 3.9b on the wide kernel (S = 18 001)
    tg = _targets(rng, 9000, 32, 0)
    states = _planted_path(30000, tg, amp=40.0, cycles=3.0)
    lp1, t1, l1, lo1 = _flat([(_planted_lp(rng, states, tg, 32, 0, bonus=4.0), tg)])
    _, _, _, _, info = _check(kab, lp1, t1, l1, lo1, 32, 0, long_form=True, what="wide: ", planted=True)
    assert info.n_class[3] == 1


def test_banded_plans_whose_windows_clip(kab):
    rng = np.random.default_rng(12)
    items = []
    for T, L, amp in [(800, 300, 10.0), (3000, 1200, 30.0), (5000, 2000, 60.0)]:
        tg = _targets(rng, L, 32, 0)
        items.append((_planted_lp(rng, _planted_path(T, tg, amp=amp), tg, 32, 0, bonus=3.0), tg))
    lp, t_off, labels, l_off = _flat(items)
    for W in (64, 200, 1000):
        _check(kab, lp, t_off, labels, l_off, 32, 0, W, what=f"W = {W}: ")


def test_wide_vocabulary(kab):
    rng = np.random.default_rng(13)
    V, blank = 1025, 1024
    items = _items(rng, [(300, 100), (900, 400), (2000, 700)], V, blank)
    items[2] = (items[2][0], rng.permutation(1024)[:700].astype(np.int32))   # > 511 distinct ids: the generic route
    lp, t_off, labels, l_off = _flat(items)
    _, _, _, _, info = _check(kab, lp, t_off, labels, l_off, V, blank)
    assert info.n_class[2] >= 1
    _check(kab, lp, t_off, labels, l_off, V, blank, 300, what="banded: ")
    # rows read from global memory: a window too wide for the ring of 1025-column rows next to the state buffers
    tg = _targets(rng, 13900, V, blank, repeat_p=0.0)
    big = _flat([(_planted_lp(rng, _planted_path(15500, tg), tg, V, blank), tg)])
    _check(kab, *big, V, blank, 27800, what="unstaged rows: ", planted=True)


def test_ties_masks_and_statuses(kab):
    rng = np.random.default_rng(14)
    items = _items(rng, [(200, 50), (300, 100), (120, 40)], 8, 3, quant=2.0)          # tie-heavy
    items += _items(rng, [(250, 60), (400, 150)], 8, 3, neginf=0.3)                    # -inf masks
    nan_lp = _random_lp(rng, 100, 8)
    nan_lp[37, 2] = np.nan
    items.append((nan_lp, _targets(rng, 20, 8, 3)))                                    # status 3
    items.append((_random_lp(rng, 50, 8), np.array([1, 9, 2], np.int32)))              # status 2: bad label
    items.append((_random_lp(rng, 4, 8), np.array([1, 1, 1], np.int32)))              # status 1: T < L + R
    dead = _random_lp(rng, 40, 8)
    dead[-1, :] = -np.inf                                                              # both end states -inf
    items.append((dead, _targets(rng, 10, 8, 3)))
    lp, t_off, labels, l_off = _flat(items)
    _, st, post, ll, _ = _check(kab, lp, t_off, labels, l_off, 8, 3)
    assert list(st[-4:]) == [3, 2, 1, 0] and ll[-1] == -np.inf
    # a band that loses every path: status 1 in a banded plan
    lost = _random_lp(rng, 40, 8)
    tg = np.array([1, 2, 4], np.int32)
    lost[:35, tg] = -np.inf
    lp2, t2, l2, lo2 = _flat(items[:2] + [(lost, tg)])
    _, st, _, _, _ = _check(kab, lp2, t2, l2, lo2, 8, 3, 2)
    assert st[-1] == 1


def test_planted_chapter_under_beam(kab):
    rng = np.random.default_rng(15)
    tg = _targets(rng, 6000, 32, 0)
    states = _planted_path(36000, tg, amp=80.0, cycles=5.0)
    lp, t_off, labels, l_off = _flat([(_planted_lp(rng, states, tg, 32, 0, bonus=5.0), tg)])
    path, _, post, _, _ = _check(kab, lp, t_off, labels, l_off, 32, 0, 1000, planted=True)
    assert np.median(post) > 0.5


def test_arbitrary_state_paths(kab):
    rng = np.random.default_rng(16)
    items = _items(rng, [(300, 80), (1000, 300)], 32, 0)
    lp, t_off, labels, l_off = _flat(items)
    for W in (None, 120):
        n = int(t_off[-1])
        path = np.concatenate([np.clip(np.cumsum(rng.integers(-1, 3, int(t_off[b + 1] - t_off[b]))), -2,
                                       2 * int(l_off[b + 1] - l_off[b]) + 2) for b in range(2)]).astype(np.int32)
        path[rng.random(n) < 0.05] = -1
        got_path, st, post, ll, _ = _run(kab, lp, t_off, labels, l_off, 32, 0, W, path=path)
        _check_values(post, ll, lp, t_off, labels, l_off, path, st, 0, W, f"W = {W}: ")


def test_posteriors_keep_the_alignment_and_match_ctc_loss(kab):
    import torch
    rng = np.random.default_rng(17)
    B, T_max, V = 6, 400, 32
    lp = torch.from_numpy(np.stack([_random_lp(rng, T_max, V) for _ in range(B)]))
    tl = torch.tensor([400, 350, 120, 399, 200, 64])
    ll_t = torch.tensor([100, 90, 40, 150, 3, 20])
    tg = torch.from_numpy(np.stack([np.pad(_targets(rng, int(n), V, 0), (0, 150 - int(n)), constant_values=1)
                                    for n in ll_t])).long()
    for dev in ("cuda", "cpu"):
        x, y = lp.to(dev), tg.to(dev)
        p0, s0 = kab.forced_align_batch(x, y, tl, ll_t)
        p1, s1, post, loglik = kab.forced_align_batch(x, y, tl, ll_t, posteriors=True)
        assert post.device.type == dev and loglik.dtype == torch.float64 and post.shape == s1.shape
        assert p0.cpu().numpy().tobytes() == p1.cpu().numpy().tobytes()
        assert s0.cpu().numpy().tobytes() == s1.cpu().numpy().tobytes()
        for b in range(B):
            assert not post[b, int(tl[b]):].any()
        ref = -torch.nn.functional.ctc_loss(lp.double().transpose(0, 1), tg, tl, ll_t, blank=0, reduction="none")
        err = np.abs(loglik.cpu().numpy() - ref.numpy())
        assert (err <= np.maximum(1e-3, 2e-6 * np.abs(ref.numpy()))).all(), err
        spans = kab.merge_tokens_batch(p1, post, tl)
        assert bool(((spans.score >= 0) & (spans.score <= 1)).all())
    # one item, forced_align, on a non-default stream and on the CPU
    x, y = lp[:1, :350], tg[:1, :90]
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        p, sc, post, loglik = kab.forced_align(x.cuda(), y.cuda(), posteriors=True)
    s.synchronize()
    pc, scc, postc, loglikc = kab.forced_align(x, y, posteriors=True)
    assert postc.device.type == "cpu" and torch.equal(post.cpu(), postc) and torch.equal(loglik.cpu(), loglikc)
    assert torch.equal(pc, p.cpu()) and loglik.shape == (1,)
    ref = -torch.nn.functional.ctc_loss(x.double().transpose(0, 1), y, torch.tensor([350]), torch.tensor([90]), blank=0,
                                        reduction="sum")
    assert abs(float(loglik[0]) - float(ref)) <= max(1e-3, 2e-6 * abs(float(ref)))


def test_non_default_stream_and_rejections(kab):
    import torch
    rng = np.random.default_rng(18)
    lp, t_off, labels, l_off = _flat(_items(rng, [(300, 100), (500, 200)], 32, 0))
    s = torch.cuda.Stream()
    path, st, post, ll, _ = _run(kab, lp, t_off, labels, l_off, 32, 0, stream=s)
    _check_values(post, ll, lp, t_off, labels, l_off, path, st, 0, None)
    x, y = torch.from_numpy(lp[:300])[None], torch.from_numpy(labels[:100])[None].long()
    with pytest.raises(ValueError, match="free_ends"):
        kab.forced_align(x, y, free_ends=True, posteriors=True)
    with pytest.raises(ValueError, match="free_ends"):
        kab.forced_align_batch(x, y, free_ends=True, posteriors=True)
    with pytest.raises(ValueError, match=r"item 1: .*S = 30001"):
        kab.forced_align_batch(torch.zeros(2, 16000, 32), (torch.arange(15000) % 2 + 1).repeat(2, 1),
                               target_lengths=torch.tensor([10, 15000]), posteriors=True)
    d_lp = torch.from_numpy(lp).cuda()
    with kab.AlignPlan.ctc(t_off, labels, l_off, 32, 0, free_ends=True) as plan:
        path, _, _, _, st = plan.run_torch(d_lp)
        with pytest.raises(kab.KabError, match="unsupported"):
            plan.ctc_posteriors_torch(d_lp, path, st)
    with kab.AlignPlan(t_off, labels, l_off, 32, 1000, 4) as plan:   # a Kokoro-mode plan
        path, _, _, _, st = plan.run_torch(d_lp)
        with pytest.raises(kab.KabError, match="unsupported"):
            plan.ctc_posteriors_torch(d_lp, path, st)
