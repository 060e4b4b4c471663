"""Forward-backward posteriors of unbanded long-form lattices above KAB_POSTERIOR_MAX_STATES on the chain-of-warps
pass (kab_ctc_posterior_chain_kernel, DESIGN.md 3.9g), held to the float64 restatement (tests/ctc_posteriors_np.py)
at 3.9f's tolerances: log-likelihood within max(1e-3, 2e-6 |ref|), posteriors within 1e-4 (T <= 4000) or 1e-3.

KAB_POSTERIOR_CHAIN_MIN_STATES (read at a plan's first posterior call) moves smaller lattices of long-form plans
onto the chain, so that its slice geometry (128 pairs = 256 states per warp), FIFO and value edges are checked on
lattices the restatement handles in seconds, and against the single-CTA kernel on the same inputs.
KAB_POSTERIOR_CHAIN_SERIAL runs the two directions one after the other, as on a grid too large for both."""
import numpy as np
import pytest

from tests.test_gpu_ctc_posteriors import _check_values
from tests.test_gpu_forced_align import _flat
from tests.test_gpu_forced_align_band import _planted_lp, _planted_path, _random_lp, _targets

pytestmark = pytest.mark.gpu

MAX_STATES = 28000
LONG_MAX_STATES = 324001


@pytest.fixture(scope="module")
def kab():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from kokoro_align_b200 import align
    return align


@pytest.fixture
def chain(monkeypatch):
    """Every lattice of a long-form plan created from here on takes the chain pass."""
    monkeypatch.setenv("KAB_POSTERIOR_CHAIN_MIN_STATES", "0")
    return monkeypatch


def _run(kab, lp, t_off, labels, l_off, V, blank, path=None, stream=None, long_form=True, W=None):
    import torch
    with kab.AlignPlan.ctc(t_off, labels, l_off, V, blank, long_form=long_form, beam_size=W) as plan:
        d_lp = torch.from_numpy(lp).cuda()
        best, _, sc, _, st = plan.run_torch(d_lp)
        if path is not None:
            best = torch.from_numpy(np.ascontiguousarray(path, np.int32)).cuda()
        post, ll = plan.ctc_posteriors_torch(d_lp, best, st, stream=stream)
        if stream is not None:
            stream.synchronize()
        return best.cpu().numpy(), sc.cpu().numpy(), st.cpu().numpy(), post.cpu().numpy(), ll.cpu().numpy(), plan.info


def _check_chain(kab, monkeypatch, items, V, blank, path=None, what=""):
    """The chain pass (both directions side by side, then one after the other: the same bytes) against the
    restatement and against the single-CTA pass on the same inputs."""
    lp, t_off, labels, l_off = _flat(items)
    monkeypatch.delenv("KAB_POSTERIOR_CHAIN_MIN_STATES", raising=False)
    best, _, st, post1, ll1, _ = _run(kab, lp, t_off, labels, l_off, V, blank, path)
    monkeypatch.setenv("KAB_POSTERIOR_CHAIN_MIN_STATES", "0")
    best2, _, st2, post, ll, _ = _run(kab, lp, t_off, labels, l_off, V, blank, path)
    assert np.array_equal(best, best2) and np.array_equal(st, st2)
    _check_values(post, ll, lp, t_off, labels, l_off, best, st, blank, None, what)
    ok = st == 0
    np.testing.assert_allclose(ll[ok], ll1[ok], rtol=2e-6, atol=1e-3)
    assert np.abs(post.astype(np.float64) - post1).max() <= 1e-3
    monkeypatch.setenv("KAB_POSTERIOR_CHAIN_SERIAL", "1")
    _, _, _, post_s, ll_s, _ = _run(kab, lp, t_off, labels, l_off, V, blank, path)
    monkeypatch.delenv("KAB_POSTERIOR_CHAIN_SERIAL")
    assert post_s.tobytes() == post.tobytes() and ll_s.tobytes() == ll.tobytes()
    return best, st, post, ll


def _random_items(rng, shapes, V=32, blank=0, **kw):
    return [(_random_lp(rng, T, V), _targets(rng, L, V, blank, **kw)) for T, L in shapes]


@pytest.mark.parametrize("shapes", [
    [(1, 1), (5, 2), (16, 6), (300, 126)],                   # T = 1, T within the start-up lag; S = 253: one warp
    [(400, 127), (400, 128), (500, 129)],                    # S = 255 (one warp), 257 (S-1 alone in warp 1), 259
    [(700, 255), (700, 256), (900, 383), (900, 384)],        # two warps exactly, one state more; three / four
])
def test_slice_geometry(kab, chain, shapes):
    rng = np.random.default_rng(sum(L for _, L in shapes))
    _check_chain(kab, chain, _random_items(rng, shapes), 32, 0)


def test_repeated_labels_across_warp_boundaries(kab, chain):
    """Move 2 is forbidden between equal labels: here across the forward boundary (labels 127 / 128: states
    255 and 257, pairs of warps 0 and 1) and the backward one (labels 126 / 127: states 253 and 255), and in
    the middle of a warp."""
    rng = np.random.default_rng(21)
    items = []
    for reps in ([127], [126], [126, 127, 255], [60]):
        tg = _targets(rng, 400, 32, 0, repeat_p=0.0)
        for r in reps:
            tg[r + 1] = tg[r]
        items.append((_random_lp(rng, 900, 32), tg))
    _check_chain(kab, chain, items, 32, 0)


def test_fifo_lapping(kab, chain):
    """5 warps per direction over 375 groups of 8 frames: the 32-message FIFOs lap about 12 times."""
    rng = np.random.default_rng(22)
    tg = _targets(rng, 600, 32, 0)
    items = [(_planted_lp(rng, _planted_path(3000, tg, amp=30.0, cycles=4.0), tg, 32, 0, bonus=2.0), tg)]
    items += _random_items(rng, [(2500, 700)])
    _check_chain(kab, chain, items, 32, 0)


def test_masks_dead_ends_and_statuses(kab, chain):
    rng = np.random.default_rng(23)
    items = []
    tg = _targets(rng, 300, 8, 3)
    st = _planted_path(1200, tg, amp=20.0)
    lp = _planted_lp(rng, st, tg, 8, 3, bonus=2.0)
    lp[rng.random(lp.shape) < 0.05] = -np.inf         # -inf masks, some on the planted path
    ext = np.full(601, 3)
    ext[1::2] = tg
    lp[np.arange(1200)[::97], ext[st[::97]]] = -np.inf
    items.append((lp, tg))
    dead = _random_lp(rng, 800, 8)
    dead[-1, :] = -np.inf                              # both end states -inf: log Z = -inf, posteriors 0
    items.append((dead, _targets(rng, 300, 8, 3)))
    nan_lp = _random_lp(rng, 700, 8)
    nan_lp[345, 2] = np.nan                            # status 3
    items.append((nan_lp, _targets(rng, 260, 8, 3)))
    items.append((_random_lp(rng, 500, 8), np.r_[_targets(rng, 200, 8, 3), 9].astype(np.int32)))   # status 2
    items.append((_random_lp(rng, 300, 8), np.ones(299, np.int32)))                               # status 1
    items += [(_random_lp(rng, 600, 8, quant=2.0), _targets(rng, 270, 8, 3))]                     # ties
    best, st, post, ll = _check_chain(kab, chain, items, 8, 3)
    assert list(st[1:5]) == [0, 3, 2, 1] and ll[1] == -np.inf and np.isnan(ll[2:5]).all()


def test_arbitrary_state_paths(kab, chain):
    rng = np.random.default_rng(24)
    items = _random_items(rng, [(700, 260), (1500, 600)])
    t_off = np.cumsum([0] + [x[0].shape[0] for x in items])
    path = np.concatenate([np.clip(np.cumsum(rng.integers(-1, 3, x[0].shape[0])), -3, 2 * len(x[1]) + 3)
                           for x in items]).astype(np.int32)
    path[rng.random(int(t_off[-1])) < 0.05] = -1
    path[rng.random(int(t_off[-1])) < 0.02] = 100000    # outside [0, S)
    _check_chain(kab, chain, items, 32, 0, path=path)


def test_wide_vocabulary(kab, chain):
    rng = np.random.default_rng(25)
    V, blank = 1025, 1024
    items = _random_items(rng, [(900, 300)], V, blank)
    items.append((_random_lp(rng, 1500, V), rng.permutation(1024)[:700].astype(np.int32)))   # > 511 distinct ids
    _check_chain(kab, chain, items, V, blank)


def _long_item(rng, T, L, V=32, blank=0, amp=40.0, cycles=3.0, bonus=4.0, pool=None):
    tg = _targets(rng, L, V, blank, repeat_p=0.05, pool=pool)
    return _planted_lp(rng, _planted_path(T, tg, amp=amp, cycles=cycles), tg, V, blank, bonus=bonus), tg


def test_just_above_the_limit(kab):
    """S = 28 001 and S = 40 001 over 60 000 frames, on the default route of long-form plans."""
    rng = np.random.default_rng(26)
    for T, L in [(16000, 14000), (60000, 20000)]:
        lp, t_off, labels, l_off = _flat([_long_item(rng, T, L)])
        best, _, st, post, ll, info = _run(kab, lp, t_off, labels, l_off, 32, 0)
        assert st[0] == 0 and info.n_class[3] == 1
        _check_values(post, ll, lp, t_off, labels, l_off, best, st, 0, None, f"S = {2 * L + 1}: ")


def test_mixed_plan_keeps_the_short_lattices(kab):
    """A long lattice next to warp, band, generic and wide-class short ones (V = 1025: an item with more than 511
    distinct ids aligns on the generic kernel): the short ones get exactly the bytes of a plan without it."""
    rng = np.random.default_rng(27)
    V, blank, pool = 1025, 1024, np.arange(200, 500)
    short = _random_items(rng, [(60, 20), (150, 60), (700, 300)], V, blank)
    short.append((_random_lp(rng, 1500, V), rng.permutation(1024)[:600].astype(np.int32)))
    short.append(_long_item(rng, 12000, 3000, V, blank, pool=pool))           # S = 6001: the wide kernel
    long_ = _long_item(rng, 20000, 15000, V, blank, amp=20.0, pool=pool)      # S = 30 001: the chain
    lp0, t0, lab0, lo0 = _flat(short)
    _, _, st0, post0, ll0, info0 = _run(kab, lp0, t0, lab0, lo0, V, blank)
    assert info0.n_class[2] and info0.n_class[3] and info0.n_class[0] + info0.n_class[1] == 3
    lp, t_off, labels, l_off = _flat(short[:2] + [long_] + short[2:])
    best, _, st, post, ll, _ = _run(kab, lp, t_off, labels, l_off, V, blank)
    _check_values(post, ll, lp, t_off, labels, l_off, best, st, blank, None)
    keep = np.r_[0:2, 3:len(short) + 1]
    assert ll[keep].tobytes() == ll0.tobytes()
    rows = np.concatenate([np.arange(t_off[b], t_off[b + 1]) for b in keep])
    assert post[rows].tobytes() == post0.tobytes()


def test_one_hour_chapter_against_a_covering_band(kab):
    """T = 180 000, L = 54 000 (S = 108 001) on planted emissions: the unbanded log Z is no smaller than the
    band's at beam_size = 20 000 (which holds practically all the mass), and both agree; so do the posteriors.
    posteriors=True leaves the paths and scores of the long-form alignment byte for byte."""
    import torch
    rng = np.random.default_rng(28)
    lp, tg = _long_item(rng, 180000, 54000, amp=60.0, cycles=5.0, bonus=4.0)
    x, y = torch.from_numpy(lp)[None], torch.from_numpy(tg)[None].long()
    p0, s0 = kab.forced_align(x.cuda(), y.cuda(), long_form=True)
    p1, s1, post, ll = kab.forced_align(x.cuda(), y.cuda(), long_form=True, posteriors=True)
    assert p0.cpu().numpy().tobytes() == p1.cpu().numpy().tobytes()
    assert s0.cpu().numpy().tobytes() == s1.cpu().numpy().tobytes()
    lpf, t_off, labels, l_off = _flat([(lp, tg)])
    best, _, st, post2, ll2, info = _run(kab, lpf, t_off, labels, l_off, 32, 0)
    assert st[0] == 0 and info.n_class[3] == 1
    assert post2.tobytes() == post.cpu().numpy()[0].tobytes() and ll2.tobytes() == ll.cpu().numpy().tobytes()
    _, _, stb, postb, llb, _ = _run(kab, lpf, t_off, labels, l_off, 32, 0, path=best, long_form=False, W=20000)
    assert stb[0] == 0
    z, zb = float(ll2[0]), float(llb[0])
    tol = max(1e-3, 2e-6 * abs(zb))
    assert z >= zb - tol and abs(z - zb) <= tol, (z, zb)
    assert np.abs(post2.astype(np.float64) - postb).max() <= 1e-3
    assert float(np.median(post2)) > 0.5


def test_entry_points(kab):
    import torch
    rng = np.random.default_rng(29)
    items = [_long_item(rng, 18000, 14500, amp=15.0), (_random_lp(rng, 18000, 32), _targets(rng, 300, 32, 0))]
    T_max, L_max = 18000, 14500
    lp = torch.from_numpy(np.stack([x[0] for x in items]))
    tg = torch.from_numpy(np.stack([np.pad(x[1], (0, L_max - len(x[1])), constant_values=1) for x in items])).long()
    tl, ll_t = torch.tensor([18000, 18000]), torch.tensor([14500, 300])
    ref = -torch.nn.functional.ctc_loss(lp.double().cuda().transpose(0, 1), tg.cuda(), tl, ll_t, blank=0,
                                        reduction="none").cpu().numpy()
    outs = {}
    for dev in ("cuda", "cpu"):
        p0, s0 = kab.forced_align_batch(lp.to(dev), tg.to(dev), tl, ll_t, long_form=True)
        p1, s1, post, loglik = kab.forced_align_batch(lp.to(dev), tg.to(dev), tl, ll_t, long_form=True, posteriors=True)
        assert post.device.type == dev and loglik.dtype == torch.float64 and post.shape == (2, T_max)
        assert torch.equal(p0, p1) and torch.equal(s0, s1)
        assert (np.abs(loglik.cpu().numpy() - ref) <= np.maximum(1e-3, 2e-6 * np.abs(ref))).all()
        outs[dev] = post.cpu(), loglik.cpu()
    assert torch.equal(outs["cuda"][0], outs["cpu"][0]) and torch.equal(outs["cuda"][1], outs["cpu"][1])
    x, y = lp[:1], tg[:1]
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        p, sc, post, loglik = kab.forced_align(x.cuda(), y.cuda(), long_form=True, posteriors=True)
    s.synchronize()
    assert torch.equal(post.cpu(), outs["cpu"][0][:1]) and torch.equal(loglik.cpu(), outs["cpu"][1][:1])
    pc, scc, postc, loglikc = kab.forced_align(x, y, long_form=True, posteriors=True)
    assert postc.device.type == "cpu" and torch.equal(postc, post.cpu()) and torch.equal(loglikc, loglik.cpu())


def test_limits_and_refusals(kab):
    import torch
    # above the long-form limit: ValueError naming the item and its S
    L = (LONG_MAX_STATES + 1) // 2
    with pytest.raises(ValueError, match=rf"item 1: .*S = {2 * L + 1}"):
        kab.forced_align_batch(torch.zeros(2, L + 10, 32), (torch.arange(L) % 2 + 1).repeat(2, 1),
                               target_lengths=torch.tensor([10, L]), long_form=True, posteriors=True)
    # default, banded and free-ends plans still refuse windows above KAB_POSTERIOR_MAX_STATES
    rng = np.random.default_rng(30)
    lp, t_off, labels, l_off = _flat([_long_item(rng, 20000, 14500, amp=10.0)])
    d_lp = torch.from_numpy(lp).cuda()
    for kw in ({}, {"beam_size": MAX_STATES + 1}, {"beam_size": 40000}, {"long_form": True, "free_ends": True}):
        with kab.AlignPlan.ctc(t_off, labels, l_off, 32, 0, **kw) as plan:
            path, _, _, _, st = plan.run_torch(d_lp)
            with pytest.raises(kab.KabError, match="unsupported"):
                plan.ctc_posteriors_torch(d_lp, path, st)
    x, y = torch.from_numpy(lp)[None], torch.from_numpy(labels)[None].long()
    with pytest.raises(ValueError, match="beam_size"):
        kab.forced_align(x, y, posteriors=True)
    with pytest.raises(ValueError, match="free_ends"):
        kab.forced_align(x, y, long_form=True, free_ends=True, posteriors=True)
