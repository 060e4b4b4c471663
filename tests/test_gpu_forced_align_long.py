"""Long-form CTC forced alignment on the B200 (kab_plan_create_ctc_long, long_form=True): lattices with
more than 3296 states on the wide kernel (kab_wide_ctc_kernel), bit-exact against the restatement and
torchaudio's CPU forced_align, and byte-equal to the default plans, which run them on the generic kernel."""
import functools
import types

import numpy as np
import pytest

from oracle.forced_align_np import forced_align_batch_np, forced_align_np
from tests.test_gpu_forced_align import _check_plan as _check_plan_default
from tests.test_gpu_forced_align import _flat, _random_items, _torchaudio

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def kab():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from kokoro_align_b200 import align
    return align


def _check_plan(kab, lp, t_off, labels, l_off, V, blank, ta_check=True, long_form=True):
    """_check_plan of the default-plan tests, on a plan built with AlignPlan.ctc(..., long_form)."""
    shim = types.SimpleNamespace(AlignPlan=types.SimpleNamespace(ctc=functools.partial(kab.AlignPlan.ctc, long_form=long_form)))
    return _check_plan_default(shim, lp, t_off, labels, l_off, V, blank, ta_check)


def _item(rng, L, V, blank, t_kind, repeat_p=0.2):
    """One lattice of L labels whose frame count is of the kind t_kind: "tight" (T = L + R), "tight1"
    (L + R + 1) or (residue, modulus) -- the smallest T >= 1.25 (L + R) with T = residue mod modulus."""
    pool = np.array([x for x in range(V) if x != blank])
    tg = rng.choice(pool, L)
    rep = rng.random(L) < repeat_p
    rep[0] = False
    tg[rep] = tg[np.flatnonzero(rep) - 1]
    need = L + int((tg[1:] == tg[:-1]).sum())
    if t_kind == "tight":
        T = need
    elif t_kind == "tight1":
        T = need + 1
    else:
        res, mod = t_kind
        T = int(1.25 * need)
        T += (res - T) % mod
    lp = np.log(rng.dirichlet(np.full(V, 0.5), T)).astype(np.float32)
    return lp, tg.astype(np.int32)


# (S, V, blank, T): S = 3297 the smallest wide lattice (32 warps); 3329 = 1 mod 104, S-1 alone in the top
# warp and S-2 below it; 3431 33 warps (the last CTA has 3 spare warps); 3743 36 warps.  V = 5 / 32: 16-frame
# emission stages, V = 129 / 256: 8-frame stages.  T mod 8 in {0, 1, 7}, T mod 128 in {0, 1}: the edges of
# the frame groups and of the backtrack blocks.
EDGES = [
    (3297, 32, 0, "tight"), (3297, 5, 4, "tight1"), (3297, 129, 128, (0, 128)), (3297, 256, 100, (7, 8)),
    (3329, 32, 16, (0, 128)), (3329, 256, 255, (1, 128)), (3329, 5, 2, "tight1"), (3329, 129, 0, (1, 8)),
    (3431, 129, 64, (7, 8)), (3431, 5, 0, (1, 8)), (3431, 32, 31, "tight"),
    (3743, 256, 0, (0, 8)), (3743, 32, 31, "tight"), (3743, 129, 7, (1, 128)),
]


@pytest.mark.parametrize("S,V,blank,t_kind", EDGES, ids=[f"S{s}-V{v}-b{b}-T{t if isinstance(t, str) else f'{t[0]}m{t[1]}'}"
                                                        for s, v, b, t in EDGES])
def test_geometry_edges(kab, S, V, blank, t_kind):
    rng = np.random.default_rng(S * 1000 + V + blank)
    lp, tg = _item(rng, (S - 1) // 2, V, blank, t_kind)
    info = _check_plan(kab, *_flat([(lp, tg)]), V, blank)
    assert info.n_class[3] == 1, list(info.n_class)
    T = lp.shape[0]
    nww = -(-S // 104)
    assert info.backptr_bytes == nww * -(-T // 8) * 256   # 2 bits per cell, not the generic kernel's byte


def test_repeats_ties_and_masks(kab):
    """Repeated labels (p = 0.4) with quantised log-probs (ties everywhere), and 5 % -inf masking."""
    rng = np.random.default_rng(31)
    V, blank = 32, 9
    items = _random_items(rng, 3, V, blank, (4500, 6000), quant=2, repeat_p=0.4, l_frac=(0.38, 0.45)) \
        + _random_items(rng, 2, V, blank, (4500, 6000), quant=1, repeat_p=0.4, l_frac=(0.38, 0.45)) \
        + _random_items(rng, 3, V, blank, (4500, 6000), neginf=0.05, l_frac=(0.38, 0.45))
    lp, t_off, labels, l_off = _flat(items)
    assert (2 * np.diff(l_off) + 1 > 3296).all()
    info = _check_plan(kab, lp, t_off, labels, l_off, V, blank)
    assert info.n_class[3] == len(items)


def test_both_end_states_neginf(kab):
    """Both end states -inf at the last frame: the restatement's path (torchaudio's is undefined there)."""
    rng = np.random.default_rng(32)
    V, blank = 32, 0
    items = _random_items(rng, 2, V, blank, (4000, 5000), l_frac=(0.4, 0.45))
    for lp, tg in items:
        lp[-1, blank] = -np.inf
        lp[-1, tg[-1]] = -np.inf
    lp, t_off, labels, l_off = _flat(items)
    rs, rp, rsc, rf, rst = forced_align_batch_np(lp, t_off, labels, l_off, blank)
    assert np.isneginf(rf).all()
    info = _check_plan(kab, lp, t_off, labels, l_off, V, blank, ta_check=False)
    assert info.n_class[3] == 2


def test_statuses(kab):
    """NaN and +inf: status 3; T < L + R: 1; a label equal to the blank: 2 -- among good wide lattices."""
    rng = np.random.default_rng(33)
    V, blank = 32, 5
    items = _random_items(rng, 6, V, blank, (4000, 4500), l_frac=(0.42, 0.45))
    items[1][0][1234, 7] = np.nan
    items[2][0][-1, 30] = np.inf
    lp3, tg3 = items[3]
    items[3] = (lp3[:len(tg3) - 1], tg3)             # T < L: no path
    items[4][1][100] = blank
    lp, t_off, labels, l_off = _flat(items)
    info = _check_plan(kab, lp, t_off, labels, l_off, V, blank)
    with kab.AlignPlan.ctc(t_off, labels, l_off, V, blank, long_form=True) as plan:
        status = plan.run_host(lp)[4]
    assert status.tolist() == [0, 3, 3, 1, 2, 0]
    assert info.n_class[3] == 4


def test_mixed_long_form_plan_equals_default(kab):
    """Warp, band and several wide lattices in one long-form plan: warp and band lattices keep their
    classes; the default plan of the same batch sends S > 3296 to the generic kernel, byte for byte equal."""
    rng = np.random.default_rng(34)
    V, blank = 32, 7
    items = _random_items(rng, 30, V, blank, (20, 300)) + _random_items(rng, 5, V, blank, (900, 4000), l_frac=(0.2, 0.35)) \
        + _random_items(rng, 4, V, blank, (9000, 12000), l_frac=(0.3, 0.4))
    lp, t_off, labels, l_off = _flat(items)
    S = 2 * np.diff(l_off) + 1
    info = _check_plan(kab, lp, t_off, labels, l_off, V, blank)
    assert info.n_class[0] == int((S <= 248).sum()) > 0
    assert info.n_class[1] == int(((S > 248) & (S <= 3296)).sum()) > 0
    assert info.n_class[3] == int((S > 3296).sum()) == 4 and info.n_class[2] == 0
    with kab.AlignPlan.ctc(t_off, labels, l_off, V, blank, long_form=True) as plan:
        out_long = plan.run_host(lp)
    with kab.AlignPlan.ctc(t_off, labels, l_off, V, blank) as plan:
        out_def = plan.run_host(lp)
        assert plan.info.n_class[2] == 4 and plan.info.n_class[3] == 0
        assert plan.info.n_class[:2] == info.n_class[:2]
    for a, b in zip(out_long, out_def):
        assert a.tobytes() == b.tobytes()


def test_fallbacks(kab):
    """V = 512: the wide kernel's emission stages do not fit shared memory -> generic.  A lattice whose
    CTAs exceed the resident capacity -> generic (plan info only)."""
    import torch
    rng = np.random.default_rng(35)
    items = _random_items(rng, 1, 512, 511, (4000, 4200), l_frac=(0.42, 0.45))
    info = _check_plan(kab, *_flat(items), 512, 511)
    assert info.n_class[2] == 1 and info.n_class[3] == 0
    # V = 129: 8-frame stages, one CTA per SM; 4 compute warps of 104 states per CTA plus the backtrack CTA
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    s_max = (sms - 1) * 4 * 104
    for L, cls in (((s_max - 1) // 2, 3), ((s_max + 1) // 2, 2)):
        tg = (np.arange(L) % 128 + 1).astype(np.int32)   # no repeats
        with kab.AlignPlan.ctc([0, L + 8], tg, [0, L], 129, 0, long_form=True) as plan:
            assert plan.info.n_class[cls] == 1, (L, list(plan.info.n_class))


@pytest.mark.parametrize("n,cls", [(8, 3), (64, 2)])
def test_selection(kab, n, cls):
    """The wide kernel runs its lattices one after another, the generic kernel side by side: a few lattices
    of S = 3401 go wide, 64 of them stay generic (the makespan estimate; plan info only)."""
    L, T = 1700, 3500
    tg = (np.arange(n * L) % 31 + 1).astype(np.int32)
    t_off, l_off = np.arange(n + 1) * T, np.arange(n + 1) * L
    with kab.AlignPlan.ctc(t_off, tg, l_off, 32, 0, long_form=True) as plan:
        assert plan.info.n_class[cls] == n, list(plan.info.n_class)


def test_chapter_length(kab):
    """T = 60 000, L = 16 000 (1.9e9 cells): long-form plan vs the default (generic) plan, the
    restatement and torchaudio CPU."""
    rng = np.random.default_rng(36)
    V, blank, T, L = 32, 0, 60000, 16000
    tg = rng.integers(1, V, L).astype(np.int32)
    lp = np.log(rng.dirichlet(np.full(V, 0.5), T)).astype(np.float32)
    t_off, l_off = np.array([0, T]), np.array([0, L])
    outs = []
    for long_form in (True, False):
        with kab.AlignPlan.ctc(t_off, tg, l_off, V, blank, long_form=long_form) as plan:
            assert plan.info.n_class[3 if long_form else 2] == 1
            outs.append(plan.run_host(lp))
    for a, b in zip(*outs):
        assert a.tobytes() == b.tobytes()
    path, labs, scores, final, status = outs[0]
    states, paths, sc, f = forced_align_np(lp, tg, blank)
    assert status[0] == 0
    np.testing.assert_array_equal(path, states)
    np.testing.assert_array_equal(labs, paths)
    assert scores.tobytes() == sc.tobytes() and final[0].tobytes() == f.tobytes()
    F = _torchaudio()
    if F is not None:
        import torch
        p, s = F.forced_align(torch.from_numpy(lp)[None], torch.from_numpy(tg)[None], blank=blank)
        np.testing.assert_array_equal(labs, p[0].numpy())
        assert scores.tobytes() == s[0].numpy().tobytes()


def test_run_torch_and_run_host_children(kab, monkeypatch):
    """run_torch of a long-form plan; run_host cutting the batch into child plans, which inherit the
    long form (the wide kernel runs, the generic one does not)."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    rng = np.random.default_rng(37)
    V, blank = 32, 3
    items = []
    for k in range(3):   # every child plan gets a wide lattice
        items += _random_items(rng, 1, V, blank, (4000, 5000), l_frac=(0.42, 0.45)) + _random_items(rng, 8, V, blank, (100, 1500))
    lp, t_off, labels, l_off = _flat(items)
    rs, rp, rsc, rf, rst = forced_align_batch_np(lp, t_off, labels, l_off, blank)
    assert (rst == 0).all()
    with kab.AlignPlan.ctc(t_off, labels, l_off, V, blank, long_form=True) as plan:
        assert plan.info.n_class[3] == 3 and plan.info.n_class[2] == 0
        outs = [tuple(x.cpu().numpy() for x in plan.run_torch(torch.from_numpy(lp).cuda()))]
    monkeypatch.setenv("KAB_HOST_SEGMENTS", "3")
    with kab.AlignPlan.ctc(t_off, labels, l_off, V, blank, long_form=True) as plan:
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            outs.append(plan.run_host(lp))
            torch.cuda.synchronize()
    names = {e.key for e in prof.key_averages()}
    assert any("kab_wide_ctc_kernel" in n for n in names), sorted(names)
    assert not any("kab_generic_ctc_kernel" in n for n in names), sorted(names)
    for path, labs, scores, final, status in outs:
        np.testing.assert_array_equal(status, rst)
        np.testing.assert_array_equal(path, rs)
        np.testing.assert_array_equal(labs, rp)
        assert scores.tobytes() == rsc.tobytes() and final.tobytes() == rf.tobytes()


def test_python_entry_points(kab):
    """forced_align(long_form=True) on CPU and CUDA tensors, forced_align_batch(long_form=True), and
    merge_tokens_batch of a long path (one span per target)."""
    import torch
    rng = np.random.default_rng(38)
    V, blank = 32, 0
    items = _random_items(rng, 3, V, blank, (4000, 6000), l_frac=(0.4, 0.45))
    lp0, tg0 = items[0]
    states, paths, sc, _ = forced_align_np(lp0, tg0, blank)
    T = lp0.shape[0]
    for dev in ("cpu", "cuda"):
        p, s = kab.forced_align(torch.from_numpy(lp0)[None].to(dev), torch.from_numpy(tg0)[None].to(dev),
                                blank=blank, long_form=True)
        assert p.device.type == dev and p.dtype == torch.int32 and p.shape == (1, T) and s.shape == (1, T)
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
        p, s = kab.forced_align_batch(torch.from_numpy(lpp).to(dev), torch.from_numpy(tgp).to(dev), tl, ll,
                                      blank=blank, long_form=True)
        assert p.device.type == dev and p.dtype == torch.int64 and p.shape == (B, T_max)
        for b, (x, tg) in enumerate(items):
            _, rp, rsc, _ = forced_align_np(x, tg, blank)
            n = x.shape[0]
            np.testing.assert_array_equal(p[b, :n].cpu().numpy(), rp)
            assert s[b, :n].cpu().numpy().tobytes() == rsc.tobytes()
            assert (p[b, n:] == blank).all() and (s[b, n:] == 0).all()
        spans = kab.merge_tokens_batch(p, s, tl, blank=blank)
        np.testing.assert_array_equal(spans.count.cpu().numpy(), ll.numpy())
        for b, (x, tg) in enumerate(items):
            np.testing.assert_array_equal(spans.token[b, :len(tg)].cpu().numpy(), tg)


@pytest.mark.parametrize("V", [39, 129])
def test_kokoro_wide_unaffected(kab, V):
    """A Kokoro-mode wide plan before and after a long-form CTC plan on the same device: both equal the C
    oracle.  V = 129 (8-frame emission stages) also checks the first group of frames of warp 0, whose staged
    backpointers once overlapped an mbarrier in shared memory."""
    from oracle import ctc_oracle
    rng = np.random.default_rng(39)
    items = _random_items(rng, 2, V, 0, (4000, 5000), l_frac=(0.45, 0.5))
    lp, t_off, labels, l_off = _flat(items)
    S = 2 * np.diff(l_off) + 1
    assert (S > 3296).all()
    beam = 2 * int(S.max()) + 2
    rp, rl, rs, rf, rst = ctc_oracle.ctc_best_path_batch(lp, t_off, labels, l_off, beam, 4, n_threads=2)
    outs = []
    for ctc_first in (False, True):
        if ctc_first:
            with kab.AlignPlan.ctc(t_off, labels, l_off, V, 0, long_form=True) as cplan:
                assert cplan.info.n_class[3] == 2
                cplan.run_host(lp)
        with kab.AlignPlan(t_off, labels, l_off, V, beam_size=beam) as plan:
            assert plan.info.n_class[3] == 2
            outs.append(plan.run_host(lp))
    for path, labs, scores, final, status in outs:
        np.testing.assert_array_equal(status, rst)
        np.testing.assert_array_equal(path, rp)
        np.testing.assert_array_equal(labs, rl)
        assert scores.tobytes() == rs.tobytes() and final.tobytes() == rf.tobytes()
