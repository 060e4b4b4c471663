"""CTC forced alignment on the B200 (kab_plan_create_ctc and the Python entry points), bit-exact
against torchaudio's CPU forced_align and the goldens: paths, labels, scores and final score."""
import numpy as np
import pytest

from oracle.forced_align_np import forced_align_batch_np, forced_align_np
from tests.test_forced_align_oracle import CASES

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
        F.forced_align(torch.zeros(1, 2, 3), torch.ones(1, 1, dtype=torch.int32))
        return F
    except Exception:  # noqa: BLE001
        return None


def _flat(items):
    """[(lp [T, V], targets [L])] -> flat batch (lp, t_off, labels, l_off)."""
    t_off = np.concatenate([[0], np.cumsum([x[0].shape[0] for x in items])]).astype(np.int64)
    l_off = np.concatenate([[0], np.cumsum([len(x[1]) for x in items])]).astype(np.int64)
    lp = np.ascontiguousarray(np.concatenate([x[0] for x in items]), np.float32)
    labels = np.concatenate([np.asarray(x[1], np.int32) for x in items]).astype(np.int32)
    return lp, t_off, labels, l_off


def _check_plan(kab, lp, t_off, labels, l_off, V, blank, ta_check=True):
    """run_host of a CTC plan vs the restatement (and torchaudio CPU where its result is defined)."""
    rs, rp, rsc, rf, rst = forced_align_batch_np(lp, t_off, labels, l_off, blank)
    with kab.AlignPlan.ctc(t_off, labels, l_off, V, blank) as plan:
        path, labs, scores, final, status = plan.run_host(lp)
        info = plan.info
    np.testing.assert_array_equal(status, rst)
    F = _torchaudio() if ta_check else None
    for b in range(len(t_off) - 1):
        if rst[b] != 0:
            continue
        a, e = int(t_off[b]), int(t_off[b + 1])
        np.testing.assert_array_equal(path[a:e], rs[a:e], err_msg=f"lattice {b}")
        np.testing.assert_array_equal(labs[a:e], rp[a:e], err_msg=f"lattice {b}")
        assert scores[a:e].tobytes() == rsc[a:e].tobytes(), f"lattice {b}"
        assert final[b].tobytes() == rf[b].tobytes(), f"lattice {b}"
        if F is not None and np.isfinite(rf[b]):
            import torch
            tg = torch.from_numpy(labels[int(l_off[b]):int(l_off[b + 1])])[None]
            p, s = F.forced_align(torch.from_numpy(lp[a:e])[None], tg, blank=blank)
            np.testing.assert_array_equal(labs[a:e], p[0].numpy(), err_msg=f"lattice {b} vs torchaudio")
            assert scores[a:e].tobytes() == s[0].numpy().tobytes(), f"lattice {b} vs torchaudio"
    return info


@pytest.mark.parametrize("name,case", CASES, ids=[n for n, _ in CASES])
def test_golden(kab, name, case):
    import torch
    lp, tg, blank = case["lp"], case["targets"], int(case["blank"])
    T, V = lp.shape
    with kab.AlignPlan.ctc([0, T], tg, [0, len(tg)], V, blank) as plan:
        path, labs, scores, final, status = plan.run_host(lp)
        S = 2 * len(tg) + 1
        expect = 0 if V <= 512 and S <= 248 else (1 if V <= 512 and S <= 3296 else 2)
        assert plan.info.n_class[expect] == 1, (name, list(plan.info.n_class))
    assert status[0] == 0
    np.testing.assert_array_equal(path, case["states"])
    np.testing.assert_array_equal(labs, case["paths"])
    assert scores.tobytes() == case["scores"].tobytes()
    assert final[0].tobytes() == case["final"].tobytes()
    # the torchaudio drop-in, CPU and CUDA tensors
    for dev in ("cpu", "cuda"):
        p, s = kab.forced_align(torch.from_numpy(lp)[None].to(dev), torch.from_numpy(tg)[None].to(dev), blank=blank)
        assert p.device.type == dev and p.dtype == torch.int32 and p.shape == (1, T) and s.shape == (1, T)
        np.testing.assert_array_equal(p[0].cpu().numpy(), case["paths"])
        assert s[0].cpu().numpy().tobytes() == case["scores"].tobytes()


def _random_items(rng, n, V, blank, t_range, quant=None, repeat_p=0.2, neginf=0.0, l_frac=(0.1, 0.45)):
    items = []
    pool = np.array([x for x in range(V) if x != blank])
    for _ in range(n):
        T = int(rng.integers(*t_range))
        L = max(1, int(T * rng.uniform(*l_frac)))
        tg = rng.choice(pool, L)
        rep = rng.random(L) < repeat_p
        rep[0] = False
        tg[rep] = tg[np.flatnonzero(rep) - 1]
        T = max(T, L + int((tg[1:] == tg[:-1]).sum()))
        lp = np.log(rng.dirichlet(np.full(V, 0.5), T)).astype(np.float32)
        if quant:
            lp = (np.round(lp * quant) / quant).astype(np.float32)
        if neginf:
            lp[rng.random(lp.shape) < neginf] = -np.inf
        items.append((lp, tg.astype(np.int32)))
    return items


def test_mixed_batch_all_classes(kab):
    """Warp (S <= 248), band (S <= 3296) and generic (S > 3296) lattices in one plan."""
    rng = np.random.default_rng(11)
    V, blank = 32, 7
    items = _random_items(rng, 40, V, blank, (20, 300)) + _random_items(rng, 6, V, blank, (900, 4000), l_frac=(0.2, 0.35)) \
        + _random_items(rng, 2, V, blank, (9000, 11000), l_frac=(0.3, 0.4))
    lp, t_off, labels, l_off = _flat(items)
    S = 2 * np.diff(l_off) + 1
    info = _check_plan(kab, lp, t_off, labels, l_off, V, blank)
    assert info.n_class[0] == int((S <= 248).sum()) > 0
    assert info.n_class[1] == int(((S > 248) & (S <= 3296)).sum()) > 0
    assert info.n_class[2] == int((S > 3296).sum()) > 0
    assert info.n_class[3] == 0 and info.cells_eval == int((np.diff(t_off) * S).sum())


@pytest.mark.parametrize("quant,blank", [(2, 0), (4, 31), (1, 15)])
def test_tie_stress(kab, quant, blank):
    rng = np.random.default_rng(100 + quant)
    items = _random_items(rng, 60, 32, blank, (10, 200), quant=quant, repeat_p=0.4) \
        + _random_items(rng, 4, 32, blank, (700, 1500), quant=quant, repeat_p=0.4, neginf=0.05)
    _check_plan(kab, *_flat(items), 32, blank)


def test_neginf_masks_and_wide_vocab(kab):
    rng = np.random.default_rng(5)
    items = _random_items(rng, 30, 512, 511, (20, 200), neginf=0.1) + _random_items(rng, 3, 512, 511, (600, 900), neginf=0.02)
    _check_plan(kab, *_flat(items), 512, 511)
    _check_plan(kab, *_flat(_random_items(rng, 20, 600, 3, (20, 120))), 600, 3)   # V > 512: generic kernel


def test_band_lattice_1e8_cells(kab):
    """One band-class lattice of 1e8 cells (S = 3295, T = 30 350)."""
    rng = np.random.default_rng(8)
    V, blank, L, T = 32, 0, 1647, 30350
    tg = rng.integers(1, V, L).astype(np.int32)
    lp = np.log(rng.dirichlet(np.full(V, 0.5), T)).astype(np.float32)
    t_off, l_off = np.array([0, T]), np.array([0, L])
    with kab.AlignPlan.ctc(t_off, tg, l_off, V, blank) as plan:
        assert plan.info.n_class[1] == 1 and plan.info.cells_eval >= 10 ** 8
        path, labs, scores, final, status = plan.run_host(lp)
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


def test_run_torch_and_batch_api(kab):
    import torch
    rng = np.random.default_rng(21)
    V, blank = 32, 3
    items = _random_items(rng, 25, V, blank, (30, 600), quant=2)
    lp, t_off, labels, l_off = _flat(items)
    rs, rp, rsc, rf, rst = forced_align_batch_np(lp, t_off, labels, l_off, blank)
    with kab.AlignPlan.ctc(t_off, labels, l_off, V, blank) as plan:
        path, labs, scores, final, status = (x.cpu().numpy() for x in plan.run_torch(torch.from_numpy(lp).cuda()))
        with pytest.raises(kab.KabError):   # align()'s segment records are Kokoro-specific
            plan.run_host_segments(lp, [np.array([int(t_off[b + 1] - t_off[b])]) for b in range(len(items))])
    assert (status == 0).all() and (rst == 0).all()
    np.testing.assert_array_equal(path, rs)
    np.testing.assert_array_equal(labs, rp)
    assert scores.tobytes() == rsc.tobytes() and final.tobytes() == rf.tobytes()
    # forced_align_batch: padded in, padded out, CPU and CUDA
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
        p, s = p.cpu().numpy(), s.cpu().numpy()
        for b in range(B):
            a, e = int(t_off[b]), int(t_off[b + 1])
            np.testing.assert_array_equal(p[b, :e - a], rp[a:e])
            assert s[b, :e - a].tobytes() == rsc[a:e].tobytes()
            assert (p[b, e - a:] == blank).all() and (s[b, e - a:] == 0).all()


def test_statuses_and_errors(kab):
    import torch
    rng = np.random.default_rng(3)
    V = 6
    lp = np.log(rng.dirichlet(np.ones(V), 40)).astype(np.float32)
    lp[25, 4] = np.nan
    lp[33, 1] = np.inf
    lp[5, 2] = -np.inf   # accepted
    t_off = np.array([0, 10, 13, 20, 30, 36, 40])
    labels = np.array([1, 2, 3, 2, 2, 2, 0, 4, 1, 5, 5, 1, 2, 3], np.int32)
    l_off = np.array([0, 3, 6, 7, 9, 11, 14])
    # 0 ok (-inf inside), 1 [2,2,2] in 3 frames: dead, 2 label == blank (0): bad label,
    # 3 NaN, 4 +inf, 5 label 5 ok with blank 0
    with kab.AlignPlan.ctc(t_off, labels, l_off, V, 0) as plan:
        _, _, _, _, status = plan.run_host(lp)
    assert status.tolist() == [0, 1, 2, 3, 3, 0]
    with pytest.raises(kab.KabError):
        kab.AlignPlan.ctc(t_off, labels, l_off, V, V)   # blank outside [0, V)
    x = torch.from_numpy(lp[20:30])[None]
    for dev in ("cpu", "cuda"):
        with pytest.raises(ValueError):
            kab.forced_align(x.to(dev), torch.tensor([[1, 5]], device=dev))
    with pytest.raises(ValueError, match="item 1"):
        kab.forced_align_batch(torch.from_numpy(lp[10:30].reshape(2, 10, V)).cuda(),
                               torch.tensor([[1, 2], [4, 1]], device="cuda"))


def test_kokoro_mode_unaffected(kab):
    """A Kokoro-mode plan of the same batch, before and after a CTC plan ran on it: same outputs."""
    from oracle import ctc_oracle
    rng = np.random.default_rng(4)
    items = _random_items(rng, 30, 39, 0, (50, 400)) + _random_items(rng, 2, 39, 0, (2000, 3000))
    lp, t_off, labels, l_off = _flat(items)
    rp, rl, rs, rf, rst = ctc_oracle.ctc_best_path_batch(lp, t_off, labels, l_off, 1000, 4, n_threads=4)
    outs = []
    for ctc_first in (False, True):
        if ctc_first:
            with kab.AlignPlan.ctc(t_off, labels, l_off, 39, 0) as cplan:
                cplan.run_host(lp)
        with kab.AlignPlan(t_off, labels, l_off, 39) as plan:
            outs.append(plan.run_host(lp))
    for path, labs, scores, final, status in outs:
        np.testing.assert_array_equal(status, rst)
        np.testing.assert_array_equal(path, rp)
        np.testing.assert_array_equal(labs, rl)
        assert scores.tobytes() == rs.tobytes() and final.tobytes() == rf.tobytes()
