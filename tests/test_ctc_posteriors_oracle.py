"""CPU checks of the posterior restatement (tests/ctc_posteriors_np.py) that the GPU tests hold the device to:
against a brute force over every CTC path, against torch's float64 ctc_loss and its gradient, and against its
own invariants -- on repeats, a blank that is not 0, -inf masks, banded windows that clip and lattices whose two
end states are both -inf."""
import numpy as np
import pytest

from tests.ctc_posteriors_np import ctc_posteriors_batch_np, ctc_posteriors_np, full_alpha_beta, path_values
from tests.forced_align_band_np import windows


def _lp(rng, T, V, neginf=0.0):
    lp = np.log(rng.dirichlet(np.full(V, 0.7), T))
    if neginf:
        lp[rng.random(lp.shape) < neginf] = -np.inf
    return lp


def _brute(lp, tg, blank, beam_size):
    """log Z and gamma [T, S] by enumerating every state path inside the windows."""
    T = lp.shape[0]
    S = 2 * len(tg) + 1
    ext = np.full(S, blank)
    ext[1::2] = tg
    lo, hi, _ = windows(T, S, beam_size)
    probs, occ = [], np.zeros((T, S))
    paths = []
    for v0 in (0, 1):
        if v0 < S:
            paths.append([v0])
    for t in range(1, T):
        nxt = []
        for p in paths:
            v = p[-1]
            for m in (0, 1, 2):
                w = v + m
                if w >= S or (m == 2 and (w % 2 == 0 or w < 3 or ext[w] == ext[w - 2])):
                    continue
                nxt.append(p + [w])
        paths = nxt
    for p in paths:
        if p[-1] < S - 2 or any(not lo[t] <= p[t] < hi[t] for t in range(T)):
            continue
        sc = sum(lp[t, ext[p[t]]] for t in range(T))
        probs.append(np.exp(sc))
        for t in range(T):
            occ[t, p[t]] += np.exp(sc)
    z = sum(probs)
    return (np.log(z) if z > 0 else -np.inf), (occ / z if z > 0 else occ)


CASES = [  # (T, targets, V, blank, beam_size)
    (5, [1, 2], 4, 0, None), (6, [1, 1], 3, 0, None), (8, [2, 2, 2], 3, 0, None), (7, [1, 2, 1], 4, 3, None),
    (4, [1], 2, 0, None), (8, [1, 2, 3], 4, 0, 3), (7, [1, 1, 2], 3, 0, 4), (8, [2, 1], 3, 0, 2), (6, [3, 3], 4, 0, 5),
    (8, [1, 2, 1], 4, 3, 3),
]


@pytest.mark.parametrize("T,tg,V,blank,W", CASES)
def test_brute_force_every_state(T, tg, V, blank, W):
    rng = np.random.default_rng(T * 100 + len(tg) * 10 + (W or 0))
    lp = _lp(rng, T, V)
    z_ref, g_ref = _brute(lp, np.array(tg), blank, W)
    S = 2 * len(tg) + 1
    for v in range(S):
        g, z = ctc_posteriors_np(lp, tg, np.full(T, v), blank, W)
        assert z == pytest.approx(z_ref, abs=1e-12)
        np.testing.assert_allclose(g, g_ref[:, v], atol=1e-12)
    rnd = rng.integers(-1, S + 1, T)   # an arbitrary path, some frames outside the lattice
    g, _ = ctc_posteriors_np(lp, tg, rnd, blank, W)
    want = np.array([g_ref[t, p] if 0 <= p < S else 0.0 for t, p in enumerate(rnd)])
    np.testing.assert_allclose(g, want, atol=1e-12)


def test_brute_force_with_masks_and_dead_ends():
    rng = np.random.default_rng(5)
    for _ in range(30):
        T, L = int(rng.integers(3, 8)), int(rng.integers(1, 4))
        tg = rng.integers(1, 4, L)
        lp = _lp(rng, T, 4, neginf=0.3)
        for W in (None, 2, 3):
            z_ref, g_ref = _brute(lp, tg, 0, W)
            for v in range(2 * L + 1):
                g, z = ctc_posteriors_np(lp, tg, np.full(T, v), 0, W)
                assert (z == z_ref) if z_ref == -np.inf else z == pytest.approx(z_ref, abs=1e-12)
                assert not np.isnan(g).any()
                np.testing.assert_allclose(g, g_ref[:, v], atol=1e-12)


@pytest.mark.parametrize("T,tg,blank", [(40, [1, 2, 2, 3, 1, 4, 1], 0), (30, [3, 3, 3, 1], 5), (25, [2, 1, 2], 0)])
def test_against_torch_ctc_loss_and_its_gradient(T, tg, blank):
    torch = pytest.importorskip("torch")
    V = 6
    rng = np.random.default_rng(T)
    lp_np = _lp(rng, T, V)
    lp = torch.tensor(lp_np[:, None, :], dtype=torch.float64, requires_grad=True)
    loss = torch.nn.functional.ctc_loss(lp, torch.tensor([tg]), torch.tensor([T]), torch.tensor([len(tg)]), blank=blank,
                                        reduction="sum")
    loss.backward()
    occ_ref = (lp.detach().exp() - lp.grad)[:, 0].numpy()
    al, be = full_alpha_beta(lp_np, tg, blank)
    z = np.logaddexp(al[-1, -1], al[-1, -2])
    assert z == pytest.approx(-loss.item(), abs=1e-10)
    g = np.exp(al + be - z)
    ext = np.full(2 * len(tg) + 1, blank)
    ext[1::2] = tg
    occ = np.zeros((T, V))
    for v, c in enumerate(ext):
        occ[:, c] += g[:, v]
    np.testing.assert_allclose(occ, occ_ref, atol=1e-12)
    _, z2 = ctc_posteriors_np(lp_np, tg, np.zeros(T, int), blank)
    assert z2 == pytest.approx(-loss.item(), abs=1e-10)


@pytest.mark.parametrize("W", [None, 5, 8, 11])
def test_invariants(W):
    rng = np.random.default_rng(7 + (W or 0))
    T, tg, blank = 50, np.array([1, 2, 2, 3, 1, 1, 4]), 4
    lp = _lp(rng, T, 5, neginf=0.05)
    al, be = full_alpha_beta(lp, tg, blank, W)
    z = np.logaddexp(al[-1, -1], al[-1, -2])
    assert np.isfinite(z)
    z_back = np.logaddexp(be[0, 0] + lp[0, blank], be[0, 1] + lp[0, tg[0]])   # beta_0 plus the start emissions
    assert z_back == pytest.approx(z, abs=1e-10)
    np.testing.assert_allclose(np.exp(al + be - z).sum(axis=1), 1.0, atol=1e-10)
    path = rng.integers(0, 2 * len(tg) + 1, T)
    fwd, bwd, z2 = path_values(lp, tg, path, blank, W)
    np.testing.assert_array_equal(fwd, al[np.arange(T), path])
    np.testing.assert_allclose(bwd, be[np.arange(T), path], atol=1e-10)
    assert z2 == z


def test_both_end_states_dead_and_the_batch_statuses():
    tg = np.array([1, 2])
    lp = np.log(np.full((6, 3), 1 / 3))
    lp[-1, :] = -np.inf   # no path can end
    g, z = ctc_posteriors_np(lp, tg, np.full(6, 3), 0)
    assert z == -np.inf and not g.any()
    lp2 = np.log(np.full((5, 3), 1 / 3))
    big = np.concatenate([lp, lp2])
    post, ll = ctc_posteriors_batch_np(big, [0, 6, 11], np.array([1, 2, 2, 1]), [0, 2, 4], np.full(11, 1), [0, 2])
    assert ll[0] == -np.inf and np.isnan(ll[1]) and not post.any()


def test_long_lattice_checks_quickly():
    rng = np.random.default_rng(3)
    T, L = 30000, 4000
    tg = rng.integers(1, 32, L)
    lp = np.log(rng.dirichlet(np.full(32, 0.5), T))
    fwd, bwd, z = path_values(lp, tg, np.linspace(0, 2 * L, T).astype(int), 0, 200)
    assert fwd.shape == (T,) and np.isfinite(z)
