"""The warp kernel's checkpointed backtrack on the GPU, on the shapes that stress it (see
tests/test_warp_ckpt_emulation.py): every block shape and K class, S = 1, paths that fall three
states in every frame, tie stress, max_move < 4 and vocabularies other than 39.  Bit for bit
against the C oracle."""
import numpy as np
import pytest

from tools.emulate_warp_ckpt import C, falling_lattice

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def kab():
    import torch
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from kokoro_align_b200 import align
    return align


def _batch(V):
    from kokoro_align_b200 import synth
    lats = []
    for T in (1, C - 1, C, C + 1, 2 * C + 1, 861):
        for L in (0, 1, 20, 50, 80, 115, 123):
            if 2 * L <= 3 * T:
                lats.append(synth.make_lattice_exact(T, L, V, seed=11 * T + L, planted=True))
    for T in (2, 8, 16, 24, 80):
        lats.append(falling_lattice(T, V=V, seed=T))
    for n, (T, L) in enumerate([(30, 40), (100, 61), (200, 120), (300, 123), (861, 123), (500, 70)]):
        lats.append(synth.make_lattice_exact(T, L, V, seed=900 + n, levels=3, repeat_labels=True))
    T = np.array([lp.shape[0] for lp, _ in lats])
    L = np.array([len(lab) for _, lab in lats])
    t_off = np.concatenate([[0], np.cumsum(T)]).astype(np.int64)
    l_off = np.concatenate([[0], np.cumsum(L)]).astype(np.int64)
    lp = np.concatenate([lp for lp, _ in lats]).astype(np.float32)
    labels = np.concatenate([np.asarray(lab, np.int32) for _, lab in lats]).astype(np.int32)
    return lp, t_off, labels, l_off


@pytest.mark.parametrize("V", [39, 17, 100])
@pytest.mark.parametrize("max_move", [4, 3, 2])
def test_adversarial_shapes_bit_exact(kab, V, max_move):
    from oracle import ctc_oracle
    lp, t_off, labels, l_off = _batch(V)
    B = len(t_off) - 1
    rp, rl, rs, rf, rst = ctc_oracle.ctc_best_path_batch(lp, t_off, labels, l_off, 1000, max_move, n_threads=8)
    with kab.AlignPlan(t_off, labels, l_off, V, 1000, max_move) as plan:
        path, labs, scores, final, status = plan.run_host(lp)
        assert plan.info.n_class[0] == B  # every lattice on the warp kernel
    np.testing.assert_array_equal(status, rst)
    assert (rst == 0).sum() >= B - 2
    for b in range(B):
        if rst[b] != 0:
            continue
        a, e = int(t_off[b]), int(t_off[b + 1])
        np.testing.assert_array_equal(path[a:e], rp[a:e], err_msg=f"lattice {b}")
        np.testing.assert_array_equal(labs[a:e], rl[a:e], err_msg=f"lattice {b}")
        assert scores[a:e].tobytes() == rs[a:e].tobytes(), f"lattice {b}"
        assert final[b].tobytes() == rf[b].tobytes(), f"lattice {b}"
