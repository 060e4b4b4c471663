"""The warp kernel's checkpointed backtrack (tools/emulate_warp_ckpt.py, DESIGN.md 3.1) against the
C oracle, bit for bit: the goldens' warp-shaped cases, tie stress, paths that fall three states in
every frame, every block shape and every K class.  CPU only."""
import numpy as np
import pytest

from kokoro_align_b200 import synth
from tests.golden_util import case_inputs, golden_names
from tools.emulate_warp_ckpt import C, check, falling_lattice, k_class


def _warp_shaped(case, arrays):
    if case["outcome"] != "ok" or case["max_move"] > 4:
        return False
    lp, labels = case_inputs(case, arrays)
    T, S, W = lp.shape[0], 2 * len(labels) + 1, case["beam_size"]
    full = W >= S and (S * (T - 1)) // T <= W // 2
    return full and S <= 248 and (len(labels) == 0 or labels.min() >= 1)


def test_golden_warp_cases(golden):
    index, arrays = golden
    cases = [c for c in index if _warp_shaped(c, arrays)]
    assert len(cases) >= 5
    for case in cases:
        lp, labels = case_inputs(case, arrays)
        check(lp, labels, case["max_move"])


# T: one frame, partial / exact / one-past blocks, the longest config-2 segment; L: S = 1 and the K
# classes 2, 4, 6, 8, wherever a path can reach the end (S <= 3T + 1)
SHAPES = [(T, L) for T in (1, C - 1, C, C + 1, 2 * C + 1, 861) for L in (0, 1, 20, 50, 80, 115) if 2 * L <= 3 * T]


@pytest.mark.parametrize("T,L", SHAPES)
def test_block_shapes_and_classes(T, L):
    lp, labels = synth.make_lattice_exact(T, L, 39, seed=7 * T + L, planted=True)
    for max_move in (4, 3, 1):
        check(lp, labels, max_move, junk_seed=T + L)


def test_every_k_class_is_covered():
    assert sorted({k_class(2 * L + 1) for L in (0, 20, 50, 80, 115)}) == [2, 4, 6, 8]


@pytest.mark.parametrize("T", [2, 8, 16, 24, 80])
def test_paths_falling_three_states_every_frame(T):
    lp, labels = falling_lattice(T, seed=T)
    check(lp, labels)


def test_tie_stress_batch():
    T, L = synth.segment_lengths(40, seed=2100, t_min=1, t_max=200)
    for n, (t, l) in enumerate(zip(T, L)):
        if 2 * l + 1 > 248:
            continue
        lp, labels = synth.make_lattice(int(t), int(l), 39, 2101 + n)
        lp = (np.round(lp * 2) / 2).astype(np.float32)
        check(lp, labels, junk_seed=n)


def test_tie_stress_exact_levels():
    for n, (T, L) in enumerate([(30, 40), (100, 61), (200, 120), (300, 123)]):
        lp, labels = synth.make_lattice_exact(T, L, 39, seed=500 + n, levels=3, repeat_labels=True)
        check(lp, labels, junk_seed=n)
