"""The long-form posterior limit of the C header and its Python mirror, and the ValueError above it (no GPU)."""
import os
import re

import numpy as np
import pytest

from kokoro_align_b200 import _lib, align

HEADER = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include", "kokoro_align_b200.h")


def _define(name):
    with open(HEADER) as f:
        m = re.search(rf"#define\s+{name}\s+(\d+)", f.read())
    assert m, name
    return int(m.group(1))


def test_long_posterior_limit_matches_the_header():
    assert _define("KAB_POSTERIOR_LONG_MAX_STATES") == _lib.POSTERIOR_LONG_MAX_STATES
    assert _define("KAB_POSTERIOR_MAX_STATES") == _lib.POSTERIOR_MAX_STATES
    assert _lib.POSTERIOR_LONG_MAX_STATES >= 108001   # a one-hour chapter (DESIGN.md 3.9b)


def test_long_form_limit_names_the_item():
    import torch
    L = (_lib.POSTERIOR_LONG_MAX_STATES + 1) // 2   # S = 2 L + 1: two states above the limit
    lp = torch.zeros(2, L + 4, 8)
    tg = (torch.arange(L) % 2 + 1).repeat(2, 1)
    with pytest.raises(ValueError, match=rf"item 1: long-form posteriors .*S = {2 * L + 1}"):
        align.forced_align_batch(lp, tg, target_lengths=torch.tensor([3, L]), long_form=True, posteriors=True)
    with pytest.raises(ValueError, match=rf"S = {2 * L + 1}"):
        align.forced_align(lp[:1], tg[:1], long_form=True, posteriors=True)
    # without long_form, the single-CTA limit and its beam_size advice are unchanged
    with pytest.raises(ValueError, match=r"item 1: .*S = 30001.*beam_size"):
        align._check_posteriors(False, None, np.array([11, 30001]), lambda b: f"item {b}: ")
    align._check_posteriors(False, None, np.array([11, 30001]), long_form=True)
