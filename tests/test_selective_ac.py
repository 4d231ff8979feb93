"""Selective-recompute placement must reproduce the reference patterns bit-for-bit
(reference tests/test_selective_ac.py:12-64, rule at fms_fsdp/policies/ac_handler.py:43-58)."""
import pytest

from fms_fsdp_b200.models.llama import LLaMABlock
from fms_fsdp_b200.policies import apply_fsdp_checkpointing, is_checkpointed, selection_mask
from fms_fsdp_b200.policies.ac_handler import parse_fraction

T, F = True, False
CASES = [
    (0, [F] * 15), (1 / 100, [F] * 15), (-1, [F] * 15),
    (1 / 5, [F, F, T, F, F] * 3), (1 / 3, [F, T, F] * 5), (1 / 2, [T, F] * 7 + [T]),
    (3 / 5, [T, F, T, F, T] * 3), (2 / 3, [T, F, T] * 5), (1, [T] * 15), (5 / 3, [T] * 15),
    ("1/3", [F, T, F] * 5), ("1/2", [T, F] * 7 + [T]),
]


@pytest.mark.parametrize("p,expected", CASES)
def test_patterns(narrow_model_factory, p, expected):
    model = narrow_model_factory(15)
    apply_fsdp_checkpointing(model, LLaMABlock, p)
    assert [is_checkpointed(b) for b in model.layers] == expected
    assert selection_mask(15, p) == expected


def test_fraction_parser_is_not_eval():
    assert parse_fraction("1/4") == 0.25
    assert parse_fraction(0.5) == 0.5
    with pytest.raises(Exception):
        parse_fraction("__import__('os').system('true')")


def test_non_reentrant_wrapper_marks_a_single_block():
    import torch.nn as nn
    from fms_fsdp_b200.policies.ac_handler import is_checkpointed, non_reentrant_wrapper
    blk = nn.Linear(2, 2)
    assert not is_checkpointed(blk)
    assert non_reentrant_wrapper(blk) is blk and is_checkpointed(blk)


def test_selection_equals_what_the_reference_install_wraps():
    """Which blocks the original ``apply_fsdp_checkpointing`` (torch ``checkpoint_wrapper``) wrapped on stacks of plain
    blocks, for the depths of the model zoo and a sweep of fractions (tests/golden/reference/ac_selection.json, "1" =
    wrapped), equals ``selection_mask``."""
    import json
    import os
    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference", "ac_selection.json")) as f:
        theirs = json.load(f)
    fracs = ["1/7", "1/4", "1/3", "2/5", "1/2", "3/5", "2/3", "3/4", "9/10", "1"]
    depths = [10, 24, 32, 40, 48, 80]
    assert len(theirs) == len(fracs) * len(depths)
    for n in depths:
        for p in fracs:
            assert selection_mask(n, p) == [c == "1" for c in theirs[f"{n}:{p}"]], (n, p)
