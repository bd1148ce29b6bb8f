"""``repeat_expand_2d`` (reference utils.py:482-496) - bit-identical to a literal restatement of the reference's walk, and to the
reference's own function's outputs (tests/golden/repeat_expand_2d.pt)."""
import pytest
import torch

from ns2vc_b200.frontend import repeat_expand_2d, repeat_expand_index

CASES = [(1, 1), (1, 7), (50, 94), (213, 400), (400, 213), (37, 37), (300, 1024), (7, 0), (1024, 1023), (3, 1000)]


def walk(content, target_len):
    """utils.py:482-496, statement by statement (test-side oracle)."""
    src_len = content.shape[-1]
    target = torch.zeros([content.shape[0], target_len], dtype=torch.float)
    temp = torch.arange(src_len + 1) * target_len / src_len
    current_pos = 0
    for i in range(target_len):
        if i < temp[current_pos + 1]:
            target[:, i] = content[:, current_pos]
        else:
            current_pos += 1
            target[:, i] = content[:, current_pos]
    return target


@pytest.mark.parametrize("src,tgt", CASES)
def test_matches_the_walk(src, tgt):
    c = torch.randn((5, src), generator=torch.Generator().manual_seed(src * 1000 + tgt))
    got = repeat_expand_2d(c, tgt)
    assert got.dtype == torch.float32 and got.shape == (5, tgt)
    assert torch.equal(got, walk(c, tgt))
    idx = repeat_expand_index(src, tgt)
    assert all(0 <= a <= b < src for a, b in zip(idx, idx[1:])) or tgt <= 1      # monotone, in range
    assert all(b - a <= 1 for a, b in zip(idx, idx[1:]))                          # at most one column per frame (the reference's lag)


def test_other_dtypes_and_errors():
    c = torch.arange(12, dtype=torch.float64).view(3, 4)
    assert torch.equal(repeat_expand_2d(c, 9), walk(c.float(), 9))
    with pytest.raises(ValueError):
        repeat_expand_2d(torch.zeros(4), 3)
    with pytest.raises(ValueError):
        repeat_expand_index(0, 3)


def test_matches_the_reference_function(gold):
    cases = gold("repeat_expand_2d.pt")                # the reference's own function on these inputs (oracle/make_golden_dropin.py)
    assert [(c["src"], c["tgt"]) for c in cases] == CASES
    for c in cases:
        x = torch.randn((4, c["src"]), generator=torch.Generator().manual_seed(c["seed"]))
        assert torch.equal(repeat_expand_2d(x, c["tgt"]), c["output"]), (c["src"], c["tgt"])
