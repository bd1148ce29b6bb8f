"""Oracle of the condition encoders (`Pre_model`, SURVEY.md §8(f) rank 1 — the step before the denoiser) against
fixtures produced by the unmodified reference (oracle/make_golden_pre.py).  CPU only; groundwork for the next row."""
import os

import pytest
import torch

from oracle import pre_model_oracle as po

GOLD = os.path.join(os.path.dirname(__file__), "golden")


def _inputs(B, T, S, c_in, seed):
    g = torch.Generator().manual_seed(seed)
    c = torch.randn((B, c_in, T), generator=g)
    refer = torch.randn((B, 100, S), generator=g)
    lengths = torch.tensor([max(1, T - 13 * i) for i in range(B)], dtype=torch.int64)
    refer_lengths = torch.tensor([max(1, S - 7 * i) for i in range(B)], dtype=torch.int64)
    return c, refer, lengths, refer_lengths


@pytest.mark.parametrize("name", ["tiny", "full"])
def test_pre_model_oracle_matches_reference_fixture(name):
    """In float64 on both sides (the reference's run is stored rounded to float32, <= 2.4e-7 here): in float32 the outputs
    move by a few 1e-6 with the host's summation order (thread count, vector ISA), which is not what this test checks."""
    g = torch.load(os.path.join(GOLD, f"pre_model_{name}.pt"))
    sd = po.synth_state_dict(g["shapes"], seed=0)
    assert sum(v.numel() for v in sd.values()) == g["n_params"]
    if name == "full":
        assert g["n_params"] == 34923404                      # demo.ipynb:447 "pre params"
    cfg = g["cfg"]
    c, refer, lengths, refer_lengths = _inputs(g["B"], g["T"], g["S"], cfg["phoneme_encoder"]["in_channels"], g["input_seed"])
    taps = {}
    with torch.no_grad():
        content, prompt = po.pre_model_infer({k: v.double() for k, v in sd.items()}, c.double(), refer.double(), lengths,
                                             refer_lengths, cfg["phoneme_encoder"]["n_layers"], cfg["prompt_encoder"]["n_layers"], taps)
    assert g["taps_f64"] or name == "full"
    for k, v in g["taps_f64"].items():                        # per-layer activations (tiny fixture only)
        assert torch.allclose(taps[k], v.double(), rtol=0, atol=2e-6), k
    assert content.shape == g["content_f64"].shape and prompt.shape == g["prompt_f64"].shape
    assert torch.allclose(content, g["content_f64"].double(), rtol=0, atol=2e-6)
    assert torch.allclose(prompt, g["prompt_f64"].double(), rtol=0, atol=2e-6)
    # padded frames are exactly zero (model.py:146-148, 188-190)
    for b in range(g["B"]):
        assert (content[lengths[b]:, b] == 0).all() and (prompt[refer_lengths[b]:, b] == 0).all()
