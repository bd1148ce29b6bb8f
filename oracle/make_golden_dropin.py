"""Record what the UNMODIFIED reference's ``model.py`` and ``utils.py`` expect of the drop-in classes, so the tests check the
drop-in against the reference without the reference tree, and write tests/golden/{reference_model,repeat_expand_2d}.pt:

    NS2VC_REFERENCE=<reference tree> python oracle/make_golden_dropin.py

reference_model.pt: the shipped config.json, the ordered key -> shape list of the reference's own ``Pre_model(cfg)`` and of a
``NaturalSpeech2(cfg)`` checkpoint, the keyword arguments ``Diffusion_Encoder`` passes to ``UNet1DConditionModel`` (model.py:391-400),
the parameter counts, and the names model.py imports from the modules ``ns2vc_b200.install()`` aliases.
repeat_expand_2d.pt: input seeds and outputs of the reference's ``utils.repeat_expand_2d`` (utils.py:482-496) over the
(source, target) lengths of tests/test_frontend.py.  model.py imports matplotlib / vocos / accelerate / librosa / soundfile, which
are never touched here: they are stubbed.
"""
from __future__ import annotations

import ast
import json
import os
import sys
from unittest.mock import MagicMock

import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.environ.get("NS2VC_REFERENCE", "/root/reference")
sys.path.insert(0, REPO)
sys.path.insert(0, REF)
for name in ("matplotlib", "matplotlib.pyplot", "vocos", "accelerate", "librosa", "soundfile", "tensorboardX"):
    sys.modules.setdefault(name, MagicMock())

GOLD = os.path.join(REPO, "tests", "golden")
ALIASED = ("unet1d.unet_1d_condition", "sampler.dpm_solver", "sampler.uni_pc")     # the modules ns2vc_b200.install() replaces


def model_py_imports():
    """{module: [names]} of every ``from <aliased module> import ...`` in model.py (module level and inside functions)."""
    tree = ast.parse(open(os.path.join(REF, "model.py")).read())
    out = {m: [] for m in ALIASED}
    for node in ast.walk(tree):
        if isinstance(node, ast.ImportFrom) and node.module in out:
            out[node.module] += [a.name for a in node.names if a.name not in out[node.module]]
    return out


def reference_model():
    import model as ref_model
    cfg = json.load(open(os.path.join(REF, "config.json")))
    unet_kwargs = []

    class Recording(ref_model.UNet1DConditionModel):
        def __init__(self, **kw):
            unet_kwargs.append(dict(kw))
            super().__init__(**kw)

    real = ref_model.UNet1DConditionModel
    ref_model.UNet1DConditionModel = Recording
    try:
        ns2 = ref_model.NaturalSpeech2(cfg)
    finally:
        ref_model.UNet1DConditionModel = real
    assert len(unet_kwargs) == 1
    pre = ref_model.Pre_model(cfg)
    rec = {"config": cfg, "unet_kwargs": unet_kwargs[0], "imports": model_py_imports(),
           "pre_model_shapes": [(k, tuple(v.shape)) for k, v in pre.state_dict().items()],
           "checkpoint_shapes": [(k, tuple(v.shape)) for k, v in ns2.state_dict().items()],
           "pre_model_params": sum(p.numel() for p in ns2.pre_model.parameters()),
           "unet_params": sum(p.numel() for p in ns2.diff_model.unet.parameters())}
    torch.save(rec, os.path.join(GOLD, "reference_model.pt"))
    print(f"reference_model.pt: {len(rec['checkpoint_shapes'])} checkpoint keys, Pre_model {rec['pre_model_params']} params, "
          f"UNet {rec['unet_params']} params, imports {rec['imports']}")


def repeat_expand():
    import utils as ref_utils
    cases = []
    for src, tgt in [(1, 1), (1, 7), (50, 94), (213, 400), (400, 213), (37, 37), (300, 1024), (7, 0), (1024, 1023), (3, 1000)]:
        seed = src + 7 * tgt                                # input: torch.randn((4, src)) from this seed
        c = torch.randn((4, src), generator=torch.Generator().manual_seed(seed))
        cases.append({"src": src, "tgt": tgt, "seed": seed, "output": ref_utils.repeat_expand_2d(c, tgt)})
    torch.save(cases, os.path.join(GOLD, "repeat_expand_2d.pt"))
    print(f"repeat_expand_2d.pt: {len(cases)} cases")


if __name__ == "__main__":
    os.makedirs(GOLD, exist_ok=True)
    reference_model()
    repeat_expand()
