"""Drop-in check against what the reference's own model.py builds (tests/golden/reference_model.pt, recorded from the unmodified
reference by oracle/make_golden_dropin.py).  After `ns2vc_b200.install()` / `install_pre_model()` the names model.py imports
resolve to the B200 classes, and those classes, built with model.py's arguments, expose the reference's state_dict contract
and strict-load a reference-shaped checkpoint."""
import importlib
import sys
import types

import torch


def test_reference_model_py_builds_on_our_unet(gold):
    import ns2vc_b200
    from ns2vc_b200 import dpm_solver, uni_pc, unet as unet_mod
    from ns2vc_b200.arch import ns2vc_denoiser_config, param_shapes
    from ns2vc_b200.pre_model import Pre_model
    from ns2vc_b200.unet import UNet1DConditionModel
    g = gold("reference_model.pt")
    cfg = g["config"]

    # every name model.py imports from the aliased modules resolves to ours
    saved = {k: v for k, v in sys.modules.items() if k.split(".")[0] in ("unet1d", "sampler")}
    try:
        ns2vc_b200.install()
        ours = {"unet1d.unet_1d_condition": unet_mod, "sampler.dpm_solver": dpm_solver, "sampler.uni_pc": uni_pc}
        assert set(g["imports"]) == set(ours)
        for mod, names in g["imports"].items():
            assert names and importlib.import_module(mod) is ours[mod]
            for name in names:
                assert getattr(importlib.import_module(mod), name) is getattr(ours[mod], name), (mod, name)
    finally:
        for k in list(sys.modules):
            if k.split(".")[0] in ("unet1d", "sampler"):
                del sys.modules[k]
        sys.modules.update(saved)

    # model.py:451 looks Pre_model up by its global name
    model_py = types.ModuleType("model")
    model_py.Pre_model = object
    ns2vc_b200.install_pre_model(model_py)
    assert model_py.Pre_model is Pre_model
    pre = model_py.Pre_model(cfg)
    assert [(k, tuple(v.shape)) for k, v in pre.state_dict().items()] == g["pre_model_shapes"]   # keys, order, shapes
    assert sum(p.numel() for p in pre.parameters()) == g["pre_model_params"] == 34923404

    # Diffusion_Encoder's constructor call (model.py:391-400)
    unet = UNet1DConditionModel(**g["unet_kwargs"])
    assert sum(p.numel() for p in unet.parameters()) == g["unet_params"] == 66076900
    assert unet.latent_channels == cfg["diffusion_encoder"]["in_channels"]

    # a checkpoint written by the reference: its diff_model.unet. and pre_model. entries are exactly our state_dicts
    ckpt = g["checkpoint_shapes"]
    unet_keys = [(k[len("diff_model.unet."):], s) for k, s in ckpt if k.startswith("diff_model.unet.")]
    assert unet_keys == [(k, tuple(v.shape)) for k, v in unet.state_dict().items()]
    assert [k for k, _ in unet_keys] == list(param_shapes(ns2vc_denoiser_config()).keys())
    assert [(k[len("pre_model."):], s) for k, s in ckpt if k.startswith("pre_model.")] == g["pre_model_shapes"]
    assert not [k for k, _ in ckpt if k.startswith("diff_model.") and not k.startswith("diff_model.unet.")]
    unet.load_state_dict({k: torch.zeros(s) for k, s in unet_keys}, strict=True)
    pre.load_state_dict({k: torch.zeros(s) for k, s in g["pre_model_shapes"]}, strict=True)
