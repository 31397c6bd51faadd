"""Checkpoint ingest (SURVEY.md §8(f) rank 3): reference-prefixed `.safetensors` / `.ckpt` files through the strict=False load that
`DiffusionEngine.init_from_ckpt` performs (models/diffusion.py:191-219) — no key of the replaced modules may be skipped."""
import json
import os
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from gcd_b200 import checkpoint, spec, synthetic  # noqa: E402
from gcd_b200.unet import VideoUNet  # noqa: E402
from gcd_b200.vae import Encoder, VideoDecoder  # noqa: E402


def _root():
    return checkpoint.HotPathRoot(VideoUNet(**spec.unet_ctor_kwargs(spec.UNET_TINY)),
                                  VideoDecoder(**spec.decoder_ctor_kwargs(spec.VAE_TINY)),
                                  Encoder(**spec.encoder_ctor_kwargs(spec.VAE_ENCODER_TINY)))


def _engine_state():
    """A DiffusionEngine-style state dict: reference prefixes for the hot-path tensors + keys of components this package does
    not replace (conditioner / EMA bookkeeping), as they appear in an SVD / GCD checkpoint."""
    sd = {}
    for k, v in synthetic.seeded_state(spec.unet_param_shapes(spec.UNET_TINY), seed=1).items():
        sd["model.diffusion_model." + k] = v
    for k, v in synthetic.seeded_state(spec.decoder_param_shapes(spec.VAE_TINY), seed=2).items():
        sd["first_stage_model.decoder." + k] = v
    for k, v in synthetic.seeded_state(spec.encoder_param_shapes(spec.VAE_ENCODER_TINY), seed=3).items():
        sd["first_stage_model.encoder." + k] = v
    sd["first_stage_model.quant_conv.weight"] = torch.randn(8, 8, 1, 1)
    sd["first_stage_model.quant_conv.bias"] = torch.randn(8)
    extra = {"conditioner.embedders.0.open_clip.model.positional_embedding": torch.randn(4, 4),
             "model_ema.decay": torch.tensor(0.9999), "model_ema.num_updates": torch.tensor(7)}
    sd.update(extra)
    return sd, sorted(extra)


@pytest.mark.parametrize("fmt", ["safetensors", "ckpt"])
def test_prefixed_checkpoint_round_trip_skips_nothing(tmp_path, fmt):
    sd, extra = _engine_state()
    path = str(tmp_path / f"engine.{fmt}")
    if fmt == "safetensors":
        from safetensors.torch import save_file
        save_file({k: v.contiguous() for k, v in sd.items()}, path)
    else:
        torch.save({"state_dict": sd, "global_step": 1}, path)
    root = _root()
    missing, unexpected = root.init_from_ckpt(path)
    assert missing == [], missing[:5]                       # every parameter of the replaced modules was found in the file
    assert sorted(unexpected) == extra                      # and nothing but the foreign components was left over
    got = root.state_dict()
    for k, v in sd.items():
        if k not in extra:
            assert torch.equal(got[k], v), k
    # a renamed tensor is REPORTED (strict=False would otherwise skip it silently: the failure mode spec.py guards against)
    bad = dict(sd)
    bad["model.diffusion_model.input_blocks.0.0.weight_renamed"] = bad.pop("model.diffusion_model.input_blocks.0.0.weight")
    p2 = str(tmp_path / "bad.ckpt")
    torch.save({"state_dict": bad}, p2)
    missing, unexpected = _root().init_from_ckpt(p2)
    assert missing == ["model.diffusion_model.input_blocks.0.0.weight"]
    assert "model.diffusion_model.input_blocks.0.0.weight_renamed" in unexpected


def test_ema_shadows_replace_the_unet_weights(tmp_path):
    """use_ema: `model_ema.<name without dots>` shadows (LitEma, modules/ema.py) overwrite the UNet parameters; checked against
    the shadow names the reference's own LitEma gave `HotPathRoot.model` (tests/golden/host_api.json)."""
    sd, _ = _engine_state()
    ema = {k: v * 0.5 + 0.25 for k, v in synthetic.seeded_state(spec.unet_param_shapes(spec.UNET_TINY), seed=1).items()}
    for k, v in ema.items():
        sd["model_ema." + checkpoint.ema_key("diffusion_model." + k)] = v
    path = str(tmp_path / "ema.ckpt")
    torch.save({"state_dict": sd}, path)
    root = _root()
    missing, unexpected = root.init_from_ckpt(path, use_ema=True)
    assert missing == [] and not any(k.startswith("model_ema.") for k in unexpected)
    got = root.model.diffusion_model.state_dict()
    assert all(torch.equal(got[k], v) for k, v in ema.items())
    with pytest.raises(KeyError):
        p2 = str(tmp_path / "noema.ckpt")
        torch.save({"state_dict": {k: v for k, v in sd.items() if not k.startswith("model_ema.")}}, p2)
        _root().init_from_ckpt(p2, use_ema=True)
    with open(os.path.join(ROOT, "tests", "golden", "host_api.json")) as f:
        shadows = json.load(f)["litema_shadows_of_model"]      # reference naming of the shadows of `model`
    assert all(checkpoint.ema_key("diffusion_model." + k) == shadows["diffusion_model." + k] for k in ema)
