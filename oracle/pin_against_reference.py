"""Pins the oracle to the reference and writes tests/golden/ (run in the BUILD CONTAINER only; needs /root/reference).

    python -m oracle.pin_against_reference [--full]

For each case the REFERENCE's own modules (imported through oracle/ref_shim.py) are run on CPU fp32 with seeded
weights/inputs (oracle/weights.py); the golden tensors stored are the reference outputs, and the oracle restatement is
asserted to agree with them (max-abs relative to output scale < 2e-5). Also dumps the reference state-dict key/shape
lists used by tests/test_spec_cpu.py and the reference helpers' view of the modules (host_api.json). `--full` adds the full-width Kubric architecture (1.5 B parameters).
"""
import json
import os
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import gcd_oracle as O  # noqa: E402
from oracle import ref_shim, weights  # noqa: E402

GOLD = os.path.join(ROOT, "tests", "golden")
UNET_TINY = dict(O.UNET_KUBRIC, model_channels=64)
VAE_TINY = dict(O.VAE_DECODER, ch=64)
torch.set_grad_enabled(False)


def maxrel(a, b):
    return ((a - b).abs().max() / b.abs().max()).item()


def pin_unet(tag, cfg, B, T, H, W, steps):
    t0 = time.time()
    net = ref_shim.build_ref_unet(cfg)
    shapes = {k: tuple(v.shape) for k, v in net.state_dict().items()}
    json.dump({k: list(v) for k, v in shapes.items()}, open(os.path.join(GOLD, f"unet_{tag}_keys.json"), "w"))
    sd = weights.seeded_state(shapes, seed=0)
    net.load_state_dict(sd, strict=True)
    x, c, uc, ioi = weights.seeded_inputs(cfg, B, T, H, W)
    # ---- single forward through Denoiser + OpenAIWrapper + VideoUNet (reference classes)
    from sgm.modules.diffusionmodules.denoiser import Denoiser
    from sgm.modules.diffusionmodules.wrappers import OpenAIWrapper
    from sgm.modules.diffusionmodules.sampling import EulerEDMSampler
    den = Denoiser({"target": "sgm.modules.diffusionmodules.denoiser_scaling.VScalingWithEDMcNoise"})
    wrapped = OpenAIWrapper(net)
    BT = B * T
    sigma = torch.full((2 * BT,), 10.0)
    c_cat = {k: torch.cat((uc[k], c[k]), 0) for k in c}
    extra = dict(image_only_indicator=ioi, num_video_frames=T)
    ref_den = den(wrapped, torch.cat([x, x]) * 3.0, sigma, c_cat, **extra)
    net_fn = lambda xin, t, ctx, y, **kw: O.unet_forward(sd, cfg, xin, t, ctx, y, kw["num_video_frames"],
                                                         kw["image_only_indicator"])
    ora_den = O.denoise(net_fn, torch.cat([x, x]) * 3.0, sigma, c_cat, **extra)
    e1 = maxrel(ora_den, ref_den)
    # raw network output (what the CUDA VideoUNet must reproduce)
    cs, co, ci, cn = O.vscaling_edm_cnoise(sigma.view(-1, 1, 1, 1))
    xin = torch.cat((torch.cat([x, x]) * 3.0 * ci, c_cat["concat"]), 1)
    ref_net = net(xin, cn.reshape(-1), context=c_cat["crossattn"], y=c_cat["vector"], **extra)
    # ---- full sampler loop (reference EulerEDMSampler + LinearPredictionGuider)
    sampler = EulerEDMSampler(
        discretization_config={"target": "sgm.modules.diffusionmodules.discretizer.EDMDiscretization",
                               "params": {"sigma_max": 700.0}},
        num_steps=steps,
        guider_config={"target": "sgm.modules.diffusionmodules.guiders.LinearPredictionGuider",
                       "params": {"num_frames": T, "max_scale": 1.5, "min_scale": 1.0}},
        device="cpu")
    denoiser_fn = lambda inp, sig, cc: den(wrapped, inp, sig, cc, **extra)
    ref_samp = sampler(denoiser_fn, x.clone(), cond=c, uc=uc)
    ora_samp = O.euler_edm_sample(net_fn, x.clone(), c, uc, steps, T, 1.5, 1.0, **extra)
    e2 = maxrel(ora_samp, ref_samp)
    sig_ref = sampler.discretization(steps, device="cpu")
    assert torch.equal(sig_ref, O.edm_sigmas(steps)), "sigma schedule must be bit-exact"
    print(f"[unet {tag}] oracle vs reference: denoise {e1:.2e}  sample({steps} steps) {e2:.2e}  ({time.time()-t0:.0f}s)")
    assert e1 < 2e-5 and e2 < 2e-4, (e1, e2)
    torch.save({"cfg": cfg, "B": B, "T": T, "H": H, "W": W, "steps": steps, "sigma": 10.0, "x_mul": 3.0,
                "net_out": ref_net.clone(), "denoised": ref_den.clone(), "sampled": ref_samp.clone()},
               os.path.join(GOLD, f"unet_{tag}.pt"))


def pin_decoder(tag, cfg, T, H, W):
    dec = ref_shim.build_ref_decoder(cfg)
    shapes = {k: tuple(v.shape) for k, v in dec.state_dict().items()}
    json.dump({k: list(v) for k, v in shapes.items()}, open(os.path.join(GOLD, f"vae_{tag}_keys.json"), "w"))
    sd = weights.seeded_state(shapes, seed=0)
    dec.load_state_dict(sd, strict=True)
    g = torch.Generator().manual_seed(4321)
    z = torch.randn(T, cfg["z_channels"], H, W, generator=g)
    ref = dec(z / 0.18215, timesteps=T)
    ora = O.decode_first_stage(sd, cfg, z, T)
    e = maxrel(ora, ref)
    print(f"[vae {tag}] oracle vs reference: {e:.2e}")
    assert e < 2e-5, e
    torch.save({"cfg": cfg, "T": T, "H": H, "W": W, "z_seed": 4321, "decoded": ref.clone()},
               os.path.join(GOLD, f"vae_{tag}.pt"))


def pin_encoder(tag, cfg, n, H, W):
    """Reference Encoder + quant_conv + DiagonalGaussianDistribution.mode() (the pieces of AutoencoderKLModeOnly.encode that
    import here; the LightningModule wrapper itself needs pytorch_lightning)."""
    enc = ref_shim.build_ref_encoder(cfg)
    shapes = {k: tuple(v.shape) for k, v in enc.state_dict().items()}
    json.dump({k: list(v) for k, v in shapes.items()}, open(os.path.join(GOLD, f"enc_{tag}_keys.json"), "w"))
    sd = weights.seeded_state(shapes, seed=0)
    enc.load_state_dict(sd, strict=True)
    g = torch.Generator().manual_seed(777)
    x = torch.randn(n, cfg["in_channels"], H, W, generator=g).clamp_(-1, 1)
    zc = cfg["z_channels"]
    qw = torch.randn(2 * zc, 2 * zc, 1, 1, generator=g) * 0.4
    qb = torch.randn(2 * zc, generator=g) * 0.1
    from sgm.modules.distributions.distributions import DiagonalGaussianDistribution
    moments = enc(x)
    mode = DiagonalGaussianDistribution(torch.nn.functional.conv2d(moments, qw, qb)).mode() * 0.18215
    e1 = maxrel(O.encoder_forward(sd, cfg, x), moments)
    e2 = maxrel(O.encode_cond_frames(sd, cfg, x, qw, qb), mode)
    print(f"[enc {tag}] oracle vs reference: moments {e1:.2e}, mode*scale {e2:.2e}")
    assert e1 < 2e-5 and e2 < 2e-5, (e1, e2)
    torch.save({"cfg": cfg, "n": n, "H": H, "W": W, "x": x, "quant_w": qw, "quant_b": qb, "moments": moments.clone(),
                "mode_scaled": mode.clone()}, os.path.join(GOLD, f"enc_{tag}.pt"))


def pin_embedders():
    Concat, Spherical = ref_shim.ref_embedder_classes()
    g = torch.Generator().manual_seed(99)
    out = {}
    x1 = torch.tensor([6.0, 127.0, 0.02, 1.0])                       # fps_id / motion_bucket_id / cond_aug style scalars
    x2 = torch.randn(5, 3, generator=g) * 3.0
    out["concat_x1"], out["concat_x2"] = x1, x2
    out["concat_y1"], out["concat_y2"] = Concat(256)(x1), Concat(256)(x2)
    sph = Spherical(128)
    w = torch.randn(128, 13, generator=g) * 0.3
    b = torch.randn(128, generator=g) * 0.1
    sph.proj.weight.data.copy_(w); sph.proj.bias.data.copy_(b)
    xs = torch.cat([torch.randn(28, 2, generator=g) * 2.0, torch.rand(28, 1, generator=g) * 6.0], 1)
    out["sph_w"], out["sph_b"], out["sph_x"], out["sph_y"] = w, b, xs, sph(xs)
    assert torch.equal(O.concat_timestep_embedder_nd(x1, 256), out["concat_y1"])
    assert torch.equal(O.concat_timestep_embedder_nd(x2, 256), out["concat_y2"])
    e = maxrel(O.spherical_embedder(w, b, xs), out["sph_y"])
    print(f"[embedders] ConcatTimestepEmbedderND bit-exact; SphericalEmbedder oracle vs reference {e:.2e}")
    assert e < 1e-6
    torch.save(out, os.path.join(GOLD, "embedders.pt"))


def pin_host_api():
    """What the reference's host-side helpers make of this package's modules, so the tests need no reference tree:
    the LitEma shadow names of `HotPathRoot.model` (modules/ema.py) and the embedder attributes the GeneralConditioner
    reads and sets (encoders/modules.py:40-81, 93-130). The two conditioner classes are cut out of the reference source
    with `ast` and executed against the repo's embedders, as in ref_shim.ref_embedder_classes."""
    import ast
    import importlib
    import types
    import typing
    import torch.nn as nn
    from gcd_b200 import checkpoint, spec
    from gcd_b200.sampling import instantiate_from_config
    from gcd_b200.unet import VideoUNet
    from gcd_b200.vae import Encoder, VideoDecoder
    ref_shim.install()
    from sgm.modules.ema import LitEma
    root = checkpoint.HotPathRoot(VideoUNet(**spec.unet_ctor_kwargs(spec.UNET_TINY)),
                                  VideoDecoder(**spec.decoder_ctor_kwargs(spec.VAE_TINY)),
                                  Encoder(**spec.encoder_ctor_kwargs(spec.VAE_ENCODER_TINY)))
    out = {"litema_shadows_of_model": LitEma(root.model, decay=0.999).m_name2s_name}
    path = os.path.join(ref_shim.REF, "sgm", "modules", "encoders", "modules.py")
    body = [n for n in ast.parse(open(path).read()).body
            if isinstance(n, ast.ClassDef) and n.name in ("AbstractEmbModel", "GeneralConditioner")]
    ns = {"torch": torch, "nn": nn, "Union": typing.Union, "List": typing.List, "Dict": typing.Dict,
          "Optional": typing.Optional, "ListConfig": list, "instantiate_from_config": instantiate_from_config,
          "disabled_train": lambda self, mode=True: self, "count_params": lambda m, verbose=False: 0,
          "print": lambda *a, **k: None}
    exec(compile(ast.Module(body=body, type_ignores=[]), path, "exec"), ns)
    base = ns["AbstractEmbModel"]
    out["abstract_emb_model"] = {k: getattr(base(), k) for k, v in vars(base).items() if isinstance(v, property)}
    fake = types.ModuleType("sgm.modules.encoders.modules")
    fake.AbstractEmbModel = base
    pkg = types.ModuleType("sgm.modules.encoders")
    pkg.__path__ = []
    sys.modules["sgm.modules.encoders"], sys.modules["sgm.modules.encoders.modules"] = pkg, fake
    import gcd_b200.embedders as E
    importlib.reload(E)
    configs = [{"target": "gcd_b200.embedders.ConcatTimestepEmbedderND", "params": {"outdim": 256}, "input_key": "fps_id",
                "is_trainable": False},
               {"target": "gcd_b200.embedders.SphericalEmbedder", "params": {"embed_dim": 128}, "input_key": "spherical",
                "is_trainable": False, "ucg_rate": 0.1}]
    cond = ns["GeneralConditioner"](configs)
    out["general_conditioner"] = [
        {"config": cfg, "class": type(e).__name__, "input_key": e.input_key, "ucg_rate": e.ucg_rate,
         "is_trainable": e.is_trainable, "legacy_ucg_val": e.legacy_ucg_val, "training": e.training,
         "requires_grad": [p.requires_grad for p in e.parameters()]} for cfg, e in zip(configs, cond.embedders)]
    del sys.modules["sgm.modules.encoders"], sys.modules["sgm.modules.encoders.modules"]
    importlib.reload(E)
    json.dump(out, open(os.path.join(GOLD, "host_api.json"), "w"), indent=0, sort_keys=True)
    print(f"[host api] {len(out['litema_shadows_of_model'])} LitEma shadows; conditioner accepted "
          f"{[d['class'] for d in out['general_conditioner']]}")


def pin_closed_forms():
    """Known-answer values derivable from the source (SURVEY.md §8(c))."""
    ref_shim.install()
    from sgm.modules.diffusionmodules.discretizer import EDMDiscretization
    from sgm.modules.diffusionmodules.guiders import LinearPredictionGuider
    from sgm.modules.diffusionmodules.util import timestep_embedding
    out = {}
    for n in (25, 50):
        out[f"sigmas_{n}"] = EDMDiscretization(sigma_max=700.0)(n, device="cpu")
    out["scale_1.5"] = LinearPredictionGuider(1.5, 14, 1.0).scale
    out["scale_2.5"] = LinearPredictionGuider(2.5, 14, 1.0).scale
    t = torch.tensor([0.5756, -0.37, 1.23])
    out["temb_t"] = t
    out["temb_320"] = timestep_embedding(t, 320)
    torch.save(out, os.path.join(GOLD, "closed_forms.pt"))
    assert torch.equal(out["sigmas_25"], O.edm_sigmas(25)) and torch.equal(out["sigmas_50"], O.edm_sigmas(50))
    assert torch.equal(out["scale_1.5"], O.guider_scale(14, 1.5)) and torch.equal(out["temb_320"], O.timestep_embedding(t, 320))
    print("[closed forms] sigma schedule / guider scale / timestep embedding: bit-exact")


if __name__ == "__main__":
    os.makedirs(GOLD, exist_ok=True)
    torch.manual_seed(0)
    pin_closed_forms()
    pin_unet("tiny", UNET_TINY, B=1, T=3, H=16, W=24, steps=4)
    pin_decoder("tiny", VAE_TINY, T=3, H=8, W=8)
    pin_encoder("tiny", dict(O.VAE_ENCODER, ch=64), n=2, H=64, W=96)
    pin_embedders()
    pin_host_api()
    if "--full" in sys.argv:
        pin_unet("kubric", O.UNET_KUBRIC, B=1, T=2, H=16, W=16, steps=2)
        pin_unet("pardom", O.UNET_PARDOM, B=1, T=2, H=8, W=8, steps=1)
        pin_decoder("full", O.VAE_DECODER, T=2, H=8, W=8)
        pin_encoder("full", O.VAE_ENCODER, n=1, H=64, W=64)
