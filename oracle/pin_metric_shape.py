"""Reference goldens AT THE METRIC SHAPE (TEST INFRASTRUCTURE; run in the BUILD CONTAINER only, needs /root/reference).

    python -m oracle.pin_metric_shape [unet_kubric] [unet_pardom] [traj25] [traj50] [vae_fullres]     (default: all)

Everything stored is an output of the REFERENCE's own modules (imported through oracle/ref_shim.py) on CPU fp32 with the
seeded weights / inputs of oracle/weights.py — the CUDA path is compared with these in tests/test_metric_shape_gpu.py:

  unet_{kubric,pardom}_metric.pt  one CFG forward (28 frames) of the full-width VideoUNet at latent 72x128, the shape
                                  bench.py measures (video_model.py:461-540): exercises the BN=160 pair tiles at
                                  M=258 048, the 9216-token attention instantiation, T=14 temporal GroupNorm. Stored at
                                  1152 seeded pixel positions (every frame and channel) + per-frame, per-channel moments.
  traj25.pt                       the complete 25-step EulerEDMSampler trajectory (sampling.py:123-144) at 14x32x48, full
                                  width, LinearPredictionGuider 1.0 -> 1.5 (BASELINE.md §4.4); x after steps 1, 5, 10, 25,
                                  at 512 seeded pixel positions + moments of the final sample.
  traj50.pt                       config 4: 50 steps, guider max scale 2.5, at 14x16x24, full width; x after 1, 10, 25, 50,
                                  every pixel.
  vae_fullres.pt                  VideoDecoder (temporal_ae.py:293-349) of 14 frames at latent 72x128 -> 576x1024 px, stored
                                  as 2304 seeded positions of the 8x strided subsample + three full-resolution 64x64 crops +
                                  per-frame moments.

Samples keep every golden file under 1 MB; the pixel indices are stored with the values they select.
"""
import os
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import gcd_oracle as O  # noqa: E402
from oracle import ref_shim, weights  # noqa: E402

GOLD = os.path.join(ROOT, "tests", "golden")
torch.set_grad_enabled(False)

CROPS = [(0, 0, 0), (7, 256, 480), (13, 512, 960)]          # (frame, y0, x0) of the 64x64 full-resolution crops


def pixel_sample(h, w, n, seed):
    """n distinct flat pixel indices of an h x w image, ascending, from a seeded generator."""
    g = torch.Generator().manual_seed(seed)
    return torch.randperm(h * w, generator=g)[:n].sort().values


def at_pixels(x, pix):
    """[..., H, W] -> [..., len(pix)]: the values at the flat pixel indices `pix`."""
    return x.flatten(-2)[..., pix].contiguous()


def moments(x):
    """Per-frame, per-channel mean and mean square of [N, C, H, W] over the whole image."""
    return {"mean": x.mean(dim=(2, 3)), "sqmean": x.pow(2).mean(dim=(2, 3))}


def pack_unet_metric(cfg, T, H, W, net_out):
    pix = pixel_sample(H, W, 1152, seed=72128)
    return {"cfg": cfg, "B": 1, "T": T, "H": H, "W": W, "sigma": 10.0, "x_mul": 3.0, "pix": pix,
            "net_out_pix": at_pixels(net_out, pix), **moments(net_out)}


def pack_traj(cfg, T, H, W, steps, max_scale, states, final, n_pix):
    pix = pixel_sample(H, W, n_pix, seed=steps)
    return {"cfg": cfg, "B": 1, "T": T, "H": H, "W": W, "steps": steps, "max_scale": max_scale, "min_scale": 1.0, "pix": pix,
            "after_steps_pix": {k: at_pixels(v, pix) for k, v in states.items()}, "sampled_pix": at_pixels(final, pix),
            **moments(final)}


def pack_decoder_fullres(cfg, T, H, W, sub8, crops, mean, sqmean, norm):
    pix = pixel_sample(H, W, 2304, seed=4321)
    return {"cfg": cfg, "T": T, "H": H, "W": W, "z_seed": 4321, "pix": pix, "sub8_pix": at_pixels(sub8, pix), "crops": crops,
            "crop_pos": CROPS, "mean": mean, "sqmean": sqmean, "norm": norm}


def _loaded_ref_unet(cfg):
    net = ref_shim.build_ref_unet(cfg)
    shapes = {k: tuple(v.shape) for k, v in net.state_dict().items()}
    sd = weights.seeded_state(shapes, seed=0)
    net.load_state_dict(sd, strict=True)
    return net


def pin_unet_metric(tag, cfg, T=14, H=72, W=128):
    t0 = time.time()
    net = _loaded_ref_unet(cfg)
    x, c, uc, ioi = weights.seeded_inputs(cfg, 1, T, H, W)
    sigma = torch.full((2 * T,), 10.0)
    c_cat = {k: torch.cat((uc[k], c[k]), 0) for k in c}
    cs, co, ci, cn = O.vscaling_edm_cnoise(sigma.view(-1, 1, 1, 1))
    xin = torch.cat((torch.cat([x, x]) * 3.0 * ci, c_cat["concat"]), 1)
    out = net(xin, cn.reshape(-1), context=c_cat["crossattn"], y=c_cat["vector"], image_only_indicator=ioi,
              num_video_frames=T)
    print(f"[unet {tag} metric] reference forward {tuple(out.shape)} in {time.time() - t0:.0f} s, rms {out.pow(2).mean().sqrt():.4f}",
          flush=True)
    torch.save(pack_unet_metric(cfg, T, H, W, out), os.path.join(GOLD, f"unet_{tag}_metric.pt"))


def pin_traj(tag, cfg, T, H, W, steps, max_scale, keep, n_pix):
    t0 = time.time()
    net = _loaded_ref_unet(cfg)
    from sgm.modules.diffusionmodules.denoiser import Denoiser
    from sgm.modules.diffusionmodules.sampling import EulerEDMSampler
    from sgm.modules.diffusionmodules.wrappers import OpenAIWrapper
    den = Denoiser({"target": "sgm.modules.diffusionmodules.denoiser_scaling.VScalingWithEDMcNoise"})
    wrapped = OpenAIWrapper(net)
    x, c, uc, ioi = weights.seeded_inputs(cfg, 1, T, H, W)
    extra = dict(image_only_indicator=ioi, num_video_frames=T)
    sampler = EulerEDMSampler(
        discretization_config={"target": "sgm.modules.diffusionmodules.discretizer.EDMDiscretization",
                               "params": {"sigma_max": 700.0}},
        num_steps=steps,
        guider_config={"target": "sgm.modules.diffusionmodules.guiders.LinearPredictionGuider",
                       "params": {"num_frames": T, "max_scale": max_scale, "min_scale": 1.0}},
        device="cpu")
    seen = []          # the denoiser's input at call i is cat([x_i] * 2): x_i = state BEFORE step i (x_0 = scaled noise)

    def denoiser_fn(inp, sig, cc):
        seen.append(inp[:T].clone())
        print(f"  [{tag}] step {len(seen)}/{steps}  sigma {sig[0].item():.4f}  ({time.time() - t0:.0f} s)", flush=True)
        return den(wrapped, inp, sig, cc, **extra)

    final = sampler(denoiser_fn, x.clone(), cond=c, uc=uc)
    states = {k: (seen[k].clone() if k < steps else final.clone()) for k in keep}      # x after k steps
    torch.save(pack_traj(cfg, T, H, W, steps, max_scale, states, final, n_pix), os.path.join(GOLD, f"{tag}.pt"))
    print(f"[{tag}] reference {steps}-step trajectory at {T}x{H}x{W} in {time.time() - t0:.0f} s; |x| {final.abs().mean():.4f}", flush=True)


def pin_decoder_fullres(T=14, H=72, W=128):
    t0 = time.time()
    cfg = O.VAE_DECODER
    dec = ref_shim.build_ref_decoder(cfg)
    shapes = {k: tuple(v.shape) for k, v in dec.state_dict().items()}
    dec.load_state_dict(weights.seeded_state(shapes, seed=0), strict=True)
    g = torch.Generator().manual_seed(4321)
    z = torch.randn(T, cfg["z_channels"], H, W, generator=g)
    out = dec(z / 0.18215, timesteps=T)                                   # [14, 3, 576, 1024]
    crops = [out[f, :, y0:y0 + 64, x0:x0 + 64].clone() for f, y0, x0 in CROPS]
    m = moments(out)
    torch.save(pack_decoder_fullres(cfg, T, H, W, out[:, :, ::8, ::8], crops, m["mean"], m["sqmean"], out.norm().item()),
               os.path.join(GOLD, "vae_fullres.pt"))
    print(f"[vae fullres] reference decode {tuple(out.shape)} in {time.time() - t0:.0f} s", flush=True)


if __name__ == "__main__":
    want = sys.argv[1:] or ["unet_kubric", "unet_pardom", "traj25", "traj50", "vae_fullres"]
    torch.manual_seed(0)
    if "unet_kubric" in want:
        pin_unet_metric("kubric", O.UNET_KUBRIC)
    if "unet_pardom" in want:
        pin_unet_metric("pardom", O.UNET_PARDOM)
    if "traj50" in want:
        pin_traj("traj50", O.UNET_KUBRIC, 14, 16, 24, 50, 2.5, keep=(1, 10, 25, 50), n_pix=16 * 24)
    if "traj25" in want:
        pin_traj("traj25", O.UNET_KUBRIC, 14, 32, 48, 25, 1.5, keep=(1, 5, 10, 25), n_pix=512)
    if "vae_fullres" in want:
        pin_decoder_fullres()
