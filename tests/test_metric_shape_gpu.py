"""GPU parity AT THE METRIC SHAPE against outputs of the REFERENCE's own modules (tests/golden/*_metric.pt, traj25.pt,
traj50.pt, vae_fullres.pt — written by oracle/pin_metric_shape.py; outputs are stored at seeded pixel positions that cover
every frame and channel, with whole-image moments, to keep each file under 1 MB):

* one CFG forward of the full-width VideoUNet at latent 28x72x128 — the shape bench.py times: BN=160 pair tiles at M=258 048,
  the 9216-token attention instantiation (`attn_kernel<4,1>`), rbufs=2 residual epilogues, T=14 temporal GroupNorm over
  129 024 rows (Kubric and ParDom conditioning widths);
* the complete 25-step Euler trajectory at 14x32x48, full width (BASELINE.md §4.4), and the 50-step / max-scale-2.5 one of
  BASELINE config 4 at 14x16x24, intermediate states included;
* the VideoDecoder at 576x1024 px (14 frames), against a strided subsample, full-resolution crops and per-frame moments;
* the sigma schedule the product puts on the DEVICE, bit for bit against the reference's values.

Stated tolerances (relative L2 vs the fp32 reference; 16-bit tensor-core operands, fp32 accumulate / residual / norms):
network output 4e-3, multi-step sample 1.5e-2, VAE decode 5e-3; schedule: bit-exact.
"""
import os
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
GOLD = os.path.join(ROOT, "tests", "golden")

TOL_NET, TOL_SAMPLE, TOL_DECODE = 4e-3, 1.5e-2, 5e-3


def relerr(a, b):
    a, b = a.float().cpu(), b.float().cpu()
    return ((a - b).norm() / b.norm()).item()


def _gold(name):
    return torch.load(os.path.join(GOLD, name))


def at_pixels(x, pix):
    """[..., H, W] -> [..., len(pix)] at the golden's flat pixel indices (oracle/pin_metric_shape.py)."""
    return x.float().cpu().flatten(-2)[..., pix]


def moment_errors(x, gold):
    """Whole-image per-frame, per-channel moments vs the golden's: (max |d mean| / max rms, rel-L2 of the mean squares)."""
    x = x.float().cpu()
    e_mean = (x.mean(dim=(2, 3)) - gold["mean"]).abs().max().item() / gold["sqmean"].sqrt().max().item()
    return e_mean, relerr(x.pow(2).mean(dim=(2, 3)), gold["sqmean"])


_NETS = {}


def _net(cfg):
    """Full-width VideoUNet with the seeded weights, built once per architecture (1.5 B parameters from host generators)."""
    from gcd_b200 import spec
    from gcd_b200.unet import VideoUNet
    from oracle import weights
    key = tuple(sorted((k, str(v)) for k, v in cfg.items()))
    if key not in _NETS:
        _NETS.clear()                                   # one 6 GB fp32 parameter set at a time
        net = VideoUNet(**spec.unet_ctor_kwargs(cfg))
        net.load_state_dict(weights.seeded_state(spec.unet_param_shapes(cfg), seed=0), strict=True)
        _NETS[key] = net.cuda()
    return _NETS[key]


def test_sigma_schedule_on_device_is_bit_exact():
    from gcd_b200 import sampling
    g = torch.load(os.path.join(GOLD, "closed_forms.pt"))
    for n in (25, 50):
        s = sampling.EulerEDMSampler(
            discretization_config={"target": "gcd_b200.sampling.EDMDiscretization", "params": {"sigma_max": 700.0}},
            num_steps=n, guider_config={"target": "gcd_b200.sampling.LinearPredictionGuider",
                                        "params": {"num_frames": 14, "max_scale": 1.5}}, device="cuda")
        x = torch.ones(14, 4, 8, 8, device="cuda")
        _, _, sigmas, num_sigmas, _, _ = s.prepare_sampling_loop(x, {}, {})
        assert sigmas.is_cuda and num_sigmas == n + 1
        assert torch.equal(sigmas.cpu(), g[f"sigmas_{n}"])
        assert torch.equal(x.cpu(), torch.ones(14, 4, 8, 8) * torch.sqrt(1.0 + g[f"sigmas_{n}"][0] ** 2.0))


@pytest.mark.parametrize("tag", ["kubric", "pardom"])
def test_unet_forward_at_metric_shape_vs_reference(tag):
    from oracle import gcd_oracle as O, weights
    gold = _gold(f"unet_{tag}_metric.pt")
    cfg, T, H, W = gold["cfg"], gold["T"], gold["H"], gold["W"]
    assert (2 * T, H, W) == (28, 72, 128)
    net = _net(cfg)
    x, c, uc, ioi = weights.seeded_inputs(cfg, 1, T, H, W)
    sigma = torch.full((2 * T,), gold["sigma"])
    c_cat = {k: torch.cat((uc[k], c[k]), 0) for k in c}
    cs, co, ci, cn = O.vscaling_edm_cnoise(sigma.view(-1, 1, 1, 1))
    xin = torch.cat((torch.cat([x, x]) * gold["x_mul"] * ci, c_cat["concat"]), 1)
    out = net(xin.cuda(), cn.reshape(-1).cuda(), context=c_cat["crossattn"].cuda(), y=c_cat["vector"].cuda(),
              num_video_frames=T, image_only_indicator=ioi.cuda())
    assert out.shape == (2 * T, cfg["out_channels"], H, W)
    got, ref = at_pixels(out, gold["pix"]), gold["net_out_pix"]
    e = relerr(got, ref)
    worst = max(relerr(got[f], ref[f]) for f in range(2 * T))
    e_mean, e_sq = moment_errors(out, gold)
    print(f"unet[{tag}] 28x72x128 rel-L2 vs reference: {e:.3e} (worst frame {worst:.3e}), frame means {e_mean:.3e}, "
          f"second moments {e_sq:.3e}")
    assert e < TOL_NET and worst < 2 * TOL_NET and e_mean < TOL_NET and e_sq < TOL_NET


def _sample(gold):
    from gcd_b200 import sampling
    from oracle import weights
    cfg, T, H, W = gold["cfg"], gold["T"], gold["H"], gold["W"]
    net = _net(cfg)
    den = sampling.Denoiser({"target": "gcd_b200.sampling.VScalingWithEDMcNoise"})
    sampler = sampling.EulerEDMSampler(
        discretization_config={"target": "gcd_b200.sampling.EDMDiscretization", "params": {"sigma_max": 700.0}},
        num_steps=gold["steps"],
        guider_config={"target": "gcd_b200.sampling.LinearPredictionGuider",
                       "params": {"num_frames": T, "max_scale": gold["max_scale"], "min_scale": gold["min_scale"]}},
        device="cuda")
    sampler.trace_steps = set(gold["after_steps_pix"].keys())
    x, c, uc, ioi = weights.seeded_inputs(cfg, 1, T, H, W)
    cuda = lambda d: {k: v.cuda() for k, v in d.items()}
    fd = sampling.FusedDenoiser(den, sampling.OpenAIWrapper(net), image_only_indicator=ioi.cuda(), num_video_frames=T)
    out = sampler(fd, x.cuda(), cond=cuda(c), uc=cuda(uc))
    assert sampler.last_path == "fused"
    return out, sampler.trace


@pytest.mark.parametrize("name", ["traj25", "traj50"])
def test_full_trajectory_vs_reference(name):
    """The whole sampler loop (sampling.py:123-144): state after selected step counts and the final sample."""
    gold = _gold(f"{name}.pt")
    out, trace = _sample(gold)
    pix = gold["pix"]
    errs = {k: relerr(at_pixels(trace[k], pix), v) for k, v in sorted(gold["after_steps_pix"].items()) if k in trace}
    e = relerr(at_pixels(out, pix), gold["sampled_pix"])
    e_mean, e_sq = moment_errors(out, gold)
    print(f"{name}: {gold['steps']} steps at 14x{gold['H']}x{gold['W']}, max scale {gold['max_scale']}: rel-L2 after k steps "
          f"{ {k: f'{v:.2e}' for k, v in errs.items()} }, final {e:.3e}, frame means {e_mean:.3e}, second moments {e_sq:.3e}")
    assert len(errs) >= 3 and all(v < TOL_SAMPLE for v in errs.values())
    assert e < TOL_SAMPLE and e_mean < TOL_SAMPLE and e_sq < TOL_SAMPLE


def test_vae_decode_full_resolution_vs_reference():
    from gcd_b200 import spec
    from gcd_b200.vae import VideoDecoder
    from oracle import weights
    gold = _gold("vae_fullres.pt")
    cfg, T, H, W = gold["cfg"], gold["T"], gold["H"], gold["W"]
    assert (T, H, W) == (14, 72, 128)
    _NETS.clear()
    dec = VideoDecoder(**spec.decoder_ctor_kwargs(cfg))
    dec.load_state_dict(weights.seeded_state(spec.decoder_param_shapes(cfg), seed=0), strict=True)
    dec = dec.cuda()
    g = torch.Generator().manual_seed(gold["z_seed"])
    z = torch.randn(T, cfg["z_channels"], H, W, generator=g)
    out = dec((z / 0.18215).cuda(), timesteps=T)
    assert out.shape == (T, 3, 8 * H, 8 * W)
    e_sub = relerr(at_pixels(out[:, :, ::8, ::8], gold["pix"]), gold["sub8_pix"])
    e_crop = max(relerr(out[f, :, y0:y0 + 64, x0:x0 + 64], cr) for (f, y0, x0), cr in zip(gold["crop_pos"], gold["crops"]))
    e_mean, e_sq = moment_errors(out, gold)
    print(f"vae 14x576x1024: rel-L2 subsample {e_sub:.3e}, crops {e_crop:.3e}, frame means {e_mean:.3e}, second moments {e_sq:.3e}")
    assert e_sub < TOL_DECODE and e_crop < TOL_DECODE and e_mean < TOL_DECODE and e_sq < TOL_DECODE
