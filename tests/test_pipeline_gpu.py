"""GPU parity: EDM/Euler sampler loop (generic + fused paths) and the temporal VAE decoder against golden outputs of
the REFERENCE's own EulerEDMSampler / VideoDecoder (tests/golden, oracle/pin_against_reference.py)."""
import os
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
GOLD = os.path.join(ROOT, "tests", "golden")

# stated tolerances (relative L2 vs the fp32 reference; fp16 tensor-core operands, fp32 accumulation/residuals)
TOL_SAMPLE = 1.5e-2     # after the full multi-step trajectory (errors compound through the Euler steps)
TOL_DECODE = 5e-3


def relerr(a, b):
    a, b = a.float().cpu(), b.float().cpu()
    return ((a - b).norm() / b.norm()).item()


def _build(tag):
    from gcd_b200 import sampling, spec
    from gcd_b200.unet import VideoUNet
    from oracle import weights
    gold = torch.load(os.path.join(GOLD, f"unet_{tag}.pt"))
    cfg = gold["cfg"]
    net = VideoUNet(**spec.unet_ctor_kwargs(cfg))
    net.load_state_dict(weights.seeded_state(spec.unet_param_shapes(cfg), seed=0))
    net = net.cuda()
    den = sampling.Denoiser({"target": "gcd_b200.sampling.VScalingWithEDMcNoise"})
    model = sampling.OpenAIWrapper(net)
    sampler = sampling.EulerEDMSampler(
        discretization_config={"target": "gcd_b200.sampling.EDMDiscretization", "params": {"sigma_max": 700.0}},
        num_steps=gold["steps"],
        guider_config={"target": "gcd_b200.sampling.LinearPredictionGuider",
                       "params": {"num_frames": gold["T"], "max_scale": 1.5, "min_scale": 1.0}},
        device="cuda")
    x, c, uc, ioi = weights.seeded_inputs(cfg, gold["B"], gold["T"], gold["H"], gold["W"])
    cuda = lambda d: {k: v.cuda() for k, v in d.items()}
    extra = dict(image_only_indicator=ioi.cuda(), num_video_frames=gold["T"])
    return gold, den, model, sampler, x.cuda(), cuda(c), cuda(uc), extra


@pytest.mark.parametrize("tag", ["tiny", "kubric"])
def test_sampler_generic_and_fused_vs_reference(tag):
    from gcd_b200 import sampling
    if not os.path.exists(os.path.join(GOLD, f"unet_{tag}.pt")):
        pytest.skip("golden not generated")
    gold, den, model, sampler, x, c, uc, extra = _build(tag)
    # generic path: an opaque closure (not recognisable), reference control flow
    opaque = lambda inp, sig, cc, _d=den, _m=model, _e=extra: _d(_m, inp, sig, cc, **_e)
    out_g = sampler(opaque, x.clone(), cond=c, uc=uc)
    assert sampler.last_path == "generic"
    eg = relerr(out_g, gold["sampled"])
    # fused path: explicit handle
    out_f = sampler(sampling.FusedDenoiser(den, model, **extra), x.clone(), cond=c, uc=uc)
    assert sampler.last_path == "fused"
    ef = relerr(out_f, gold["sampled"])
    print(f"sampler[{tag}] {gold['steps']} steps: generic {eg:.3e}  fused {ef:.3e}  fused-vs-generic {relerr(out_f, out_g):.3e}")
    assert eg < TOL_SAMPLE and ef < TOL_SAMPLE


def test_sampler_recognises_diffusion_engine_closure():
    """The closure shape of DiffusionEngine.sample_video (models/diffusion.py:531-532) takes the fused path."""
    gold, den, model, sampler, x, c, uc, extra = _build("tiny")

    class Engine:  # stands in for DiffusionEngine: attributes `denoiser` and `model`
        pass

    self = Engine()
    self.denoiser, self.model = den, model
    additional_model_inputs = extra

    def denoiser(input, sigma, c):
        return self.denoiser(self.model, input, sigma, c, **additional_model_inputs)

    out = sampler(denoiser, x.clone(), cond=c, uc=uc)
    assert sampler.last_path == "fused"
    assert relerr(out, gold["sampled"]) < TOL_SAMPLE


@pytest.mark.parametrize("tag", ["tiny", "full"])
def test_decoder_vs_reference(tag):
    from gcd_b200 import spec
    from gcd_b200.vae import VideoDecoder
    from oracle import weights
    path = os.path.join(GOLD, f"vae_{tag}.pt")
    if not os.path.exists(path):
        pytest.skip("golden not generated")
    gold = torch.load(path)
    cfg = gold["cfg"]
    dec = VideoDecoder(**spec.decoder_ctor_kwargs(cfg))
    dec.load_state_dict(weights.seeded_state(spec.decoder_param_shapes(cfg), seed=0), strict=True)
    dec = dec.cuda()
    g = torch.Generator().manual_seed(gold["z_seed"])
    z = torch.randn(gold["T"], cfg["z_channels"], gold["H"], gold["W"], generator=g)
    out = dec((z / 0.18215).cuda(), timesteps=gold["T"])
    assert out.shape == gold["decoded"].shape
    e = relerr(out, gold["decoded"])
    print(f"vae[{tag}] rel-L2 vs reference golden: {e:.3e}")
    assert e < TOL_DECODE


def test_decode_first_stage_in_ragged_chunks_vs_oracle():
    """DiffusionEngine.decode_first_stage decodes `en_and_decode_n_samples_a_time` frames at a time, each chunk with
    timesteps = its own length (models/diffusion.py:233-251): 14 frames in chunks of 5 -> 5, 5, 4 (ragged last chunk; the temporal
    convolutions and clip-wide GroupNorms see only their chunk)."""
    from gcd_b200 import spec, synthetic
    from gcd_b200.pipeline import GCDHotPath
    from oracle import gcd_oracle as O
    pipe = GCDHotPath(spec.UNET_TINY, spec.VAE_TINY, num_steps=2, num_frames=14, device="cuda")
    vst = synthetic.seeded_state(spec.decoder_param_shapes(spec.VAE_TINY), seed=0)
    pipe.decoder.load_state_dict(vst, strict=True)
    pipe.decoder.cuda()
    z = torch.randn(14, 4, 8, 16, generator=torch.Generator().manual_seed(3))
    out = pipe.decode_first_stage(z.cuda(), decoding_t=5)
    with torch.no_grad():
        ref = torch.cat([O.decode_first_stage(vst, spec.VAE_TINY, z[i:i + 5], min(5, 14 - i)) for i in range(0, 14, 5)], 0)
    assert out.shape == ref.shape == (14, 3, 64, 128)
    assert relerr(out, ref) < TOL_DECODE
    full = pipe.decode_first_stage(z.cuda())                      # one chunk of 14: a different function of z
    assert relerr(full[:5], ref[:5]) > 1e-3


@pytest.mark.parametrize("tag", ["tiny", "full"])
def test_encoder_vs_reference(tag):
    """SURVEY.md §8(f) rank 1: VAE Encoder of the conditioning frames vs the reference Encoder's own outputs; the fused
    quant_conv + mode + scale path vs reference quant_conv -> DiagonalGaussianDistribution.mode() * scale_factor."""
    from gcd_b200 import spec
    from gcd_b200.vae import Encoder
    from oracle import weights
    path = os.path.join(GOLD, f"enc_{tag}.pt")
    if not os.path.exists(path):
        pytest.skip("golden not generated")
    gold = torch.load(path)
    cfg = gold["cfg"]
    enc = Encoder(**spec.encoder_ctor_kwargs(cfg))
    enc.load_state_dict(weights.seeded_state(spec.encoder_param_shapes(cfg), seed=0), strict=True)
    enc = enc.cuda()
    out = enc(gold["x"].cuda())
    assert out.shape == gold["moments"].shape
    e1 = relerr(out, gold["moments"])
    z = enc.encode_mode(gold["x"].cuda(), gold["quant_w"].cuda(), gold["quant_b"].cuda(), 0.18215)
    assert z.shape == gold["mode_scaled"].shape
    e2 = relerr(z, gold["mode_scaled"])
    print(f"enc[{tag}] rel-L2 vs reference golden: moments {e1:.3e}, scaled mode {e2:.3e}")
    assert e1 < TOL_DECODE and e2 < TOL_DECODE


def test_encoder_live_oracle_ragged_shape():
    """A non-square size whose level sizes (40x192, 20x96, 10x48, 5x24) leave ragged tiles, two frames."""
    from gcd_b200 import spec
    from gcd_b200.vae import Encoder
    from oracle import gcd_oracle as O, weights
    cfg = spec.VAE_ENCODER_TINY
    sd = weights.seeded_state(spec.encoder_param_shapes(cfg), seed=3)
    enc = Encoder(**spec.encoder_ctor_kwargs(cfg))
    enc.load_state_dict(sd, strict=True)
    enc = enc.cuda()
    x = torch.randn(2, 3, 40, 192, generator=torch.Generator().manual_seed(5)).clamp_(-1, 1)
    with torch.no_grad():
        ref = O.encoder_forward(sd, cfg, x)
    assert relerr(enc(x.cuda()), ref) < TOL_DECODE
    with pytest.raises(ValueError):
        enc(torch.zeros(1, 3, 36, 64).cuda())          # not a multiple of 8
    with pytest.raises(ValueError):
        enc(torch.zeros(1, 3, 40, 88).cuda())          # 5 x 11 mid-attention tokens: rows not 16-byte aligned


def test_sampler_50_steps_scale_2p5_fused_equals_generic():
    """Config 4 of BASELINE.json (50 steps, guider max scale 2.5) on the tiny network: fused == generic control flow."""
    from gcd_b200 import sampling, spec
    from gcd_b200.unet import VideoUNet
    from oracle import weights
    cfg = spec.UNET_TINY
    net = VideoUNet(**spec.unet_ctor_kwargs(cfg))
    net.load_state_dict(weights.seeded_state(spec.unet_param_shapes(cfg), seed=0))
    net = net.cuda()
    T = 2
    den = sampling.Denoiser({"target": "gcd_b200.sampling.VScalingWithEDMcNoise"})
    model = sampling.OpenAIWrapper(net)
    sampler = sampling.EulerEDMSampler(
        {"target": "gcd_b200.sampling.EDMDiscretization", "params": {"sigma_max": 700.0}}, num_steps=50,
        guider_config={"target": "gcd_b200.sampling.LinearPredictionGuider", "params": {"num_frames": T, "max_scale": 2.5}},
        device="cuda")
    x, c, uc, ioi = weights.seeded_inputs(cfg, 1, T, 8, 8)
    cuda = lambda d: {k: v.cuda() for k, v in d.items()}
    extra = dict(image_only_indicator=torch.zeros(2, T).cuda(), num_video_frames=T)
    opaque = lambda inp, sig, cc: den(model, inp, sig, cc, **extra)
    a = sampler(opaque, x.clone().cuda(), cond=cuda(c), uc=cuda(uc))
    b = sampler(sampling.FusedDenoiser(den, model, **extra), x.clone().cuda(), cond=cuda(c), uc=cuda(uc))
    assert sampler.last_path == "fused" and torch.isfinite(a).all()
    assert relerr(b, a) < 1e-2


def test_bench_dump_outputs_are_reproducible(tmp_path):
    """`bench.py --dump-outputs DIR` writes the last timed step's latents and frames as float32 .npy; two runs with the same
    arguments sample the same seeded inputs, so their dumps agree to the run-to-run noise of the fp64 statistics atomics."""
    import json
    import subprocess
    import numpy as np
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    dumps = []
    for run in range(2):
        d = tmp_path / f"run{run}"
        r = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--gpus", "1", "--steps", "2", "--warmup", "0",
                            "--workload", "tiny-selftest", "--no-cpu-baseline", "--dump-outputs", str(d)],
                           capture_output=True, text=True, timeout=900)
        assert r.returncode == 0, r.stderr[-2000:]
        line = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
        assert line["steps"] == 2
        dumps.append({n: np.load(d / f"{n}.npy") for n in ("latents", "frames")})
        assert sorted(os.listdir(d)) == ["frames.npy", "latents.npy"]
    for n, shape in (("latents", (14, 4, 16, 24)), ("frames", (14, 3, 128, 192))):
        a, b = dumps[0][n], dumps[1][n]
        assert a.dtype == np.float32 and a.shape == shape and np.isfinite(a).all() and np.abs(a).max() > 0
        assert np.linalg.norm(a - b) / np.linalg.norm(b) < 1e-4, n


def test_cfg_parallel_two_gpus():
    """SURVEY.md §8(f) rank 2 on real hardware (skipped on a 1-GPU box): one clip over two GPUs (uc | c) with NCCL equals the
    single-GPU fused sampler within the 16-bit noise floor and leaves both ranks with bit-identical latents."""
    import json
    import subprocess
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", str(29700 + os.getpid() % 200), os.path.join(root, "tools", "cfg_parallel_check.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    out = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
    assert out["ranks_bit_identical"] and out["tiny_rel_l2_vs_single_gpu"] < 5e-3
