"""CPU tests: oracle pinned to the reference's golden vectors, host-side sampler classes, FLOP model, C-ABI exports,
and the world_size-2 gloo path of the clip sharding/gather."""
import json
import os
import re
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
GOLD = os.path.join(ROOT, "tests", "golden")

from gcd_b200 import flops, sampling, spec, synthetic  # noqa: E402
from oracle import gcd_oracle as O  # noqa: E402


def maxrel(a, b):
    return ((a - b).abs().max() / b.abs().max()).item()


# ------------------------------------------------------------------------------------------- oracle vs reference goldens
def test_closed_forms_bit_exact():
    g = torch.load(os.path.join(GOLD, "closed_forms.pt"))
    for n in (25, 50):
        assert torch.equal(O.edm_sigmas(n), g[f"sigmas_{n}"])
        assert torch.equal(sampling.EDMDiscretization(sigma_max=700.0)(n, device="cpu"), g[f"sigmas_{n}"])
    assert abs(g["sigmas_25"][0].item() - 700.0001) < 1e-3 and g["sigmas_25"][-1].item() == 0.0
    assert torch.equal(O.guider_scale(14, 1.5), g["scale_1.5"]) and torch.equal(O.guider_scale(14, 2.5), g["scale_2.5"])
    assert torch.equal(sampling.LinearPredictionGuider(1.5, 14, 1.0).scale, g["scale_1.5"])
    assert torch.equal(O.timestep_embedding(g["temb_t"], 320), g["temb_320"])


def test_oracle_unet_and_sampler_vs_reference_golden():
    gold = torch.load(os.path.join(GOLD, "unet_tiny.pt"))
    cfg, B, T, H, W = gold["cfg"], gold["B"], gold["T"], gold["H"], gold["W"]
    sd = synthetic.seeded_state(spec.unet_param_shapes(cfg), seed=0)
    x, c, uc, ioi = synthetic.seeded_inputs(cfg, B, T, H, W)
    net = lambda xin, t, ctx, y, **kw: O.unet_forward(sd, cfg, xin, t, ctx, y, kw["num_video_frames"], kw["image_only_indicator"])
    extra = dict(image_only_indicator=ioi, num_video_frames=T)
    c_cat = {k: torch.cat((uc[k], c[k]), 0) for k in c}
    with torch.no_grad():
        den = O.denoise(net, torch.cat([x, x]) * gold["x_mul"], torch.full((2 * B * T,), gold["sigma"]), c_cat, **extra)
        samp = O.euler_edm_sample(net, x.clone(), c, uc, gold["steps"], T, 1.5, 1.0, **extra)
    assert maxrel(den, gold["denoised"]) < 2e-5
    assert maxrel(samp, gold["sampled"]) < 2e-4


def test_oracle_decoder_vs_reference_golden():
    gold = torch.load(os.path.join(GOLD, "vae_tiny.pt"))
    cfg = gold["cfg"]
    sd = synthetic.seeded_state(spec.decoder_param_shapes(cfg), seed=0)
    g = torch.Generator().manual_seed(gold["z_seed"])
    z = torch.randn(gold["T"], cfg["z_channels"], gold["H"], gold["W"], generator=g)
    with torch.no_grad():
        out = O.decode_first_stage(sd, cfg, z, gold["T"])
    assert maxrel(out, gold["decoded"]) < 2e-5


def test_oracle_encoder_vs_reference_golden():
    """SURVEY.md §8(f) rank 1: Encoder moments and the scaled mode (quant_conv + DiagonalGaussian.mode) vs the reference."""
    gold = torch.load(os.path.join(GOLD, "enc_tiny.pt"))
    cfg = gold["cfg"]
    sd = synthetic.seeded_state(spec.encoder_param_shapes(cfg), seed=0)
    with torch.no_grad():
        assert maxrel(O.encoder_forward(sd, cfg, gold["x"]), gold["moments"]) < 2e-5
        assert maxrel(O.encode_cond_frames(sd, cfg, gold["x"], gold["quant_w"], gold["quant_b"]), gold["mode_scaled"]) < 2e-5


def test_oracle_embedders_vs_reference_golden():
    """ConcatTimestepEmbedderND / SphericalEmbedder restatements vs outputs of the reference's own classes."""
    gold = torch.load(os.path.join(GOLD, "embedders.pt"))
    assert torch.equal(O.concat_timestep_embedder_nd(gold["concat_x1"], 256), gold["concat_y1"])
    assert torch.equal(O.concat_timestep_embedder_nd(gold["concat_x2"], 256), gold["concat_y2"])
    assert maxrel(O.spherical_embedder(gold["sph_w"], gold["sph_b"], gold["sph_x"]), gold["sph_y"]) < 1e-6
    from gcd_b200.embedders import ConcatTimestepEmbedderND, SphericalEmbedder
    with pytest.raises(RuntimeError):
        ConcatTimestepEmbedderND(256)(gold["concat_x1"])           # CPU tensor: no CPU path
    with pytest.raises(RuntimeError):
        SphericalEmbedder(128)(gold["sph_x"])
    assert list(SphericalEmbedder(128).state_dict().keys()) == ["proj.weight", "proj.bias"]


def test_len1_cross_attention_is_a_bias():
    """SURVEY.md §8(a) fact 1: with one context token attn2(x, ctx) == to_out(to_v(ctx)), independent of x."""
    torch.manual_seed(0)
    C, ctxd = 128, 1024
    sd = {"a.to_q.weight": torch.randn(C, C), "a.to_k.weight": torch.randn(C, ctxd), "a.to_v.weight": torch.randn(C, ctxd),
          "a.to_out.0.weight": torch.randn(C, C), "a.to_out.0.bias": torch.randn(C)}
    x, ctx = torch.randn(3, 17, C), torch.randn(3, 1, ctxd)
    full = O.attention(sd, "a", x, ctx, heads=2)
    vec = torch.nn.functional.linear(torch.nn.functional.linear(ctx, sd["a.to_v.weight"]), sd["a.to_out.0.weight"], sd["a.to_out.0.bias"])
    assert torch.allclose(full, vec.expand_as(full), atol=1e-4, rtol=1e-4)


# ------------------------------------------------------------------------------------------- host-side sampler classes
def test_generic_sampler_matches_oracle_with_fake_network():
    T, B, H, W = 3, 2, 4, 4
    torch.manual_seed(0)
    x = torch.randn(B * T, 4, H, W)
    c = {"vector": torch.randn(B * T, 8), "crossattn": torch.randn(B * T, 1, 16), "concat": torch.randn(B * T, 4, H, W)}
    uc = {"vector": c["vector"].clone(), "crossattn": torch.zeros_like(c["crossattn"]), "concat": torch.zeros_like(c["concat"])}

    class Net(torch.nn.Module):   # any network obeying the VideoUNet call contract
        def forward(self, x, timesteps=None, context=None, y=None, **kw):
            return torch.tanh(x[:, :4] * 0.5 + x[:, 4:] * 0.1 + timesteps.view(-1, 1, 1, 1) + context.mean() + y.mean())

    net = Net()
    den = sampling.Denoiser({"target": "gcd_b200.sampling.VScalingWithEDMcNoise"})
    model = sampling.OpenAIWrapper(net)
    sampler = sampling.EulerEDMSampler(
        {"target": "sgm.modules.diffusionmodules.discretizer.EDMDiscretization", "params": {"sigma_max": 700.0}},  # alias
        num_steps=6, guider_config={"target": "gcd_b200.sampling.LinearPredictionGuider",
                                    "params": {"num_frames": T, "max_scale": 2.5, "min_scale": 1.0}}, device="cpu")
    out = sampler(lambda i, s, cc: den(model, i, s, cc, num_video_frames=T), x.clone(), cond=c, uc=uc)
    assert sampler.last_path == "generic"
    ref = O.euler_edm_sample(lambda xin, t, ctx, y, **kw: net(xin, timesteps=t, context=ctx, y=y), x.clone(), c, uc, 6, T, 2.5, 1.0)
    assert torch.allclose(out, ref, atol=1e-5, rtol=1e-5)
    # last Euler step lands exactly on the denoised sample (sigma_next = 0), sampling.py:86-87
    assert sampler.discretization(6)[-1] == 0


def test_unsupported_options_fail_loudly():
    from gcd_b200.unet import VideoUNet
    kw = spec.unet_ctor_kwargs(spec.UNET_TINY)
    with pytest.raises(NotImplementedError):
        VideoUNet(**dict(kw, num_head_channels=32))
    with pytest.raises(NotImplementedError):
        VideoUNet(**dict(kw, merge_strategy="fixed"))
    net = VideoUNet(**kw)
    with pytest.raises(RuntimeError):   # no CPU fallback
        net(torch.zeros(2, 8, 8, 8), torch.zeros(2), context=torch.zeros(2, 1, 1024), y=torch.zeros(2, 896), num_video_frames=2)


def test_encoder_rejects_unsupported_options_and_cpu_tensors():
    from gcd_b200.vae import Encoder
    kw = spec.encoder_ctor_kwargs(spec.VAE_ENCODER_TINY)
    with pytest.raises(NotImplementedError):
        Encoder(**dict(kw, attn_resolutions=[32]))
    with pytest.raises(NotImplementedError):
        Encoder(**dict(kw, resamp_with_conv=False))
    with pytest.raises(RuntimeError):
        Encoder(**kw)(torch.zeros(1, 3, 64, 64))


def test_flop_model_matches_survey():
    u = flops.unet_forward_flops(spec.UNET_KUBRIC, 28, 72, 128)
    v = flops.decoder_flops(spec.VAE_DECODER, 14, 72, 128)
    assert abs(u / 1e12 - 86.160) < 0.01 and abs(v / 1e12 - 97.202) < 0.01
    assert abs(flops.clip_flops(spec.UNET_KUBRIC, spec.VAE_DECODER, 14, 72, 128, 25) / 14e12 - 160.8) < 0.05


# ------------------------------------------------------------------------------------------- C ABI
def test_c_abi_exports_every_declared_symbol():
    from gcd_b200 import _lib, build
    build.build()                                  # cross-compiles for sm_100a; no GPU needed
    hdr = open(os.path.join(ROOT, "include", "gcd_b200.h")).read()
    declared = set(re.findall(r"\b(gcd_[a-z0-9_]+)\s*\(", hdr))
    lib = _lib.load()
    assert declared == set(_lib.EXPORTS), declared ^ set(_lib.EXPORTS)
    for name in declared:
        assert getattr(lib, name) is not None
    assert lib.gcd_version() >= 100 and lib.gcd_act_dtype() in (0, 1)


# ------------------------------------------------------------------------------------------- multi-process (gloo, 2 ranks)
def _worker(rank, world, port, q):
    import torch.distributed as dist
    from gcd_b200.pipeline import gather_clips, shard_clips
    dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world)
    num_clips = 5
    mine = shard_clips(num_clips, rank, world)
    local = [torch.full((14, 4, 2, 2), float(i)) for i in mine]
    out = gather_clips(local, num_clips, rank, world)
    ok = all(bool((out[i] == float(i)).all()) for i in range(num_clips))
    q.put((rank, mine, ok))
    dist.destroy_process_group()


def test_clip_sharding_and_gather_world2_gloo():
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29500 + os.getpid() % 500
    ps = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    [p.start() for p in ps]
    res = sorted(q.get(timeout=120) for _ in ps)
    [p.join(timeout=60) for p in ps]
    assert res[0][1] == [0, 2, 4] and res[1][1] == [1, 3] and all(r[2] for r in res)


# ---- cfg-parallel (one clip over two ranks): host logic with a stand-in engine and torch versions of the two step kernels
class _FakePool:
    def __init__(self):
        self.b = {}

    def get(self, name, shape, dtype):
        k = (name, tuple(shape), dtype)
        if k not in self.b:
            self.b[k] = torch.zeros(*shape, dtype=dtype)
        return self.b[k]


class _FakeEngine:
    """forward_cl depends on every routed input (its batch slice of x_cl, ctx, y, t) so a mis-routed half is detected."""
    AD = torch.float32

    def __init__(self):
        self.pool = _FakePool()

    def cross_attn_vectors(self, ctx, T, static=False):
        return ctx[:, 0, :4].clone()

    def forward_graphed(self, x_cl, n, H, W, t_in, ctx, y, T, ca):        # the engine replays a CUDA graph of forward_cl
        return self.forward_cl(x_cl, n, H, W, t_in, ctx, y, T, ca=ca)

    def forward_cl(self, x_cl, n, H, W, t_in, ctx, y, T, ca=None):
        res = torch.zeros(n * H * W, 16)
        v = x_cl[..., :4] * 0.5 - x_cl[..., 4:8] * 0.25 + (ca[:, None, None, :] + y[:, None, None, :4]) * t_in.view(-1, 1, 1, 1) * 0.01
        res[:, :4] = torch.tanh(v).reshape(n * H * W, 4)
        return res


class _FakeOps:
    @staticmethod
    def sampler_prep(x, ucc, cc, BT, H, W, c_in, x_cl):                      # elem.cu sampler_prep_kernel
        xs = (x * c_in).permute(0, 2, 3, 1)
        x_cl.zero_()
        x_cl[:BT, ..., :4], x_cl[BT:, ..., :4] = xs, xs
        x_cl[:BT, ..., 4:8], x_cl[BT:, ..., 4:8] = ucc.permute(0, 2, 3, 1), cc.permute(0, 2, 3, 1)

    @staticmethod
    def sampler_update(x, net, ld, BT, T, H, W, c_out, c_skip, sigma, dt, scale):   # elem.cu sampler_update_kernel
        n4 = net.view(2 * BT, H, W, ld)[..., :4].permute(0, 3, 1, 2)
        den = n4 * c_out + torch.cat([x, x]) * c_skip
        du, dc = den[:BT], den[BT:]
        d = du + scale.repeat(BT // T).view(BT, 1, 1, 1) * (dc - du)
        x += dt * (x - d) / sigma


def _cfg_case():
    g = torch.Generator().manual_seed(11)
    BT, T, H, W = 4, 2, 3, 5
    r = lambda *s: torch.randn(*s, generator=g)
    steps = 3
    host = [[3.0, 2.0, 1.0], [0.3, 0.4, 0.5], [-0.9, -0.8, -0.7], [0.3, 0.45, 0.7], [-1.0, -1.0, -1.0]]
    return dict(BT=BT, T=T, H=H, W=W, x=r(BT, 4, H, W), ucc=r(BT, 4, H, W), cc=r(BT, 4, H, W), ctx=r(2 * BT, 1, 8),
                y=r(2 * BT, 6), scale=torch.tensor([1.0, 1.5]), host=host, c_noise=r(steps))


def _cfg_run(group):
    from gcd_b200 import sampling
    k = _cfg_case()
    eng = _FakeEngine()
    smp = sampling.EulerEDMSampler.__new__(sampling.EulerEDMSampler)
    smp.cfg_group = group
    x = k["x"].clone()
    x_cl = torch.zeros(2 * k["BT"], k["H"], k["W"], 64)
    t_in = torch.zeros(2 * k["BT"])
    old = sampling.ops
    sampling.ops = _FakeOps
    try:
        if group is not None:
            return smp._run_fused_cfg_parallel(eng, x, k["ucc"], k["cc"], k["ctx"], k["y"], k["scale"], k["host"], k["c_noise"],
                                               x_cl, t_in, k["T"])
        ca = eng.cross_attn_vectors(k["ctx"], k["T"])                      # the single-process loop of _run_fused
        for i in range(3):
            _FakeOps.sampler_prep(x, k["ucc"], k["cc"], k["BT"], k["H"], k["W"], k["host"][3][i], x_cl)
            t_in.copy_(k["c_noise"][i].expand(2 * k["BT"]))
            res = eng.forward_cl(x_cl, 2 * k["BT"], k["H"], k["W"], t_in, k["ctx"], k["y"], k["T"], ca=ca)
            _FakeOps.sampler_update(x, res, 16, k["BT"], k["T"], k["H"], k["W"], k["host"][2][i], k["host"][1][i], k["host"][0][i],
                                    k["host"][4][i], k["scale"])
        return x
    finally:
        sampling.ops = old


def _cfg_worker(rank, world, port, q):
    import torch.distributed as dist
    dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world)
    out = _cfg_run(dist.new_group([0, 1]))
    q.put((rank, out))
    dist.destroy_process_group()


def test_cfg_parallel_world2_gloo_equals_single_process():
    """SURVEY.md §8(f) rank 2: rank 0 = unconditional half, rank 1 = conditional half, one all_gather per step."""
    import torch.multiprocessing as mp
    ref = _cfg_run(None)
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 30100 + os.getpid() % 500
    ps = [ctx.Process(target=_cfg_worker, args=(r, 2, port, q)) for r in range(2)]
    [p.start() for p in ps]
    res = dict(q.get(timeout=120) for _ in ps)
    [p.join(timeout=60) for p in ps]
    assert torch.equal(res[0], res[1])
    assert torch.allclose(res[0], ref, rtol=0, atol=1e-6)
    from gcd_b200 import sampling
    with pytest.raises(ValueError):
        class G: pass
        import torch.distributed as dist
        orig = dist.get_world_size
        dist.get_world_size = lambda g=None: 3
        try:
            sampling.EulerEDMSampler.set_cfg_parallel(sampling.EulerEDMSampler.__new__(sampling.EulerEDMSampler), G())
        finally:
            dist.get_world_size = orig


# ------------------------------------------------------------------------------------------- bench.py contract (CPU legs)
def test_bench_reference_arm_json_contract_and_no_cpu_fallback():
    """`bench.py --impl reference` (the CPU port timed on the host cores) prints one JSON line with the contract's keys;
    the product arm refuses to run without a CUDA device instead of falling back to the CPU."""
    import json
    import subprocess
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    # the reduced-width self-test workload keeps this to seconds (the full one builds 1.5 B seeded weights on the host first)
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                        "--workload", "tiny-selftest"], capture_output=True, text=True, timeout=900, env=env)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in line, k
    assert line["impl"] == "reference" and line["metric"] == "latent-frames/sec" and line["value"] > 0
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["d2h_bytes_per_step"] == 0
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "0"],
                       capture_output=True, text=True, timeout=600, env=env)
    assert r.returncode != 0 and "no CPU fallback" in (r.stderr + r.stdout)


def test_bench_cpu_leg_falls_back_to_a_bounded_sample_when_the_full_size_one_cannot_run():
    """The CPU-oracle leg runs in a child process with a time limit; if it cannot finish (host memory limit, slow host) bench.py
    times a bounded sample instead, scales it by the algorithmic-FLOP ratios and says so — it never takes the bench line down."""
    import json
    import subprocess
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="", GCD_CPU_LEG_TIMEOUT="1")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                        "--workload", "tiny-selftest"], capture_output=True, text=True, timeout=900, env=env)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])
    assert line["impl"] == "reference" and line["value"] > 0
    assert "FULL-SIZE SAMPLE UNAVAILABLE" in line["cpu_baseline"]["sample"] and "exceeded 1 s" in line["cpu_baseline"]["sample"]


# ------------------------------------------------------------------------------------------- weight (re)load / EMA swap
def test_engine_key_sees_data_copy_and_litema_shadows_every_parameter():
    """ADVICE r1: `param.data.copy_` (what the reference's LitEma.copy_to / restore do, modules/ema.py) does not bump
    `_version`; the engine cache key must still change, and LitEma must find parameters to shadow (requires_grad)."""
    from gcd_b200.unet import VideoUNet, weights_key
    net = VideoUNet(**spec.unet_ctor_kwargs(spec.UNET_TINY))
    net.load_state_dict(synthetic.seeded_state(spec.unet_param_shapes(spec.UNET_TINY), seed=0))
    k0 = weights_key(net, "cpu")
    assert weights_key(net, "cpu") == k0
    other = synthetic.seeded_state(spec.unet_param_shapes(spec.UNET_TINY), seed=5)
    with torch.no_grad():
        for name, p in net.named_parameters():
            v = p._version
            p.data.copy_(other[name])
            assert p._version == v                      # the blind spot the content probe covers
    assert weights_key(net, "cpu") != k0
    n_params = sum(1 for _ in net.parameters())
    assert all(p.requires_grad for p in net.parameters())
    # the parameters the reference's LitEma shadowed in this network (tests/golden/host_api.json, recorded from
    # LitEma(HotPathRoot.model) by oracle/pin_against_reference.py): every weight has a shadow => `model_ema.*` keys load
    shadows = json.load(open(os.path.join(GOLD, "host_api.json")))["litema_shadows_of_model"]
    mine = {"diffusion_model." + name for name, p in net.named_parameters() if p.requires_grad}
    assert set(shadows) == mine and len(shadows) == n_params
    # ema_scope (models/diffusion.py): LitEma.store clones the weights, copy_to and restore write through `param.data.copy_`
    k1 = weights_key(net, "cpu")
    stored = [p.detach().clone() for p in net.parameters()]
    with torch.no_grad():
        for p in net.parameters():
            p.data.copy_(p.data * 0.5)
    assert weights_key(net, "cpu") != k1
    with torch.no_grad():
        for p, s in zip(net.parameters(), stored):
            p.data.copy_(s)
    assert weights_key(net, "cpu") == k1


def test_embedders_pass_the_general_conditioner_gate():
    """ADVICE r1: GeneralConditioner asserts isinstance(embedder, AbstractEmbModel) (encoders/modules.py:93-96). What the
    reference's own classes made of the repo's embedders is recorded in tests/golden/host_api.json: the properties of
    AbstractEmbModel with their defaults, and each embedder's state after GeneralConditioner accepted it. Standalone the
    embedders carry the same properties; with an `sgm.modules.encoders.modules` importable they derive from its
    AbstractEmbModel (a stand-in class here) and take the conditioner's settings to the recorded state."""
    import importlib
    import types
    import torch.nn as nn
    from gcd_b200.sampling import instantiate_from_config
    gold = json.load(open(os.path.join(GOLD, "host_api.json")))
    import gcd_b200.embedders as E
    for cls, args in ((E.ConcatTimestepEmbedderND, (256,)), (E.SphericalEmbedder, (128,))):
        emb = cls(*args)
        assert {k: getattr(emb, k) for k in gold["abstract_emb_model"]} == gold["abstract_emb_model"]

    class AbstractEmbModel(nn.Module):
        def __init__(self):
            super().__init__()
            for k, v in gold["abstract_emb_model"].items():
                setattr(self, k, v)

    fake = types.ModuleType("sgm.modules.encoders.modules")
    fake.AbstractEmbModel = AbstractEmbModel
    pkg = types.ModuleType("sgm.modules.encoders")
    pkg.__path__ = []
    saved = {k: sys.modules.get(k) for k in ("sgm.modules.encoders", "sgm.modules.encoders.modules")}
    sys.modules["sgm.modules.encoders"], sys.modules["sgm.modules.encoders.modules"] = pkg, fake
    try:
        E = importlib.reload(E)
        assert issubclass(E.ConcatTimestepEmbedderND, AbstractEmbModel) and issubclass(E.SphericalEmbedder, AbstractEmbModel)
        for rec in gold["general_conditioner"]:
            cfg = rec["config"]
            emb = instantiate_from_config(cfg)
            assert isinstance(emb, AbstractEmbModel) and type(emb).__name__ == rec["class"]
            emb.is_trainable, emb.ucg_rate = cfg.get("is_trainable", False), cfg.get("ucg_rate", 0.0)
            emb.input_key, emb.legacy_ucg_val = cfg["input_key"], cfg.get("legacy_ucg_value", None)
            for p in emb.parameters():
                p.requires_grad = False
            got = {"input_key": emb.input_key, "ucg_rate": emb.ucg_rate, "is_trainable": emb.is_trainable,
                   "legacy_ucg_val": emb.legacy_ucg_val, "requires_grad": [p.requires_grad for p in emb.parameters()]}
            assert got == {k: rec[k] for k in got}, (got, rec)
    finally:
        for k, v in saved.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v
        importlib.reload(E)


def test_stats_arena_slots_and_growth():
    """GroupNorm statistics arena (unet.StatsArena): one memset per forward, one slot per producer, slot size follows the batch."""
    from gcd_b200 import unet as U

    class Pool:
        def __init__(self):
            self.bufs = {}

        def get(self, name, shape, dtype):
            return self.bufs.setdefault((name, tuple(shape), dtype), torch.zeros(shape, dtype=dtype))

    zeroed = []
    orig = U.ops.zero_tensor
    U.ops.zero_tensor = lambda t: (zeroed.append(t.numel()), t.zero_())
    try:
        a = U.StatsArena(Pool())
        a.reset(28)
        s0, s1 = a.take(28), a.take(2)
        assert s0.numel() == s1.numel() == 64 * 64 and s0.data_ptr() != s1.data_ptr() and zeroed == [U.StatsArena.SLOTS * 4096]
        s0[:10] = 1.0
        a.reset(28)                                            # next forward: same storage, zeroed again by ONE memset
        assert a.take(28).data_ptr() == s0.data_ptr() and float(s0.sum()) == 0.0 and len(zeroed) == 2
        a.reset(200)                                           # bigger batch -> bigger slots
        assert a.take(200).numel() == 200 * 64
        with pytest.raises(AssertionError):
            a.take(500)
    finally:
        U.ops.zero_tensor = orig
