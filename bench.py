#!/usr/bin/env python
"""bench.py — latent-frames/sec through the full GCD denoising hot path on B200.

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--workload kubric|pardom|direct50] [--dump-outputs DIR]

A "step" = one pass of the hot path over one batch: per GPU ONE clip of 14 latent frames, 72x128 (576x1024 px):
25 EDM/Euler steps of the CFG-doubled SVD VideoUNet (28 frames per forward) + the temporal VAE decode of the 14 frames
(BASELINE.json configs[1]; `direct50` = configs[3]: 50 steps, guider max scale 2.5). Clips are independent, so N GPUs run
N clips (weak scaling) with one NCCL all_gather of the sampled latents per step. Synthetic inputs, seeded random weights
(no checkpoints offline; zero-init tensors overwritten — gcd_b200/synthetic.py).

JSON line (rank 0): `value` = whole-job latent-frames/s with inputs resident in HBM (CUDA-event timed, max over ranks);
`e2e` = same metric through the public API gcd_b200.pipeline.GCDHotPath.sample_video with pinned HOST inputs and a
device->host read of the decoded frames inside the timed region; `roofline` = tensor-core roofline of the dominant kernel
class (tc_gemm implicit-GEMM conv/linear) from CUDA events on the launching stream + whole-path fraction; `cpu_baseline` =
the CPU oracle port (oracle/gcd_oracle.py) timed on this box's host cores on a bounded sample.
`--impl reference` times only that CPU port (the reference's own PyTorch code cannot travel to the GPU box).
`--dump-outputs DIR` writes what the last timed step returned (rank 0) as float32 .npy files, for comparing two builds on
identical seeded inputs: latents.npy [14, 4, h, w]; frames.npy, or frames_sample.npy (a fixed seeded sample of 2^23
values of the flattened [14, 3, 8h, 8w] frames) when the frames exceed that; latents_gathered.npy [N, 14, 4, h, w] with N > 1.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import torch

sys.dont_write_bytecode = True       # the tree may be read-only; nothing is cached next to the sources
ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

T_FRAMES, LAT_H, LAT_W = 14, 72, 128
WORKLOADS = {
    "kubric": dict(unet="UNET_KUBRIC", steps=25, max_scale=1.5, name="Kubric-4D gradual max90, 25-step Euler sample, 14x72x128 latent (576x1024 px)"),
    "pardom": dict(unet="UNET_PARDOM", steps=25, max_scale=1.5, name="ParallelDomain-4D gradual RGB, 25-step sample, 14x72x128 latent"),
    "direct50": dict(unet="UNET_KUBRIC", steps=50, max_scale=2.5, name="Kubric-4D direct max180, CFG 2.5, 50-step sample, 14x72x128 latent"),
    # reduced-width network: only for tests of this script's plumbing (tests/test_host_cpu.py), never a reported number
    "tiny-selftest": dict(unet="UNET_TINY", vae="VAE_TINY", steps=25, max_scale=1.5, latent=(16, 24),
                          name="SELF-TEST ONLY: width-64 network at latent 16x24, not a benchmark"),
}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(tflops=d["bf16_tflops_sustained"], burst=d["bf16_tflops"], hbm=d["hbm_gbs"], src="measured (MEASURED_PEAKS.json, sustained bf16)")
    return dict(tflops=1400.0, burst=1590.0, hbm=6650.0, src="fallback (B200_PROFILING.md)")


class ClockSampler:
    """nvidia-smi clock / throttle-reason samples during the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200",
                                       "-i", str(index)], stdout=self.f, stderr=subprocess.DEVNULL)
        except OSError:
            self.p = None

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        rows = [l.strip().split(", ") for l in self.f.read().strip().splitlines() if l.strip()]
        rows = [r for r in rows if len(r) == 6 and r[0].isdigit()]
        os.unlink(self.f.name)
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        sm = sorted(int(r[0]) for r in rows)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(r[2 + i].strip() == "Active" for r in rows)]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": int(rows[0][1]), "reasons": reasons, "samples": len(rows)}


# ------------------------------------------------------------------------------------------------------ CPU oracle leg
_CPU_CACHE = {}


def _cpu_leg_worker(spec_json):
    """Child process of cpu_oracle_sample (python bench.py --cpu-leg '<json>'): times the CPU oracle and prints one JSON line.
    Runs in its own process so that a host-memory limit or a timeout on the GPU box cannot take the bench line down with it."""
    from gcd_b200 import flops, spec, synthetic
    from oracle import gcd_oracle as O
    a = json.loads(spec_json)
    unet_cfg, vae_cfg, (h, w), (vh, vw) = a["unet_cfg"], a["vae_cfg"], a["lat_hw"], a["vae_hw"]
    # Measured on the pool's 128-vCPU B200 hosts (tools/cpu_threads.py, same UNet sample): 16 threads 1.9 s, 32 threads
    # 2.1 s, 64 threads 3.9 s, 128 threads 121 s (the cgroup quota is far below 128 cores) -> use the fastest setting.
    cores = min(os.cpu_count() or 1, 32)
    torch.set_num_threads(cores)
    unet_state = synthetic.seeded_state(spec.unet_param_shapes(unet_cfg), seed=0)
    vae_state = synthetic.seeded_state(spec.decoder_param_shapes(vae_cfg), seed=0)
    n = 2 * T_FRAMES

    def inputs(hh, ww):
        x, c, uc, ioi = synthetic.seeded_inputs(unet_cfg, 1, T_FRAMES, hh, ww)
        xin = torch.cat((torch.cat([x, x]), torch.cat((uc["concat"], c["concat"]))), 1)
        return xin, torch.cat((uc["crossattn"], c["crossattn"])), torch.cat((uc["vector"], c["vector"])), ioi

    t = torch.full((n,), 0.5756)
    with torch.no_grad():
        xin, ctx, y, ioi = inputs(8, 8)                                        # warm-up, untimed
        O.unet_forward(unet_state, unet_cfg, xin, t, ctx, y, T_FRAMES, ioi)
        O.decode_first_stage(vae_state, vae_cfg, torch.randn(T_FRAMES, 4, 8, 8), T_FRAMES)
        xin, ctx, y, ioi = inputs(h, w)
        t0 = time.perf_counter()
        O.unet_forward(unet_state, unet_cfg, xin, t, ctx, y, T_FRAMES, ioi)
        tu = time.perf_counter() - t0
        del xin
        z = torch.randn(T_FRAMES, 4, vh, vw)
        t0 = time.perf_counter()
        O.decode_first_stage(vae_state, vae_cfg, z, T_FRAMES)
        tv = time.perf_counter() - t0
    print(json.dumps({"cpu_leg": True, "tu": tu, "tv": tv, "cores": cores}), flush=True)


def _run_cpu_leg(unet_cfg, vae_cfg, lat_hw, vae_hw, timeout):
    arg = json.dumps({"unet_cfg": unet_cfg, "vae_cfg": vae_cfg, "lat_hw": list(lat_hw), "vae_hw": list(vae_hw)})
    env = dict(os.environ)
    for k in ("RANK", "LOCAL_RANK", "WORLD_SIZE", "MASTER_ADDR", "MASTER_PORT", "OMP_NUM_THREADS"):
        env.pop(k, None)                      # torchrun pins OMP_NUM_THREADS=1 for its workers
    env["CUDA_VISIBLE_DEVICES"] = ""
    try:
        r = subprocess.run([sys.executable, os.path.abspath(__file__), "--cpu-leg", arg], capture_output=True, text=True,
                           timeout=timeout, env=env)
        for line in r.stdout.splitlines():
            if line.startswith("{") and "cpu_leg" in line:
                return json.loads(line), None
        return None, f"CPU leg exited {r.returncode}: {r.stderr.strip()[-200:]}"
    except subprocess.TimeoutExpired:
        return None, f"CPU leg exceeded {timeout} s"


def cpu_oracle_sample(unet_cfg, vae_cfg, steps, lat_hw=(LAT_H, LAT_W)):
    """Times the CPU oracle port (restatement of the reference's PyTorch path, oracle/gcd_oracle.py) on THIS workload's own
    shapes: ONE CFG UNet forward (28 frames at `lat_hw` = 72x128) and ONE VAE decode of the 14 frames at that size, fp32, after a
    small warm-up call (thread pool / allocator). One clip = `steps` such forwards + one decode; every sampler step runs the
    identical network on identically shaped inputs, so clip time = steps x t_forward + t_decode ("extrapolated from 1 step":
    a full 25-step clip is ~1 h of host time). The same routine serves `cpu_baseline` and `--impl reference`, so the two legs
    agree by construction. The measurement runs in a child process with a time limit (GCD_CPU_LEG_TIMEOUT, default 900 s; the full-size sample takes ~5 min on the pool's hosts);
    if the full-size sample cannot run on this host (memory limit, time), a bounded sample (latent 16x24 / decode 8x8) is timed
    instead and scaled by the exact algorithmic-FLOP ratios — and labelled as such.
    Returns (latent_frames_per_s, description, cores, seconds_measured)."""
    from gcd_b200 import flops
    key = (tuple(sorted((k, str(v)) for k, v in unet_cfg.items())), tuple(sorted((k, str(v)) for k, v in vae_cfg.items())), steps, lat_hw)
    if key in _CPU_CACHE:
        return _CPU_CACHE[key]
    h, w = lat_hw
    tmo = int(os.environ.get("GCD_CPU_LEG_TIMEOUT", "900"))
    res, err = _run_cpu_leg(unet_cfg, vae_cfg, (h, w), (h, w), tmo)
    if res is not None:
        tu, tv, cores = res["tu"], res["tv"], res["cores"]
        desc = (f"1 CFG UNet forward (28 frames, latent {h}x{w}: {tu:.1f} s) + 1 VAE decode of 14 frames at latent {h}x{w} "
                f"({tv:.1f} s), fp32, {cores} threads, measured once after a small warm-up call; clip = {steps} x forward + decode "
                f"(extrapolated from 1 step: the steps are identical network calls)")
        full_s = steps * tu + tv
    else:
        sh, sw = min(h, 16), min(w, 24)
        res, err2 = _run_cpu_leg(unet_cfg, vae_cfg, (sh, sw), (8, 8), 600)
        if res is None:
            out = (None, f"CPU oracle could not be timed on this host ({err}; bounded sample: {err2})", 0, 0.0)
            _CPU_CACHE[key] = out
            return out
        tu, tv, cores = res["tu"], res["tv"], res["cores"]
        n = 2 * T_FRAMES
        ru = flops.unet_forward_flops(unet_cfg, n, h, w) / flops.unet_forward_flops(unet_cfg, n, sh, sw)
        rv = flops.decoder_flops(vae_cfg, T_FRAMES, h, w) / flops.decoder_flops(vae_cfg, T_FRAMES, 8, 8)
        full_s = steps * tu * ru + tv * rv
        desc = (f"FULL-SIZE SAMPLE UNAVAILABLE ({err}); bounded sample instead: 1 CFG UNet forward at latent {sh}x{sw} ({tu:.2f} s) "
                f"+ 1 VAE decode at latent 8x8 ({tv:.2f} s), fp32, {cores} threads, scaled to {steps} steps at {h}x{w} by "
                f"algorithmic FLOP ratios x{ru:.1f} / x{rv:.1f}")
    _CPU_CACHE[key] = (T_FRAMES / full_s, desc, cores, tu + tv)
    return _CPU_CACHE[key]


def run_reference(args, wl):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from gcd_b200 import spec
    unet_cfg, vae_cfg = getattr(spec, wl["unet"]), getattr(spec, wl.get("vae", "VAE_DECODER"))
    lat = tuple(wl.get("latent", (LAT_H, LAT_W)))
    # measured once (one full-size forward + decode is minutes of host time) and reused for every --warmup/--steps iteration
    v, desc, cores, secs = cpu_oracle_sample(unet_cfg, vae_cfg, wl["steps"], lat_hw=lat)
    if v is None:
        print(json.dumps({"impl": "reference", "unavailable": desc}), flush=True)
        return
    line = {"impl": "reference", "metric": "latent-frames/sec", "value": v, "unit": "latent-frames/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * T_FRAMES / v, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic (seeded random weights, random latents/conditioning)",
            "config": {"workload": wl["name"], "latent": [T_FRAMES, 4, lat[0], lat[1]], "sampler_steps": wl["steps"],
                       "measured_once": True,
                       "impl_note": "CPU port of the reference PyTorch path (oracle/gcd_oracle.py) at the workload's own shapes; "
                                    "the reference itself is pure Python under /root/reference and cannot travel to the GPU box"},
            "cpu_baseline": {"value": v, "unit": "latent-frames/s", "cores": cores, "kind": "port", "sample": desc},
            "e2e": {"value": v, "unit": "latent-frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------------ extra workloads
def run_extra_workloads(args, wl, pipe, ust, dev, rank, world, lat, timed, gathered):
    """BASELINE.json configs 3 and 4 and the single-clip latency mode, measured in the same process right after the main
    line so the driver's N = 1/2/4/8 runs record them (one clip per rank each, CUDA events, max over ranks):
      direct50     config 4: Kubric-4D direct max180 — 50 Euler steps, guider max scale 2.5 (pretrained/*.yaml:135), + decode,
                   clips sharded one per rank + the NCCL gather of the latents;
      pardom       config 3: ParallelDomain-4D network (no auxiliary embedding), 25 steps + decode, same sharding;
      cfg_parallel N >= 2: ONE clip on ranks 0 and 1, the CFG pair split across them (EulerEDMSampler.set_cfg_parallel) —
                   ms per clip and rel-L2 of its latents vs the same clip sampled on one GPU.
    Not part of `value`. Skipped for the self-test workload and under --no-extra."""
    import torch.distributed as dist
    from gcd_b200 import spec, synthetic
    from gcd_b200.pipeline import GCDHotPath
    if wl.get("unet") != "UNET_KUBRIC" or args.workload != "kubric":
        return None
    LH, LW = lat
    out = {}

    def clip_inputs(cfg):
        x0, c, uc, _ = synthetic.seeded_inputs(cfg, 1, T_FRAMES, LH, LW, seed=4321 + rank)
        return x0.to(dev), {k: v.to(dev) for k, v in c.items()}, {k: v.to(dev) for k, v in uc.items()}

    def one_clip(p, x, c, uc):
        z = p.sample_latents(x.clone(), c, uc)
        fr = p.decode_first_stage(z)
        if world > 1:
            dist.all_gather(gathered, z.contiguous())
        return z, fr

    def measure(name, p, cfg, note):
        x, c, uc = clip_inputs(cfg)
        one_clip(p, x, c, uc)                                           # warm-up (workspaces, graph capture)
        ms = timed(lambda: one_clip(p, x, c, uc), 1)
        out[name] = {"ms_per_clip": round(ms, 1), "latent_frames_per_s": round(world * T_FRAMES / (ms / 1e3), 3),
                     "clips": world, "config": note}

    # ---- config 4: same network, 50 steps, max scale 2.5
    p50 = GCDHotPath(pipe.unet_cfg, pipe.vae_cfg, num_steps=50, num_frames=T_FRAMES, max_scale=2.5, device=dev,
                     unet=pipe.unet, decoder=pipe.decoder)              # share the loaded modules (and their packed engines)
    measure("direct50", p50, pipe.unet_cfg, WORKLOADS["direct50"]["name"])
    # ---- single-clip latency over 2 GPUs (before the ParDom network replaces nothing: it uses the Kubric modules)
    if world >= 2:
        grp = dist.new_group([0, 1])                                    # every rank must take part in group creation
        if rank < 2:
            x0, c, uc, _ = synthetic.seeded_inputs(pipe.unet_cfg, 1, T_FRAMES, LH, LW, seed=777)      # the SAME clip on both ranks
            x, c, uc = x0.to(dev), {k: v.to(dev) for k, v in c.items()}, {k: v.to(dev) for k, v in uc.items()}
            z_ref = pipe.sample_latents(x.clone(), c, uc)
            pipe.set_cfg_parallel(grp)
            pipe.sample_latents(x.clone(), c, uc)                       # warm-up
            torch.cuda.synchronize()
            dist.barrier(group=grp)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            z = pipe.sample_latents(x.clone(), c, uc)
            if rank == 0:
                pipe.decode_first_stage(z)
            e1.record()
            torch.cuda.synchronize()
            pipe.set_cfg_parallel(None)
            ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
            dist.all_reduce(ms, op=dist.ReduceOp.MAX, group=grp)
            out["cfg_parallel"] = {"ms_per_clip": round(ms.item(), 1), "gpus": 2,
                                   "rel_l2_vs_single_gpu_latents": float(((z - z_ref).norm() / z_ref.norm()).item()),
                                   "config": "one clip, CFG pair split over ranks 0/1, one NCCL all_gather of the network "
                                             "output per step; 25 steps + decode on rank 0"}
        dist.barrier()
    # ---- config 3: ParDom network = the Kubric state without the auxiliary-embedding tensors (seeded per tensor name)
    pcfg = spec.UNET_PARDOM
    shapes = spec.unet_param_shapes(pcfg)
    pst = {k: ust[k] for k in shapes} if ust is not None else synthetic.seeded_state(shapes, seed=0)
    pp = GCDHotPath(pcfg, pipe.vae_cfg, num_steps=25, num_frames=T_FRAMES, max_scale=1.5, device=dev, decoder=pipe.decoder)
    pp.unet.load_state_dict(pst, strict=True)
    pp.unet.to(dev)
    measure("pardom", pp, pcfg, WORKLOADS["pardom"]["name"])
    del pp
    return out


# ------------------------------------------------------------------------------------------------------ output dump
DUMP_FRAMES_SAMPLE = 1 << 23          # float32 values: 32 MiB of the 99 MB of frames of a 576x1024 clip
DUMP_LIMIT = 64 << 20


def dump_outputs(out_dir, z, frames, gathered):
    """Writes the arrays of one timed step as float32 .npy files (see the module docstring); at most DUMP_LIMIT bytes."""
    import numpy as np
    arrays = {"latents": z}
    if frames is not None:
        if frames.numel() <= DUMP_FRAMES_SAMPLE:
            arrays["frames"] = frames
        else:
            g = torch.Generator().manual_seed(0)
            idx = torch.randperm(frames.numel(), generator=g)[:DUMP_FRAMES_SAMPLE].sort().values
            arrays["frames_sample"] = frames.reshape(-1)[idx.to(frames.device)]
    if gathered is not None:
        arrays["latents_gathered"] = torch.stack(gathered)
    total = sum(a.numel() * 4 for a in arrays.values())
    assert total <= DUMP_LIMIT, f"--dump-outputs: {total} bytes exceed {DUMP_LIMIT}"
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a.detach().float().cpu().numpy())


def positive_int(v):
    n = int(v)
    if n < 1:
        raise argparse.ArgumentTypeError(f"must be >= 1, got {v}")
    return n


# ------------------------------------------------------------------------------------------------------ product arm
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=positive_int, default=2, help="timed steps (one clip per GPU each)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="kubric", choices=list(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-decode", action="store_true", help=argparse.SUPPRESS)
    ap.add_argument("--cpu-leg", default=None, help=argparse.SUPPRESS)
    ap.add_argument("--no-extra", action="store_true", help="skip the extra_workloads block (BASELINE configs 3/4, CFG-parallel)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the latents and frames of the last timed step (rank 0) to DIR/<name>.npy, float32")
    ap.add_argument("--profile-run", action="store_true",
                    help="for ncu: exactly --warmup/--steps resident steps, no e2e / instrumented / CPU passes, no JSON claims")
    args = ap.parse_args()
    if args.cpu_leg is not None:
        return _cpu_leg_worker(args.cpu_leg)
    wl = WORKLOADS[args.workload]
    if args.impl == "reference":
        if args.dump_outputs:
            ap.error("--dump-outputs needs the product arm: --impl reference only times the CPU port")
        return run_reference(args, wl)

    import torch.distributed as dist
    from gcd_b200 import flops, ops, spec, synthetic
    from gcd_b200.pipeline import GCDHotPath
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — the product path has no CPU fallback (use --impl reference for the CPU port)")
    ops.lib()  # fail loudly if libgcd_b200.so is missing
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        import datetime
        dist.init_process_group("nccl", device_id=dev, timeout=datetime.timedelta(seconds=1200))   # ranks build 1.5 B seeded weights on shared host cores first
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world} (launch with torch.distributed.run)"

    unet_cfg, vae_cfg = getattr(spec, wl["unet"]), getattr(spec, wl.get("vae", "VAE_DECODER"))
    pipe = GCDHotPath(unet_cfg, vae_cfg, num_steps=wl["steps"], num_frames=T_FRAMES, max_scale=wl["max_scale"], device=dev)
    ust = synthetic.seeded_state(spec.unet_param_shapes(unet_cfg), seed=0)
    vst = synthetic.seeded_state(spec.decoder_param_shapes(vae_cfg), seed=0)
    pipe.load_state(ust, vst)
    # rank r samples its own clip: seed 1234 + r (scripts/test.py:1059-1084 strides examples over workers the same way)
    LH, LW = tuple(wl.get("latent", (LAT_H, LAT_W)))
    x0, c, uc, _ = synthetic.seeded_inputs(unet_cfg, 1, T_FRAMES, LH, LW, seed=1234 + rank)
    pin = lambda t: t.pin_memory()
    hx, hc, huc = pin(x0), {k: pin(v) for k, v in c.items()}, {k: pin(v) for k, v in uc.items()}
    dx, dc, duc = x0.to(dev), {k: v.to(dev) for k, v in c.items()}, {k: v.to(dev) for k, v in uc.items()}
    h2d = sum(t.numel() * t.element_size() for t in [hx, *hc.values(), *huc.values()])
    frames_host = torch.empty(T_FRAMES, 3, LH * 8, LW * 8, dtype=torch.float32).pin_memory()
    d2h = frames_host.numel() * 4
    gathered = [torch.empty(T_FRAMES, 4, LH, LW, device=dev) for _ in range(world)] if world > 1 else None

    def step_resident(collective=True):
        z = pipe.sample_latents(dx.clone(), dc, duc)
        fr = None if args.no_decode else pipe.decode_first_stage(z)
        if world > 1 and collective:
            dist.all_gather(gathered, z.contiguous())     # the path's only collective: final gather over NVLink
        return z, fr

    last = {}

    def step_resident_kept():
        last["z"], last["frames"] = step_resident()

    def step_e2e():
        z, fr = pipe.sample_video(hx, hc, huc, decode=not args.no_decode)
        if fr is not None:
            frames_host.copy_(fr, non_blocking=True)
        if world > 1:
            dist.all_gather(gathered, z.contiguous())
        torch.cuda.current_stream().synchronize()        # the caller holds the frames on the host when the step ends
        return z

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, k):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(k):
            fn()
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return ms.item()

    if args.profile_run:
        for _ in range(args.warmup):
            step_resident()
        ms = timed(step_resident, args.steps)
        if rank == 0:
            print(json.dumps({"profile_run": True, "ms_per_step_under_profiler": ms / args.steps}))
        return
    for _ in range(max(args.warmup, 3)):
        step_resident()
    clocks = ClockSampler(local) if rank == 0 else None
    l0 = ops.launch_count()
    ms = timed(step_resident_kept, args.steps)
    launches = ops.launch_count() - l0
    clk = clocks.stop() if clocks else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last["z"], last["frames"], gathered)
    last.clear()
    step_e2e()
    ms_e2e = timed(step_e2e, args.steps)

    extra = None if args.no_extra else run_extra_workloads(args, wl, pipe, ust, dev, rank, world, (LH, LW), timed, gathered)

    frames_total = world * args.steps * T_FRAMES
    value = frames_total / (ms / 1e3)
    e2e_value = frames_total / (ms_e2e / 1e3)

    # ---- per-kernel-class roofline (one extra, untimed, instrumented step on rank 0)
    line = None
    if rank == 0:
        pk = measured_peaks()
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with ops.profile() as prof:
            g0.record()
            step_resident(collective=False)       # rank 0 only: must not enter a collective
            g1.record()
        summ = prof.summary()
        prof_wall_ms = g0.elapsed_time(g1)        # eager, per-launch events: slower than the timed (graph-replay) steps
        tc = summ.get("tc_gemm", dict(ms=1e-9, flops=0.0, launches=0))
        tot_ms = sum(d["ms"] for d in summ.values())
        tc_tflops = tc["flops"] / (tc["ms"] / 1e3) / 1e12
        per_frame = flops.clip_flops(unet_cfg, vae_cfg, T_FRAMES, LH, LW, wl["steps"]) / T_FRAMES
        path_tflops = per_frame * (value / world) / 1e12
        traffic, traffic_detail = None, None
        tp = os.path.join(ROOT, "profiles", "r2_traffic.json")
        if os.path.exists(tp):
            traffic_detail = json.load(open(tp))       # one representative tc_gemm launch from `ncu --set full`
            traffic = traffic_detail.get("dram_bytes")  # dram__bytes_read.sum + dram__bytes_write.sum of that launch
        roof = {"bound": "tensor", "kernel": "tc_gemm_kernel (tcgen05 implicit-GEMM conv / linear)",
                "achieved": round(tc_tflops, 1), "peak": pk["tflops"], "unit": "TFLOP/s", "frac": round(tc_tflops / pk["tflops"], 4),
                "traffic": traffic, "traffic_detail": traffic_detail, "peak_source": pk["src"],
                "kernel_share_of_step": round(tc["ms"] / max(tot_ms, 1e-9), 4),
                "instrumented_step": {"wall_ms": round(prof_wall_ms, 2), "class_sum_ms": round(tot_ms, 2),
                                      "gap_ms": round(prof_wall_ms - tot_ms, 2),
                                      "note": "one extra eager step with CUDA events around every launch (all kernel classes "
                                              "incl. `elem`); gap = time between kernels + torch glue; the timed steps replay the "
                                              "UNet forward from a CUDA graph"},
                "whole_path": {"algorithmic_tflop_per_latent_frame": round(per_frame / 1e12, 1),
                               "achieved": round(path_tflops, 1), "frac": round(path_tflops / pk["tflops"], 4)},
                "classes": {k: {"ms": round(d["ms"], 2), "launches": d["launches"],
                                "tflops": round(d["flops"] / max(d["ms"], 1e-9) / 1e9, 1),
                                "gbs": round(d["bytes"] / max(d["ms"], 1e-9) / 1e6, 1)} for k, d in summ.items()}}
        line = {"metric": "latent-frames/sec", "value": round(value, 4), "unit": "latent-frames/s", "n_gpus": world,
                "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": round(ms / args.steps, 2),
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "bf16" if ops.lib().gcd_act_dtype() == 1 else "f16",
                "data": "synthetic (seeded random weights of the named architecture, random latents/conditioning)",
                "config": {"workload": wl["name"], "clips_per_gpu_per_step": 1, "latent": [T_FRAMES, 4, LH, LW],
                           "sampler_steps": wl["steps"], "cfg_batch": 2 * T_FRAMES, "decode": not args.no_decode,
                           "parallelism": f"clips x{world} (one NCCL all_gather of latents per step)" if world > 1 else "single GPU",
                           "l2": "no explicit flush: per-step working set (3.2 GB fp16 weights + multi-GB activations) >> 126 MB L2",
                           "precision": "fp16 tensor-core operands, fp32 accumulate / residual stream / norms (UNet = the reference's fp16-autocast arithmetic; the VAE decode uses the same 16-bit operands where the reference decodes in fp32: 7.4e-4 rel-L2 at 576x1024)"},
                "e2e": {"value": round(e2e_value, 4), "unit": "latent-frames/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                        "ms_per_step": round(ms_e2e / args.steps, 2),
                        "api": "gcd_b200.pipeline.GCDHotPath.sample_video(pinned host noise/cond) + frames -> pinned host"},
                "gpu_launches": int(launches), "clocks": clk, "roofline": roof}
        if extra:
            line["extra_workloads"] = extra
        if world == 1 and not args.no_cpu_baseline and not args.profile_run:
            del ust, vst                   # the CPU leg runs in a child process: release the 6 GB of host weights first
            v, desc, cores, _ = cpu_oracle_sample(unet_cfg, vae_cfg, wl["steps"], lat_hw=tuple(wl.get("latent", (LAT_H, LAT_W))))
            line["cpu_baseline"] = {"value": v, "unit": "latent-frames/s", "cores": cores, "kind": "port", "sample": desc}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
