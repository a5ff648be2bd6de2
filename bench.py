#!/usr/bin/env python
"""Benchmark of the DDPO hot path on B200 (contract: see the task brief / DESIGN.md §Measurement).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--phase sample|ppo] [--dump-outputs DIR]

Workload = BASELINE.json configs[1]: DDPO, SD2-base 512 px (64x64x4 latents, 77x1024 context), 50-step
DDIM, CFG 5.0, eta 1.0, per-GPU sample batch 8 (global batch 64 on 8 GPUs), synthetic latents/prompt
embeddings, random-init U-Net weights.  One bench "step" is one pass of the hot path over one batch:
  phase=sample : one denoising step of the 8-sample batch (U-Net on the 2x8 CFG batch + fused
                 CFG/DDIM/log-prob/noise kernel)                          -> denoising steps/s
  phase=ppo    : one PPO train pass: 10 timesteps of the train batch of 2 (reference micro-batch, train_cfg) stacked
                 into one U-Net fwd+bwd of batch 40, log-prob, PPO loss (per-micro-batch means), gradient accumulate;
                 plus the optimizer update (all-reduce + clip + AdamW) timed separately  -> PPO samples/s
The headline `value` is PPO samples/s when the training path is available (a PPO sample = 50 sampling
steps + 50 train steps of one trajectory), else denoising steps/s.
One process per GPU (torchrun for N>1), max-over-ranks CUDA-event timing.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

T_STEPS = 50
SAMPLE_BATCH = 8
TRAIN_BATCH = 2
TRAIN_MACRO = int(os.environ.get("DDPO_BENCH_MACRO", "25"))  # timesteps of the same train batch evaluated in one U-Net pass (same parameters, see train_step doc)
GUIDANCE, ETA, CLIP = 5.0, 1.0, 1e-4
UNET_GFLOP = 804.3  # algorithmic GFLOP of one SD2-base U-Net application (SURVEY.md §8d / BASELINE.md §2)
WORKLOAD = "DDPO SD2-base 512px, 50-step DDIM, CFG 5.0, eta 1.0, sample batch 8/GPU (BASELINE configs[1])"
GRAD_SAMPLE = 1 << 20  # gradient entries --dump-outputs keeps (4 MB; the whole fp32 gradient is 3.5 GB)


def _write_outputs(path, arrays):
    """--dump-outputs: one float32 .npy per array, so that two builds can be compared output for output."""
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), np.ascontiguousarray(a, dtype=np.float32))


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return d.get("bf16_tflops_sustained", 1387.8), d.get("bf16_tflops", 1645.5), d.get("hbm_gbs", 6576.4), "measured"
    return 1400.0, 1590.0, 6650.0, "fallback"


class ClockSampler(threading.Thread):
    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.samples = []
        self.reasons = set()
        self.max_mhz = None
        self.stop_flag = False

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i",
                                      str(self.index)], capture_output=True, text=True, timeout=5).stdout.strip()
                f = [x.strip() for x in out.split(",")]
                self.samples.append(float(f[0]))
                self.max_mhz = float(f[1])
                for n, v in zip(names, f[2:]):
                    if v.lower().startswith("active"):
                        self.reasons.add(n)
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons)}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons)}


# ------------------------------------------------------------------- CPU arm ----
UNIT = "PPO samples/s"   # ONE unit string for both arms (the driver divides the two values only if metric/unit agree)
UNIT_DETAIL = ("a PPO sample = 50 denoising steps (both CFG branches) + VAE decode of the final latent + 50 PPO train "
               "steps (cond + uncond U-Net forward and backward) + its share of the optimizer update")


def parity_inputs():
    """The one-sample workload both arms evaluate for the parity block: x_T from threefry key (0, 7), its step key, and
    N(0,1) prompt / negative-prompt embeddings (seeded torch CPU generator -> identical bytes on both sides)."""
    import torch
    from oracle import threefry
    g = torch.Generator().manual_seed(1)
    ctx = torch.randn(2, 77, 1024, generator=g)                       # [uncond ; cond]
    x = threefry.normal(np.array((0, 7), np.uint32), (1, 4, 64, 64)).astype(np.float32)
    return x, ctx, (0, 11)


def _cpu_threads():
    """Threads of the CPU arm = PHYSICAL cores this process may use.  torchrun exports OMP_NUM_THREADS=1 (rank 0 is the
    only rank that runs the CPU arm and must still use the whole host), while one thread per hyper-thread (128 on the
    64-core GPU box) makes oneDNN's autograd path collapse -- measured: the 34 s train step did not finish in 10 minutes."""
    import torch
    n = None
    try:
        import psutil
        n = psutil.cpu_count(logical=False)
    except Exception:
        pass
    avail = os.cpu_count() or 1
    try:
        avail = len(os.sched_getaffinity(0))
    except Exception:
        pass
    n = max(1, min(n or avail, avail))
    if torch.get_num_threads() != n:
        torch.set_num_threads(n)
    return torch.get_num_threads()


def _oracle_net():
    from ddpo_b200 import unet_spec
    from oracle.unet import UNetOracle
    cfg = unet_spec.SD2_BASE
    flat = unet_spec.init_flat_params(cfg, 0)
    return cfg, flat, UNetOracle(cfg, unet_spec.views(flat, cfg))


def cpu_step_seconds(n_steps, net=None):
    """Times the CPU oracle (restated reference path: oracle/unet.py + oracle/scheduler.py) on denoising steps of ONE
    sample (2 U-Net applications each, SD2-base, fp32) -- bounded sample.  The first (untimed, warm-up) step runs on
    `parity_inputs()` and its outputs are returned for the GPU-vs-oracle parity block."""
    import torch
    from oracle import scheduler as OS, ppo as OPPO
    cores = _cpu_threads()
    if net is None:
        _, _, net = _oracle_net()
    st = OS.set_timesteps(OS.SD_CONFIG, OS.create_state(OS.SD_CONFIG), T_STEPS)
    x0, ctx, key = parity_inputs()
    x = torch.from_numpy(x0)
    times, first = [], None
    for s in range(n_steps + 1):
        t0 = time.perf_counter()
        with torch.no_grad():
            e = net(torch.cat([x, x]), torch.full((2,), int(st.timesteps[s])), ctx).numpy()
        eps = OPPO.cfg_combine(e[:1], e[1:], GUIDANCE)
        xn, _, lp = OS.step(OS.SD_CONFIG, st, eps, int(st.timesteps[s]), x.numpy(),
                            key=np.array(key if s == 0 else (1, s), np.uint32), eta=ETA)
        if s == 0:
            first = {"eps_u": e[:1].copy(), "eps_c": e[1:].copy(), "prev": xn.copy(), "logp": np.asarray(lp).copy()}
        x = torch.from_numpy(xn)
        if s > 0:  # first step = warm-up (allocator, thread pool)
            times.append(time.perf_counter() - t0)
    return float(np.mean(times)), cores, first


def cpu_unet_application_seconds(net, n_timed, n_warm):
    """Reference-arm step: ONE U-Net application of one sample (alternating uncond / cond context)."""
    import torch
    x0, ctx, _ = parity_inputs()
    x = torch.from_numpy(x0)
    ts = []
    for i in range(n_warm + n_timed):
        t0 = time.perf_counter()
        with torch.no_grad():
            net(x, torch.full((1,), 981 - 20 * (i % 50)), ctx[i % 2:i % 2 + 1])
        if i >= n_warm:
            ts.append(time.perf_counter() - t0)
    return ts


def cpu_vae_decode_seconds():
    """One image through the oracle's Flax VAE decoder (oracle/vae.py; reference pipeline/policy_gradient.py:174-182)."""
    import torch
    from ddpo_b200 import vae as V
    from oracle import vae as OV
    vflat = V.init_flat_params(V.SD_VAE, 1)
    z = torch.randn(1, 4, 64, 64, generator=torch.Generator().manual_seed(5)) * 0.18215
    t0 = time.perf_counter()
    with torch.no_grad():
        OV.decode(V.views(vflat, V.SD_VAE), V.SD_VAE, z)
    return time.perf_counter() - t0


def _ncu_traffic():
    """Average DRAM bytes (read + write) per igemm launch of one denoising step, from the committed ncu capture of
    `bench.py --ncu sample` (profiles/r1_traffic.json, written by profiles/make_launch_summary.py); None if absent."""
    for name in ("r2_launches_summary.json",):
        try:
            with open(os.path.join(ROOT, "profiles", name)) as f:
                return json.load(f)["sample"]["igemm"]["dram_bytes_per_launch"]
        except Exception:
            continue
    return None


def _dump_shapes(prof, tags, path):
    """Per-(kernel, shape) table of the eager CUDA-event profile: which GEMM shapes the time goes to."""
    agg = {}
    for (name, work, a, b), tag in zip(prof, tags):
        d = agg.setdefault((name, tag), [0.0, 0.0, 0])
        d[0] += a.elapsed_time(b)
        d[1] += work
        d[2] += 1
    tot = sum(v[0] for v in agg.values())
    os.makedirs(os.path.dirname(path), exist_ok=True)
    with open(path, "w") as f:
        f.write(f"total {tot:.3f} ms\n")
        for (name, tag), v in sorted(agg.items(), key=lambda kv: -kv[1][0]):
            tf = f"{v[1] / (v[0] * 1e-3) / 1e12:7.1f} TF/s" if v[1] > 0 else ""
            f.write(f"{v[0]:8.3f} ms {100 * v[0] / tot:5.1f}%  n={v[2]:3d}  {v[0] / v[2] * 1e3:8.1f} us/launch  {name:16s} {tag}  {tf}\n")


def cpu_train_step_seconds():
    """Times the CPU oracle's PPO train step (oracle/pipeline.py::train_loss, the restated
    ddpo/training/policy_gradient.py:86-138: cond + uncond U-Net forward, CFG, score-mode log-prob, clipped loss, and
    jax.grad's counterpart -- torch autograd through both U-Net applications) for ONE sample at ONE timestep."""
    import torch
    from ddpo_b200 import unet_spec
    from oracle import pipeline as OP, scheduler as OS
    from oracle.unet import UNetOracle
    _cpu_threads()
    cfg = unet_spec.SD2_BASE
    # every parameter its own autograd leaf, as in the reference's pytree (slices of one flat leaf would make each
    # of the 686 SliceBackward nodes materialise a 3.5 GB zero tensor)
    flat = unet_spec.init_flat_params(cfg, 0)
    params = {k: v.clone().requires_grad_(True) for k, v in unet_spec.views(flat, cfg).items()}
    del flat
    net = UNetOracle(cfg, params)
    st = OS.set_timesteps(OS.SD_CONFIG, OS.create_state(OS.SD_CONFIG), T_STEPS)
    g = torch.Generator().manual_seed(2)
    batch = {"latents": torch.randn(1, 4, 64, 64, generator=g).numpy(), "next_latents": torch.randn(1, 4, 64, 64, generator=g).numpy(),
             "ts": np.array([int(st.timesteps[3])], np.int32), "log_probs": np.array([-1.4], np.float32),
             "advantages": np.array([1.0], np.float32), "prompt_embeds": torch.randn(1, 77, 1024, generator=g).numpy(),
             "uncond_embeds": torch.randn(1, 77, 1024, generator=g).numpy()}
    t0 = time.perf_counter()
    loss, info, lp = OP.train_loss(net, OS.SD_CONFIG, st, batch, True, GUIDANCE, ETA, CLIP)
    loss.backward()
    dt = time.perf_counter() - t0
    assert params["conv_in/kernel"].grad is not None
    return dt


def cpu_ppo_samples_per_sec(n_denoise):
    """The headline metric on the host cores from a BOUNDED sample: `n_denoise` timed denoising steps of one sample
    (after one warm-up step), one VAE decode of one image and one PPO train step of one sample, extrapolated linearly to
    a PPO sample = 50 denoising steps + decode + 50 train steps (every step of the trajectory costs the same: the scan /
    loop bodies are step-invariant).  Returns a dict (value, pieces, threads, first-step outputs for the parity block)."""
    per_step, cores, first = cpu_step_seconds(n_denoise)
    t_vae = cpu_vae_decode_seconds()
    t_train = cpu_train_step_seconds()
    s_per_sample = T_STEPS * per_step + t_vae + T_STEPS * t_train
    return {"value": 1.0 / s_per_sample, "denoising_steps_per_sec": 1.0 / per_step, "seconds_per_train_step": t_train,
            "seconds_per_vae_decode": t_vae, "cores": cores, "first": first}


def run_reference(args):
    """Reference arm: the reference's own path cannot be installed here (jax / flax / diffusers are absent and there
    is no network, DESIGN.md section 1), so this times the oracle port of it on the host cores -- same metric, unit and
    workload as the B200 arm.  A timed "step" is ONE U-Net application of one sample (what `ms_per_step` and `steps`
    describe, so steps x ms_per_step is time really spent in this run); one VAE decode and one PPO train step (forward +
    autograd backward through both CFG branches) are timed once each; `value` extrapolates those pieces to a PPO sample
    (`extrapolated: true`): 100 applications + decode + 50 train steps."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = _cpu_threads()
    _, _, net = _oracle_net()
    ts = cpu_unet_application_seconds(net, max(1, int(args.steps)), max(0, int(args.warmup)))
    del net
    t_app = float(np.mean(ts))
    t_vae = cpu_vae_decode_seconds()
    t_train = cpu_train_step_seconds()
    s_per_sample = 2 * T_STEPS * t_app + t_vae + T_STEPS * t_train
    v = 1.0 / s_per_sample
    sample = (f"{len(ts)} timed U-Net applications of 1 sample (fp32, SD2-base) + 1 VAE decode of 1 image + 1 PPO train "
              f"step of 1 sample (2 U-Net forward + backward), torch-CPU oracle port on {cores} threads; extrapolated to "
              f"100 applications + decode + 50 train steps")
    print(json.dumps({
        "impl": "reference", "metric": "ppo_samples_per_sec", "value": v, "unit": UNIT, "unit_detail": UNIT_DETAIL,
        "n_gpus": args.gpus, "steps": len(ts), "warmup": max(0, int(args.warmup)), "ms_per_step": 1e3 * t_app,
        "step_is": "one U-Net application of one sample on the host cores", "extrapolated": True,
        "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "denoising_steps_per_sec": 1.0 / (2 * t_app), "seconds_per_train_step": t_train, "seconds_per_vae_decode": t_vae,
        "config": {"workload": WORKLOAD, "cpu_arm": "1 sample at a time"},
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


# ------------------------------------------------------------------- GPU arm ----
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--phase", default="auto", choices=["auto", "sample", "ppo"])
    ap.add_argument("--cpu-steps", type=int, default=2)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--ncu", default="", choices=["", "sample", "train"],
                    help="run under `ncu --profile-from-start off`: bracket ONE eager denoising step / train pass with "
                         "cudaProfilerStart/Stop, print nothing, exit (profiles/README.md has the command lines)")
    ap.add_argument("--shapes", action="store_true", help="also write per-shape kernel tables to gpurun_out/shapes_*.txt")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak: 8 samples per GPU per epoch (default); strong: 64 samples per epoch for the whole job "
                         "(SURVEY 8d: sample batch 8 x 8/N batches per GPU), visible in the epoch-driver e2e number")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="after the timed steps, write what the last timed step of each phase returned as DIR/<name>.npy "
                         "(float32; rank 0): sample_next_latents, sample_log_probs, ppo_loss, ppo_approx_kl, ppo_clipfrac "
                         "and ppo_grad_sample, the accumulated U-Net gradient at %d fixed indices (numpy default_rng(0))"
                         % GRAD_SAMPLE)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")  # keep stdout to the single JSON line
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)

    from ddpo_b200 import ops, unet_spec
    from ddpo_b200.diffusers_patch import DDIMScheduler, StableDiffusionPipeline
    from ddpo_b200.unet import UNet
    sus_tf, burst_tf, hbm_gbs, peak_src = _peaks()

    cfg = unet_spec.SD2_BASE
    # random-init weights from the seeded CPU generator: identical on every rank AND identical to what the CPU oracle
    # leg builds, so the parity block below compares like with like
    flat = unet_spec.init_flat_params(cfg, 0)
    net = UNet(cfg, flat, dev)
    del flat
    sched = DDIMScheduler(1000, 0.00085, 0.012, "scaled_linear", None, False, 1, "epsilon", device=dev)
    pipe = StableDiffusionPipeline(net, sched, vae_scale_factor=8)
    state = sched.create_state()

    B = SAMPLE_BATCH
    gh = torch.Generator().manual_seed(1 + rank)
    emb_host = torch.randn(B, 77, 1024, generator=gh).pin_memory()
    neg_host = torch.randn(1, 77, 1024, generator=torch.Generator().manual_seed(2)).expand(B, -1, -1).contiguous().pin_memory()
    seed_key = ops.threefry_split(ops.prng_key(0), max(2, world))[rank % max(2, world)]

    # ---------------- phase: sample (device-resident timing of K denoising steps) ----------------
    emb, neg = emb_host.to(dev), neg_host.to(dev)
    st = sched.set_timesteps(state, T_STEPS)
    ratio = 1000 // T_STEPS
    net.prepare_context(torch.cat([neg, emb]))
    S = pipe._step_buffers(B, 64, 64, dev)
    ops.threefry_normal(ops.key_tensor([seed_key], dev), S["x_cur"].view(-1))
    ts_dev = torch.as_tensor(np.asarray(st.timesteps, np.int32), device=dev)
    S["t_dev"].copy_(ts_dev[0:1])
    S["key_dev"].copy_(ops.key_tensor([seed_key], dev)[0])

    def one_step():
        pipe._one_step(S, B, st, ratio, GUIDANCE, ETA)

    lc0 = ops.LAUNCH_COUNT
    one_step()
    torch.cuda.synchronize()
    launches_per_step = ops.LAUNCH_COUNT - lc0
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        one_step()

    def step(i):
        S["t_dev"].copy_(ts_dev[i % T_STEPS:i % T_STEPS + 1])
        graph.replay()
        S["x_cur"].copy_(S["x_next"])

    for i in range(max(3, args.warmup)):
        step(i)
    sampler = ClockSampler(local)
    sampler.start()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(args.steps):
        step(i)
    e1.record()
    torch.cuda.synchronize()
    outputs = {}   # what the last timed step of each phase returned, for --dump-outputs
    if args.dump_outputs:
        outputs["sample_next_latents"] = S["x_next"].view(B, 4, 64, 64).cpu().numpy()
        outputs["sample_log_probs"] = S["logp"].cpu().numpy()
    if world > 1:
        dist.barrier()
    ms = e0.elapsed_time(e1)
    sampler.stop_flag = True
    tms = torch.tensor([ms], device=dev)
    if world > 1:
        dist.all_reduce(tms, op=dist.ReduceOp.MAX)
    ms = tms.item()
    ms_per_step = ms / args.steps
    steps_per_s = world * B * args.steps / (ms / 1e3)  # denoising steps of one sample, whole job

    if args.ncu == "sample":
        torch.cuda.synchronize()
        torch.cuda.profiler.start()
        one_step()
        torch.cuda.synchronize()
        torch.cuda.profiler.stop()
        return
    # ---------------- kernel profile (eager, CUDA events per launch) ----------------
    ops.PROFILE, ops.PROFILE_TAGS = [], []
    one_step()
    torch.cuda.synchronize()
    prof = ops.PROFILE
    ops.PROFILE = None
    if args.shapes and rank == 0:
        _dump_shapes(prof, ops.PROFILE_TAGS, "gpurun_out/shapes_sample.txt")
    agg = {}
    for name, work, a, b in prof:
        d = agg.setdefault(name, [0.0, 0.0, 0])
        d[0] += a.elapsed_time(b)
        d[1] += work
        d[2] += 1
    tot_ms = sum(v[0] for v in agg.values())
    ig = agg.get("igemm", [1e-9, 0, 0])
    igemm_tflops = ig[1] / (ig[0] * 1e-3) / 1e12
    gn = agg.get("groupnorm_fwd", [1e-9, 0, 0])
    breakdown = {k: {"ms": round(v[0], 3), "launches": v[2], "share": round(v[0] / tot_ms, 4)} for k, v in agg.items()}
    at = agg.get("attention_fwd", [1e-9, 0, 0])
    breakdown["igemm"]["tflops"] = round(igemm_tflops, 1)
    breakdown["attention_fwd"]["tflops"] = round(at[1] / (at[0] * 1e-3) / 1e12, 1)
    breakdown["groupnorm_fwd"]["gbs"] = round(gn[1] / (gn[0] * 1e-3) / 1e9, 1)

    # ---------------- e2e: the public pipeline call with host buffers ----------------
    def e2e_call():
        e = emb_host.to(dev, non_blocking=True)
        n_ = neg_host.to(dev, non_blocking=True)
        final, lat, nxt, lps, ts = pipe(e, n_, {"unet": net.params, "scheduler": state}, seed_key, T_STEPS, 512, 512,
                                        GUIDANCE, ETA)
        return final.cpu(), lps.cpu()

    e2e_call()  # warm (captures the pipeline's own graph)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    fin, lps = e2e_call()
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    tdt = torch.tensor([dt], device=dev)
    if world > 1:
        dist.all_reduce(tdt, op=dist.ReduceOp.MAX)
    e2e_steps_per_s = world * B * T_STEPS / tdt.item()
    h2d = (emb_host.numel() + neg_host.numel()) * 4 / T_STEPS
    d2h = (fin.numel() + lps.numel()) * 4 / T_STEPS

    # ---------------- VAE decode of the sample batch (the step between sampling and the reward, reference
    # pipeline/policy_gradient.py:271-275): device time per batch and end to end (images copied to the host) ------------
    vae_info = None
    try:
        from ddpo_b200.vae import SD_VAE, VAEDecoder
        dec = VAEDecoder(SD_VAE, device=dev, seed=1, decode_batch=2)
        lat8 = (S["x_cur"].view(B, 4, 64, 64) * 0.18215).contiguous()
        lcv = ops.LAUNCH_COUNT
        dec.decode(lat8)
        torch.cuda.synchronize()
        vae_launches = ops.LAUNCH_COUNT - lcv
        v0, v1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        v0.record()
        for _ in range(2):
            img = dec.decode(lat8)
        v1.record()
        torch.cuda.synchronize()
        ms_decode = v0.elapsed_time(v1) / 2
        tv = time.perf_counter()
        img_host = dec.decode(lat8).cpu()
        ms_decode_e2e = (time.perf_counter() - tv) * 1e3
        ok = bool(torch.isfinite(img).all().item()) and float(img.min()) >= 0.0 and float(img.max()) <= 1.0
        vae_info = {"ms_per_batch": ms_decode, "ms_per_batch_e2e": ms_decode_e2e, "images": B, "launches": vae_launches,
                    "d2h_bytes": img_host.numel() * 4, "finite_in_unit_range": ok,
                    "tflops": B * 1.24e12 / (ms_decode * 1e-3) / 1e12}
        del dec, img, img_host
        torch.cuda.empty_cache()
    except Exception as ex:  # reported, never hidden: the headline then excludes the decode and says so
        vae_info = {"error": repr(ex)[:300]}

    # ---------------- parity of THIS build at THIS config against the fp32 oracle (N = 1 only: it needs the CPU leg);
    # taken BEFORE the PPO phase: the optimizer updates below change the weights the oracle leg is built from ----
    # one denoising step of one sample on `parity_inputs()`: eps of both CFG branches, the sampled x_{t-1} and its log-prob,
    # and -- the number PPO's importance ratio depends on -- the score-mode log-prob of the ORACLE's x_{t-1} under the
    # GPU's eps (reference pipeline_flax_stable_diffusion.py:204-241, training/policy_gradient.py:103-125)
    parity_gpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        x0, pctx, pkey = parity_inputs()
        xg = torch.from_numpy(x0).to(dev).view(1, -1)
        net.prepare_context(pctx.to(dev))
        eps_g = net.forward(torch.cat([xg, xg]).view(2, 4, 64, 64), ts_dev[0:1]).view(2, -1)
        prev_g, lp_g = torch.empty_like(xg), torch.empty(1, device=dev)
        ws1 = ops.ddim_workspace(1, dev)
        ops.ddim_step_sample(eps_g[:1], eps_g[1:], xg, st.common.alphas_cumprod, ts_dev[0:1], st.final_alpha_cumprod, ratio,
                             GUIDANCE, ETA, ops.key_tensor([pkey], dev), prev_g, lp_g, ws1)
        torch.cuda.synchronize()
        parity_gpu = dict(eps=eps_g.cpu().numpy(), prev=prev_g.cpu().numpy(), logp=lp_g.cpu().numpy(), xg=xg, eps_dev=eps_g,
                          ws=ws1)

    # ---------------- phase: ppo train steps (fwd+bwd of the 2x2 CFG batch) + one optimizer update ----------------
    ppo = None
    if args.phase in ("auto", "ppo"):
        from ddpo_b200.training import policy_gradient as pg
        Bt = TRAIN_BATCH
        # pmean_info=False below: as the epoch driver does, the (3-float) info of a pass is not all-reduced after every pass
        # but once per inner epoch -- the only per-pass collective of the reference loop that is not the gradient
        tstate = pg.AccumulatingTrainState(apply_fn=net)
        # a short real trajectory to train on (device resident)
        final, lat, nxt, lps, tss = pipe(emb[:Bt], neg[:Bt], {"unet": net.params, "scheduler": state}, seed_key, T_STEPS,
                                         512, 512, GUIDANCE, ETA)
        adv = torch.tensor([1.0, -1.0], device=dev)

        J = TRAIN_MACRO

        def make_batch(j0, host=False):
            """J consecutive (shuffled-order) timesteps of the Bt samples, stacked micro-batch major"""
            js = [(j0 + i) % T_STEPS for i in range(J)]
            st_ = lambda x: torch.stack([x[:, j] for j in js], 0).reshape(J * Bt, *x.shape[2:]).contiguous()
            rep = lambda x: x.unsqueeze(0).expand(J, *x.shape).reshape(J * Bt, *x.shape[1:]).contiguous()
            bt = {"latents": st_(lat), "next_latents": st_(nxt), "ts": st_(tss), "log_probs": st_(lps),
                  "advantages": rep(adv), "prompt_embeds": rep(emb[:Bt]), "uncond_embeds": rep(neg[:Bt])}
            if host:
                bt = {k: v.cpu().pin_memory() for k, v in bt.items()}
            return bt

        batches = [make_batch((j * J) % T_STEPS) for j in range(5)]
        lc0 = ops.LAUNCH_COUNT
        pg.USE_CUDA_GRAPH = False
        pg.train_step(tstate, batches[0], st, sched, True, GUIDANCE, ETA, CLIP, False, micro_batch_size=Bt, pmean_info=False)
        torch.cuda.synchronize()
        train_launches = ops.LAUNCH_COUNT - lc0
        pg.USE_CUDA_GRAPH = True
        for i in range(max(3, args.warmup)):
            _, info = pg.train_step(tstate, batches[i % len(batches)], st, sched, True, GUIDANCE, ETA, CLIP, False, micro_batch_size=Bt, pmean_info=False)
        first_pass_kl = float(info["approx_kl"].item())
        if args.ncu == "train":
            pg.USE_CUDA_GRAPH = False
            torch.cuda.synchronize()
            torch.cuda.profiler.start()
            pg.train_step(tstate, batches[1], st, sched, True, GUIDANCE, ETA, CLIP, False, micro_batch_size=Bt, pmean_info=False)
            torch.cuda.synchronize()
            torch.cuda.profiler.stop()
            return
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        t0e, t1e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0e.record()
        for i in range(args.steps):
            _, last_info = pg.train_step(tstate, batches[i % len(batches)], st, sched, True, GUIDANCE, ETA, CLIP, False,
                                         micro_batch_size=Bt, pmean_info=False)
        t1e.record()
        torch.cuda.synchronize()
        if args.dump_outputs:
            for k, v in last_info.items():
                outputs[f"ppo_{k}"] = v.cpu().numpy().reshape(1)
            idx = np.random.default_rng(0).integers(0, tstate.grad_acc.numel(), GRAD_SAMPLE)
            outputs["ppo_grad_sample"] = tstate.grad_acc[torch.from_numpy(idx).to(dev)].cpu().numpy()
        if world > 1:
            dist.barrier()
        tt = torch.tensor([t0e.elapsed_time(t1e)], device=dev)
        # one optimizer update: NCCL all-reduce of the flat gradient + global norm + clip/AdamW + bf16 weight refresh
        u0, u1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        u0.record()
        pg.train_step(tstate, batches[0], st, sched, True, GUIDANCE, ETA, CLIP, True, micro_batch_size=Bt, pmean_info=False)
        u1.record()
        torch.cuda.synchronize()
        tu = torch.tensor([u0.elapsed_time(u1)], device=dev)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            dist.all_reduce(tu, op=dist.ReduceOp.MAX)
        ms_train = tt.item() / args.steps
        ms_update = max(0.0, tu.item() - ms_train)
        # the data-path collective on its own: sum all-reduce of the flat fp32 gradient (what one optimizer update issues)
        allreduce_ms = allreduce_busbw = None
        if world > 1:
            from ddpo_b200.training import distributed as D
            gbuf = tstate.grad_acc
            D.allreduce_sum_(gbuf)
            torch.cuda.synchronize()
            dist.barrier()
            a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a0.record()
            for _ in range(3):
                D.allreduce_sum_(gbuf)
            a1.record()
            torch.cuda.synchronize()
            ta = torch.tensor([a0.elapsed_time(a1) / 3], device=dev)
            dist.all_reduce(ta, op=dist.ReduceOp.MAX)
            allreduce_ms = ta.item()
            allreduce_busbw = 2 * (world - 1) / world * gbuf.numel() * 4 / (allreduce_ms * 1e-3) / 1e9
            gbuf.zero_()
        # e2e train step: host-resident batch in, loss out
        hb = make_batch(1, host=True)
        pg.train_step(tstate, hb, st, sched, True, GUIDANCE, ETA, CLIP, False, micro_batch_size=Bt, pmean_info=False)
        torch.cuda.synchronize()
        te0 = time.perf_counter()
        for _ in range(3):
            _, info = pg.train_step(tstate, hb, st, sched, True, GUIDANCE, ETA, CLIP, False, micro_batch_size=Bt, pmean_info=False)
            _loss = float(info["loss"].item())
        ms_train_e2e = (time.perf_counter() - te0) / 3 * 1e3
        # profile one eager train step
        pg.USE_CUDA_GRAPH = False
        ops.PROFILE, ops.PROFILE_TAGS = [], []
        pg.train_step(tstate, batches[1], st, sched, True, GUIDANCE, ETA, CLIP, False, micro_batch_size=Bt, pmean_info=False)
        torch.cuda.synchronize()
        tprof = ops.PROFILE
        ops.PROFILE = None
        if args.shapes and rank == 0:
            _dump_shapes(tprof, ops.PROFILE_TAGS, "gpurun_out/shapes_train.txt")
        pg.USE_CUDA_GRAPH = True
        tagg = {}
        for name, work, a, b in tprof:
            d = tagg.setdefault(name, [0.0, 0.0, 0])
            d[0] += a.elapsed_time(b)
            d[1] += work
            d[2] += 1
        ttot = sum(v[0] for v in tagg.values())
        tbreak = {k: {"ms": round(v[0], 3), "launches": v[2], "share": round(v[0] / ttot, 4)} for k, v in tagg.items()}
        for k in ("igemm", "wgrad", "attention_fwd", "attention_bwd"):
            if k in tagg and tagg[k][0] > 0:
                tbreak[k]["tflops"] = round(tagg[k][1] / (tagg[k][0] * 1e-3) / 1e12, 1)
        # one PPO sample = T sampling steps (batch 8) + T train steps (batch 2) + its share of the update
        # (a macro train step covers J timesteps of Bt samples)
        dec_ms = vae_info.get("ms_per_batch", 0.0) / B if vae_info else 0.0          # VAE decode share per sample
        dec_ms_e2e = vae_info.get("ms_per_batch_e2e", 0.0) / B if vae_info else 0.0
        s_per_sample = T_STEPS * (ms_per_step / B) + dec_ms + (T_STEPS / J) * (ms_train / Bt) + ms_update / Bt
        s_per_sample_e2e = (T_STEPS * (1e3 / (e2e_steps_per_s / world)) + dec_ms_e2e + (T_STEPS / J) * (ms_train_e2e / Bt)
                            + ms_update / Bt)
        ppo = {"ms_per_train_step": ms_train, "ms_per_update": ms_update, "train_launches": train_launches,
               "allreduce_ms": allreduce_ms, "allreduce_busbw_gbs": allreduce_busbw,
               "samples_per_s": world * 1e3 / s_per_sample, "samples_per_s_e2e": world * 1e3 / s_per_sample_e2e,
               "ms_train_step_e2e": ms_train_e2e, "first_pass_approx_kl": first_pass_kl,
               "train_tflops_per_gpu": 3 * 2 * Bt * J * UNET_GFLOP * 1e9 / (ms_train * 1e-3) / 1e12,
               "train_batch": Bt, "timesteps_per_train_pass": J, "unet_batch_per_train_pass": 2 * Bt * J, "kernels": tbreak}

    # ---------------- e2e through the epoch driver (the call a user makes): pipeline/policy_gradient.main ------------
    # prompts -> CLIP text tower (GPU) -> 50-step sampling of 8 samples -> VAE decode -> images to the host -> JPEG reward on the
    # driver's thread pool -> advantages -> shuffles -> on-device gathers -> 20 macro train passes + 4 optimizer updates.
    # Epoch 0 warms up (graph capture); epoch 1 is timed by the driver's own wall clock (includes every H2D / D2H).
    driver = None
    if ppo is not None and vae_info is not None and "error" not in vae_info and not args.ncu:
        try:
            import contextlib
            from ddpo_b200.pipeline import policy_gradient as PG
            from ddpo_b200.text_encoder import SD2_TEXT, CLIPTextEncoder
            from ddpo_b200.utils.text_stub import StubTokenizer
            from ddpo_b200.vae import SD_VAE, VAEDecoder
            pipe.vae = VAEDecoder(SD_VAE, device=dev, seed=1, decode_batch=2)
            net.grads.zero_()  # the timing passes above accumulated gradients the driver's fresh train state must not see
            # prompts are embedded by the CLIP text tower on the GPU (random-init SD2 tower; ids from the stub tokenizer:
            # no vocabulary files offline)
            pipe.tokenizer, pipe.text_encoder = StubTokenizer(), CLIPTextEncoder(SD2_TEXT, device=dev, seed=2)
            nsb = max(1, 8 // world) if args.scaling == "strong" else 1   # strong: 64 samples per epoch over the whole job
            argv = ["--dataset", "compressed_animals", "--sample_batch_size", str(B), "--num_sample_batches_per_epoch", str(nsb),
                    "--train_batch_size", str(TRAIN_BATCH), "--train_macro", str(TRAIN_MACRO), "--num_train_epochs", "3",
                    "--save_freq", "1000000", "--savepath", f"bench_driver_{rank}", "--seed", "0"]
            # the driver writes its logs/ (args, sample images, rewards) under the working directory: a temporary one, so
            # that the benchmark leaves the source tree untouched and runs from a read-only one
            with tempfile.TemporaryDirectory() as tmp, contextlib.chdir(tmp), contextlib.redirect_stdout(sys.stderr):
                out = PG.main(argv, models=(pipe, {"unet": net.params, "scheduler": state, "text_encoder": {}}),
                              max_epochs=3, save_last=False)
            # epoch 0 warms up (graph capture, arena growth); of the two steady-state epochs the faster one is reported
            # (the host side -- JPEG threads, Python -- jitters by a few per cent between epochs)
            h = min(out["history"][1:], key=lambda e: e["sample_seconds"] + e["train_seconds"])
            tsec = torch.tensor([h["sample_seconds"], h["train_seconds"]], device=dev, dtype=torch.float64)
            if world > 1:
                dist.all_reduce(tsec, op=dist.ReduceOp.MAX)
            ssec, trsec = tsec.tolist()
            kl = out["history"][0]["infos"][0]["approx_kl"]
            NB = B * nsb                                                   # samples per epoch on this GPU
            driver = {"samples_per_s": world * NB / (ssec + trsec), "sample_seconds": ssec, "train_seconds": trsec,
                      "samples_per_epoch_per_gpu": NB, "samples_per_epoch": world * NB, "mean_reward": h["mean_reward"],
                      "epoch0_first_pass_approx_kl": float(kl[0]),
                      "optimizer_updates_per_epoch": NB // TRAIN_BATCH,
                      "h2d_bytes_per_epoch": (NB + 1) * 77 * 8 + (NB // TRAIN_BATCH) * (T_STEPS // TRAIN_MACRO) * TRAIN_MACRO * TRAIN_BATCH * 40,
                      # images leave as uint8 (the JPEG reward's own cast, done on the device: pipeline/policy_gradient.images_to_host)
                      "d2h_bytes_per_epoch": NB * 512 * 512 * 3 * 1 + NB * T_STEPS * 8 + (NB // TRAIN_BATCH) * (T_STEPS // TRAIN_MACRO) * 12}
        except Exception as ex:  # reported, never hidden
            driver = {"error": repr(ex)[:300]}

    if rank == 0:
        cpu, parity = None, None
        if not args.no_cpu and world == 1:   # the CPU baseline is reported by the N = 1 run only
            c = cpu_ppo_samples_per_sec(args.cpu_steps)
            cpu = {"value": c["value"], "unit": UNIT, "cores": c["cores"], "kind": "port",
                   "denoising_steps_per_sec": c["denoising_steps_per_sec"], "seconds_per_train_step": c["seconds_per_train_step"],
                   "seconds_per_vae_decode": c["seconds_per_vae_decode"],
                   "sample": f"{args.cpu_steps} denoising steps of 1 sample (2 U-Net applications each) + 1 VAE decode + 1 PPO "
                             f"train step of 1 sample (2 U-Net forward + backward), torch-CPU oracle port, extrapolated to "
                             f"50 steps + decode + 50 train steps"}
            f, g_ = c["first"], parity_gpu
            rel = lambda a, b: float(np.linalg.norm(a.ravel() - b.ravel()) / np.linalg.norm(b.ravel()))
            lp_s = torch.empty(1, device=dev)
            ops.ddim_logprob_fwd(g_["eps_dev"][:1], g_["eps_dev"][1:], g_["xg"], torch.from_numpy(f["prev"]).to(dev).view(1, -1),
                                 st.common.alphas_cumprod, ts_dev[0:1], st.final_alpha_cumprod, ratio, GUIDANCE, ETA, lp_s, g_["ws"])
            lp_score = float(lp_s.item())
            parity = {"what": "one denoising step (t=981) of one sample, SD2-base, this build vs the fp32 CPU oracle on the same "
                              "weights / inputs / threefry key",
                      "eps_rel": rel(g_["eps"], np.concatenate([f["eps_u"], f["eps_c"]]).reshape(2, -1)),
                      "latents_rel": rel(g_["prev"], f["prev"]),
                      "logp_rel": float(abs(g_["logp"][0] / f["logp"].ravel()[0] - 1.0)),
                      "logp_score_rel": float(abs(lp_score / f["logp"].ravel()[0] - 1.0)),
                      "ratio_minus_1": float(abs(np.exp(lp_score - float(f["logp"].ravel()[0])) - 1.0)),
                      "logp_oracle": float(f["logp"].ravel()[0]), "logp_gpu": float(g_["logp"][0]), "logp_gpu_score_mode": lp_score,
                      "tolerance": "north-star: per-step log_prob within 1e-3 relative"}
        step_flops = 2 * B * UNET_GFLOP * 1e9
        if ppo is not None:
            head = {"metric": "ppo_samples_per_sec", "value": ppo["samples_per_s"], "unit": UNIT, "unit_detail": UNIT_DETAIL}
        else:
            head = {"metric": "denoising_steps_per_sec", "value": steps_per_s,
                    "unit": "denoising steps/s (1 sample, both CFG branches)"}
        line = {
            **head, "denoising_steps_per_sec": steps_per_s, "denoising_steps_per_sec_per_gpu": steps_per_s / world,
            "n_gpus": world, "steps": args.steps, "warmup": max(3, args.warmup), "ms_per_step": ms_per_step,
            "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "bf16 (fp32 accumulate, fp32 residual stream/norms)",
            "data": "synthetic",
            "config": {"workload": WORKLOAD,
                       "per_step": "one denoising step of the 8-sample batch (U-Net batch 16)",
                       "samples_per_epoch": "8 per GPU (weak scaling; BASELINE's batch 64 = 8 GPUs x 8; per-sample work is identical)"
                                            if args.scaling == "weak" else "64 over the whole job (strong scaling)",
                       "l2": "per-step working set (1.7 GB bf16 weights + activations) exceeds the 126 MB L2; no explicit flush",
                       "cuda_graph": True, "per_gpu_steps_per_s": steps_per_s / world,
                       "unet_tflops_per_gpu": step_flops / (ms_per_step * 1e-3) / 1e12},
            "clocks": sampler.summary(),
            "e2e": ({"value": ppo["samples_per_s_e2e"], "unit": UNIT, "h2d_bytes_per_step": h2d + TRAIN_MACRO * TRAIN_BATCH * (2 * 65536 + 2 * 77 * 1024 * 4 + 12),
                     "d2h_bytes_per_step": d2h + 12, "denoising_steps_per_sec": e2e_steps_per_s,
                     "what": "pipeline(...) from pinned host embeddings to host latents/log-probs + train_step(...) from a pinned host batch to host loss"}
                    if ppo is not None else
                    {"value": e2e_steps_per_s, "unit": "denoising steps/s", "h2d_bytes_per_step": h2d,
                     "d2h_bytes_per_step": d2h, "what": "pipeline(...) 50-step call from pinned host embeddings to host final latents + log-probs"}),
            "e2e_driver": driver,
            "e2e_composed": None,
            "parity": parity,
            "ms_per_train_step": ppo["ms_per_train_step"] if ppo else None,
            "ms_per_update": ppo["ms_per_update"] if ppo else None,
            "allreduce_ms": ppo["allreduce_ms"] if ppo else None,
            "allreduce_busbw_gbs": ppo["allreduce_busbw_gbs"] if ppo else None,
            "gpu_launches": launches_per_step * args.steps + (ppo["train_launches"] * args.steps if ppo else 0),
            "ppo": ppo,
            "vae_decode": vae_info,
            "roofline": {"bound": "tensor", "achieved": igemm_tflops, "peak": sus_tf, "unit": "TFLOP/s",
                         "frac": igemm_tflops / sus_tf, "traffic": _ncu_traffic(), "kernel": "igemm2_kernel (CTA-pair implicit GEMM; igemm_kernel below 1024 rows)",
                         "peak_source": f"{peak_src} bf16_tflops_sustained",
                         "how": "sum of algorithmic 2MNK over the igemm launches of one step / sum of their CUDA-event durations"},
            "kernels": breakdown,
            "kernels_note": "per-kernel CUDA-event times of ONE EAGER step: every launch carries a few microseconds of event / launch "
                            "overhead (407 launches per denoising step), so their sum exceeds the graph-replayed ms_per_step; shares "
                            "are what to compare with the ncu launch lists in profiles/",
            "cpu_baseline": cpu,
        }
        if ppo is not None and driver is not None and "error" not in driver:
            # the call a user makes is the epoch driver: its wall-clock samples/s is THE end-to-end number; the figure
            # composed from pipeline(...) + train_step(...) with host buffers is kept next to it
            line["e2e_composed"] = dict(line["e2e"])
            nb_ = driver["samples_per_epoch_per_gpu"]
            steps_per_epoch = (nb_ // SAMPLE_BATCH) * T_STEPS + (nb_ // TRAIN_BATCH) * (T_STEPS // TRAIN_MACRO)
            line["e2e"] = {"value": driver["samples_per_s"], "unit": UNIT,
                           "h2d_bytes_per_step": driver["h2d_bytes_per_epoch"] / steps_per_epoch,
                           "d2h_bytes_per_step": driver["d2h_bytes_per_epoch"] / steps_per_epoch,
                           "what": "ddpo_b200.pipeline.policy_gradient.main (faster of epochs 1-2 of 3, the driver's wall clock): prompts -> "
                                   "text embedding -> 50-step sampling in batches of 8 samples/GPU -> VAE decode -> images to the host -> "
                                   "JPEG reward (thread pool) -> advantages -> shuffles -> on-device gathers -> 5 train passes "
                                   "+ 1 optimizer update per 2 samples; a step = one denoising step or one train pass",
                           "samples_per_epoch_per_gpu": nb_}
        line["gpu_mem_peak_gb"] = round(torch.cuda.max_memory_allocated() / 2 ** 30, 2)
        if args.dump_outputs:
            _write_outputs(args.dump_outputs, outputs)
        print(json.dumps(line))
    # orderly teardown: drop captured graphs and cached buffers before the process exits
    torch.cuda.synchronize()
    if ppo is not None:
        pg._GRAPHS.clear()
    pipe._graphs.clear()
    del graph
    import gc
    gc.collect()
    torch.cuda.empty_cache()
    torch.cuda.synchronize()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
