#!/usr/bin/env python
"""bench.py - rollout latents/sec, SD3.5-medium 1024^2 30-step GRPO sampling (BASELINE.json metric, config C2).

  python bench.py --gpus N --steps K --warmup W              # our arm (one rank per GPU; torchrun for N > 1)
  python bench.py --impl reference --gpus N --steps K --warmup W   # the reference's own CPU classes (oracle/_ref) on host cores
  python bench.py --gpus 1 --steps K --warmup W --dump-outputs DIR  # also writes what the last timed rollout returned, DIR/<name>.npy

A "step" is ONE ROLLOUT: `batch` prompts per rank x 30 denoise steps x (2 transformer forwards with CFG) + the fused
Euler/SDE + log-prob step, synthetic inputs of the BASELINE shape, random-init weights of the SD3.5-medium architecture
(no checkpoints offline).  `value` = whole-job latents/s with inputs resident in HBM, device-timed (CUDA events, max over
ranks); `e2e` = the same metric through the public adapter API with HOST (pinned) inputs and host outputs, copies inside
the timed region.  Working set (4.5 GB of weights + GBs of activations per step) is far larger than the 126 MB L2.
`roofline`: the single kernel shape with the largest time share of a step (joint attention, 46 %), `roofline_gemm`: the GEMM kernel (49 %
over its 216 launches) at the shape with the largest FLOP share (MLP-up); both timed live here, alone before the rollouts and again right
after them; DRAM traffic from the committed ncu captures.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "rollout latents/sec SD3.5-medium 1024^2 30-step"


def ncu_traffic(kernel: str, shape: str):
    """dram__bytes_read.sum + dram__bytes_write.sum of ONE launch of `kernel` at `shape`, read from profiles/ncu_traffic.json - the table
    tools/ncu_traffic.py extracts from the `ncu --set full` captures of exactly these launches; None when that shape was never captured."""
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as f:
            return json.load(f)[kernel][shape]["dram_bytes"]
    except Exception:
        return None


def launch_shares():
    """Kernel shares of one denoise step from the committed ncu launch list of this command (profiles/launch_shares.json, written by
    tools/launchlist_summary.py); empty when absent."""
    try:
        with open(os.path.join(ROOT, "profiles", "launch_shares.json")) as f:
            return json.load(f)
    except Exception:
        return {}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=8, help="prompts per rank per rollout (reference example default: per_device_batch_size 8)")
    ap.add_argument("--height", type=int, default=1024)
    ap.add_argument("--width", type=int, default=1024)
    ap.add_argument("--num-inference-steps", type=int, default=30)
    ap.add_argument("--guidance", type=float, default=4.5)
    ap.add_argument("--n-text", type=int, default=333)
    ap.add_argument("--num-sde-steps", type=int, default=1)
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--skip-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed rollouts, write what the last one returned to its caller (rank 0: kept latents, log-probs, final "
                         "latents and timesteps of the batch) as DIR/<name>.npy in float32, at most 64 MB in all; the inputs are seeded, so "
                         "two builds run with the same arguments can be compared output for output")
    ap.add_argument("--config", default="sd35", choices=["sd35", "flux1", "wan21", "qwen_image"],
                    help="BASELINE.json config: sd35 = C2 (the metric's, default); flux1 / wan21 / qwen_image = configs 3-5, each through its own "
                         "bench tool under tools/ with the same line contract (examples/grpo/*/{flux1/default,wan21/t2v,qwen_image/default}.yaml)")
    return ap.parse_args()


# ------------------------------------------------------------------------------------------------ helpers
def load_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return json.load(f), "measured"
    except Exception:
        return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


class ClockSampler:
    """nvidia-smi clocks + throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx, self.proc, self.lines = gpu_index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200",
                                          "-i", str(self.idx)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            pass
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            p = [x.strip() for x in ln.split(",")]
            if len(p) < 9:
                continue
            try:
                sm.append(float(p[1])); mx.append(float(p[2]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), p[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def flops_per_latent(cfg, ni, nt, T, cfg_on):
    from flow_factory_b200.synth import flops_per_forward
    lin, att = flops_per_forward(cfg, ni, nt)
    return (lin + att) * T * (2 if cfg_on else 1)


DUMP_LIMIT_BYTES = 63_000_000      # 64 MB with room for the .npy headers


def dump_outputs(directory: str, arrays) -> None:
    """Write `arrays` (name -> tensor; None entries skipped) as DIR/<name>.npy, float64 kept, everything else as float32.  When they would
    take more than DUMP_LIMIT_BYTES in all, every array above 1 MB is cut to the same fraction of its flattened elements, at positions drawn
    from a fixed seed, so that two runs with the same arguments write the same positions."""
    import numpy as np
    arrays = {k: v.detach() for k, v in arrays.items() if v is not None}
    size = lambda v: v.numel() * (8 if v.dtype == torch.float64 else 4)
    large = {k for k, v in arrays.items() if size(v) > 1_000_000}
    small_bytes = sum(size(v) for k, v in arrays.items() if k not in large)
    large_bytes = sum(size(arrays[k]) for k in large)
    os.makedirs(directory, exist_ok=True)
    for name, v in arrays.items():
        if name in large and small_bytes + large_bytes > DUMP_LIMIT_BYTES:
            keep = v.numel() * (DUMP_LIMIT_BYTES - small_bytes) // large_bytes
            idx = torch.randint(v.numel(), (keep,), generator=torch.Generator().manual_seed(0)).sort().values
            v = v.flatten()[idx.to(v.device)]
        v = v.cpu().double() if v.dtype == torch.float64 else v.cpu().float()
        np.save(os.path.join(directory, name + ".npy"), v.numpy())


# ------------------------------------------------------------------------------------------------ CPU baseline: the reference's own code
CPU_STEP_BUDGET_S = 12.0      # a timed C2 sample longer than this is cut to the first L blocks (and scaled by FLOPs; stated in `sample`)
CPU_MAX_SAMPLES = 5


def cpu_reference(args, steps: int, warmup: int, full: bool = True):
    """The reference's CPU path through its OWN classes (oracle/ref_runner.py over oracle/_ref: SD3Transformer2DModel.forward +
    FlowMatchEulerDiscreteSDEScheduler.step as SD3_5Adapter.forward calls them, bf16 CPU autocast) on the physical cores of one NUMA node.
      * BASELINE config C1 (256^2, 4 steps, B=1, no CFG) is timed IN FULL (BASELINE.md section 3);
      * config C2 (the metric's): `steps` timed samples of ONE full denoising step at B=1 with CFG (2 transformer forwards at 1024^2 +
        scheduler.step) after `warmup` untimed ones - or, when a full step would take longer than CPU_STEP_BUDGET_S, of its first L blocks,
        scaled to 24 blocks by FLOPs; latents/s = 1 / (best step x T).
    Falls back to the oracle PORT (kind "port") only where oracle/_ref is absent."""
    from oracle import ref_runner as R
    from oracle import sd3_oracle as O
    cfg = O.sd35_medium()
    cores = R.pick_cores()
    R.pin(cores)
    T, g, n_text = args.num_inference_steps, args.guidance, args.n_text
    ni = (args.height // 16) * (args.width // 16)
    kind = "reference" if R.available() else "port"
    dev = "cuda" if torch.cuda.is_available() else "cpu"
    w = {k: v.cpu() for k, v in O.make_weights(cfg, seed=0, dtype=torch.bfloat16, device=dev).items()}
    info = {"cores": cores["n"], "cpu_model": cores["model"], "logical_cpus_allowed": cores["logical_allowed"], "kind": kind}
    if kind == "port":
        return _cpu_port(args, cfg, w, cores, info, steps, warmup)
    model = R.build_model(cfg, w)
    del w
    lin, att = O.flops_per_forward(cfg, ni, n_text)
    # calibration on 2 blocks (also warms oneDNN's primitive cache for these shapes)
    m2 = R.truncated(model, 2)
    R.time_c2_step(cfg, m2, g, n_text, args.height, T)
    t2 = min(R.time_c2_step(cfg, m2, g, n_text, args.height, T) for _ in range(2))
    est_full = t2 * (lin + att) / R.block_flops(cfg, ni, n_text, 2)
    L = cfg.num_layers if est_full <= CPU_STEP_BUDGET_S else max(2, min(cfg.num_layers, int(cfg.num_layers * CPU_STEP_BUDGET_S / est_full)))
    mL = model if L == cfg.num_layers else R.truncated(model, L)
    scale = 1.0 if L == cfg.num_layers else (lin + att) / R.block_flops(cfg, ni, n_text, L)
    for _ in range(max(0, warmup)):
        R.time_c2_step(cfg, mL, g, n_text, args.height, T)
    n = max(1, min(steps, CPU_MAX_SAMPLES))
    times = [R.time_c2_step(cfg, mL, g, n_text, args.height, T) for _ in range(n)]
    best = min(times) * scale
    value = 1.0 / (best * T)
    info.update({"value": value, "unit": "latents/s", "c2_step_s": best, "c2_step_samples_s": [round(t * scale, 3) for t in times],
                 "sample": (f"{n} timed samples (min taken) of ONE full C2 denoising step at B=1 (CFG: 2 forwards of the real SD3Transformer2DModel at "
                            f"{args.height}^2 + scheduler.step, bf16 CPU autocast)" + ("" if L == cfg.num_layers else f", first {L} of {cfg.num_layers} blocks scaled by FLOPs") +
                            f", x{T} steps; {cores['n']} threads pinned to the physical cores of one NUMA node")})
    if full:
        R.time_c1_full(cfg, model)                                   # warm the 256^2 shapes
        c1_s, c1_v = R.time_c1_full(cfg, model)
        info["c1_full"] = {"seconds": c1_s, "latents_per_s": c1_v, "config": "SD3.5-medium 256^2 4-step, B=1, guidance 1.0, CPU bf16 autocast, timed in full"}
    return info, sum(times) / len(times)


def gpu_eager_reference(args, B, cfg_on):
    """Informational: the reference NUMERICS run eagerly on this GPU - the oracle's transformer forward (the reference's torch ops in the
    reference's order: F.linear / cuBLAS, F.scaled_dot_product_attention, F.layer_norm ...) under CUDA bf16 autocast at the bench's
    forward batch, timed with CUDA events; latents/s = B / (T x forward) ignores the scheduler step and every host sync of the reference
    loop, so it flatters the reference.  Part of the reference leg (the only place bench.py may execute oracle/)."""
    try:
        from oracle import sd3_oracle as O
        cfg = O.sd35_medium()
        dev = "cuda"
        w = O.make_weights(cfg, seed=0, dtype=torch.bfloat16, device=dev)
        Bp = B * (2 if cfg_on else 1)
        lat = args.height // 8
        g = torch.Generator(device=dev).manual_seed(3)
        x = torch.randn(Bp, cfg.in_channels, lat, lat, generator=g, device=dev).half()
        pe = torch.randn(Bp, args.n_text, cfg.joint_attention_dim, generator=g, device=dev).bfloat16()
        pp = torch.randn(Bp, cfg.pooled_projection_dim, generator=g, device=dev).bfloat16()
        tt = torch.full((Bp,), 612.5, device=dev).half()
        def fwd():
            with torch.no_grad(), torch.autocast("cuda", dtype=torch.bfloat16):
                return O.transformer_forward(w, cfg, x, pe, pp, tt)
        fwd(); fwd()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); fwd(); fwd(); fwd(); e1.record(); torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / 3
        del w
        torch.cuda.empty_cache()
        return {"ms_per_forward": ms, "forward_batch": Bp, "value": B / (args.num_inference_steps * ms / 1e3), "unit": "latents/s",
                "what": "oracle transformer forward (reference numerics, torch eager: cuBLAS + SDPA) under CUDA bf16 autocast; no scheduler step, no host syncs"}
    except Exception as exc:                        # informational only
        return {"unavailable": f"{type(exc).__name__}: {exc}"}


def _cpu_port(args, cfg, w, cores, info, steps, warmup):
    """oracle/_ref absent: the oracle port's 2-block sample (round-1 method), min of the timed samples."""
    from oracle import sd3_oracle as O
    T, g, n_text, res = args.num_inference_steps, args.guidance, args.n_text, args.height
    lat = res // 8
    ni = (lat // 2) ** 2
    inp = O.make_inputs(cfg, 1, lat, lat, n_text, seed=1)
    ts, sig = O.make_schedule(T, 3.0)
    x = inp["x0"].half()

    def sample():
        t0 = time.perf_counter()
        with torch.no_grad(), torch.autocast("cpu", dtype=torch.bfloat16):
            v = O.transformer_forward(w, cfg, x, inp["prompt_embeds"].bfloat16(), inp["pooled"].bfloat16(), ts[3].expand(1).half(), max_layers=2)
        O.sde_step(v, x, (ts[3] / 1000).item(), (ts[4] / 1000).item(), 0.7, float(sig[1]), noise=torch.randn(x.shape), compute_log_prob=True)
        return time.perf_counter() - t0
    for _ in range(max(1, warmup)):
        sample()
    times = [sample() for _ in range(max(1, min(steps, CPU_MAX_SAMPLES)))]
    from oracle import ref_runner as R
    lin, att = O.flops_per_forward(cfg, ni, n_text)
    t_fwd = min(times) * (lin + att) / R.block_flops(cfg, ni, n_text, 2)
    value = 1.0 / (t_fwd * T * (2 if g > 1.0 else 1))
    info.update({"value": value, "unit": "latents/s",
                 "sample": f"oracle PORT (oracle/_ref absent): 2 of 24 blocks of one forward at {res}^2 B=1 + scheduler.step, scaled by FLOPs, x{T} x{2 if g > 1 else 1}"})
    return info, sum(times) / len(times)


def run_reference(args):
    """`--impl reference`: the reference's own CPU implementation of the path on this box's host cores (see cpu_reference)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    t0 = time.perf_counter()
    info, mean_sample_s = cpu_reference(args, steps=args.steps, warmup=max(2, args.warmup), full=True)
    wall = time.perf_counter() - t0
    T = args.num_inference_steps
    line = {"metric": METRIC, "value": info["value"], "unit": "latents/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1000.0 * mean_sample_s, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "bf16", "data": "synthetic", "impl": "reference",
            "config": {"workload": f"SD3.5-medium {args.height}x{args.width} {T}-step GRPO rollout, guidance {args.guidance}, random-init weights",
                       "timing": "host wall clock; a step = one bounded sample (see cpu_baseline.sample)", "wall_s": wall},
            "cpu_baseline": info,
            "e2e": {"value": info["value"], "unit": "latents/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def time_roofline_kernels(cfg, args, dev, B, cfg_on, ni):
    """Isolated launches of the two roofline kernels at the bench shapes (CUDA events on the launching stream, 256 MB L2 flush between
    repetitions, median of 10 after 3 warm-ups): the MLP-up GEMM (bias + GELU epilogue) and the joint attention exactly as the engine
    launches it (RMS-normed q / k heads, keys pre-scaled by softmax_scale * log2(e) in the QKV GEMM epilogue, csrc/softmax.cuh).  Returns (gemm_ms, (M, N, K), att_ms | None, note)."""
    from flow_factory_b200.ops import linear as op_linear
    Bp = B * (2 if cfg_on else 1)
    M, N, K = Bp * ni, 4 * cfg.inner_dim, cfg.inner_dim
    A = torch.randn(M, K, device=dev).bfloat16(); Wt = (torch.randn(N, K, device=dev) / K ** 0.5).bfloat16()
    bb = torch.zeros(N, device=dev).bfloat16(); oo = torch.empty(M, N, device=dev, dtype=torch.bfloat16)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def median_ms(fn):
        for _ in range(3):
            fn()
        ts = []
        for _ in range(10):
            flush.zero_()
            a, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(); fn(); b_.record(); torch.cuda.synchronize()
            ts.append(a.elapsed_time(b_))
        return sorted(ts)[len(ts) // 2]
    gemm_ms = median_ms(lambda: op_linear(A, Wt, bb, oo, epi=1))
    del A, Wt, oo
    att_ms, note = None, None
    try:
        # the engine's own launch (ffb200_attention_normed): q / k heads as the QKV epilogue leaves them - per-head RMS-normed (unit weights
        # here, as in the random-init model), keys pre-scaled by softmax_scale * log2(e)
        from flow_factory_b200.ops import attention_normed as op_attention
        S_joint, Hh = ni + args.n_text, cfg.num_attention_heads
        x = torch.randn(Bp, S_joint, 3, Hh, 64, device=dev)
        x[:, :, :2] = x[:, :, :2] * torch.rsqrt(x[:, :, :2].pow(2).mean(-1, keepdim=True) + 1e-6)
        x[:, :, 1] *= 64 ** -0.5 * 1.4426950408889634
        qkv = x.reshape(Bp, S_joint, 3 * cfg.inner_dim).bfloat16()
        del x
        w_norm = torch.ones(64, device=dev).bfloat16()
        ao = torch.empty(Bp, S_joint, cfg.inner_dim, device=dev, dtype=torch.bfloat16)
        att_ms = median_ms(lambda: op_attention(qkv, Hh, w_norm, w_norm, out=ao))
        del qkv, ao
    except Exception as exc:   # the attention micro-timing is reporting only: never lose the bench line over it
        note = f"{type(exc).__name__}: {exc}"
    del flush
    torch.cuda.empty_cache()
    return gemm_ms, (M, N, K), att_ms, note


# ------------------------------------------------------------------------------------------------ our arm
def run_b200(args):
    import torch.distributed as dist
    from flow_factory_b200 import FlowMatchEulerDiscreteSDEScheduler, RolloutEngine, _lib
    from flow_factory_b200.adapter import B200SD3_5Adapter
    from flow_factory_b200.dist import all_gather_rollout
    from flow_factory_b200.trajectory import compute_trajectory_indices
    from flow_factory_b200.synth import random_inputs, random_weights, sd35_medium   # the engine arm never touches oracle/

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    torch.manual_seed(1 + rank)     # the adapter draws each rollout's noise seed from the global generator: same arguments, same noise
    cfg = sd35_medium()
    T, B = args.num_inference_steps, args.batch
    lat_h, lat_w = args.height // 8, args.width // 8
    ni = (lat_h // 2) * (lat_w // 2)
    cfg_on = args.guidance > 1.0
    w = random_weights(cfg, seed=0, dtype=torch.bfloat16, device=f"cuda:{local}")
    sched = FlowMatchEulerDiscreteSDEScheduler(noise_level=0.7, shift=3.0, num_sde_steps=args.num_sde_steps, seed=42)
    adapter = B200SD3_5Adapter(cfg, w, device=dev, scheduler=sched, rng="philox", use_graph=not args.no_graph)
    adapter.rollout()
    del w
    sched.set_timesteps(T, seq_len=ni)
    traj_idx = compute_trajectory_indices(sched.train_timesteps, T)
    inp = random_inputs(cfg, B, lat_h, lat_w, args.n_text, seed=1 + rank, device=dev)
    kw = dict(height=args.height, width=args.width, num_inference_steps=T, guidance_scale=args.guidance, compute_log_prob=True,
              trajectory_indices=traj_idx)

    def rollout_device():
        s = adapter.inference(prompt_embeds=inp["prompt_embeds"], pooled_prompt_embeds=inp["pooled"],
                              negative_prompt_embeds=inp["neg_prompt_embeds"], negative_pooled_prompt_embeds=inp["neg_pooled"],
                              latents=inp["x0"], **kw)
        if world > 1:   # the single collective of the path: one all-gather of {kept latents | log-probs} per rollout
            lat = torch.stack([x.all_latents for x in s]); lp = torch.stack([x.log_probs for x in s])
            all_gather_rollout(lat, lp)
        return s

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---------------- the two roofline kernels, each timed ALONE on an idle GPU (burst peak is the matching denominator) ----------------
    roof_cold = time_roofline_kernels(cfg, args, dev, B, cfg_on, ni) if rank == 0 else None
    barrier()

    # ---------------- device-resident timing ----------------
    for _ in range(args.warmup):
        rollout_device()
    barrier()
    launches_per_rollout = RolloutEngine.last_launch_count()
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_wall = time.perf_counter()
    e0.record()
    for _ in range(args.steps):
        last = rollout_device()
    e1.record()
    barrier()
    wall = time.perf_counter() - t_wall
    ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms_total = float(ms)
    clk = clocks.stop() if rank == 0 else None
    value = world * B * args.steps / (ms_total / 1e3)
    if args.dump_outputs and rank == 0:       # now: the legs below reuse the engine's output buffers
        stack = lambda name: None if getattr(last[0], name) is None else torch.stack([getattr(x, name) for x in last])
        dump_outputs(args.dump_outputs, {"all_latents": stack("all_latents"), "log_probs": stack("log_probs"),
                                         "final_latents": stack("final_latents"), "timesteps": last[0].timesteps})

    # ---------------- the same rollout with the WHOLE SDE window noisy (num_sde_steps = T - 1 = 29: noise + log-prob on every step but the
    # last; SURVEY 8d asks for {1, 29}) - one warm-up (the graph is re-used, only the step coefficients change), then timed ----------------
    sde_all = None
    if args.num_sde_steps is not None and args.steps > 0:
        sched._num_sde_steps = None
        sched.set_timesteps(T, seq_len=ni)
        kw_all = dict(kw, trajectory_indices=compute_trajectory_indices(sched.train_timesteps, T))      # every step is a train timestep now

        def rollout_all():
            s = adapter.inference(prompt_embeds=inp["prompt_embeds"], pooled_prompt_embeds=inp["pooled"],
                                  negative_prompt_embeds=inp["neg_prompt_embeds"], negative_pooled_prompt_embeds=inp["neg_pooled"],
                                  latents=inp["x0"], **kw_all)
            if world > 1:
                all_gather_rollout(torch.stack([x.all_latents for x in s]), torch.stack([x.log_probs for x in s]))
            return s
        rollout_all(); barrier()
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        f0.record(); s_all = rollout_all(); f1.record(); barrier()
        ms_all = torch.tensor([f0.elapsed_time(f1)], device=dev)
        if world > 1:
            dist.all_reduce(ms_all, op=dist.ReduceOp.MAX)
        sde_all = {"num_sde_steps": T - 1, "value": world * B / (float(ms_all) / 1e3), "unit": "latents/s", "ms_per_step": float(ms_all),
                   "log_probs_per_sample": int(s_all[0].log_probs.numel()), "latents_kept_per_sample": int(s_all[0].all_latents.shape[0])}
        sched._num_sde_steps = args.num_sde_steps
        sched.set_timesteps(T, seq_len=ni)
        rollout_device(); barrier()

    # ---------------- end to end through the public API with host buffers ----------------
    host = {k: v.cpu().pin_memory() for k, v in inp.items() if k != "x0"}
    h2d = sum(v.numel() * v.element_size() for v in host.values())

    def rollout_e2e():
        s = adapter.inference(prompt_embeds=host["prompt_embeds"].to(dev, non_blocking=True),
                              pooled_prompt_embeds=host["pooled"].to(dev, non_blocking=True),
                              negative_prompt_embeds=host["neg_prompt_embeds"].to(dev, non_blocking=True),
                              negative_pooled_prompt_embeds=host["neg_pooled"].to(dev, non_blocking=True), **kw)
        lat = torch.stack([x.all_latents for x in s]); lp = torch.stack([x.log_probs for x in s])
        fin = torch.stack([x.extra_kwargs["final_latents"] for x in s])
        if world > 1:
            lat, lp = all_gather_rollout(lat, lp)
        out = (lat.cpu(), lp.cpu(), fin.cpu())     # device -> host read of the rollout's result
        return sum(t.numel() * t.element_size() for t in out)

    d2h = rollout_e2e()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        rollout_e2e()
    barrier()
    e2e_s = torch.tensor([time.perf_counter() - t0], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(e2e_s, op=dist.ReduceOp.MAX)
    e2e_value = world * B * args.steps / float(e2e_s)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---------------- rooflines: the tcgen05 GEMM (MLP-up shape of this batch) and the joint attention ----------------
    # `achieved` / `frac`: the kernel timed alone before the rollouts (idle GPU, full clocks) against the measured BURST cuBLAS figure;
    # `achieved_after_rollouts`: the same launches repeated right after the timed rollouts, when the GPU sits at its power cap (see `clocks`),
    # against the SUSTAINED figure - the state the kernel runs in inside a step.
    peaks, peak_kind = load_peaks()
    roof_hot = time_roofline_kernels(cfg, args, dev, B, cfg_on, ni)
    gemm_ms, (M, N, K), att_ms, att_note = roof_cold
    gemm_ms_hot, _, att_ms_hot, _ = roof_hot
    Bp = B * (2 if cfg_on else 1)
    gemm_tf, gemm_tf_hot = 2.0 * M * N * K / gemm_ms / 1e9, 2.0 * M * N * K / gemm_ms_hot / 1e9
    fl_latent = flops_per_latent(cfg, ni, args.n_text, T, cfg_on)
    step_tf = value * fl_latent / 1e12
    shares = launch_shares()
    # DRAM bytes of one launch of this kernel from the committed `ncu --set full` capture of this shape (profiles/ncu_traffic.json), else null.
    # Algorithmic bytes of the launch: A + W + out = 2 * (M*K + N*K + M*N).
    traffic = ncu_traffic("gemm_mlp_up", f"{M}x{N}x{K}")
    roofline_gemm = {"bound": "tensor", "kernel": "gemm_bf16_kernel<256> (MLP up, bias+GELU epilogue)", "achieved": gemm_tf,
                     "peak": peaks["bf16_tflops"], "unit": "TFLOP/s", "frac": gemm_tf / peaks["bf16_tflops"], "traffic": traffic,
                     "traffic_unit": "bytes/launch (ncu dram read+write)", "algorithmic_bytes_per_launch": 2.0 * (M * K + N * K + M * N),
                     "peak_source": f"{peak_kind} cuBLAS bf16 burst", "flops_per_launch": 2.0 * M * N * K, "launch_ms": gemm_ms,
                     "achieved_after_rollouts": gemm_tf_hot, "frac_of_sustained_after_rollouts": gemm_tf_hot / peaks["bf16_tflops_sustained"],
                     "time_share_of_step": shares.get("gemm")}
    # The single kernel shape with the largest TIME share of the step is the joint attention: it is the `roofline` entry; the GEMM kernel
    # (the larger share over all its launches since round 2) is reported beside it as `roofline_gemm` at its most FLOP-heavy shape.
    whole = {"whole_step_achieved_per_gpu": step_tf / world, "whole_step_frac_of_sustained": step_tf / world / peaks["bf16_tflops_sustained"],
             "flops_per_latent": fl_latent}
    if att_ms is not None and att_ms_hot is not None:
        S_joint, Hh = ni + args.n_text, cfg.num_attention_heads
        att_fl = 4.0 * Bp * Hh * S_joint * S_joint * 64
        att_tf, att_tf_hot = att_fl / att_ms / 1e9, att_fl / att_ms_hot / 1e9
        roofline = {"bound": "tensor", "kernel": "attention_kernel (joint image+text attention, head_dim 64)", "achieved": att_tf,
                    "peak": peaks["bf16_tflops"], "unit": "TFLOP/s", "frac": att_tf / peaks["bf16_tflops"],
                    "traffic": ncu_traffic("attention_d64", f"{Bp}x{S_joint}x{Hh}"), "traffic_unit": "bytes/launch (ncu dram read+write)",
                    "algorithmic_bytes_per_launch": 2.0 * Bp * S_joint * 4 * cfg.inner_dim, "peak_source": f"{peak_kind} cuBLAS bf16 burst",
                    "flops_per_launch": att_fl, "launch_ms": att_ms,
                    "achieved_after_rollouts": att_tf_hot, "frac_of_sustained_after_rollouts": att_tf_hot / peaks["bf16_tflops_sustained"],
                    "time_share_of_step": shares.get("attention"),
                    "note": "SIMT-softmax-limited at head_dim 64 (MUFU and FMA pipes balanced, DESIGN.md section 4; cuDNN SDPA on the same shape: 0.53 of the measured burst peak), "
                            "see DESIGN.md section 4 / profiles/r02_attention_experiments.md", **whole}
    else:
        roofline = dict(roofline_gemm, note=f"attention roofline unavailable ({att_note}); GEMM reported instead", **whole)

    # ---------------- CPU baseline: the reference's own classes on this box's host cores, bounded sample (rank 0, N=1 only) ----------------
    cpu = None
    if not args.skip_cpu_baseline and world == 1:
        cpu, _ = cpu_reference(args, steps=3, warmup=2, full=True)
        cpu["gpu_eager_reference"] = gpu_eager_reference(args, B, cfg_on)

    line = {"metric": METRIC, "value": value, "unit": "latents/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
            "data": "synthetic", "impl": "b200",
            "config": {"workload": f"SD3.5-medium {args.height}x{args.width} {T}-step GRPO rollout (Flow-SDE, noise 0.7, num_sde_steps {args.num_sde_steps}), "
                                   f"guidance {args.guidance}, {args.n_text} text tokens, random-init weights",
                       "per_rank_batch": B, "global_batch": B * world, "parallelism": f"dp{world} (prompt-sharded, 1 all-gather/rollout)",
                       "l2": "working set >> 126 MB L2 (4.5 GB weights re-read every forward)", "cuda_graph": not args.no_graph,
                       "rng": "in-kernel Philox4x32-10"},
            "clocks": clk,
            "e2e": {"value": e2e_value, "unit": "latents/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
            "gpu_launches": int(launches_per_rollout * args.steps),
            "roofline": roofline, "roofline_gemm": roofline_gemm, "cpu_baseline": cpu, "sde_window_all": sde_all,
            "wall_s_timed_region": wall}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def run_other_config(args):
    """BASELINE configs 3-5 behind the same entry point: hands over (same process, so torchrun's environment carries) to the model's
    bench tool, which prints one JSON line with the same contract (metric, value, e2e, clocks, gpu_launches, roofline ...)."""
    import runpy
    tool, extra = {
        "flux1": ("tools/flux_bench.py", ["--num-inference-steps", "28"]),                       # FLUX.1-dev 1024^2 28-step
        "wan21": ("tools/wan_bench.py", ["--frames", "49", "--num-inference-steps", "40"]),      # Wan2.1-T2V-1.3B 480p 49-frame 40-step
        "qwen_image": ("tools/qwen_bench.py", ["--num-inference-steps", "50"]),                  # Qwen-Image 20B 1024^2 50-step DGPO (ODE)
    }[args.config]
    sys.argv = [os.path.join(ROOT, tool), "--gpus", str(args.gpus), "--steps", str(args.steps), "--warmup", str(args.warmup)] + extra
    runpy.run_path(sys.argv[0], run_name="__main__")


def main():
    args = parse()
    if args.dump_outputs and (args.impl != "b200" or args.config != "sd35"):
        raise SystemExit("--dump-outputs is implemented for the engine arm of the sd35 config")
    if args.impl == "reference":
        run_reference(args)
    else:
        if not torch.cuda.is_available():
            raise SystemExit("bench.py needs a B200 (no CPU fallback for the engine arm); use --impl reference for the CPU baseline")
        if args.config != "sd35":
            run_other_config(args)
        else:
            run_b200(args)


if __name__ == "__main__":
    main()
