#!/usr/bin/env python
"""bench.py — imagined frames/s of the DIAMOND sampler hot path on B200 (BASELINE.json metric).

A "step" = one DiffusionSampler.sample() call over a batch of `--envs` imagined environments per GPU
(frame-stack 4 x 64x64x3 fp32 + 4 actions -> next frame, 3 Euler denoising steps = 3 U-Net forwards).
`value` is device-resident throughput, `e2e` the same call with pinned HOST buffers in and out, `roofline` the dominant conv
kernel timed alone.  Secondary blocks on the same line (each under a watchdog, so the headline line is always printed):
`train_denoiser` (cfg 2: Denoiser.forward + backward + ONE flat-buffer NCCL all-reduce + clip + AdamW, + the wgrad kernel's
roofline), `imagination_update` (cfg 3: 32 envs x horizon 15 through WorldModelEnv + policy BPTT + all-reduce + AdamW),
`gpu_baseline` (the reference's GPU path on this GPU: eager and torch.compile), `cpu_baseline` (its CPU path on the host cores).
Multi-GPU is weak scaling: imagination needs no collective (SURVEY.md 8e); both training blocks all-reduce their gradients.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--envs B] [--impl native|reference] [--dump-outputs DIR]

Prints ONE JSON line (rank 0).  `--impl reference` times the reference algorithm's CPU path (the oracle port — the
reference is pure Python and /root/reference does not travel to the GPU box) on the host cores.

`--dump-outputs DIR` also writes what the last timed sample() call returned (rank 0's environments) as DIR/x.npy and
DIR/trajectory.npy.  Inputs and sampler noise are seeded, so two builds run with the same arguments can be compared output
for output.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the benchmark writes nothing into the tree it runs from (which may be read-only)

METRIC = "imagined frames/sec (64x64, 3 denoise steps)"
GFLOP_PER_FRAME = 18.266  # SURVEY.md 8d: 3 x 6.0888 GFLOP denoiser forwards
TRS = os.environ.get("DMD_CONV_TRS", "0") != "0"  # the executor's weight layout for 3x3 convs (tap-major; DMD_CONV_TRS=1 selects the tap-row-stacked experiment)
DUMP_LIMIT_BYTES = 64 << 20


def load_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return p, "measured (MEASURED_PEAKS.json)"
    except Exception:
        return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback (B200_PROFILING.md)"


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons sampled every 200 ms while the timed region runs."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag = index, [], threading.Event()

    def run(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i",
                                          str(self.index), "-lms", "200"], stdout=subprocess.PIPE, text=True)
            for line in self.proc.stdout:
                self.rows.append([x.strip() for x in line.split(",")])
                if self.stop_flag.is_set():
                    break
        except Exception:
            pass

    def finish(self):
        self.stop_flag.set()
        try:
            self.proc.terminate()
        except Exception:
            pass
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                continue
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def build_oracle_model(depths=(2, 2, 2, 2)):
    from oracle import torch_oracle as O

    inner = O.InnerCfg(depths=list(depths))
    sd = O.seeded_state_dict(O.inner_model_shapes(inner), 2024)
    return O, inner, sd


def pick_cpu_threads():
    """torch's CPU convolutions stop scaling (and collapse) with very many intra-op threads on these small images, so the
    baseline gets the thread count that is FASTEST for it among {8, 16, 32, 64, all}: fair to the reference."""
    import torch

    avail = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    O, inner, sd = build_oracle_model()
    cfg = O.DenoiserCfg(inner=inner)
    obs, act, x0 = O.synthetic_inputs(2, inner, 64, 64, 5)
    sig = torch.tensor([1.0, 1.0])
    best, best_t = None, None
    for th in sorted({t for t in (8, 16, 32, 64, avail) if t <= avail}):
        torch.set_num_threads(th)
        with torch.no_grad():
            O.model_output(x0, sig, obs.reshape(2, -1, 64, 64), act, sd, cfg)
            t0 = time.perf_counter()
            O.model_output(x0, sig, obs.reshape(2, -1, 64, 64), act, sd, cfg)
            dt = time.perf_counter() - t0
        if best_t is None or dt < best_t:
            best, best_t = th, dt
        if dt > 4 * best_t:
            break
    return best, avail


def cpu_frames_per_s(envs: int, repeats: int, threads: int):
    """Reference algorithm on the host cores: oracle port of DiffusionSampler.sample (3 Euler steps), fp32."""
    import torch

    O, inner, sd = build_oracle_model()
    torch.set_num_threads(threads)
    cfg, sc = O.DenoiserCfg(inner=inner), O.SamplerCfg(3)
    obs, act, x0 = O.synthetic_inputs(envs, inner, 64, 64, 5)
    times = []
    with torch.no_grad():
        O.sample(obs[:1], act[:1], x0[:1], sd, cfg, sc)  # warm-up (thread pool, oneDNN primitives)
        for _ in range(repeats):
            t0 = time.perf_counter()
            O.sample(obs, act, x0, sd, cfg, sc)
            times.append(time.perf_counter() - t0)
    return envs / statistics.median(times), times


def run_reference(args):
    """--impl reference: CPU path of the reference algorithm; rank 0 only."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch

    cores, avail = pick_cpu_threads()
    envs = args.envs  # the declared workload (CPU throughput is flat in batch, so this costs ~1.5 s per sample())
    O, inner, sd = build_oracle_model()
    torch.set_num_threads(cores)
    cfg, sc = O.DenoiserCfg(inner=inner), O.SamplerCfg(3)
    obs, act, x0 = O.synthetic_inputs(envs, inner, 64, 64, 5)
    steps = args.steps
    warmups = 0
    with torch.no_grad():
        for _ in range(max(1, min(args.warmup, 2))):
            t0 = time.perf_counter()
            O.sample(obs, act, x0, sd, cfg, sc)
            t_one = time.perf_counter() - t0
            warmups += 1
            if t_one > 15.0:      # a host shared with other jobs: at most one warm-up of a slow arm
                break
        t0 = time.perf_counter()
        for _ in range(steps):
            x, traj = O.sample(obs, act, x0, sd, cfg, sc)
        dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, x, torch.stack(traj))
    val = envs * steps / dt
    sample = f"{envs} envs x {steps} sample() calls (the full {args.envs}-env workload per step), torch {torch.__version__} CPU fp32, {cores} threads (fastest of 8/16/32/64/{avail} available)"
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": val, "unit": "frames/s", "n_gpus": args.gpus, "steps": steps,
        "warmup": warmups, "ms_per_step": 1e3 * dt / steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "fp32", "data": "synthetic",
        "config": workload_config(args),
        "cpu_baseline": {"value": val, "unit": "frames/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": val, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def dump_outputs(out_dir: str, x, traj) -> None:
    """What one sample() call returned -- the next frames x (B, C, H, W) and the denoising trajectory (num_sigmas, B, C, H, W)
    -- as float32 out_dir/x.npy and out_dir/trajectory.npy.  When the two exceed DUMP_LIMIT_BYTES, a fixed seeded subset of
    the B environments is written (the same rows of both, in ascending order)."""
    import numpy as np
    import torch

    b = x.shape[0]
    per_env = 4 * (x[0].numel() + traj[:, 0].numel())
    keep = min(b, DUMP_LIMIT_BYTES // per_env)
    rows = np.arange(b) if keep == b else np.sort(np.random.default_rng(0).choice(b, keep, replace=False))
    rows = torch.from_numpy(rows).to(x.device)
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "x.npy"), x.index_select(0, rows).float().cpu().numpy())
    np.save(os.path.join(out_dir, "trajectory.npy"), traj.index_select(1, rows).float().cpu().numpy())


def workload_config(args, envs_override=None):
    envs = envs_override or args.envs
    return {"workload": "DiffusionSampler.sample: Breakout-shape imagination, frame-stack 4, 64x64x3, 3 Euler denoise steps, "
                        "default agent config (4.4 M-param U-Net), random-init de-zeroed weights",
            "envs_per_gpu": envs, "global_envs": envs * args.gpus, "parallelism": f"dp{args.gpus} (independent envs per rank, no collective)",
            "l2": "256 MiB L2 flush between timed steps (untimed)", "cuda_graph": True, "programmatic_dependent_launch": True}


def rank_inputs(envs: int, rank: int):
    """Synthetic frame stacks / actions of one rank (weak scaling: every rank imagines its own envs)."""
    from diamond_b200.synthetic import frame_stacks

    obs, act, _ = frame_stacks(envs, 4, 3, 64, 64, 4, 100 + rank)
    return obs, act


def max_over_ranks(values, device):
    """Device timings are reduced with MAX over ranks (a multi-GPU step is as slow as its slowest rank)."""
    import torch
    import torch.distributed as dist

    t = torch.tensor(values, device=device, dtype=torch.float64)
    if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return [float(v) for v in t]


def whole_job_value(frames_per_rank: int, world: int, ms: float) -> float:
    return frames_per_rank * world / (ms * 1e-3)


def conv_roofline(dev, envs, peaks, peaks_src):
    """Dominant kernel: conv_tc_kernel<64>, 3x3 64->64 at 64x64 (Appendix A row 2; 8 launches per forward + the 128->64
    and upsample variants share the code).  Timed live with CUDA events on the launching stream, rotating through
    buffer sets larger than L2."""
    import torch

    from diamond_b200 import ops

    g = torch.Generator().manual_seed(0)
    wt = (torch.randn(64, 64, 3, 3, generator=g) / 24).to(dev)
    wpk, cp = ops.pack_conv_weight(wt, 64, trs=TRS)
    bias = torch.zeros(64, device=dev)
    nset = 6  # rotating operand / output sets: 6 x (17 MB operand + 33.5 MB output) at 32 envs > 126 MB L2
    xs = [torch.randn(envs, 64, 64, 64, device=dev) for _ in range(nset)]
    film = torch.randn(envs, 128, device=dev) * 0.1
    sts = [ops.gn_stats(x, 32) for x in xs]
    outs = [torch.empty(envs, 64, 64, 64, device=dev) for _ in range(nset)]
    ost = [torch.zeros(envs, 2, 2, device=dev, dtype=torch.float64) for _ in range(nset)]
    opnd = [ops.prep_act(xs[i], mode=1, silu=True, stats0=sts[i], gs0=32, film=film)[0] for i in range(nset)]
    iters = 24

    def launch(i):
        k = i % nset
        ops.conv2d_operand(opnd[k], None, 64, 0, envs, 64, 64, wpk, 64, cp, bias=bias, out_gs=32, out=outs[k], ostats=ost[k], trs=TRS)

    def launch_prep(i):
        k = i % nset
        ops.prep_act(xs[k], mode=1, silu=True, stats0=sts[k], gs0=32, film=film)

    def time_graph(fn):
        for i in range(5):
            fn(i)
        torch.cuda.synchronize()
        # Python call overhead exceeds the kernel time, so the launches are captured in a CUDA graph and the replay is
        # what is timed (events on the replay stream)
        graph = torch.cuda.CUDAGraph()
        side = torch.cuda.Stream()
        with torch.cuda.stream(side):
            with torch.cuda.graph(graph, stream=side):
                for i in range(iters):
                    fn(i)
            torch.cuda.synchronize()
            graph.replay()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            reps = 5
            e0.record(side)
            for _ in range(reps):
                graph.replay()
            e1.record(side)
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / (iters * reps)

    ms = time_graph(launch)
    ms_prep = time_graph(launch_prep)
    flops = 2.0 * 576 * 64 * 4096 * envs
    traffic, traffic_src = conv_traffic_from_profile()
    achieved = flops / (ms * 1e-3) / 1e12
    peak = float(peaks.get("bf16_tflops", 1590.0))
    return {"bound": "tensor", "kernel": ("conv_tc_kernel<256,3> (tap-row-stacked: 3 MMAs of N=192 per slab)" if TRS else "conv_tc_kernel<64,0> (tap-major: 9 MMAs of N=64 per slab)") + " 3x3 64->64 @64x64 on a PLC16 fp16 operand, bias + GroupNorm-stats epilogue",
            "prep_us_per_launch": ms_prep * 1e3,
            # the operand pass that precedes every conv (GroupNorm / FiLM / SiLU -> fp16 PLC16): HBM-bound; algorithmic bytes =
            # 256 B read (fp32 NHWC, 64 channels) + 128 B written per pixel
            "prep": {"bound": "hbm", "kernel": "prep_fast_kernel<8,0>", "achieved": (256.0 + 128.0) * 4096.0 * envs / (ms_prep * 1e-3) / 1e9,
                     "peak": float(peaks.get("hbm_gbs", 6650.0)), "unit": "GB/s",
                     "frac": (256.0 + 128.0) * 4096.0 * envs / (ms_prep * 1e-3) / 1e9 / float(peaks.get("hbm_gbs", 6650.0))},
            "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
            "traffic": traffic, "traffic_source": traffic_src, "algorithmic_bytes": (128 * 1.0 + 256) * 4096.0 * envs,
            "us_per_launch": ms * 1e3, "flop_per_launch": flops, "peak_source": peaks_src + " bf16 burst (fp16 and bf16 share the tensor-pipe rate)"}


def gpu_baseline(dev, envs: int, steps: int = 5):
    """The reference's own GPU path on this B200 (what north_star's ">= 50x" is stated against, SURVEY.md 8d): the oracle
    port of DiffusionSampler.sample (same torch ops as the reference modules: cuDNN convs, ATen norms, cuBLAS linears) on
    `dev`, fp32 with TF32 matmul (src/trainer.py:41), in the reference's two modes: eager, and the per-step denoise under
    torch.compile(mode="reduce-overhead") (src/trainer.py:182-184, its default).  /root/reference cannot travel to the GPU
    box, so the port stands in for it; it runs the reference's per-step device->host syncs (diffusion_sampler.py:39,47)."""
    import torch

    O, inner, sd = build_oracle_model()
    torch.backends.cuda.matmul.allow_tf32 = True
    sdd = {k: v.to(dev) for k, v in sd.items()}
    cfg, sc = O.DenoiserCfg(inner=inner), O.SamplerCfg(3)
    obs, act, _ = O.synthetic_inputs(envs, inner, 64, 64, 5)
    obs, act = obs.to(dev), act.to(dev)
    b, t, c, h, w = obs.shape
    prev_obs = obs.reshape(b, t * c, h, w)
    sigmas = O.build_sigmas(sc.num_steps_denoising, sc.sigma_min, sc.sigma_max, sc.rho).to(dev)

    def denoise_eager(x, sigma):
        return O.denoise(x, sigma, prev_obs, act, sdd, cfg)

    def sample(denoise_fn):
        x = torch.randn(b, c, h, w, device=dev)
        for sigma, next_sigma in zip(sigmas[:-1], sigmas[1:]):
            gamma = 0.0 if not (0 <= sigma <= float("inf")) else 0.0  # s_churn = 0; keeps the reference's host sync (:39)
            sigma_hat = sigma * (gamma + 1)
            denoised = denoise_fn(x, sigma)
            d = (x - denoised) / sigma_hat
            dt = next_sigma - sigma_hat
            if next_sigma == 0:  # host sync (:47)
                x = x + d * dt
            else:
                x = x + d * dt
        return x

    def timed(fn, n):
        with torch.no_grad():
            for _ in range(3):
                sample(fn)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(n):
                sample(fn)
            e1.record()
            torch.cuda.synchronize()
        return envs * n / (e0.elapsed_time(e1) * 1e-3)

    out = {"unit": "frames/s", "envs": envs, "steps": steps, "dtype": "fp32, TF32 matmul (src/trainer.py:41)",
           "kind": "port (oracle restatement of the reference modules run on cuda; torch " + torch.__version__ + ")"}
    try:
        out["eager"] = timed(denoise_eager, steps)
    except Exception as e:  # noqa: BLE001
        out["eager"] = None
        out["eager_error"] = repr(e)[:200]
    try:
        t0 = time.perf_counter()
        compiled = torch.compile(denoise_eager, mode="reduce-overhead")
        out["compiled_reduce_overhead"] = timed(compiled, steps)
        out["compile_s"] = time.perf_counter() - t0
    except Exception as e:  # noqa: BLE001
        out["compiled_reduce_overhead"] = None
        out["compile_error"] = repr(e)[:300]
    return out


def conv_traffic_from_profile():
    """roofline.traffic = dram__bytes_read.sum + dram__bytes_write.sum of conv_tc_kernel, parsed from the newest committed
    `profiles/r*_prof_conv_*_summary.csv` (one `ncu --set full` capture of the same kernel); None when no capture exists."""
    import csv
    import glob

    files = sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_prof_conv_*_summary.csv")))
    for path in reversed(files):
        try:
            vals = {}
            with open(path) as f:
                for row in csv.reader(f):
                    for i, cell in enumerate(row):
                        if cell in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
                            unit, num = row[i + 1].strip().lower(), float(row[i + 2].replace(",", ""))
                            mult = {"byte": 1.0, "kbyte": 1e3, "mbyte": 1e6, "gbyte": 1e9}.get(unit, 1.0)
                            vals[cell] = num * mult
            if len(vals) == 2:
                return vals["dram__bytes_read.sum"] + vals["dram__bytes_write.sum"], os.path.relpath(path, ROOT)
        except Exception:
            continue
    return None, None


def train_block(dev, world, rank, batch, steps=5, warmup=2):
    """cfg 2 of BASELINE.json: denoiser training step (Denoiser.forward + backward on the native path, ONE flat-buffer NCCL
    all-reduce of the 17.6 MB gradient when world > 1, clip + AdamW as src/trainer.py:365-378), batch `batch` per GPU,
    frame-stack 4 + 1 autoregressive step, synthetic frames.  Returns samples/s (whole job) and the time split."""
    import torch
    import torch.distributed as dist

    from diamond_b200.models.diffusion import Denoiser, DenoiserConfig, InnerModelConfig, SigmaDistributionConfig
    from diamond_b200.synthetic import frame_stacks, randomize_module_
    from diamond_b200.utils import allreduce_native_gradients

    den = Denoiser(DenoiserConfig(InnerModelConfig(3, 4, 256, [2, 2, 2, 2], [64] * 4, [0] * 4, 4), 0.5, 0.3))
    randomize_module_(den.inner_model, 2024)
    den = den.to(dev).train()
    den.setup_training(SigmaDistributionConfig(-0.4, 1.2, 2e-3, 20))
    opt = torch.optim.AdamW(den.parameters(), lr=1e-4, weight_decay=1e-2, eps=1e-8)
    obs, act, _ = frame_stacks(batch, 5, 3, 64, 64, 4, 300 + rank)

    class B_:
        pass

    b = B_()
    b.obs, b.act, b.mask_padding = obs.to(dev), act.to(dev), torch.ones(batch, 5, dtype=torch.bool, device=dev)
    ev = lambda: torch.cuda.Event(enable_timing=True)  # noqa: E731
    t_fb = t_ar = t_opt = 0.0
    for it in range(warmup + steps):
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1, e2, e3 = ev(), ev(), ev(), ev()
        e0.record()
        opt.zero_grad(set_to_none=True)
        loss, _ = den(b)
        loss.backward()
        e1.record()
        ncoll = allreduce_native_gradients(den.inner_model)
        e2.record()
        torch.nn.utils.clip_grad_norm_(den.parameters(), 1.0)
        opt.step()
        e3.record()
        torch.cuda.synchronize()
        if it >= warmup:
            t_fb += e0.elapsed_time(e1); t_ar += e1.elapsed_time(e2); t_opt += e2.elapsed_time(e3)
    tot = max_over_ranks([t_fb + t_ar + t_opt, t_fb, t_ar, t_opt], dev)
    ms = tot[0] / steps
    gflop = 3 * 6.0888 * batch  # fwd + dgrad + wgrad (SURVEY.md 8d: 18.27 GFLOP / sample / AR step)
    return {"workload": "Denoiser.forward + backward + gradient all-reduce + clip + AdamW (cfg 2), batch %d per GPU, 1 AR step" % batch,
            "value": batch * world / (ms * 1e-3), "unit": "samples/s", "ms_per_step": ms, "fwd_bwd_ms": tot[1] / steps,
            "allreduce_ms": tot[2] / steps, "clip_adamw_ms": tot[3] / steps, "collectives_per_step": ncoll if world > 1 else 0,
            "allreduce_bytes": int(sum(p.numel() for p in den.parameters()) * 4), "loss": float(loss.detach()),
            "achieved_tflops_per_gpu": gflop / (tot[1] / steps), "steps": steps, "warmup": warmup}


def imagination_block(dev, world, rank, envs=32, horizon=15, updates=3, warmup=1):
    """cfg 3 of BASELINE.json: one actor-critic update in imagination = `horizon` imagined steps of `envs` environments
    (native sampler, 3 denoising steps, + native reward/termination model + native policy with autograd nodes), then the loss,
    BPTT through the rollout, gradient all-reduce when world > 1, clip + AdamW (src/trainer.py:365-378).  Everything on the
    step path is native; the environment is fed by a synthetic in-memory loader (no dataset on the box)."""
    import types

    import torch
    import torch.distributed as dist

    from diamond_b200.envs import WorldModelEnv, WorldModelEnvConfig
    from diamond_b200.models.actor_critic import ActorCritic, ActorCriticConfig, ActorCriticLossConfig
    from diamond_b200.models.diffusion import Denoiser, DenoiserConfig, DiffusionSamplerConfig, InnerModelConfig
    from diamond_b200.models.rew_end_model import RewEndModel, RewEndModelConfig
    from diamond_b200.synthetic import frame_stacks, randomize_module_
    from diamond_b200.utils import allreduce_native_gradients

    den = Denoiser(DenoiserConfig(InnerModelConfig(3, 4, 256, [2, 2, 2, 2], [64] * 4, [0] * 4, 4), 0.5, 0.3))
    randomize_module_(den.inner_model, 2024)
    rem = RewEndModel(RewEndModelConfig(512, 3, 64, 128, [2, 2, 2, 2], [32] * 4, [0] * 4, 4))
    randomize_module_(rem, 2025)
    ac = ActorCritic(ActorCriticConfig(512, 3, 64, [32, 32, 64, 64], [1, 1, 1, 1], 4))
    randomize_module_(ac, 2026)
    den, rem, ac = den.to(dev).eval(), rem.to(dev).eval(), ac.to(dev).train()

    # A trained reward/termination model ends episodes rarely; a random-init one ends ~half of them at every step, which turns the
    # rollout into a stream of resets + burn-ins.  The synthetic model's two termination logits are therefore tied to
    # +/- 0.05 * sum(hidden) (the head has no bias, rew_end_model.py:40), i.e. P(end) of a few per cent.
    with torch.no_grad():
        last = [m for m in rem.modules() if isinstance(m, torch.nn.Linear)][-1]
        last.weight[3].fill_(0.05); last.weight[4].fill_(-0.05)

    pool = [frame_stacks(envs, 4, 3, 64, 64, 4, 1000 * (rank + 1) + k)[:2] for k in range(8)]   # in-memory "dataset": no per-batch RNG cost

    class Loader:
        batch_sampler = types.SimpleNamespace(batch_size=envs)

        def __iter__(self):
            k = 0
            while True:
                obs, act = pool[k % len(pool)]
                k += 1
                yield types.SimpleNamespace(obs=obs, act=act)

    env = WorldModelEnv(den, rem, Loader(), WorldModelEnvConfig(horizon, 4, DiffusionSamplerConfig(3)))
    ac.setup_training(env, ActorCriticLossConfig(horizon, 0.985, 0.95, 1.0, 0.001))
    opt = torch.optim.AdamW(ac.parameters(), lr=1e-4, weight_decay=1e-2, eps=1e-8)
    ev = lambda: torch.cuda.Event(enable_timing=True)  # noqa: E731
    t_roll = t_bwd = t_rest = 0.0
    for it in range(warmup + updates):
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1, e2, e3 = ev(), ev(), ev(), ev()
        e0.record()
        opt.zero_grad(set_to_none=True)
        loss, logs = ac()
        e1.record()
        loss.backward()
        e2.record()
        allreduce_native_gradients(ac)   # the BPTT nodes accumulated into ONE flat buffer: one collective
        torch.nn.utils.clip_grad_norm_(ac.parameters(), 100.0)
        opt.step()
        e3.record()
        torch.cuda.synchronize()
        if it >= warmup:
            t_roll += e0.elapsed_time(e1); t_bwd += e1.elapsed_time(e2); t_rest += e2.elapsed_time(e3)
    tot = max_over_ranks([t_roll + t_bwd + t_rest, t_roll, t_bwd, t_rest], dev)
    ms = tot[0] / updates
    return {"workload": "ActorCritic.forward() over WorldModelEnv (%d envs x horizon %d, 3 denoise steps) + backward + clip + AdamW (cfg 3)" % (envs, horizon),
            "value": envs * horizon * world / (ms * 1e-3), "unit": "imagined frames/s (incl. policy update)", "ms_per_update": ms,
            "rollout_ms": tot[1] / updates, "backward_ms": tot[2] / updates, "allreduce_clip_adamw_ms": tot[3] / updates,
            "loss": float(loss.detach()), "updates": updates, "warmup": warmup}


def wgrad_roofline(dev, batch, peaks):
    """tcgen05 wgrad kernel, 3x3 64->64 at 64x64 over `batch` images (the dominant backward-filter shape), timed alone."""
    import torch

    from diamond_b200 import ops

    x = torch.randn(batch, 64, 64, 64, device=dev)
    g = torch.randn(batch, 64, 64, 64, device=dev)
    xo, go = ops.prep_act(x)[0], ops.prep_act(g)[0]
    dw = torch.zeros(64, 64, 9, device=dev)
    for _ in range(3):
        ops.conv2d_wgrad(go, 64, xo, 64, batch, 64, 64, 64, 64, 9, dw=dw)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 10
    e0.record()
    for _ in range(reps):
        ops.conv2d_wgrad(go, 64, xo, 64, batch, 64, 64, 64, 64, 9, dw=dw)
    e1.record()
    torch.cuda.synchronize()
    us = e0.elapsed_time(e1) / reps * 1e3
    flops = 2.0 * 576 * 64 * 4096 * batch
    peak = float(peaks.get("bf16_tflops", 1590.0))
    return {"kernel": "wgrad_tc_kernel + fixed-order reduce, 3x3 64->64 @64x64, %d images" % batch, "us_per_launch": us,
            "achieved": flops / (us * 1e-6) / 1e12, "peak": peak, "unit": "TFLOP/s", "frac": flops / (us * 1e-6) / 1e12 / peak}


class SecondaryBlocks:
    """Runs the optional blocks of the bench line after the headline numbers exist.  Every block gets a watchdog (its own limit,
    clipped to what is left of a budget shared by all blocks); when a watchdog fires, rank 0 prints the line as far as it got --
    tagged in `incomplete` -- and the process exits 0.  A block whose turn comes after the budget is spent is skipped."""

    def __init__(self, rank: int, line, budget_s: float, exit_fn=os._exit, out=None):
        self.rank, self.line, self.exit_fn, self.out = rank, line, exit_fn, out
        self.deadline = time.monotonic() + budget_s

    def _give_up(self, what: str) -> None:
        if self.rank == 0 and self.line is not None:
            self.line.setdefault("incomplete", []).append(what + ": watchdog timeout")
            print(json.dumps(self.line), file=self.out or sys.stdout, flush=True)
        self.exit_fn(0)

    def run(self, what: str, seconds: float, fn):
        left = self.deadline - time.monotonic()
        if left < 3.0:
            if self.rank == 0 and self.line is not None:
                self.line.setdefault("incomplete", []).append(what + ": skipped, secondary time budget spent")
            return {"skipped": "secondary time budget spent"}
        timer = threading.Timer(min(seconds, left), self._give_up, args=(what,))
        timer.daemon = True
        timer.start()
        try:
            return fn()
        except Exception as e:  # noqa: BLE001
            return {"error": repr(e)[:300]}
        finally:
            timer.cancel()


def run_native(args):
    import torch
    import torch.distributed as dist

    from diamond_b200 import _lib
    from diamond_b200.models.diffusion import (Denoiser, DenoiserConfig, DiffusionSampler, DiffusionSamplerConfig,
                                               InnerModelConfig)

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch with torchrun for --gpus > 1")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    lib = _lib.lib()  # no fallback: raises if the sm_100a library is missing

    from diamond_b200.synthetic import randomize_module_

    den = Denoiser(DenoiserConfig(InnerModelConfig(3, 4, 256, [2, 2, 2, 2], [64] * 4, [0] * 4, 4), 0.5, 0.3))
    randomize_module_(den.inner_model, 2024)  # same PCG64 rule as the oracle's seeded_state_dict(…, 2024)
    den = den.to(dev).eval()
    sampler = DiffusionSampler(den, DiffusionSamplerConfig(3))
    B = args.envs
    obs, act = rank_inputs(B, rank)
    obs_d, act_d = obs.to(dev), act.to(dev)
    obs_h, act_h = obs.pin_memory(), act.pin_memory()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    torch.manual_seed(0)  # sample() draws its initial noise from torch's generator: same arguments, same outputs

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident throughput
    clk = ClockSampler(local); clk.start()  # samples clocks / throttle reasons from warm-up to the end of the timed regions
    for _ in range(max(args.warmup, 3)):
        sampler.sample(obs_d, act_d)
    barrier()
    lib.dmd_launch_count(1)
    evs = []
    t_wall0 = time.perf_counter()
    for _ in range(args.steps):
        flush.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        x, traj = sampler.sample(obs_d, act_d)
        b.record()
        evs.append((a, b))
    barrier()
    t_wall = time.perf_counter() - t_wall0
    launches = int(lib.dmd_launch_count(0))
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, x, torch.stack(traj))
    dev_ms = sum(a.elapsed_time(b) for a, b in evs)

    # ---- end to end through the public API with host buffers (H2D of the frame stack + actions, D2H of the frame)
    for _ in range(3):
        x, _ = sampler.sample(obs_h.to(dev, non_blocking=True), act_h.to(dev, non_blocking=True)); x.cpu()
    barrier()
    e2e_evs = []
    out_h = torch.empty(B, 3, 64, 64).pin_memory()
    for _ in range(args.steps):
        flush.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        x, _ = sampler.sample(obs_h.to(dev, non_blocking=True), act_h.to(dev, non_blocking=True))
        out_h.copy_(x, non_blocking=True)
        b.record()
        e2e_evs.append((a, b))
    barrier()
    e2e_ms = sum(a.elapsed_time(b) for a, b in e2e_evs)

    dev_ms, e2e_ms = max_over_ranks([dev_ms, e2e_ms], dev)
    frames = B * args.steps * world
    line = None
    if rank == 0:
        peaks, peaks_src = load_peaks()
        roof = conv_roofline(dev, B, peaks, peaks_src)
        clocks = clk.finish()  # warm-up, both timed loops and the roofline loop are inside the sampling window
        value = whole_job_value(B * args.steps, world, dev_ms)
        line = {
            "metric": METRIC, "value": value, "unit": "frames/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": dev_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "fp16 tensor-core operands (split-fp16 on the residual-stream 1x1/conv_in layers), fp32 accumulate, fp32 activations", "data": "synthetic",
            "config": workload_config(args),
            "e2e": {"value": frames / (e2e_ms * 1e-3), "unit": "frames/s", "h2d_bytes_per_step": int(obs_h.numel() * 4 + act_h.numel() * 8),
                    "d2h_bytes_per_step": int(out_h.numel() * 4)},
            "gpu_launches": launches, "clocks": clocks, "roofline": roof,
            "model_flop_util": {"gflop_per_frame": GFLOP_PER_FRAME, "achieved_tflops": value * GFLOP_PER_FRAME / 1e3 / world,
                                "frac_of_peak": value * GFLOP_PER_FRAME / 1e3 / world / float(peaks.get("bf16_tflops_sustained", 1400.0))},
            "wall_s_timed_loop": t_wall,
            "parity": {"tolerance": "1e-3 RELATIVE L2 over the whole pre-quantisation model-output tensor vs the reference-pinned oracle "
                                    "(not max-per-element); outputs behind the truncating uint8 quantiser: never more than one level off",
                       "tests": "tests/test_gpu_denoiser.py (B=1, 2, 3, 5, the benchmarked B=32, and the padded 60x62 case)"},
        }
    else:
        clk.finish()

    # The headline line is complete here.  The secondary blocks (cfg 2 training step, cfg 3 imagination update, the reference's GPU
    # and CPU paths) run under a watchdog and a shared time budget: if one of them hangs (a rank lost inside a collective, a compile
    # that never returns) or the host is slow, the line is printed without it instead of the run ending with no result.
    guarded = SecondaryBlocks(rank, line, args.secondary_budget).run

    train = guarded("train_denoiser", 240, lambda: train_block(dev, world, rank, args.train_batch)) if not args.skip_train else None
    imag = guarded("imagination_update", 240, lambda: imagination_block(dev, world, rank, envs=B)) if not args.skip_imagination else None
    if rank == 0:
        if train is not None:
            line["train_denoiser"] = train
            if "error" not in train and "skipped" not in train:
                line["train_denoiser"]["wgrad_roofline"] = guarded("wgrad_roofline", 60, lambda: wgrad_roofline(dev, min(args.train_batch, 64), peaks))
        if imag is not None:
            line["imagination_update"] = imag
        if world == 1 and not args.skip_cpu_baseline:
            def cpu_leg():
                cores, avail = pick_cpu_threads()
                cpu_envs = 4
                cpu_val, _ = cpu_frames_per_s(cpu_envs, 3, cores)
                return {"value": cpu_val, "unit": "frames/s", "cores": cores, "kind": "port",
                        "sample": f"{cpu_envs} envs x 3 sample() calls of the same workload (oracle port of the reference, torch CPU fp32, {cores} threads = fastest of 8/16/32/64/{avail} available)"}
            line["cpu_baseline"] = guarded("cpu_baseline", 300, cpu_leg)
        if world == 1 and not args.skip_gpu_baseline:
            gpu_base = guarded("gpu_baseline", 300, lambda: gpu_baseline(dev, B))
            line["gpu_baseline"] = gpu_base
            for k in ("eager", "compiled_reduce_overhead"):
                if gpu_base.get(k):
                    gpu_base["e2e_speedup_vs_" + k] = line["e2e"]["value"] / gpu_base[k]
        print(json.dumps(line), flush=True)
    if world > 1:
        watchdog = threading.Timer(60, lambda: os._exit(0))   # the line is out: never hang in teardown
        watchdog.daemon = True
        watchdog.start()
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--envs", type=int, default=32, help="imagined environments per GPU (config/trainer.yaml actor_critic batch 32)")
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--skip-cpu-baseline", action="store_true", help="development runs: omit the (minutes-long) cpu_baseline leg")
    ap.add_argument("--skip-imagination", action="store_true", help="omit the imagination + actor-critic update block (cfg 3)")
    ap.add_argument("--skip-train", action="store_true", help="omit the denoiser-training block (cfg 2)")
    ap.add_argument("--train-batch", type=int, default=256, help="denoiser training batch per GPU (config/trainer.yaml: 32; BASELINE cfg 2: 256)")
    ap.add_argument("--skip-gpu-baseline", action="store_true", help="omit the reference-GPU-path leg (eager + torch.compile of the oracle port)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed sample() call returned (rank 0) as DIR/x.npy and "
                    "DIR/trajectory.npy, float32, at most 64 MB (a fixed seeded subset of the environments beyond that)")
    ap.add_argument("--secondary-budget", type=float, default=200.0, help="seconds shared by the blocks that follow the headline numbers (training, imagination, baselines); ~55 s are used on a healthy box")
    args = ap.parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_native(args)


if __name__ == "__main__":
    main()
