#!/usr/bin/env python
"""bench.py — headline benchmark: images/sec of one ImageGPT CIFAR-10-shaped training step.

A "step" is the reference's `Trainer._train_one_batch` (reference trainer.py:173-193) on one synthetic batch:
zero_grad -> forward -> BCE loss -> backward (+ DDP gradient all-reduce when N > 1) ->
clip_grad_norm_(params, 1e50) -> Adam step -> MultiplicativeLR step -> loss.item(), norm.item().

    python bench.py [--gpus N --steps K --warmup W]            our arm (N>1: launched by torch.distributed.run)
    python bench.py --impl reference [...]                      the reference's CPU path (oracle port), rank 0 only
    python bench.py --dump-outputs DIR [...]                    also write the last timed step's outputs (dump_outputs)

One JSON line on stdout (rank 0).  `value` has the batch resident in HBM when the timed region starts; `e2e`
goes through the public Module API with the batch in pinned host memory (H2D copy + loss/grad-norm D2H read
inside the timed region).  `roofline` is for the dominant kernel (the tcgen05 channel-contraction GEMM), timed
with CUDA events around every launch inside the timed region.  `cpu_baseline` is the oracle port on the host
cores on a bounded sample (rank 0, N=1 only).
"""

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

CONFIGS = {
    # BASELINE.json configs[4] — the configuration the metric is quoted on (fits one GPU)
    "c5": dict(name="ImageGPT 3x32x32 CIFAR-10-shaped, 24 blocks / 8 heads / 512 ch", cls="ImageGPT", oracle="image_gpt",
               cfg=dict(in_channels=3, out_channels=3, in_size=32, n_transformer_blocks=24, n_attention_heads=8,
                        n_embedding_channels=512),
               shape=(3, 32, 32), batch=64, lr=5e-3, algo_gflop_per_img=541.289, cpu_batch=2),
    # BASELINE.json configs[1]
    "c2": dict(name="ImageGPT 1x28x28 MNIST-shaped, 8 blocks / 4 heads / 64 ch", cls="ImageGPT", oracle="image_gpt",
               cfg=dict(in_channels=1, out_channels=1, in_size=28, n_transformer_blocks=8, n_attention_heads=4,
                        n_embedding_channels=64),
               shape=(1, 28, 28), batch=64, lr=5e-3, algo_gflop_per_img=3.742, cpu_batch=16),
    # the other BASELINE.json configs (secondary numbers, `--config cN`; the conv models compose the drop-in modules)
    "c1": dict(name="PixelCNN 1x28x28 binarized-MNIST-shaped, 15 residual / 16 ch", cls="PixelCNN", oracle="pixel_cnn",
               cfg=dict(in_channels=1, out_channels=1, n_residual=15, residual_channels=16, head_channels=32),
               shape=(1, 28, 28), batch=16, lr=1e-3, algo_gflop_per_img=0.171, cpu_batch=16),
    "c3": dict(name="GatedPixelCNN 3x32x32 CIFAR-10-shaped, 15 gated layers / 128 ch", cls="GatedPixelCNN",
               oracle="gated_pixel_cnn",
               cfg=dict(in_channels=3, out_channels=3, n_gated=15, gated_channels=128, head_channels=32),
               shape=(3, 32, 32), batch=128, lr=1e-3, algo_gflop_per_img=30.164, cpu_batch=8),
    "c4": dict(name="PixelSNAIL 3x32x32 CIFAR-10-shaped, 8 blocks / 256 ch, key 16 / value 128", cls="PixelSNAIL",
               oracle="pixel_snail",
               cfg=dict(in_channels=3, out_channels=3, n_channels=256, n_pixel_snail_blocks=8, n_residual_blocks=2,
                        attention_key_channels=16, attention_value_channels=128),
               shape=(3, 32, 32), batch=128, lr=1e-3, algo_gflop_per_img=92.061, cpu_batch=4),
}


def synthetic_batch(n, shape, seed):
    """CIFAR-shaped: uint8/255 like ToTensor (reference datasets.py:170); MNIST-shaped: Bernoulli(0.5)."""
    g = torch.Generator().manual_seed(seed)
    if shape[0] == 1:
        return torch.bernoulli(torch.full((n, *shape), 0.5), generator=g)
    return torch.randint(0, 256, (n, *shape), generator=g).float() / 255


def recipe_loss(x, _, preds):
    """loss_fn of the reference recipes (image_gpt.py:158-162)."""
    b = x.shape[0]
    x, preds = x.reshape(b, -1), preds.reshape(b, -1)
    loss = torch.nn.functional.binary_cross_entropy_with_logits(preds, x, reduction="none")
    return loss.sum(dim=1).mean()


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return dict(hbm_gbs=p["hbm_gbs"], tf_burst=p["bf16_tflops"], tf_sustained=p["bf16_tflops_sustained"],
                    source="measured (MEASURED_PEAKS.json)")
    return dict(hbm_gbs=6650.0, tf_burst=1590.0, tf_sustained=1400.0, source="fallback (B200_PROFILING.md)")


def measured_traffic():
    """DRAM bytes per GEMM launch from the committed ncu capture (None when the profile is absent)."""
    for name in ("r02_gemm_traffic.json", "r01_gemm_traffic.json"):
        path = os.path.join(ROOT, "profiles", name)
        if os.path.exists(path):
            return round(json.load(open(path))["traffic_bytes_per_launch"])
    return None


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons while the timed region runs."""

    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self._stop, self._t = index, [], threading.Event(), None

    def _run(self):
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits",
                                      "-i", str(self.index)], capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            self._stop.wait(0.2)

    def __enter__(self):
        self._t = threading.Thread(target=self._run, daemon=True)
        self._t.start()
        return self

    def __exit__(self, *exc):
        self._stop.set()
        self._t.join(timeout=6)

    def summary(self):
        sm = sorted(int(float(r[0])) for r in self.rows if r and r[0].replace(".", "").isdigit())
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        reasons = []
        for name, col in (("hw_slowdown", 3), ("hw_thermal_slowdown", 4), ("sw_thermal_slowdown", 5), ("sw_power_cap", 6)):
            if any(len(r) > col and r[col].lower().startswith("active") for r in self.rows):
                reasons.append(name)
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": int(float(self.rows[0][1])), "reasons": reasons,
                "samples": len(sm)}


class _stdout_to_stderr:
    """Routes file descriptor 1 to stderr for the duration of the block (C libraries that write to stdout)."""

    def __enter__(self):
        sys.stdout.flush()
        self._saved = os.dup(1)
        os.dup2(2, 1)

    def __exit__(self, *exc):
        sys.stdout.flush()
        os.dup2(self._saved, 1)
        os.close(self._saved)
        return False


def dump_outputs(out_dir, last, logits, model, per_tensor=4096, seed=0, max_logits=8 << 20):
    """Writes what the caller of the timed step holds after its last step, for comparing two builds output for output:
    loss.npy and grad_norm.npy (float64, the step's two return values), logits.npy (float32, the forward's output, cut
    to the leading images that fit in `max_logits` elements; eager steps only, the graphed step does not keep it) and
    weights.npy (float32, the updated weights: up to `per_tensor` elements of every parameter at fixed seeded positions,
    concatenated in named_parameters() order)."""
    import numpy as np

    os.makedirs(out_dir, exist_ok=True)
    arrays = {"loss": np.array(last[0], dtype=np.float64), "grad_norm": np.array(last[1], dtype=np.float64)}
    if logits is not None:
        keep = max(1, max_logits // max(1, logits[0].numel()))
        arrays["logits"] = logits[:keep].float().cpu().numpy()
    g = torch.Generator().manual_seed(seed)
    picks = []
    for _, p in model.named_parameters():
        flat = p.detach().reshape(-1)
        if flat.numel() > per_tensor:
            flat = flat[torch.randint(0, flat.numel(), (per_tensor,), generator=g).sort().values.to(flat.device)]
        picks.append(flat.float().cpu())
    arrays["weights"] = torch.cat(picks).numpy()
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


# --------------------------------------------------------------------------------------------------
# Our arm
# --------------------------------------------------------------------------------------------------
def run_ours(args):
    import torch.distributed as dist

    from pytorch_generative_b200 import _lib as L
    from pytorch_generative_b200 import losses, models, optim, parallel

    spec = CONFIGS[args.config]
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            sys.exit("bench.py --gpus N>1 must be launched with torch.distributed.run (one rank per GPU)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        parallel.configure_nccl()  # few NCCL CTAs: the gradient buckets need a fraction of NVLink, the GEMMs need the SMs
        with _stdout_to_stderr():  # NCCL prints its version banner on stdout; stdout carries the one JSON line only
            dist.init_process_group("nccl", device_id=dev)
            dist.barrier()
    L.load()

    batch = args.batch or spec["batch"]
    torch.manual_seed(0)
    model = getattr(models, spec["cls"])(**spec["cfg"]).to(dev)
    train_model = model
    parallel.broadcast_parameters(model)       # rank 0's weights everywhere (what DDP does at construction)
    params = [p for p in model.parameters()]
    # block-bucketed all-reduce overlapped with backward (ImageGPT) + one flat bucket for the rest; no-op at world size 1
    grad_avg = parallel.OverlappedGradAverager(model, params) if os.environ.get("PG_DP_OVERLAP", "1") != "0" \
        else parallel.FlatGradAverager(params)
    fused_opt = os.environ.get("PG_BENCH_TORCH_ADAM") != "1"
    opt = optim.FusedAdam(params, lr=spec["lr"]) if fused_opt else torch.optim.Adam(params, lr=spec["lr"])
    sched = torch.optim.lr_scheduler.MultiplicativeLR(opt, lr_lambda=lambda _: 0.999977)
    x_host = synthetic_batch(batch, spec["shape"], seed=parallel.shard_seed(0, rank)).pin_memory()  # rank r: seed r
    x_dev = x_host.to(dev)

    graphed = None
    if args.graph and world == 1:
        from pytorch_generative_b200 import trainstep

        model.train()
        graphed = trainstep.GraphedTrainStep(model, params, lambda preds, x: losses.bce_with_logits_sum_mean(preds, x), x_dev,
                                             lr=spec["lr"], lr_gamma=0.999977)

    last_logits = {}

    def step(x):
        if graphed is not None:
            return graphed(x)
        train_model.train()
        opt.zero_grad()
        preds = train_model(x)
        if args.dump_outputs:
            last_logits["logits"] = preds.detach()
        loss = losses.bce_with_logits_sum_mean(preds, x)  # the recipes' loss_fn (image_gpt.py:158-162), fused kernel
        loss.backward()
        grad_avg.average_()
        if fused_opt:  # clip_grad_norm_(params, 1e50) + Adam: two kernels over all parameters (optim.FusedAdam)
            norm = opt.clip_and_step(1e50)
        else:
            norm = torch.nn.utils.clip_grad_norm_(params, 1e50)
            opt.step()
        sched.step()
        return loss.item(), norm.item()

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        last = None
        for _ in range(steps):
            last = fn()
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return ms.item(), last

    for _ in range(max(args.warmup, 3)):
        step(x_dev)

    # ---- device-resident timing: `value` (no instrumentation inside the timed region) ----
    launches0 = L.launch_count()
    with ClockSampler(local_rank) as clocks:
        ms_total, last = timed(lambda: step(x_dev), args.steps)
    launches = L.launch_count() - launches0
    if args.dump_outputs and rank == 0:  # before the passes below move the weights on
        dump_outputs(args.dump_outputs, last, last_logits.get("logits"), model)

    # ---- the same steps again with CUDA events around every GEMM launch, for the roofline line only ----
    gemm_events = []
    L.gemm_timing_hook = lambda flops, a, b, io: gemm_events.append((flops, a, b, io))
    ms_instr, _ = timed(lambda: step(x_dev), args.steps)
    L.gemm_timing_hook = None
    gemm_ms = sum(a.elapsed_time(b) for _, a, b, _ in gemm_events)
    gemm_flops = sum(f for f, _, _, _ in gemm_events)
    gemm_bytes = sum(io for _, _, _, io in gemm_events)

    sample_ms = None
    if args.sample and rank == 0:
        # sample() latency (reference trainer.py:212-220 draws n=16): raster scan through the public API, wall clock
        model.eval()
        sample_ms = []
        for _ in range(2):  # first call builds the sampler (weight packing, graph capture), second is steady state
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            model.sample(n_samples=16)
            torch.cuda.synchronize()
            sample_ms.append((time.perf_counter() - t0) * 1e3)

    # ---- end-to-end: pinned host batch -> H2D -> step -> D2H scalars, through the Module API ----
    def e2e_step():
        return step(x_host.to(dev, non_blocking=True))

    e2e_step()
    ms_e2e, _ = timed(e2e_step, args.steps)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    pk = peaks()
    ms_step = ms_total / args.steps
    imgs = batch * world
    value = imgs / (ms_step / 1e3)
    e2e_value = imgs / (ms_e2e / args.steps / 1e3)
    achieved_tf = gemm_flops / (gemm_ms / 1e3) / 1e12 if gemm_ms > 0 else 0.0
    n_gemm = len(gemm_events)
    out = {
        "metric": "images/sec training step (ImageGPT CIFAR-10 32x32)" if args.config == "c5" else
        f"images/sec training step ({spec['name']})", "value": round(value, 2), "unit": "images/sec",
        "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": round(ms_step, 3),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": {"workload": spec["name"] + f", per-GPU batch {batch}, Adam lr {spec['lr']}, fp32 master weights, "
                   "bf16 tensor-core operands, fp32 residual stream", "global_batch": imgs, "parallelism": f"dp{world}",
                   "l2": "working set per step (~29 GB of activations at batch 64) >> 126 MB L2; no explicit flush needed",
                   "baseline_config": "BASELINE.json configs[4] (the metric's configuration)",
                   "step_launch": "one CUDA graph replay per step" if graphed is not None else "eager launches",
                   "optimizer": "FusedAdam (pg_grad_sqnorm + pg_adam_step)" if fused_opt and graphed is None else "torch.optim.Adam"},
        "e2e": {"value": round(e2e_value, 2), "unit": "images/sec", "h2d_bytes_per_step": x_host.numel() * 4,
                "d2h_bytes_per_step": 8},
        "gpu_launches": int(launches),
        "clocks": clocks.summary(),
        "roofline": {"bound": "tensor", "kernel": "gemm_tc_kernel (pg_gemm_bf16, tcgen05 1x1-conv fwd/dgrad/wgrad)",
                     "achieved": round(achieved_tf, 1), "peak": pk["tf_sustained"], "unit": "TFLOP/s",
                     "frac": round(achieved_tf / pk["tf_sustained"], 4), "traffic": measured_traffic(),
                     "traffic_unit": "DRAM bytes per launch (ncu dram__bytes_read+write over the 291 GEMMs of one step, "
                                     "profiles/r02_gemm_traffic.json)",
                     "algo_bytes_per_launch": round(gemm_bytes / max(n_gemm, 1)),
                     "flops_per_launch": round(gemm_flops / max(n_gemm, 1)),
                     "launches_timed": n_gemm, "share_of_step": round(gemm_ms / ms_instr, 4),
                     "timed_in": "a second pass of the same steps with CUDA events around every GEMM launch "
                                 f"({round(ms_instr / args.steps, 3)} ms/step instrumented)", "peak_source": pk["source"],
                     "step_algo_tflops": round(spec["algo_gflop_per_img"] * value / world / 1e3, 1),
                     "step_frac_of_peak": round(spec["algo_gflop_per_img"] * value / world / 1e3 / pk["tf_sustained"], 4)},
        "last_loss": last[0], "last_grad_norm": last[1],
    }
    if sample_ms is not None:
        out["sample"] = {"n_samples": 16, "pixels": spec["shape"][1] * spec["shape"][2],
                         "ms_first_call": round(sample_ms[0], 1), "ms": round(sample_ms[1], 1),
                         "method": "model.sample(n_samples=16): raster order and sample_fn hook of base.py:97-120; every "
                                   "model evaluates each pixel incrementally (line buffers / KV caches, one graph-replayed "
                                   "per-pixel program)"}
    if world == 1 and not args.no_cpu_baseline:
        out["cpu_baseline"] = cpu_baseline(spec, steps=2, warmup=1)
    print(json.dumps(out), flush=True)
    if world > 1:
        dist.destroy_process_group()


# --------------------------------------------------------------------------------------------------
# Reference arm / cpu_baseline: the oracle port of the reference's CPU path on the host cores
# --------------------------------------------------------------------------------------------------
def _thread_sweep(spec, candidates):
    """Picks the intra-op thread count for the CPU arm: one forward + backward of a depth-reduced copy of the model
    (2 blocks / layers, same widths, batch 1) at each candidate count; torch's CPU pool stops scaling -- and on a
    128-thread host gets slower -- well below the core count on this workload, so "all cores" (BASELINE.md §4) is
    resolved to the fastest measured count, and the sweep is reported next to the result."""
    from oracle import reference_path as O

    cfg = dict(spec["cfg"])
    for k in ("n_transformer_blocks", "n_residual", "n_gated", "n_pixel_snail_blocks"):
        if k in cfg:
            cfg[k] = min(cfg[k], 2)
    state = O.init_state(spec["oracle"], cfg)
    x = synthetic_batch(1, spec["shape"], seed=0)
    out = {}
    for t in candidates:
        torch.set_num_threads(t)
        best = float("inf")
        for _ in range(2):
            t0 = time.perf_counter()
            O.loss_and_grads(spec["oracle"], state, x, cfg)
            best = min(best, time.perf_counter() - t0)
        out[t] = round(best * 1e3, 1)
    return out


def cpu_baseline(spec, steps, warmup, budget_s=60.0):
    """Times the reference's CPU path (the oracle port: the same torch ops in the same order, bit-identical to the live
    reference on this torch build, tests/test_oracle.py) on the host cores at BASELINE.md §4's reduced batch; bounded:
    stops adding steps once `budget_s` is spent."""
    from oracle import reference_path as O

    try:
        avail = len(os.sched_getaffinity(0))
    except AttributeError:
        avail = os.cpu_count() or 1
    candidates = sorted({c for c in (8, 16, 32, 64, avail) if c <= avail})
    sweep = _thread_sweep(spec, candidates)
    threads = min(sweep, key=sweep.get)
    torch.set_num_threads(threads)
    nb = spec["cpu_batch"]
    ts = O.TrainState(spec["oracle"], O.init_state(spec["oracle"], spec["cfg"]), spec["cfg"], lr=spec["lr"])
    x = synthetic_batch(nb, spec["shape"], seed=0)
    times, t_start = [], time.perf_counter()
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        ts.step(x)
        times.append(time.perf_counter() - t0)
        if time.perf_counter() - t_start > budget_s and len(times) >= 1:
            break
    timed = times[warmup:] if len(times) > warmup else times[-1:]
    dt = sum(timed) / len(timed)
    return {"value": round(nb / dt, 4), "unit": "images/sec", "cores": threads, "host_cores": avail, "kind": "port",
            "ms_per_step": round(dt * 1e3, 1), "thread_sweep_ms": {str(k): v for k, v in sweep.items()},
            "sample": f"{len(timed)} timed step(s) after {min(warmup, len(times) - len(timed))} warm-up of the same training "
                      f"step at batch {nb} on the host CPU (oracle/reference_path.py = the reference's torch-CPU fp32 path); "
                      f"threads = fastest of a sweep over {candidates} on a 2-block copy of the model"}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    spec = CONFIGS[args.config]
    steps = min(args.steps, 3)
    cb = cpu_baseline(spec, steps=steps, warmup=1)
    world = int(os.environ.get("WORLD_SIZE", "1"))
    out = {
        "impl": "reference",
        "metric": "images/sec training step (ImageGPT CIFAR-10 32x32)" if args.config == "c5" else
        f"images/sec training step ({spec['name']})", "value": cb["value"],
        "unit": "images/sec", "n_gpus": world, "steps": steps, "warmup": 1, "ms_per_step": cb["ms_per_step"],
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": spec["name"] + f", CPU batch {spec['cpu_batch']} (bounded sample)", "parallelism": "cpu"},
        "cpu_baseline": cb,
        "e2e": {"value": cb["value"], "unit": "images/sec", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(out), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="c5", choices=sorted(CONFIGS))
    ap.add_argument("--batch", type=int, default=0, help="per-GPU batch (default: the recipe's)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--sample", action="store_true", help="also time model.sample(n_samples=16)")
    ap.add_argument("--graph", action="store_true", help="replay the whole training step as one CUDA graph (small configs)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
