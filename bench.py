#!/usr/bin/env python
"""bench.py — headline benchmark of the B200-native single-step denoising engine.

    python bench.py --gpus N --steps K --warmup W            (torchrun launches N>1, one rank per GPU)
    python bench.py --impl reference --gpus N --steps K --warmup W
    python bench.py --workload {marigold,normals,geowizard,train} [--res R] [--batch B]      (BASELINE.json configs 2-5)
    python bench.py ... --dump-outputs DIR        (+ what the last timed step returned, as DIR/<name>.npy)

Default workload = BASELINE.json configs[1]: marigold-e2e-ft-depth inference, bs=8 per GPU, fp16 operands,
processing_res=768, 1 denoising step, zeros noise, synthetic 3x768x768 RGB, seeded random weights.
One "step" = one `MarigoldPipeline.single_infer` over a batch (VAE encode -> UNet -> x0 -> VAE decode
-> depth post-ops).  Metric: 768x768 depth images / second (whole job, all GPUs).

  value      device-timed throughput, inputs resident in HBM
  e2e        same through the public pipeline API from pinned fp32 HOST buffers (H2D + D2H inside the timing)
  roofline   implicit-GEMM conv kernel (the dominant kernel): algorithmic FLOPs / CUDA-event time of its
             launches inside the timed region, against the measured bf16 peak (MEASURED_PEAKS.json)
  train_step BASELINE.json configs[2] (training/train.py:469-568, bs=2 per GPU, 768x768, fp32 masters): forward /
             backward / optimizer split and the gradient all-reduce (NCCL over NVLink at N > 1) with the bucketed
             overlap on and off — the one collective of this workload, driver-run at every N
  cpu_baseline / --impl reference: the ORACLE (oracle/, plain PyTorch fp32 restatement of the reference's
             diffusers path, which is not installable here) on the host cores, at the REAL config: one 3x768x768
             image per `single_infer` (BASELINE.json configs[0]), the same fixed resolution in both legs.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# tensor-pipe FLOPs (2*MAC) per image, SURVEY.md §8(d): UNet / VAE enc / VAE dec
TFLOP_PER_IMAGE = {768: 10.501, 512: 4.429, 384: 2.444, 256: 1.10, 128: 0.28, 64: 0.07}
METRIC = "images_per_sec_768x768_depth"
DUMP_BYTES = 64 * 10 ** 6          # --dump-outputs writes at most this; larger outputs are stored as a fixed seeded sample


def dump_outputs(arrays, out_dir, seed=0):
    """Write every array as <out_dir>/<name>.npy in float32.  If together they exceed DUMP_BYTES, each keeps the same
    share of its elements, at flat indices drawn by a generator seeded with `seed` and stored in index order: runs with
    the same arguments store the same positions, so two builds can be compared element for element."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    total = sum(a.numel() for a in arrays.values())
    cap = (DUMP_BYTES - 1024 * len(arrays)) // 4          # float32 elements, leaving room for the .npy headers
    info = {}
    for name, a in arrays.items():
        a = a.detach().float().cpu()
        n = a.numel()
        info[name] = {"shape": list(a.shape), "stored": "all"}
        if total > cap:
            k = n * cap // total
            idx = torch.randperm(n, generator=torch.Generator().manual_seed(seed))[:k].sort().values
            a = a.reshape(-1)[idx]
            info[name]["stored"] = f"{k} of {n} elements at seeded flat indices (torch.randperm seed {seed}), ascending"
        np.save(os.path.join(out_dir, name + ".npy"), a.numpy())
    return info


def shard_range(total, rank, world):
    """Contiguous shard [lo, hi) of `total` images for `rank` (independent images: no collective)."""
    per = (total + world - 1) // world
    lo = min(total, rank * per)
    return lo, min(total, lo + per)


def max_over_ranks(ms, device):
    import torch
    import torch.distributed as dist
    if not (dist.is_available() and dist.is_initialized()):
        return ms
    t = torch.tensor([ms], dtype=torch.float64, device=device)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(tflops_burst=d["bf16_tflops"], tflops_sustained=d["bf16_tflops_sustained"],
                    hbm_gbs=d["hbm_gbs"], source="measured")
    return dict(tflops_burst=1590.0, tflops_sustained=1400.0, hbm_gbs=6650.0, source="fallback")


class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(gpu_index), f"--query-gpu={self.Q}",
                                       "--format=csv,noheader,nounits", "-lms", "100"], stdout=self.f,
                                      stderr=subprocess.DEVNULL)
        except OSError:
            self.p = None

    def stop(self):
        if self.p is None:
            return None
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.p.kill()
        self.f.flush()
        rows = [l.strip().split(", ") for l in open(self.f.name) if l.strip()]
        os.unlink(self.f.name)
        sm, mx, reasons = [], 0.0, set()
        for r in rows:
            try:
                sm.append(float(r[1]))
                mx = max(mx, float(r[2]))
            except (ValueError, IndexError):
                continue
            names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
            for n, v in zip(names, r[5:9]):
                if v.strip().lower().startswith("active"):
                    reasons.add(n)
        if not sm:
            return None
        sm.sort()
        return dict(sm_mhz=sm[len(sm) // 2], sm_max_mhz=mx, reasons=sorted(reasons), samples=len(sm))


# --------------------------------------------------------------------------------------------- oracle legs
CPU_RES = 768                      # BASELINE.json configs[0]: one 3x768x768 image per single_infer — both CPU legs use it
CPU_BUDGET_S = 150.0               # wall-clock cap of the timed CPU steps (a 768^2 image takes ~20-30 s on the host cores)


def build_oracle(seed=1234, full=True):
    """Oracle modules with cheap synthetic weights (timing only): built on the meta device, then filled
    with U(-1/sqrt(fan_in), 1/sqrt(fan_in)) in place (default nn init of 950 M parameters takes ~45 s)."""
    import torch
    from oracle.unet import UNet2DConditionRef, UNetConfig, tiny_config
    from oracle.vae import AutoencoderKLRef, VAEConfig, tiny_vae_config
    g = torch.Generator().manual_seed(seed)
    with torch.device("meta"):
        unet = UNet2DConditionRef(UNetConfig() if full else tiny_config())
        vae = AutoencoderKLRef(VAEConfig() if full else tiny_vae_config())
    for m in (unet, vae):
        m.to_empty(device="cpu")
        with torch.no_grad():
            for name, p in m.named_parameters():
                if p.dim() >= 2:
                    p.uniform_(-1.0, 1.0, generator=g).mul_(1.0 / (p[0].numel() ** 0.5))
                elif "norm" in name and name.endswith("weight"):
                    p.fill_(1.0)
                else:
                    p.zero_()
        m.eval()
    return unet, vae


def oracle_step(unet, vae, res, batch=1):
    import torch
    from oracle import pipeline as OP
    g = torch.Generator().manual_seed(0)
    rgb = torch.rand(batch, 3, res, res, generator=g) * 2 - 1
    ete = torch.randn(1, 2, unet.config.cross_attention_dim, generator=g) * 0.5
    t0 = time.perf_counter()
    with torch.no_grad():
        OP.marigold_single_infer(unet, vae, OP.DDIMOneStep(), rgb, ete)
    return time.perf_counter() - t0


def pick_cpu_threads(unet, vae):
    """Host thread count for the oracle: all cores is often NOT fastest on a 128-way shared host
    (oversubscribed oneDNN thread pools), so calibrate on a tiny problem and keep the best."""
    import torch
    try:
        avail = len(os.sched_getaffinity(0))
    except AttributeError:
        avail = os.cpu_count() or 1
    cands = sorted({c for c in (avail, 64, 32, 16, 8) if 1 <= c <= avail}, reverse=True)
    best, best_t = cands[-1], float("inf")
    for c in cands:
        torch.set_num_threads(c)
        oracle_step(unet, vae, 64)
        t = oracle_step(unet, vae, 64)
        if t < best_t:
            best, best_t = c, t
    torch.set_num_threads(best)
    return best


def cpu_reference_run(steps, warmup, budget_s=CPU_BUDGET_S):
    """The reference's CPU path (oracle restatement, fp32, PyTorch CPU kernels) at the real config: every step is one
    `single_infer` of ONE 3x768x768 image.  At most `steps` timed steps, stopped early once `budget_s` is spent (never
    fewer than one); at most one untimed warm-up."""
    unet, vae = build_oracle()
    cores = pick_cpu_threads(unet, vae)
    n_warm = min(1, warmup)
    for _ in range(n_warm):
        oracle_step(unet, vae, CPU_RES)
    times = []
    while len(times) < max(1, steps) and (not times or sum(times) + times[-1] <= budget_s):
        times.append(oracle_step(unet, vae, CPU_RES))
    dt = sum(times)
    sample = (f"{len(times)} timed + {n_warm} warm-up oracle single_infer call(s), each ONE 3x{CPU_RES}x{CPU_RES} image "
              f"(BASELINE.json configs[0]), fp32, {cores} host threads; per image "
              f"{min(times):.1f}-{max(times):.1f} s; capped at {budget_s:.0f} s of timed CPU work")
    return dict(value=len(times) / dt, steps=len(times), warmup=n_warm, seconds=dt, cores=cores, sample=sample)


def run_reference(args):
    """The reference's own (CPU, fp32, PyTorch) path on the host cores: the oracle restatement, since
    diffusers==0.30.2 cannot be installed offline (DESIGN.md §Reference arm)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    r = cpu_reference_run(args.steps, args.warmup)
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": r["value"], "unit": "images/s", "n_gpus": args.gpus,
        "steps": r["steps"], "warmup": r["warmup"], "steps_requested": args.steps,
        "ms_per_step": r["seconds"] / r["steps"] * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "fp32", "data": "synthetic",
        "config": {"workload": "marigold-e2e-ft-depth single_infer, 1 step, zeros noise, one 3x768x768 image per step "
                               "(CPU oracle = the reference's diffusers graph restated; BASELINE.json configs[0])",
                   "global_batch": 1},
        "cpu_baseline": {"value": r["value"], "unit": "images/s", "cores": r["cores"], "kind": "port",
                         "sample": r["sample"]},
        "e2e": {"value": r["value"], "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def cpu_baseline_leg():
    r = cpu_reference_run(1, 0, budget_s=60.0)
    return {"value": r["value"], "unit": "images/s", "cores": r["cores"], "kind": "port", "sample": r["sample"]}


# --------------------------------------------------------------------------------------------- engine
def build_engine(device, stream_dtype, module_dtype, workload="marigold", seed=1234, vae_stream_dtype=None):
    import torch
    from diffusion_e2e_ft_b200 import (B200AutoencoderKL, B200UNet2DConditionModel, DDIMScheduler,
                                       DepthNormalEstimationPipeline, MarigoldPipeline)
    torch.manual_seed(seed)
    with torch.device(device):
        if workload == "geowizard":
            # SURVEY.md §8(d) config 4: SD-2 widths, class-embedding projection (10), 1 x 768 image-embedding token,
            # joint depth/normal self-attention
            unet = B200UNet2DConditionModel(stream_dtype=stream_dtype, class_embed_type="projection",
                                            projection_class_embeddings_input_dim=10, cross_attention_dim=768,
                                            joint_attention=True)
        else:
            unet = B200UNet2DConditionModel(stream_dtype=stream_dtype)
        vae = B200AutoencoderKL(stream_dtype=vae_stream_dtype or stream_dtype)
    unet.to(module_dtype).eval().requires_grad_(False)
    vae.to(module_dtype).eval().requires_grad_(False)
    if workload == "geowizard":
        # geowizard_pipeline.py:232-248,283-288: the CLIP ViT-L/14 image encoder runs for every input image
        from diffusion_e2e_ft_b200 import B200CLIPVisionModelWithProjection, CLIPImageProcessorConfig
        with torch.device(device):
            enc = B200CLIPVisionModelWithProjection()
        enc.to(module_dtype).eval().requires_grad_(False)
        return DepthNormalEstimationPipeline(unet, vae, DDIMScheduler(), image_encoder=enc,
                                             feature_extractor=CLIPImageProcessorConfig(224))
    ete = (torch.randn(1, 2, 1024, device=device) * 0.5).to(module_dtype)
    return MarigoldPipeline(unet, vae, DDIMScheduler(), empty_text_embed=ete)


def _dist_setup():
    import datetime
    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a B200 (no CPU fallback); use --impl reference for the CPU path")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        # a collective that never completes raises after the timeout instead of hanging the whole bench
        dist.init_process_group("nccl", device_id=dev, timeout=datetime.timedelta(seconds=180))
    return world, rank, local, dev


def train_leg(dev, rank, world, res=768, batch=2, steps=3, warmup=2, modality="depth"):
    """BASELINE.json configs[2] / SURVEY.md §8(d) config 3: training/train.py:469-568 step semantics — SD-2 UNet with the
    8-channel conv_in, fp32 master weights, bs `batch` per GPU, rgb U(-1,1), GT depth U(0.1,10), mask all-true, ctx
    [1,77,1024], data parallel over `world` ranks (one gradient all-reduce per optimizer step, NCCL over NVLink).
    Device-timed (CUDA events), max over ranks.  Three timings of the same step: all bucket all-reduces launched after
    backward (FlatTrainer's default, see its docstring), launched from backward hooks so they overlap it, and the
    all-reduce of the flat gradient buffer alone."""
    import torch
    import torch.distributed as dist
    from diffusion_e2e_ft_b200 import B200AutoencoderKL, B200UNet2DConditionModel, DDIMScheduler, ops
    from diffusion_e2e_ft_b200.training import FlatTrainer, e2e_ft_loss
    torch.manual_seed(4321)
    with torch.device(dev):
        unet = B200UNet2DConditionModel()
        vae = B200AutoencoderKL()
    vae.eval().requires_grad_(False)
    unet.train().requires_grad_(True)
    tr = FlatTrainer(unet, lr=3e-5, weight_decay=1e-2, max_grad_norm=1.0)
    g = torch.Generator(device=dev).manual_seed(5 + rank)                      # different images per rank
    rgb = torch.rand(batch, 3, res, res, device=dev, generator=g) * 2 - 1
    gt = torch.rand(batch, 1, res, res, device=dev, generator=g) * 9.9 + 0.1
    mask = torch.ones(batch, 1, res, res, device=dev, dtype=torch.bool)
    ete = torch.randn(1, 77, 1024, device=dev, generator=g) * 0.5
    sched = DDIMScheduler()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def one_step():
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
        ev[0].record()
        loss, _ = e2e_ft_loss(unet, vae, sched, rgb, gt, mask, ete, modality)
        ev[1].record()
        tr.backward(loss)
        ev[2].record()
        tr.step()
        ev[3].record()
        return loss, ev

    def timed_steps(n):
        barrier()
        evs, losses = [], []
        for _ in range(n):
            loss, ev = one_step()
            evs.append(ev)
            losses.append(loss)
        barrier()
        # per-step device times; the MEDIAN step is reported (the caching allocator still grows in the first steps of a
        # 66 GB working set: single steps of 2x the steady-state time were observed right after warm-up)
        per = sorted(((e[0].elapsed_time(e[3]), e[0].elapsed_time(e[1]), e[1].elapsed_time(e[2]), e[2].elapsed_time(e[3]))
                      for e in evs))
        tot, f, b, o = per[len(per) // 2]
        return [f, b, o, tot], [float(l) for l in losses]

    for _ in range(warmup):
        one_step()
    ops.STATS.reset()
    t_on, losses = timed_steps(steps)
    flops = sum(ops.STATS.flops.values()) / steps
    launches = ops.STATS.launches // steps
    t_off, ar = None, 0.0
    if world > 1:
        tr.overlap = True                     # the alternative: bucket all-reduces launched from backward hooks
        one_step()
        t_off, _ = timed_steps(steps)
        tr.overlap = False
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        a0.record()
        for _ in range(3):
            dist.all_reduce(tr.flat_grad)
        a1.record()
        barrier()
        ar = a0.elapsed_time(a1) / 3
        tr.flat_grad.zero_()
    vals = t_on + (t_off or [0.0] * 4) + [ar]
    if world > 1:
        t = torch.tensor(vals, dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        vals = [float(v) for v in t]
    f, b, o, tot = vals[:4]
    out = {
        "config": f"training/train.py step, SD-2 UNet (8-ch conv_in) + frozen VAE, {modality} recipe, bs={batch}/GPU "
                  f"{res}x{res}, fp32 masters, fp16 GEMM operands, dynamic loss scale, dp{world} (BASELINE.json configs[2])",
        "ms_per_step": tot, "ms_per_step_is": "median of the timed steps", "samples_per_s": world * batch / (tot / 1e3),
        "forward_ms": f, "backward_ms": b,
        "optimizer_ms": o, "grad_bytes": int(tr.flat_grad.numel()) * 4, "buckets": len(tr._buckets),
        "tensor_tflops_per_gpu": flops / (tot / 1e3) / 1e12, "gpu_launches_per_step": launches,
        "losses": losses, "finite": all(l == l and abs(l) < 1e9 for l in losses),
        "applied_steps": tr.applied_steps(), "skipped_steps": tr.skipped_steps(), "loss_scale": tr.loss_scale(),
        "peak_mem_gb": torch.cuda.max_memory_allocated(dev) / 2 ** 30,
    }
    if world > 1:
        out["allreduce"] = {
            "collective": "NCCL all-reduce(sum) of the flat fp32 gradient in 256 MB buckets, after backward (default)",
            "alone_ms": vals[8], "bus_gbs": 2 * (world - 1) / world * out["grad_bytes"] / (vals[8] / 1e3) / 1e9,
            "step_ms": tot, "exposed_ms": vals[8],
            "step_ms_overlap_with_backward": vals[7],
            "note": "overlap with backward is N-dependent on this engine (persistent one-CTA-per-SM GEMM grids vs NCCL's "
                    "channel CTAs): measured 515 vs 260 ms at 2 ranks (P2P ring), 178 vs 182 ms at 8 ranks (NVLS); the "
                    "default keeps the exchange after backward, where it costs alone_ms"}
    del tr, unet, vae
    torch.cuda.empty_cache()
    return out


def run_train(args):
    import torch.distributed as dist
    world, rank, local, dev = _dist_setup()
    t = train_leg(dev, rank, world, res=args.res, batch=args.batch or 2, steps=args.steps, warmup=max(args.warmup, 3))
    if rank == 0:
        print(json.dumps({
            "metric": "train_samples_per_sec_768x768", "value": t["samples_per_s"], "unit": "samples/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": t["ms_per_step"],
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "fp16", "data": "synthetic",
            "config": {"workload": t["config"], "global_batch": (args.batch or 2) * world, "parallelism": f"dp{world}"},
            "gpu_launches": t["gpu_launches_per_step"] * args.steps, "train_step": t}))
    if world > 1:
        dist.destroy_process_group()


def run_engine(args):
    import torch
    import torch.distributed as dist
    from diffusion_e2e_ft_b200 import ops
    world, rank, local, dev = _dist_setup()
    wl = args.workload
    bs = args.batch or {"marigold": 8, "normals": 16, "geowizard": 4}[wl]
    res = args.res
    sdt = torch.float16 if args.stream == "fp16" else torch.float32
    vsdt = torch.float16 if args.stream == "mixed" else None            # mixed: fp32 UNet stream, fp16 VAE stream
    pipe = build_engine(dev, sdt, torch.float16, wl, vae_stream_dtype=vsdt)
    g = torch.Generator(device="cpu").manual_seed(1000 + rank)
    # the reference API hands the pipeline fp32 images (marigold_pipeline.py:245-247): fp32 pinned host buffers
    host_rgb = (torch.rand(bs, 3, res, res, generator=g) * 2 - 1).pin_memory()
    out_ch = {"marigold": 1, "normals": 3, "geowizard": 4}[wl]
    host_out = torch.empty(bs, out_ch, res, res, dtype=torch.float32).pin_memory()
    dev_rgb = host_rgb.to(dev)

    def infer(x):
        if wl == "geowizard":
            d, n = pipe.single_infer(x, 1, "indoor")       # resize + CLIP image encoder + VAE + joint UNet + 2 decodes
            return torch.cat([d, n], 1)
        return pipe.single_infer(x, 1, False, noise="zeros", normals=(wl == "normals"))

    def step_resident():
        return infer(dev_rgb)

    def step_e2e():
        x = host_rgb.to(dev, non_blocking=True)
        y = infer(x)
        host_out.copy_(y, non_blocking=True)
        return y

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    last = None                        # what the last timed step returned

    def timed(fn, steps, time_conv=False):
        nonlocal last
        ops.STATS.reset()
        ops.STATS.time_kind = ("gemm" if args.dump_shapes else "conv") if time_conv else None
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            last = fn()
        e1.record()
        barrier()
        ops.STATS.time_kind = None
        return max_over_ranks(e0.elapsed_time(e1), dev)

    # ---- timed region A: the step as a user runs it (CUDA-graph replay inside the pipeline)
    for _ in range(max(args.warmup, 3)):
        step_resident()
    sampler = ClockSampler(local) if rank == 0 else None
    ms = timed(step_resident, args.steps)
    clocks = sampler.stop() if sampler else None
    launches = ops.STATS.launches
    total_flops = sum(ops.STATS.flops.values())
    flops_by_kind = {k: v / args.steps for k, v in ops.STATS.flops.items()}
    dumped = None
    if args.dump_outputs and rank == 0:
        # what single_infer handed back in the last timed step
        if wl == "geowizard":                          # infer() concatenates its (depth, normal)
            arrays = {"depth": last[:, :1], "normal": last[:, 1:]}
        else:
            arrays = {"normals" if wl == "normals" else "depth": last}
        dumped = {"dir": os.path.abspath(args.dump_outputs), "arrays": dump_outputs(arrays, args.dump_outputs)}

    # ---- timed region B (roofline leg): the same step launched eagerly so every implicit-GEMM conv
    # launch can be bracketed with CUDA events on the launching stream
    pipe.use_cuda_graph = False
    step_resident()
    rsteps = min(args.steps, 3)
    eager_ms = timed(step_resident, rsteps, time_conv=True)
    stats = ops.STATS
    conv_ms = sum(e[0].elapsed_time(e[1]) for e in stats.events)
    conv_flops = sum(e[2] for e in stats.events)
    if args.dump_shapes and rank == 0:
        os.makedirs(os.path.join(ROOT, 'gpurun_out'), exist_ok=True)
        for name, events in (("linear", stats.lin_events), ("conv", stats.events)):
            agg = {}
            for e in events:
                a = agg.setdefault(str(e[3]), [0, 0.0, 0])
                a[0] += 1; a[1] += e[0].elapsed_time(e[1]); a[2] += e[2]
            rows = sorted(((k, n, ms_, fl / (ms_ / 1e3) / 1e12) for k, (n, ms_, fl) in agg.items()), key=lambda r: -r[2])
            with open(os.path.join(ROOT, 'gpurun_out', f'{name}_shapes.txt'), 'w') as f:
                f.write(('(B,M,N,K,act,residual,out)' if name == "linear" else '(NB,H,W,Cin,C2,Cout,taps,stride,out)')
                        + f' launches total_ms TFLOP/s   [{rsteps} eager steps]\n')
                for k, n, ms_, tf in rows:
                    f.write(f'{k:55s} {n:4d} {ms_:9.3f} {tf:8.1f}\n')
    n_conv = len(stats.events)
    # per-op breakdown of one eager step (CUDA events around every op)
    ops.STATS.time_all = True
    ops.STATS.op_events = []
    step_resident()
    torch.cuda.synchronize()
    ops.STATS.time_all = False
    breakdown = {}
    for name, a, b2 in ops.STATS.op_events:
        breakdown[name] = breakdown.get(name, 0.0) + a.elapsed_time(b2)
    ops.STATS.op_events = []
    pipe.use_cuda_graph = True

    # ---- UNet-only forward (part of the headline metric triple), graph-replayed: 8-channel random latent, t = 999, the
    # batch-shared 2-token context exactly as the pipeline passes it (constant-context cross-attention, cached temb)
    unet_ms = unet_flops = None
    if wl != "geowizard":
        lat = torch.randn(bs, 8, res // 8, res // 8, device=dev, dtype=torch.float16)
        ctx = pipe.empty_text_embed.expand(bs, -1, -1)
        with torch.no_grad():
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                for _ in range(2):
                    pipe.unet(lat, 999, encoder_hidden_states=ctx)
            torch.cuda.current_stream().wait_stream(side)
            torch.cuda.synchronize()
            ops.STATS.reset()
            ug = torch.cuda.CUDAGraph()
            with torch.cuda.graph(ug):
                pipe.unet(lat, 999, encoder_hidden_states=ctx)
            unet_flops = sum(ops.STATS.flops.values())
            ug.replay()
            unet_ms = timed(ug.replay, args.steps) / args.steps
            del ug

    for _ in range(2):
        step_e2e()
    e2e_ms = timed(step_e2e, args.steps)

    # ---- fast mode (fp16 residual stream, the dtype layout of the reference's own fp16 path): reported beside the
    # default fp32-stream number, never instead of it
    fast = None
    if args.stream == "fp32" and not args.no_fast:
        try:
            del pipe._graphs
            fpipe = build_engine(dev, torch.float16, torch.float16, wl)
            pipe_keep, pipe = pipe, fpipe
            for _ in range(3):
                step_resident()
            fms = timed(step_resident, args.steps)
            fast = {"stream_dtype": "fp16", "value": bs * world * args.steps / (fms / 1e3), "ms_per_step": fms / args.steps}
            pipe = pipe_keep
            fpipe.__dict__.pop("_graphs", None)     # graph entries hold closures over the pipeline (reference cycle)
            del fpipe
        except Exception as e:  # noqa: BLE001
            fast = {"error": repr(e)[:200]}

    peaks = measured_peaks()
    images = bs * world * args.steps
    value = images / (ms / 1e3)
    e2e_value = images / (e2e_ms / 1e3)
    out = None
    if rank == 0:
        conv_tf = conv_flops / (conv_ms / 1e3) / 1e12 if conv_ms > 0 else 0.0
        ms_eager = eager_ms / rsteps
        peak = peaks["tflops_sustained"]
        traffic, traffic_of = None, None
        tp = os.path.join(ROOT, "profiles", "conv_traffic.json")
        if os.path.exists(tp):
            tj = json.load(open(tp))
            traffic = tj.get("dram_bytes_per_launch")
            traffic_of = (f"one ncu --set full capture of {tj.get('kernel')} on {tj.get('shape')}: "
                          f"{tj.get('algorithmic_flops', 0) / 1e12:.3f} TFLOP, algorithmic bytes >= "
                          f"{tj.get('algorithmic_bytes_min', 0) / 1e9:.3f} GB ({tj.get('source')})")
        names = {"marigold": ("marigold-e2e-ft-depth single_infer", "BASELINE.json configs[1]"),
                 "normals": ("marigold-e2e-ft-normals single_infer", "BASELINE.json configs[4]"),
                 "geowizard": ("geowizard-e2e-ft joint depth+normals single_infer (indoor), CLIP ViT-L/14 image encoder per image included", "BASELINE.json configs[3]")}[wl]
        out = {
            "metric": METRIC if (wl == "marigold" and res == 768) else f"images_per_sec_{res}x{res}_{wl}",
            "value": value, "unit": "images/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "fp16", "data": "synthetic",
            "config": {"workload": f"{names[0]} bs={bs}/GPU {res}x{res}, 1 step, zeros noise ({names[1]})",
                       "global_batch": bs * world, "parallelism": f"dp{world} (independent images, no collective)",
                       "stream_dtype": args.stream, "operands": "fp16 x fp16 -> fp32 accumulate",
                       "l2": "per-step working set (GBs of activations + 1.9 GB weights) >> 126 MB L2; no flush needed"},
            "e2e": {"value": e2e_value, "unit": "images/s", "h2d_bytes_per_step": host_rgb.numel() * 4,
                    "d2h_bytes_per_step": host_out.numel() * 4, "ms_per_step": e2e_ms / args.steps,
                    "host_dtype": "fp32 pinned"},
            "gpu_launches": launches,
            "step_tensor_tflops": total_flops / (ms / 1e3) / 1e12,
            "step_tensor_frac": total_flops / (ms / 1e3) / 1e12 / peak,
            "tensor_flops_per_step_by_kind": flops_by_kind,
            "breakdown_ms_eager_step": {k: round(v, 2) for k, v in sorted(breakdown.items(), key=lambda kv: -kv[1])},
            "roofline": {"kernel": "gemm_conv_kernel (implicit-GEMM conv3x3, tcgen05+TMA)", "bound": "tensor",
                         "achieved": conv_tf, "peak": peak, "unit": "TFLOP/s", "frac": conv_tf / peak,
                         "traffic": traffic, "traffic_of": traffic_of, "peak_source": f"{peaks['source']} bf16_tflops_sustained (kernel timed inside a long step)",
                         "launches_timed": n_conv, "avg_launch_ms": conv_ms / max(1, n_conv),
                         "share_of_step": (conv_ms / rsteps) / (ms / args.steps),
                         "timed_in": f"{rsteps} eagerly launched steps of the same workload ({ms_eager:.1f} ms/step eager)"},
            "clocks": clocks,
        }
        if unet_ms is not None:
            out["unet_fwd_ms"] = unet_ms
            out["unet_tensor_frac"] = unet_flops / (unet_ms / 1e3) / 1e12 / peak
        if fast is not None:
            out["fast_mode"] = fast
        if dumped is not None:
            out["dumped_outputs"] = dumped

    # ---- BASELINE.json configs[2]: the training step with its gradient all-reduce.  Every rank runs it in a CHILD
    # process with its own process group (MASTER_PORT + 1): a fault or a stuck collective in the training leg can then
    # never take the headline line down with it — the child is killed by PID after the timeout and its error recorded.
    if wl == "marigold" and not args.no_train:
        # release EVERYTHING this process holds on the GPU first: the child peaks at ~93 GB, and captured graphs keep their
        # private pools (tens of GB of activations) alive through reference cycles until the cyclic GC runs — a child
        # squeezed by the parent's leftovers spends its step in allocator retries (observed: 160 -> 240 -> 425 ms)
        import gc
        pipe.__dict__.pop("_graphs", None)
        del pipe
        infer = step_resident = step_e2e = None     # closures over the pipeline
        gc.collect()
        torch.cuda.empty_cache()
        free_b, total_b = torch.cuda.mem_get_info(dev)
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        t = _train_subprocess(world, rank, local, args.steps, max(args.warmup, 4))
        if rank == 0:
            if isinstance(t, dict):
                t["gpu_free_gb_at_start"] = free_b / 2 ** 30
            out["train_step"] = t
        world_pg = False
    else:
        world_pg = world > 1
    if world_pg:
        dist.barrier()
    if rank == 0:
        if not args.no_cpu_baseline and world == 1:
            try:
                out["cpu_baseline"] = cpu_baseline_leg()
            except Exception as e:  # noqa: BLE001
                out["cpu_baseline"] = {"error": repr(e)[:200]}
        print(json.dumps(out))
    if world_pg:
        dist.destroy_process_group()


def _train_subprocess(world, rank, local, steps, warmup, timeout_s=420):
    """Run `bench.py --workload train --steps steps` for this rank in a child process (own NCCL group on
    MASTER_PORT + 1)."""
    env = dict(os.environ)
    env.update(RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(local),
               MASTER_ADDR=env.get("MASTER_ADDR", "127.0.0.1"), MASTER_PORT=str(int(env.get("MASTER_PORT", "29500")) + 1))
    for k in ("TORCHELASTIC_RUN_ID", "TORCHELASTIC_RESTART_COUNT", "TORCHELASTIC_MAX_RESTARTS",
              "TORCHELASTIC_USE_AGENT_STORE", "TORCH_NCCL_ASYNC_ERROR_HANDLING"):
        env.pop(k, None)                       # the child rendezvous is a plain env:// TCP store on the new port
    cmd = [sys.executable, os.path.abspath(__file__), "--workload", "train", "--gpus", str(world), "--steps", str(steps),
           "--warmup", str(warmup), "--res", "768", "--batch", "2"]
    try:
        p = subprocess.Popen(cmd, env=env, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
        try:
            so, se = p.communicate(timeout=timeout_s)
        except subprocess.TimeoutExpired:
            p.kill()                           # exact PID of the child this rank started
            so, se = p.communicate()
            return {"error": f"training leg timed out after {timeout_s} s", "stderr_tail": (se or "")[-300:]}
        if rank != 0:
            return None
        for line in reversed((so or "").strip().splitlines()):
            if line.startswith("{"):
                return json.loads(line).get("train_step")
        return {"error": f"training leg rc={p.returncode}", "stderr_tail": (se or "")[-300:]}
    except Exception as e:  # noqa: BLE001
        return {"error": repr(e)[:300]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="engine", choices=["engine", "reference"])
    ap.add_argument("--workload", default="marigold", choices=["marigold", "normals", "geowizard", "train"],
                    help="marigold = configs[1] (headline); normals = configs[4] (bs 16, --res sweep); geowizard = "
                         "configs[3] (bs 4, joint attention); train = configs[2] (bs 2/GPU training step)")
    ap.add_argument("--batch", type=int, default=0, help="images per GPU per step (default: the config's)")
    ap.add_argument("--res", type=int, default=768)
    ap.add_argument("--stream", default="fp32", choices=["fp32", "mixed", "fp16"],
                    help="residual-stream dtype in the engine (mixed = fp32 in the UNet, fp16 in the VAE)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-train", action="store_true", help="skip the configs[2] training-step leg of the default line")
    ap.add_argument("--no-fast", action="store_true", help="skip the fp16-stream timing of the default line")
    ap.add_argument("--dump-shapes", action="store_true", help="write per-shape conv timings to gpurun_out/")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one returned as DIR/<name>.npy (float32, rank 0; "
                         "a fixed seeded sample when above 64 MB in all; inputs and weights are seeded)")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl == "reference" or args.workload == "train"):
        ap.error("--dump-outputs covers the engine's inference workloads")
    if args.impl == "reference":
        run_reference(args)
    elif args.workload == "train":
        run_train(args)
    else:
        run_engine(args)


if __name__ == "__main__":
    main()
