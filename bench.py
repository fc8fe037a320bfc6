#!/usr/bin/env python
"""Benchmark of the APTP hot path: mixed-expert gated SD-2.1 U-Net denoising step on B200.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

One "step" = one U-Net forward over one batch of synthetic input (BASELINE.json configs[1]: bf16,
batch 64 per GPU, 64x64 latent, 8 architecture codes with width + depth gating, random-init weights).
`value` is timed with the inputs resident in HBM; `e2e` runs the same step through the public API
(`UNet2DConditionModelGated.forward`) from pinned HOST buffers with the H2D / D2H copies inside the
timed region. `--impl reference` times the reference's CPU path (the fp32 oracle restatement; the
reference has no separate CPU implementation and diffusers is not installable offline) on the host
cores, on a bounded sample of the same workload.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "mixed_expert_unet_samples_steps_per_s"
UNIT = "samples*steps/s"
BATCH, LATENT, N_CODES, N_CTX, CTX_DIM = 64, 64, 8, 77, 1024
DENSE_TFLOP_PER_SAMPLE = 0.7767  # SURVEY Appendix C: 388.35 GMACs at 64x64


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"tflops": d["bf16_tflops"], "tflops_sustained": d.get("bf16_tflops_sustained"), "hbm": d["hbm_gbs"],
                "source": "measured (MEASURED_PEAKS.json)"}
    return {"tflops": 1590.0, "tflops_sustained": 1400.0, "hbm": 6650.0, "source": "fallback (B200_PROFILING.md)"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region. The sampler is started before the warm-up
    (nvidia-smi can take longer than a short timed region to print its first line); every line is time-stamped on
    arrival and only lines inside [begin(), end()] count. If fewer than 3 lines fell inside (very short runs), the
    caller keeps the same workload running untimed until enough samples under load exist (`extend`)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.proc, self.lines = index, None, []
        self.t0, self.t1, self.extended = None, None, False

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "50", "-i", str(self.index)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:  # noqa: BLE001
            self.proc = None
        self.t0 = time.time()

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def begin(self):
        self.t0 = time.time()

    def end(self):
        self.t1 = time.time()

    def in_window(self):
        t1 = self.t1 if self.t1 is not None else time.time()
        return [ln for ts, ln in self.lines if self.t0 <= ts <= t1 + 0.02]

    def extend(self, fn, min_samples: int = 3, max_seconds: float = 3.0):
        """Keep `fn` (one more untimed step of the same workload) running until min_samples lines exist under load."""
        import torch
        if self.proc is None or len(self.in_window()) >= min_samples:
            return
        self.extended = True
        t_stop = time.time() + max_seconds
        while time.time() < t_stop:
            fn()
            torch.cuda.synchronize()
            self.t1 = time.time()
            if len(self.in_window()) >= min_samples:
                break

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        if self.t1 is None:
            self.t1 = time.time()
        time.sleep(0.08)
        self.proc.terminate()
        sm, smax, reasons = [], None, set()
        for ln in self.in_window():
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1]))
                smax = float(f[2])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        out = {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": smax, "reasons": sorted(reasons),
               "samples": len(sm)}
        if self.extended:
            out["note"] = "timed region shorter than the sampling latency: samples taken while the same step kept running"
        return out


_DIST = {}


def init_dist():
    """(rank, world, local, device); the NCCL process group is created once per process and shared by every workload
    measured in this run (forward, then the `secondary` train / sampling numbers)."""
    import torch
    import torch.distributed as dist
    if _DIST:
        return _DIST["v"]
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the product path has no CPU fallback")
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    if world > 1 and not dist.is_initialized():
        dist.init_process_group("nccl", device_id=device)
    _DIST["v"] = (rank, world, local, device)
    return _DIST["v"]


def finish_dist():
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized():
        dist.destroy_process_group()


def dump_outputs(args, world, rank, **arrays):
    """--dump-outputs DIR: each array as DIR/<name>.npy in float32, or DIR/<name>_rank<k>.npy when several ranks run
    (every rank draws its own seeded inputs)."""
    if not args.dump_outputs:
        return
    import numpy as np
    os.makedirs(args.dump_outputs, exist_ok=True)
    suffix = f"_rank{rank}" if world > 1 else ""
    for name, a in arrays.items():
        np.save(os.path.join(args.dump_outputs, f"{name}{suffix}.npy"), a.detach().float().cpu().numpy())


def sampled_entries(tensors, n: int, seed: int = 0):
    """A fixed, seeded sample of n entries (positions drawn with replacement, sorted) of the concatenation of
    `tensors`, for outputs too large to store whole."""
    import torch
    sizes = torch.tensor([t.numel() for t in tensors])
    ends = torch.cumsum(sizes, 0)
    pos = torch.randint(0, int(ends[-1]), (n,), generator=torch.Generator().manual_seed(seed)).sort().values
    which = torch.searchsorted(ends, pos, right=True)
    off = pos - (ends - sizes)[which]
    parts = []
    for i in which.unique().tolist():
        sel = which == i
        parts.append(tensors[i].detach().reshape(-1)[off[sel].to(tensors[i].device)].float().cpu())
    return torch.cat(parts)


def make_workload(device, seed):
    import torch
    from diffusion_pruning_b200.synthetic import split_arch, synthetic_codes
    from diffusion_pruning_b200.unet import UNet2DConditionModelGated
    torch.manual_seed(seed)
    with torch.device(device):
        model = UNet2DConditionModelGated()  # SD-2.1 layout, PyTorch default (random) init, on the GPU
    model.eval()
    st = model.get_structure()
    codes = synthetic_codes(st, N_CODES, seed=2)
    g = torch.Generator().manual_seed(3)
    assign = torch.arange(BATCH) % N_CODES
    assign = assign[torch.randperm(BATCH, generator=g)]
    arch = codes[assign].to(device)
    model.set_structure(split_arch(arch, st))
    g = torch.Generator().manual_seed(seed + 11)
    sample = torch.randn(BATCH, 4, LATENT, LATENT, generator=g)
    ctx = torch.randn(BATCH, N_CTX, CTX_DIM, generator=g)
    t = torch.randint(0, 1000, (BATCH,), generator=g).float()
    return model, codes, assign, sample, ctx, t


def run_ours(args):
    import torch
    import torch.distributed as dist
    rank, world, local, device = init_dist()
    from diffusion_pruning_b200 import kernels as K
    model, codes, assign, sample, ctx, t = make_workload(device, seed=1234 + rank)
    sample_h, ctx_h, t_h = sample.pin_memory(), ctx.pin_memory(), t.pin_memory()
    out_h = torch.empty(BATCH, 4, LATENT, LATENT).pin_memory()
    sample_d, ctx_d, t_d = sample.to(device), ctx.to(device), t.to(device)

    def step_resident():
        with torch.no_grad():
            return model(sample_d, t_d, ctx_d).sample

    def step_e2e():
        with torch.no_grad():
            s = sample_h.to(device, non_blocking=True)
            c = ctx_h.to(device, non_blocking=True)
            tt = t_h.to(device, non_blocking=True)
            y = model(s, tt, c).sample
            out_h.copy_(y, non_blocking=True)
        torch.cuda.current_stream().synchronize()  # the user reads the result every step

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        """(ms over `steps` calls of fn, what the last call returned)"""
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            y = fn()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        if world > 1:
            tt = torch.tensor([ms], device=device)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            ms = float(tt.item())
        barrier()
        return ms, y

    clocks = ClockSampler(local)
    clocks.start()
    for _ in range(max(args.warmup, 3)):
        step_resident()
    K.check_abort()
    if os.environ.get("APTP_CUDA_PROFILE"):  # ncu --profile-from-start off: capture exactly one step
        torch.cuda.profiler.start()
        step_resident()
        torch.cuda.synchronize()
        torch.cuda.profiler.stop()
    clocks.begin()
    ms_total, y_last = timed(step_resident, args.steps)
    clocks.end()
    clocks.extend(step_resident)
    clk = clocks.stop()
    # the forward returns a fresh tensor every step (a graph replay returns a copy of its static output), so y_last
    # still holds the prediction of the last timed step
    dump_outputs(args, world, rank, sample=y_last)
    del y_last
    eng = model._engine
    launches_per_step = eng.launches
    kept_flops = eng.flops
    gemm_alg_bytes = eng.gemm_bytes
    # end-to-end through the public API with host buffers
    for _ in range(2):
        step_e2e()
    t0 = time.perf_counter()
    ms_e2e_dev, _ = timed(step_e2e, args.steps)
    ms_e2e = ms_e2e_dev
    # per-kernel timing of the dominant kernel, live, with CUDA events on the launching stream
    # (eager launches, each bracketed by two events. The GPU is first parked on a spin kernel so that the host has queued the
    # whole forward before the first kernel runs -- otherwise an event pair also times the host's launch latency whenever
    # the GPU catches up with the launching thread -- and every launch takes the median of three such passes.)
    passes = []
    for _ in range(3):
        eng.profile = []
        torch.cuda._sleep(int(60e6))  # ~35 ms at 1.7 GHz
        step_resident()
        torch.cuda.synchronize()
        passes.append(eng.profile)
    eng.profile = None
    prof = []
    for i, (kind, a, b, fl, label) in enumerate(passes[0]):
        ms = sorted(p_[i][1].elapsed_time(p_[i][2]) for p_ in passes)[1]
        prof.append((kind, ms, fl, label))
    if os.environ.get("APTP_PROFILE_DUMP") and rank == 0:
        with open(os.environ["APTP_PROFILE_DUMP"], "w") as f:
            for kind, ms, fl, label in prof:
                f.write(f"{kind}\t{ms:.4f}\t{fl / 1e9:.2f}\t{fl / max(ms, 1e-6) / 1e9:.1f}\t{label}\n")
    gemm = [(ms, fl) for kind, ms, fl, _ in prof if kind == "gemm" and fl > 0]
    attn = [(ms, fl) for kind, ms, fl, _ in prof if kind == "attn"]
    hbm = [(ms, nb) for kind, ms, nb, _ in prof if kind == "hbm"]
    g_ms, g_fl = sum(x for x, _ in gemm), sum(f for _, f in gemm)
    a_ms, a_fl = sum(x for x, _ in attn), sum(f for _, f in attn)
    h_ms, h_bytes = sum(x for x, _ in hbm), sum(b for _, b in hbm)
    K.check_abort()
    peaks = load_peaks()
    traffic, traffic_src = {}, None
    tp = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tp):  # ncu DRAM bytes of the same command (tools/gpu_ncu.sh), per launch
        tj = json.load(open(tp))
        traffic, traffic_src = tj.get("grouped_gemm_kernel", {}), tj.get("source")
    ms_step = ms_total / args.steps
    value = BATCH * world * args.steps / (ms_total / 1e3)
    e2e_value = BATCH * world * args.steps / (ms_e2e / 1e3)
    out = {
        "metric": METRIC, "value": round(value, 2), "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": round(ms_step, 3), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": {"workload": "configs[1]: mixed-expert gated SD-2.1 U-Net forward, bf16, batch 64/GPU, 64x64 latent, "
                               "8 codes with width+depth gating, random-init weights",
                   "batch_per_gpu": BATCH, "latent": LATENT, "codes": N_CODES, "parallelism": f"dp{world} over prompts",
                   "l2": "activations per step (several GB) exceed the 126 MB L2; no explicit flush",
                   "kept_tflop_per_step_per_gpu": round(kept_flops / 1e12, 3),
                   "dense_tflop_per_step_per_gpu": round(BATCH * DENSE_TFLOP_PER_SAMPLE, 3)},
        "e2e": {"value": round(e2e_value, 2), "unit": UNIT,
                "h2d_bytes_per_step": int(sample_h.numel() * 4 + ctx_h.numel() * 4 + t_h.numel() * 4),
                "d2h_bytes_per_step": int(out_h.numel() * 4), "ms_per_step": round(ms_e2e / args.steps, 3)},
        "gpu_launches": int(launches_per_step * args.steps),
        "clocks": clk,
        "roofline": {"bound": "tensor", "kernel": "grouped_gemm_kernel (tcgen05 grouped GEMM / implicit conv)",
                     "achieved": round(g_fl / (g_ms / 1e3) / 1e12, 1) if g_ms else None, "peak": peaks["tflops"],
                     "unit": "TFLOP/s", "frac": round(g_fl / (g_ms / 1e3) / 1e12 / peaks["tflops"], 4) if g_ms else None,
                     "traffic": traffic.get("dram_bytes_per_launch"), "traffic_source": traffic_src,
                     "algorithmic_bytes_per_launch": round(gemm_alg_bytes / max(len(gemm), 1)),
                     "algorithmic_flop_per_launch": round(g_fl / max(len(gemm), 1)),
                     "peak_source": peaks["source"], "peak_sustained": peaks["tflops_sustained"],
                     "launches": len(gemm), "kernel_ms_per_step": round(g_ms, 3),
                     "attention": {"achieved": round(a_fl / (a_ms / 1e3) / 1e12, 1) if a_ms else None,
                                   "kernel_ms_per_step": round(a_ms, 3), "launches": len(attn)},
                     "step_frac_of_peak_kept_work": round(kept_flops / (ms_step / 1e3) / 1e12 / peaks["tflops"], 4),
                     "dense_equivalent_tflops": round(BATCH * DENSE_TFLOP_PER_SAMPLE / (ms_step / 1e3), 1)},
    }
    # Re-structuring cost (the reference calls set_structure for every prompt batch, pruning_pipelines.py:757-759): a
    # FRESH random prompt -> expert assignment of the same 8 codes, set_structure, first forward, host-timed with a
    # synchronize on both sides; and the throughput when EVERY step brings a new assignment (no CUDA-graph reuse unless
    # the engine can key its cached state on something coarser than the exact assignment).
    from diffusion_pruning_b200.synthetic import split_arch as _split
    st_ = model.get_structure()
    gr = torch.Generator().manual_seed(99 + rank)

    def fresh_arch():
        a = torch.randint(0, N_CODES, (BATCH,), generator=gr)
        return codes[a].to(device)
    restruct = []
    for _ in range(3):
        arch_new = fresh_arch()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        model.set_structure(_split(arch_new, st_))
        step_resident()
        torch.cuda.synchronize()
        restruct.append((time.perf_counter() - t0) * 1e3)
    n_fresh = max(4, min(args.steps, 10))
    archs = [fresh_arch() for _ in range(n_fresh)]
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for a in archs:
        model.set_structure(_split(a, st_))
        step_resident()
    torch.cuda.synchronize()
    fresh_ms = (time.perf_counter() - t0) * 1e3 / n_fresh
    out["restructure_ms"] = round(sorted(restruct)[1], 2)
    out["restructure_note"] = ("host-timed median of 3: fresh random assignment of the same codes -> set_structure -> first "
                               "forward -> synchronize (bucketing, schedule builds for new bucket sizes, eager forward)")
    out["value_fresh_assignment"] = round(BATCH * world / (fresh_ms / 1e3), 2)
    out["ms_per_step_fresh_assignment"] = round(fresh_ms, 3)
    # flat copies of the per-kernel-class numbers (the nested dict above is kept for continuity with round 1)
    out.update({
        "attention_tflops": round(a_fl / (a_ms / 1e3) / 1e12, 1) if a_ms else None, "attention_ms": round(a_ms, 3),
        "attention_frac": round(a_fl / (a_ms / 1e3) / 1e12 / peaks["tflops"], 4) if a_ms else None,
        "gemm_tflops": round(g_fl / (g_ms / 1e3) / 1e12, 1) if g_ms else None, "gemm_ms": round(g_ms, 3),
        "hbm_kernels_gbs": round(h_bytes / (h_ms / 1e3) / 1e9, 1) if h_ms else None, "hbm_kernels_ms": round(h_ms, 3),
        "hbm_frac": round(h_bytes / (h_ms / 1e3) / 1e9 / peaks["hbm"], 4) if h_ms else None, "hbm_peak_gbs": peaks["hbm"],
        "hbm_kernels": "GroupNorm statistics + apply(+SiLU/gate), LayerNorm: algorithmic bytes (read once, write once) "
                       "/ CUDA-event time of each launch",
        "step_frac_of_peak_kept_work": out["roofline"]["step_frac_of_peak_kept_work"],
    })
    # free the forward model before the other workloads
    del model, eng
    torch.cuda.empty_cache()
    if world == 1 and not args.no_library_baseline:
        lb = library_baseline(device, codes, assign) if rank == 0 else None
        if rank == 0:
            out["library_baseline"] = lb
            if lb.get("mixed_expert"):
                out["vs_library_mixed"] = round(value / lb["mixed_expert"]["value"], 3)
                out["vs_library_dense"] = round(value / lb["dense"]["value"], 3)
    if not args.no_secondary:
        sec = secondary_workloads(args)
        out["secondary"] = sec
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        out["cpu_baseline"], _ = cpu_baseline(sample_steps=1)
    if rank == 0:
        print(json.dumps(out), flush=True)


def measure_train(args):
    """BASELINE configs[2]: pruning train step (DDPM + distillation + block + resource + contrastive losses, gate
    backward, Sinkhorn router, AdamW on hypernet + codebook), 32 samples per GPU at 64x64, data parallel with a
    gradient all-reduce. Secondary workload (`--workload train`); the default bench line stays configs[1]."""
    import torch
    import torch.distributed as dist
    rank, world, local, device = init_dist()
    from diffusion_pruning_b200 import HyperStructure, StructureVectorQuantizer
    from diffusion_pruning_b200 import kernels as K
    from diffusion_pruning_b200 import pruning_step as PS
    from diffusion_pruning_b200.synthetic import DEPTH_ORDER
    from diffusion_pruning_b200.unet import UNet2DConditionModelGated
    Bt = args.train_batch
    torch.manual_seed(1234)
    with torch.device(device):
        unet = UNet2DConditionModelGated()
    unet.eval()
    unet.freeze()
    st = unet.get_structure()
    torch.manual_seed(7)
    hyper = HyperStructure(structure=st, input_dim=768, wn_flag=False, linear_bias=True).to(device)
    quant = StructureVectorQuantizer(n_e=N_CODES, structure=st, beta=0.25, temperature=0.4, base=3,
                                     depth_order=list(DEPTH_ORDER), non_zero_width=True,
                                     resource_aware_normalization=False, optimal_transport=True).to(device)
    quant.train()
    hyper.train()
    unet.count_macs(LATENT, LATENT)
    cfg = PS.PruningLossConfig()
    p_actual = PS.actual_pruning_target(unet, cfg.pruning_target)
    taps = PS.BlockTaps(unet)
    params = [p for p in list(hyper.parameters()) + list(quant.parameters()) if p.requires_grad]
    opt = torch.optim.AdamW(params, lr=2e-4)
    g = torch.Generator().manual_seed(100 + rank)
    host = {"noisy_latents": torch.randn(Bt, 4, LATENT, LATENT, generator=g).pin_memory(),
            "timesteps": torch.randint(0, 1000, (Bt,), generator=g).pin_memory(),
            "target": torch.randn(Bt, 4, LATENT, LATENT, generator=g).pin_memory(),
            "encoder_hidden_states": torch.randn(Bt, N_CTX, CTX_DIM, generator=g).pin_memory(),
            "mpnet_embeddings": torch.randn(Bt, 768, generator=g).pin_memory()}
    acp = PS.alphas_cumprod().to(device)
    # DDP semantics (trainer.py:782, :922) without per-parameter copies: every trainable gradient is a VIEW of one flat
    # fp32 buffer (autograd accumulates into the views in place), so the mean over ranks is ONE NCCL all-reduce of
    # 1.26 M floats and "zero_grad" is one memset. The all-reduce is timed with CUDA events on its own.
    flat = torch.zeros(sum(p.numel() for p in params), device=device)
    off = 0
    for p in params:
        p.grad = flat[off:off + p.numel()].view_as(p)
        off += p.numel()
    ar_events = []

    def step():
        batch = {k: v.to(device, non_blocking=True) for k, v in host.items()}
        out = PS.pruning_step(unet, hyper, quant, batch, cfg, taps, p_actual, acp=acp)
        flat.zero_()
        out["loss"].backward()
        if world > 1:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            dist.all_reduce(flat)
            flat.div_(world)
            e1.record()
            ar_events.append((e0, e1))
        opt.step()
        return out["loss"].detach()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(args.warmup, 3)):
        loss = step()
    K.check_abort()
    if os.environ.get("APTP_CUDA_PROFILE"):  # ncu --profile-from-start off: capture exactly one train step
        torch.cuda.synchronize()
        torch.cuda.profiler.start()
        step()
        torch.cuda.synchronize()
        torch.cuda.profiler.stop()
    clocks = ClockSampler(local)
    clocks.start()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        loss = step()
        loss_h = float(loss)  # the trainer reads the loss every step (D2H)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    if world > 1:
        tt = torch.tensor([ms], device=device)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        ms = float(tt.item())
    clk = clocks.stop()
    K.check_abort()
    dump_outputs(args, world, rank, train_loss=loss, train_grad=flat)  # flat: the last step's (reduced) gradients
    peaks = load_peaks()
    value = Bt * world * args.steps / (ms / 1e3)
    tflop_per_sample = 2.52  # SURVEY 8(d): two forwards + dgrad-only backward at 64x64
    out = {"metric": "pruning_train_samples_steps_per_s", "value": round(value, 2), "unit": UNIT, "n_gpus": world,
           "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": round(ms / args.steps, 3),
           "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
           "config": {"workload": "configs[2]: pruning train step (teacher + student forward, backward to the gates, "
                                  "Sinkhorn router, 7 losses, AdamW on hypernet + codebook), 64x64 latent",
                      "batch_per_gpu": Bt, "latent": LATENT, "codes": N_CODES, "parallelism": f"dp{world} + grad all-reduce",
                      "l2": "activations exceed L2"},
           "e2e": {"value": round(value, 2), "unit": UNIT,
                   "h2d_bytes_per_step": int(sum(v.numel() * v.element_size() for v in host.values())),
                   "d2h_bytes_per_step": 4},
           "gpu_launches": None, "clocks": clk, "final_loss": loss_h,
           "grad_allreduce_ms": (round(sum(a.elapsed_time(b) for a, b in ar_events[-args.steps:]) / args.steps, 3)
                                 if ar_events else None),
           "roofline": {"bound": "tensor", "achieved": round(Bt * tflop_per_sample / (ms / args.steps / 1e3), 1),
                        "peak": peaks["tflops"], "unit": "TFLOP/s",
                        "frac": round(Bt * tflop_per_sample / (ms / args.steps / 1e3) / peaks["tflops"], 4),
                        "note": "whole-step dense-equivalent FLOPs (2.52 TFLOP/sample) / step time", "traffic": None}}
    taps.remove() if hasattr(taps, "remove") else None
    return out


def measure_sample(args):
    """BASELINE configs[3]: expert-routed 25-step DDIM sampling at 96x96 latents with classifier-free guidance. Every
    rank routes its own prompts (hypernet + eval cosine argmax), an all-to-all sends each prompt to the GPU that owns
    its expert (expert e lives on rank e % world), the whole scheduler loop runs there (gated U-Net on the doubled CFG
    batch + the fused CFG/DDIM kernel), a second all-to-all returns the final latents. A bench "step" is one such
    sampling pass over the rank's prompts; value counts prompt x DDIM-step units (each is TWO U-Net samples: cond +
    uncond)."""
    import torch
    import torch.distributed as dist
    rank, world, local, device = init_dist()
    from diffusion_pruning_b200 import HyperStructure, StructureVectorQuantizer
    from diffusion_pruning_b200 import kernels as K
    from diffusion_pruning_b200 import sampling as S
    from diffusion_pruning_b200.synthetic import DEPTH_ORDER, synthetic_codes
    from diffusion_pruning_b200.unet import UNet2DConditionModelGated
    P, H, STEPS = args.prompts, args.sample_latent, args.ddim_steps
    torch.manual_seed(1234)
    with torch.device(device):
        unet = UNet2DConditionModelGated()
    unet.eval()
    st = unet.get_structure()
    torch.manual_seed(7)
    hyper = HyperStructure(structure=st, input_dim=768, wn_flag=False, linear_bias=True).to(device).eval()
    quant = StructureVectorQuantizer(n_e=N_CODES, structure=st, beta=0.25, temperature=0.4, base=3,
                                     depth_order=list(DEPTH_ORDER), non_zero_width=True,
                                     resource_aware_normalization=False, optimal_transport=True).to(device)
    quant.eval()
    codes = synthetic_codes(st, N_CODES).float()
    quant.embedding_gs.data = (codes * 0.9 + 0.05).to(device)  # soft codebook rows; eval routing thresholds them
    g = torch.Generator().manual_seed(300 + rank)
    # Synthetic prompt embeddings that the (random-init, linear) hypernet maps near the codes in round-robin order, so
    # that the router really spreads the prompts over the experts: least-squares pre-images of +-4 logits, plus noise.
    with torch.no_grad():
        Wh = torch.cat([l.weight for l in hyper.mh_fc], 0).float().cpu()
        bh = torch.cat([l.bias for l in hyper.mh_fc], 0).float().cpu()
        want = (2.0 * codes[(torch.arange(P) + rank * P) % N_CODES] - 1.0) * 4.0 - bh
        prompt = torch.linalg.lstsq(Wh, want.t()).solution.t().contiguous()
        prompt = prompt + 0.02 * prompt.std() * torch.randn(P, 768, generator=g)
    host = {"prompt": prompt.pin_memory(),
            "latents": torch.randn(P, 4, H, H, generator=g).pin_memory(),
            "cond": torch.randn(P, N_CTX, CTX_DIM, generator=g).pin_memory(),
            "uncond": torch.randn(1, N_CTX, CTX_DIM, generator=g).expand(P, -1, -1).contiguous().pin_memory()}
    acp = S.alphas_cumprod()
    result = torch.empty(P, 4, H, H).pin_memory()

    def step():
        d = {k: v.to(device, non_blocking=True) for k, v in host.items()}
        out, idx = S.routed_sampling(unet, hyper, quant, d["prompt"], d["latents"], d["cond"], d["uncond"],
                                     num_inference_steps=STEPS, guidance_scale=7.5, acp=acp)
        result.copy_(out, non_blocking=True)
        return idx

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(args.warmup, 1)):
        idx = step()
    K.check_abort()
    clocks = ClockSampler(local)
    clocks.start()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        idx = step()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    counts = torch.bincount(idx, minlength=N_CODES).float()
    if world > 1:
        tt = torch.tensor([ms], device=device)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        ms = float(tt.item())
        dist.all_reduce(counts)
    clk = clocks.stop()
    K.check_abort()
    assert torch.isfinite(result).all(), "sampling produced non-finite latents"
    dump_outputs(args, world, rank, sample_latents=result, sample_experts=idx)
    value = P * world * STEPS * args.steps / (ms / 1e3)
    if True:
        out = {"metric": "routed_sampling_prompt_steps_per_s", "value": round(value, 2), "unit": "prompts*steps/s",
               "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 1),
               "ms_per_step": round(ms / args.steps, 3), "higher_is_better": True, "scaling": "weak",
               "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
               "config": {"workload": f"configs[3]: expert-routed {STEPS}-step DDIM sampling with CFG 7.5, {H}x{H} "
                                      f"latent, {N_CODES} experts (expert e on rank e % world), all-to-all prompt "
                                      f"dispatch + return, random-init weights",
                          "prompts_per_gpu": P, "latent": H, "ddim_steps": STEPS, "codes": N_CODES,
                          "unet_samples_per_prompt_step": 2, "parallelism": f"ep{world} over experts",
                          "prompts_per_expert": [int(c) for c in counts.tolist()],
                          "l2": "activations exceed L2"},
               "prompts_per_s": round(P * world * args.steps / (ms / 1e3), 3),
               "unet_samples_steps_per_s": round(2 * value, 2),
               "e2e": {"value": round(value, 2), "unit": "prompts*steps/s",
                       "h2d_bytes_per_step": int(sum(v.numel() * v.element_size() for v in host.values())),
                       "d2h_bytes_per_step": int(result.numel() * result.element_size())},
               "gpu_launches": None, "clocks": clk}
    return out


def measure_finetune(args):
    """SURVEY 8(f) rank 4: the fine-tune step of one static expert (FineTuner.step, trainer.py:1683-1765, from the encoded
    batch on): dense teacher forward (no grad), student forward + backward to EVERY U-Net parameter (dgrad + tcgen05
    wgrad + norm-affine + attention backward), DDPM / distillation / block losses, AdamW over the 866 M parameters."""
    import torch
    import torch.distributed as dist
    rank, world, local, device = init_dist()
    from diffusion_pruning_b200 import finetune as FT
    from diffusion_pruning_b200 import kernels as K
    from diffusion_pruning_b200 import pruning_step as PS
    from diffusion_pruning_b200.synthetic import split_arch, synthetic_codes
    from diffusion_pruning_b200.unet import UNet2DConditionModelGated, UNet2DConditionModelPruned
    Bt = args.train_batch
    torch.manual_seed(1234)
    with torch.device(device):
        unet = UNet2DConditionModelPruned()   # what FineTuner trains (trainer.py:1452-1462): prune() semantics
        teacher = UNet2DConditionModelGated()
    teacher.load_state_dict(unet.state_dict())
    teacher.eval()
    teacher.freeze()
    teacher.set_all_ones_structure(1, device=device)
    unet.train()
    st = unet.get_structure()
    code = synthetic_codes(st, N_CODES)[3:4].float().to(device)
    unet.prune_to(code * 0.9 + 0.05)      # soft codebook row (quantizer_embeddings.pt), thresholded like prune()
    unet.enable_weight_training(True)
    cfg = FT.FinetuneLossConfig()
    taps, ttaps = PS.BlockTaps(unet), PS.BlockTaps(teacher)
    params = [p for p in unet.parameters() if p.requires_grad]
    opt = torch.optim.AdamW(params, lr=1e-5, weight_decay=0.0, fused=True)
    g = torch.Generator().manual_seed(100 + rank)
    host = {"noisy_latents": torch.randn(Bt, 4, LATENT, LATENT, generator=g).pin_memory(),
            "timesteps": torch.randint(0, 1000, (Bt,), generator=g).pin_memory(),
            "target": torch.randn(Bt, 4, LATENT, LATENT, generator=g).pin_memory(),
            "encoder_hidden_states": torch.randn(Bt, N_CTX, CTX_DIM, generator=g).pin_memory()}
    acp = PS.alphas_cumprod().to(device)

    def step():
        batch = {k: v.to(device, non_blocking=True) for k, v in host.items()}
        out = FT.finetune_step(unet, teacher, batch, cfg, taps, ttaps, acp=acp)
        opt.zero_grad(set_to_none=True)
        out["loss"].backward()
        if world > 1:  # DDP semantics: mean of the gradients
            for p in params:
                if p.grad is not None:
                    dist.all_reduce(p.grad)
                    p.grad.div_(world)
        opt.step()
        return out["loss"].detach()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(args.warmup, 3)):
        loss = step()
    K.check_abort()
    if os.environ.get("APTP_CUDA_PROFILE"):
        torch.cuda.synchronize()
        torch.cuda.profiler.start()
        step()
        torch.cuda.synchronize()
        torch.cuda.profiler.stop()
    clocks = ClockSampler(local)
    clocks.start()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        loss = step()
        loss_h = float(loss)  # the trainer reads the loss every step (D2H)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    if world > 1:
        tt = torch.tensor([ms], device=device)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        ms = float(tt.item())
    clk = clocks.stop()
    K.check_abort()
    if args.dump_outputs:  # the last step's gradients cover 866 M parameters: a fixed sample of 2^20 of them
        dump_outputs(args, world, rank, finetune_loss=loss,
                     finetune_grad_sample=sampled_entries([p.grad for p in params if p.grad is not None], 1 << 20))
    peaks = load_peaks()
    value = Bt * world * args.steps / (ms / 1e3)
    # dense-equivalent FLOPs per sample: teacher forward + student forward + dgrad + wgrad of the conv / linear layers
    # (+ 2.5x forward attention FLOPs for its backward): 2 * (2 * 388.35 + 2 * 325.3 + 2.5 * 63.0) GMAC
    flop_per_sample = 2.0 * (2 * 388.35 + 2 * 325.3 + 2.5 * 63.0) * 1e9
    if True:
        out = {"metric": "finetune_samples_steps_per_s", "value": round(value, 2), "unit": UNIT, "n_gpus": world,
               "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": round(ms / args.steps, 3),
               "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
               "config": {"workload": "fine-tune step of one static expert (SURVEY 8f rank 4; FineTuner.step): dense teacher "
                                      "forward, student forward + backward to all 866 M U-Net parameters, 3 losses, AdamW, "
                                      "64x64 latent", "batch_per_gpu": Bt, "latent": LATENT,
                          "parallelism": f"dp{world} + grad all-reduce", "l2": "activations exceed L2"},
               "e2e": {"value": round(value, 2), "unit": UNIT,
                       "h2d_bytes_per_step": int(sum(v.numel() * v.element_size() for v in host.values())),
                       "d2h_bytes_per_step": 4},
               "gpu_launches": None, "clocks": clk, "final_loss": loss_h,
               "roofline": {"bound": "tensor", "achieved": round(flop_per_sample * Bt * args.steps / (ms / 1e3) / 1e12, 1),
                            "peak": peaks["tflops"], "unit": "TFLOP/s",
                            "frac": round(flop_per_sample * Bt * args.steps / (ms / 1e3) / 1e12 / peaks["tflops"], 4),
                            "traffic": None,
                            "note": "whole-step dense-equivalent FLOPs (3.17 TFLOP/sample) / step time; the student computes "
                                    "gated-off channels too (dense weights)"}}
    return out


def build_oracle_fast():
    """Full-size fp32 oracle with cheap deterministic init (fan-in scaled uniform)."""
    import math
    import torch
    from oracle.unet_oracle import GatedUNetOracle
    with torch.device("meta"):
        o = GatedUNetOracle()
    o = o.to_empty(device="cpu").eval()
    g = torch.Generator().manual_seed(0)
    with torch.no_grad():
        for name, p in o.named_parameters():
            if p.ndim >= 2:
                a = 1.0 / math.sqrt(p[0].numel())
                p.uniform_(-a, a, generator=g)
            elif "norm" in name and name.endswith("weight"):
                p.fill_(1.0)
            else:
                p.zero_()
    return o


def library_baseline(device, codes, assign, steps: int = 20, warmup: int = 5):
    """The "library bar" (SURVEY 8(d), BASELINE.md section 3): what the reference's real execution path -- eager PyTorch on
    cuDNN / cuBLAS / flash-SDPA -- does on the SAME B200 for the SAME workload (configs[1]: batch 64, 64x64 latent, the same
    8 codes and assignment). The reference U-Net (restated: oracle/unet_oracle.py; diffusers is not installable) is moved
    to the GPU in bf16 / channels_last, hard gates are MULTIPLIED as the reference does (nothing is skipped), and the
    dense case (all-ones gates) is timed beside it. A reported baseline, measured with CUDA events after warm-up."""
    import torch
    from diffusion_pruning_b200.synthetic import split_arch
    out = {"unit": UNIT, "kind": "eager PyTorch " + torch.__version__ + " (cuDNN / cuBLAS / SDPA), bf16 weights and "
                                 "activations, channels_last, torch.no_grad, gates multiplied as in the reference",
           "steps": steps, "warmup": warmup, "batch": BATCH, "latent": LATENT}
    try:
        torch.backends.cudnn.benchmark = True
        o = build_oracle_fast().to(device=device, dtype=torch.bfloat16).to(memory_format=torch.channels_last)
        st = o.get_structure()
        g = torch.Generator().manual_seed(11)
        sample = torch.randn(BATCH, 4, LATENT, LATENT, generator=g).to(device, torch.bfloat16)
        sample = sample.contiguous(memory_format=torch.channels_last)
        ctx = torch.randn(BATCH, N_CTX, CTX_DIM, generator=g).to(device, torch.bfloat16)
        t = torch.randint(0, 1000, (BATCH,), generator=g).to(device)
        for name, arch in (("mixed_expert", codes[assign]), ("dense", torch.ones(BATCH, codes.shape[1]))):
            o.set_structure(split_arch(arch.to(device, torch.bfloat16), st))
            with torch.no_grad():
                for _ in range(warmup):
                    o(sample, t, ctx)
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(steps):
                    y = o(sample, t, ctx)
                e1.record()
                torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / steps
            assert torch.isfinite(y.float()).all()
            out[name] = {"value": round(BATCH / (ms / 1e3), 2), "ms_per_step": round(ms, 3),
                         "dense_equivalent_tflops": round(BATCH * DENSE_TFLOP_PER_SAMPLE / (ms / 1e3), 1)}
        del o, sample, ctx, y
        torch.cuda.empty_cache()
    except Exception as e:  # noqa: BLE001 -- a baseline leg must not take the bench line down with it
        out["error"] = repr(e)[:300]
    return out


def secondary_workloads(args):
    """BASELINE configs[2] (pruning train step, gradient all-reduce) and configs[3] (expert-routed sampling, all-to-all)
    measured in the SAME process group as the headline forward, so the driver's per-N lines carry the two multi-GPU
    splits north_star names. Flat keys."""
    import copy
    import torch
    sec = {}
    a = copy.copy(args)
    a.steps, a.warmup = args.secondary_train_steps, 6  # (the allocator re-grows its pools after the library-baseline leg)
    a.dump_outputs = None  # --dump-outputs records the headline forward only
    try:
        tr = measure_train(a)
        sec.update(train_samples_steps_per_s=tr["value"], train_ms=tr["ms_per_step"], train_batch_per_gpu=a.train_batch,
                   train_frac_of_peak=tr["roofline"]["frac"], train_grad_allreduce_ms=tr.get("grad_allreduce_ms"),
                   train_final_loss=tr.get("final_loss"))
    except Exception as e:  # noqa: BLE001
        sec["train_error"] = repr(e)[:300]
    torch.cuda.empty_cache()
    a = copy.copy(args)
    a.steps, a.warmup = 1, 1
    a.dump_outputs = None
    try:
        sm = measure_sample(a)
        sec.update(sample_prompt_steps_per_s=sm["value"], sample_ms_per_pass=sm["ms_per_step"],
                   sample_prompts_per_gpu=a.prompts, sample_latent=a.sample_latent, sample_ddim_steps=a.ddim_steps,
                   sample_unet_samples_steps_per_s=sm["unet_samples_steps_per_s"],
                   sample_prompts_per_expert=sm["config"]["prompts_per_expert"])
    except Exception as e:  # noqa: BLE001
        sec["sample_error"] = repr(e)[:300]
    torch.cuda.empty_cache()
    return sec


def cpu_baseline(sample_steps: int = 1):
    """The reference's CPU path (fp32 oracle restatement) on the host cores: config 1 (batch 4, 64x64). Returns (numbers,
    prediction of the last timed forward)."""
    import torch
    from diffusion_pruning_b200.synthetic import split_arch, synthetic_codes
    threads = os.cpu_count() or 1
    torch.set_num_threads(threads)
    o = build_oracle_fast()
    st = o.get_structure()
    codes = synthetic_codes(st, N_CODES, seed=2)
    arch = codes[[0, 3, 3, 7]]
    g = torch.Generator().manual_seed(1)
    sample = torch.randn(4, 4, LATENT, LATENT, generator=g)
    ctx = torch.randn(4, N_CTX, CTX_DIM, generator=g)
    t = torch.tensor([981, 661, 341, 21])
    o.set_structure(split_arch(arch.clone(), st))
    with torch.no_grad():
        o.set_all_ones(1)
        o(sample[:1], t[:1], ctx[:1])  # warm-up (allocator, thread pool)
        o.set_structure(split_arch(arch.clone(), st))
        t0 = time.perf_counter()
        for _ in range(sample_steps):
            y = o(sample, t, ctx)
        dt = time.perf_counter() - t0
    return {"value": round(4 * sample_steps / dt, 4), "unit": UNIT, "cores": threads, "kind": "port",
            "sample": f"{sample_steps} forward(s) of BASELINE configs[0] (batch 4, 64x64 latent, fp32, hard gates "
                      f"multiplied as in the reference) on {threads} host threads, {dt:.1f} s"}, y


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    world = int(os.environ.get("WORLD_SIZE", "1"))
    cb, y = cpu_baseline(sample_steps=args.steps)
    dump_outputs(args, 1, rank, reference_sample=y)
    out = {"impl": "reference", "metric": METRIC, "value": cb["value"], "unit": UNIT, "n_gpus": world,
           "steps": args.steps, "warmup": 1, "ms_per_step": round(4e3 / cb["value"], 1),
           "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
           "config": {"workload": "configs[1] workload, bounded sample: batch-4 slices (configs[0] size) per step on "
                                  "the host CPU", "latent": LATENT, "codes": N_CODES},
           "cpu_baseline": cb,
           "e2e": {"value": cb["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(out), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-library-baseline", action="store_true", help="skip the eager-PyTorch-on-GPU library bar (N=1)")
    ap.add_argument("--no-secondary", action="store_true", help="skip the configs[2] / configs[3] numbers")
    ap.add_argument("--secondary-train-steps", type=int, default=6)
    ap.add_argument("--workload", default="forward", choices=["forward", "train", "sample", "finetune"])
    ap.add_argument("--train-batch", type=int, default=32)
    ap.add_argument("--prompts", type=int, default=16, help="--workload sample: prompts per GPU")
    ap.add_argument("--sample-latent", type=int, default=96)
    ap.add_argument("--ddim-steps", type=int, default=25)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step returned as float32 DIR/<name>.npy (DIR/<name>_rank<k>.npy "
                         "with several ranks): forward sample; train loss + gradients; sample latents + expert per "
                         "prompt; finetune loss + a fixed sample of the gradients; --impl reference sample. The seeded "
                         "inputs are the same in every run with the same arguments")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        run_reference(args)
        return
    if args.workload == "forward":
        run_ours(args)
    else:
        out = {"train": measure_train, "sample": measure_sample, "finetune": measure_finetune}[args.workload](args)
        if int(os.environ.get("RANK", "0")) == 0:
            print(json.dumps(out), flush=True)
    finish_dist()


if __name__ == "__main__":
    main()
