"""Cost of the sampling schedulers at the BASELINE configs[3] shape: full-width SD-2.1 (seeded random init), 8 synthetic
codes, 16 prompts spread round-robin over them, 96x96 latents, CFG 7.5, one GPU (sampling.denoise: the loop that
routed_sampling runs on each rank; routing and dispatch are left out).

  pass      ms per sampling pass for DDIM 25, DDIM 25 eta 1, DDIM 25 guidance_rescale 0.7 and DPM-Solver++(2M) at 15, 20
            and 25 steps: CUDA events around each pass, one warm-up pass per configuration, median of --passes.
  kernels   us per scheduler step of aptp_cfg_ddim_step, aptp_cfg_sampler_step (DDIM eta 1: + noise; DPM 2M: + x0
            history) and aptp_cfg_pred_stats at the same shape, in a separate pass: median of single launches timed with
            CUDA events after a 256 MB write that evicts L2 (cold, the inputs come from HBM), and the mean of back-to-back
            launches (hot, the 14 MB working set stays in the 126 MB L2). Achieved bytes/s = bytes the kernel must move
            (from the shapes) / time, against the 7.7 TB/s HBM3e data-sheet figure.

Prints one JSON line per measurement with the GPU name and power limit read in the same run. Needs a GPU.

  python tools/sampler_bench.py [--passes 3] [--out FILE]
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from diffusion_pruning_b200 import HyperStructure  # noqa: E402
from diffusion_pruning_b200 import kernels as K  # noqa: E402
from diffusion_pruning_b200 import sampling as S  # noqa: E402
from diffusion_pruning_b200.synthetic import synthetic_codes  # noqa: E402
from diffusion_pruning_b200.unet import UNet2DConditionModelGated  # noqa: E402

N_CODES, N_CTX, CTX_DIM, HBM_TBPS = 8, 77, 1024, 7.7
CONFIGS = [("ddim 25", 25, {}), ("ddim 25 eta 1", 25, dict(eta=1.0)),
           ("ddim 25 rescale 0.7", 25, dict(guidance_rescale=0.7)),
           ("dpmsolver++(2M) 15", 15, dict(scheduler="dpmsolver++")),
           ("dpmsolver++(2M) 20", 20, dict(scheduler="dpmsolver++")),
           ("dpmsolver++(2M) 25", 25, dict(scheduler="dpmsolver++"))]


def gpu_info() -> dict:
    info = {"gpu": torch.cuda.get_device_name(), "power_limit_w": "not measured"}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits",
                            "-i", str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30)
        info["power_limit_w"] = float(q.stdout.strip().splitlines()[0])
    except (OSError, ValueError, IndexError, subprocess.TimeoutExpired):
        pass
    return info


def measure_passes(args, info, emit):
    device = torch.device("cuda")
    torch.manual_seed(1234)
    with torch.device(device):
        unet = UNet2DConditionModelGated()
    unet.eval()
    st = unet.get_structure()
    hyper = HyperStructure(structure=st, input_dim=768, wn_flag=False, linear_bias=True).to(device).eval()
    P, H = args.prompts, args.latent
    arch = synthetic_codes(st, N_CODES).float()[torch.arange(P) % N_CODES].to(device)
    g = torch.Generator().manual_seed(300)
    lat = torch.randn(P, 4, H, H, generator=g).to(device)
    cond = torch.randn(P, N_CTX, CTX_DIM, generator=g).to(device)
    unc = torch.randn(1, N_CTX, CTX_DIM, generator=g).expand(P, -1, -1).contiguous().to(device)
    acp = S.alphas_cumprod()
    base = None
    for name, steps, kw in CONFIGS:
        def run():
            gen = torch.Generator().manual_seed(7) if kw.get("eta", 0) > 0 else None
            return S.denoise(unet, hyper, arch, lat, cond, unc, num_inference_steps=steps, guidance_scale=7.5, acp=acp,
                             generator=gen, **kw)
        out = run()
        torch.cuda.synchronize()
        times = []
        for _ in range(args.passes):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            out = run()
            e1.record()
            torch.cuda.synchronize()
            times.append(e0.elapsed_time(e1))
        K.check_abort()
        assert torch.isfinite(out).all(), name
        ms = statistics.median(times)
        base = ms if base is None else base
        emit({"measurement": "sampling pass", "config": name, "steps": steps, "ms_per_pass": round(ms, 2),
              "ms_per_step": round(ms / steps, 2), "pass_ms_all": [round(t, 2) for t in times],
              "vs_ddim25": round(ms / base, 3), "prompts": P, "latent": H, "guidance": 7.5, **info})
    del unet


def measure_kernels(args, info, emit):
    B, H = args.prompts, args.latent
    n = 4 * H * H
    g = torch.Generator(device="cuda").manual_seed(1)
    pred = torch.randn(2 * B, 4, H, H, device="cuda", generator=g)
    x = torch.randn(B, 4, H, H, device="cuda", generator=g)
    out = torch.empty_like(x)
    hist = torch.randn_like(x)
    noise = torch.randn(B, 25, 4, H, H, device="cuda", generator=g)
    partials = torch.empty(B, K.SAMPLER_STAT_CHUNKS, 4, device="cuda", dtype=torch.float64)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    ddim1 = S.sampler_plan("ddim", 25, 1.0)[10]
    dpm2 = S.sampler_plan("dpmsolver++", 25)[10]
    K.cfg_pred_stats(pred, n, B, 7.5, partials)
    e = 4 * B * n    # bytes of one fp32 latent block
    launches = {
        "aptp_cfg_ddim_step": (lambda: K.cfg_ddim_step(pred, x, out, B * n, 7.5, 0.5, 0.6), 4 * e),
        "aptp_cfg_sampler_step ddim eta 1": (
            lambda: K.cfg_sampler_step(pred, x, out, n, B, 7.5, 0.0, None, ddim1.coeffs, noise=noise[:, 10],
                                       noise_ld=noise.stride(0)), 5 * e),
        "aptp_cfg_sampler_step dpm 2M": (
            lambda: K.cfg_sampler_step(pred, x, out, n, B, 7.5, 0.0, None, dpm2.coeffs, hist, hist), 6 * e),
        "aptp_cfg_sampler_step dpm 2M rescale 0.7": (
            lambda: K.cfg_sampler_step(pred, x, out, n, B, 7.5, 0.7, partials, dpm2.coeffs, hist, hist), 6 * e),
        "aptp_cfg_pred_stats": (lambda: K.cfg_pred_stats(pred, n, B, 7.5, partials), 2 * e),
    }
    for name, (fn, nbytes) in launches.items():
        for _ in range(10):
            fn()
        cold = []
        for _ in range(args.kernel_iters):
            flush.fill_(1)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            cold.append(e0.elapsed_time(e1) * 1e3)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.kernel_iters):
            fn()
        e1.record()
        torch.cuda.synchronize()
        hot = e0.elapsed_time(e1) * 1e3 / args.kernel_iters
        us = statistics.median(cold)
        emit({"measurement": "scheduler kernel", "kernel": name, "batch": B, "n_per_sample": n, "bytes": nbytes,
              "us_cold_l2_flushed": round(us, 2), "tbps_cold": round(nbytes / us / 1e6, 3),
              "frac_of_7.7tbps_cold": round(nbytes / us / 1e6 / HBM_TBPS, 3), "us_hot_back_to_back": round(hot, 2),
              "tbps_hot": round(nbytes / hot / 1e6, 3), **info})
    K.check_abort()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--prompts", type=int, default=16)
    ap.add_argument("--latent", type=int, default=96)
    ap.add_argument("--passes", type=int, default=3)
    ap.add_argument("--kernel-iters", type=int, default=100)
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "sampler_bench needs a GPU"
    info = gpu_info()

    def emit(row):
        line = json.dumps(row)
        print(line, flush=True)
        if args.out:
            os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
            with open(args.out, "a") as f:
                f.write(line + "\n")

    with torch.no_grad():
        measure_kernels(args, info, emit)
        measure_passes(args, info, emit)


if __name__ == "__main__":
    main()
