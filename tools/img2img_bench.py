"""Cost of image-to-image and inpainting sampling at the BASELINE configs[3] shape: full-width SD-2.1 (seeded random init),
8 synthetic codes, 16 prompts spread round-robin over them, 96x96 latents, CFG 7.5, a 25-step grid, one GPU
(sampling.denoise: the loop that routed_sampling runs on each rank; routing and dispatch are left out).

  pass      ms per sampling pass for text-to-image DDIM 25 (reference), img2img at strength 1.0 / 0.6 / 0.3 and
            inpainting with a half-image mask at strength 1.0 / 0.6, each with DDIM and DPM-Solver++(2M): CUDA events
            around each pass, one warm-up pass per configuration, median of --passes. Executed steps =
            min(int(25 * strength), 25).
  kernels   us per step of aptp_cfg_sampler_step_masked next to aptp_cfg_sampler_step with the same coefficients (DDIM
            eta 0, DPM 2M with x0 history) at the same shape: median of single launches timed with CUDA events after a
            256 MB write that evicts L2 (inputs from HBM), and the mean of back-to-back launches (the working set stays
            in L2). Achieved bytes/s = bytes the kernel must move (from the shapes) / time.

Prints one JSON line per measurement with the GPU name and power limit read in the same run. Needs a GPU.

  python tools/img2img_bench.py [--passes 3] [--out FILE]
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

from diffusion_pruning_b200 import HyperStructure  # noqa: E402
from diffusion_pruning_b200 import kernels as K  # noqa: E402
from diffusion_pruning_b200 import sampling as S  # noqa: E402
from diffusion_pruning_b200.synthetic import synthetic_codes  # noqa: E402
from diffusion_pruning_b200.unet import UNet2DConditionModelGated  # noqa: E402
from sampler_bench import CTX_DIM, HBM_TBPS, N_CODES, N_CTX, gpu_info  # noqa: E402

STEPS = 25
CONFIGS = [("txt2img ddim", {}, None)]
for _sched, _kw in (("ddim", {}), ("dpmsolver++(2M)", dict(scheduler="dpmsolver++"))):
    CONFIGS += [(f"img2img {_sched} strength {s}", _kw, ("img2img", s)) for s in (1.0, 0.6, 0.3)]
    CONFIGS += [(f"inpaint half mask {_sched} strength {s}", _kw, ("inpaint", s)) for s in (1.0, 0.6)]


def half_mask(B, H, W, device):
    m = torch.zeros(B, 1, H, W, device=device)
    m[..., : W // 2] = 1.0
    return m


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
    image = torch.randn(P, 4, H, H, generator=g).to(device)
    mask = half_mask(P, H, H, device)
    acp = S.alphas_cumprod()
    base = None
    for name, kw, mode in CONFIGS:
        img_kw = {}
        if mode is not None:
            img_kw = dict(image_latents=image, strength=mode[1])
            if mode[0] == "inpaint":
                img_kw["mask"] = mask
        executed = STEPS - (S.img2img_start(STEPS, mode[1]) if mode else 0)

        def run():
            return S.denoise(unet, hyper, arch, lat, cond, unc, num_inference_steps=STEPS, guidance_scale=7.5,
                             acp=acp, **kw, **img_kw)
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
        emit({"measurement": "img2img pass", "config": name, "grid_steps": STEPS, "executed_steps": executed,
              "ms_per_pass": round(ms, 2), "ms_per_executed_step": round(ms / executed, 2),
              "pass_ms_all": [round(t, 2) for t in times], "vs_txt2img_ddim25": round(ms / base, 3), "prompts": P,
              "latent": H, "guidance": 7.5, **info})
    del unet


def measure_kernels(args, info, emit):
    B, H = args.prompts, args.latent
    n = 4 * H * H
    g = torch.Generator(device="cuda").manual_seed(1)
    pred = torch.randn(2 * B, 4, H, H, device="cuda", generator=g)
    x = torch.randn(B, 4, H, H, device="cuda", generator=g)
    out = torch.empty_like(x)
    hist = torch.randn_like(x)
    image = torch.randn_like(x)
    init = torch.randn_like(x)
    mask = half_mask(B, H, H, "cuda")
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    ddim = S.sampler_plan("ddim", STEPS)[10]
    dpm2 = S.sampler_plan("dpmsolver++", STEPS)[10]
    e = 4 * B * n    # bytes of one fp32 latent block
    blend_bytes = 2 * e + e // 4   # image, init noise, one mask plane per sample
    launches = {
        "aptp_cfg_sampler_step ddim eta 0": (
            lambda: K.cfg_sampler_step(pred, x, out, n, B, 7.5, 0.0, None, ddim.coeffs), 4 * e),
        "aptp_cfg_sampler_step_masked ddim eta 0": (
            lambda: K.cfg_sampler_step_masked(pred, x, out, n, B, 7.5, 0.0, None, ddim.coeffs, image, mask, H * H,
                                              init, 0.6, 0.8), 4 * e + blend_bytes),
        "aptp_cfg_sampler_step dpm 2M": (
            lambda: K.cfg_sampler_step(pred, x, out, n, B, 7.5, 0.0, None, dpm2.coeffs, hist, hist), 6 * e),
        "aptp_cfg_sampler_step_masked dpm 2M": (
            lambda: K.cfg_sampler_step_masked(pred, x, out, n, B, 7.5, 0.0, None, dpm2.coeffs, image, mask, H * H,
                                              init, 0.6, 0.8, hist, hist), 6 * e + blend_bytes),
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
    assert torch.cuda.is_available(), "img2img_bench needs a GPU"
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
