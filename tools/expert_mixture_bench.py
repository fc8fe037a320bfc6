"""Fine-tuned experts served as one batch (PrunedExpertMixture) vs the per-expert path.

Eight synthetic fine-tuned SD-2.1 experts: seeded random weights, a seeded perturbation of every parameter per expert,
the eight bench codes (bench.py / synthetic_codes). Two measurements on the same prompts and inputs:

  sampling  BASELINE configs[3] size (96x96 latents, CFG 7.5, 25 DDIM steps):
              (a) the mixture, every prompt in one batch;
              (b) one UNet2DConditionModelPruned per expert, one sampling loop per expert (the reference's serving
                  form: one job per expert);
            timed alternately in the same process, two repeats. Parity: one U-Net evaluation of the loop (the CFG-doubled
            batch at the first timestep) through (a) and through (b) must meet the U-Net contract (cosine >= 0.9999,
            max-abs <= 2e-2 of scale). After 25 guided steps the two trajectories are compared too, next to the spread
            of today's path against itself ((b) vs the same loop with one prompt per run), since guidance 7.5 amplifies
            bf16 rounding differences from step to step.
  forward   BASELINE configs[1] size (64 samples, 64x64): the mixture (8 weight sets) vs the gated U-Net with one weight
            set on the same codes and inputs: the cost of per-expert weights on the layers that used to share one.

Prints one JSON line per measurement with the GPU name and power limit read in the same run. Needs a GPU.

  python tools/expert_mixture_bench.py [--prompts 16] [--steps 2] [--forward-iters 10] [--out FILE]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from diffusion_pruning_b200 import PrunedExpertMixture, UNet2DConditionModelPruned  # noqa: E402
from diffusion_pruning_b200 import kernels as K  # noqa: E402
from diffusion_pruning_b200 import sampling as S  # noqa: E402
from diffusion_pruning_b200.synthetic import split_arch, synthetic_codes  # noqa: E402
from diffusion_pruning_b200.unet import UNet2DConditionModelGated  # noqa: E402

N_EXPERTS, N_CTX, CTX_DIM = 8, 77, 1024


def gpu_info() -> dict:
    info = {"gpu": torch.cuda.get_device_name(), "power_limit_w": "not measured"}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits",
                            "-i", str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30)
        info["power_limit_w"] = float(q.stdout.strip().splitlines()[0])
    except (OSError, ValueError, IndexError, subprocess.TimeoutExpired):
        pass
    return info


def build(device):
    """(base gated model, 8 fine-tuned experts, codes [8, dim])."""
    torch.manual_seed(1234)
    with torch.device(device):
        base = UNet2DConditionModelGated()   # SD-2.1 layout, seeded random init
    base.eval()
    st = base.get_structure()
    codes = synthetic_codes(st, N_EXPERTS, seed=2)
    experts = []
    for k in range(N_EXPERTS):
        with torch.device(device):
            m = UNet2DConditionModelPruned()
        m.load_state_dict(base.state_dict())
        with torch.no_grad():
            for i, p in enumerate(m.parameters()):
                g = torch.Generator(device=device).manual_seed(7919 * (k + 1) + i)
                p.add_(torch.randn(p.shape, generator=g, device=device) * (0.05 * float(p.abs().mean()) + 1e-4))
        m.prune_to(codes[k:k + 1].clone())
        experts.append(m.eval())
    return base, experts, codes


class _Split:
    """hyper_net stand-in for sampling.denoise: hands the codes to set_structure (HyperStructure.transform_structure_vector)."""

    def __init__(self, st):
        self.st = st

    def transform_structure_vector(self, arch):
        return split_arch(arch, self.st)


def timed(fn, n):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(n):
        out = fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) / n, out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--prompts", type=int, default=16)
    ap.add_argument("--latent", type=int, default=96)
    ap.add_argument("--ddim-steps", type=int, default=25)
    ap.add_argument("--steps", type=int, default=2, help="sampling passes per timed repeat")
    ap.add_argument("--forward-batch", type=int, default=64)
    ap.add_argument("--forward-latent", type=int, default=64)
    ap.add_argument("--forward-iters", type=int, default=10)
    ap.add_argument("--repeats", type=int, default=2)
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("expert_mixture_bench.py measures the B200 path: no CUDA device found")
    dev = torch.device("cuda")
    info = gpu_info()
    base, experts, codes = build(dev)
    mix = PrunedExpertMixture(experts)
    st = base.get_structure()
    lines = []

    def emit(d):
        d.update(info)
        s = json.dumps(d)
        print(s, flush=True)
        lines.append(s)

    # ---------------- sampling: (a) mixture in one batch, (b) one loop per expert ----------------
    P, H, T = args.prompts, args.latent, args.ddim_steps
    g = torch.Generator().manual_seed(300)
    lat = torch.randn(P, 4, H, H, generator=g).to(dev)
    cond = torch.randn(P, N_CTX, CTX_DIM, generator=g).to(dev)
    unc = torch.randn(1, N_CTX, CTX_DIM, generator=g).expand(P, -1, -1).contiguous().to(dev)
    eidx = (torch.arange(P) % N_EXPERTS)[torch.randperm(P, generator=g)].to(dev)
    acp = S.alphas_cumprod()
    split = _Split(st)
    groups = [(k, torch.nonzero(eidx == k).reshape(-1)) for k in range(N_EXPERTS)]
    groups = [(k, rows) for k, rows in groups if rows.numel()]

    def run_a():
        return S.denoise(None, None, None, lat, cond, unc, T, 7.5, acp, experts=mix, expert_index=eidx)

    def run_b(one_prompt_per_run=False):
        out = torch.empty_like(lat)
        for k, rows in groups:
            for r in (rows.split(1) if one_prompt_per_run else [rows]):
                out[r] = S.denoise(experts[k], split, codes[k:k + 1].expand(r.numel(), -1).to(dev), lat[r], cond[r],
                                   unc[r], T, 7.5, acp)
        return out

    def metrics(got, ref):
        got, ref = got.float().cpu().flatten(), ref.float().cpu().flatten()
        return ((got - ref).abs().max().item() / max(1.0, ref.abs().max().item()),
                torch.nn.functional.cosine_similarity(got, ref, dim=0).item())

    # one U-Net evaluation of the loop: the CFG-doubled batch at the first timestep, (a) vs (b)
    with torch.no_grad():
        x2, emb = torch.cat([lat, lat]), torch.cat([unc, cond])
        tt = torch.full((2 * P,), float(S.ddim_timesteps(T)[0]), device=dev)
        one_a = mix(x2, tt, emb, eidx).sample
        one_b = torch.empty_like(one_a)
        for k, rows in groups:
            r2 = torch.cat([rows, rows + P])
            experts[k].set_structure(split_arch(codes[k:k + 1].expand(r2.numel(), -1).to(dev), st))
            one_b[r2] = experts[k](x2[r2], tt[r2], emb[r2]).sample
    step_abs, step_cos = metrics(one_a, one_b)
    parity_ok = step_abs <= 2e-2 and step_cos >= 0.9999

    ya, yb = run_a(), run_b()          # warm-up: packs, schedules, CUDA graphs of both paths
    ya, yb = run_a(), run_b()
    K.check_abort()
    max_abs, cos = metrics(ya, yb)
    spread_abs, spread_cos = metrics(run_b(one_prompt_per_run=True), yb)
    times = {"a_mixture": [], "b_per_expert_loop": []}
    for _ in range(args.repeats):     # alternate (a) and (b)
        times["a_mixture"].append(timed(run_a, args.steps)[0])
        times["b_per_expert_loop"].append(timed(run_b, args.steps)[0])
    for name, ts in times.items():
        ms_step = [1e3 * t / T for t in ts]
        emit({"measure": "sampling", "path": name,
              "config": f"configs[3] size: {P} prompts on {len(groups)} experts, {H}x{H}, CFG 7.5, {T} DDIM steps",
              "ms_per_ddim_step": [round(v, 3) for v in ms_step],
              "samples_steps_per_s": [round(P * T / t, 1) for t in ts],
              "parity_one_unet_step_a_vs_b": {"max_abs_over_scale": round(step_abs, 6), "cosine": round(step_cos, 7),
                                              "ok": parity_ok},
              f"after_{T}_steps_a_vs_b": {"max_abs_over_scale": round(max_abs, 6), "cosine": round(cos, 7)},
              f"after_{T}_steps_b_vs_b_one_prompt_per_run": {"max_abs_over_scale": round(spread_abs, 6),
                                                            "cosine": round(spread_cos, 7)}})

    # ---------------- forward: mixture (8 weight sets) vs gated model (one weight set) ----------------
    B, L = args.forward_batch, args.forward_latent
    g = torch.Generator().manual_seed(3)
    assign = (torch.arange(B) % N_EXPERTS)[torch.randperm(B, generator=g)]
    base.set_structure(split_arch(codes[assign].to(dev), st))
    g = torch.Generator().manual_seed(11)
    x = torch.randn(B, 4, L, L, generator=g).to(dev)
    ctx = torch.randn(B, N_CTX, CTX_DIM, generator=g).to(dev)
    t = torch.randint(0, 1000, (B,), generator=g).float().to(dev)
    aidx = assign.to(dev)

    def fwd_mix():
        return mix(x, t, ctx, aidx).sample

    def fwd_gated():
        return base(x, t, ctx).sample

    with torch.no_grad():
        for _ in range(3):
            fwd_mix()
            fwd_gated()
        K.check_abort()
        ft = {"mixture_8_weight_sets": [], "gated_1_weight_set": []}
        for _ in range(args.repeats):
            ft["mixture_8_weight_sets"].append(timed(fwd_mix, args.forward_iters)[0])
            ft["gated_1_weight_set"].append(timed(fwd_gated, args.forward_iters)[0])
    for name, ts in ft.items():
        emit({"measure": "forward", "path": name, "config": f"configs[1] size: batch {B}, {L}x{L}, 8 codes",
              "ms_per_forward": [round(1e3 * v, 3) for v in ts],
              "samples_per_s": [round(B / v, 1) for v in ts]})
    mem = torch.cuda.max_memory_allocated() / 2 ** 30
    emit({"measure": "memory", "max_allocated_gib": round(mem, 2),
          "note": "8 experts' fp32 weights + their bf16 packs (mixture and per-expert engines) + the gated model"})
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "a") as f:
            f.write("\n".join(lines) + "\n")
    if not parity_ok:
        raise SystemExit(f"one U-Net step of (a) and (b) disagree: max-abs {step_abs:.3g} of scale, cosine {step_cos:.6f}")


if __name__ == "__main__":
    main()
