"""Expert-routed DDIM sampling on the B200 hot path: a restatement of the denoising part of
`StableDiffusionPruningPipeline.__call__` (pdm/pipelines/pruning_pipelines.py:746-820) from the encoded prompts
on (CLIP / VAE are out of scope), plus the expert-per-GPU serving form of BASELINE configs[3]:

  route: hyper_net(prompt embedding) -> quantizer (eval: cosine argmax, hard_concrete)   :746-751
  unet.set_structure(codes of the batch)                                                  :757-759
  per step: latent_model_input = cat([x] * 2); unet(...); CFG combine; scheduler.step     :790-814
            -> one gated U-Net step on the doubled batch + ONE fused CFG+DDIM kernel

With N GPUs, expert e lives on GPU e % N: every rank routes its own prompts, an NCCL all-to-all moves
(latent, cond, uncond) to the owner, the whole loop runs there with no further communication, and a second
all-to-all returns the final latents (the reference instead launches one job per expert:
cluster_scripts/slurm/img_generation/sd2-1_cc3m.slurm:45-60).
"""
from __future__ import annotations

import math
from typing import List, NamedTuple, Optional, Tuple

import torch
import torch.distributed as dist

from . import kernels as K
from .pruning_step import alphas_cumprod


def ddim_timesteps(num_inference_steps: int, num_train_timesteps: int = 1000, steps_offset: int = 1) -> List[int]:
    """DDIMScheduler.set_timesteps with the SD-2.1 scheduler config ("leading" spacing, steps_offset 1)."""
    ratio = num_train_timesteps // num_inference_steps
    return [int(i * ratio) + steps_offset for i in range(num_inference_steps)][::-1]


SCHEDULERS = ("ddim", "dpmsolver++")


class SamplerStep(NamedTuple):
    """One step of a sampling loop: the model runs at timestep t; coeffs = (sa, sb, c_x, c_0, c_h, c_e, c_n) are the
    arguments of kernels.cfg_sampler_step; store_x0: the step keeps its x0 for the next (second-order) step."""
    t: int
    coeffs: Tuple[float, float, float, float, float, float, float]
    store_x0: bool


def sampler_plan(scheduler: str, steps: int, eta: float = 0.0, solver_order: int = 2,
                 acp: Optional[torch.Tensor] = None, start: int = 0) -> List[SamplerStep]:
    """Per-step coefficients of x_prev = c_x x + c_0 x0 + c_h x0_last + c_e eps + c_n z on the ddim_timesteps(steps) grid
    (the last step goes to acp[0]), computed once in float64. With abar = alphas_cumprod, a = sqrt(abar),
    s = sqrt(1 - abar), lambda = log(a / s), t the current and p the previous timestep:
      "ddim" (DDIMScheduler.step):  std = eta sqrt((1 - abar_p) / (1 - abar_t) (1 - abar_t / abar_p)),
                                    x_prev = a_p x0 + sqrt(1 - abar_p - std^2) eps + std z
      "dpmsolver++" (multistep, data prediction, midpoint form): h = lambda_p - lambda_t,
                                    x_prev = (s_p / s_t) x - a_p (e^-h - 1) D,
        D = x0 at order 1, D = (1 + 1/2r) x0 - (1/2r) x0_last with r = h_last / h at order 2. The first step is order
        1, and so is the last when steps < 15 (lower_order_final).
    x0 and eps are derived from the guided model output as in cfg_ddim_step (sa = a_t, sb = s_t).
    start > 0 (img2img, img2img_start) returns the steps of ddim_timesteps(steps)[start:] only: DDIM's coefficients are
    unchanged; for DPM-Solver++ the first executed step is order 1, h_last is the previous executed step's, and
    lower_order_final still keys on the full `steps`."""
    _check_sampler_args(scheduler, eta, 0.0, solver_order)
    if not 0 <= start < steps:
        raise ValueError(f"start must lie in [0, {steps}), got {start}")
    acp = (alphas_cumprod() if acp is None else acp).detach().double().cpu()
    ratio = 1000 // steps
    plan, h_last = [], None
    for i, t in enumerate(ddim_timesteps(steps)):
        if i < start:
            continue
        ab_t = float(acp[t])
        ab_p = float(acp[t - ratio]) if t - ratio >= 0 else float(acp[0])   # set_alpha_to_one = False
        sa, sb, ap, sp = math.sqrt(ab_t), math.sqrt(1.0 - ab_t), math.sqrt(ab_p), math.sqrt(1.0 - ab_p)
        if scheduler == "ddim":
            std = eta * math.sqrt((1.0 - ab_p) / (1.0 - ab_t) * (1.0 - ab_t / ab_p))
            plan.append(SamplerStep(t, (sa, sb, 0.0, ap, 0.0, math.sqrt(1.0 - ab_p - std * std), std), False))
            continue
        h = math.log(ap / sp) - math.log(sa / sb)
        phi = -ap * math.expm1(-h)
        second = solver_order == 2 and i > start and not (i == steps - 1 and steps < 15)
        if second:
            r = h_last / h
            c_0, c_h = phi * (1.0 + 0.5 / r), -phi * 0.5 / r
        else:
            c_0, c_h = phi, 0.0
        plan.append(SamplerStep(t, (sa, sb, sp / sb, c_0, c_h, 0.0, 0.0), solver_order == 2 and i < steps - 1))
        h_last = h
    return plan


def draw_step_noise(generator, steps: int, B: int, shape, device) -> torch.Tensor:
    """The noise every step of a stochastic scheduler draws, drawn up front: [B, steps, *shape] fp32 on `device`.
    Same order as diffusers' randn_tensor(model_output.shape, generator) once per step: step-major; with a list of
    generators prompt b's rows come from generator[b] (drawn on that generator's device), with one generator (or None:
    the global RNG, on `device`) each step is one batch draw. Every prompt thus sees the sequence the diffusers pipeline
    would give it. Memory: steps x B x 4 x prod(shape) bytes (59 MB at 16 prompts, 4x96x96 latents, 25 steps)."""
    shape = tuple(shape)
    out = torch.empty(B, steps, *shape, device=device, dtype=torch.float32)
    for i in range(steps):
        if isinstance(generator, (list, tuple)):
            for b, g in enumerate(generator):
                out[b, i] = torch.randn((1, *shape), generator=g, device=g.device)[0].to(device)
        else:
            dev = device if generator is None else generator.device
            out[:, i] = torch.randn((B, *shape), generator=generator, device=dev).to(device)
    return out


def img2img_start(steps: int, strength: float) -> int:
    """Index of the first executed step of an img2img / inpainting pass (diffusers get_timesteps): the loop runs
    ddim_timesteps(steps)[start:], the last min(int(steps * strength), steps) steps of the grid."""
    if not 0.0 < strength <= 1.0:
        raise ValueError(f"strength must lie in (0, 1], got {strength}")
    init = min(int(steps * strength), steps)
    if init < 1:
        raise ValueError(f"strength {strength} leaves no step of a {steps}-step grid (int(steps * strength) = {init})")
    return steps - init


def _check_sampler_args(scheduler, eta, guidance_rescale, solver_order, generator=None, B=None, *, steps=None,
                        latents=None, image_latents=None, strength=1.0, mask=None) -> None:
    if image_latents is None:
        if mask is not None:
            raise ValueError("mask needs image_latents (inpainting regenerates the masked region of an image)")
        if strength != 1.0:
            raise ValueError(f"strength needs image_latents (got strength={strength})")
    else:
        if steps is not None:
            img2img_start(steps, strength)
        if latents is not None and tuple(image_latents.shape) != tuple(latents.shape):
            raise ValueError(f"image_latents must have the shape of latents {list(latents.shape)}, "
                             f"got {list(image_latents.shape)}")
        if mask is not None and latents is not None and (
                mask.dim() != 4 or tuple(mask.shape) != (latents.shape[0], 1, *latents.shape[2:])):
            raise ValueError(f"mask must be [{latents.shape[0]}, 1, {', '.join(map(str, latents.shape[2:]))}], "
                             f"got {list(mask.shape)}")
    if scheduler not in SCHEDULERS:
        raise ValueError(f"scheduler must be one of {SCHEDULERS}, got {scheduler!r}")
    if eta < 0 or (eta > 0 and scheduler != "ddim"):
        raise ValueError(f"eta must be >= 0 and is a DDIM option (scheduler={scheduler!r}, eta={eta})")
    if not 0.0 <= guidance_rescale <= 1.0:
        raise ValueError(f"guidance_rescale must lie in [0, 1], got {guidance_rescale}")
    if solver_order not in (1, 2):
        raise ValueError(f"solver_order must be 1 or 2, got {solver_order}")
    if isinstance(generator, (list, tuple)) and len(generator) != B:
        raise ValueError(f"got {len(generator)} generators for {B} prompts")


@torch.no_grad()
def route_prompts(hyper_net, quantizer, prompt_embeddings: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
    """pruning_pipelines.py:746-751 in eval mode: returns (hard architecture vectors [B,1620], code index [B])."""
    assert not quantizer.training, "routing for sampling uses the eval path (cosine argmax + hard_concrete)"
    arch = hyper_net(prompt_embeddings)
    z_q, (_, _, idx) = quantizer(arch)
    return z_q, idx


@torch.no_grad()
def denoise(unet, hyper_net, arch_vectors: torch.Tensor, latents: torch.Tensor, cond: torch.Tensor,
            uncond: torch.Tensor, num_inference_steps: int = 25, guidance_scale: float = 7.5,
            acp: Optional[torch.Tensor] = None, prediction_type: str = "v_prediction", experts=None,
            expert_index: Optional[torch.Tensor] = None, *, scheduler: str = "ddim", eta: float = 0.0,
            generator=None, guidance_rescale: float = 0.0, solver_order: int = 2,
            step_noise: Optional[torch.Tensor] = None, image_latents: Optional[torch.Tensor] = None,
            strength: float = 1.0, mask: Optional[torch.Tensor] = None) -> torch.Tensor:
    """The scheduler loop (pruning_pipelines.py:757-820) for one batch of prompts whose hard architecture
    vectors are `arch_vectors` (any mix of experts). latents [B,4,H,W] fp32 ~ N(0,1) (init_noise_sigma = 1).
    With `experts` (a PrunedExpertMixture) each prompt runs on its fine-tuned expert `expert_index` [B] instead: `unet`,
    `hyper_net` and `arch_vectors` are not used.

    The pipeline's scheduler controls (sampler_plan has the definitions):
      scheduler: "ddim" or "dpmsolver++" (DPMSolverMultistepScheduler, data prediction; solver_order 1 or 2);
      eta: DDIM noise level (>= 0); the noise of every step comes from `generator` (None, one torch.Generator or a list
           of B, one per prompt) in draw_step_noise's order, or is given as step_noise [B, steps, 4, H, W] fp32
           (steps x B x 16 H W bytes: 59 MB at 16 prompts, 96x96 latents, 25 steps);
      guidance_rescale: diffusers rescale_noise_cfg factor in [0, 1].
    The defaults (DDIM, eta 0, no rescale) run the fused cfg_ddim_step loop; anything else runs cfg_sampler_step (and
    cfg_pred_stats when guidance_rescale > 0).

    Image-to-image and inpainting (StableDiffusionImg2ImgPipeline / StableDiffusionInpaintPipeline with a 4-channel
    U-Net; DESIGN section 4 has the definitions):
      image_latents [B,4,H,W]: the encoded image (the caller runs the VAE); `latents` is then the noise of diffusers'
           prepare_latents. The loop runs ddim_timesteps(steps)[img2img_start(steps, strength):] from
           x = sqrt(abar_t0) image + sqrt(1 - abar_t0) noise (one add_noise_velocity launch), t0 its first timestep;
      strength in (0, 1];
      mask [B,1,H,W] fp32 in [0, 1], 1 = regenerate: every step runs cfg_sampler_step_masked, which resets the known
           region to the image re-noised to the next timestep (to the image itself after the last step). At strength 1
           the masked pass starts from the noise.
    With eta > 0 the step noise covers the executed steps only ([B, executed steps, 4, H, W])."""
    B = latents.shape[0]
    _check_sampler_args(scheduler, eta, guidance_rescale, solver_order, generator, B, steps=num_inference_steps,
                        latents=latents, image_latents=image_latents, strength=strength, mask=mask)
    if B == 0:
        return latents
    acp = (alphas_cumprod() if acp is None else acp).cpu()
    start = 0 if image_latents is None else img2img_start(num_inference_steps, strength)
    ts = ddim_timesteps(num_inference_steps)[start:]
    ratio = 1000 // num_inference_steps
    if experts is None:
        unet.set_structure(hyper_net.transform_structure_vector(arch_vectors))   # gates tile over [uncond; cond]
        model = unet
    else:
        if expert_index is None or expert_index.shape != (B,):
            raise ValueError(f"experts= needs expert_index [{B}] (one expert per prompt)")
        model = lambda x, t, e: experts(x, t, e, expert_index)  # noqa: E731  (the index tiles over [uncond; cond])
    emb = torch.cat([uncond, cond], dim=0)                                   # :764-765
    x = latents.float().contiguous()
    blend = None
    if image_latents is not None:
        noise0, image = x, image_latents.to(x.device, torch.float32).contiguous()
        if mask is None or strength < 1.0:                                   # inpainting at strength 1 starts from noise
            x = _start_latents(image, noise0, ts[0], acp)
        if mask is not None:
            blend = (image, mask.to(x.device, torch.float32).contiguous(), noise0)
    x2 = torch.empty(2 * B, *x.shape[1:], device=x.device, dtype=torch.float32)
    nxt = torch.empty_like(x)
    if scheduler != "ddim" or eta != 0 or guidance_rescale != 0 or blend is not None:
        return _sampler_loop(model, emb, x, x2, nxt, num_inference_steps, guidance_scale, acp, prediction_type,
                             scheduler, eta, generator, guidance_rescale, solver_order, step_noise, start, blend)
    for t in ts:                                                             # :790
        x2[:B].copy_(x)                                                      # :792 cat([latents] * 2)
        x2[B:].copy_(x)
        tt = torch.full((2 * B,), float(t), device=x.device)
        pred = model(x2, tt, emb).sample                                     # :796-802
        prev = t - ratio
        a_t = float(acp[t])
        a_prev = float(acp[prev]) if prev >= 0 else float(acp[0])            # set_alpha_to_one = False
        K.cfg_ddim_step(pred.contiguous(), x, nxt, x.numel(), guidance_scale, a_t, a_prev,
                        prediction_type == "v_prediction")                   # :805-814 fused
        x, nxt = nxt, x
    return x


def _start_latents(image, noise, t0, acp):
    """sqrt(abar_t0) image + sqrt(1 - abar_t0) noise (DDIMScheduler.add_noise), in one add_noise_velocity launch."""
    from .losses import NoiseTables
    tables = NoiseTables(acp, image.device)
    out = torch.empty_like(image)
    t = torch.full((image.shape[0],), int(t0), device=image.device, dtype=torch.int64)
    K.add_noise_velocity(image, noise, t, tables.sqrt_acp, tables.sqrt_1m_acp, out, None, image.shape[0],
                         image[0].numel())
    return out


def _sampler_loop(model, emb, x, x2, nxt, steps, guidance_scale, acp, prediction_type, scheduler, eta, generator,
                  guidance_rescale, solver_order, step_noise, start=0, blend=None):
    B, n = x.shape[0], x[0].numel()
    x = x.clone()   # the ping-pong writes into x every other step; it may be the caller's latents
    plan = sampler_plan(scheduler, steps, eta, solver_order, acp, start)
    executed = len(plan)
    noise = None
    if eta > 0:
        if step_noise is None:
            step_noise = draw_step_noise(generator, executed, B, x.shape[1:], x.device)
        if tuple(step_noise.shape) != (B, executed, *x.shape[1:]):
            raise ValueError(f"step_noise must be [{B}, {executed}, {', '.join(map(str, x.shape[1:]))}], "
                             f"got {list(step_noise.shape)}")
        noise = step_noise.to(x.device, torch.float32).contiguous()
    if blend is not None:
        image, mask, noise0 = blend
        acp64 = acp.detach().double().cpu()
        plane = mask[0].numel()
    hist = torch.empty_like(x) if any(st.store_x0 for st in plan) else None
    partials = (torch.empty(B, K.SAMPLER_STAT_CHUNKS, 4, device=x.device, dtype=torch.float64)
                if guidance_rescale > 0 else None)
    vpred = prediction_type == "v_prediction"
    for i, st in enumerate(plan):
        x2[:B].copy_(x)
        x2[B:].copy_(x)
        tt = torch.full((2 * B,), float(st.t), device=x.device)
        pred = model(x2, tt, emb).sample.contiguous()
        if partials is not None:
            K.cfg_pred_stats(pred, n, B, guidance_scale, partials)
        step_args = (hist if st.coeffs[4] != 0 else None, hist if st.store_x0 else None,
                     None if noise is None else noise[:, i], 0 if noise is None else noise.stride(0), vpred)
        if blend is None:
            K.cfg_sampler_step(pred, x, nxt, n, B, guidance_scale, guidance_rescale, partials, st.coeffs, *step_args)
        else:
            # the known region at the next executed timestep; after the last step the image itself
            ab = float(acp64[plan[i + 1].t]) if i + 1 < executed else 1.0
            K.cfg_sampler_step_masked(pred, x, nxt, n, B, guidance_scale, guidance_rescale, partials, st.coeffs,
                                      image, mask, plane, noise0, math.sqrt(ab), math.sqrt(1.0 - ab), *step_args)
        x, nxt = nxt, x
    return x


def plan_dispatch(idx: torch.Tensor, n_experts: int, policy: str = "balanced") -> torch.Tensor:
    """Destination rank of every local prompt.

    "expert_mod": expert e lives on rank e % world (round 1). Eval routing is an unbalanced cosine argmax
    (pdm/models/vq/quantizer.py:264-271; SURVEY section 7 measured 47 ... 1212 of 4096 prompts per code), so this leaves
    most GPUs idle behind the one that owns the hot expert.
    "balanced" (default): the GLOBAL prompt list is sorted by expert and cut into `world` contiguous chunks of equal
    size. A hot expert spans several ranks (replicas), cold experts share one, every rank still sees few distinct
    experts (its compacted weight packs stay cached), and no rank gets more than ceil(total / world) prompts. Every
    rank holds the full dense U-Net, so any rank can serve any expert. Needs one all-gather of the per-expert counts."""
    world = dist.get_world_size() if dist.is_available() and dist.is_initialized() else 1
    if world == 1:
        return torch.zeros_like(idx)
    if policy == "expert_mod":
        return idx % world
    assert policy == "balanced", policy
    rank = dist.get_rank()
    counts = torch.bincount(idx, minlength=n_experts).to(torch.int64)
    all_counts = torch.empty(world, n_experts, dtype=torch.int64, device=idx.device)
    dist.all_gather_into_tensor(all_counts, counts.reshape(1, n_experts))
    tot_e = all_counts.sum(0)
    start_e = torch.cumsum(tot_e, 0) - tot_e                  # first global position of each expert's block
    before = all_counts[:rank].sum(0)                          # this expert's prompts held by lower ranks
    order = torch.argsort(idx, stable=True)
    first = torch.cumsum(counts, 0) - counts                   # first local sorted position of each expert
    within = torch.empty_like(idx)
    within[order] = torch.arange(idx.numel(), device=idx.device) - first[idx[order]]
    gpos = start_e[idx] + before[idx] + within
    total = int(tot_e.sum().item())
    chunk = max(1, (total + world - 1) // world)
    return torch.clamp(gpos // chunk, max=world - 1)


def _all_to_all_rows(t: torch.Tensor, send_counts: List[int], recv_counts: List[int]) -> torch.Tensor:
    out = torch.empty(sum(recv_counts), *t.shape[1:], device=t.device, dtype=t.dtype)
    dist.all_to_all_single(out, t.contiguous(), output_split_sizes=recv_counts, input_split_sizes=send_counts)
    return out


@torch.no_grad()
def routed_sampling(unet, hyper_net, quantizer, prompt_embeddings: torch.Tensor, latents: torch.Tensor,
                    cond: torch.Tensor, uncond: torch.Tensor, num_inference_steps: int = 25,
                    guidance_scale: float = 7.5, acp: Optional[torch.Tensor] = None, dispatch: str = "balanced",
                    experts=None, code_to_expert: Optional[torch.Tensor] = None, *, scheduler: str = "ddim",
                    eta: float = 0.0, generator=None, guidance_rescale: float = 0.0, solver_order: int = 2,
                    image_latents: Optional[torch.Tensor] = None, strength: float = 1.0,
                    mask: Optional[torch.Tensor] = None):
    """BASELINE configs[3]: route local prompts, dispatch them (all-to-all over NVLink) to the GPU chosen by
    plan_dispatch -- the rank(s) serving their expert, load-balanced --, denoise there, return the final latents to
    the rank that asked. Returns (latents, code index).
    With `experts` (a PrunedExpertMixture, held whole by every rank) each prompt is denoised by the fine-tuned expert of
    its routed code: `code_to_expert` [n_codes] maps a code index to a mixture position (default:
    experts.code_to_expert(quantizer.n_e), from the experts' code ids). Routing and dispatch are unchanged.
    scheduler / eta / generator / guidance_rescale / solver_order are denoise's. With eta > 0 the asking rank draws
    every step's noise of its prompts up front (draw_step_noise: one generator for the batch or one per prompt) and
    ships it with the prompts, so a prompt gets the same noise whichever rank serves it.
    image_latents / strength / mask are denoise's img2img and inpainting inputs; the image latents and masks travel with
    their prompts like the step noise, which then covers the executed steps only."""
    B = latents.shape[0]
    _check_sampler_args(scheduler, eta, guidance_rescale, solver_order, generator, B, steps=num_inference_steps,
                        latents=latents, image_latents=image_latents, strength=strength, mask=mask)
    sampler_kw = {k: v for k, v, default in (("scheduler", scheduler, "ddim"), ("eta", eta, 0.0),
                                             ("guidance_rescale", guidance_rescale, 0.0),
                                             ("solver_order", solver_order, 2), ("strength", strength, 1.0))
                  if v != default}
    step_noise = None
    if eta > 0:
        executed = num_inference_steps - (0 if image_latents is None else img2img_start(num_inference_steps, strength))
        step_noise = draw_step_noise(generator, executed, B, latents.shape[1:], latents.device)
    arch, idx = route_prompts(hyper_net, quantizer, prompt_embeddings)
    eidx = None
    if experts is not None:
        cmap = experts.code_to_expert(quantizer.n_e) if code_to_expert is None else torch.as_tensor(code_to_expert)
        eidx = cmap.to(idx.device, torch.int64)[idx]
        if bool((eidx < 0).any()):
            raise ValueError(f"prompts were routed to codes without a fine-tuned expert: "
                             f"{sorted(set(idx[eidx < 0].tolist()))}")
    world = dist.get_world_size() if dist.is_available() and dist.is_initialized() else 1
    per_prompt = (("expert_index", eidx), ("step_noise", step_noise), ("image_latents", image_latents), ("mask", mask))
    if world == 1:
        kw = {k: t for k, t in per_prompt if t is not None}
        if experts is not None:
            kw["experts"] = experts
        return denoise(unet, hyper_net, arch, latents, cond, uncond, num_inference_steps, guidance_scale, acp, **kw,
                       **sampler_kw), idx
    owner = plan_dispatch(idx, quantizer.n_e, dispatch)
    order = torch.argsort(owner, stable=True)
    send = torch.bincount(owner, minlength=world)
    recv = torch.empty_like(send)
    dist.all_to_all_single(recv, send)
    sc, rc = send.tolist(), recv.tolist()
    payload = [arch[order], latents[order].float(), cond[order], uncond[order]]
    extra = [(k, t) for k, t in per_prompt if t is not None]
    arch_r, lat_r, cond_r, unc_r, *extra_r = [_all_to_all_rows(p, sc, rc) for p in payload + [t[order] for _, t in extra]]
    kw = dict(zip([k for k, _ in extra], extra_r))
    if experts is not None:
        kw["experts"] = experts
    out_r = denoise(unet, hyper_net, arch_r, lat_r, cond_r, unc_r, num_inference_steps, guidance_scale, acp, **kw,
                    **sampler_kw)
    back = _all_to_all_rows(out_r, rc, sc)
    out = torch.empty_like(back)
    out[order] = back
    return out, idx
