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

from typing import List, Optional, Tuple

import torch
import torch.distributed as dist

from . import kernels as K
from .pruning_step import alphas_cumprod


def ddim_timesteps(num_inference_steps: int, num_train_timesteps: int = 1000, steps_offset: int = 1) -> List[int]:
    """DDIMScheduler.set_timesteps with the SD-2.1 scheduler config ("leading" spacing, steps_offset 1)."""
    ratio = num_train_timesteps // num_inference_steps
    return [int(i * ratio) + steps_offset for i in range(num_inference_steps)][::-1]


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
            expert_index: Optional[torch.Tensor] = None) -> torch.Tensor:
    """The scheduler loop (pruning_pipelines.py:757-820) for one batch of prompts whose hard architecture
    vectors are `arch_vectors` (any mix of experts). latents [B,4,H,W] fp32 ~ N(0,1) (init_noise_sigma = 1).
    With `experts` (a PrunedExpertMixture) each prompt runs on its fine-tuned expert `expert_index` [B] instead: `unet`,
    `hyper_net` and `arch_vectors` are not used."""
    B = latents.shape[0]
    if B == 0:
        return latents
    acp = (alphas_cumprod() if acp is None else acp).cpu()
    ts = ddim_timesteps(num_inference_steps)
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
    x2 = torch.empty(2 * B, *x.shape[1:], device=x.device, dtype=torch.float32)
    nxt = torch.empty_like(x)
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
                    experts=None, code_to_expert: Optional[torch.Tensor] = None):
    """BASELINE configs[3]: route local prompts, dispatch them (all-to-all over NVLink) to the GPU chosen by
    plan_dispatch -- the rank(s) serving their expert, load-balanced --, denoise there, return the final latents to
    the rank that asked. Returns (latents, code index).
    With `experts` (a PrunedExpertMixture, held whole by every rank) each prompt is denoised by the fine-tuned expert of
    its routed code: `code_to_expert` [n_codes] maps a code index to a mixture position (default:
    experts.code_to_expert(quantizer.n_e), from the experts' code ids). Routing and dispatch are unchanged."""
    arch, idx = route_prompts(hyper_net, quantizer, prompt_embeddings)
    eidx = None
    if experts is not None:
        cmap = experts.code_to_expert(quantizer.n_e) if code_to_expert is None else torch.as_tensor(code_to_expert)
        eidx = cmap.to(idx.device, torch.int64)[idx]
        if bool((eidx < 0).any()):
            raise ValueError(f"prompts were routed to codes without a fine-tuned expert: "
                             f"{sorted(set(idx[eidx < 0].tolist()))}")
    world = dist.get_world_size() if dist.is_available() and dist.is_initialized() else 1
    if world == 1:
        kw = {} if experts is None else dict(experts=experts, expert_index=eidx)
        return denoise(unet, hyper_net, arch, latents, cond, uncond, num_inference_steps, guidance_scale, acp, **kw), idx
    owner = plan_dispatch(idx, quantizer.n_e, dispatch)
    order = torch.argsort(owner, stable=True)
    send = torch.bincount(owner, minlength=world)
    recv = torch.empty_like(send)
    dist.all_to_all_single(recv, send)
    sc, rc = send.tolist(), recv.tolist()
    payload = [arch[order], latents[order].float(), cond[order], uncond[order]]
    if eidx is not None:
        payload.append(eidx[order])
    arch_r, lat_r, cond_r, unc_r, *eidx_r = [_all_to_all_rows(p, sc, rc) for p in payload]
    kw = {} if experts is None else dict(experts=experts, expert_index=eidx_r[0])
    out_r = denoise(unet, hyper_net, arch_r, lat_r, cond_r, unc_r, num_inference_steps, guidance_scale, acp, **kw)
    back = _all_to_all_rows(out_r, rc, sc)
    out = torch.empty_like(back)
    out[order] = back
    return out, idx
