"""Float64 restatement of image-to-image and inpainting sampling -- TEST INFRASTRUCTURE. diffusers
StableDiffusionImg2ImgPipeline and StableDiffusionInpaintPipeline (4-channel U-Net) on the grid of oracle.sampling_oracle,
written from their definitions: get_timesteps, prepare_latents / add_noise, and the inpainting blend after every
scheduler.step. The per-step updates are oracle.sampler_oracle's. Independent of diffusion_pruning_b200.sampling."""
from __future__ import annotations

import torch

from oracle.sampler_oracle import ddim_update, dpm_update, rescale, x0_eps
from oracle.sampling_oracle import ddim_timesteps
from oracle.step_oracle import alphas_cumprod


def add_noise(image, noise, abar):
    """DDIMScheduler.add_noise at one timestep."""
    return abar ** 0.5 * image + (1 - abar) ** 0.5 * noise


@torch.no_grad()
def denoise(model, latents, steps=25, guidance=7.5, scheduler="ddim", eta=0.0, solver_order=2, guidance_rescale=0.0,
            noise=None, v_prediction=True, acp=None, image_latents=None, strength=1.0, mask=None):
    """model(x2 [2B, ...] float64, t) -> prediction [2B, ...] of [uncond | cond]. noise [B, executed steps, ...]
    (eta > 0). Without image_latents this is oracle.sampler_oracle.denoise.

    With image_latents, `latents` is the noise of prepare_latents; get_timesteps keeps the last
    min(int(steps * strength), steps) timesteps; the loop starts from add_noise(image, latents, first kept timestep), or
    from latents for an inpainting run at strength 1. With mask [B, 1, ...] (1 = regenerate), after every step
      x = (1 - mask) * add_noise(image, latents, next kept timestep) + mask * x,
    with the image itself after the last step. DPM-Solver++ keeps the unblended x0 as its history, its first kept step is
    first order, and lower_order_final looks at the full grid's length."""
    acp = (alphas_cumprod() if acp is None else acp).double()
    B = latents.shape[0]
    ratio = 1000 // steps
    timesteps = ddim_timesteps(steps)
    if image_latents is None:
        x = latents.double().clone()
    else:
        keep = min(int(steps * strength), steps)
        timesteps = timesteps[steps - keep:]
        img, nz = image_latents.double(), latents.double()
        x = nz.clone() if mask is not None and strength == 1 else add_noise(img, nz, acp[timesteps[0]])
    x0_last = h_last = None
    for i, t in enumerate(timesteps):
        pred = model(torch.cat([x] * 2), t).double()
        pu, pc = pred[:B], pred[B:]
        m = pu + guidance * (pc - pu)
        if guidance_rescale > 0:
            m = rescale(m, pc, guidance_rescale)
        abar_t = acp[t]
        abar_p = acp[t - ratio] if t - ratio >= 0 else acp[0]
        x0, eps = x0_eps(m, x, abar_t, v_prediction)
        last = i == len(timesteps) - 1
        if scheduler == "ddim":
            x = ddim_update(x0, eps, abar_t, abar_p, eta, None if noise is None else noise[:, i].double())
        else:
            assert scheduler == "dpmsolver++", scheduler
            second = solver_order == 2 and i > 0 and not (last and steps < 15)
            x, h_last = dpm_update(x, x0, x0_last if second else None, abar_t, abar_p, h_last)
            x0_last = x0
        if mask is not None:
            proper = img if last else add_noise(img, nz, acp[timesteps[i + 1]])
            x = (1 - mask.double()) * proper + mask.double() * x
    return x
