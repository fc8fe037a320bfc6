"""Float64 oracle of the sampling loop's schedulers beyond DDIM eta 0 -- TEST INFRASTRUCTURE. Restates the updates from
their definitions (diffusers DDIMScheduler.step with eta, DPMSolverMultistepScheduler "dpmsolver++" / midpoint, and
rescale_noise_cfg) on the SD-2.1 grid of oracle.sampling_oracle (leading spacing, steps_offset 1, the last step to
alphas_cumprod[0]). Independent of diffusion_pruning_b200.sampling.sampler_plan."""
from __future__ import annotations

import torch

from .sampling_oracle import ddim_timesteps
from .step_oracle import alphas_cumprod


def rescale(m: torch.Tensor, m_text: torch.Tensor, g_r: float) -> torch.Tensor:
    """diffusers rescale_noise_cfg: per sample, unbiased std over every non-batch dimension."""
    dims = list(range(1, m.ndim))
    std_text = m_text.std(dim=dims, keepdim=True)
    std_cfg = m.std(dim=dims, keepdim=True)
    return g_r * (m * (std_text / std_cfg)) + (1 - g_r) * m


def x0_eps(m, x, abar_t, v_prediction=True):
    a, s = abar_t ** 0.5, (1 - abar_t) ** 0.5
    if v_prediction:
        return a * x - s * m, a * m + s * x
    return (x - s * m) / a, m


def ddim_update(x0, eps, abar_t, abar_p, eta=0.0, z=None):
    """DDIMScheduler.step: x_prev = sqrt(abar_p) x0 + sqrt(1 - abar_p - std^2) eps + std z."""
    std = eta * ((1 - abar_p) / (1 - abar_t) * (1 - abar_t / abar_p)) ** 0.5
    out = abar_p ** 0.5 * x0 + (1 - abar_p - std ** 2) ** 0.5 * eps
    return out + std * z if eta > 0 else out


def lam(abar):
    return 0.5 * (torch.log(abar) - torch.log(1 - abar))


def dpm_update(x, x0, x0_last, abar_t, abar_p, h_last=None):
    """DPM-Solver++ multistep (data prediction, midpoint): order 1 without x0_last, order 2 with it. Returns
    (x_prev, h)."""
    h = lam(abar_p) - lam(abar_t)
    a_p, s_p, s_t = abar_p ** 0.5, (1 - abar_p) ** 0.5, (1 - abar_t) ** 0.5
    d = x0
    if x0_last is not None:
        r = h_last / h
        d = (1 + 1 / (2 * r)) * x0 - (1 / (2 * r)) * x0_last
    return (s_p / s_t) * x - a_p * torch.expm1(-h) * d, h


@torch.no_grad()
def denoise(model, latents, steps=25, guidance=7.5, scheduler="ddim", eta=0.0, solver_order=2, guidance_rescale=0.0,
            noise=None, v_prediction=True, acp=None):
    """model(x2 [2B, ...] float64, t) -> prediction [2B, ...] of [uncond | cond]. noise [B, steps, ...] (eta > 0)."""
    acp = (alphas_cumprod() if acp is None else acp).double()
    x = latents.double().clone()
    B = x.shape[0]
    ratio = 1000 // steps
    x0_last = h_last = None
    for i, t in enumerate(ddim_timesteps(steps)):
        pred = model(torch.cat([x] * 2), t).double()
        pu, pc = pred[:B], pred[B:]
        m = pu + guidance * (pc - pu)
        if guidance_rescale > 0:
            m = rescale(m, pc, guidance_rescale)
        abar_t = acp[t]
        abar_p = acp[t - ratio] if t - ratio >= 0 else acp[0]
        x0, eps = x0_eps(m, x, abar_t, v_prediction)
        if scheduler == "ddim":
            x = ddim_update(x0, eps, abar_t, abar_p, eta, None if noise is None else noise[:, i].double())
            continue
        assert scheduler == "dpmsolver++", scheduler
        second = solver_order == 2 and i > 0 and not (i == steps - 1 and steps < 15)
        x, h_last = dpm_update(x, x0, x0_last if second else None, abar_t, abar_p, h_last)
        x0_last = x0
    return x
