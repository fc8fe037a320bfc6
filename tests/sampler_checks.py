"""Shared pieces of the scheduler tests: a closed-form denoiser and a float64 numpy restatement of the sampler step.

Data x0 ~ N(0, s^2) per element; at abar = alphas_cumprod[t] (a = sqrt(abar), sigma = sqrt(1 - abar)) the exact
posterior mean is x0_hat = a s^2 x / (a^2 s^2 + sigma^2), i.e. v = (a x - x0_hat) / sigma, and the probability-flow ODE
carries x_T to x_T sqrt((a_e^2 s^2 + sigma_e^2) / (a_T^2 s^2 + sigma_T^2))."""
from __future__ import annotations

import numpy as np
import torch

from oracle.step_oracle import alphas_cumprod


def analytic_v(x, abar, s):
    a, sg = abar ** 0.5, (1 - abar) ** 0.5
    x0 = a * s * s * x / (a * a * s * s + sg * sg)
    return (a * x - x0) / sg


def analytic_model(s_uncond, s_cond, acp=None):
    """model(x2, t) for oracle.sampler_oracle.denoise: exact v of N(0, s_uncond^2) on the uncond half and of
    N(0, s_cond^2) on the cond half."""
    acp = (alphas_cumprod() if acp is None else acp).double()

    def model(x2, t):
        B = x2.shape[0] // 2
        ab = acp[int(t)].to(x2.dtype)
        return torch.cat([analytic_v(x2[:B], ab, s_uncond), analytic_v(x2[B:], ab, s_cond)])
    return model


def ode_endpoint(x_T, T, s, acp=None):
    acp = (alphas_cumprod() if acp is None else acp).double()
    a_e, a_T = acp[0], acp[T]
    return x_T * ((a_e * s * s + 1 - a_e) / (a_T * s * s + 1 - a_T)) ** 0.5


def plan_loop(plan, model, latents, guidance, guidance_rescale=0.0, noise=None, v_prediction=True):
    """sampling.sampler_plan applied as the kernel applies it, in float64 numpy."""
    x = latents.double().numpy()
    B = x.shape[0]
    hist = np.zeros_like(x)
    axes = tuple(range(1, x.ndim))
    for i, st in enumerate(plan):
        sa, sb, c_x, c_0, c_h, c_e, c_n = st.coeffs
        pred = model(torch.from_numpy(np.concatenate([x, x])), st.t).double().numpy()
        pu, pc = pred[:B], pred[B:]
        m = pu + guidance * (pc - pu)
        if guidance_rescale > 0:
            f = pc.std(axis=axes, ddof=1, keepdims=True) / m.std(axis=axes, ddof=1, keepdims=True)
            m = m * (guidance_rescale * f + 1 - guidance_rescale)
        if v_prediction:
            x0, eps = sa * x - sb * m, sa * m + sb * x
        else:
            x0, eps = (x - sb * m) / sa, m
        z = 0.0 if noise is None else noise[:, i].double().numpy()
        out = c_x * x + c_0 * x0 + c_h * hist + c_e * eps + c_n * z
        if st.store_x0:
            hist = x0
        x = out
    return torch.from_numpy(x)


def rel_err(a, b):
    return float((a - b).abs().max() / b.abs().max())
