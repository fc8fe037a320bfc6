"""Schedulers of the sampling loop without a GPU: the float64 oracle against identities and closed-form solutions,
sampling.sampler_plan against the oracle, the noise order, argument validation, and the routing of per-prompt noise
over gloo."""
import os
import socket
import sys
import types

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import sampler_checks as SC
from diffusion_pruning_b200 import sampling as S
from oracle import sampler_oracle as SO2
from oracle import sampling_oracle as SO

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)


def _latents(B=3, H=5, seed=0):
    return torch.randn(B, 4, H, H, generator=torch.Generator().manual_seed(seed), dtype=torch.float64)


@pytest.mark.parametrize("steps", [5, 25, 50])
def test_dpm_order1_is_ddim_eta0(steps):
    model = SC.analytic_model(0.7, 1.6)   # uncond and cond differ: CFG at 7.5 is not the identity
    x = _latents()
    ddim = SO2.denoise(model, x, steps, 7.5, "ddim")
    dpm1 = SO2.denoise(model, x, steps, 7.5, "dpmsolver++", solver_order=1)
    assert SC.rel_err(dpm1, ddim) <= 1e-12


def test_oracle_ddim_matches_sampling_oracle():
    """oracle.sampling_oracle.denoise (fp32, the DDIM eta 0 loop every existing sampling test uses) against the float64
    restatement: same update up to fp32 rounding."""
    model = SC.analytic_model(0.7, 1.6)

    class AnalyticUNet:
        def set_structure(self, structure):
            pass

        def __call__(self, x2, t, emb):
            return model(x2.double(), int(t[0])).float()
    layout = types.SimpleNamespace(width_starts=[0], width_list=[], n_width=0, n_depth=0)
    x = _latents()
    emb = torch.zeros(3, 1, 1)
    ref = SO.denoise(AnalyticUNet(), layout, torch.zeros(3, 1), x.float(), emb, emb, steps=10, guidance=7.5)
    got = SO2.denoise(model, x, 10, 7.5, "ddim")
    assert SC.rel_err(got, ref.double()) <= 2e-6


@pytest.mark.parametrize("case", [
    dict(scheduler="ddim"), dict(scheduler="ddim", eta=0.5), dict(scheduler="ddim", eta=1.0, guidance_rescale=0.7),
    dict(scheduler="dpmsolver++", solver_order=1), dict(scheduler="dpmsolver++", solver_order=2),
    dict(scheduler="dpmsolver++", solver_order=2, guidance_rescale=1.0),
    dict(scheduler="dpmsolver++", solver_order=2, v_prediction=False)])
@pytest.mark.parametrize("steps", [4, 20])
def test_plan_reproduces_oracle(case, steps):
    """sampler_plan's coefficients applied as the kernel applies them (float64 numpy) = the oracle's updates; 20 steps
    exercises the second-order final step (lower_order_final applies below 15 steps)."""
    case = dict(case)
    vpred = case.pop("v_prediction", True)
    eta, g_r = case.get("eta", 0.0), case.pop("guidance_rescale", 0.0)
    model = SC.analytic_model(0.7, 1.6)
    x = _latents()
    noise = S.draw_step_noise(torch.Generator().manual_seed(3), steps, 3, x.shape[1:], "cpu") if eta > 0 else None
    plan = S.sampler_plan(case["scheduler"], steps, eta, case.get("solver_order", 2))
    got = SC.plan_loop(plan, model, x, 7.5, g_r, noise, vpred)
    ref = SO2.denoise(model, x, steps, 7.5, guidance_rescale=g_r, noise=noise, v_prediction=vpred, **case)
    assert SC.rel_err(got, ref) <= 1e-12


def test_convergence_on_gaussian_data():
    """Endpoint error of the probability-flow ODE for x0 ~ N(0, 2^2) with the exact denoiser. Measured (float64, max
    error over max |exact|):
      steps      16       20       32       64
      DDIM       6.08e-2  4.99e-2  3.15e-2  1.53e-2    (ratio per doubling 1.93, 2.05)
      DPM++(2M)  1.86e-2  1.30e-2  5.89e-3  1.77e-3    (ratio per doubling 3.16, 3.33)
    Second order shows as >= 3x per doubling rather than 4x: the grid's last step (t = 1 to alphas_cumprod[0]) has the
    same size at every step count."""
    s = 2.0
    model = SC.analytic_model(s, s)
    x = _latents(B=2, H=8)
    err = {}
    for sched in ("ddim", "dpmsolver++"):
        for n in (16, 20, 32, 64):
            exact = SC.ode_endpoint(x, S.ddim_timesteps(n)[0], s)
            err[sched, n] = SC.rel_err(SO2.denoise(model, x, n, 7.5, sched), exact)
    for a, b in ((16, 32), (32, 64)):
        assert err["dpmsolver++", a] / err["dpmsolver++", b] >= 3.0, err
        assert 1.8 <= err["ddim", a] / err["ddim", b] <= 2.2, err
    assert err["dpmsolver++", 20] * 3 <= err["ddim", 20], err


def test_rescale_matches_text_std():
    g = torch.Generator().manual_seed(1)
    m = torch.randn(3, 4, 6, 7, generator=g, dtype=torch.float64) * torch.tensor([0.5, 2.0, 7.0]).view(3, 1, 1, 1)
    m_text = torch.randn(3, 4, 6, 7, generator=g, dtype=torch.float64) * torch.tensor([1.0, 0.3, 4.0]).view(3, 1, 1, 1)
    r1 = SO2.rescale(m, m_text, 1.0)
    for b in range(3):
        assert abs(float(r1[b].std()) / float(m_text[b].std()) - 1) <= 1e-12
    assert torch.equal(SO2.rescale(m, m_text, 0.0), m)


def test_draw_step_noise_order():
    steps, B, shape = 3, 4, (4, 5, 5)
    gens = [torch.Generator().manual_seed(10 + b) for b in range(B)]
    got = S.draw_step_noise(gens, steps, B, shape, "cpu")
    ref_gens = [torch.Generator().manual_seed(10 + b) for b in range(B)]
    for i in range(steps):       # diffusers randn_tensor with a generator list, once per step
        ref = torch.cat([torch.randn((1, *shape), generator=ref_gens[b]) for b in range(B)])
        assert torch.equal(got[:, i], ref)
    got1 = S.draw_step_noise(torch.Generator().manual_seed(5), steps, B, shape, "cpu")
    g = torch.Generator().manual_seed(5)
    for i in range(steps):
        assert torch.equal(got1[:, i], torch.randn((B, *shape), generator=g))


@pytest.mark.parametrize("kw", [dict(scheduler="euler"), dict(eta=-0.1), dict(scheduler="dpmsolver++", eta=0.5),
                                dict(guidance_rescale=-0.01), dict(guidance_rescale=1.5), dict(solver_order=3),
                                dict(solver_order=0), dict(eta=1.0, generator=[torch.Generator()] * 2)])
def test_rejected_arguments(kw):
    lat = torch.zeros(3, 4, 4, 4)
    with pytest.raises(ValueError):
        S.denoise(None, None, None, lat, None, None, num_inference_steps=2, **kw)
    with pytest.raises(ValueError):
        S.routed_sampling(None, None, None, None, lat, None, None, num_inference_steps=2, **kw)


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _noise_worker(rank, world, port, out_path, P, steps):
    sys.path.insert(0, ROOT)
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from diffusion_pruning_b200 import sampling as S
    g = torch.Generator().manual_seed(80 + rank)
    latents = torch.randn(P, 4, 6, 6, generator=g)
    cond = torch.randn(P, 5, 16, generator=g)
    uncond = torch.randn(P, 5, 16, generator=g)
    idx = torch.randint(0, 8, (P,), generator=g)
    arch = torch.nn.functional.one_hot(idx, 8).float()
    seen = {}

    def fake_route(hyper_net, quantizer, prompt_embeddings):
        return arch, idx

    def fake_denoise(unet, hyper_net, arch_vectors, lat, c, u, num_inference_steps=25, guidance_scale=7.5, acp=None,
                     prediction_type="v_prediction", *, scheduler="ddim", eta=0.0, generator=None,
                     guidance_rescale=0.0, solver_order=2, step_noise=None):
        codes = arch_vectors.argmax(dim=1)
        assert bool((codes % world == rank).all()), (rank, codes)
        seen.update(scheduler=scheduler, eta=eta, generator=generator, guidance_rescale=guidance_rescale,
                    solver_order=solver_order)
        assert step_noise.shape == (lat.shape[0], num_inference_steps, 4, 6, 6), step_noise.shape
        w = torch.arange(1, num_inference_steps + 1, dtype=torch.float32).view(1, -1, 1, 1, 1)
        tag = c.mean(dim=(1, 2)) + 2.0 * u.mean(dim=(1, 2))
        return lat * 2.0 + (step_noise * w).sum(1) + tag[:, None, None, None] + 1000.0 * rank

    S.route_prompts, S.denoise = fake_route, fake_denoise
    gens = [torch.Generator().manual_seed(1000 * rank + b) for b in range(P)]
    out, _ = S.routed_sampling(None, None, types.SimpleNamespace(n_e=8), torch.zeros(P, 8), latents, cond, uncond,
                               num_inference_steps=steps, dispatch="expert_mod", eta=1.0, generator=gens,
                               guidance_rescale=0.3)
    noise = torch.stack([torch.stack([torch.randn(4, 6, 6, generator=gg) for _ in range(steps)])
                         for gg in [torch.Generator().manual_seed(1000 * rank + b) for b in range(P)]])
    w = torch.arange(1, steps + 1, dtype=torch.float32).view(1, -1, 1, 1, 1)
    tag = cond.mean(dim=(1, 2)) + 2.0 * uncond.mean(dim=(1, 2))
    want = latents * 2.0 + (noise * w).sum(1) + tag[:, None, None, None] + 1000.0 * (idx % world)[:, None, None, None]
    kw_ok = not seen or seen == dict(scheduler="ddim", eta=1.0, generator=None, guidance_rescale=0.3, solver_order=2)
    torch.save({"ok": bool(torch.allclose(out, want, rtol=0, atol=1e-4)), "kw_ok": kw_ok}, f"{out_path}.{rank}")
    dist.destroy_process_group()


@pytest.mark.timeout(300)
@pytest.mark.parametrize("world", [2, 3])
def test_routed_step_noise_travels_with_its_prompt(tmp_path, world):
    """routed_sampling with eta > 0 and one generator per prompt: the asking rank draws each prompt's noise, the rows
    arrive with the prompt on the rank serving its expert, the outputs return in the caller's order, and only the
    non-default options are forwarded (as step_noise, not the generators)."""
    out = str(tmp_path / "res")
    mp.spawn(_noise_worker, args=(world, _free_port(), out, 7, 3), nprocs=world, join=True)
    res = [torch.load(f"{out}.{r}") for r in range(world)]
    assert all(r["ok"] and r["kw_ok"] for r in res), res
