"""Image-to-image and inpainting in the sampling loop without a GPU: sampler_plan on the strength-truncated grid against
the float64 oracle, convergence on the truncated grid, the oracle's mask edge cases, the noise order, argument
validation, and the routing of image latents and masks over gloo."""
import os
import socket
import sys
import types

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import img2img_oracle as IO
import sampler_checks as SC
from diffusion_pruning_b200 import sampling as S
from oracle import sampler_oracle as SO2

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)


def _pair(B=3, H=5, seed=0):
    """(noise, image latents) float64."""
    g = torch.Generator().manual_seed(seed)
    return (torch.randn(B, 4, H, H, generator=g, dtype=torch.float64),
            torch.randn(B, 4, H, H, generator=g, dtype=torch.float64) * 1.5)


def _half_mask(B, H, W):
    """Left half regenerated, right half kept; one sample with a fractional ramp."""
    m = torch.zeros(B, 1, H, W, dtype=torch.float64)
    m[..., : W // 2] = 1.0
    m[-1] = torch.linspace(0, 1, H * W, dtype=torch.float64).view(1, H, W)
    return m


def test_img2img_start_is_get_timesteps():
    """diffusers get_timesteps: init = min(int(steps * strength), steps), t_start = steps - init."""
    assert S.img2img_start(25, 1.0) == 0
    assert S.img2img_start(25, 0.6) == 10
    assert S.img2img_start(25, 0.3) == 18     # int(7.5) = 7 steps run
    assert S.img2img_start(4, 0.75) == 1
    assert S.img2img_start(4, 0.25) == 3
    assert S.ddim_timesteps(25)[S.img2img_start(25, 0.6):] == S.ddim_timesteps(25)[10:]


@pytest.mark.parametrize("case", [
    dict(scheduler="ddim"), dict(scheduler="ddim", eta=1.0), dict(scheduler="dpmsolver++", solver_order=1),
    dict(scheduler="dpmsolver++", solver_order=2), dict(scheduler="dpmsolver++", solver_order=2, v_prediction=False)])
@pytest.mark.parametrize("steps", [4, 20])
@pytest.mark.parametrize("strength", [0.75, 0.6, 0.3])
def test_plan_with_start_reproduces_oracle(case, steps, strength):
    """sampler_plan(start=k) applied as the kernel applies it, from the oracle's start latents, = the oracle's truncated
    loop. At 20 steps the truncated DPM grid ends with a second-order step; at 4 it ends with lower_order_final."""
    case = dict(case)
    vpred = case.pop("v_prediction", True)
    eta = case.get("eta", 0.0)
    model = SC.analytic_model(0.7, 1.6)
    noise, img = _pair()
    start = S.img2img_start(steps, strength)
    plan = S.sampler_plan(case["scheduler"], steps, eta, case.get("solver_order", 2), start=start)
    assert [st.t for st in plan] == S.ddim_timesteps(steps)[start:]
    step_noise = (S.draw_step_noise(torch.Generator().manual_seed(3), len(plan), 3, noise.shape[1:], "cpu")
                  if eta > 0 else None)
    x_t0 = IO.add_noise(img, noise, S.alphas_cumprod().double()[plan[0].t])
    got = SC.plan_loop(plan, model, x_t0, 7.5, 0.0, step_noise, vpred)
    ref = IO.denoise(model, noise, steps, 7.5, noise=step_noise, v_prediction=vpred, image_latents=img,
                     strength=strength, **case)
    assert SC.rel_err(got, ref) <= 1e-12


def test_dpm_first_executed_step_is_first_order():
    full = S.sampler_plan("dpmsolver++", 20)
    cut = S.sampler_plan("dpmsolver++", 20, start=8)
    assert cut[0].coeffs[4] == 0.0 and full[8].coeffs[4] != 0.0      # no x0 history on the first executed step
    assert cut[1].coeffs == full[9].coeffs                              # h_last of the previous executed step
    assert S.sampler_plan("ddim", 20, 1.0, start=8) == S.sampler_plan("ddim", 20, 1.0)[8:]
    last4 = S.sampler_plan("dpmsolver++", 4, start=1)
    assert last4[-1].coeffs[4] == 0.0    # lower_order_final keys on the full 4-step grid, not on 3 executed steps


def test_img2img_convergence_on_truncated_grid():
    """Endpoint error of the probability-flow ODE from x_t0 = add_noise(image, noise, t0) to acp[0], for x0 ~ N(0, 2^2)
    with the exact denoiser and no guidance (identical cond and uncond). t0 depends on the step count through the
    integer grid ratio, so every run is compared to its own ode_endpoint(x_t0, t0). Measured (float64, max error over
    max |exact|, ratio per doubling of 16 -> 32 -> 64 -> 128 steps):
      strength 0.5  DDIM       1.79  2.03  2.27     DPM-Solver++(2M)  3.18  3.32  3.61
      strength 0.8  DDIM       1.74  2.02  2.30     DPM-Solver++(2M)  3.17  3.30  3.60
    The truncated grid keeps the full grid's behaviour: first order for DDIM, >= 3x per doubling for the 2M solver
    (its first executed step is first order, as the full grid's is)."""
    s = 2.0
    model = SC.analytic_model(s, s)
    noise, _ = _pair(B=2, H=8)
    img = _pair(B=2, H=8, seed=1)[1] * (s / 1.5)
    acp = S.alphas_cumprod().double()
    for strength in (0.5, 0.8):
        err = {}
        for sched in ("ddim", "dpmsolver++"):
            for n in (16, 32, 64, 128):
                t0 = S.ddim_timesteps(n)[S.img2img_start(n, strength)]
                exact = SC.ode_endpoint(IO.add_noise(img, noise, acp[t0]), t0, s)
                got = IO.denoise(model, noise, n, 7.5, sched, image_latents=img, strength=strength)
                err[sched, n] = SC.rel_err(got, exact)
        for a, b in ((16, 32), (32, 64), (64, 128)):
            r_dpm, r_ddim = err["dpmsolver++", a] / err["dpmsolver++", b], err["ddim", a] / err["ddim", b]
            assert r_dpm >= 3.0, (strength, a, err)
            assert 1.6 <= r_ddim <= 2.4, (strength, a, err)
            assert r_dpm >= r_ddim + 0.9, (strength, a, err)
        assert err["dpmsolver++", 32] * 2 <= err["ddim", 32], err


@pytest.mark.parametrize("sched", [dict(scheduler="ddim"), dict(scheduler="ddim", eta=1.0),
                                   dict(scheduler="dpmsolver++")])
def test_oracle_mask_edge_cases(sched):
    """Mask 0 returns image_latents exactly; mask 1 returns the unmasked img2img run exactly, and at strength 1 the
    text-to-image run from the same noise (the masked pass starts from the noise)."""
    model = SC.analytic_model(0.7, 1.6)
    noise, img = _pair()
    steps = 10
    zeros, ones = torch.zeros(3, 1, 5, 5, dtype=torch.float64), torch.ones(3, 1, 5, 5, dtype=torch.float64)
    for strength in (0.6, 1.0):
        executed = steps - S.img2img_start(steps, strength)
        kw = dict(sched)
        if kw.get("eta", 0) > 0:
            kw["noise"] = S.draw_step_noise(torch.Generator().manual_seed(9), executed, 3, noise.shape[1:], "cpu")
        kept = IO.denoise(model, noise, steps, 7.5, image_latents=img, strength=strength, mask=zeros, **kw)
        assert torch.equal(kept, img)
        whole = IO.denoise(model, noise, steps, 7.5, image_latents=img, strength=strength, mask=ones, **kw)
        plain = (IO.denoise(model, noise, steps, 7.5, image_latents=img, strength=strength, **kw) if strength < 1
                else SO2.denoise(model, noise, steps, 7.5, **kw))
        assert torch.equal(whole, plain), (strength, SC.rel_err(whole, plain))
    half = IO.denoise(model, noise, steps, 7.5, image_latents=img, strength=1.0, mask=_half_mask(3, 5, 5), **kw)
    assert torch.equal(half[:2, ..., 2:], img[:2, ..., 2:])     # the kept half ends on the image


class _Recorder:
    def __init__(self):
        self.kw = None

    def route(self, hyper_net, quantizer, prompt_embeddings):
        B = prompt_embeddings.shape[0]
        return torch.zeros(B, 8), torch.zeros(B, dtype=torch.int64)

    def denoise(self, *a, **kw):
        self.kw = kw
        return a[3]


@pytest.mark.parametrize("per_prompt", [False, True])
def test_noise_order_start_noise_then_executed_steps(monkeypatch, per_prompt):
    """The caller draws the start noise (`latents`) first; routed_sampling then draws one step-noise batch per executed
    step from the same generator(s), in draw_step_noise order."""
    B, steps, strength, shape = 3, 10, 0.6, (4, 6, 6)
    executed = steps - S.img2img_start(steps, strength)
    rec = _Recorder()
    monkeypatch.setattr(S, "route_prompts", rec.route)
    monkeypatch.setattr(S, "denoise", rec.denoise)

    def gens():
        return ([torch.Generator().manual_seed(20 + b) for b in range(B)] if per_prompt
                else torch.Generator().manual_seed(20))
    g = gens()
    if per_prompt:
        latents = torch.cat([torch.randn((1, *shape), generator=gb) for gb in g])
    else:
        latents = torch.randn((B, *shape), generator=g)
    img = torch.randn(B, *shape)
    S.routed_sampling(None, None, types.SimpleNamespace(n_e=8), torch.zeros(B, 8), latents, None, None,
                      num_inference_steps=steps, eta=1.0, generator=g, image_latents=img, strength=strength)
    got = rec.kw["step_noise"]
    assert got.shape == (B, executed, *shape)
    ref_g = gens()
    if per_prompt:
        for b in range(B):
            assert torch.equal(torch.randn((1, *shape), generator=ref_g[b])[0], latents[b])
            for i in range(executed):
                assert torch.equal(got[b, i], torch.randn((1, *shape), generator=ref_g[b])[0])
    else:
        assert torch.equal(torch.randn((B, *shape), generator=ref_g), latents)
        for i in range(executed):
            assert torch.equal(got[:, i], torch.randn((B, *shape), generator=ref_g))
    assert rec.kw["strength"] == strength and rec.kw["image_latents"] is img and "mask" not in rec.kw


_LAT = torch.zeros(3, 4, 4, 4)


@pytest.mark.parametrize("kw", [
    dict(image_latents=_LAT, strength=0.0), dict(image_latents=_LAT, strength=1.5),
    dict(image_latents=_LAT, strength=-0.5), dict(image_latents=_LAT, strength=0.2),   # int(4 * 0.2) = 0 steps
    dict(mask=torch.ones(3, 1, 4, 4)), dict(strength=0.5),
    dict(image_latents=torch.zeros(3, 4, 4, 5)), dict(image_latents=torch.zeros(2, 4, 4, 4)),
    dict(image_latents=_LAT, mask=torch.ones(3, 4, 4, 4)), dict(image_latents=_LAT, mask=torch.ones(3, 1, 4, 5)),
    dict(image_latents=_LAT, mask=torch.ones(3, 4, 4))])
def test_rejected_img2img_arguments(kw):
    with pytest.raises(ValueError):
        S.denoise(None, None, None, _LAT, None, None, num_inference_steps=4, **kw)
    with pytest.raises(ValueError):
        S.routed_sampling(None, None, None, None, _LAT, None, None, num_inference_steps=4, **kw)


def test_plan_start_out_of_range():
    for start in (-1, 4, 5):
        with pytest.raises(ValueError):
            S.sampler_plan("ddim", 4, start=start)


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _image_worker(rank, world, port, out_path, P, steps):
    sys.path.insert(0, ROOT)
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from diffusion_pruning_b200 import sampling as S
    g = torch.Generator().manual_seed(80 + rank)
    latents = torch.randn(P, 4, 6, 6, generator=g)
    image = torch.randn(P, 4, 6, 6, generator=g)
    mask = torch.rand(P, 1, 6, 6, generator=g)
    cond = torch.randn(P, 5, 16, generator=g)
    uncond = torch.randn(P, 5, 16, generator=g)
    idx = torch.randint(0, 8, (P,), generator=g)
    arch = torch.nn.functional.one_hot(idx, 8).float()
    seen = {}

    def fake_route(hyper_net, quantizer, prompt_embeddings):
        return arch, idx

    def fake_denoise(unet, hyper_net, arch_vectors, lat, c, u, num_inference_steps=25, guidance_scale=7.5, acp=None,
                     prediction_type="v_prediction", *, scheduler="ddim", eta=0.0, generator=None,
                     guidance_rescale=0.0, solver_order=2, step_noise=None, image_latents=None, strength=1.0,
                     mask=None):
        codes = arch_vectors.argmax(dim=1)
        assert bool((codes % world == rank).all()), (rank, codes)
        seen.update(scheduler=scheduler, eta=eta, strength=strength, step_noise=step_noise is not None)
        assert image_latents.shape == lat.shape and mask.shape == (lat.shape[0], 1, 6, 6)
        tag = c.mean(dim=(1, 2)) + 2.0 * u.mean(dim=(1, 2))
        return lat * 2.0 + image_latents * 3.0 + mask * 5.0 + tag[:, None, None, None] + 1000.0 * rank

    S.route_prompts, S.denoise = fake_route, fake_denoise
    out, _ = S.routed_sampling(None, None, types.SimpleNamespace(n_e=8), torch.zeros(P, 8), latents, cond, uncond,
                               num_inference_steps=steps, dispatch="expert_mod", scheduler="dpmsolver++",
                               image_latents=image, strength=0.6, mask=mask)
    tag = cond.mean(dim=(1, 2)) + 2.0 * uncond.mean(dim=(1, 2))
    want = (latents * 2.0 + image * 3.0 + mask * 5.0 + tag[:, None, None, None]
            + 1000.0 * (idx % world)[:, None, None, None])
    kw_ok = not seen or seen == dict(scheduler="dpmsolver++", eta=0.0, strength=0.6, step_noise=False)
    torch.save({"ok": bool(torch.allclose(out, want, rtol=0, atol=1e-4)), "kw_ok": kw_ok}, f"{out_path}.{rank}")
    dist.destroy_process_group()


@pytest.mark.timeout(300)
@pytest.mark.parametrize("world", [2, 3])
def test_routed_image_latents_and_masks_travel_with_their_prompt(tmp_path, world):
    """routed_sampling with image_latents and mask: each prompt's image and mask arrive with it on the rank serving its
    expert, the outputs return in the caller's order, and strength is forwarded only because it is not the default."""
    out = str(tmp_path / "res")
    mp.spawn(_image_worker, args=(world, _free_port(), out, 7, 5), nprocs=world, join=True)
    res = [torch.load(f"{out}.{r}") for r in range(world)]
    assert all(r["ok"] and r["kw_ok"] for r in res), res
