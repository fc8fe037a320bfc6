"""Image-to-image and inpainting in the sampling loop on the B200: aptp_cfg_sampler_step_masked against float64 and at its
bit-exact edges, the launches of the default and img2img paths, the GPU loop against the float64 oracle with a
closed-form model, the tiny U-Net and expert-mixture loops, and routed inpainting over two ranks."""
import os

import pytest
import torch

import img2img_oracle as IO
import sampler_checks as SC
from diffusion_pruning_b200 import kernels as K
from diffusion_pruning_b200 import sampling as S
from oracle import sampler_oracle as SO2
from test_samplers_gpu import KERNEL_CASES, LOOP_COS, LOOP_MAX_ABS, _analytic_experts, _tiny_problem, loop_bound

pytestmark = pytest.mark.gpu


def _mask(B, H, W, g, fractional=True):
    """Left half regenerated (1), right half kept (0); with `fractional`, uniform values in [0, 1] in a middle band."""
    m = torch.zeros(B, 1, H, W)
    m[..., : W // 2] = 1.0
    if fractional:
        band = slice(H // 3, 2 * H // 3)
        m[:, :, band] = torch.rand(B, 1, m[:, :, band].shape[2], W, generator=g)
    return m


def _step_inputs(case, B, H, W, seed):
    scheduler, order, eta, step, inplace = KERNEL_CASES[case]
    st = S.sampler_plan(scheduler, 25, eta, order)[step]
    g = torch.Generator().manual_seed(seed)
    pred = torch.randn(2 * B, 4, H, W, generator=g)
    pred[B:] = pred[B:] * 1.3 + 0.2
    d = dict(pred=pred, x=torch.randn(B, 4, H, W, generator=g), hist=torch.randn(B, 4, H, W, generator=g),
             noise=torch.randn(B, 5, 4, H, W, generator=g), image=torch.randn(B, 4, H, W, generator=g) * 1.5,
             init=torch.randn(B, 4, H, W, generator=g), mask=_mask(B, H, W, g))
    return st, inplace, d


def _launch(masked, st, inplace, d, vpred, rescale, guidance=7.5, a_next=0.6, s_next=0.8):
    """One step kernel on the cuda copies of d; returns (x_out, x0 history out or None)."""
    B, n = d["x"].shape[0], d["x"][0].numel()
    out = torch.full_like(d["x"], float("nan"))
    hist_in = d["hist"].clone()
    hist_out = hist_in if inplace else torch.full_like(d["x"], float("nan"))
    partials = None
    if rescale > 0:
        partials = torch.empty(B, K.SAMPLER_STAT_CHUNKS, 4, device="cuda", dtype=torch.float64)
        K.cfg_pred_stats(d["pred"], n, B, guidance, partials)
    uses_h, uses_z = st.coeffs[4] != 0, st.coeffs[6] != 0
    tail = dict(x0_hist_in=hist_in if uses_h else None, x0_hist_out=hist_out if st.store_x0 or inplace else None,
                noise=d["noise"][:, 2] if uses_z else None, noise_ld=d["noise"].stride(0), v_prediction=vpred)
    if masked:
        K.cfg_sampler_step_masked(d["pred"], d["x"], out, n, B, guidance, rescale, partials, st.coeffs, d["image"],
                                  d["mask"], d["mask"][0].numel(), d["init"], a_next, s_next, **tail)
    else:
        K.cfg_sampler_step(d["pred"], d["x"], out, n, B, guidance, rescale, partials, st.coeffs, **tail)
    torch.cuda.synchronize()
    return out, (hist_out if st.store_x0 or inplace else None)


def _masked_vs_float64(case, vpred, rescale, B, H, W, seed=0):
    st, inplace, d = _step_inputs(case, B, H, W, seed)
    a_next, s_next = 0.6, 0.8
    out, hist_out = _launch(True, st, inplace, {k: v.cuda() for k, v in d.items()}, vpred, rescale, a_next=a_next,
                            s_next=s_next)
    p = d["pred"].double()
    m = p[:B] + 7.5 * (p[B:] - p[:B])
    if rescale > 0:
        m = SO2.rescale(m, p[B:], rescale)
    sa, sb, c_x, c_0, c_h, c_e, c_n = st.coeffs
    xd = d["x"].double()
    x0, eps = SO2.x0_eps(m, xd, sa * sa, vpred)
    x_step = c_x * xd + c_0 * x0 + c_h * d["hist"].double() + c_e * eps + c_n * d["noise"][:, 2].double()
    mk = d["mask"].double()
    ref = (1 - mk) * (a_next * d["image"].double() + s_next * d["init"].double()) + mk * x_step
    err = SC.rel_err(out.cpu().double(), ref)
    assert err <= 1e-5, (case, vpred, rescale, err)
    if hist_out is not None:
        assert SC.rel_err(hist_out.cpu().double(), x0) <= 1e-5, (case, "x0 history is the unblended x0")


@pytest.mark.parametrize("case", list(KERNEL_CASES))
@pytest.mark.parametrize("vpred", [True, False])
@pytest.mark.parametrize("rescale", [0.0, 0.7])
def test_masked_step_kernel_vs_float64(case, vpred, rescale):
    """Odd batch, H x W = 17 x 23: the plane size is not a multiple of 4, so float4s straddle channel planes and the
    mask is indexed per element; fractional mask values."""
    _masked_vs_float64(case, vpred, rescale, B=3, H=17, W=23)


def test_masked_step_kernel_at_sampling_shape():
    """16 x 4 x 96^2 (the plane is a multiple of 4: one float4 of mask per float4 of x)."""
    for case in ("ddim eta 1", "dpm order 2 in-place history"):
        _masked_vs_float64(case, True, 0.7, B=16, H=96, W=96, seed=1)


@pytest.mark.parametrize("HW", [(17, 23), (16, 20)])
@pytest.mark.parametrize("case", ["ddim eta 1", "dpm order 2", "dpm order 2 in-place history"])
def test_masked_step_kernel_edges_are_bit_exact(case, HW):
    """Mask 0 with a_next = 1, s_next = 0 (the last step) gives image_latents exactly; mask 1 gives exactly the output
    and x0 history of aptp_cfg_sampler_step with the same coefficients."""
    H, W = HW
    st, inplace, d = _step_inputs(case, 3, H, W, seed=4)
    d = {k: v.cuda() for k, v in d.items()}
    for rescale in (0.0, 0.7):
        d["mask"].zero_()
        kept, _ = _launch(True, st, inplace, d, True, rescale, a_next=1.0, s_next=0.0)
        assert torch.equal(kept, d["image"]), (case, HW, rescale)
        d["mask"].fill_(1.0)
        got, got_h = _launch(True, st, inplace, d, True, rescale)
        want, want_h = _launch(False, st, inplace, d, True, rescale)
        assert torch.equal(got, want), (case, HW, rescale)
        if want_h is not None:
            assert torch.equal(got_h, want_h), (case, HW, rescale)


def _count_launches(monkeypatch, names):
    calls = dict.fromkeys(names, 0)
    for name in names:
        orig = getattr(K, name)

        def counted(*a, _orig=orig, _name=name, **kw):
            calls[_name] += 1
            return _orig(*a, **kw)
        monkeypatch.setattr(K, name, counted)
    return calls


def test_launches_of_default_img2img_and_inpainting(monkeypatch):
    """Without the new arguments only cfg_ddim_step runs; unmasked DDIM img2img adds one add_noise_velocity and runs
    cfg_ddim_step per executed step; a masked run uses cfg_sampler_step_masked on every executed step, also for DDIM
    with eta 0, and starts from the noise at strength 1."""
    gpu, _, lat = _tiny_problem()
    g = torch.Generator().manual_seed(12)
    img = torch.randn(lat.shape, generator=g).cuda()
    mask = _mask(lat.shape[0], lat.shape[2], lat.shape[3], g).cuda()
    names = ("cfg_ddim_step", "cfg_sampler_step", "cfg_sampler_step_masked", "cfg_pred_stats", "add_noise_velocity")
    calls = _count_launches(monkeypatch, names)

    def expect(**want):
        assert calls == {k: want.get(k, 0) for k in names}, calls
        calls.update(dict.fromkeys(names, 0))
    default = gpu(steps=4)
    expect(cfg_ddim_step=4)
    assert torch.equal(default, gpu(steps=4, strength=1.0, mask=None, image_latents=None))
    expect(cfg_ddim_step=4)
    gpu(steps=4, image_latents=img, strength=0.75)
    expect(add_noise_velocity=1, cfg_ddim_step=3)
    gpu(steps=4, image_latents=img, strength=0.75, mask=mask)
    expect(add_noise_velocity=1, cfg_sampler_step_masked=3)
    gpu(steps=4, image_latents=img, mask=mask)
    expect(cfg_sampler_step_masked=4)
    gpu(steps=4, image_latents=img, strength=0.5, scheduler="dpmsolver++", guidance_rescale=0.5)
    expect(add_noise_velocity=1, cfg_sampler_step=2, cfg_pred_stats=2)


IMG_CASES = {
    "ddim": dict(steps=25),
    "ddim eta 1": dict(steps=25, eta=1.0),
    "ddim rescale 0.7": dict(steps=25, guidance_rescale=0.7),
    "dpm 2M 20": dict(steps=20, scheduler="dpmsolver++"),
    "dpm 2M 8": dict(steps=8, scheduler="dpmsolver++"),
}


def _analytic_img_run(kw, strength, masked, B=3, H=12, fractional=True):
    kw = dict(kw)
    steps = kw.pop("steps")
    g = torch.Generator().manual_seed(11)
    lat = torch.randn(B, 4, H, H, generator=g)
    img = torch.randn(B, 4, H, H, generator=g) * 1.5
    mask = _mask(B, H, H, g, fractional) if masked else None
    emb = torch.zeros(B, 1, 8)
    executed = steps - S.img2img_start(steps, strength)
    noise = None
    if kw.get("eta", 0) > 0:
        kw["generator"] = [torch.Generator().manual_seed(40 + b) for b in range(B)]
        noise = S.draw_step_noise([torch.Generator().manual_seed(40 + b) for b in range(B)], executed, B,
                                  lat.shape[1:], "cpu")
    got = S.denoise(None, None, None, lat.cuda(), emb.cuda(), emb.cuda(), num_inference_steps=steps,
                    guidance_scale=7.5, experts=_analytic_experts(0.7, 1.6), expert_index=torch.zeros(B).cuda(),
                    image_latents=img.cuda(), strength=strength, mask=None if mask is None else mask.cuda(), **kw)
    torch.cuda.synchronize()
    K.check_abort()
    ref = IO.denoise(SC.analytic_model(0.7, 1.6), lat, steps, 7.5, kw.get("scheduler", "ddim"), kw.get("eta", 0.0),
                     kw.get("solver_order", 2), kw.get("guidance_rescale", 0.0), noise, image_latents=img,
                     strength=strength, mask=mask)
    return got.cpu().double(), ref, img, mask


@pytest.mark.parametrize("case", list(IMG_CASES))
@pytest.mark.parametrize("strength", [0.6, 1.0])
@pytest.mark.parametrize("masked", [False, True])
def test_gpu_img2img_loop_with_closed_form_model_vs_oracle(case, strength, masked):
    got, ref, _, _ = _analytic_img_run(IMG_CASES[case], strength, masked)
    assert SC.rel_err(got, ref) <= 1e-4, (case, strength, masked, SC.rel_err(got, ref))


@pytest.mark.parametrize("case", ["ddim", "ddim eta 1", "dpm 2M 20", "dpm 2M 8"])
def test_inpainting_regions_with_elementwise_model(case):
    """The closed-form model is element-wise, so with a 0/1 mask and no rescale the regenerated elements follow the
    unmasked img2img run and the kept ones end on the image exactly. Both runs step the regenerated elements with the
    same fp32 operations where both use cfg_sampler_step; unmasked DDIM eta 0 runs cfg_ddim_step instead, whose
    rounding differs."""
    inpaint, _, img, mask = _analytic_img_run(IMG_CASES[case], 0.6, True, fractional=False)
    plain, _, _, _ = _analytic_img_run(IMG_CASES[case], 0.6, False)
    regen = mask.expand_as(img).bool()
    assert torch.equal(inpaint[~regen], img.double()[~regen]), case
    if case == "ddim":
        assert SC.rel_err(inpaint[regen], plain[regen]) <= 1e-5, case
    else:
        assert torch.equal(inpaint[regen], plain[regen]), case


TINY_IMG_CASES = {
    "ddim": dict(),
    "dpm 2M": dict(scheduler="dpmsolver++"),
    "ddim eta 1": dict(eta=1.0),
    "ddim rescale 0.7": dict(guidance_rescale=0.7),
}


def _img_inputs(lat, masked, seed):
    g = torch.Generator().manual_seed(seed)
    img = torch.randn(lat.shape, generator=g) * 1.2
    mask = _mask(lat.shape[0], lat.shape[2], lat.shape[3], g) if masked else None
    return img, mask


@pytest.mark.parametrize("case", list(TINY_IMG_CASES))
@pytest.mark.parametrize("masked", [False, True])
def test_tiny_unet_img2img_loop_vs_oracle_loop(case, masked):
    """4-step grid at strength 0.75: three executed steps."""
    import unet_checks as U
    gpu, oracle_model, lat = _tiny_problem()
    img, mask = _img_inputs(lat, masked, 70)
    kw = dict(TINY_IMG_CASES[case])
    noise = None
    if kw.get("eta", 0) > 0:
        kw["generator"] = [torch.Generator().manual_seed(60 + b) for b in range(lat.shape[0])]
        noise = S.draw_step_noise([torch.Generator().manual_seed(60 + b) for b in range(lat.shape[0])], 3,
                                  lat.shape[0], lat.shape[1:], "cpu")
    got = gpu(image_latents=img.cuda(), strength=0.75, mask=None if mask is None else mask.cuda(), **kw)
    ref = IO.denoise(oracle_model, lat, 4, 7.5, kw.get("scheduler", "ddim"), kw.get("eta", 0.0), 2,
                     kw.get("guidance_rescale", 0.0), noise, image_latents=img, strength=0.75, mask=mask)
    max_abs, cos = U.record(f"img2img loop tiny B=3 H=16 4 steps strength 0.75 {case} mask={masked}", got, ref)
    tol_abs, tol_cos = loop_bound(kw.get("scheduler", "ddim"))
    assert max_abs <= tol_abs and cos >= tol_cos, (case, masked, max_abs, cos)


@pytest.mark.parametrize("case", ["ddim", "dpm 2M", "ddim eta 1"])
@pytest.mark.parametrize("masked", [False, True])
def test_mixture_img2img_loop_vs_per_expert_oracle(case, masked):
    import unet_checks as U
    from diffusion_pruning_b200 import PrunedExpertMixture
    from test_expert_mixture_gpu import TINY, build_experts
    experts, oracles, _ = build_experts()
    mixture = PrunedExpertMixture(experts).cuda()
    idx = torch.tensor([3, 1, 0, 1, 2])
    B, H, steps = 5, 16, 4
    g = torch.Generator().manual_seed(5)
    lat = torch.randn(B, 4, H, H, generator=g)
    cond = torch.randn(B, 77, TINY["cross_attention_dim"], generator=g)
    unc = torch.randn(B, 77, TINY["cross_attention_dim"], generator=g)
    img, mask = _img_inputs(lat, masked, 71)
    kw = dict(TINY_IMG_CASES[case])
    noise = None
    if kw.get("eta", 0) > 0:
        noise = S.draw_step_noise([torch.Generator().manual_seed(90 + b) for b in range(B)], 3, B, lat.shape[1:],
                                  "cpu")
        kw["step_noise"] = noise.cuda()
    got = S.denoise(None, None, None, lat.cuda(), cond.cuda(), unc.cuda(), num_inference_steps=steps,
                    guidance_scale=7.5, experts=mixture, expert_index=idx.cuda(), image_latents=img.cuda(),
                    strength=0.75, mask=None if mask is None else mask.cuda(), **kw)
    torch.cuda.synchronize()
    refs = []
    for b, e in enumerate(idx.tolist()):
        emb = torch.cat([unc[b:b + 1], cond[b:b + 1]])

        def model(x2, t, _o=oracles[e], _emb=emb):
            with torch.no_grad():
                return _o(x2.float(), torch.full((2,), t), _emb).double()
        refs.append(IO.denoise(model, lat[b:b + 1], steps, 7.5, kw.get("scheduler", "ddim"), kw.get("eta", 0.0), 2,
                               0.0, None if noise is None else noise[b:b + 1], image_latents=img[b:b + 1],
                               strength=0.75, mask=None if mask is None else mask[b:b + 1]))
    max_abs, cos = U.record(f"expert mixture img2img loop 4 steps strength 0.75 B=5 H=16 {case} mask={masked}", got,
                            torch.cat(refs))
    tol_abs, tol_cos = loop_bound(kw.get("scheduler", "ddim"))
    assert max_abs <= tol_abs and cos >= tol_cos, (case, masked, max_abs, cos)


def _routed_image_inputs(rank, lat):
    g = torch.Generator().manual_seed(700 + rank)
    img = torch.randn(lat.shape, generator=g)
    return img.cuda(), _mask(lat.shape[0], lat.shape[2], lat.shape[3], g).cuda()


def _routed_inpaint_worker(rank, world, port, out_path):
    import sys
    import torch.distributed as dist
    here = os.path.dirname(os.path.abspath(__file__))
    sys.path[:0] = [os.path.dirname(here), here]
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    from diffusion_pruning_b200 import sampling as S
    from test_expert_mixture_gpu import _routed_inputs, _routed_setup
    mix, hyper, quant, code_map = _routed_setup()
    prompt, lat, cond, unc = [t.cuda() for t in _routed_inputs(rank)]
    img, mask = _routed_image_inputs(rank, lat.cpu())
    out, idx = S.routed_sampling(None, hyper, quant, prompt, lat, cond, unc, num_inference_steps=4, guidance_scale=7.5,
                                 experts=mix, code_to_expert=code_map, scheduler="dpmsolver++", image_latents=img,
                                 strength=0.75, mask=mask)
    torch.cuda.synchronize()
    torch.save({"out": out.cpu(), "idx": idx.cpu()}, f"{out_path}.{rank}")
    dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_routed_inpainting_two_ranks(tmp_path):
    """Inpainting at strength 0.75 over 2 NCCL ranks = the single-process run of the same prompts. A misrouted image or
    mask row changes a prompt's output by O(1), far above the loop tolerance."""
    import socket

    import torch.multiprocessing as mp
    import unet_checks as U
    from test_expert_mixture_gpu import _routed_inputs, _routed_setup
    with socket.socket() as sk:
        sk.bind(("127.0.0.1", 0))
        port = sk.getsockname()[1]
    out = str(tmp_path / "inpaint")
    mp.spawn(_routed_inpaint_worker, args=(2, port, out), nprocs=2, join=True)
    mix, hyper, quant, code_map = _routed_setup()
    for r in range(2):
        res = torch.load(f"{out}.{r}")
        prompt, lat, cond, unc = [t.cuda() for t in _routed_inputs(r)]
        img, mask = _routed_image_inputs(r, lat.cpu())
        local, idx = S.routed_sampling(None, hyper, quant, prompt, lat, cond, unc, num_inference_steps=4,
                                       guidance_scale=7.5, experts=mix, code_to_expert=code_map,
                                       scheduler="dpmsolver++", image_latents=img, strength=0.75, mask=mask)
        assert torch.equal(idx.cpu(), res["idx"])
        max_abs, cos = U.metrics(res["out"], local.cpu())
        assert max_abs <= LOOP_MAX_ABS and cos >= LOOP_COS, (r, max_abs, cos)
