"""Schedulers of the sampling loop on the B200: aptp_cfg_pred_stats / aptp_cfg_sampler_step against float64, the default
path's launches, the GPU loop against the float64 oracle loop with a closed-form model, the tiny U-Net and an expert
mixture."""
import os
import types

import pytest
import torch

import sampler_checks as SC
from diffusion_pruning_b200 import kernels as K
from diffusion_pruning_b200 import sampling as S
from oracle import sampler_oracle as SO2

pytestmark = pytest.mark.gpu

LOOP_MAX_ABS, LOOP_COS = 6e-2, 0.998   # the 4-step guided loop bound of tests/test_sampling_gpu.py


def loop_bound(scheduler):
    """(max-abs over scale, cosine) bound of a 4-step guided loop against the fp32 oracle loop. DPM-Solver++(2M) gets the
    DDIM bound with twice the max-abs and 1 - cosine: on the 4-step grid its second-order step at t = 251 extrapolates
    x0 with weights 2.5 and -1.6 (r = h_last / h = 0.29), so the endpoint is more sensitive to the U-Net's bf16 error
    in x0. Summed in quadrature over the steps, that sensitivity (from sampler_plan's coefficients, model Jacobian left
    out) is 2.10 for DPM-Solver++(2M) and 0.73 for DDIM. Measured on a B200 (1000 W): tiny U-Net 8.2e-2 / 0.99823,
    mixture 6.6e-2 / 0.99812 (DDIM eta 1 on the same problems: 5.0e-2 / 0.99872, 5.4e-2 / 0.99904)."""
    if scheduler == "dpmsolver++":
        return 2 * LOOP_MAX_ABS, 1 - 2 * (1 - LOOP_COS)
    return LOOP_MAX_ABS, LOOP_COS


def _step_case(scheduler, order, step, steps=25, eta=0.0):
    plan = S.sampler_plan(scheduler, steps, eta, order)
    return plan[step]


KERNEL_CASES = {
    "ddim eta 0": ("ddim", 2, 0.0, 3, False),
    "ddim eta 0.5": ("ddim", 2, 0.5, 3, False),
    "ddim eta 1": ("ddim", 2, 1.0, 24, False),
    "dpm order 1": ("dpmsolver++", 1, 0.0, 0, False),
    "dpm order 2": ("dpmsolver++", 2, 0.0, 7, False),
    "dpm order 2 in-place history": ("dpmsolver++", 2, 0.0, 7, True),
}


def _kernel_vs_float64(case, vpred, rescale, B, H, W, guidance=7.5, seed=0):
    scheduler, order, eta, step, inplace = KERNEL_CASES[case]
    st = _step_case(scheduler, order, step, eta=eta)
    n = 4 * H * W
    g = torch.Generator().manual_seed(seed)
    pred = torch.randn(2 * B, 4, H, W, generator=g)
    pred[B:] = pred[B:] * 1.3 + 0.2
    x = torch.randn(B, 4, H, W, generator=g)
    hist = torch.randn(B, 4, H, W, generator=g)
    steps = 5
    noise_all = torch.randn(B, steps, 4, H, W, generator=g)   # step 2 of a [B, steps, ...] block: strided rows
    d = {k: v.cuda() for k, v in dict(pred=pred, x=x, hist=hist, noise=noise_all).items()}
    out = torch.full_like(d["x"], float("nan"))
    hist_out = d["hist"] if inplace else torch.full_like(d["x"], float("nan"))
    partials = None
    if rescale > 0:
        partials = torch.empty(B, K.SAMPLER_STAT_CHUNKS, 4, device="cuda", dtype=torch.float64)
        K.cfg_pred_stats(d["pred"], n, B, guidance, partials)
    uses_h, uses_z = st.coeffs[4] != 0, st.coeffs[6] != 0
    K.cfg_sampler_step(d["pred"], d["x"], out, n, B, guidance, rescale, partials, st.coeffs,
                       d["hist"] if uses_h else None, hist_out if st.store_x0 or inplace else None,
                       d["noise"][:, 2] if uses_z else None, d["noise"].stride(0), vpred)
    torch.cuda.synchronize()
    # float64 reference
    p, xd, hd, z = pred.double(), x.double(), hist.double(), noise_all[:, 2].double()
    m = p[:B] + guidance * (p[B:] - p[:B])
    if rescale > 0:
        m = SO2.rescale(m, p[B:], rescale)
    sa, sb, c_x, c_0, c_h, c_e, c_n = st.coeffs
    x0, eps = SO2.x0_eps(m, xd, sa * sa, vpred)
    ref = c_x * xd + c_0 * x0 + c_h * hd + c_e * eps + c_n * z
    err = SC.rel_err(out.cpu().double(), ref)
    assert err <= 1e-5, (case, vpred, rescale, err)
    if st.store_x0 or inplace:
        assert SC.rel_err(hist_out.cpu().double(), x0) <= 1e-5, (case, "x0 history")
    return partials


@pytest.mark.parametrize("case", list(KERNEL_CASES))
@pytest.mark.parametrize("vpred", [True, False])
@pytest.mark.parametrize("rescale", [0.0, 0.7, 1.0])
def test_sampler_step_kernel_vs_float64(case, vpred, rescale):
    """Odd batch, n_per_sample = 4 x 17 x 23 (not a multiple of the statistics chunks' vector count)."""
    _kernel_vs_float64(case, vpred, rescale, B=3, H=17, W=23)


def test_sampler_step_kernel_at_sampling_shape():
    for case in ("ddim eta 1", "dpm order 2 in-place history"):
        _kernel_vs_float64(case, True, 0.7, B=16, H=96, W=96, seed=1)


def test_pred_stats_bit_reproducible_and_exact():
    B, H, W, guidance = 5, 33, 29, 7.5
    n = 4 * H * W
    g = torch.Generator().manual_seed(2)
    pred = (torch.randn(2 * B, 4, H, W, generator=g) * 3 + 0.5).cuda()
    a = torch.empty(B, K.SAMPLER_STAT_CHUNKS, 4, device="cuda", dtype=torch.float64)
    b = torch.empty_like(a)
    K.cfg_pred_stats(pred, n, B, guidance, a)
    K.cfg_pred_stats(pred, n, B, guidance, b)
    torch.cuda.synchronize()
    assert torch.equal(a, b), "cfg_pred_stats is not bit-reproducible"
    p = pred.double().cpu().view(2 * B, -1)
    m = p[:B] + guidance * (p[B:] - p[:B])
    want = torch.stack([p[B:].sum(1), (p[B:] ** 2).sum(1), m.sum(1), (m ** 2).sum(1)], 1)
    got = a.sum(1).cpu()
    assert torch.allclose(got[:, :2], want[:, :2], rtol=1e-12, atol=1e-9), (got, want)
    assert torch.allclose(got[:, 2:], want[:, 2:], rtol=1e-6, atol=1e-3), (got, want)


def _tiny_problem(B=3, H=16, code_ids=(0, 3, 7), seed=3):
    from diffusion_pruning_b200 import HyperStructure
    from diffusion_pruning_b200.synthetic import DEPTH_ORDER, synthetic_codes
    from oracle import router_oracle as R
    from oracle.step_oracle import split
    from unet_checks import build_pair
    model, oracle = build_pair(True, beta_std=0.1)
    st = model.get_structure()
    arch = synthetic_codes(st, 8)[list(code_ids)]
    layout = R.ArchLayout(st, DEPTH_ORDER)
    hyper = HyperStructure(structure=st, input_dim=16, wn_flag=False, linear_bias=True)
    g = torch.Generator().manual_seed(seed)
    cd = model.config["cross_attention_dim"]
    lat = torch.randn(B, 4, H, H, generator=g)
    cond = torch.randn(B, 77, cd, generator=g)
    unc = torch.randn(B, 77, cd, generator=g)
    oracle.set_structure(split(arch.clone(), layout))
    emb = torch.cat([unc, cond])

    def oracle_model(x2, t):
        with torch.no_grad():
            return oracle(x2.float(), torch.full((x2.shape[0],), t), emb).double()

    def gpu(**kw):
        out = S.denoise(model, hyper, arch.clone().cuda(), lat.cuda(), cond.cuda(), unc.cuda(),
                        num_inference_steps=kw.pop("steps", 4), guidance_scale=7.5, **kw)
        torch.cuda.synchronize()
        K.check_abort()
        return out
    return gpu, oracle_model, lat


def test_default_denoise_launches_only_cfg_ddim_step(monkeypatch):
    gpu, _, _ = _tiny_problem()
    calls = {"cfg_ddim_step": 0, "cfg_sampler_step": 0, "cfg_pred_stats": 0}
    for name in calls:
        orig = getattr(K, name)

        def counted(*a, _orig=orig, _name=name, **kw):
            calls[_name] += 1
            return _orig(*a, **kw)
        monkeypatch.setattr(K, name, counted)
    default = gpu(steps=3)
    assert calls == {"cfg_ddim_step": 3, "cfg_sampler_step": 0, "cfg_pred_stats": 0}, calls
    spelled = gpu(steps=3, scheduler="ddim", eta=0.0, guidance_rescale=0.0)
    assert torch.equal(default, spelled)
    assert calls == {"cfg_ddim_step": 6, "cfg_sampler_step": 0, "cfg_pred_stats": 0}, calls
    gpu(steps=3, scheduler="dpmsolver++", guidance_rescale=0.5)
    assert calls == {"cfg_ddim_step": 6, "cfg_sampler_step": 3, "cfg_pred_stats": 3}, calls


def _analytic_experts(s_uncond, s_cond):
    acp = S.alphas_cumprod().double().cuda()

    def experts(x2, t, emb, expert_index):
        B = x2.shape[0] // 2
        ab = acp[int(t[0].item())].float()
        v = torch.cat([SC.analytic_v(x2[:B], ab, s_uncond), SC.analytic_v(x2[B:], ab, s_cond)])
        return types.SimpleNamespace(sample=v)
    return experts


ANALYTIC_CASES = {
    "ddim 25": dict(steps=25),
    "ddim 25 eta 1": dict(steps=25, eta=1.0),
    "ddim 25 rescale 0.7": dict(steps=25, guidance_rescale=0.7),
    "dpm order 1 25": dict(steps=25, scheduler="dpmsolver++", solver_order=1),
    "dpm 2M 8": dict(steps=8, scheduler="dpmsolver++"),
    "dpm 2M 20 rescale 1": dict(steps=20, scheduler="dpmsolver++", guidance_rescale=1.0),
}


def _analytic_run(kw, B=3, H=12):
    kw = dict(kw)
    steps = kw.pop("steps")
    g = torch.Generator().manual_seed(11)
    lat = torch.randn(B, 4, H, H, generator=g)
    emb = torch.zeros(B, 1, 8)
    noise = None
    if kw.get("eta", 0) > 0:
        kw["generator"] = [torch.Generator().manual_seed(40 + b) for b in range(B)]
        noise = S.draw_step_noise([torch.Generator().manual_seed(40 + b) for b in range(B)], steps, B, lat.shape[1:],
                                  "cpu")
    got = S.denoise(None, None, None, lat.cuda(), emb.cuda(), emb.cuda(), num_inference_steps=steps,
                    guidance_scale=7.5, experts=_analytic_experts(0.7, 1.6), expert_index=torch.zeros(B).cuda(), **kw)
    torch.cuda.synchronize()
    ref = SO2.denoise(SC.analytic_model(0.7, 1.6), lat, steps, 7.5, kw.get("scheduler", "ddim"), kw.get("eta", 0.0),
                      kw.get("solver_order", 2), kw.get("guidance_rescale", 0.0), noise)
    return got.cpu().double(), ref


@pytest.mark.parametrize("case", list(ANALYTIC_CASES))
def test_gpu_loop_with_closed_form_model_vs_oracle(case):
    got, ref = _analytic_run(ANALYTIC_CASES[case])
    assert SC.rel_err(got, ref) <= 1e-4, (case, SC.rel_err(got, ref))


def test_gpu_dpm_order1_equals_ddim():
    a, _ = _analytic_run(ANALYTIC_CASES["dpm order 1 25"])
    b, _ = _analytic_run(ANALYTIC_CASES["ddim 25"])
    assert SC.rel_err(a, b) <= 1e-5, SC.rel_err(a, b)


TINY_CASES = {
    "dpm 2M": dict(scheduler="dpmsolver++"),
    "ddim eta 1": dict(eta=1.0),
    "ddim rescale 0.7": dict(guidance_rescale=0.7),
}


@pytest.mark.parametrize("case", list(TINY_CASES))
def test_tiny_unet_loop_vs_oracle_loop(case):
    import unet_checks as U
    gpu, oracle_model, lat = _tiny_problem()
    kw = dict(TINY_CASES[case])
    noise = None
    if kw.get("eta", 0) > 0:
        kw["generator"] = [torch.Generator().manual_seed(60 + b) for b in range(lat.shape[0])]
        noise = S.draw_step_noise([torch.Generator().manual_seed(60 + b) for b in range(lat.shape[0])], 4,
                                  lat.shape[0], lat.shape[1:], "cpu")
    got = gpu(**kw)
    ref = SO2.denoise(oracle_model, lat, 4, 7.5, kw.get("scheduler", "ddim"), kw.get("eta", 0.0), 2,
                      kw.get("guidance_rescale", 0.0), noise)
    max_abs, cos = U.record(f"sampler loop tiny B=3 H=16 4 steps {case}", got, ref)
    tol_abs, tol_cos = loop_bound(kw.get("scheduler", "ddim"))
    assert max_abs <= tol_abs and cos >= tol_cos, (case, max_abs, cos)


@pytest.mark.parametrize("case", ["dpm 2M", "ddim eta 1"])
def test_mixture_loop_vs_per_expert_oracle(case):
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
    kw = dict(TINY_CASES[case])
    noise = None
    if kw.get("eta", 0) > 0:
        noise = S.draw_step_noise([torch.Generator().manual_seed(90 + b) for b in range(B)], steps, B, lat.shape[1:],
                                  "cpu")
        kw["step_noise"] = noise.cuda()
    got = S.denoise(None, None, None, lat.cuda(), cond.cuda(), unc.cuda(), num_inference_steps=steps,
                    guidance_scale=7.5, experts=mixture, expert_index=idx.cuda(), **kw)
    torch.cuda.synchronize()
    refs = []
    for b, e in enumerate(idx.tolist()):
        emb = torch.cat([unc[b:b + 1], cond[b:b + 1]])

        def model(x2, t, _o=oracles[e], _emb=emb):
            with torch.no_grad():
                return _o(x2.float(), torch.full((2,), t), _emb).double()
        refs.append(SO2.denoise(model, lat[b:b + 1], steps, 7.5, kw.get("scheduler", "ddim"), kw.get("eta", 0.0), 2,
                                0.0, None if noise is None else noise[b:b + 1]))
    max_abs, cos = U.record(f"expert mixture sampler loop 4 steps B=5 H=16 {case}", got, torch.cat(refs))
    tol_abs, tol_cos = loop_bound(kw.get("scheduler", "ddim"))
    assert max_abs <= tol_abs and cos >= tol_cos, (case, max_abs, cos)


def _routed_noise_worker(rank, world, port, out_path):
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
    gens = [torch.Generator().manual_seed(500 + 10 * rank + b) for b in range(lat.shape[0])]
    out, idx = S.routed_sampling(None, hyper, quant, prompt, lat, cond, unc, num_inference_steps=3, guidance_scale=7.5,
                                 experts=mix, code_to_expert=code_map, eta=1.0, generator=gens)
    torch.cuda.synchronize()
    torch.save({"out": out.cpu(), "idx": idx.cpu()}, f"{out_path}.{rank}")
    dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_routed_stochastic_sampling_two_ranks(tmp_path):
    """eta = 1 with one generator per prompt over 2 NCCL ranks = the single-process denoise of the same prompts. A
    misrouted noise row changes a prompt's output by O(1), far above the loop tolerance."""
    import socket

    import torch.multiprocessing as mp
    import unet_checks as U
    from test_expert_mixture_gpu import _routed_inputs, _routed_setup
    with socket.socket() as sk:
        sk.bind(("127.0.0.1", 0))
        port = sk.getsockname()[1]
    out = str(tmp_path / "noise")
    mp.spawn(_routed_noise_worker, args=(2, port, out), nprocs=2, join=True)
    mix, hyper, quant, code_map = _routed_setup()
    for r in range(2):
        res = torch.load(f"{out}.{r}")
        prompt, lat, cond, unc = [t.cuda() for t in _routed_inputs(r)]
        gens = [torch.Generator().manual_seed(500 + 10 * r + b) for b in range(lat.shape[0])]
        local, idx = S.routed_sampling(None, hyper, quant, prompt, lat, cond, unc, num_inference_steps=3,
                                       guidance_scale=7.5, experts=mix, code_to_expert=code_map, eta=1.0,
                                       generator=gens)
        assert torch.equal(idx.cpu(), res["idx"])
        max_abs, cos = U.metrics(res["out"], local.cpu())
        assert max_abs <= LOOP_MAX_ABS and cos >= LOOP_COS, (r, max_abs, cos)
