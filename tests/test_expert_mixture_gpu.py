"""PrunedExpertMixture on the B200: fine-tuned experts (every parameter their own) served as one mixed batch, against
the fp32 oracle copy of each sample's own expert after prune()."""
import copy
import os

import pytest
import torch

from diffusion_pruning_b200 import PrunedExpertMixture, UNet2DConditionModelPruned
from diffusion_pruning_b200.synthetic import split_arch, synthetic_codes
from oracle.unet_oracle import GatedUNetOracle, UNetConfig, seeded_init

pytestmark = pytest.mark.gpu

TINY = dict(block_out_channels=(64, 128, 256, 256), attention_head_dim=(1, 2, 4, 4), cross_attention_dim=128)
CODE_OF_EXPERT = (3, 3, 0, 7)   # experts 0 and 1 share code 3: only their weights tell them apart
MAX_ABS_TOL, COS_TOL = 2e-2, 0.9999


def build_experts(beta_std=0.1, perturb=0.1):
    """Four tiny experts fine-tuned from one seeded base: every parameter of expert k perturbed by its own seed
    (GroupNorm / LayerNorm beta != 0). Returns (experts, pruned fp32 oracles, codes [4, dim])."""
    base = GatedUNetOracle(UNetConfig.tiny()).eval()
    seeded_init(base, 0, beta_std)
    st = base.get_structure()
    all_codes = synthetic_codes(st, 8)
    experts, oracles = [], []
    for k, c in enumerate(CODE_OF_EXPERT):
        o = copy.deepcopy(base)
        with torch.no_grad():
            for i, p in enumerate(o.parameters()):
                g = torch.Generator().manual_seed(7919 * (k + 1) + i)
                p.add_(torch.randn(p.shape, generator=g) * (perturb * float(p.abs().mean()) + 1e-3))
        m = UNet2DConditionModelPruned(**TINY)
        m.load_state_dict(o.state_dict())
        m.prune_to(all_codes[c:c + 1].clone())
        o.set_structure(split_arch(all_codes[c:c + 1].clone(), st))
        o.prune()
        experts.append(m.eval())
        oracles.append(o)
    return experts, oracles, all_codes[list(CODE_OF_EXPERT)]


def mixed_inputs(B, H, seed=1):
    g = torch.Generator().manual_seed(seed)
    sample = torch.randn(B, 4, H, H, generator=g)
    ctx = torch.randn(B, 77, TINY["cross_attention_dim"], generator=g)
    t = torch.tensor([981, 661, 341, 21, 500, 3, 777, 150][:B])
    return sample, t, ctx


def oracle_per_sample(oracles, idx, sample, t, ctx):
    with torch.no_grad():
        return torch.cat([oracles[int(e)](sample[b:b + 1], t[b:b + 1], ctx[b:b + 1]) for b, e in enumerate(idx)])


@pytest.fixture(scope="module")
def experts():
    return build_experts()


@pytest.fixture(scope="module")
def mixture(experts):
    return PrunedExpertMixture([copy.deepcopy(e) for e in experts[0]]).cuda()


def test_mixed_batch_vs_own_expert_oracle(experts, mixture):
    """B = 6 at 32x32, experts shuffled, two sharing one code, depth-dropped blocks: every sample against the pruned
    oracle of its own expert."""
    import unet_checks as U
    _, oracles, codes = experts
    assert (codes[:, -14:] == 0).any(), "the case needs a depth-dropped block"
    idx = torch.tensor([1, 3, 0, 2, 1, 0])
    sample, t, ctx = mixed_inputs(6, 32)
    ref = oracle_per_sample(oracles, idx, sample, t, ctx)
    got = mixture(sample.cuda(), t.cuda(), ctx.cuda(), idx.cuda()).sample
    torch.cuda.synchronize()
    for b in range(6):
        max_abs, cos = U.record(f"expert mixture B=6 H=32 sample {b} expert {int(idx[b])}", got[b], ref[b])
        assert max_abs <= MAX_ABS_TOL and cos >= COS_TOL, (b, int(idx[b]), max_abs, cos)
    # CUDA-graph replays (third forward with the same bucket sizes on) and a new assignment with the same sizes
    for perm in (idx, idx, idx[[2, 3, 0, 1, 5, 4]]):
        got2 = mixture(sample.cuda(), t.cuda(), ctx.cuda(), perm.clone().cuda()).sample
        ref2 = oracle_per_sample(oracles, perm, sample, t, ctx)
        max_abs, cos = U.metrics(got2, ref2)
        assert max_abs <= MAX_ABS_TOL and cos >= COS_TOL, (perm.tolist(), max_abs, cos)


def test_same_code_experts_differ(experts):
    """Negative control: the two experts that share a code give outputs more than 10x the tolerance apart, so a launch
    that read the other expert's block could not pass the mixed-batch case."""
    import unet_checks as U
    _, oracles, codes = experts
    assert torch.equal(codes[0], codes[1])
    sample, t, ctx = mixed_inputs(2, 32)
    with torch.no_grad():
        a, b = oracles[0](sample, t, ctx), oracles[1](sample, t, ctx)
    max_abs, _ = U.metrics(a, b)
    assert max_abs > 10 * MAX_ABS_TOL, max_abs


def _reference_with_w2_rows(ref):
    """cpu_kernel_sim.grouped_gemm reads the second operand pair's weights from row 0 of `w2` (what every launch but a
    mixture's passes). This reference adds the record's w2_row_off: the schedule is split by distinct offset and the
    unchanged reference runs once per group (tiles of that group's segments only) on w2 viewed from that row."""
    import dataclasses

    import numpy as np

    def grouped_gemm(a, w, out, sched, **kw):
        segs = sched.segs.cpu().numpy()[:sched.n_segs]
        if kw.get("w2") is None or not segs[:, 9].any():
            return ref(a, w, out, sched, **kw)
        seg_of_tile = sched.tiles[:, 0].cpu().numpy()
        for off in np.unique(segs[:, 9]):
            keep = np.isin(seg_of_tile, np.nonzero(segs[:, 9] == off)[0])
            if keep.any():
                sub = dataclasses.replace(sched, tiles=sched.tiles[torch.as_tensor(keep, device=sched.tiles.device)],
                                          n_tiles=int(keep.sum()))
                ref(a, w, out, sub, **dict(kw, w2=kw["w2"][int(off):]))
    return grouped_gemm


def test_mixture_launch_replay(experts, monkeypatch):
    """Every launch of a mixture forward against its float64 contract, 0 unchecked GEMM launches. At 64x64 the 16x16
    level's ResNet shortcuts are fused into conv2 (2-SM halo scheme): those launches must read two or more blocks of
    w2, and the layers that used to share one weight set (conv_in, time MLP, proj_in / proj_out, samplers, conv_out)
    must run with one segment per expert."""
    import cpu_kernel_sim
    import launch_replay as LR
    from diffusion_pruning_b200.unet import _Engine
    mix = PrunedExpertMixture([copy.deepcopy(e) for e in experts[0]]).cuda()
    idx = torch.tensor([2, 0, 3, 1])
    sample, t, ctx = mixed_inputs(4, 64)
    mix._prepare_index(idx, 4)
    eng = _Engine(mix.experts[0], torch.device("cuda"), sources=list(mix.experts), gates=mix)
    segs_of, w2_blocks = {}, []
    orig = LR.gemm_tags

    def tags(kw, sched):
        segs_of[eng._label] = max(segs_of.get(eng._label, 0), sched.n_segs)
        if kw.get("a2") is not None:
            live = sched.tiles[:, 0].cpu().unique().tolist()
            w2_blocks.append(len({int(sched.segs[si, 9]) for si in live}))
        return orig(kw, sched)
    monkeypatch.setattr(LR, "gemm_tags", tags)
    monkeypatch.setattr(cpu_kernel_sim, "grouped_gemm", _reference_with_w2_rows(cpu_kernel_sim.grouped_gemm))
    rec = LR.Recorder(cdt=torch.float64, label=lambda: eng._label).install(monkeypatch.setattr)
    with torch.no_grad():
        eng.run(sample.cuda(), t.cuda(), ctx.cuda())
    report = rec.report()
    print(report)
    rec.dump("expert_mixture_b4_64")
    rec.assert_clean()
    assert rec.counts["grouped_gemm"] > 50 and rec.unchecked["grouped_gemm"] == 0, report
    assert rec.has("halo", "a2") and max(w2_blocks, default=0) >= 2, (w2_blocks, report)
    for lab in ("('conv_in',", "('te', 'te1')", "('te', 'te2')", "('lin', 'pi.", "('lin', 'po.", "('conv', 'ds.",
                "('conv', 'us.", "('conv_out',"):
        hits = [n for k, n in segs_of.items() if k.startswith(lab)]
        assert hits and min(hits) > 1, (lab, hits, sorted(segs_of))


def test_routed_sampling_with_experts(experts, mixture):
    """4-step CFG DDIM at 16x16 with experts=: against a per-expert loop of the oracle sampler (loop bound of
    tests/test_sampling_gpu.py)."""
    import unet_checks as U
    from diffusion_pruning_b200 import sampling as S
    from oracle import router_oracle as R
    from oracle import sampling_oracle as SO
    from diffusion_pruning_b200.synthetic import DEPTH_ORDER
    _, oracles, codes = experts
    st = mixture.experts[0].get_structure()
    layout = R.ArchLayout(st, DEPTH_ORDER)
    idx = torch.tensor([3, 1, 0, 1, 2])
    g = torch.Generator().manual_seed(5)
    B, H = 5, 16
    lat = torch.randn(B, 4, H, H, generator=g)
    cond = torch.randn(B, 77, TINY["cross_attention_dim"], generator=g)
    unc = torch.randn(B, 77, TINY["cross_attention_dim"], generator=g)
    got = S.denoise(None, None, None, lat.cuda(), cond.cuda(), unc.cuda(), num_inference_steps=4, guidance_scale=7.5,
                    experts=mixture, expert_index=idx.cuda())
    ref = torch.cat([SO.denoise(oracles[int(e)], layout, codes[int(e)][None].clone(), lat[b:b + 1], cond[b:b + 1],
                                unc[b:b + 1], steps=4, guidance=7.5) for b, e in enumerate(idx)])
    max_abs, cos = U.record("expert mixture sampling 4 steps B=5 H=16", got, ref)
    assert max_abs <= 6e-2 and cos >= 0.998, (max_abs, cos)


def _routed_setup():
    from diffusion_pruning_b200 import HyperStructure, StructureVectorQuantizer
    from diffusion_pruning_b200.synthetic import DEPTH_ORDER
    experts, _, _ = build_experts()
    mix = PrunedExpertMixture(experts, expert_ids=[5, 1, 0, 7]).cuda()
    st = mix.experts[0].get_structure()
    torch.manual_seed(9)
    hyper = HyperStructure(structure=st, input_dim=16, wn_flag=False, linear_bias=True).cuda().eval()
    quant = StructureVectorQuantizer(n_e=8, structure=st, beta=0.25, temperature=0.4, base=3,
                                     depth_order=list(DEPTH_ORDER), non_zero_width=True,
                                     resource_aware_normalization=False, optimal_transport=True).cuda().eval()
    quant.embedding_gs.data = (synthetic_codes(st, 8).float() * 0.9 + 0.05).cuda()
    code_map = torch.arange(8) % 4   # every code served by an expert; experts serve several codes
    return mix, hyper, quant, code_map


def _routed_inputs(rank, B=4):
    g = torch.Generator().manual_seed(100 + rank)
    return (torch.randn(B, 16, generator=g), torch.randn(B, 4, 16, 16, generator=g),
            torch.randn(B, 77, TINY["cross_attention_dim"], generator=g),
            torch.randn(B, 77, TINY["cross_attention_dim"], generator=g))


def _routed_worker(rank, world, port, out_path):
    import sys
    import torch.distributed as dist
    here = os.path.dirname(os.path.abspath(__file__))
    sys.path[:0] = [os.path.dirname(here), here]
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    from diffusion_pruning_b200 import sampling as S
    mix, hyper, quant, code_map = _routed_setup()
    prompt, lat, cond, unc = [t.cuda() for t in _routed_inputs(rank)]
    out, idx = S.routed_sampling(None, hyper, quant, prompt, lat, cond, unc, num_inference_steps=3,
                                 guidance_scale=7.5, experts=mix, code_to_expert=code_map)
    torch.cuda.synchronize()
    torch.save({"out": out.cpu(), "idx": idx.cpu()}, f"{out_path}.{rank}")
    dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_routed_sampling_with_experts_two_ranks(tmp_path):
    """A 2-rank NCCL run of routed_sampling(experts=...) matches the single-process result on each rank's prompts."""
    import socket
    import torch.multiprocessing as mp
    from diffusion_pruning_b200 import sampling as S
    with socket.socket() as sk:
        sk.bind(("127.0.0.1", 0))
        port = sk.getsockname()[1]
    out = str(tmp_path / "mix")
    mp.spawn(_routed_worker, args=(2, port, out), nprocs=2, join=True)
    mix, hyper, quant, code_map = _routed_setup()
    for r in range(2):
        res = torch.load(f"{out}.{r}")
        prompt, lat, cond, unc = [t.cuda() for t in _routed_inputs(r)]
        local, idx = S.routed_sampling(None, hyper, quant, prompt, lat, cond, unc, num_inference_steps=3,
                                       guidance_scale=7.5, experts=mix, code_to_expert=code_map)
        assert torch.equal(idx.cpu(), res["idx"])
        assert torch.allclose(local.cpu(), res["out"], rtol=0, atol=1e-4), (local.cpu() - res["out"]).abs().max()
