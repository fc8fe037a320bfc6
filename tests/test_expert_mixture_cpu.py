"""PrunedExpertMixture host logic without a GPU: loading fine-tuned experts, rejected inputs, the code -> expert map, the
packed segment table's w2_row_off, and the whole mixture forward with the kernels replaced by their torch emulation
(tests/cpu_kernel_sim.py) against each sample's own pruned fp32 oracle."""
import copy

import numpy as np
import pytest
import torch

import cpu_kernel_sim
from diffusion_pruning_b200 import PrunedExpertMixture, UNet2DConditionModelPruned
from diffusion_pruning_b200 import kernels as K
from diffusion_pruning_b200.unet import _Engine
from test_expert_mixture_gpu import TINY, build_experts, mixed_inputs, oracle_per_sample

# bf16 bound of the engine's CPU emulation (tests/test_engine_cpu.py)
MAX_ABS_TOL, COS_TOL = 2e-2, 0.9998


@pytest.fixture(scope="module")
def experts():
    return build_experts()


def _metrics(got, ref):
    scale = max(1.0, ref.abs().max().item())
    return ((got - ref).abs().max().item() / scale,
            torch.nn.functional.cosine_similarity(got.flatten(), ref.flatten(), dim=0).item())


def _run_sim(mix, idx, sample, t, ctx):
    mix._prepare_index(idx, sample.shape[0])
    eng = _Engine(mix.experts[0], torch.device("cpu"), sources=list(mix.experts), gates=mix)
    with torch.no_grad():
        out, _ = eng.run(sample, t, ctx)
    return out, eng


def test_mixed_batch_cpu_emulation(experts, monkeypatch):
    """Shuffled experts, two sharing a code, depth-dropped blocks, CFG-style tiling of a [B/2] index."""
    cpu_kernel_sim.install(monkeypatch)
    models, oracles, _ = experts
    mix = PrunedExpertMixture(models)
    sample, t, ctx = mixed_inputs(6, 16)
    idx = torch.tensor([1, 3, 0, 2, 1, 0])
    got, eng = _run_sim(mix, idx, sample, t, ctx)
    ref = oracle_per_sample(oracles, idx, sample, t, ctx)
    for b in range(6):
        err, cos = _metrics(got[b], ref[b])
        assert err < MAX_ABS_TOL and cos > COS_TOL, (b, err, cos)
    # every prunable pack has one variant per expert in the batch, even where two experts share a code
    assert all(d["V"] == 4 for k, d in eng.expert.items() if isinstance(d, dict) and "V" in d)
    # [B/2] index on a doubled batch: sample b runs on expert idx[b % 3]
    half = torch.tensor([2, 0, 1])
    got2, _ = _run_sim(mix, half, sample, t, ctx)
    ref2 = oracle_per_sample(oracles, half.repeat(2), sample, t, ctx)
    err, cos = _metrics(got2, ref2)
    assert err < MAX_ABS_TOL and cos > COS_TOL, (err, cos)


def test_one_expert_mixture_issues_the_experts_launches(experts, monkeypatch):
    """A mixture of one expert is the expert's own engine: the same segment tables launch for launch, the same
    output bit for bit."""
    cpu_kernel_sim.install(monkeypatch)
    model = copy.deepcopy(experts[0][2])
    tables = {"model": [], "mix": []}
    real = K.grouped_gemm
    which = ["model"]

    def spy(a, w, out, sched, **kw):
        tables[which[0]].append(sched.segs.cpu().numpy()[:sched.n_segs].copy())
        return real(a, w, out, sched, **kw)
    monkeypatch.setattr(K, "grouped_gemm", spy)
    sample, t, ctx = mixed_inputs(3, 16)
    with torch.no_grad():
        ref, _ = _Engine(model, torch.device("cpu")).run(sample, t, ctx)
    which[0] = "mix"
    got, _ = _run_sim(PrunedExpertMixture([model]), torch.zeros(3, dtype=torch.long), sample, t, ctx)
    assert len(tables["model"]) == len(tables["mix"]) > 50
    for i, (a, b) in enumerate(zip(tables["model"], tables["mix"])):
        assert np.array_equal(a, b), f"launch {i}: {a} != {b}"
    assert torch.equal(got, ref)


def test_segment_table_carries_w2_row_off():
    segs = [K.Segment(0, 256, 320, 5), K.Segment(256, 512, 320, 5, w_row_off=320, w2_row_off=320)]
    sched = K.build_schedule(segs, 160, "cpu")
    tab = sched.segs.numpy()
    assert tab.shape == (2, 12)
    assert tab[:, 9].tolist() == [0, 320]
    assert tab[:, 5].tolist() == [0, 320]


def test_loader_sliced_and_dense_round_trip(experts, tmp_path):
    """Fine-tuned experts as FineTuner writes them: `<dir>/unet/` (diffusers layout, physically sliced or dense
    tensors) and `<dir>/arch_vector.pt`."""
    models = experts[0]
    dirs = []
    for k, m in enumerate(models[:3]):
        d = tmp_path / f"expert{k}"
        m.save_pretrained(str(d / "unet"), sliced=(k != 1))
        torch.save(m.arch_vector, d / "arch_vector.pt")
        dirs.append(str(d))
    mix = PrunedExpertMixture.from_pretrained(dirs, expert_ids=[4, 2, 6])
    assert mix.n_experts == 3 and mix.expert_ids == [4, 2, 6]
    for k in range(3):
        assert torch.equal(mix.experts[k].arch_vector, models[k].arch_vector)
        a, b = mix.experts[k].sliced_state_dict(), models[k].sliced_state_dict()
        assert a.keys() == b.keys()
        assert all(torch.equal(a[n], b[n]) for n in a), k
    assert np.array_equal(mix.codes, PrunedExpertMixture(models[:3]).codes)


def test_code_to_expert_map(experts):
    mix = PrunedExpertMixture(experts[0], expert_ids=[5, 1, 0, 7])
    assert mix.code_to_expert(8).tolist() == [2, 1, -1, -1, -1, 0, -1, 3]
    with pytest.raises(ValueError):
        mix.code_to_expert(6)   # expert 3 was fine-tuned for code 7
    with pytest.raises(ValueError):
        PrunedExpertMixture(experts[0], expert_ids=[0, 0, 1, 2])


def test_rejected_inputs(experts):
    models = experts[0]
    other = UNet2DConditionModelPruned(**dict(TINY, cross_attention_dim=64), arch_vector=models[0].arch_vector)
    with pytest.raises(ValueError, match="different config"):
        PrunedExpertMixture([models[0], other])
    with pytest.raises(ValueError, match="no architecture vector"):
        PrunedExpertMixture([models[0], UNet2DConditionModelPruned(**TINY)])
    with pytest.raises(ValueError):
        PrunedExpertMixture([])
    mix = PrunedExpertMixture(models)
    sample, t, ctx = mixed_inputs(4, 16)
    for bad in (torch.tensor([0, 1, 4, 2]), torch.tensor([0, -1, 1, 2])):
        with pytest.raises(IndexError):
            mix(sample, t, ctx, bad)
    with pytest.raises(ValueError):
        mix(sample, t, ctx, torch.tensor([0, 1, 2]))           # 4 samples, 3 indices
    with pytest.raises(TypeError):
        mix(sample, t, ctx, torch.tensor([0.0, 1.0, 2.0, 3.0]))
    with pytest.raises(RuntimeError, match="CUDA"):
        mix(sample, t, ctx, torch.tensor([0, 1, 2, 3]))         # CPU inputs
    with pytest.raises(NotImplementedError):
        mix.enable_weight_training()
