"""Every kernel launch of full-width (SD-2.1) U-Net forwards and train steps replayed against a float64 reference of
its contract (tests/launch_replay.py): the production launch shapes -- 2-SM scheme, multi-bucket schedules, placeholder tiles,
conv boxes, fused epilogues -- checked one launch at a time instead of only through end-to-end parity. Each case
also asserts that the engine still issues the feature combinations it is meant to check."""
import pytest
import torch

pytestmark = pytest.mark.gpu

# (case id, batch, latent size, gates: code ids or "soft", reference dtype, env, GEMM feature sets that must occur)
CASES = [
    ("hard_b5_24", 5, 24, (0, 7, 4, 4, 2), torch.float64, {}, [
        ("2sm", "geglu", "lnfold", "multiseg"),
        ("2sm", "linear", "multiseg", "unaligned_start", "placeholder"),
        ("2sm", "conv_s2"),
        ("box8x8x2", "multiseg"), ("box4x4x8", "multiseg"), ("box2x2x32", "multiseg"), ("box1x1x128", "multiseg"),
        ("inactive_seg", "multiseg"), ("1sm", "col_off", "multiseg", "lnfold"), ("balanced", "ragged"),
        ("res_f32", "2sm", "conv"), ("nchw",),
    ]),
    ("hard_b4_32", 4, 32, (0, 3, 3, 7), torch.float64, {}, [
        ("halo", "multiseg", "colstat"),
        ("halo", "a2", "multiseg"),
        ("2sm", "conv_s2", "colstat"),
        ("rowstat", "residual", "multiseg"),
    ]),
    ("soft_b3_16", 3, 16, "soft", torch.float64, {}, [
        ("gate", "geglu", "lnfold"), ("gate", "linear", "col_off"), ("halo", "a2"),
    ]),
    ("hard_b8_64", 8, 64, (0, 1, 2, 3, 4, 5, 6, 7), torch.float32, {}, [
        ("multi_tile_pairs", "2sm", "conv", "multiseg"), ("multi_tile_pairs", "linear", "multiseg"),
        ("multi_tile_pairs", "halo"),
    ]),
    ("hard_b4_32_a_stat", 4, 32, (0, 3, 3, 7), torch.float64, {"APTP_A_STAT": "1"}, [
        ("a_stat", "1sm", "linear", "multiseg"),
    ]),
]


@pytest.fixture(scope="module")
def full_model():
    import unet_checks as U
    model, oracle = U.build_pair(tiny=False)
    del oracle
    return model


@pytest.mark.parametrize("case", [c[0] for c in CASES])
def test_launch_replay(case, full_model, monkeypatch):
    import launch_replay as LR
    from diffusion_pruning_b200.synthetic import synthetic_codes
    _, B, H, gates, cdt, env, want = next(c for c in CASES if c[0] == case)
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    model = full_model
    st = model.get_structure()
    if gates == "soft":
        dim = sum(w for ws in st["width"] for w in ws) + 14
        arch = torch.rand(B, dim, generator=torch.Generator().manual_seed(9)) * 0.9 + 0.05
    else:
        arch = synthetic_codes(st, 8)[list(gates)]
    rec, eng = LR.replay_forward(model, arch, B, H, model.config["cross_attention_dim"], "cuda", monkeypatch.setattr,
                                 cdt=cdt)
    report = rec.report()
    print(f"\n== {case} ==\n{report}")
    rec.dump(case)
    rec.assert_clean()
    missing = [w for w in want if not rec.has(*w)]
    assert not missing, f"{case}: the engine no longer issues GEMM launches with {missing}\n{report}"
    assert rec.counts["grouped_gemm"] > 100 and rec.counts["attention"] > 0


def _train_step(model, arch, monkeypatch):
    """One forward + backward through the training path (train.py) under a Recorder; GEMM launches of the backward
    carry the "bwd" tag."""
    import launch_replay as LR
    import train_checks as T
    from diffusion_pruning_b200.synthetic import split_arch
    from unet_checks import inputs
    sample, t, ctx = inputs(2, 16, model.config["cross_attention_dim"])
    model.set_structure(split_arch(arch, model.get_structure()))
    rec = LR.Recorder(cdt=torch.float64).install(monkeypatch.setattr)
    pred = model(sample.cuda(), t.cuda(), ctx.cuda()).sample
    rec.phase = "bwd"
    T._loss(pred, []).backward()
    torch.cuda.synchronize()
    return rec


def _check(case, rec, want, counts):
    report = rec.report()
    print(f"\n== {case} ==\n{report}")
    rec.dump(case)
    rec.assert_clean()
    missing = [w for w in want if not rec.has(*w)]
    assert not missing, f"{case}: the training path no longer issues launches with {missing}\n{report}"
    for name in counts:
        assert rec.counts[name] > 0 and not rec.unchecked[name], f"{case}: no checked {name} launch\n{report}"


def test_launch_replay_train_soft_gates(full_model, monkeypatch):
    """Soft-gate forward + backward to the gates (the pruning stage): dgrad through the grouped GEMM at full width,
    attention with its log-sum-exp, attention backward."""
    st = full_model.get_structure()
    dim = sum(w for ws in st["width"] for w in ws) + 14
    arch = (torch.rand(2, dim, generator=torch.Generator().manual_seed(9)) * 0.9 + 0.05).cuda().requires_grad_(True)
    rec = _train_step(full_model, arch, monkeypatch)
    assert arch.grad is not None and torch.isfinite(arch.grad).all()
    _check("train_soft_b2_16", rec, [("bwd", "2sm", "linear"), ("bwd", "2sm", "conv"), ("bwd", "1sm", "linear")],
           ["attention", "attention_bwd", "grouped_gemm"])


def test_launch_replay_finetune_backward(full_model, monkeypatch):
    """Fine-tune backward of one static expert (weights trainable): full-width aptp_wgrad launches, linear and 3x3
    stride 1 / 2, accumulated with += into the gradient buffers."""
    from diffusion_pruning_b200.synthetic import synthetic_codes
    arch = synthetic_codes(full_model.get_structure(), 8)[[3, 3]].float().cuda()
    full_model.enable_weight_training(True)
    try:
        rec = _train_step(full_model, arch, monkeypatch)
    finally:
        full_model.enable_weight_training(False)
        full_model.zero_grad(set_to_none=True)
    _check("finetune_b2_16", rec, [("wgrad", "linear", "width1280"), ("wgrad", "conv", "width1280"),
                                   ("wgrad", "conv_s2"), ("bwd", "2sm", "linear")],
           ["wgrad", "attention_bwd"])
