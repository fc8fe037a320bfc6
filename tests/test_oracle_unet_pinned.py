"""Pins oracle/unet_oracle.py to outputs of the REFERENCE'S OWN code (tests/golden/unet_ref.npz, produced by
tests/golden/make_unet_goldens.py executing pdm/models/unet/blocks.py, unet_2d_conditional.py and pdm/utils/op_counter.py
in place over constructor-only diffusers stand-ins). CPU only.

Bar: bit-for-bit in fp32 wherever the oracle performs the same torch ops in the same order as the reference (every
gated forward); <= 1e-5 where the reference's prune() physically slices weights and the oracle keeps exact-zero gates
(a different summation length in the following GEMM), and for MAC totals accumulated in a different order."""
import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))

from oracle import unet_oracle as O  # noqa: E402
from diffusion_pruning_b200.synthetic import split_arch, synthetic_codes  # noqa: E402
import make_unet_goldens as G  # noqa: E402

GOLD = np.load(os.path.join(ROOT, "tests", "golden", "unet_ref.npz"))


@pytest.fixture(scope="module", autouse=True)
def golden_threads():
    """Sum in the order the goldens were recorded in: same intra-op thread count (make_unet_goldens.THREADS)."""
    n = torch.get_num_threads()
    torch.set_num_threads(G.THREADS)
    yield
    torch.set_num_threads(n)


def _exact(got: torch.Tensor, key: str, tol: float = 0.0):
    ref = torch.from_numpy(GOLD[key])
    assert got.shape == ref.shape, (key, got.shape, ref.shape)
    diff = (got - ref).abs().max().item()
    if tol == 0.0:
        # same ops, same order, same machine class: expected identical; a different BLAS build may differ in the last
        # bits, which is reported rather than hidden
        assert torch.equal(got, ref) or diff <= 2e-6, f"{key}: max diff {diff}"
    else:
        assert diff <= tol, f"{key}: max diff {diff} > {tol}"
    return diff


@pytest.fixture(scope="module")
def tiny_oracle():
    torch.manual_seed(0)
    cfg = O.UNetConfig.tiny()
    oracle = O.GatedUNetOracle(cfg).eval()
    O.seeded_init(oracle, 0, 0.1)
    return cfg, oracle


@pytest.mark.parametrize("case", ["hard", "soft", "cfg", "ones"])
def test_unet_forward_matches_reference_forward(tiny_oracle, case):
    """UNet2DConditionModelGated.forward (unet_2d_conditional.py:1415-1726) incl. every gated layer forward."""
    cfg, oracle = tiny_oracle
    st = oracle.get_structure()
    arch, B = G.unet_cases(st)[case]
    sample, t, ctx = G.unet_inputs(B, G.TINY_H, cfg.cross_attention_dim)
    oracle.set_structure(split_arch(arch.clone(), st))
    with torch.no_grad():
        out, taps = oracle(sample, t, ctx, return_blocks=True)
    _exact(out, f"unet_{case}")
    if case == "hard":  # the nine hooked block outputs (trainer.py:496-511)
        assert len(taps) == 9
        for i, tp in enumerate(taps):
            _exact(tp, f"hard_tap{i}")


def test_macs_match_reference_op_counter_and_calc_macs(tiny_oracle):
    """count_ops_and_params (op_counter.py:19) + calc_macs (unet_2d_conditional.py:2124-2163) as the reference ran them."""
    cfg, oracle = tiny_oracle
    st = oracle.get_structure()
    oracle.count_macs(G.TINY_H, G.TINY_H, 77)
    dim = sum(w for ws in st["width"] for w in ws) + 14
    oracle.set_structure(split_arch(torch.ones(1, dim), st))
    d = oracle.calc_macs()
    ref = GOLD["macs_ones"]
    assert float(d["total_macs"]) == ref[0] and float(d["prunable_macs"]) == ref[1]
    assert abs(float(d["cur_prunable_macs"]) - ref[2]) <= 1e-6 * ref[2]
    assert abs(float(d["cur_total_macs"]) - ref[3]) <= 1e-6 * ref[3]
    codes = synthetic_codes(st, 8)
    oracle.set_structure(split_arch(codes.clone(), st))
    d8 = oracle.calc_macs()
    np.testing.assert_allclose(d8["cur_prunable_macs"].double().numpy(), GOLD["macs_codes_cur_prunable"], rtol=1e-6)
    np.testing.assert_allclose(d8["cur_total_macs"].double().numpy(), GOLD["macs_codes_cur_total"], rtol=1e-6)


def test_pruned_unet_matches_reference_prune_sweep(tiny_oracle):
    """The prune() / prune_module() sweep of unet_2d_conditional.py:2425-2436 for one code, then a dense forward."""
    import copy
    cfg, oracle = tiny_oracle
    st = oracle.get_structure()
    code = synthetic_codes(st, 8)[3:4]
    pruned = copy.deepcopy(oracle)
    pruned.set_structure(split_arch(code.clone(), st))
    pruned.prune()
    sample, t, ctx = G.unet_inputs(3, G.TINY_H, cfg.cross_attention_dim)
    with torch.no_grad():
        out = pruned(sample, t, ctx)
    _exact(out, "unet_pruned_code3", tol=1e-5)


# ---------------------------------------------------------------------------------------------------------------
# layers
# ---------------------------------------------------------------------------------------------------------------
def _seeded(mod, seed):
    O.seeded_init(mod, seed, 0.1)
    return mod.eval()


def test_layers_match_reference_layer_forwards():
    """Replays tests/golden/make_unet_goldens.layer_goldens with the oracle's layers (same seeds, same draw order)."""
    import copy
    lc = G.layer_cases()
    g = torch.Generator().manual_seed(21)
    B, H = lc["B"], lc["H"]
    for tag, cin, skip in (("res", lc["C_in"], None), ("res_same", lc["C_out"], None), ("res_up", lc["C_out"] + 32, 32)):
        x = torch.randn(B, cin, H, H, generator=g)
        temb = torch.randn(B, lc["temb"], generator=g)
        gate = (torch.rand(lc["bg"], lc["groups"], generator=g) > 0.4).float()
        gate[:, 0] = 1.0
        soft = torch.rand(lc["bg"], lc["groups"], generator=g) * 0.9 + 0.05
        depth = torch.tensor([0.3, 1.0])
        r1 = _seeded(O.Resnet(cin, lc["C_out"], lc["temb"], lc["groups"], 1e-5), 31)
        has2 = skip is not None or cin == lc["C_out"]
        r2 = _seeded(O.Resnet(cin, lc["C_out"], lc["temb"], lc["groups"], 1e-5, depth_gated=True, skip_dim=skip), 31) \
            if has2 else None
        for gname, gv in (("hard", gate), ("soft", soft)):
            r1.gate = gv
            with torch.no_grad():
                _exact(r1(x, temb), f"layer_{tag}_width_{gname}")
            if r2 is not None:
                r2.gate, r2.depth = gv, depth
                with torch.no_grad():
                    _exact(r2(x, temb), f"layer_{tag}_widthdepth_{gname}")
        r1.gate = gate[:1]
        r1.prune()
        with torch.no_grad():
            _exact(r1(x, temb), f"layer_{tag}_width_pruned")  # physically sliced like blocks.py:424-465
        if r2 is not None:
            for dtag, dval in (("kept", 1.0), ("dropped", 0.0)):
                r3 = _seeded(O.Resnet(cin, lc["C_out"], lc["temb"], lc["groups"], 1e-5, depth_gated=True, skip_dim=skip), 31)
                r3.gate, r3.depth = gate[:1], torch.tensor([dval])
                r3.prune()
                with torch.no_grad():
                    _exact(r3(x, temb), f"layer_{tag}_widthdepth_pruned_{dtag}")

    dim, heads, N = lc["dim"], lc["heads"], H * H
    xs = torch.randn(B, N, dim, generator=g)
    ctx = torch.randn(B, lc["n_ctx"], lc["ctx_dim"], generator=g)
    hg = torch.tensor([[1., 0., 1.], [0.5, 1., 0.25]])
    a_self = _seeded(O.Attention(dim, heads), 41)
    a_cross = _seeded(O.Attention(dim, heads, lc["ctx_dim"]), 42)
    a_self.gate = a_cross.gate = hg
    with torch.no_grad():
        _exact(a_self(xs), "layer_attn_self")
        _exact(a_cross(xs, ctx), "layer_attn_cross")
        a_self.gate = hg[:1]
        _exact(a_self(xs), "layer_attn_self_pruned", tol=1e-5)  # reference slices heads (blocks.py:153-187)
    fg = (torch.rand(lc["bg"], 32, generator=g) > 0.5).float()
    fg[:, 0] = 1.0
    ff = _seeded(O.FeedForward(dim, 32), 43)
    with torch.no_grad():
        ff.gate = fg
        _exact(ff(xs), "layer_ff_hard")
        ff.gate = torch.rand(lc["bg"], 32, generator=g)
        _exact(ff(xs), "layer_ff_soft")
        ff.gate = fg[:1]
        _exact(ff(xs), "layer_ff_pruned", tol=1e-5)               # reference slices proj rows / net.2 columns (:52-67,:121-129)
    tb = _seeded(O.BasicTransformerBlock(dim, heads, lc["ctx_dim"], 32), 44)
    tb.attn1.gate, tb.attn2.gate, tb.ff.gate = hg, hg.flip(0), fg
    with torch.no_grad():
        _exact(tb(xs, ctx), "layer_tblock")
    x4 = torch.randn(B, dim, H, H, generator=g)
    tr = _seeded(O.Transformer(dim, heads, lc["ctx_dim"], 32, 32, depth_gated=True), 45)
    t0 = tr.transformer_blocks[0]
    t0.attn1.gate, t0.attn2.gate, t0.ff.gate = hg, hg.flip(0), fg
    tr.depth = torch.tensor([0.3, 1.0])
    with torch.no_grad():
        _exact(tr(x4, ctx), "layer_transformer_lerp")
        # depth-dropped + prune_module() (blocks.py:1427-1438, :1190-1194): identity
        assert torch.equal(torch.from_numpy(GOLD["layer_transformer_dropped"]), x4)
        tr.depth = torch.tensor([0.0])
        t0.attn1.gate, t0.attn2.gate, t0.ff.gate = hg[:1], hg[:1], fg[:1]
        _exact(tr(x4, ctx), "layer_transformer_dropped")
    del copy
