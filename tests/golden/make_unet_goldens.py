"""U-Net golden vectors produced by EXECUTING THE REFERENCE'S OWN blocks.py / unet_2d_conditional.py / op_counter.py.

Run in the build container only (needs /root/reference):  python tests/golden/make_unet_goldens.py
The reference sources are executed in place on top of constructor-only stand-ins for their diffusers 0.23.1 base
classes (oracle/ref_shim/diffusers_stubs.py lists what is stubbed and what therefore stays restated); nothing is
copied. Inputs and weights are seeded (oracle.unet_oracle.seeded_init + torch.Generator), so only OUTPUTS are stored:

  tests/golden/unet_ref.npz
    whole-U-Net tiny configuration (64/128/256/256 channels, 1/2/4/4 heads, GroupNorm beta != 0):
      UNet2DConditionModelGated.forward (unet_2d_conditional.py:1415-1726) for hard mixed-expert codes, soft gates,
      CFG batch doubling, all-ones gates; the nine hooked block outputs (trainer.py:496-511) of the hard case;
      calc_macs() (unet_2d_conditional.py:2124-2163) after the reference's count_ops_and_params (op_counter.py:19);
      the physically pruned model (the prune()/prune_module() sweep of unet_2d_conditional.py:2425-2436).
    layers, each run through the reference class's own forward / prune():
      ResnetBlock2DWidthGated / WidthDepthGated (blocks.py:293-371, :482-584, prune :424-465, :641-697),
      GEGLUGated + FeedForwardWidthGated (:41-50, :70-129), GatedAttention + HeadGatedAttnProcessor2 (:132-280),
      BasicTransformerBlockWidthGated (:763-851), Transformer2DModelWidthDepthGated (:1139-1355, :1427-1438).
"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
OUT = os.path.dirname(os.path.abspath(__file__))

from oracle import unet_oracle as O  # noqa: E402
from diffusion_pruning_b200.synthetic import split_arch, synthetic_codes  # noqa: E402

TINY_H = 16
# CPU intra-op threads the goldens are recorded and checked with: PyTorch's CPU convolutions split their reductions by
# thread count, so another count sums in another order and changes the last bits of the fp32 outputs
THREADS = 8


def unet_inputs(B, H, ctx_dim, seed=1):
    g = torch.Generator().manual_seed(seed)
    sample = torch.randn(B, 4, H, H, generator=g)
    ctx = torch.randn(B, 77, ctx_dim, generator=g)
    t = torch.tensor([981, 661, 341, 21] * ((B + 3) // 4))[:B]
    return sample, t, ctx


def unet_cases(structure):
    """name -> (arch [b, dim], batch): shared by the generator and the tests."""
    codes = synthetic_codes(structure, 8)
    dim = codes.shape[1]
    g = torch.Generator().manual_seed(9)
    return {
        "hard": (codes[[0, 3, 3, 7]], 4),
        "soft": (torch.rand(3, dim, generator=g) * 0.9 + 0.05, 3),
        "cfg": (codes[[1, 5]], 4),           # gates for 2 prompts, batch [uncond; cond] (gates.py:18-19)
        "ones": (torch.ones(2, dim), 2),
    }


def build_reference_unet(ref, cfg, oracle):
    m = ref["unet"].UNet2DConditionModelGated(
        sample_size=32, block_out_channels=cfg.block_out_channels, attention_head_dim=cfg.num_heads,
        cross_attention_dim=cfg.cross_attention_dim, use_linear_projection=True, gated_ff=True, ff_gate_width=32)
    m.load_state_dict(oracle.state_dict())
    return m.eval()


def layer_cases():
    """Small shapes for the per-layer goldens (shared with the tests)."""
    return dict(C_in=64, C_out=96, temb=128, groups=32, heads=3, dim=192, ctx_dim=80, n_ctx=7, B=2, bg=2, H=6)


def _seeded(mod, seed):
    O.seeded_init(mod, seed, 0.1)
    return mod.eval()


def layer_goldens(ref):
    bl = ref["blocks"]
    lc = layer_cases()
    out = {}
    g = torch.Generator().manual_seed(21)
    B, H = lc["B"], lc["H"]

    # ---- ResNets: width gate per GroupNorm group BEFORE norm2 (blocks.py:345-348), depth lerp (:577-582) ----
    for tag, cin, skip in (("res", lc["C_in"], None), ("res_same", lc["C_out"], None), ("res_up", lc["C_out"] + 32, 32)):
        x = torch.randn(B, cin, H, H, generator=g)
        temb = torch.randn(B, lc["temb"], generator=g)
        gate = (torch.rand(lc["bg"], lc["groups"], generator=g) > 0.4).float()
        gate[:, 0] = 1.0
        soft = torch.rand(lc["bg"], lc["groups"], generator=g) * 0.9 + 0.05
        depth = torch.tensor([0.3, 1.0])
        kw = dict(in_channels=cin, out_channels=lc["C_out"], temb_channels=lc["temb"], eps=1e-5, groups=lc["groups"])
        r1 = _seeded(bl.ResnetBlock2DWidthGated(**kw), 31)
        r2 = _seeded(bl.ResnetBlock2DWidthDepthGated(skip_connection_dim=skip, is_input_concatenated=skip is not None,
                                                     **kw), 31) if (skip is not None or cin == lc["C_out"]) else None
        for gname, gv in (("hard", gate), ("soft", soft)):
            r1.gate.set_structure_value(gv)
            out[f"{tag}_width_{gname}"] = r1(x, temb).detach().numpy()
            if r2 is not None:
                r2.gate.set_structure_value(gv)
                r2.depth_gate.set_structure_value(depth)
                out[f"{tag}_widthdepth_{gname}"] = r2(x, temb).detach().numpy()
        # prune() for one code (batch-1 gates): the compacted module's forward
        r1.gate.set_structure_value(gate[:1])
        r1.prune()
        out[f"{tag}_width_pruned"] = r1(x, temb).detach().numpy()
        if r2 is not None:
            for dtag, dval in (("kept", 1.0), ("dropped", 0.0)):
                r3 = _seeded(bl.ResnetBlock2DWidthDepthGated(skip_connection_dim=skip,
                                                             is_input_concatenated=skip is not None, **kw), 31)
                r3.gate.set_structure_value(gate[:1])
                r3.depth_gate.set_structure_value(torch.tensor([dval]))
                r3.prune()
                out[f"{tag}_widthdepth_pruned_{dtag}"] = r3(x, temb).detach().numpy()

    # ---- attention (head gates on q, k, v: blocks.py:250-255), FF (both GEGLU halves gated: :45-48) ----
    dim, heads, N = lc["dim"], lc["heads"], H * H
    xs = torch.randn(B, N, dim, generator=g)
    ctx = torch.randn(B, lc["n_ctx"], lc["ctx_dim"], generator=g)
    hg = torch.tensor([[1., 0., 1.], [0.5, 1., 0.25]])
    a_self = _seeded(bl.GatedAttention(query_dim=dim, heads=heads, dim_head=64), 41)
    a_cross = _seeded(bl.GatedAttention(query_dim=dim, cross_attention_dim=lc["ctx_dim"], heads=heads, dim_head=64), 42)
    a_self.gate.set_structure_value(hg)
    a_cross.gate.set_structure_value(hg)
    out["attn_self"] = a_self(xs).detach().numpy()
    out["attn_cross"] = a_cross(xs, encoder_hidden_states=ctx).detach().numpy()
    a_self.gate.set_structure_value(hg[:1])
    a_self.prune()
    out["attn_self_pruned"] = a_self(xs).detach().numpy()
    fg = (torch.rand(lc["bg"], 32, generator=g) > 0.5).float()
    fg[:, 0] = 1.0
    ff = _seeded(bl.FeedForwardWidthGated(dim, gate_width=32), 43)
    ff.net[0].gate.set_structure_value(fg)
    out["ff_hard"] = ff(xs).detach().numpy()
    ff.net[0].gate.set_structure_value(torch.rand(lc["bg"], 32, generator=g))
    out["ff_soft"] = ff(xs).detach().numpy()
    ff.net[0].gate.set_structure_value(fg[:1])
    ff.prune()
    out["ff_pruned"] = ff(xs).detach().numpy()

    # ---- transformer block / Transformer2DModelWidthDepthGated ----
    tb = _seeded(bl.BasicTransformerBlockWidthGated(dim, heads, 64, cross_attention_dim=lc["ctx_dim"], gated_ff=True,
                                                    ff_gate_width=32), 44)
    tb.set_gate_structure({"width": [hg, hg.flip(0), fg], "depth": []})
    out["tblock"] = tb(xs, encoder_hidden_states=ctx).detach().numpy()
    x4 = torch.randn(B, dim, H, H, generator=g)
    for dtag, dv in (("lerp", torch.tensor([0.3, 1.0])),):
        tr = _seeded(bl.Transformer2DModelWidthDepthGated(heads, 64, in_channels=dim, cross_attention_dim=lc["ctx_dim"],
                                                          norm_num_groups=32, use_linear_projection=True,
                                                          gated_ff=True, ff_gate_width=32), 45)
        tr.set_gate_structure({"width": [hg, hg.flip(0), fg], "depth": [dv]})
        out[f"transformer_{dtag}"] = tr(x4, encoder_hidden_states=ctx, return_dict=False)[0].detach().numpy()
    tr.set_gate_structure({"width": [hg[:1], hg[:1], fg[:1]], "depth": [torch.tensor([0.0])]})
    tr.prune_module()
    out["transformer_dropped"] = tr(x4, encoder_hidden_states=ctx, return_dict=False)[0].detach().numpy()
    return out


def unet_goldens():
    from oracle.ref_shim.diffusers_stubs import load_unet_reference
    ref = load_unet_reference()
    assert ref["unet"] is not None, ref["unet_error"]
    torch.manual_seed(0)
    cfg = O.UNetConfig.tiny()
    oracle = O.GatedUNetOracle(cfg).eval()
    O.seeded_init(oracle, 0, 0.1)
    m = build_reference_unet(ref, cfg, oracle)
    st = m.get_structure()
    assert st == oracle.get_structure()
    out = {}
    taps = {}

    def hook(name):
        def fn(mod, inp, o):
            taps[name] = (o[0] if isinstance(o, tuple) else o).detach().numpy()
        return fn
    for name, (arch, B) in unet_cases(st).items():
        sample, t, ctx = unet_inputs(B, TINY_H, cfg.cross_attention_dim)
        m.set_structure(split_arch(arch.clone(), st))
        handles = []
        if name == "hard":
            blocks = list(m.down_blocks) + [m.mid_block] + list(m.up_blocks)
            handles = [b.register_forward_hook(hook(f"hard_tap{i}")) for i, b in enumerate(blocks)]
        with torch.no_grad():
            out[f"unet_{name}"] = m(sample, t, ctx).sample.numpy()
        for h in handles:
            h.remove()
    out.update(taps)

    # ---- MAC accounting: Pruner.count_macs sequence (trainer.py:1257-1296) on the reference's own hooks ----
    dim = sum(w for ws in st["width"] for w in ws) + sum(1 for d in st["depth"] if d == [1])
    m.set_structure(split_arch(torch.ones(1, dim), st))
    sample, t, ctx = unet_inputs(1, TINY_H, cfg.cross_attention_dim)
    macs, params = ref["op_counter"].count_ops_and_params(
        m, {"sample": sample, "timestep": t, "encoder_hidden_states": ctx})
    d1 = m.calc_macs()
    out["macs_counter_total"] = np.asarray([macs, params], dtype=np.float64)
    out["macs_ones"] = np.asarray([float(d1["total_macs"]), float(d1["prunable_macs"]),
                                   float(d1["cur_prunable_macs"]), float(d1["cur_total_macs"])], dtype=np.float64)
    codes = synthetic_codes(st, 8)
    m.set_structure(split_arch(codes.clone(), st))
    d8 = m.calc_macs()
    out["macs_codes_cur_prunable"] = d8["cur_prunable_macs"].detach().double().numpy()
    out["macs_codes_cur_total"] = d8["cur_total_macs"].detach().double().numpy()
    pm = m.get_prunable_macs()
    out["macs_prunable_list"] = np.asarray([e for elem in pm for e in elem], dtype=np.float64)

    # ---- physically pruned expert: the sweep of unet_2d_conditional.py:2425-2436 for code 3 ----
    m2 = build_reference_unet(ref, cfg, oracle)
    code = codes[3:4]
    m2.set_structure(ref["hypernet"].HyperStructure.transform_arch_vector(code.clone(), m2.get_structure()))
    for _, mod in m2.named_modules():
        if hasattr(mod, "prune"):
            mod.prune()
    for mod in m2.modules():
        if hasattr(mod, "prune_module"):
            mod.prune_module()
    sample, t, ctx = unet_inputs(3, TINY_H, cfg.cross_attention_dim)
    with torch.no_grad():
        out["unet_pruned_code3"] = m2(sample, t, ctx).sample.numpy()
    out["pruned_state_shapes"] = np.asarray(
        [list(v.shape) + [0] * (4 - v.dim()) for v in m2.state_dict().values()], dtype=np.int64)
    out["pruned_state_keys"] = np.asarray(list(m2.state_dict().keys()))

    out.update({"layer_" + k: v for k, v in layer_goldens(ref).items()})
    np.savez_compressed(os.path.join(OUT, "unet_ref.npz"), **out)
    print(f"unet goldens written: {len(out)} arrays, "
          f"{os.path.getsize(os.path.join(OUT, 'unet_ref.npz')) / 1e6:.2f} MB")


if __name__ == "__main__":
    torch.set_num_threads(THREADS)
    unet_goldens()
