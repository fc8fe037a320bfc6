"""CPU oracle of the APTP gated SD-2.1 U-Net -- TEST INFRASTRUCTURE, not product code.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may import
this module; the product path (diffusion_pruning_b200/) never does.

It is a plain-PyTorch fp32 restatement of the reference forward. The gating logic follows the
reference file by file (citations below, relative to /root/reference); the generic U-Net arithmetic
the reference inherits from diffusers 0.23.1 (env.yaml:114 -- NOT vendored, NOT installed here) is
restated from that version's published behaviour (SURVEY.md Appendix B).

Pinning status (round 2): PINNED to reference-executed code except for the stubbed diffusers base classes.
The reference ships no tests or golden vectors (SURVEY.md section 4), and diffusers 0.23.1 is absent, but the gating
arithmetic is written out in the reference's own files. tests/golden/make_unet_goldens.py executes
pdm/models/unet/blocks.py, pdm/models/unet/unet_2d_conditional.py and pdm/utils/op_counter.py IN PLACE on top of
constructor-only stand-ins for their diffusers base classes (oracle/ref_shim/diffusers_stubs.py) and records
  * UNet2DConditionModelGated.forward (unet_2d_conditional.py:1415-1726) on a tiny configuration: hard mixed-expert
    codes, soft gates, CFG batch doubling, all-ones gates, the nine hooked block outputs, GroupNorm beta != 0;
  * every gated layer's own forward and prune(): blocks.py:41-50, :70-129, :132-280, :293-371, :424-465, :482-584,
    :641-697, :763-851, :1139-1355, :1427-1438, and the prune sweep of unet_2d_conditional.py:2425-2436;
  * count_ops_and_params + calc_macs (op_counter.py:19-116, :259-306; unet_2d_conditional.py:2124-2163);
tests/test_oracle_unet_pinned.py holds this file to those outputs bit-for-bit in fp32 (<= 1e-5 where the reference
slices weights and this file keeps exact-zero gates).
Still restated, hence the only unpinned arithmetic: what the stubs themselves implement -- the container loops the
reference inherits (resnet -> attention order, skip concatenation, samplers), Transformer2DModel.forward of the
width-only variant, Downsample2D / Upsample2D, Timesteps / TimestepEmbedding, GEGLU.gelu, and PyTorch 2.11 (not 2.1.0)
as the executor of conv / group_norm / SDPA. Structure is additionally pinned by the public SD-2.1 parameter count
865,910,724, the diffusers state-dict key names and the reference's gate layout 70 / 1606 / 14
(tests/test_oracle_unet_cpu.py).
"""
from __future__ import annotations

import math
from dataclasses import dataclass, field
from typing import Dict, List, Optional, Sequence, Tuple

import torch
import torch.nn as nn
import torch.nn.functional as F


@dataclass
class UNetConfig:
    """SD-2.1 layout by default (configs/pruning/sd-2-1_cc3m.yaml:11-26 + the SD-2.1 unet config)."""
    in_channels: int = 4
    out_channels: int = 4
    block_out_channels: Tuple[int, ...] = (320, 640, 1280, 1280)
    num_heads: Tuple[int, ...] = (5, 10, 20, 20)  # SD-2.1 `attention_head_dim` (really heads per block)
    layers_per_block: int = 2
    cross_attention_dim: int = 1024
    norm_num_groups: int = 32
    norm_eps: float = 1e-5
    ff_gate_width: int = 32
    # which down blocks carry transformers (CrossAttnDownBlock2DHalfGated) -- last one is DownBlock2DHalfGated
    down_has_attn: Tuple[bool, ...] = (True, True, True, False)

    @property
    def time_embed_dim(self) -> int:
        return self.block_out_channels[0] * 4

    @property
    def up_has_attn(self) -> Tuple[bool, ...]:
        return tuple(reversed(self.down_has_attn))

    @staticmethod
    def tiny() -> "UNetConfig":
        return UNetConfig(block_out_channels=(64, 128, 256, 256), num_heads=(1, 2, 4, 4), cross_attention_dim=128)


def hard_concrete(x: torch.Tensor) -> torch.Tensor:
    """pdm/utils/estimation_utils.py:67-75 (forward value: exact 0/1; straight-through gradient)."""
    hard = (x >= 0.5).to(x.dtype)
    return (hard - x).detach() + x


# ------------------------------------------------------------------------------------------------
# gates -- pdm/models/unet/gates.py
# ------------------------------------------------------------------------------------------------
def width_gate(x: torch.Tensor, g: torch.Tensor) -> torch.Tensor:
    """WidthGate.forward (gates.py:15-21): x [B,C,...], g [b,width]; CFG batch doubling via repeat."""
    mask = g.repeat_interleave(x.shape[1] // g.shape[1], dim=1).unsqueeze(-1).unsqueeze(-1)
    if mask.shape[0] != x.shape[0]:
        mask = mask.repeat(x.shape[0] // mask.shape[0], 1, 1, 1)
    return mask.expand_as(x) * x


def linear_width_gate(x: torch.Tensor, g: torch.Tensor) -> torch.Tensor:
    """LinearWidthGate.forward (gates.py:49-55): x [B,N,C]."""
    mask = g.repeat_interleave(x.shape[-1] // g.shape[1], dim=1).unsqueeze(1)
    if mask.shape[0] != x.shape[0]:
        mask = mask.repeat(x.shape[0] // mask.shape[0], 1, 1)
    return mask.expand_as(x) * x


def depth_gate(x_in: torch.Tensor, y: torch.Tensor, d: torch.Tensor) -> torch.Tensor:
    """DepthGate.forward (gates.py:36-42): d [b]."""
    mask = d.unsqueeze(-1).unsqueeze(-1).unsqueeze(-1)
    if mask.shape[0] != y.shape[0]:
        mask = mask.repeat(y.shape[0] // mask.shape[0], 1, 1, 1)
    return (1 - mask) * x_in + mask * y


# ------------------------------------------------------------------------------------------------
# layers (diffusers 0.23.1 module / key names)
# ------------------------------------------------------------------------------------------------
class Resnet(nn.Module):
    """ResnetBlock2DWidthGated / ...WidthDepthGated (blocks.py:283-371, :468-584)."""

    def __init__(self, cin, cout, temb, groups, eps, depth_gated=False, skip_dim=None):
        super().__init__()
        self.norm1 = nn.GroupNorm(groups, cin, eps=eps)
        self.conv1 = nn.Conv2d(cin, cout, 3, padding=1)
        self.time_emb_proj = nn.Linear(temb, cout)
        self.norm2 = nn.GroupNorm(groups, cout, eps=eps)
        self.conv2 = nn.Conv2d(cout, cout, 3, padding=1)
        self.conv_shortcut = nn.Conv2d(cin, cout, 1) if cin != cout else None
        self.cin, self.cout, self.groups = cin, cout, groups
        self.depth_gated, self.skip_dim = depth_gated, skip_dim
        self.gate = torch.ones(1, groups)
        self.depth = torch.ones(1)
        self.pruned = self.dropped = False

    def widths(self):
        return [self.groups]

    @torch.no_grad()
    def prune(self):
        """Physical compaction for ONE code (blocks.py:424-465; depth-gated variant :641-697): conv1 rows, the
        time-embedding rows, norm2 (kept groups only) and conv2 input columns are sliced by the kept GroupNorm
        groups; a depth-dropped block becomes the identity on its (non-skip) input."""
        assert self.gate.shape[0] == 1 and self.depth.shape[0] == 1, "Pruning is only supported for single batch size"
        if self.depth_gated and float(self.depth[0]) < 0.5:
            self.dropped = True
            return
        keep_g = self.gate[0] >= 0.5
        gs = self.cout // self.groups
        keep = keep_g.repeat_interleave(gs)
        n = int(keep.sum())
        conv1 = nn.Conv2d(self.cin, n, 3, padding=1)
        conv1.weight.data, conv1.bias.data = self.conv1.weight.data[keep].clone(), self.conv1.bias.data[keep].clone()
        tproj = nn.Linear(self.time_emb_proj.in_features, n)
        tproj.weight.data, tproj.bias.data = (self.time_emb_proj.weight.data[keep].clone(),
                                              self.time_emb_proj.bias.data[keep].clone())
        norm2 = nn.GroupNorm(int(keep_g.sum()), n, eps=self.norm2.eps)
        norm2.weight.data, norm2.bias.data = self.norm2.weight.data[keep].clone(), self.norm2.bias.data[keep].clone()
        conv2 = nn.Conv2d(n, self.cout, 3, padding=1)
        conv2.weight.data, conv2.bias.data = self.conv2.weight.data[:, keep].clone(), self.conv2.bias.data.clone()
        self.conv1, self.time_emb_proj, self.norm2, self.conv2 = conv1, tproj, norm2, conv2
        self.pruned = True

    def forward(self, x, temb):
        # blocks.py:485-495: depth-gate input is the non-skip part of the concatenated up-block input
        x_in = x[:, : x.shape[1] - self.skip_dim] if (self.depth_gated and self.skip_dim) else x
        if self.dropped:  # blocks.py:497-498
            return x_in
        h = F.silu(self.norm1(x))
        h = self.conv1(h)
        h = h + self.time_emb_proj(F.silu(temb))[:, :, None, None]
        if not self.pruned:
            h = width_gate(h, self.gate)  # blocks.py:345-348 -- BEFORE norm2
        h = F.silu(self.norm2(h))
        h = self.conv2(h)
        sc = self.conv_shortcut(x) if self.conv_shortcut is not None else x
        out = sc + h  # output_scale_factor = 1
        if self.depth_gated and not self.pruned:
            out = depth_gate(x_in, out, self.depth)  # blocks.py:577-582
        return out

    def macs(self, hw_in: int, hw: int) -> Tuple[float, float]:
        """(prunable, total) following blocks.py:384-416 with op_counter hook formulas."""
        conv1 = 9 * self.cin * self.cout * hw + self.cout * hw
        tproj = self.time_emb_proj.in_features * self.cout + self.cout
        norm2 = 2 * self.cout * hw
        conv2 = 9 * self.cout * self.cout * hw + self.cout * hw
        prunable = conv1 + tproj + norm2 + conv2
        total = prunable + 2 * self.cin * hw
        if self.conv_shortcut is not None:
            total += self.cin * self.cout * hw + self.cout * hw
        return float(prunable), float(total)


class Attention(nn.Module):
    """GatedAttention + HeadGatedAttnProcessor2 (blocks.py:132-142, :194-280)."""

    def __init__(self, dim, heads, ctx_dim=None):
        super().__init__()
        self.to_q = nn.Linear(dim, dim, bias=False)
        self.to_k = nn.Linear(ctx_dim or dim, dim, bias=False)
        self.to_v = nn.Linear(ctx_dim or dim, dim, bias=False)
        self.to_out = nn.ModuleList([nn.Linear(dim, dim), nn.Dropout(0.0)])
        self.heads, self.dim = heads, dim
        self.gate = torch.ones(1, heads)

    def forward(self, x, ctx=None):
        B = x.shape[0]
        ctx = x if ctx is None else ctx
        hd = self.dim // self.heads
        q = self.to_q(x).view(B, -1, self.heads, hd).transpose(1, 2)
        k = self.to_k(ctx).view(B, -1, self.heads, hd).transpose(1, 2)
        v = self.to_v(ctx).view(B, -1, self.heads, hd).transpose(1, 2)
        q, k, v = width_gate(q, self.gate), width_gate(k, self.gate), width_gate(v, self.gate)  # blocks.py:250-255
        o = F.scaled_dot_product_attention(q, k, v)
        o = o.transpose(1, 2).reshape(B, -1, self.dim)
        return self.to_out[0](o)

    def macs(self, n_q: int, n_ctx: int, ctx_dim: int) -> float:
        """op_counter.py:259-306: seq_len is the *query* length for self AND cross attention."""
        lin = lambda n, i, o, bias: n * i * o + (o if bias else 0)
        hd = self.dim // self.heads
        m = lin(n_q, self.dim, self.dim, False) + 2 * lin(n_ctx, ctx_dim, self.dim, False)
        m += self.heads * (2 * n_q * n_q * hd + n_q * n_q)
        m += lin(n_q, self.dim, self.dim, True)
        return float(m)


class GEGLU(nn.Module):
    def __init__(self, dim, inner):
        super().__init__()
        self.proj = nn.Linear(dim, inner * 2)


class FeedForward(nn.Module):
    """FeedForwardWidthGated with GEGLUGated (blocks.py:24-50, :70-101)."""

    def __init__(self, dim, gate_width):
        super().__init__()
        self.net = nn.ModuleList([GEGLU(dim, dim * 4), nn.Dropout(0.0), nn.Linear(dim * 4, dim)])
        self.gate = torch.ones(1, gate_width)
        self.dim = dim

    def forward(self, x):
        h, g = self.net[0].proj(x).chunk(2, dim=-1)
        h, g = linear_width_gate(h, self.gate), linear_width_gate(g, self.gate)  # blocks.py:45-48
        return self.net[2](h * F.gelu(g))

    def macs(self, n: int) -> float:
        d = self.dim
        return float(n * d * 8 * d + 8 * d + n * 4 * d * d + d)


class BasicTransformerBlock(nn.Module):
    """BasicTransformerBlockWidthGated.forward (blocks.py:763-851)."""

    def __init__(self, dim, heads, ctx_dim, gate_width):
        super().__init__()
        self.norm1 = nn.LayerNorm(dim)
        self.attn1 = Attention(dim, heads)
        self.norm2 = nn.LayerNorm(dim)
        self.attn2 = Attention(dim, heads, ctx_dim)
        self.norm3 = nn.LayerNorm(dim)
        self.ff = FeedForward(dim, gate_width)

    def forward(self, x, ctx):
        x = self.attn1(self.norm1(x)) + x
        x = self.attn2(self.norm2(x), ctx) + x
        x = self.ff(self.norm3(x)) + x
        return x


class Transformer(nn.Module):
    """Transformer2DModelWidthGated / ...WidthDepthGated (blocks.py:941-1068, :1070-1438), continuous
    input, use_linear_projection=True, GroupNorm eps 1e-6."""

    def __init__(self, dim, heads, ctx_dim, groups, gate_width, depth_gated=False):
        super().__init__()
        self.norm = nn.GroupNorm(groups, dim, eps=1e-6)
        self.proj_in = nn.Linear(dim, dim)
        self.transformer_blocks = nn.ModuleList([BasicTransformerBlock(dim, heads, ctx_dim, gate_width)])
        self.proj_out = nn.Linear(dim, dim)
        self.dim, self.heads, self.ctx_dim, self.gate_width = dim, heads, ctx_dim, gate_width
        self.depth_gated = depth_gated
        self.depth = torch.ones(1)

    def widths(self):
        return [self.heads, self.heads, self.gate_width]  # blocks.py:853-859

    def forward(self, x, ctx):
        B, C, H, W = x.shape
        h = self.norm(x)
        h = h.permute(0, 2, 3, 1).reshape(B, H * W, C)
        h = self.proj_in(h)
        for blk in self.transformer_blocks:
            h = blk(h, ctx)
        h = self.proj_out(h)
        h = h.reshape(B, H, W, C).permute(0, 3, 1, 2).contiguous()
        out = h + x
        if self.depth_gated:
            out = depth_gate(x, out, self.depth)  # blocks.py:1345-1348
        return out

    def macs(self, hw: int, n_ctx: int) -> Dict[str, float]:
        tb = self.transformer_blocks[0]
        d = self.dim
        a1 = tb.attn1.macs(hw, hw, d)
        a2 = tb.attn2.macs(hw, n_ctx, self.ctx_dim)
        ff = tb.ff.macs(hw)
        fixed = 2 * d * hw + 2 * (hw * d * d + d) + 3 * hw * d  # GN + proj_in/out + 3 LN
        return {"attn1": a1, "attn2": a2, "ff": ff, "fixed": float(fixed)}


class Downsample(nn.Module):
    def __init__(self, c):
        super().__init__()
        self.conv = nn.Conv2d(c, c, 3, stride=2, padding=1)

    def forward(self, x):
        return self.conv(x)


class Upsample(nn.Module):
    def __init__(self, c):
        super().__init__()
        self.conv = nn.Conv2d(c, c, 3, padding=1)

    def forward(self, x):
        return self.conv(F.interpolate(x, scale_factor=2.0, mode="nearest"))


class DownBlock(nn.Module):
    """CrossAttnDownBlock2DWidthHalfDepthGated / DownBlock2DWidthHalfDepthGated (blocks.py:1677-1909,
    :2290-2416): first n-1 layers width gated, last width+depth gated; forward inherited from diffusers."""

    def __init__(self, cfg: UNetConfig, cin, cout, heads, has_attn, add_down):
        super().__init__()
        n = cfg.layers_per_block
        self.resnets = nn.ModuleList([
            Resnet(cin if i == 0 else cout, cout, cfg.time_embed_dim, cfg.norm_num_groups, cfg.norm_eps,
                   depth_gated=(i == n - 1)) for i in range(n)])
        self.attentions = nn.ModuleList([
            Transformer(cout, heads, cfg.cross_attention_dim, cfg.norm_num_groups, cfg.ff_gate_width,
                        depth_gated=(i == n - 1)) for i in range(n)]) if has_attn else None
        self.downsamplers = nn.ModuleList([Downsample(cout)]) if add_down else None

    def forward(self, x, temb, ctx):
        outs = ()
        for i, r in enumerate(self.resnets):
            x = r(x, temb)
            if self.attentions is not None:
                x = self.attentions[i](x, ctx)
            outs += (x,)
        if self.downsamplers is not None:
            x = self.downsamplers[0](x)
            outs += (x,)
        return x, outs


class MidBlock(nn.Module):
    """UNetMidBlock2DCrossAttnWidthGated (blocks.py:2554-2736): width gates only."""

    def __init__(self, cfg: UNetConfig, c, heads):
        super().__init__()
        self.resnets = nn.ModuleList([Resnet(c, c, cfg.time_embed_dim, cfg.norm_num_groups, cfg.norm_eps) for _ in range(2)])
        self.attentions = nn.ModuleList([Transformer(c, heads, cfg.cross_attention_dim, cfg.norm_num_groups, cfg.ff_gate_width)])

    def forward(self, x, temb, ctx):
        x = self.resnets[0](x, temb)
        x = self.attentions[0](x, ctx)
        x = self.resnets[1](x, temb)
        return x


class UpBlock(nn.Module):
    """CrossAttnUpBlock2DWidthHalfDepthGated / UpBlock2DWidthHalfDepthGated (blocks.py:2004-2243, :2419-2550)."""

    def __init__(self, cfg: UNetConfig, cin, cout, prev, heads, has_attn, add_up):
        super().__init__()
        n = cfg.layers_per_block + 1
        res = []
        for i in range(n):
            skip = cin if i == n - 1 else cout
            rin = prev if i == 0 else cout
            res.append(Resnet(rin + skip, cout, cfg.time_embed_dim, cfg.norm_num_groups, cfg.norm_eps,
                              depth_gated=(i == n - 1), skip_dim=skip if i == n - 1 else None))
        self.resnets = nn.ModuleList(res)
        self.attentions = nn.ModuleList([
            Transformer(cout, heads, cfg.cross_attention_dim, cfg.norm_num_groups, cfg.ff_gate_width,
                        depth_gated=(i == n - 1)) for i in range(n)]) if has_attn else None
        self.upsamplers = nn.ModuleList([Upsample(cout)]) if add_up else None

    def forward(self, x, skips: List[torch.Tensor], temb, ctx):
        for i, r in enumerate(self.resnets):
            x = torch.cat([x, skips.pop()], dim=1)
            x = r(x, temb)
            if self.attentions is not None:
                x = self.attentions[i](x, ctx)
        if self.upsamplers is not None:
            x = self.upsamplers[0](x)
        return x


class TimestepEmbedding(nn.Module):
    def __init__(self, cin, dim):
        super().__init__()
        self.linear_1 = nn.Linear(cin, dim)
        self.linear_2 = nn.Linear(dim, dim)

    def forward(self, x):
        return self.linear_2(F.silu(self.linear_1(x)))


def timestep_sinusoid(t: torch.Tensor, dim: int) -> torch.Tensor:
    """diffusers Timesteps(dim, flip_sin_to_cos=True, downscale_freq_shift=0)."""
    half = dim // 2
    freqs = torch.exp(-math.log(10000.0) * torch.arange(half, dtype=torch.float32, device=t.device) / half)
    arg = t.float()[:, None] * freqs[None]
    return torch.cat([torch.cos(arg), torch.sin(arg)], dim=-1)


class GatedUNetOracle(nn.Module):
    """UNet2DConditionModelGated (pdm/models/unet/unet_2d_conditional.py:628-2181) restated."""

    def __init__(self, cfg: Optional[UNetConfig] = None):
        super().__init__()
        cfg = cfg or UNetConfig()
        self.cfg = cfg
        ch = cfg.block_out_channels
        self.conv_in = nn.Conv2d(cfg.in_channels, ch[0], 3, padding=1)
        self.time_embedding = TimestepEmbedding(ch[0], cfg.time_embed_dim)
        downs, out_c = [], ch[0]
        for i, c in enumerate(ch):
            in_c, out_c = out_c, c
            downs.append(DownBlock(cfg, in_c, out_c, cfg.num_heads[i], cfg.down_has_attn[i], add_down=i < len(ch) - 1))
        self.down_blocks = nn.ModuleList(downs)
        self.mid_block = MidBlock(cfg, ch[-1], cfg.num_heads[-1])
        rev, rev_heads = list(reversed(ch)), list(reversed(cfg.num_heads))
        ups, out_c = [], rev[0]
        for i in range(len(ch)):
            prev, out_c = out_c, rev[i]
            in_c = rev[min(i + 1, len(ch) - 1)]
            ups.append(UpBlock(cfg, in_c, out_c, prev, rev_heads[i], cfg.up_has_attn[i], add_up=i < len(ch) - 1))
        self.up_blocks = nn.ModuleList(ups)
        self.conv_norm_out = nn.GroupNorm(cfg.norm_num_groups, ch[0], eps=cfg.norm_eps)
        self.conv_out = nn.Conv2d(ch[0], cfg.out_channels, 3, padding=1)
        self.resource_info = None

    # ---- gate plumbing: resnets-then-attentions order per block (blocks.py:1814-1861) ----
    def gated_modules(self) -> List[nn.Module]:
        mods = []
        for blk in list(self.down_blocks) + [self.mid_block] + list(self.up_blocks):
            mods += list(blk.resnets)
            if blk.attentions is not None:
                mods += list(blk.attentions)
        return mods

    def get_structure(self) -> Dict[str, List[List[int]]]:
        """unet_2d_conditional.py:1332-1363."""
        mods = self.gated_modules()
        return {"width": [m.widths() for m in mods],
                "depth": [[1] if m.depth_gated else [0] for m in mods]}

    def set_structure(self, arch: Dict[str, List[torch.Tensor]]) -> None:
        """unet_2d_conditional.py:1365-1413 (pops from the caller's lists, like the reference)."""
        width, depth = arch["width"], arch["depth"]
        for blk in list(self.down_blocks) + [self.mid_block] + list(self.up_blocks):
            mods = list(blk.resnets) + (list(blk.attentions) if blk.attentions is not None else [])
            w_take = [[width.pop(0) for _ in m.widths()] for m in mods]
            d_take = [depth.pop(0) if m.depth_gated else None for m in mods]
            for m, ws, d in zip(mods, w_take, d_take):
                if isinstance(m, Resnet):
                    assert ws[0].shape[1] == m.groups
                    m.gate = ws[0]
                else:
                    tb = m.transformer_blocks[0]
                    tb.attn1.gate, tb.attn2.gate, tb.ff.gate = ws
                if d is not None:
                    m.depth = d

    @torch.no_grad()
    def prune(self) -> None:
        """UNet2DConditionModelPruned.from_pretrained (unet_2d_conditional.py:2425-2436) for the code currently set
        with batch-1 hard gates: ResNets are compacted physically (Resnet.prune). Attention heads, FF groups and
        depth-dropped transformers keep their (hard) gates: gating there yields exact zeros, so it equals the
        reference's slicing (blocks.py:52-67, :121-129, :153-187, :1427-1438) bit for bit in fp32."""
        for m in self.modules():
            if isinstance(m, Resnet):
                m.prune()

    def set_all_ones(self, batch: int = 1) -> None:
        st = self.get_structure()
        self.set_structure({"width": [torch.ones(batch, w) for ws in st["width"] for w in ws],
                            "depth": [torch.ones(batch) for d in st["depth"] if d == [1]]})

    # ---- forward: unet_2d_conditional.py:1415-1726 ----
    def forward(self, sample, timestep, encoder_hidden_states, return_blocks: bool = False):
        t = timestep.expand(sample.shape[0]) if timestep.ndim else timestep[None].expand(sample.shape[0])
        temb = self.time_embedding(timestep_sinusoid(t, self.cfg.block_out_channels[0]).to(sample.dtype))
        x = self.conv_in(sample)
        skips, taps = [x], []
        for blk in self.down_blocks:
            x, outs = blk(x, temb, encoder_hidden_states)
            skips += list(outs)
            taps.append(x)
        x = self.mid_block(x, temb, encoder_hidden_states)
        taps.append(x)
        for blk in self.up_blocks:
            x = blk(x, skips, temb, encoder_hidden_states)
            taps.append(x)
        x = self.conv_out(F.silu(self.conv_norm_out(x)))
        return (x, taps) if return_blocks else x

    # ---- MAC accounting: unet_2d_conditional.py:2124-2163 and SURVEY Appendix F ----
    def count_macs(self, H: int, W: int, n_ctx: int = 77) -> None:
        """Closed form of Pruner.count_macs (trainer.py:1257-1296): per-sample constants at latent HxW."""
        info = []
        h, w = H, W
        ch = self.cfg.block_out_channels
        fixed_total = 0.0
        te = self.time_embedding
        fixed_total += te.linear_1.in_features * te.linear_1.out_features + te.linear_1.out_features
        fixed_total += 2 * te.linear_1.out_features
        fixed_total += te.linear_2.in_features * te.linear_2.out_features + te.linear_2.out_features
        fixed_total += 9 * self.cfg.in_channels * ch[0] * h * w + ch[0] * h * w  # conv_in
        for blk in self.down_blocks:
            hw = h * w
            for i, r in enumerate(blk.resnets):
                info.append(("res", r, r.macs(hw, hw)))
                if blk.attentions is not None:
                    pass
            if blk.attentions is not None:
                for a in blk.attentions:
                    info.append(("attn", a, a.macs(hw, n_ctx)))
            if blk.downsamplers is not None:
                h, w = h // 2, w // 2
                c = blk.downsamplers[0].conv.in_channels
                fixed_total += 9 * c * c * h * w + c * h * w
        hw = h * w
        mb = self.mid_block
        info.append(("res", mb.resnets[0], mb.resnets[0].macs(hw, hw)))
        info.append(("res", mb.resnets[1], mb.resnets[1].macs(hw, hw)))
        info.append(("attn", mb.attentions[0], mb.attentions[0].macs(hw, n_ctx)))
        for blk in self.up_blocks:
            hw = h * w
            for r in blk.resnets:
                info.append(("res", r, r.macs(hw, hw)))
            if blk.attentions is not None:
                for a in blk.attentions:
                    info.append(("attn", a, a.macs(hw, n_ctx)))
            if blk.upsamplers is not None:
                h, w = h * 2, w * 2
                c = blk.upsamplers[0].conv.in_channels
                fixed_total += 9 * c * c * h * w + c * h * w
        fixed_total += 2 * ch[0] * h * w + 2 * ch[0] * h * w  # conv_norm_out + conv_act (SiLU hook: 2*numel)
        fixed_total += 9 * ch[0] * self.cfg.out_channels * h * w + self.cfg.out_channels * h * w
        self.resource_info = (info, float(fixed_total))

    def calc_macs(self) -> Dict[str, object]:
        assert self.resource_info is not None, "call count_macs(H, W) first"
        info, fixed_total = self.resource_info
        total, prunable = fixed_total, 0.0
        cur_p, cur_t = 0.0, fixed_total
        ratio = lambda g: hard_concrete(g).sum(dim=1, keepdim=True) / g.shape[1]
        for kind, m, mm in info:
            if kind == "res":
                P, T = mm
                r = ratio(m.gate)
                cp = r * P
                ct = r.detach() * P + (T - P)
                if m.depth_gated:
                    d = hard_concrete(m.depth).unsqueeze(1)
                    cp = (r * P + (T - P)) * d  # blocks.py:630-633
                    ct = ct * d.detach()
            else:
                tb = m.transformer_blocks[0]
                P = mm["attn1"] + mm["attn2"] + mm["ff"]
                T = P + mm["fixed"]
                r1, r2, rf = ratio(tb.attn1.gate), ratio(tb.attn2.gate), ratio(tb.ff.gate)
                cp = r1 * mm["attn1"] + r2 * mm["attn2"] + rf * mm["ff"]
                ct = (r1.detach() * mm["attn1"] + r2.detach() * mm["attn2"] + rf.detach() * mm["ff"]) + mm["fixed"]
                if m.depth_gated:
                    d = hard_concrete(m.depth).unsqueeze(1)
                    cp = (cp + T - P) * d  # blocks.py:1409-1411
                    ct = ct * d.detach()
            total += T
            prunable += P
            cur_p = cur_p + cp
            cur_t = cur_t + ct
        return {"total_macs": total, "prunable_macs": prunable, "cur_prunable_macs": cur_p, "cur_total_macs": cur_t}


def seeded_init(model: nn.Module, seed: int = 0, beta_std: float = 0.0) -> None:
    """Deterministic synthetic weights (there are no checkpoints offline): every tensor is filled from
    its own generator seeded by (seed, parameter index), fan-in scaled so activations stay O(1).
    beta_std > 0 gives GroupNorm/LayerNorm biases a non-zero spread (exercises SURVEY Appendix D-1)."""
    with torch.no_grad():
        for idx, (name, p) in enumerate(model.named_parameters()):
            g = torch.Generator().manual_seed(seed * 100003 + idx)
            if p.ndim >= 2:
                fan_in = p[0].numel()
                p.copy_(torch.randn(p.shape, generator=g) * (1.0 / math.sqrt(fan_in)))
            elif "norm" in name and name.endswith("weight"):
                p.copy_(1.0 + 0.1 * torch.randn(p.shape, generator=g))
            elif "norm" in name and name.endswith("bias"):
                p.copy_(beta_std * torch.randn(p.shape, generator=g))
            else:
                p.copy_(0.02 * torch.randn(p.shape, generator=g))
