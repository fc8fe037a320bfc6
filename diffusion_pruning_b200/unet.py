"""Drop-in `UNet2DConditionModelGated` whose forward runs on the hand-written sm_100a kernels.

Mirrors the reference interface (pdm/models/unet/unet_2d_conditional.py:628): same constructor
vocabulary for the shipped SD-2.1 layout, same module tree / state-dict keys as the diffusers SD-2.1
U-Net (gates add no parameters, pdm/models/unet/gates.py:13), same `get_structure` /
`set_structure` / `calc_macs` / `freeze` / `forward(sample, timestep, encoder_hidden_states)`.

Execution model (B200-first, not a translation of the module-by-module eager reference):
  * activations live in NHWC / token-major bf16, so 3x3 conv (implicit GEMM over shifted TMA boxes),
    1x1 conv, Linear and the transformer's [B, HW, C] view share one layout -- no permute copies;
  * hard (0/1) gates: samples are bucketed by architecture code and every prunable layer runs a
    grouped tcgen05 GEMM over per-expert *compacted* weights -- pruned channels / heads / FF groups and
    depth-dropped blocks are skipped, not multiplied by zero;
  * soft gates (training-mode codes): dense weights, gate multipliers fused into the GroupNorm pass
    and the GEMM epilogues, depth gate as one lerp kernel;
  * the nn.Module tree below only owns parameters and fires forward hooks; arithmetic happens in
    libaptp_sm100.so through diffusion_pruning_b200.kernels (no eager / CPU fallback exists).
"""
from __future__ import annotations

import contextlib
import gc
import os

import math
from collections import OrderedDict
from dataclasses import dataclass
from typing import Any, Dict, List, Optional, Sequence, Tuple

import numpy as np
import torch
import torch.nn as nn

from . import kernels as K
from . import plan as P
from ._lib import (A_CONV3X3, A_CONV3X3_S2, A_LINEAR, EPI_GEGLU, EPI_RES_F32, EPI_SILU, OUT_BF16, OUT_F32,
                   OUT_F32_NCHW)

BF16 = torch.bfloat16


@dataclass
class UNet2DConditionOutput:
    sample: torch.Tensor


@contextlib.contextmanager
def _graph_capture(g):
    """torch.cuda.graph(g) with Python's cyclic garbage collector held off for the capture. A collection inside the
    capture can free an unreachable model whose engine holds captured graphs; destroying a graph is not permitted while
    a (global-mode) capture is open, so it would invalidate this capture. The garbage is collected after the capture."""
    enabled = gc.isenabled()
    gc.disable()
    try:
        with torch.cuda.graph(g):
            yield
    finally:
        if enabled:
            gc.enable()


def _require_cuda(sample: torch.Tensor) -> None:
    if not sample.is_cuda:
        raise RuntimeError("UNet2DConditionModelGated runs on the sm_100a CUDA path only: move the model and "
                           "inputs to a CUDA device (there is no CPU fallback)")


class FrozenConfig(dict):
    """`unet.config` as the reference's callers use it: attribute access (`unet.config.sample_size`,
    pruning_pipelines.py:708, :772; trainer.py:1440) and item access, like diffusers' FrozenDict."""

    def __getattr__(self, k):
        try:
            return self[k]
        except KeyError as e:
            raise AttributeError(k) from e

    def __setattr__(self, k, v):
        raise AttributeError("the model config is read-only; use register_to_config(**kwargs)")


# diffusers UNet2DConditionModel config keys whose only supported value(s) on this path are listed; anything else raises
# instead of being silently ignored. Keys not listed here and not consumed by the constructor are kept verbatim in
# `config` (and written back by save_pretrained): they do not change the arithmetic of the SD-2.1 layout.
_ONLY_SUPPORTED = {
    "act_fn": ("silu", "swish"), "center_input_sample": (False,), "dual_cross_attention": (False,),
    "flip_sin_to_cos": (True,), "freq_shift": (0,), "downsample_padding": (1,), "mid_block_scale_factor": (1, 1.0),
    "only_cross_attention": (False,), "num_class_embeds": (None,), "class_embed_type": (None,),
    "addition_embed_type": (None,), "addition_time_embed_dim": (None,), "time_embedding_type": ("positional",),
    "time_embedding_dim": (None,), "time_embedding_act_fn": (None,), "timestep_post_act": (None,),
    "time_cond_proj_dim": (None,), "resnet_time_scale_shift": ("default",), "resnet_skip_time_act": (False,),
    "resnet_out_scale_factor": (1, 1.0), "encoder_hid_dim": (None,), "encoder_hid_dim_type": (None,),
    "transformer_layers_per_block": (1,), "conv_in_kernel": (3,), "conv_out_kernel": (3,),
    "projection_class_embeddings_input_dim": (None,), "attention_type": ("default",),
    "class_embeddings_concat": (False,), "mid_block_only_cross_attention": (None,), "cross_attention_norm": (None,),
    "dropout": (0, 0.0), "num_attention_heads": (None,), "use_linear_projection": (True,),
}


# --------------------------------------------------------------------------------------------------
# parameter containers (diffusers SD-2.1 names; their forward() is never used for arithmetic)
# --------------------------------------------------------------------------------------------------
class _Gate:
    """VirtualGate state (gates.py:9-24): a plain tensor attribute, not a parameter."""

    def __init__(self, width: int):
        self.width = width
        self.gate_f = torch.ones(1, width)

    def set_structure_value(self, value: torch.Tensor) -> None:
        self.gate_f = value


class ResnetBlock2DWidthGated(nn.Module):
    """Parameters of blocks.py:283 / :468 (depth_gated=True)."""

    def __init__(self, cin, cout, temb, groups, eps, depth_gated=False, skip_dim=None):
        super().__init__()
        self.norm1 = nn.GroupNorm(groups, cin, eps=eps)
        self.conv1 = nn.Conv2d(cin, cout, 3, padding=1)
        self.time_emb_proj = nn.Linear(temb, cout)
        self.norm2 = nn.GroupNorm(groups, cout, eps=eps)
        self.conv2 = nn.Conv2d(cout, cout, 3, padding=1)
        self.conv_shortcut = nn.Conv2d(cin, cout, 1) if cin != cout else None
        self.cin, self.cout, self.groups, self.eps = cin, cout, groups, eps
        self.gate = _Gate(groups)
        self.depth_gate = _Gate(1) if depth_gated else None
        self.skip_connection_dim = skip_dim
        self.uid = ""

    def gate_widths(self):
        return [self.groups]


class _Attention(nn.Module):
    def __init__(self, dim, heads, ctx_dim=None):
        super().__init__()
        self.to_q = nn.Linear(dim, dim, bias=False)
        self.to_k = nn.Linear(ctx_dim or dim, dim, bias=False)
        self.to_v = nn.Linear(ctx_dim or dim, dim, bias=False)
        self.to_out = nn.ModuleList([nn.Linear(dim, dim), nn.Dropout(0.0)])
        self.heads, self.dim, self.ctx_dim = heads, dim, ctx_dim
        self.gate = _Gate(heads)


class _GEGLU(nn.Module):
    def __init__(self, dim, inner, gate_width):
        super().__init__()
        self.proj = nn.Linear(dim, inner * 2)
        self.gate = _Gate(gate_width)


class _FeedForward(nn.Module):
    def __init__(self, dim, gate_width):
        super().__init__()
        self.net = nn.ModuleList([_GEGLU(dim, dim * 4, gate_width), nn.Dropout(0.0), nn.Linear(dim * 4, dim)])


class _BasicTransformerBlock(nn.Module):
    def __init__(self, dim, heads, ctx_dim, gate_width):
        super().__init__()
        self.norm1 = nn.LayerNorm(dim)
        self.attn1 = _Attention(dim, heads)
        self.norm2 = nn.LayerNorm(dim)
        self.attn2 = _Attention(dim, heads, ctx_dim)
        self.norm3 = nn.LayerNorm(dim)
        self.ff = _FeedForward(dim, gate_width)


class Transformer2DModelWidthGated(nn.Module):
    """Parameters of blocks.py:941 / :1070 (depth_gated=True)."""

    def __init__(self, dim, heads, ctx_dim, groups, gate_width, depth_gated=False):
        super().__init__()
        self.norm = nn.GroupNorm(groups, dim, eps=1e-6)
        self.proj_in = nn.Linear(dim, dim)
        self.transformer_blocks = nn.ModuleList([_BasicTransformerBlock(dim, heads, ctx_dim, gate_width)])
        self.proj_out = nn.Linear(dim, dim)
        self.dim, self.heads, self.ctx_dim, self.groups, self.gate_width = dim, heads, ctx_dim, groups, gate_width
        self.depth_gate = _Gate(1) if depth_gated else None
        self.uid = ""

    def gate_widths(self):
        return [self.heads, self.heads, self.gate_width]


class _Sampler(nn.Module):
    def __init__(self, c, stride):
        super().__init__()
        self.conv = nn.Conv2d(c, c, 3, stride=stride, padding=1)


class _Block(nn.Module):
    """Down / mid / up container. forward() runs the block on the engine so that forward hooks
    registered by the trainer (pdm/training/trainer.py:496-511) fire with the block output."""
    kind = "down"

    def forward(self, eng, x, *rest):  # pragma: no cover - dispatched in subclasses
        raise NotImplementedError


class DownBlock2DHalfGated(_Block):
    kind = "down"

    def __init__(self, cfg, cin, cout, heads, has_attn, add_down):
        super().__init__()
        n = cfg["layers_per_block"]
        self.resnets = nn.ModuleList([
            ResnetBlock2DWidthGated(cin if i == 0 else cout, cout, cfg["temb"], cfg["groups"], cfg["eps"],
                                    depth_gated=(i == n - 1)) for i in range(n)])
        self.attentions = nn.ModuleList([
            Transformer2DModelWidthGated(cout, heads, cfg["ctx_dim"], cfg["groups"], cfg["ff_gate_width"],
                                         depth_gated=(i == n - 1)) for i in range(n)]) if has_attn else None
        self.downsamplers = nn.ModuleList([_Sampler(cout, 2)]) if add_down else None
        self.has_cross_attention = has_attn

    def forward(self, eng, x):
        outs = []
        for i, r in enumerate(self.resnets):
            x = eng.resnet(r, x)
            if self.attentions is not None:
                x = eng.transformer(self.attentions[i], x)
            outs.append(x)
        if self.downsamplers is not None:
            x = eng.downsample(self.downsamplers[0], x)
            outs.append(x)
        return x, tuple(outs)


class MidBlock2DCrossAttnWidthGated(_Block):
    kind = "mid"

    def __init__(self, cfg, c, heads):
        super().__init__()
        self.resnets = nn.ModuleList([ResnetBlock2DWidthGated(c, c, cfg["temb"], cfg["groups"], cfg["eps"]) for _ in range(2)])
        self.attentions = nn.ModuleList([Transformer2DModelWidthGated(c, heads, cfg["ctx_dim"], cfg["groups"], cfg["ff_gate_width"])])
        self.has_cross_attention = True

    def forward(self, eng, x):
        x = eng.resnet(self.resnets[0], x)
        x = eng.transformer(self.attentions[0], x)
        x = eng.resnet(self.resnets[1], x)
        return x


class UpBlock2DHalfGated(_Block):
    kind = "up"

    def __init__(self, cfg, cin, cout, prev, heads, has_attn, add_up):
        super().__init__()
        n = cfg["layers_per_block"] + 1
        res = []
        for i in range(n):
            skip = cin if i == n - 1 else cout
            rin = prev if i == 0 else cout
            res.append(ResnetBlock2DWidthGated(rin + skip, cout, cfg["temb"], cfg["groups"], cfg["eps"],
                                               depth_gated=(i == n - 1), skip_dim=skip if i == n - 1 else None))
        self.resnets = nn.ModuleList(res)
        self.attentions = nn.ModuleList([
            Transformer2DModelWidthGated(cout, heads, cfg["ctx_dim"], cfg["groups"], cfg["ff_gate_width"],
                                         depth_gated=(i == n - 1)) for i in range(n)]) if has_attn else None
        self.upsamplers = nn.ModuleList([_Sampler(cout, 1)]) if add_up else None
        self.has_cross_attention = has_attn

    def forward(self, eng, x, skips):
        for i, r in enumerate(self.resnets):
            x = eng.resnet(r, x, skip=skips.pop())
            if self.attentions is not None:
                x = eng.transformer(self.attentions[i], x)
        if self.upsamplers is not None:
            x = eng.upsample(self.upsamplers[0], x)
        return x


class _TimestepEmbedding(nn.Module):
    def __init__(self, cin, dim):
        super().__init__()
        self.linear_1 = nn.Linear(cin, dim)
        self.linear_2 = nn.Linear(dim, dim)


# --------------------------------------------------------------------------------------------------
# activations in engine layout
# --------------------------------------------------------------------------------------------------
class Act:
    """[B*H*W, ld] rows of C valid channels (NHWC / token-major), samples in engine order. `t` holds bf16 rows (what
    every GEMM A operand is), `f` fp32 rows: the tensors BETWEEN blocks (ResNet / transformer / sampler outputs, i.e.
    the residual stream of unet_2d_conditional.py:1629-1715) are kept in fp32 by the inference engine so the running
    residual sum is not re-rounded to bf16 at every block (DESIGN.md section 4); a bf16 copy is made only where a GEMM
    reads the tensor directly. The training engine keeps bf16 rows throughout."""
    __slots__ = ("t", "f", "B", "H", "W", "C", "ld", "cs")

    def __init__(self, t, B, H, W, C, ld=None, f=None, cs=None):
        self.t, self.f, self.B, self.H, self.W, self.C = t, f, B, H, W, C
        self.ld = ld if ld is not None else C
        # (sum plane, sumsq plane) [B * H*W/32, C] fp32: per-channel GroupNorm partials written by the epilogue of the
        # GEMM that produced `f` (APTP_EPI_GN_STATS), or None when the shape is not eligible
        self.cs = cs

    @property
    def hw(self):
        return self.H * self.W

    @property
    def rows(self):
        return self.B * self.H * self.W

    def nchw(self) -> torch.Tensor:
        """Zero-copy [B, C, H, W] view (channels-last strides), as the reference's hooks see it."""
        src = self.t if self.t is not None else self.f
        return src.view(self.B, self.H, self.W, self.ld)[..., : self.C].permute(0, 3, 1, 2)


class UNet2DConditionModelGated(nn.Module):
    """SD-2.1 gated U-Net (reference: unet_2d_conditional.py:628). Only the shipped block layout is
    supported: CrossAttnDownBlock2DHalfGated x3 + DownBlock2DHalfGated, UNetMidBlock2DCrossAttnWidthGated,
    UpBlock2DHalfGated + CrossAttnUpBlock2DHalfGated x3 (configs/pruning/sd-2-1_cc3m.yaml:11-26)."""

    def __init__(self, in_channels=4, out_channels=4, block_out_channels=(320, 640, 1280, 1280),
                 attention_head_dim=(5, 10, 20, 20), layers_per_block=2, cross_attention_dim=1024,
                 norm_num_groups=32, norm_eps=1e-5, gated_ff=True, ff_gate_width=32,
                 down_block_types=("CrossAttnDownBlock2DHalfGated", "CrossAttnDownBlock2DHalfGated",
                                   "CrossAttnDownBlock2DHalfGated", "DownBlock2DHalfGated"),
                 mid_block_type="UNetMidBlock2DCrossAttnWidthGated",
                 up_block_types=("UpBlock2DHalfGated", "CrossAttnUpBlock2DHalfGated", "CrossAttnUpBlock2DHalfGated",
                                 "CrossAttnUpBlock2DHalfGated"), sample_size=96, **other):
        super().__init__()
        for k, v in other.items():
            if k in _ONLY_SUPPORTED and v not in _ONLY_SUPPORTED[k]:
                raise NotImplementedError(f"UNet config {k}={v!r} is not part of the APTP SD-2.1 hot path "
                                          f"(supported: {_ONLY_SUPPORTED[k]})")
        if not gated_ff:
            raise NotImplementedError("only gated_ff=True (the shipped configs) is supported")
        if mid_block_type != "UNetMidBlock2DCrossAttnWidthGated":
            raise NotImplementedError(mid_block_type)
        ch = tuple(block_out_channels)
        heads = tuple(attention_head_dim) if not isinstance(attention_head_dim, int) else (attention_head_dim,) * len(ch)
        for c, h in zip(ch, heads):
            if c != h * 64:
                raise NotImplementedError("attention head_dim must be 64 (SD-2.1); got C=%d heads=%d" % (c, h))
            if c % 8 or c % norm_num_groups:
                raise NotImplementedError("channels must be multiples of 8 and of norm_num_groups")
        down_has_attn = tuple(t.startswith("CrossAttn") for t in down_block_types)
        up_has_attn = tuple(t.startswith("CrossAttn") for t in up_block_types)
        for t in tuple(down_block_types) + tuple(up_block_types):
            if not t.endswith("HalfGated"):
                raise NotImplementedError(f"block type {t}: only the *HalfGated blocks of the shipped configs exist")
        cfg_d = {k: v for k, v in other.items() if not k.startswith("_")}  # unknown / inert keys are preserved
        cfg_d.update(in_channels=in_channels, out_channels=out_channels, block_out_channels=ch,
                     attention_head_dim=heads, layers_per_block=layers_per_block,
                     cross_attention_dim=cross_attention_dim, norm_num_groups=norm_num_groups,
                     norm_eps=norm_eps, gated_ff=gated_ff, ff_gate_width=ff_gate_width, sample_size=sample_size,
                     down_block_types=tuple(down_block_types), mid_block_type=mid_block_type,
                     up_block_types=tuple(up_block_types), use_linear_projection=True)
        object.__setattr__(self, "_config", FrozenConfig(cfg_d))
        cfg = dict(layers_per_block=layers_per_block, temb=ch[0] * 4, groups=norm_num_groups, eps=norm_eps,
                   ctx_dim=cross_attention_dim, ff_gate_width=ff_gate_width)
        self.conv_in = nn.Conv2d(in_channels, ch[0], 3, padding=1)
        self.time_embedding = _TimestepEmbedding(ch[0], ch[0] * 4)
        downs, out_c = [], ch[0]
        for i, c in enumerate(ch):
            in_c, out_c = out_c, c
            downs.append(DownBlock2DHalfGated(cfg, in_c, out_c, heads[i], down_has_attn[i], add_down=i < len(ch) - 1))
        self.down_blocks = nn.ModuleList(downs)
        self.mid_block = MidBlock2DCrossAttnWidthGated(cfg, ch[-1], heads[-1])
        rev, rev_heads = list(reversed(ch)), list(reversed(heads))
        ups, out_c = [], rev[0]
        for i in range(len(ch)):
            prev, out_c = out_c, rev[i]
            in_c = rev[min(i + 1, len(ch) - 1)]
            ups.append(UpBlock2DHalfGated(cfg, in_c, out_c, prev, rev_heads[i], up_has_attn[i], add_up=i < len(ch) - 1))
        self.up_blocks = nn.ModuleList(ups)
        self.conv_norm_out = nn.GroupNorm(norm_num_groups, ch[0], eps=norm_eps)
        self.conv_out = nn.Conv2d(ch[0], out_channels, 3, padding=1)

        # gate bookkeeping in get_structure() order
        self._gated: List[nn.Module] = []
        for bi, blk in enumerate(list(self.down_blocks) + [self.mid_block] + list(self.up_blocks)):
            mods = list(blk.resnets) + (list(blk.attentions) if blk.attentions is not None else [])
            for mi, m in enumerate(mods):
                m.uid = f"b{bi}.m{mi}"
            self._gated += mods
        self._resnets = [m for m in self.modules() if isinstance(m, ResnetBlock2DWidthGated)]
        off = 0
        self._temb_off: Dict[str, int] = {}
        for r in self._resnets:
            self._temb_off[r.uid] = off
            off += r.cout
        self._temb_total = off
        self.structure = {"width": [], "depth": []}
        self.resource_info_dict = None
        self._macs_table = None
        self.prunable_macs_list = None
        self.total_macs = None
        self._engine: Optional["_Engine"] = None
        self._gate_state: Optional[Dict[str, Any]] = None
        self._last_shape: Optional[Tuple[int, int, int]] = None  # (H, W, text tokens) of the last forward
        self.gradient_checkpointing = False
        # False: gated semantics (a zero-gated GroupNorm group still feeds silu(beta) into conv2, SURVEY Appendix D-1);
        # True: the semantics of the reference's prune() (blocks.py:451-463 deletes those channels)
        self.pruned_semantics = False
        self.set_all_ones_structure()

    # ---------------------------------------------------------------------------------------------
    # reference API: the ModelMixin / ConfigMixin surface its callers touch
    # ---------------------------------------------------------------------------------------------
    @property
    def config(self) -> FrozenConfig:
        return self.__dict__["_config"]

    def register_to_config(self, **kwargs) -> None:
        """ConfigMixin.register_to_config (unet_2d_conditional.py:872 uses it for encoder_hid_dim_type)."""
        for k, v in kwargs.items():
            if k in _ONLY_SUPPORTED and v not in _ONLY_SUPPORTED[k]:
                raise NotImplementedError(f"UNet config {k}={v!r} is not part of the APTP SD-2.1 hot path")
        d = dict(self.config)
        d.update(kwargs)
        object.__setattr__(self, "_config", FrozenConfig(d))

    @property
    def dtype(self) -> torch.dtype:
        """Parameter dtype (ModelMixin.dtype); the kernels compute in bf16 with fp32 accumulation whatever it is."""
        return next(self.parameters()).dtype

    @property
    def device(self) -> torch.device:
        return next(self.parameters()).device

    def enable_gradient_checkpointing(self) -> None:
        """trainer.py:160. Accepted and recorded; the tape engine already keeps only what the backward kernels read."""
        self.gradient_checkpointing = True

    def disable_gradient_checkpointing(self) -> None:
        self.gradient_checkpointing = False

    def enable_xformers_memory_efficient_attention(self, *args, **kwargs) -> None:
        """trainer.py:144-156. REFUSED: in the reference this call replaces HeadGatedAttnProcessor2 and silently turns head
        gating off (SURVEY section 5 / Appendix D-9); the shipped configs keep it off (configs/pruning/sd-2-1_cc3m.yaml:84).
        Attention here always runs the fused head-gated sm_100a kernel."""
        raise NotImplementedError("enable_xformers_memory_efficient_attention would disable head gating in the reference "
                                  "(blocks.py:140); attention already runs the fused head-gated tcgen05 kernel")

    def disable_xformers_memory_efficient_attention(self) -> None:
        pass

    def set_attn_processor(self, processor) -> None:
        raise NotImplementedError("attention processors are not pluggable on the sm_100a path (head gating is fused)")

    # ---------------------------------------------------------------------------------------------
    # reference API: structure
    # ---------------------------------------------------------------------------------------------
    def get_structure(self) -> Dict[str, List[List[int]]]:
        """unet_2d_conditional.py:1332-1363 -- per block, resnets first then attentions."""
        if len(self.structure["width"]) == 0:
            self.structure = {"width": [m.gate_widths() for m in self._gated],
                              "depth": [[1] if m.depth_gate is not None else [0] for m in self._gated]}
        return self.structure

    def set_structure(self, arch_vectors: Dict[str, List[torch.Tensor]]) -> None:
        """unet_2d_conditional.py:1365-1413. Consumes (pops) the caller's lists like the reference."""
        width, depth = arch_vectors["width"], arch_vectors["depth"]
        flat_w, flat_d = [], []
        for blk in list(self.down_blocks) + [self.mid_block] + list(self.up_blocks):
            mods = list(blk.resnets) + (list(blk.attentions) if blk.attentions is not None else [])
            w_take = []
            for m in mods:
                ws = []
                for wd in m.gate_widths():
                    assert wd == width[0].shape[1], f"width gate mismatch: expected {wd}, got {width[0].shape[1]}"
                    ws.append(width.pop(0))
                w_take.append(ws)
            d_take = [depth.pop(0) if m.depth_gate is not None else None for m in mods]
            for m, ws, d in zip(mods, w_take, d_take):
                if isinstance(m, ResnetBlock2DWidthGated):
                    m.gate.set_structure_value(ws[0])
                else:
                    tb = m.transformer_blocks[0]
                    tb.attn1.gate.set_structure_value(ws[0])
                    tb.attn2.gate.set_structure_value(ws[1])
                    tb.ff.net[0].gate.set_structure_value(ws[2])
                if d is not None:
                    m.depth_gate.set_structure_value(d)
                flat_w += ws
                if d is not None:
                    flat_d.append(d)
        self._gate_state = None  # re-derived lazily on the next forward
        self._flat_gates = (flat_w, flat_d)

    def set_all_ones_structure(self, batch: int = 1, device=None) -> None:
        st = self.get_structure()
        self.set_structure({"width": [torch.ones(batch, w, device=device) for ws in st["width"] for w in ws],
                            "depth": [torch.ones(batch, device=device) for d in st["depth"] if d == [1]]})

    def enable_weight_training(self, on: bool = True) -> None:
        """Opt in to the fine-tune path: forwards under autograd then differentiate w.r.t. every parameter that
        requires grad (FineTuner: `unet.train()` + an optimizer over `unet.parameters()`, trainer.py:1560-1600).
        Off (default): the U-Net is treated as frozen, as the pruning stage and sampling do."""
        self._train_weights = bool(on)
        self._engine = None
        self._train_engine = None

    def freeze(self) -> None:
        """unet_2d_conditional.py:2118-2122."""
        for name, p in self.named_parameters():
            if "gate_f" not in name:
                p.requires_grad = False

    # ---------------------------------------------------------------------------------------------
    # reference API: MAC accounting (closed form of op_counter + calc_macs tree, SURVEY Appendix F)
    # ---------------------------------------------------------------------------------------------
    def count_macs(self, H: int, W: int, n_ctx: int = 77) -> None:
        """What Pruner.count_macs (trainer.py:1257-1296) measures with forward hooks at batch 1 through
        op_counter.count_ops_and_params, as a closed form (SURVEY Appendix F); afterwards the attributes
        the trainer sets (`resource_info_dict` = calc_macs() at all-ones gates, `prunable_macs_list`
        normalised by the prunable total, `total_macs`) are filled in the same way (trainer.py:1281-1286)."""
        from .macs import build_resource_info
        self._macs_table = build_resource_info(self, H, W, n_ctx)
        dev = next(self.parameters()).device
        self.set_all_ones_structure(1, device=dev)
        d = self.calc_macs()
        self.resource_info_dict = d
        self.total_macs = d["total_macs"]
        self.prunable_macs_list = [[e / d["prunable_macs"] for e in elem] for elem in self.get_prunable_macs()]

    def calc_macs(self) -> Dict[str, Any]:
        from .macs import build_resource_info, calc_macs
        if self._macs_table is None:
            # The reference stamps `__macs__` on every leaf during ONE hooked forward (count_ops_and_params at
            # trainer.py:1272) and calc_macs() reads those stamps ever after. Here the stamps are a closed form in the
            # layer shapes, so the same call sequence -- set_structure(all ones); unet(sample, t, ctx); calc_macs() --
            # works with the hooked forward replaced by a plain one: the table is derived from the shapes of the
            # last forward, once, and kept (like the reference's stamps, it does not follow later resolutions).
            if self._last_shape is None:
                raise RuntimeError("calc_macs() needs one forward (the reference's count_ops_and_params pass, "
                                   "trainer.py:1257-1296) or count_macs(H, W) first")
            H, W, n_ctx = self._last_shape
            self._macs_table = build_resource_info(self, H, W, n_ctx)
        return calc_macs(self)

    def get_prunable_macs(self):
        from .macs import prunable_macs_list
        return prunable_macs_list(self)

    def get_block_utilization(self):
        from .macs import block_utilization
        return block_utilization(self)

    # ---------------------------------------------------------------------------------------------
    # forward
    # ---------------------------------------------------------------------------------------------
    def invalidate_weight_cache(self) -> None:
        """Call after changing parameters (the pruning workflow keeps the U-Net frozen)."""
        self._engine = None

    def _load_from_state_dict(self, *args, **kwargs):
        self._engine = None
        self._train_engine = None
        return super()._load_from_state_dict(*args, **kwargs)

    def forward(self, sample: torch.Tensor, timestep, encoder_hidden_states: torch.Tensor,
                class_labels=None, timestep_cond=None, attention_mask=None, cross_attention_kwargs=None,
                added_cond_kwargs=None, down_block_additional_residuals=None, mid_block_additional_residual=None,
                encoder_attention_mask=None, return_dict: bool = True):
        """unet_2d_conditional.py:1415-1726 for the SD-2.1 configuration (no class / added conditioning,
        no attention masks, no ControlNet residuals: those raise)."""
        for name, v in (("class_labels", class_labels), ("timestep_cond", timestep_cond),
                        ("attention_mask", attention_mask), ("added_cond_kwargs", added_cond_kwargs),
                        ("down_block_additional_residuals", down_block_additional_residuals),
                        ("mid_block_additional_residual", mid_block_additional_residual),
                        ("encoder_attention_mask", encoder_attention_mask)):
            if v is not None:
                raise NotImplementedError(f"{name} is not part of the APTP hot path")
        _require_cuda(sample)
        self._last_shape = (int(sample.shape[2]), int(sample.shape[3]), int(encoder_hidden_states.shape[1]))
        blocks = list(self.down_blocks) + [self.mid_block] + list(self.up_blocks)
        want_taps = any(len(b._forward_hooks) > 0 for b in blocks)
        flat_w, flat_d = self._flat_gates
        gates = list(flat_w) + list(flat_d)
        if torch.is_grad_enabled() and getattr(self, "_train_weights", False):
            # fine-tune stage (trainer.py:1683-1765): gradients to every U-Net parameter, gates are constants
            from .train import UNetFineTuneFunction
            params = [p for p in self.parameters() if p.requires_grad]
            outs = UNetFineTuneFunction.apply(self, sample, timestep, encoder_hidden_states, len(blocks), *params)
            out, taps = outs[0], list(outs[1:])
        elif torch.is_grad_enabled() and any(g.requires_grad for g in gates):
            # differentiable student forward of the pruning step (trainer.py:1192-1195): one autograd node
            from .train import UNetTrainFunction
            outs = UNetTrainFunction.apply(self, sample, timestep, encoder_hidden_states, len(blocks), *gates)
            out, taps = outs[0], list(outs[1:])
        else:
            if self._engine is None or self._engine.device != sample.device:
                self._engine = _Engine(self, sample.device)
            out, taps = self._engine.run_graphed(sample, timestep, encoder_hidden_states, want_taps=want_taps)
        if sample.is_cuda:
            K.poll_abort()  # no sync: reports an mbarrier timeout of an earlier launch instead of returning garbage
        if want_taps:
            # fire the hooks the trainer registers on down_blocks[i] / mid_block / up_blocks[i]
            # (trainer.py:496-511) with tensors shaped like the reference's outputs: down blocks return
            # (hidden_states, residuals) and the hook reads output[0]
            for blk, tap in zip(blocks, taps):
                o = (tap, ()) if blk.kind == "down" else tap
                for hook in list(blk._forward_hooks.values()):
                    hook(blk, (), o)
        if not return_dict:
            return (out,)
        return UNet2DConditionOutput(sample=out)

    # ---------------------------------------------------------------------------------------------
    # on-disk format: the diffusers layout the reference reads and writes (`<dir>/unet/config.json` +
    # `diffusion_pytorch_model.safetensors`; trainer.py:285-292, :1452-1462; gates add no tensors, gates.py:13)
    # ---------------------------------------------------------------------------------------------
    _STOCK_TO_GATED = {"CrossAttnDownBlock2D": "CrossAttnDownBlock2DHalfGated", "DownBlock2D": "DownBlock2DHalfGated",
                       "UpBlock2D": "UpBlock2DHalfGated", "CrossAttnUpBlock2D": "CrossAttnUpBlock2DHalfGated",
                       "UNetMidBlock2DCrossAttn": "UNetMidBlock2DCrossAttnWidthGated"}

    def save_pretrained(self, save_directory: str, sliced: bool = False, **unused) -> None:
        """`sliced=True` (UNet2DConditionModelPruned only) writes the physically sliced tensors the reference's pruned
        models hold (what its FineTuner checkpoints contain and scripts/metrics/generate_fid_images.py:100-102 loads);
        the default writes the dense SD-2.1 tensors. Either file loads back through from_pretrained."""
        import json
        import os
        from safetensors.torch import save_file
        os.makedirs(save_directory, exist_ok=True)
        cfg = {k: (list(v) if isinstance(v, tuple) else v) for k, v in self.config.items()}
        cfg.update(_class_name=type(self).__name__, gated_ff=True, mid_block_type="UNetMidBlock2DCrossAttnWidthGated",
                   use_linear_projection=True)
        with open(os.path.join(save_directory, "config.json"), "w") as f:
            json.dump(cfg, f, indent=2)
        sd = self.sliced_state_dict() if sliced else self.state_dict()
        save_file({k: v.detach().cpu().contiguous() for k, v in sd.items()},
                  os.path.join(save_directory, "diffusion_pytorch_model.safetensors"))

    @classmethod
    def from_pretrained(cls, pretrained_model_name_or_path: str, subfolder: Optional[str] = None, **overrides):
        """Local directories only (no hub access). A stock SD-2.1 `unet/config.json` is accepted: its block type
        names are mapped to the gated ones unless the caller overrides them, as the reference's callers do
        (trainer.py:730-740, :1452-1462)."""
        import json
        import os
        directory = os.path.join(pretrained_model_name_or_path, subfolder) if subfolder else pretrained_model_name_or_path
        with open(os.path.join(directory, "config.json")) as f:
            cfg = json.load(f)
        for k in ("revision", "torch_dtype", "variant", "use_safetensors", "low_cpu_mem_usage"):
            overrides.pop(k, None)
        extra = {k: overrides.pop(k) for k in ("arch_vector", "random_pruning_ratio") if k in overrides}
        cfg = {k: v for k, v in cfg.items() if not k.startswith("_")}
        cfg.update(overrides)
        for key in ("down_block_types", "up_block_types"):
            cfg[key] = tuple(cls._STOCK_TO_GATED.get(t, t) for t in cfg[key])
        cfg["mid_block_type"] = cls._STOCK_TO_GATED.get(cfg.get("mid_block_type"), cfg.get("mid_block_type"))
        cfg.setdefault("gated_ff", True)
        if not cfg.get("use_linear_projection", True):
            raise NotImplementedError("use_linear_projection=False (SD-1.x) is not part of the APTP SD-2.1 hot path")
        model = cls(**cfg)
        st_path = os.path.join(directory, "diffusion_pytorch_model.safetensors")
        if os.path.exists(st_path):
            from safetensors.torch import load_file
            sd = load_file(st_path)
        else:
            sd = torch.load(os.path.join(directory, "diffusion_pytorch_model.bin"), map_location="cpu")
        model._pre_load(directory, **extra)   # the pruned class fixes its code first (prune-then-load, :2425-2436)
        model.load_state_dict(sd)
        model.eval()
        return model

    def _pre_load(self, directory: str, **extra) -> None:
        if extra:
            raise TypeError(f"unexpected arguments for {type(self).__name__}.from_pretrained: {sorted(extra)}")

    def sliced_state_dict(self):
        raise NotImplementedError("only UNet2DConditionModelPruned (one static code) has a physically sliced layout")

    def _get_train_engine(self, device):
        from .train import TrainEngine
        device = torch.device(device)
        if device.type == "cuda" and device.index is None:  # "cuda" and "cuda:0" must not look like two devices
            device = torch.device("cuda", torch.cuda.current_device())
        te = getattr(self, "_train_engine", None)
        if te is None or te.device != device:
            te = TrainEngine(self, device)
            if self._engine is not None and self._engine.device == device:
                te.dense = self._engine.dense  # share the packed frozen weights
            self._train_engine = te
        return te


# --------------------------------------------------------------------------------------------------
# engine
# --------------------------------------------------------------------------------------------------
class UNet2DConditionModelPruned(UNet2DConditionModelGated):
    """One static expert (reference: unet_2d_conditional.py:2183-2436): the gated U-Net fixed to ONE architecture
    vector with prune() semantics. The reference slices the weights at load time (`m.prune()` / `m.prune_module()`,
    :2425-2436); here the dense diffusers weights stay as loaded and the compacted per-expert blocks the kernels
    consume are derived from them (plan.py), so the same checkpoint serves any code and `state_dict()` keeps the
    stock key names. `arch_vector` is [1, 1620] (soft values are thresholded at 0.5 like hard_concrete in prune());
    forwards of any batch size run the expert's compacted GEMMs only."""

    def __init__(self, *args, arch_vector: Optional[torch.Tensor] = None, **kwargs):
        super().__init__(*args, **kwargs)
        self.pruned_semantics = True
        self.arch_vector = None
        if arch_vector is not None:
            self.prune_to(arch_vector)

    def prune_to(self, arch_vector: torch.Tensor) -> None:
        from .hypernet import HyperStructure
        from .quantizer import hard_concrete
        assert arch_vector.dim() == 2 and arch_vector.shape[0] == 1, "Pruning is only supported for single batch size"
        self.arch_vector = arch_vector.detach().clone()
        hard = hard_concrete(arch_vector.detach().float()).detach()
        self.set_structure(HyperStructure.transform_arch_vector(hard, self.get_structure()))
        self.invalidate_weight_cache()
        self._train_engine = None

    def _pre_load(self, directory: str, arch_vector=None, random_pruning_ratio=None) -> None:
        """arch_vector.pt next to the unet/ folder (written by FineTuner, trainer.py:1449-1450), unless given. The code is
        fixed BEFORE the weights are loaded, like the reference (unet_2d_conditional.py:2425-2436 prunes, then loads), so
        that checkpoints holding physically sliced tensors can be scattered into place."""
        import os
        from .hypernet import HyperStructure
        if arch_vector is None:
            for cand in (os.path.join(os.path.dirname(os.path.normpath(directory)), "arch_vector.pt"),
                         os.path.join(directory, "arch_vector.pt")):
                if os.path.exists(cand):
                    arch_vector = torch.load(cand, map_location="cpu")
                    break
        if isinstance(arch_vector, str):
            arch_vector = torch.load(arch_vector, map_location="cpu")
        if random_pruning_ratio is not None:
            arch_vector = HyperStructure.get_random_arch_vector(random_pruning_ratio, self.get_structure())
        if arch_vector is not None:
            self.prune_to(arch_vector)

    # ---- the reference's physically sliced layout (blocks.py:52-67, :121-129, :153-187, :424-465, :641-697, :1427-1438) ----
    def _slice_plan(self):
        """[(parameter name, dim, kept index tensor | None)]: how every prunable tensor of the dense model is sliced for
        the current code; None marks a parameter of a depth-dropped block (absent from the sliced layout: the reference
        replaces those modules by nn.Identity). Parameters not listed are stored as they are."""
        assert self.arch_vector is not None, "prune_to(arch_vector) first"
        plan = []
        hard = lambda g: (g.detach().float().reshape(-1) >= 0.5)  # noqa: E731
        for name, m in self.named_modules():
            if isinstance(m, ResnetBlock2DWidthGated):
                if m.depth_gate is not None and not bool(hard(m.depth_gate.gate_f)[0]):
                    plan += [(f"{name}.{k}", 0, None) for k, _ in m.named_parameters()]
                    continue
                keep = hard(m.gate.gate_f).repeat_interleave(m.cout // m.groups).nonzero().reshape(-1)
                plan += [(f"{name}.conv1.weight", 0, keep), (f"{name}.conv1.bias", 0, keep),
                         (f"{name}.time_emb_proj.weight", 0, keep), (f"{name}.time_emb_proj.bias", 0, keep),
                         (f"{name}.norm2.weight", 0, keep), (f"{name}.norm2.bias", 0, keep),
                         (f"{name}.conv2.weight", 1, keep)]
            elif isinstance(m, Transformer2DModelWidthGated):
                if m.depth_gate is not None and not bool(hard(m.depth_gate.gate_f)[0]):
                    plan += [(f"{name}.{k}", 0, None) for k, _ in m.named_parameters()]
                    continue
                tb = m.transformer_blocks[0]
                for an, attn in (("attn1", tb.attn1), ("attn2", tb.attn2)):
                    keep = hard(attn.gate.gate_f).repeat_interleave(64).nonzero().reshape(-1)
                    pre = f"{name}.transformer_blocks.0.{an}"
                    plan += [(f"{pre}.to_q.weight", 0, keep), (f"{pre}.to_k.weight", 0, keep),
                             (f"{pre}.to_v.weight", 0, keep), (f"{pre}.to_out.0.weight", 1, keep)]
                proj = tb.ff.net[0].proj
                inner = proj.weight.shape[0] // 2
                kf = hard(tb.ff.net[0].gate.gate_f).repeat_interleave(inner // tb.ff.net[0].gate.width).nonzero().reshape(-1)
                pre = f"{name}.transformer_blocks.0.ff.net"
                both = torch.cat([kf, kf + inner])  # GEGLUGated.prune_gate: the same groups of both halves (blocks.py:55-57)
                plan += [(f"{pre}.0.proj.weight", 0, both), (f"{pre}.0.proj.bias", 0, both), (f"{pre}.2.weight", 1, kf)]
        return plan

    def sliced_state_dict(self) -> Dict[str, torch.Tensor]:
        """state_dict() as the reference's pruned model holds it: kept rows / columns only, no entries for
        depth-dropped blocks (same keys and shapes as the prune sweep of unet_2d_conditional.py:2425-2436 produces)."""
        sd = dict(self.state_dict())
        for key, dim, keep in self._slice_plan():
            if keep is None:
                sd.pop(key, None)
            else:
                sd[key] = sd[key].index_select(dim, keep.to(sd[key].device))
        return sd

    def load_state_dict(self, state_dict, strict: bool = True, assign: bool = False):
        """Accepts the dense SD-2.1 layout and, once a code is set, the reference's physically sliced layout: sliced
        tensors are scattered into the dense parameters by the kept index lists of the code (pruned rows / columns and
        depth-dropped blocks are zero-filled; prune() semantics never reads them)."""
        dense = self.state_dict()
        sliced = any(k in state_dict and tuple(state_dict[k].shape) != tuple(v.shape) for k, v in dense.items()) or \
            (self.arch_vector is not None and any(k not in state_dict for k in dense))
        if sliced:
            if self.arch_vector is None:
                raise RuntimeError("this checkpoint holds physically sliced tensors: pass arch_vector=... to from_pretrained "
                                   "or call prune_to(arch_vector) before load_state_dict (the reference prunes, then loads)")
            full = dict(state_dict)
            for key, dim, keep in self._slice_plan():
                tgt = torch.zeros_like(dense[key])
                if keep is not None and key in state_dict:
                    src = state_dict[key].to(tgt.dtype)
                    want = list(tgt.shape)
                    want[dim] = keep.numel()
                    if list(src.shape) == list(tgt.shape):
                        tgt = src.clone()  # a dense tensor inside an otherwise sliced file
                    else:
                        if list(src.shape) != want:
                            raise RuntimeError(f"{key}: sliced shape {tuple(src.shape)} does not match the code "
                                               f"(expected {tuple(want)})")
                        tgt.index_copy_(dim, keep.to(tgt.device), src.to(tgt.device))
                elif keep is not None and strict:
                    raise RuntimeError(f"missing key {key} in a sliced checkpoint")
                full[key] = tgt
            state_dict = full
        return super().load_state_dict(state_dict, strict=strict, assign=assign)


class _Engine:
    def __init__(self, model: UNet2DConditionModelGated, device, sources: Optional[Sequence[nn.Module]] = None,
                 gates: Optional[Any] = None):
        """`model` gives the module tree and config. `sources`: models of that same tree whose parameters the packs are
        built from, one per weight source (a bucket's source is ExpertSet.source; default: the model alone). `gates`:
        the owner of the gate state (`_gate_state` / `_flat_gates`; default: the model)."""
        self.m = model
        self.srcs = list(sources) if sources is not None else [model]
        self.gates = gates if gates is not None else model
        self.src_of = np.zeros(1, dtype=np.int64)  # weight source of each expert bucket of the current forward
        self.device = device
        self.dense: Dict[str, Dict[str, torch.Tensor]] = {}
        self.expert: Dict[Tuple[bytes, str], Dict[str, Any]] = {}
        self.sched: Dict[Any, Any] = {}
        self.arena: Dict[Any, torch.Tensor] = {}
        self._packs: List[tuple] = []     # (device tensors derived from parameters, their builder): see _pack()
        self._pack_graph = None
        self._pack_graph_n = -1
        self.flops = 0.0          # kept GEMM-class FLOPs of the last forward (roofline accounting)
        self.gemm_bytes = 0.0     # algorithmic HBM bytes of the grouped-GEMM launches of the last forward
        self.launches = 0
        self.count_flops = False
        self._label = ""
        self.profile: Optional[list] = None  # set to [] to bracket every GEMM / attention launch with CUDA events
        self.graphs: Dict[Any, Any] = {}     # CUDA graphs of the hard-gate forward, keyed by shapes + structure content
        self.graph_seen: Dict[Any, int] = {}
        # Bounded caches (the reference calls set_structure for EVERY prompt batch, pruning_pipelines.py:757-759, so a long
        # sampling run walks through many prompt -> expert assignments): schedules / layouts are kept for the
        # MAX_STATES most recently used (batch, code set, assignment) states, compacted weight packs for the MAX_ESETS
        # most recently used code sets; older entries are dropped together with their device buffers.
        # APTP_LN_FOLD=0 keeps the three LayerNorms of a transformer block as separate HBM passes (A/B measurements)
        self.ln_fold = os.environ.get("APTP_LN_FOLD", "1") != "0"
        # APTP_GN_EPI=0: GroupNorm statistics by the separate pass over HBM instead of the producing GEMM's epilogue
        self.gn_epi = os.environ.get("APTP_GN_EPI", "1") != "0"
        self._states: "OrderedDict[Any, int]" = OrderedDict()
        self._esets: "OrderedDict[Any, int]" = OrderedDict()
        self._next_id = 0
        self._sid = self._eid = -1
        # per-forward state
        self.B = 0
        self.compact = False
        self.eset: Optional[P.ExpertSet] = None
        self.layout: Optional[P.BatchLayout] = None
        self.soft: Dict[str, torch.Tensor] = {}

    # ---- workspace -------------------------------------------------------------------------------
    def buf(self, name: str, rows: int, cols: int, dtype=BF16) -> torch.Tensor:
        key = (name, rows, cols, dtype)
        t = self.arena.get(key)
        if t is None:
            t = torch.zeros(rows, cols, device=self.device, dtype=dtype)  # zero once: stale data stays finite
            self.arena[key] = t
        return t

    # ---- gates -> mode / experts -------------------------------------------------------------------
    # ---- parameter-derived device tensors ("packs") ---------------------------------------------------
    def _pack(self, store: dict, key, builder):
        """store[key], built once by `builder()` (a tensor, or a dict holding tensors and host-side data). The pair is
        registered so that refresh_packs() can re-derive the device tensors IN PLACE after an optimizer step changed the
        parameters (fine-tune stage); inference and the pruning stage (frozen U-Net) never refresh."""
        d = store.get(key)
        if d is None:
            d = builder()
            store[key] = d
            self._packs.append((d, builder))
        return d

    def _refresh_packs_eager(self) -> None:
        for old, builder in self._packs:
            new = builder()
            if torch.is_tensor(old):
                if new.data_ptr() != old.data_ptr():
                    old.copy_(new)
            else:
                for k, v in new.items():
                    o = old.get(k)
                    if torch.is_tensor(v) and torch.is_tensor(o) and v.data_ptr() != o.data_ptr():
                        o.copy_(v)

    def refresh_packs(self) -> None:
        """Re-derive every registered pack from the current parameter values. The builders are pure torch ops on the
        parameters' (static) storage, so the whole pass is captured once into a CUDA graph and replayed afterwards:
        one launch instead of a few thousand small ones per training step."""
        if self._pack_graph is not None and self._pack_graph_n == len(self._packs):
            self._pack_graph.replay()
            return
        self._refresh_packs_eager()
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with _graph_capture(g):
            self._refresh_packs_eager()
        self._pack_graph, self._pack_graph_n = g, len(self._packs)
        g.replay()

    MAX_STATES = 8
    MAX_ESETS = 4

    def _lru_id(self, table: "OrderedDict[Any, int]", key, limit: int, tag: str, store: dict) -> int:
        """Small integer id of `key` in an LRU table; evicting a key drops every `store` entry tagged with its id."""
        i = table.get(key)
        if i is None:
            i = self._next_id
            self._next_id += 1
            table[key] = i
            while len(table) > limit:
                _, old = table.popitem(last=False)
                dead = [k for k in store if isinstance(k, tuple) and len(k) == 2 and k[0] == (tag, old)]
                gone = {id(store.pop(k)) for k in dead}
                if tag == "es" and gone:
                    self._packs = [(d, b) for d, b in self._packs if id(d) not in gone]
                    self._pack_graph, self._pack_graph_n = None, -1
        else:
            table.move_to_end(key)
        return i

    def _prepare_gates(self, B: int):
        m = self.m
        st = self.gates._gate_state
        if st is None:
            flat_w, flat_d = m._flat_gates
            bg = flat_w[0].shape[0]
            arch = torch.cat([w.detach().reshape(bg, -1).float() for w in flat_w] +
                             [d.detach().reshape(bg, 1).float() for d in flat_d], dim=1).to(self.device)
            hard = bool(((arch == 0) | (arch == 1)).all().item())  # one host sync per set_structure
            st = {"arch": arch, "hard": hard, "bg": bg}
            widths = [w for ws in m.get_structure()["width"] for w in ws]
            st["width_starts"] = [0] + np.cumsum(widths).tolist()
            st["n_width"] = int(sum(widths))
            if hard:
                codes = arch.to(torch.uint8).cpu().numpy()
                uniq, inv = np.unique(codes, axis=0, return_inverse=True)
                st["eset"] = P.ExpertSet(codes=uniq, sample_expert=inv.reshape(-1), width_starts=st["width_starts"],
                                         n_width=st["n_width"])
            self.gates._gate_state = st
        assert B % st["bg"] == 0, f"batch {B} is not a multiple of the gate batch {st['bg']}"
        self.compact = st["hard"]
        if self.compact:
            self.eset = st["eset"]
            self.src_of = self.eset.sources()
            # Cached state (schedules, per-position tables, CUDA graph) is keyed on the BUCKET SIZES of the batch, not
            # on which sample went to which expert: a new prompt -> expert assignment with the same sizes only rewrites
            # the two permutation index buffers (device-resident, read by the gathers at the entry / exit of the forward,
            # also under CUDA-graph replay).
            est = st.setdefault(("engine", id(self)), {})  # per-engine cache inside the model's gate state
            if est.get("layout_B") != B or est.get("skey") not in self._states:
                lay = P.BatchLayout.build(self.eset.sample_expert, self.eset.n_experts, B)
                self._sid = self._lru_id(self._states, (B, self.eset.key(), lay.starts.tobytes()),
                                         self.MAX_STATES, "st", self.sched)
                self._eid = self._lru_id(self._esets, self.eset.key(), self.MAX_ESETS, "es", self.expert)
                lk = (("st", self._sid), "layout")
                cached = self.sched.get(lk)
                if cached is None:
                    self.sched[lk] = cached = lay
                else:
                    cached.perm, cached.inv_perm = lay.perm, lay.inv_perm  # expert_of_pos / starts are identical
                    for name, t in cached.__dict__.get("_dev", {}).items():
                        t.copy_(torch.as_tensor(getattr(cached, name[0])), non_blocking=True)
                est["layout_B"], est["sid"], est["eid"], est["layout"] = B, self._sid, self._eid, cached
                est["skey"] = (B, self.eset.key(), lay.starts.tobytes())
            self._sid, self._eid, self.layout = est["sid"], est["eid"], est["layout"]
            self._states.move_to_end(est["skey"])
            if self.eset.key() in self._esets:
                self._esets.move_to_end(self.eset.key())
        else:
            assert len(self.srcs) == 1, "several weight sources need hard (0/1) codes"
            self.eset, self.layout = None, None
            self.src_of = np.zeros(1, dtype=np.int64)
            self._sid = self._lru_id(self._states, (B, b"soft"), self.MAX_STATES, "st", self.sched)
            self._eid = self._lru_id(self._esets, b"soft", self.MAX_ESETS, "es", self.expert)
            arch = st["arch"]
            if B != st["bg"]:
                arch = arch.repeat(B // st["bg"], 1)  # gates.py:18-19 (CFG batch doubling)
            self.soft_arch = arch.contiguous()
        self.gate_cols = {}
        gi = 0
        di = 0
        ws = st["width_starts"]
        for mod in m._gated:
            n = len(mod.gate_widths())
            self.gate_cols[mod.uid] = {"w": list(range(gi, gi + n)), "d": (di if mod.depth_gate is not None else None)}
            gi += n
            if mod.depth_gate is not None:
                di += 1
        self.width_starts = ws
        self.n_width = st["n_width"]

    # ---- small helpers -----------------------------------------------------------------------------
    def _dev_index(self, name: str) -> torch.Tensor:
        """layout.perm / layout.inv_perm as a device tensor, uploaded once per layout (no H2D copy per forward, which
        also keeps the forward CUDA-graph capturable)."""
        cache = self.layout.__dict__.setdefault("_dev", {})
        t = cache.get((name, self.device))
        if t is None:
            t = torch.as_tensor(getattr(self.layout, name), device=self.device)
            cache[(name, self.device)] = t
        return t

    def _per_pos(self, per_expert: Sequence[int], dtype=torch.int32) -> torch.Tensor:
        arr = np.asarray(per_expert)[self.layout.expert_of_pos]
        np_dt = {torch.int32: np.int32, torch.uint8: np.uint8, torch.int64: np.int64}[dtype]
        return K.upload(arr.astype(np_dt), self.device)

    def _soft_gate(self, gate_idx: int) -> torch.Tensor:
        """Columns of one width gate as a VIEW of the [B, 1620] gate matrix: the kernels take the row pitch
        (`gate.stride(0)`), so no per-layer slice copies are launched."""
        s, e = self.width_starts[gate_idx], self.width_starts[gate_idx + 1]
        return self.soft_arch[:, s:e]

    def _soft_depth(self, depth_idx: int) -> torch.Tensor:
        """[B] contiguous depth gate: one transposed copy of the 14 depth columns per gate matrix."""
        dt = getattr(self, "_depth_T", None)
        if dt is None or self._depth_T_src is not self.soft_arch:
            dt = self.soft_arch[:, self.n_width:].t().contiguous()
            self._depth_T, self._depth_T_src = dt, self.soft_arch
        return dt[depth_idx]

    def _expert_active(self, uid: str) -> np.ndarray:
        """[E] bool: False where the block is depth-dropped for that expert."""
        d = self.gate_cols[uid]["d"]
        if d is None or not self.compact:
            return np.ones(self.eset.n_experts if self.compact else 1, dtype=bool)
        return self.eset.depth_bits(d).astype(bool)

    # ---- weight sources ------------------------------------------------------------------------------
    def _src_mod(self, mod: nn.Module, s: int) -> nn.Module:
        """The module of weight source `s` at the place `mod` (a module of self.m) has in the tree."""
        src = self.srcs[s]
        if src is self.m:
            return mod
        names = self.__dict__.get("_mod_names")
        if names is None:
            names = self._mod_names = {id(v): k for k, v in self.m.named_modules()}
        return src.get_submodule(names[id(mod)])

    def _src_stack(self, mod: nn.Module, fn) -> torch.Tensor:
        """fn(module of source s) for every source, concatenated along dim 0 in source order (block s of a stacked
        per-source tensor; a bucket finds its block at src_of * block size)."""
        parts = [fn(self._src_mod(mod, s)) for s in range(len(self.srcs))]
        return parts[0] if len(parts) == 1 else torch.cat(parts, 0).contiguous()

    def _src_off(self, block: int) -> np.ndarray:
        """[E] offset of each bucket's block in a per-source stacked tensor of `block` rows / floats per source."""
        return self.src_of * int(block)

    def _src_seg(self):
        """Per-sample affine row (weight source) for GroupNorms whose affine is stacked per source; None with one."""
        if len(self.srcs) == 1:
            return None
        return self._sched(("src_seg",), lambda: self._per_pos(self.src_of))

    def _variant_packs(self, vid: np.ndarray, kept: List[np.ndarray], build) -> Dict[str, torch.Tensor]:
        """Per-variant weight blocks, each built from the weights of its variant's own source. build(s, kept lists of
        the variants of source s) returns a dict of tensors holding one equal-sized block per variant along dim 0;
        the result holds the blocks of every variant in variant order."""
        vsrc = np.asarray([self.src_of[np.nonzero(vid == v)[0][0]] for v in range(len(kept))])
        srcs = np.unique(vsrc)
        if len(srcs) == 1:
            return build(int(srcs[0]), kept)
        parts = []
        for s in srcs:
            vs = np.nonzero(vsrc == s)[0]
            parts.append((vs, build(int(s), [kept[v] for v in vs])))
        out = {}
        for key in parts[0][1]:
            blocks: List[Optional[torch.Tensor]] = [None] * len(kept)
            for vs, d in parts:
                n = d[key].shape[0] // len(vs)
                for j, v in enumerate(vs):
                    blocks[v] = d[key][j * n:(j + 1) * n]
            out[key] = torch.cat(blocks, 0).contiguous()
        return out

    def _segments(self, hw: int, n_valid, k_chunks, w_row_off, vec_off=None, tab_off=None, n_store=None,
                  active=None, out_col_off=0, w2_row_off=None) -> List[K.Segment]:
        """One segment per expert bucket (adjacent identical buckets merged)."""
        if not self.compact:
            return [K.Segment(row_begin=0, row_end=self.B * hw, n_valid=int(n_valid[0]), k_chunks=int(k_chunks[0]),
                              w_row_off=int(w_row_off[0]), vec_off=int(vec_off[0]) if vec_off is not None else 0,
                              tab_off=int(tab_off[0]) if tab_off is not None else 0,
                              n_store=int(n_store[0]) if n_store is not None else -1, active=True,
                              out_col_off=out_col_off, w2_row_off=int(w2_row_off[0]) if w2_row_off is not None else 0)]
        segs: List[K.Segment] = []
        st = self.layout.starts
        for e in range(self.eset.n_experts):
            if st[e + 1] == st[e]:
                continue
            s = K.Segment(row_begin=int(st[e]) * hw, row_end=int(st[e + 1]) * hw, n_valid=int(n_valid[e]),
                          k_chunks=int(k_chunks[e]), w_row_off=int(w_row_off[e]),
                          vec_off=int(vec_off[e]) if vec_off is not None else 0,
                          tab_off=int(tab_off[e]) if tab_off is not None else 0,
                          n_store=int(n_store[e]) if n_store is not None else -1,
                          active=bool(active[e]) if active is not None else True, out_col_off=out_col_off,
                          w2_row_off=int(w2_row_off[e]) if w2_row_off is not None else 0)
            if segs and segs[-1].row_end == s.row_begin and \
                    (segs[-1].n_valid, segs[-1].k_chunks, segs[-1].w_row_off, segs[-1].vec_off, segs[-1].tab_off,
                     segs[-1].n_store, segs[-1].active, segs[-1].w2_row_off) == \
                    (s.n_valid, s.k_chunks, s.w_row_off, s.vec_off, s.tab_off, s.n_store, s.active, s.w2_row_off):
                segs[-1].row_end = s.row_end
            else:
                segs.append(s)
        return segs

    def _sched(self, key, builder):
        self._label = str(key[:2])
        full = (("st", self._sid), key)
        s = self.sched.get(full)
        if s is None:
            s = builder()
            self.sched[full] = s
        return s

    def _hbm(self, nbytes: float, label: str, fn) -> None:
        """Run an HBM-bound launch group; under `profile` bracket it with CUDA events and record its ALGORITHMIC bytes
        (each operand read once, the result written once) for the roofline of the norm / gate kernels."""
        if self.profile is not None:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            self.profile.append(("hbm", e0, e1, float(nbytes), label))
        else:
            fn()

    def _gemm(self, sched: K.Schedule, a, w, out, **kw):
        extra_flops = kw.pop("extra_flops", 0.0)  # work of a fused second operand pair (not in the schedule's count)
        if self.profile is not None:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            K.grouped_gemm(a, w, out, sched, **kw)
            e1.record()
            self.profile.append(("gemm", e0, e1, sched.flops + extra_flops,
                                 f"{self._label} bn{sched.bn} tiles{sched.n_tiles} mode{kw.get('mode', 0)}"))
        else:
            K.grouped_gemm(a, w, out, sched, **kw)
        self.launches += 1
        self.flops += sched.flops + extra_flops
        res_bytes = 0 if kw.get('residual') is None else (4 if kw.get('flags', 0) & EPI_RES_F32 else 2)
        self.gemm_bytes += sched.bytes_in + sched.out_elems * ((2 if kw.get('out_mode', OUT_BF16) == OUT_BF16 else 4)
                                                               + res_bytes)

    # ---- dense (unpruned) weights ---------------------------------------------------------------
    def _dense_linear(self, name: str, lin: nn.Module, n_pad_to: int = 0) -> Dict[str, torch.Tensor]:
        """Unpruned weight + bias, stacked per weight source: a bucket's rows start at src_of * max(n_out, n_pad_to),
        its bias at src_of * n_out (_dense_offs)."""
        def weight(l):
            w = l.weight.detach()
            if w.ndim == 4:
                w = P.pack_conv_weight(w) if w.shape[-1] == 3 else w.reshape(w.shape[0], w.shape[1])
            w = w.to(self.device, BF16).contiguous()
            if n_pad_to and w.shape[0] < n_pad_to:
                w = torch.cat([w, torch.zeros(n_pad_to - w.shape[0], w.shape[1], device=self.device, dtype=BF16)], 0)
            return w

        def build():
            b = self._src_stack(lin, lambda l: l.bias.detach().to(self.device, torch.float32).contiguous()) \
                if lin.bias is not None else None
            return {"w": self._src_stack(lin, weight), "b": b}
        return self._pack(self.dense, name, build)

    def _dense_offs(self, lin: nn.Module, n_pad_to: int = 0) -> Dict[str, np.ndarray]:
        """Segment offsets of each bucket into a _dense_linear pack of `lin`."""
        n = lin.weight.shape[0]
        return dict(w_row_off=self._src_off(max(n, n_pad_to)), vec_off=self._src_off(n))

    def linear(self, name: str, lin: nn.Module, x: torch.Tensor, rows: int, k: int, ld: int, out: torch.Tensor,
               out_ld: int, hw: int, *, residual=None, res_ld=0, flags=0, active=None, out_mode=OUT_BF16,
               n_out: Optional[int] = None, out_col_off: int = 0, rowstat_out=None, colstat=None):
        """Unpruned Linear / 1x1 conv over token rows (depth-dropped buckets skipped via `active`)."""
        d = self._dense_linear(name, lin)
        n = n_out if n_out is not None else lin.weight.shape[0]
        E = self.eset.n_experts if self.compact else 1

        def build():
            bn = P.choose_bn([n], k=k)
            segs = self._segments(hw, [n] * E, [(k + 63) // 64] * E, active=active, out_col_off=out_col_off,
                                  **self._dense_offs(lin))
            return K.build_schedule(segs, bn, self.device)
        sched = self._sched(("lin", name, rows, hw), build)
        self._gemm(sched, x, d["w"], out, a_ld=ld, a_k=k, a_rows=rows, out_ld=out_ld, out_mode=out_mode, bias=d["b"],
                   rows_per_sample=hw, residual=residual, res_ld=res_ld, flags=flags, rowstat_out=rowstat_out,
                   colstat=colstat)

    def conv3x3(self, name: str, conv: nn.Module, x: Act, out: torch.Tensor, out_ld: int, *, stride=1, out_mode=OUT_BF16,
                n_pad_to=0, colstat=None):
        d = self._dense_linear(name, conv, n_pad_to=n_pad_to)
        cout, cin = conv.weight.shape[0], conv.weight.shape[1]
        Ho, Wo = x.H // stride, x.W // stride
        mode = A_CONV3X3 if stride == 1 else A_CONV3X3_S2
        E = self.eset.n_experts if self.compact else 1

        def build():
            bn = P.choose_bn([max(cout, 32)], k=9 * cin)
            segs = self._segments(Ho * Wo, [cout] * E, [(cin + 63) // 64] * E, **self._dense_offs(conv, n_pad_to))
            return K.build_schedule(segs, bn, self.device, mode=mode, Ho=Ho, Wo=Wo)
        sched = self._sched(("conv", name, x.B, x.H, x.W), build)
        self._gemm(sched, x.t, d["w"], out, a_ld=x.ld, a_k=x.C, a_rows=x.rows, mode=mode, batch=x.B, H=x.H, W=x.W,
                   k_tap_pitch=cin, out_ld=out_ld, out_mode=out_mode, bias=d["b"], rows_per_sample=Ho * Wo,
                   colstat=colstat)

    # ---- group norm ------------------------------------------------------------------------------
    def groupnorm(self, x: torch.Tensor, C: int, ld: int, B: int, hw: int, groups_full: int, gs: int, eps: float,
                  gamma: torch.Tensor, beta: torch.Tensor, affine_ld: int, out: torch.Tensor, out_ld: int, silu: bool,
                  sample_seg=None, sample_channels=None, gate=None, x1: Optional[torch.Tensor] = None, c1: int = 0,
                  ld1: int = 0, alg_elems: Optional[float] = None, cs0=None, cs1=None, raw_out=None):
        """GroupNorm [+ soft width gate] [+ SiLU] -> bf16 rows. `x` (and the optional second source `x1` = the skip half
        of an up-block torch.cat) are bf16 or fp32 rows (dtype decides). Statistics: deterministic two-stage reduction
        (no atomics), see csrc/norm.cu."""
        f32 = x.dtype == torch.float32
        assert x1 is None or (x1.dtype == torch.float32) == f32
        stats = self.buf("gnstats", B, groups_full * 2, torch.float32)
        elems = float(alg_elems) if alg_elems is not None else float(B) * hw * (C + c1)
        if cs0 is not None and (x1 is None or cs1 is not None):
            # statistics from the partials the producing GEMMs' epilogues wrote: 1/4 of the tensor's bytes (two fp32
            # planes of 1/32 of its rows) instead of a full pass
            self._hbm(elems / 32 * 8, f"gn_stats_partials C{C + c1} hw{hw}",
                      lambda: K.groupnorm_stats_from_partials(cs0, C, cs1, c1, hw // 32, B, gs, sample_channels, stats,
                                                              groups_full))
        else:
            self._hbm(elems * (4 if f32 else 2), f"gn_stats C{C + c1} hw{hw} {'f32' if f32 else 'bf16'}",
                      lambda: K.groupnorm_stats(x, C, ld, x1, c1, ld1, B, hw, gs, sample_channels, stats, groups_full,
                                                x_f32=f32))
        self._hbm(elems * ((4 if f32 else 2) + 2 + (2 if raw_out is not None else 0)),
                  f"gn_apply C{C + c1} hw{hw} {'f32' if f32 else 'bf16'} silu{int(silu)}{' +raw' if raw_out is not None else ''}",
                  lambda: K.groupnorm_apply(x, C, ld, x1, c1, ld1, out, out_ld, B, hw, gs, eps, stats, groups_full, gamma,
                                            beta, affine_ld, sample_seg, sample_channels, gate,
                                            gate.stride(0) if gate is not None else groups_full, silu, x_f32=f32,
                                            raw_out=raw_out, raw_ld=raw_out.shape[1] if raw_out is not None else 0))
        self.launches += 2

    def _colstat_new(self, B: int, H: int, W: int, C: int):
        """Partial planes for a block output of shape [B, H, W, C] if its GroupNorm statistics can be gathered in the
        producing GEMM's epilogue: every 128-row tile inside one sample."""
        hw = H * W
        if not self.gn_epi or hw % 128 != 0 or K.conv_box(W, H)[2] != 1:
            return None
        return (torch.empty(B * (hw // 32), C, device=self.device, dtype=torch.float32),
                torch.empty(B * (hw // 32), C, device=self.device, dtype=torch.float32))

    def _colstat_identity(self, cs_out, x: Act, keep_c: int, drop_mask, hw: int):
        """Depth-dropped samples take the identity path (a row copy, no GEMM epilogue): their partial rows are copied from
        the input's. Returns the planes, or None if the input has none."""
        if cs_out is None or drop_mask is None:
            return cs_out
        if x.cs is None:
            return None
        nblk = hw // 32
        for src, dst in zip(x.cs, cs_out):
            K.copy_rows_cvt(src, src.shape[1], dst, dst.shape[1], src.shape[0], keep_c, drop_mask, nblk)
        self.launches += 2
        return cs_out

    def _bf16(self, x: Act) -> torch.Tensor:
        """bf16 rows of an fp32 stream tensor, for a GEMM that reads it directly (shortcut 1x1 conv, down-sampler)."""
        if x.t is None:
            t = torch.empty(x.rows, x.C, device=self.device, dtype=BF16)
            K.cast_f32_bf16(x.f, t, x.rows * x.C)
            self.launches += 1
            x.t, x.ld = t, x.C
        return x.t

    # ---- time embedding --------------------------------------------------------------------------
    def _temb_pack(self) -> Dict[str, Any]:
        """All 22 time_emb_proj Linears in one packed matrix (+ their bias + conv1 bias folded in), per
        distinct kept-set compacted in place inside each layer's block (blocks.py:442-449)."""
        key = (("es", self._eid), "temb")
        d = self.expert.get(key)
        if d is not None:
            return d
        return self._pack(self.expert, key, self._build_temb_pack)

    def _build_temb_pack(self) -> Dict[str, Any]:
        m = self.m
        E = self.eset.n_experts if self.compact else 1
        ntot = m._temb_total
        tdim = m.time_embedding.linear_2.weight.shape[0]
        w = torch.zeros(E * ntot, tdim, device=self.device, dtype=BF16)
        b = torch.zeros(E * ntot, device=self.device, dtype=torch.float32)
        for r0 in m._resnets:
            off = m._temb_off[r0.uid]
            gs = r0.cout // r0.groups
            for e in range(E):
                r = self._src_mod(r0, int(self.src_of[e]))
                wt = r.time_emb_proj.weight.detach().to(self.device)
                bt = (r.time_emb_proj.bias.detach() + r.conv1.bias.detach()).to(self.device, torch.float32)
                if self.compact:
                    kept = np.nonzero(self.eset.width_bits(self.gate_cols[r0.uid]["w"][0])[e])[0]
                    rows = torch.as_tensor(P.expand_groups(kept, gs), device=self.device, dtype=torch.long)
                else:
                    rows = torch.arange(r.cout, device=self.device)
                w[e * ntot + off: e * ntot + off + len(rows)] = wt.index_select(0, rows).to(BF16)
                b[e * ntot + off: e * ntot + off + len(rows)] = bt.index_select(0, rows)
        return {"w": w, "b": b}

    def time_embed(self, timestep: torch.Tensor):
        m = self.m
        B = self.B
        c0 = m.config["block_out_channels"][0]
        tdim = c0 * 4
        t = timestep.to(self.device, torch.float32).reshape(-1)
        if t.numel() == 1:
            t = t.expand(B)
        t = t.contiguous()
        if self.compact:
            t = t[self._dev_index("perm")].contiguous()
        emb = self.buf("t_sin", B, c0)
        K.timestep_embedding(t, emb, B, c0)
        h = self.buf("t_h", B, tdim)
        te = self.buf("t_e", B, tdim)
        E = self.eset.n_experts if self.compact else 1
        # linear_1 + SiLU, linear_2 + SiLU (every consumer applies nonlinearity(temb) first: blocks.py:333-340)
        for name, lin, src, k, dst in (("te1", m.time_embedding.linear_1, emb, c0, h),
                                       ("te2", m.time_embedding.linear_2, h, tdim, te)):
            d = self._dense_linear(name, lin)
            sched = self._sched(("te", name), lambda: K.build_schedule(
                self._segments(1, [tdim] * E, [(k + 63) // 64] * E, **self._dense_offs(lin)), P.choose_bn([tdim]),
                self.device))
            self._gemm(sched, src, d["w"], dst, a_ld=k, a_k=k, a_rows=B, out_ld=tdim, bias=d["b"], flags=EPI_SILU,
                       rows_per_sample=1)
        pack = self._temb_pack()
        ntot = m._temb_total
        rv = self.buf("t_rowvec", B, ntot, torch.float32)

        def build():
            segs = self._segments(1, [ntot] * E, [(tdim + 63) // 64] * E, [e * ntot for e in range(E)],
                                  vec_off=[e * ntot for e in range(E)])
            return K.build_schedule(segs, 256, self.device)
        sched = self._sched(("temb_all",), build)
        self._gemm(sched, te, pack["w"], rv, a_ld=tdim, a_k=tdim, a_rows=B, out_ld=ntot, out_mode=OUT_F32,
                   bias=pack["b"], rows_per_sample=1)
        self.temb_rowvec = rv

    # ---- ResNet ------------------------------------------------------------------------------------
    def _resnet_pack(self, r: ResnetBlock2DWidthGated) -> Dict[str, Any]:
        key = (("es", self._eid), r.uid)
        d = self.expert.get(key)
        if d is not None:
            return d
        return self._pack(self.expert, key, lambda: self._build_resnet_pack(r))

    def _resnet_keep_mask(self, r: ResnetBlock2DWidthGated) -> torch.Tensor:
        """[1, cout] 0/1 mask of the channels whose GroupNorm group is kept by the (single, static) expert's code: row 0 of
        the gate matrix of the current forward, thresholded like hard_concrete. Device ops only (graph-capturable)."""
        cache = self.__dict__.setdefault("_keep_masks", {})
        mask = cache.get(r.uid)
        if mask is None:
            # computed ONCE per engine into a persistent tensor: refresh_packs() replays a captured graph, which must not
            # read the per-step gate matrix (re-allocated every forward). prune_to() drops the engine when the code changes.
            gi = self.gate_cols[r.uid]["w"][0]
            s0, e0 = self.width_starts[gi], self.width_starts[gi + 1]
            keep_g = (self.soft_arch[:1, s0:e0] >= 0.5).to(torch.float32)
            mask = keep_g.repeat_interleave(r.cout // r.groups, dim=1).contiguous()
            cache[r.uid] = mask
        return mask

    def _build_resnet_pack(self, r: ResnetBlock2DWidthGated) -> Dict[str, Any]:
        if not self.compact:
            # soft gates: every channel is kept, one variant = the dense weights (pure device ops: this builder is what
            # refresh_packs() replays, under CUDA-graph capture, after each optimizer step of the fine-tune stage)
            f32 = lambda p: p.detach().to(self.device, torch.float32).contiguous()
            beta2 = f32(r.norm2.bias).reshape(1, r.cout)
            if self.m.pruned_semantics:
                # prune() semantics on dense weights (blocks.py:451-463 deletes the channels of gated-off groups, so no
                # silu(beta) of theirs reaches conv2): with the gate at 0 the group normalises to 0 and emerges as beta,
                # hence masking beta with the (hard, per-expert) gate reproduces the sliced model exactly
                beta2 = beta2 * self._resnet_keep_mask(r)
            return {"vid": np.zeros(1, dtype=np.int64), "n1": np.asarray([r.cout]), "V": 1,
                    "w1": P.pack_conv_weight(r.conv1.weight.detach().to(self.device)).to(BF16).contiguous(),
                    "w2": P.pack_conv_weight(r.conv2.weight.detach().to(self.device)).to(BF16).contiguous(),
                    "gamma2": f32(r.norm2.weight).reshape(1, r.cout), "beta2": beta2,
                    "tab": None, "b2": f32(r.conv2.bias), "g1": f32(r.norm1.weight), "b1": f32(r.norm1.bias)}
        gs = r.cout // r.groups
        if self.compact:
            bits = self.eset.width_bits(self.gate_cols[r.uid]["w"][0])
            kept_g, vid = P.kept_variants(bits, self.eset.source)
        else:
            kept_g, vid = [np.arange(r.groups)], np.zeros(1, dtype=np.int64)
        kept_c = [P.expand_groups(k, gs) for k in kept_g]
        V = len(kept_c)
        d = {"vid": vid, "n1": np.asarray([len(k) for k in kept_c]), "V": V}
        with_tab = self.compact and not self.m.pruned_semantics

        def build(s, kept):
            rs = self._src_mod(r, s)
            w1 = P.pack_conv_weight(rs.conv1.weight.detach().to(self.device))
            w2 = P.pack_conv_weight(rs.conv2.weight.detach().to(self.device))
            g2 = rs.norm2.weight.detach().to(self.device, torch.float32)
            b2 = rs.norm2.bias.detach().to(self.device, torch.float32)
            o = {"w1": P.pack_rows(w1, kept, r.cout), "w2": P.pack_cols(w2.to(BF16), kept, 9)}
            gam = torch.zeros(len(kept), r.cout, device=self.device)
            bet = torch.zeros(len(kept), r.cout, device=self.device)
            for v, k in enumerate(kept):
                idx = torch.as_tensor(k, device=self.device, dtype=torch.long)
                gam[v, :len(k)] = g2.index_select(0, idx)
                bet[v, :len(k)] = b2.index_select(0, idx)
            o["gamma2"], o["beta2"] = gam.contiguous(), bet.contiguous()
            if with_tab:
                o["tab"] = P.border_table(rs.conv2.weight.detach().to(self.device), b2,
                                          [np.setdiff1d(np.arange(r.cout), k) for k in kept])
            return o
        d.update(self._variant_packs(vid, kept_c, build))
        if with_tab:
            tab = d["tab"]
            d["tab"] = tab.contiguous() if bool((tab != 0).any().item()) else None
        else:
            # prune() removed the gated-off channels: nothing of them reaches conv2; soft gates keep every channel
            d["tab"] = None
        f32 = lambda p: p.detach().to(self.device, torch.float32).contiguous()  # noqa: E731
        d["b2"] = self._src_stack(r, lambda rs: f32(rs.conv2.bias))
        d["g1"] = self._src_stack(r, lambda rs: f32(rs.norm1.weight))
        d["b1"] = self._src_stack(r, lambda rs: f32(rs.norm1.bias))
        return d

    def resnet(self, r: ResnetBlock2DWidthGated, x: Act, skip: Optional[Act] = None) -> Act:
        """ResnetBlock2DWidthGated / WidthDepthGated forward (blocks.py:293-371, :482-584). Input and output live on the
        fp32 residual stream (Act.f); everything a GEMM reads is bf16."""
        B, H, W, hw = x.B, x.H, x.W, x.hw
        M = x.rows
        cin = x.C + (skip.C if skip is not None else 0)
        assert cin == r.cin, f"{r.uid}: expected {r.cin} input channels, got {cin}"
        pk = self._resnet_pack(r)
        E = self.eset.n_experts if self.compact else 1
        vid = pk["vid"]
        active = self._expert_active(r.uid)
        gs_in, gs = r.cin // r.groups, r.cout // r.groups
        n1_e = pk["n1"][vid]
        cidx = self.gate_cols[r.uid]

        def build_aux():
            aux = {}
            if self.compact:
                aux["ch_in"] = self._per_pos(np.where(active, r.cin, 0))
                aux["ch_mid"] = self._per_pos(np.where(active, n1_e, 0))
                aux["seg_mid"] = self._per_pos(vid)
                aux["drop_mask"] = self._per_pos((~active).astype(np.uint8), torch.uint8) if (~active).any() else None
            return aux
        aux = self._sched(("res_aux", r.uid), build_aux)
        if self.compact:  # algorithmic element counts of the two norms (dropped samples / pruned channels excluded)
            pos = self.layout.expert_of_pos
            el_in = float(np.where(active, r.cin, 0)[pos].sum()) * hw
            el_mid = float(np.where(active, n1_e, 0)[pos].sum()) * hw
        else:
            el_in, el_mid = float(M) * r.cin, float(M) * r.cout

        # norm1 + SiLU straight from the fp32 stream; an up block's torch.cat([hidden_states, res_hidden_states], 1)
        # (blocks.py: inherited UpBlock2D.forward) is read as two sources, never materialised in fp32
        a1 = self.buf("gn_a", M, r.cin)
        # the 1x1 shortcut's bf16 A operand (the concatenated, un-normalised input) is written by the same pass
        xin16 = self.buf("cat", M, r.cin) if r.conv_shortcut is not None else None
        if skip is not None:
            self.groupnorm(x.f, x.C, x.C, B, hw, r.groups, gs_in, r.eps, pk["g1"], pk["b1"], r.cin, a1, r.cin, True,
                           sample_seg=self._src_seg(), sample_channels=aux.get("ch_in"), x1=skip.f, c1=skip.C,
                           ld1=skip.C, alg_elems=el_in, cs0=x.cs, cs1=skip.cs, raw_out=xin16)
        else:
            self.groupnorm(x.f, x.C, x.C, B, hw, r.groups, gs_in, r.eps, pk["g1"], pk["b1"], r.cin, a1, r.cin, True,
                           sample_seg=self._src_seg(), sample_channels=aux.get("ch_in"), alg_elems=el_in, cs0=x.cs,
                           raw_out=xin16)
        # conv1 (N-compacted) + time embedding (+ conv1/time biases, folded into the row vector)
        h1 = self.buf("res_h1", M, r.cout)

        def build_c1():
            bn = P.choose_bn(list(pk["n1"]), k=9 * r.cin)
            segs = self._segments(hw, n1_e, [(r.cin + 63) // 64] * E, vid * r.cout, active=active,
                                  n_store=[min(P.round_up(int(n), 64), r.cout) for n in n1_e])
            return K.build_schedule(segs, bn, self.device, mode=A_CONV3X3, Ho=H, Wo=W)
        sched = self._sched(("res_c1", r.uid, H, W), build_c1)
        rv = self.temb_rowvec[:, self.m._temb_off[r.uid]:]
        # norm2's statistics (of the bf16 values conv1 stores) come from conv1's epilogue too: no statistics pass over h1
        cs_h1 = None
        if (self.gn_epi and hw % 128 == 0 and K.conv_box(W, H)[2] == 1
                and os.environ.get("APTP_GN_EPI_BF16", "1") != "0"):
            nblk = B * (hw // 32)
            cs_h1 = (self.buf("cs_h1_sum", nblk, r.cout, torch.float32), self.buf("cs_h1_sq", nblk, r.cout, torch.float32))
        self._gemm(sched, a1, pk["w1"], h1, a_ld=r.cin, a_k=r.cin, a_rows=M, mode=A_CONV3X3, batch=B, H=H, W=W,
                   k_tap_pitch=r.cin, out_ld=r.cout, rowvec=rv, rowvec_ld=self.m._temb_total, rows_per_sample=hw,
                   colstat=cs_h1)
        # width gate (soft: fused multiplier) + norm2 + SiLU on the compacted tensor
        a2 = self.buf("gn_b", M, r.cout)
        gate = self._soft_gate(cidx["w"][0]) if not self.compact else None
        self.groupnorm(h1, r.cout, r.cout, B, hw, r.groups, gs, r.eps, pk["gamma2"], pk["beta2"], r.cout, a2, r.cout,
                       True, sample_seg=aux.get("seg_mid"),
                       sample_channels=aux.get("ch_mid"), gate=gate, alg_elems=el_mid, cs0=cs_h1)
        # shortcut: 1x1 conv over the bf16 copy of the (concatenated) input, written fp32 and added in place by conv2
        out = torch.empty(M, r.cout, device=self.device, dtype=torch.float32)
        # ... unless conv2 can take it as extra K steps of its own tiles (halo-mode convs: 8 x 16-pixel boxes, 2-SM scheme)
        fuse_sc = (r.conv_shortcut is not None and W % 8 == 0 and H % 16 == 0
                   and 9 * r.cout >= int(os.environ.get("APTP_GEMM_2SM_MINK", "1280") or 1280)
                   and os.environ.get("APTP_SC_FUSE", "1") != "0" and os.environ.get("APTP_CONV_HALO", "1") != "0"
                   and os.environ.get("APTP_GEMM_1SM", "0") != "1")
        sc_kw = {}
        if fuse_sc:
            dsc = self._dense_linear("sc." + r.uid, r.conv_shortcut)
            bkey = ("b2sc", r.uid)
            b2sc = self.dense.get(bkey)
            if b2sc is None:
                b2sc = self._pack(self.dense, bkey, lambda: (pk["b2"] + dsc["b"]).contiguous())
            rows_act = float(active[self.layout.expert_of_pos].sum()) * hw if self.compact else float(M)
            sc_kw = dict(a2=xin16, a2_ld=r.cin, a2_k=r.cin, w2=dsc["w"], extra_flops=2.0 * rows_act * r.cin * r.cout)
            res, res_ld = None, 0
        elif r.conv_shortcut is not None:
            xin_ld = r.cin
            self.linear("sc." + r.uid, r.conv_shortcut, xin16, M, r.cin, xin_ld, out, r.cout, hw, active=active,
                        out_mode=OUT_F32)
            res, res_ld = out, r.cout
        else:
            assert skip is None
            res, res_ld = x.f, x.C
        # conv2 (K-compacted) + bias + border table + fp32 residual -> fp32 stream

        def build_c2():
            bn = P.choose_bn([r.cout], k=9 * int(max(pk["n1"])))
            tab_off = vid * 9 * r.cout
            # conv2 bias and the fused shortcut's weight rows / bias are stacked per weight source
            segs = self._segments(hw, [r.cout] * E, [(int(n) + 63) // 64 for n in n1_e], vid * r.cout,
                                  vec_off=self._src_off(r.cout), tab_off=tab_off, active=active,
                                  w2_row_off=self._src_off(r.cout))
            return K.build_schedule(segs, bn, self.device, mode=A_CONV3X3, Ho=H, Wo=W)
        sched = self._sched(("res_c2", r.uid, H, W), build_c2)
        cs_out = self._colstat_new(B, H, W, r.cout)
        if cs_out is not None and self.compact and aux["drop_mask"] is not None and x.cs is None:
            cs_out = None  # dropped samples would need the input's partial rows
        self._gemm(sched, a2, pk["w2"], out, a_ld=r.cout, a_k=r.cout, a_rows=M, mode=A_CONV3X3, batch=B, H=H, W=W,
                   k_tap_pitch=r.cout, out_ld=r.cout, out_mode=OUT_F32, bias=b2sc if fuse_sc else pk["b2"], residual=res,
                   res_ld=res_ld, flags=EPI_RES_F32 if res is not None else 0, rows_per_sample=hw, border_tab=pk["tab"],
                   tab_ld=r.cout, colstat=cs_out, **sc_kw)
        # depth gate: the non-skip part of the input is the identity branch (blocks.py:485-495)
        if r.depth_gate is not None:
            keep_c = x.C if skip is not None else x.C - (r.skip_connection_dim or 0)
            if self.compact:
                if aux["drop_mask"] is not None:  # dropped experts: identity on the (non-skip) input
                    K.copy_rows_cvt(x.f, x.C, out, r.cout, M, keep_c, aux["drop_mask"], hw)
                    self.launches += 1
                    cs_out = self._colstat_identity(cs_out, x, keep_c, aux["drop_mask"], hw)
            else:
                K.depth_lerp_f32(x.f, x.C, out, r.cout, out, r.cout, M, keep_c, self._soft_depth(cidx["d"]), hw)
                self.launches += 1
                cs_out = None  # the lerp changes the stored values after the epilogue gathered its statistics
        return Act(None, B, H, W, r.cout, f=out, cs=cs_out)

    # ---- transformer -------------------------------------------------------------------------------
    @staticmethod
    def _pack_vec(vec: torch.Tensor, kept: List[np.ndarray], n_pad: int) -> torch.Tensor:
        """Per-variant compaction of a per-output-row vector, laid out like P.pack_rows lays out the rows."""
        out = torch.zeros(len(kept) * n_pad, device=vec.device, dtype=torch.float32)
        for v, rows in enumerate(kept):
            idx = torch.as_tensor(rows, device=vec.device, dtype=torch.long)
            out[v * n_pad: v * n_pad + len(rows)] = vec.index_select(0, idx)
        return out

    def _attn_pack(self, uid: str, attn: _Attention, gate_idx: int, ln: nn.LayerNorm) -> Dict[str, Any]:
        """Compacted q/k/v/out weights per kept-head variant. The LayerNorm in front of the attention
        (BasicTransformerBlock.norm1 / norm2, blocks.py:782, :808-810) is FOLDED into the projections that read the
        normalised tokens (q, k, v of self-attention; q of cross-attention): weights W*gamma, bias W@beta, plus the
        column sums of the bf16 weights the epilogue needs (APTP_EPI_LN_FOLD)."""
        key = (("es", self._eid), uid)
        d = self.expert.get(key)
        if d is not None:
            return d
        C = attn.dim
        is_cross = attn.ctx_dim is not None
        if self.compact:
            kept_h, vid = P.kept_variants(self.eset.width_bits(gate_idx), self.eset.source)
        else:
            kept_h, vid = [np.arange(attn.heads)], np.zeros(1, dtype=np.int64)
        kept_c = [P.expand_groups(k, 64) for k in kept_h]
        d = {"vid": vid, "nh": np.asarray([len(k) for k in kept_h]), "V": len(kept_h)}

        def build(s, kept):
            at, ls = self._src_mod(attn, s), self._src_mod(ln, s)
            gam = ls.weight.detach().to(self.device, torch.float32)
            bet = ls.bias.detach().to(self.device, torch.float32)
            if not self.ln_fold:
                gam, bet = torch.ones_like(gam), torch.zeros_like(bet)
            o = {}
            for nm, lin in (("q", at.to_q), ("k", at.to_k), ("v", at.to_v)):
                w = lin.weight.detach().to(self.device, torch.float32)
                if nm == "q" or not is_cross:
                    o["w" + nm] = P.pack_rows(w * gam[None, :], kept, C)
                    o["b" + nm] = self._pack_vec(w @ bet, kept, C)
                else:
                    o["w" + nm] = P.pack_rows(w, kept, C)
            o["wo"] = P.pack_cols(at.to_out[0].weight.detach().to(self.device, BF16), kept, 1)
            return o
        d.update(self._variant_packs(vid, kept_c, build))
        if is_cross:
            d["cq"] = d["wq"].float().sum(1).contiguous()
            d["wkv"] = torch.cat([d["wk"], d["wv"]], 0).contiguous()
        else:
            d["wqkv"] = torch.cat([d["wq"], d["wk"], d["wv"]], 0).contiguous()
            d["bqkv"] = torch.cat([d["bq"], d["bk"], d["bv"]], 0).contiguous()
            d["cqkv"] = d["wqkv"].float().sum(1).contiguous()
        d["bo"] = self._src_stack(attn, lambda at: at.to_out[0].bias.detach().to(self.device, torch.float32).contiguous())
        self.expert[key] = d
        return d

    def _ff_pack(self, uid: str, ff: _FeedForward, gate_idx: int, ln: nn.LayerNorm) -> Dict[str, Any]:
        """GEGLU proj / net.2 per kept-FF-group variant; norm3 (blocks.py:821) is folded into the GEGLU projection."""
        key = (("es", self._eid), uid)
        d = self.expert.get(key)
        if d is not None:
            return d
        proj = ff.net[0].proj
        inner = proj.weight.shape[0] // 2
        C = proj.weight.shape[1]
        gw = ff.net[0].gate.width
        gs = inner // gw
        if self.compact:
            kept_g, vid = P.kept_variants(self.eset.width_bits(gate_idx), self.eset.source)
        else:
            kept_g, vid = [np.arange(gw)], np.zeros(1, dtype=np.int64)
        kept_c = [P.expand_groups(k, gs) for k in kept_g]
        nf = np.asarray([len(k) for k in kept_c])
        bn = P.choose_bn(list(nf), geglu=True, k=C)
        half = bn // 2
        rows_pad = ((inner + half - 1) // half) * bn
        d = {"vid": vid, "nf": nf, "V": len(kept_c), "bn": bn, "rows_pad": rows_pad, "inner": inner, "gs": gs}
        d.update(self._variant_packs(vid, kept_c, lambda s, kept: self._ff_blocks(
            self._src_mod(ff, s), self._src_mod(ln, s), kept, C, inner, bn, rows_pad)))
        d["sp"] = d["wp"].float().sum(1).contiguous()
        d["b2"] = self._src_stack(ff, lambda f: f.net[2].bias.detach().to(self.device, torch.float32).contiguous())
        self.expert[key] = d
        return d

    def _ff_blocks(self, ff: _FeedForward, ln: nn.LayerNorm, kept_c: List[np.ndarray], C: int, inner: int, bn: int,
                   rows_pad: int) -> Dict[str, torch.Tensor]:
        """GEGLU proj (norm3 folded in) and net.2 blocks of the variants `kept_c`, from the weights of `ff` / `ln`."""
        half = bn // 2
        V = len(kept_c)
        proj = ff.net[0].proj
        w = proj.weight.detach().to(self.device, torch.float32)
        gam = ln.weight.detach().to(self.device, torch.float32)
        bet = ln.bias.detach().to(self.device, torch.float32)
        if not self.ln_fold:
            gam, bet = torch.ones_like(gam), torch.zeros_like(bet)
        b = proj.bias.detach().to(self.device, torch.float32) + w @ bet
        w = w * gam[None, :]
        wp = torch.zeros(V * rows_pad, C, device=self.device, dtype=BF16)
        bp = torch.zeros(V * rows_pad, device=self.device, dtype=torch.float32)
        for v, cols in enumerate(kept_c):
            idx = torch.as_tensor(cols, device=self.device, dtype=torch.long)
            n = len(cols)
            nt = (n + half - 1) // half
            # tile t holds output columns [t*half, (t+1)*half): rows [t*bn, t*bn+half) = h, next half = g
            hsel = torch.zeros(nt * half, C, device=self.device, dtype=BF16)
            gsel = torch.zeros(nt * half, C, device=self.device, dtype=BF16)
            hsel[:n] = w.index_select(0, idx).to(BF16)
            gsel[:n] = w.index_select(0, idx + inner).to(BF16)
            hb = torch.zeros(nt * half, device=self.device)
            gb = torch.zeros(nt * half, device=self.device)
            hb[:n] = b.index_select(0, idx)
            gb[:n] = b.index_select(0, idx + inner)
            blk = torch.stack([hsel.view(nt, half, C), gsel.view(nt, half, C)], dim=1).reshape(nt * bn, C)
            bblk = torch.stack([hb.view(nt, half), gb.view(nt, half)], dim=1).reshape(nt * bn)
            wp[v * rows_pad: v * rows_pad + nt * bn] = blk
            bp[v * rows_pad: v * rows_pad + nt * bn] = bblk
        return {"wp": wp, "bp": bp, "w2": P.pack_cols(ff.net[2].weight.detach().to(self.device, BF16), kept_c, 1)}

    def _layernorm(self, tok: torch.Tensor, ln: nn.LayerNorm, M: int, C: int, hw: int, active: np.ndarray) -> torch.Tensor:
        """Un-folded LayerNorm pass (APTP_LN_FOLD=0 only): tok -> normalised bf16 rows."""
        if len(self.srcs) > 1:
            raise NotImplementedError("APTP_LN_FOLD=0 has one LayerNorm affine per launch: it cannot serve several "
                                      "weight sources in one batch")
        key = ("ln_affine", id(ln))
        d = self.dense.get(key)
        if d is None:
            d = (ln.weight.detach().to(self.device, torch.float32).contiguous(),
                 ln.bias.detach().to(self.device, torch.float32).contiguous())
            self.dense[key] = d
        xn = self.buf("ln", M, C)
        act = self._sched(("ln_act", id(ln)), lambda: self._per_pos(active.astype(np.uint8), torch.uint8)
                          if (self.compact and (~active).any()) else None)
        n_act = float(active[self.layout.expert_of_pos].sum()) if self.compact else float(self.B)
        self._hbm(n_act * hw * C * 4, f"layernorm C{C} hw{hw}",
                  lambda: K.layernorm(tok, C, xn, C, M, C, ln.eps, d[0], d[1], act, hw))
        self.launches += 1
        return xn

    def _ln_rowstats(self, part: torch.Tensor, M: int, C: int, eps: float, hw: int) -> torch.Tensor:
        """(mean, rstd) per token row from the partial sums the producing GEMM wrote: 8 bytes per row for the LN-fold
        epilogue (a 4-byte-per-element pass over `tok` in the reference's three LayerNorms becomes this)."""
        rs = self.buf("ln_rs", M, 2, torch.float32)
        self._hbm(float(M) * (part.shape[1] * 8 + 8), f"ln_rowstats C{C} hw{hw}",
                  lambda: K.ln_rowstats(part, M, C, eps, rs))
        self.launches += 1
        return rs

    def _attention(self, uid: str, attn: _Attention, gate_idx: int, ln: nn.LayerNorm, part: torch.Tensor,
                   tok: torch.Tensor, B: int, hw: int, C: int, active: np.ndarray, ctx: Optional[torch.Tensor],
                   n_ctx: int, want_stats: bool = True):
        """LayerNorm + GatedAttention + HeadGatedAttnProcessor2 (blocks.py:782-806 / :808-819, :194-280); the output is
        accumulated into `tok`. `part` holds the per-row LayerNorm partial sums of `tok` on entry (written by the GEMM
        that produced it) and, with want_stats, those of the updated `tok` on exit."""
        pk = self._attn_pack(uid, attn, gate_idx, ln)
        E = self.eset.n_experts if self.compact else 1
        vid, nh_e = pk["vid"], pk["nh"][pk["vid"]]
        M = B * hw
        is_cross = ctx is not None
        n_kv = n_ctx if is_cross else hw
        Mkv = B * n_kv
        gate = self._soft_gate(gate_idx) if not self.compact else None
        kq = C
        kkv = attn.ctx_dim if is_cross else C
        qkv = self.buf("qkv_q", M, C) if is_cross else self.buf("qkv", M, 3 * C)
        kvb = self.buf("qkv_kv", Mkv, 2 * C) if is_cross else None

        def build():
            bn = P.choose_bn([int(n) * 64 for n in pk["nh"]], k=C)
            s = {}
            nv = [int(n) * 64 for n in nh_e]
            if is_cross:
                s["q"] = K.build_schedule(self._segments(hw, nv, [(kq + 63) // 64] * E, vid * C, vec_off=vid * C,
                                                         active=active), bn, self.device)
                segs = []
                for j in range(2):
                    segs += self._segments(n_kv, nv, [(kkv + 63) // 64] * E, vid * C + j * pk["V"] * C, active=active,
                                           out_col_off=j * C)
                s["kv"] = K.build_schedule(segs, bn, self.device)
            else:
                segs = []
                for j in range(3):
                    off = vid * C + j * pk["V"] * C
                    segs += self._segments(hw, nv, [(kq + 63) // 64] * E, off, vec_off=off, active=active,
                                           out_col_off=j * C)
                s["qkv"] = K.build_schedule(segs, bn, self.device)
            s["o"] = K.build_schedule(self._segments(hw, [C] * E, [int(n) for n in nh_e], vid * C,
                                                     vec_off=self._src_off(C), active=active),
                                      P.choose_bn([C], k=64 * int(max(pk["nh"]))), self.device)
            heads = np.where(active, nh_e, 0) if self.compact else np.asarray([attn.heads])
            s["heads"] = self._per_pos(heads) if self.compact else torch.full((B,), attn.heads, device=self.device,
                                                                             dtype=torch.int32)
            s["max_heads"] = int(heads.max()) if len(heads) else 0
            s["heads_total"] = float(np.asarray(heads)[self.layout.expert_of_pos].sum()) if self.compact \
                else float(attn.heads * B)
            return s
        s = self._sched(("attn", uid, hw, n_kv), build)
        gkw = dict(gate=gate, gate_ld=gate.stride(0), gate_group=64) if gate is not None else {}
        if self.ln_fold:
            a_in = tok
            lnkw = dict(ln_rowstats=self._ln_rowstats(part, M, C, ln.eps, hw))
            lq = dict(bias=pk["bq"], ln_colsum=pk["cq"]) if is_cross else dict(bias=pk["bqkv"], ln_colsum=pk["cqkv"])
        else:
            a_in = self._layernorm(tok, ln, M, C, hw, active)
            lnkw, lq, want_stats = {}, {}, False
        if is_cross:
            self._gemm(s["q"], a_in, pk["wq"], qkv, a_ld=C, a_k=C, a_rows=M, out_ld=C, rows_per_sample=hw,
                       **lq, **lnkw, **gkw)
            self._gemm(s["kv"], ctx, pk["wkv"], kvb, a_ld=kkv, a_k=kkv, a_rows=Mkv, out_ld=2 * C, rows_per_sample=n_kv,
                       **gkw)
            q, ldq, kk, vv, ldkv = qkv, C, kvb, kvb[:, C:], 2 * C
        else:
            self._gemm(s["qkv"], a_in, pk["wqkv"], qkv, a_ld=C, a_k=C, a_rows=M, out_ld=3 * C, rows_per_sample=hw,
                       **lq, **lnkw, **gkw)
            q, ldq, kk, vv, ldkv = qkv, 3 * C, qkv[:, C:], qkv[:, 2 * C:], 3 * C
        o = self.buf("attn_o", M, C)
        if s["max_heads"] > 0:
            fl = 4.0 * hw * n_kv * 64 * s["heads_total"]
            if self.profile is not None:
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
            K.attention(q, ldq, kk, ldkv, vv, ldkv, o, C, B, hw, n_kv, s["heads"], s["max_heads"], 1.0 / 8.0)
            if self.profile is not None:
                e1.record()
                self.profile.append(("attn", e0, e1, fl, f"{uid} nq{hw} nkv{n_kv}"))
            self.launches += 1
            self.flops += fl
        # to_out (K-compacted to the kept heads) + bias + residual, in place on the token stream; its epilogue also
        # writes the LayerNorm partial sums of the updated rows for the next folded LayerNorm
        self._gemm(s["o"], o, pk["wo"], tok, a_ld=C, a_k=C, a_rows=M, out_ld=C, bias=pk["bo"], residual=tok, res_ld=C,
                   rows_per_sample=hw, rowstat_out=part if want_stats else None)

    def transformer(self, t: Transformer2DModelWidthGated, x: Act) -> Act:
        """Transformer2DModelWidth(Depth)Gated.forward (blocks.py:1139-1355) incl. the
        BasicTransformerBlockWidthGated body (blocks.py:763-851)."""
        B, H, W, hw, C = x.B, x.H, x.W, x.hw, x.C
        M = x.rows
        tb = t.transformer_blocks[0]
        cidx = self.gate_cols[t.uid]
        active = self._expert_active(t.uid)
        E = self.eset.n_experts if self.compact else 1
        key = ("tr_dense", t.uid)
        dn = self.dense.get(key)
        if dn is None:
            f32 = lambda p: p.detach().to(self.device, torch.float32).contiguous()
            dn = {"g": self._src_stack(t, lambda ts: f32(ts.norm.weight)),
                  "b": self._src_stack(t, lambda ts: f32(ts.norm.bias))}
            for i, ln in enumerate((tb.norm1, tb.norm2, tb.norm3)):
                dn[f"lg{i}"], dn[f"lb{i}"] = f32(ln.weight), f32(ln.bias)
            self.dense[key] = dn

        def build_aux():
            aux = {"ch": None, "act": None, "drop": None}
            if self.compact and (~active).any():
                aux["ch"] = self._per_pos(np.where(active, C, 0))
                aux["act"] = self._per_pos(active.astype(np.uint8), torch.uint8)
                aux["drop"] = self._per_pos((~active).astype(np.uint8), torch.uint8)
            return aux
        aux = self._sched(("tr_aux", t.uid), build_aux)
        gs = C // t.groups
        xn = self.buf("ln", M, C)
        n_act = float(active[self.layout.expert_of_pos].sum()) if self.compact else float(B)
        self.groupnorm(x.f, C, C, B, hw, t.groups, gs, 1e-6, dn["g"], dn["b"], C, xn, C, False,
                       sample_seg=self._src_seg(), sample_channels=aux["ch"], alg_elems=n_act * hw * C, cs0=x.cs)
        tok = self.buf("tok", M, C)
        # LayerNorm statistics travel with the token stream: every GEMM that writes `tok` also writes per-row
        # (sum, sumsq) partials per 32-column chunk, and the three LayerNorms of the block (norm1/2/3, blocks.py:782,
        # :808-810, :821) are folded into the GEMMs that consume them -- no LayerNorm pass over HBM at all
        part = self.buf("ln_part", M, (C // 32) * 2, torch.float32).view(M, C // 32, 2)
        self.linear("pi." + t.uid, t.proj_in, xn, M, C, C, tok, C, hw, active=active,
                    rowstat_out=part if self.ln_fold else None)
        # self-attention, cross-attention
        self._attention(t.uid + ".a1", tb.attn1, cidx["w"][0], tb.norm1, part, tok, B, hw, C, active, None, 0)
        self._attention(t.uid + ".a2", tb.attn2, cidx["w"][1], tb.norm2, part, tok, B, hw, C, active, self.ctx, self.n_ctx)
        # feed-forward: norm3 folded into GEGLU (N-compacted, gated), then Linear (K-compacted) + residual
        fk = self._ff_pack(t.uid + ".ff", tb.ff, cidx["w"][2], tb.norm3)
        vid, nf_e = fk["vid"], fk["nf"][fk["vid"]]
        inner = fk["inner"]
        ffb = self.buf("ff", M, inner)

        def build_ff():
            s = {}
            s["p"] = K.build_schedule(
                self._segments(hw, nf_e, [(C + 63) // 64] * E, vid * fk["rows_pad"], vec_off=vid * fk["rows_pad"],
                               n_store=[min(P.round_up(int(n), 64), inner) for n in nf_e], active=active),
                fk["bn"], self.device, geglu=True)
            s["o"] = K.build_schedule(
                self._segments(hw, [C] * E, [(int(n) + 63) // 64 for n in nf_e], vid * C, vec_off=self._src_off(C),
                               active=active),
                P.choose_bn([C], k=int(max(fk["nf"]))), self.device)
            return s
        s = self._sched(("ff", t.uid, hw), build_ff)
        gate = self._soft_gate(cidx["w"][2]) if not self.compact else None
        gkw = dict(gate=gate, gate_ld=gate.stride(0), gate_group=fk["gs"]) if gate is not None else {}
        if self.ln_fold:
            self._gemm(s["p"], tok, fk["wp"], ffb, a_ld=C, a_k=C, a_rows=M, out_ld=inner, bias=fk["bp"], flags=EPI_GEGLU,
                       rows_per_sample=hw, ln_colsum=fk["sp"],
                       ln_rowstats=self._ln_rowstats(part, M, C, tb.norm3.eps, hw), **gkw)
        else:
            self._gemm(s["p"], self._layernorm(tok, tb.norm3, M, C, hw, active), fk["wp"], ffb, a_ld=C, a_k=C, a_rows=M,
                       out_ld=inner, bias=fk["bp"], flags=EPI_GEGLU, rows_per_sample=hw, **gkw)
        self._gemm(s["o"], ffb, fk["w2"], tok, a_ld=inner, a_k=inner, a_rows=M, out_ld=C, bias=fk["b2"], residual=tok,
                   res_ld=C, rows_per_sample=hw)
        # proj_out + residual: back onto the fp32 stream
        out = torch.empty(M, C, device=self.device, dtype=torch.float32)
        cs_out = self._colstat_new(B, H, W, C)
        if cs_out is not None and self.compact and aux["drop"] is not None and x.cs is None:
            cs_out = None
        self.linear("po." + t.uid, t.proj_out, tok, M, C, C, out, C, hw, residual=x.f, res_ld=C, active=active,
                    out_mode=OUT_F32, flags=EPI_RES_F32, colstat=cs_out)
        if t.depth_gate is not None:
            if self.compact:
                if aux["drop"] is not None:
                    K.copy_rows_cvt(x.f, C, out, C, M, C, aux["drop"], hw)
                    self.launches += 1
                    cs_out = self._colstat_identity(cs_out, x, C, aux["drop"], hw)
            else:
                K.depth_lerp_f32(x.f, C, out, C, out, C, M, C, self._soft_depth(cidx["d"]), hw)
                self.launches += 1
                cs_out = None
        return Act(None, B, H, W, C, f=out, cs=cs_out)

    # ---- samplers ----------------------------------------------------------------------------------
    def downsample(self, s: _Sampler, x: Act) -> Act:
        out = torch.empty(x.rows // 4, x.C, device=self.device, dtype=torch.float32)
        x16 = Act(self._bf16(x), x.B, x.H, x.W, x.C)
        cs = self._colstat_new(x.B, x.H // 2, x.W // 2, x.C)
        self.conv3x3("ds.%d" % id(s), s.conv, x16, out, x.C, stride=2, out_mode=OUT_F32, colstat=cs)
        return Act(None, x.B, x.H // 2, x.W // 2, x.C, f=out, cs=cs)

    def upsample(self, s: _Sampler, x: Act) -> Act:
        up = self.buf("up", x.rows * 4, x.C)
        K.upsample2x_cvt(x.f, up, x.B, x.H, x.W, x.C)
        self.launches += 1
        xu = Act(up, x.B, x.H * 2, x.W * 2, x.C)
        out = torch.empty(xu.rows, x.C, device=self.device, dtype=torch.float32)
        cs = self._colstat_new(xu.B, xu.H, xu.W, x.C)
        self.conv3x3("us.%d" % id(s), s.conv, xu, out, x.C, out_mode=OUT_F32, colstat=cs)
        return Act(None, xu.B, xu.H, xu.W, x.C, f=out, cs=cs)

    # ---- CUDA-graph replay of the hard-gate forward -------------------------------------------------
    def run_graphed(self, sample: torch.Tensor, timestep, ctx: torch.Tensor, want_taps: bool = False):
        """`run` behind a CUDA graph. One forward is ~500 launches of this library; with hard gates their schedule
        depends only on the tensor shapes and on the CONTENT of the architecture codes, so the third forward with
        the same key is captured once and replayed afterwards (inputs are copied into the graph's static buffers,
        the prediction is returned as a fresh tensor; block taps are views of graph-owned buffers, valid until the
        next forward with the same key). Soft gates (training) and profiling runs stay eager.
        APTP_CUDA_GRAPH=0 disables the replay."""
        B = sample.shape[0]
        if (os.environ.get("APTP_CUDA_GRAPH", "1") == "0" or self.profile is not None or not torch.is_tensor(timestep)
                or torch.cuda.is_current_stream_capturing()):
            return self.run(sample, timestep, ctx, want_taps)
        self._prepare_gates(B)  # the one host sync per set_structure happens here, outside any capture
        if not self.compact:
            return self.run(sample, timestep, ctx, want_taps)
        key = (tuple(sample.shape), sample.dtype, tuple(timestep.shape), timestep.dtype, tuple(ctx.shape), ctx.dtype,
               self.eset.key(), self.layout.starts.tobytes(), bool(want_taps))
        entry = self.graphs.get(key)
        if entry is None:
            seen = self.graph_seen.get(key, 0)
            if len(self.graph_seen) >= 64 and key not in self.graph_seen:
                self.graph_seen.pop(next(iter(self.graph_seen)))
            self.graph_seen[key] = seen + 1
            if seen < 2:  # two eager forwards build every schedule / packed weight and warm the allocator
                return self.run(sample, timestep, ctx, want_taps)
            if len(self.graphs) >= 4:  # bounded: every graph pins its own activation pool
                self.graphs.pop(next(iter(self.graphs)))
            st_s, st_t, st_c = sample.clone(), timestep.clone(), ctx.clone()
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            with _graph_capture(g):
                y, taps = self.run(st_s, st_t, st_c, want_taps)
            # the captured kernels read this state's schedules and packed weights: the graph keeps them alive even if
            # the LRU caches above drop the state in the meantime
            keep = ([v for k, v in self.sched.items() if isinstance(k, tuple) and k[0] == ("st", self._sid)],
                    [v for k, v in self.expert.items() if isinstance(k, tuple) and k[0] == ("es", self._eid)])
            entry = (g, st_s, st_t, st_c, y, taps, self.flops, self.launches, self.gemm_bytes, keep)
            self.graphs[key] = entry
        g, st_s, st_t, st_c, y, taps, self.flops, self.launches, self.gemm_bytes, _keep = entry
        st_s.copy_(sample, non_blocking=True)
        st_t.copy_(timestep, non_blocking=True)
        st_c.copy_(ctx, non_blocking=True)
        g.replay()
        return y.clone(), taps

    # ---- whole forward -----------------------------------------------------------------------------
    def run(self, sample: torch.Tensor, timestep, ctx: torch.Tensor, want_taps: bool = False):
        m = self.m
        B, cin, H, W = sample.shape
        self.B = B
        self.flops = 0.0
        self.gemm_bytes = 0.0
        self.launches = 0
        self._prepare_gates(B)
        if not torch.is_tensor(timestep):
            timestep = torch.tensor([float(timestep)], device=self.device)
        sample = sample.to(torch.float32)
        ctx = ctx.to(self.device)
        if self.compact:
            perm = self._dev_index("perm")
            sample = sample.index_select(0, perm)
            ctx = ctx.index_select(0, perm)
        sample = sample.contiguous()
        ctx = ctx.contiguous()
        self.n_ctx = ctx.shape[1]
        cdim = ctx.shape[2]
        ctx16 = self.buf("ctx", B * self.n_ctx, cdim)
        if ctx.dtype == BF16:
            ctx16.copy_(ctx.reshape(B * self.n_ctx, cdim))
        else:
            K.cast_f32_bf16(ctx.to(torch.float32), ctx16, B * self.n_ctx * cdim)
        self.launches += 1
        self.ctx = ctx16
        self.time_embed(timestep)
        # conv_in as im2col (K = 36 -> 64) + GEMM
        c0 = m.config["block_out_channels"][0]
        col = self.buf("im2col", B * H * W, 64)
        K.im2col_input(sample, col, B, cin, H, W)
        self.launches += 1
        d = self.dense.get("conv_in")
        if d is None:
            def conv_in_w(conv):
                wp = torch.zeros(c0, 64, device=self.device, dtype=BF16)
                wp[:, :9 * cin] = conv.weight.detach().to(self.device).permute(0, 2, 3, 1).reshape(c0, 9 * cin).to(BF16)
                return wp
            d = {"w": self._src_stack(m.conv_in, conv_in_w),
                 "b": self._src_stack(m.conv_in, lambda c: c.bias.detach().to(self.device, torch.float32).contiguous())}
            self.dense["conv_in"] = d
        x0 = torch.empty(B * H * W, c0, device=self.device, dtype=torch.float32)
        E = self.eset.n_experts if self.compact else 1
        sched = self._sched(("conv_in", H, W), lambda: K.build_schedule(
            self._segments(H * W, [c0] * E, [1] * E, **self._dense_offs(m.conv_in)), P.choose_bn([c0]), self.device))
        cs0 = self._colstat_new(B, H, W, c0)
        self._gemm(sched, col, d["w"], x0, a_ld=64, a_k=64, a_rows=B * H * W, out_ld=c0, out_mode=OUT_F32, bias=d["b"],
                   rows_per_sample=H * W, colstat=cs0)
        x = Act(None, B, H, W, c0, f=x0, cs=cs0)
        skips = [x]
        tap_acts = []
        for blk in m.down_blocks:
            x, outs = blk.forward(self, x)
            skips += list(outs)
            tap_acts.append(x)
        x = m.mid_block.forward(self, x)
        tap_acts.append(x)
        for blk in m.up_blocks:
            x = blk.forward(self, x, skips)
            tap_acts.append(x)
        # conv_norm_out + SiLU + conv_out (fp32 NCHW result)
        key = "out_norm"
        dn = self.dense.get(key)
        if dn is None:
            dn = {"g": self._src_stack(m.conv_norm_out, lambda n: n.weight.detach().to(self.device, torch.float32)),
                  "b": self._src_stack(m.conv_norm_out, lambda n: n.bias.detach().to(self.device, torch.float32))}
            dn = {k: v.contiguous() for k, v in dn.items()}
            self.dense[key] = dn
        groups = m.config["norm_num_groups"]
        a = self.buf("gn_a", x.rows, x.C)
        self.groupnorm(x.f, x.C, x.C, B, x.hw, groups, x.C // groups, m.config["norm_eps"], dn["g"], dn["b"], x.C, a,
                       x.C, True, sample_seg=self._src_seg(), cs0=x.cs)
        cout = m.config["out_channels"]
        y = torch.empty(B, cout, x.H, x.W, device=self.device, dtype=torch.float32)
        dco = self._dense_linear("conv_out", m.conv_out, n_pad_to=32)
        sched = self._sched(("conv_out", x.H, x.W), lambda: K.build_schedule(
            self._segments(x.hw, [cout] * E, [(x.C + 63) // 64] * E, **self._dense_offs(m.conv_out, 32)), 32,
            self.device, mode=A_CONV3X3, Ho=x.H, Wo=x.W))
        self._gemm(sched, a, dco["w"], y, a_ld=x.C, a_k=x.C, a_rows=x.rows, mode=A_CONV3X3, batch=B, H=x.H, W=x.W,
                   k_tap_pitch=x.C, out_ld=cout, out_mode=OUT_F32_NCHW, bias=dco["b"], rows_per_sample=x.hw)
        taps = []
        identity = True
        if self.compact:
            identity = False  # the gather is part of the cached (graph-captured) state shared by every assignment
            inv = self._dev_index("inv_perm")
            y = y.index_select(0, inv)
        if want_taps:
            # block outputs as the reference's hooks see them ([B, C, H, W]) in bf16 channels-last (what the fused loss
            # kernels read in place): one conversion pass off the fp32 stream into a tensor the caller owns; with expert
            # bucketing the gather back to the caller's sample order runs over whole NHWC samples (contiguous chunks)
            for t in tap_acts:
                v = torch.empty(t.rows, t.C, device=self.device, dtype=BF16)
                K.copy_rows_cvt(t.f, t.C, v, t.C, t.rows, t.C)
                v = v.view(t.B, t.H, t.W, t.C)
                if not identity:
                    v = v.index_select(0, inv)
                taps.append(v.permute(0, 3, 1, 2))
        return y, taps
