"""Fine-tuned experts served as one mixed batch.

After fine-tuning (FineTuner, trainer.py:1683-1765) every expert has its own copy of EVERY U-Net parameter, not only
its own kept rows: conv_in, the time MLP, norms, projections, shortcuts, samplers and conv_out all differ between
experts. The reference serves them one job per expert (cluster_scripts/slurm/img_generation/sd2-1_cc3m.slurm:45-60).
`PrunedExpertMixture` runs a batch whose samples each name their expert through the same grouped launches as the
gated U-Net: an expert bucket is (weight source, code), every pack holds one block per expert and every segment of a
launch points at its bucket's block. Two experts may share a code; their weights still stay apart.

Memory: the K experts' fp32 weights plus, per expert, its compacted bf16 packs (the kept rows of the prunable layers
and a copy of every other layer).
"""
from __future__ import annotations

import os
from typing import Optional, Sequence

import numpy as np
import torch
import torch.nn as nn

from . import kernels as K
from . import plan as P
from .unet import UNet2DConditionModelPruned, UNet2DConditionOutput, _Engine


def _hard_code(expert: UNet2DConditionModelPruned) -> np.ndarray:
    """The expert's 0/1 code in the engine's column order (width gates, then depth gates)."""
    flat_w, flat_d = expert._flat_gates
    code = torch.cat([w.detach().reshape(1, -1).float().cpu() for w in flat_w] +
                     [d.detach().reshape(1, 1).float().cpu() for d in flat_d], dim=1)
    return code.to(torch.uint8).numpy()[0]


class PrunedExpertMixture(nn.Module):
    """K fine-tuned `UNet2DConditionModelPruned` experts of one config, run as one batch.

    forward(sample, timestep, encoder_hidden_states, expert_index): `expert_index` [B] (int) names each sample's expert
    (its position in `experts`); with a CFG-doubled batch of 2B samples a [B] index is tiled like the gates
    (pdm/models/unet/gates.py:18-19). Inference only; CUDA only. `expert_ids[k]` is the quantizer code row expert k was
    fine-tuned for (FineTuner's `expert_id`, a row of quantizer_embeddings.pt): code_to_expert() maps routed code
    indices onto the mixture."""

    def __init__(self, experts: Sequence[UNet2DConditionModelPruned], expert_ids: Optional[Sequence[int]] = None):
        super().__init__()
        experts = list(experts)
        if not experts:
            raise ValueError("PrunedExpertMixture needs at least one expert")
        for i, e in enumerate(experts):
            if not isinstance(e, UNet2DConditionModelPruned):
                raise TypeError(f"expert {i} is a {type(e).__name__}, not a UNet2DConditionModelPruned")
            if e.arch_vector is None:
                raise ValueError(f"expert {i} has no architecture vector: prune_to(arch_vector) first")
        cfg0 = dict(experts[0].config)
        for i, e in enumerate(experts[1:], 1):
            if dict(e.config) != cfg0:
                diff = sorted(k for k in set(cfg0) | set(e.config) if cfg0.get(k) != e.config.get(k))
                raise ValueError(f"expert {i} has a different config than expert 0 (keys {diff})")
        ids = list(range(len(experts))) if expert_ids is None else [int(i) for i in expert_ids]
        if len(ids) != len(experts):
            raise ValueError(f"{len(ids)} expert ids for {len(experts)} experts")
        if len(set(ids)) != len(ids):
            raise ValueError(f"expert ids must be distinct (each code row maps to one expert): {ids}")
        self.experts = nn.ModuleList(experts)
        self.expert_ids = ids
        self.codes = np.stack([_hard_code(e) for e in experts])            # [K, 1620] uint8
        st = experts[0].get_structure()
        widths = [w for ws in st["width"] for w in ws]
        self._width_starts = [0] + np.cumsum(widths).tolist()
        self._n_width = int(sum(widths))
        self._engine: Optional[_Engine] = None
        self._gate_state = None
        self._index_key = None

    @classmethod
    def from_pretrained(cls, dirs: Sequence[str], expert_ids: Optional[Sequence[int]] = None, **kwargs):
        """One fine-tuned expert per directory, read like UNet2DConditionModelPruned.from_pretrained: the diffusers
        layout (`unet/config.json` + weights, dense or physically sliced) with `arch_vector.pt` beside `unet/`. A
        directory may also be the `unet/` folder itself."""
        experts = []
        for d in dirs:
            sub = "unet" if os.path.isdir(os.path.join(d, "unet")) else None
            experts.append(UNet2DConditionModelPruned.from_pretrained(d, subfolder=sub, **kwargs))
        return cls(experts, expert_ids=expert_ids)

    @property
    def config(self):
        return self.experts[0].config

    @property
    def n_experts(self) -> int:
        return len(self.experts)

    @property
    def device(self) -> torch.device:
        return self.experts[0].device

    @property
    def dtype(self) -> torch.dtype:
        return self.experts[0].dtype

    def code_to_expert(self, n_codes: int) -> torch.Tensor:
        """[n_codes] int64: the mixture position of the expert fine-tuned for each quantizer code, -1 where none is."""
        m = torch.full((n_codes,), -1, dtype=torch.int64)
        for k, c in enumerate(self.expert_ids):
            if not 0 <= c < n_codes:
                raise ValueError(f"expert {k} has code id {c}, outside the {n_codes} codes")
            m[c] = k
        return m

    def enable_weight_training(self, on: bool = True) -> None:
        raise NotImplementedError("PrunedExpertMixture is inference only: fine-tune each expert on its own "
                                  "(UNet2DConditionModelPruned.enable_weight_training)")

    def invalidate_weight_cache(self) -> None:
        """Call after changing any expert's parameters: the packs are rebuilt on the next forward."""
        self._engine = None

    def _prepare_index(self, expert_index: torch.Tensor, batch: int) -> None:
        """Gate state of the batch: the fixed code list of the K experts, each its own weight source, and the sample ->
        expert assignment. Reused while the same index tensor is passed again unchanged (a sampling loop), so the host
        reads it once."""
        if not torch.is_tensor(expert_index) or expert_index.dim() != 1 or expert_index.dtype.is_floating_point \
                or expert_index.dtype == torch.bool or expert_index.is_complex():
            raise TypeError("expert_index must be a 1-D integer tensor")
        key = (id(expert_index), expert_index._version, batch)
        if self._index_key is not None and self._index_key[0] == key and self._index_key[1] is expert_index:
            return
        idx = expert_index.detach().cpu().numpy().astype(np.int64)
        if len(idx) == 0 or batch % len(idx) != 0:
            raise ValueError(f"batch {batch} is not a multiple of the {len(idx)} expert indices")
        if (idx < 0).any() or (idx >= self.n_experts).any():
            raise IndexError(f"expert_index out of range [0, {self.n_experts}): {idx[(idx < 0) | (idx >= self.n_experts)][:8]}")
        eset = P.ExpertSet(codes=self.codes, sample_expert=idx, width_starts=self._width_starts, n_width=self._n_width,
                           source=np.arange(self.n_experts, dtype=np.int64))
        self._gate_state = {"hard": True, "bg": len(idx), "width_starts": self._width_starts,
                            "n_width": self._n_width, "eset": eset}
        self._index_key = (key, expert_index)

    @torch.no_grad()
    def forward(self, sample: torch.Tensor, timestep, encoder_hidden_states: torch.Tensor, expert_index: torch.Tensor,
                return_dict: bool = True):
        self._prepare_index(expert_index, int(sample.shape[0]))
        if not (sample.is_cuda and encoder_hidden_states.is_cuda):
            raise RuntimeError("PrunedExpertMixture runs on the sm_100a CUDA path only: move the experts and inputs to "
                               "a CUDA device (there is no CPU fallback)")
        if self._engine is None or self._engine.device != sample.device:
            # the packs of the fixed expert list are built once: one code set, never evicted by the engine's LRU
            self._engine = _Engine(self.experts[0], sample.device, sources=list(self.experts), gates=self)
        out, _ = self._engine.run_graphed(sample, timestep, encoder_hidden_states)
        K.poll_abort()
        if not return_dict:
            return (out,)
        return UNet2DConditionOutput(sample=out)
