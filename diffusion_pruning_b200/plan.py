"""Expert bucketing and per-expert weight compaction (host logic of the hot path).

`set_structure` hands the U-Net 70 width-gate tensors + 14 depth-gate tensors per sample. With hard
(0/1) gates every distinct architecture code in the batch is an *expert*; samples are sorted by
expert so each expert owns a contiguous row range, and every prunable layer gets one compacted
weight block per distinct kept set:

  ResNet   conv1 / time_emb_proj rows, norm2 affine, conv2 input columns   <- kept GroupNorm groups
  attention to_q/to_k/to_v rows, to_out columns                             <- kept heads
  FF       GEGLU proj rows (both halves), net.2 columns                     <- kept FF groups

which is the per-expert layout the reference's prune() family produces for a single code
(pdm/models/unet/blocks.py:52-67, :121-129, :153-187, :424-465, :641-697). Unlike prune(), the
compacted conv2 keeps *gated* semantics: a zero-gated GroupNorm group still emits silu(beta_c), so its
contribution is folded into a 3x3-border-aware bias table (SURVEY Appendix D-1).
"""
from __future__ import annotations

from dataclasses import dataclass, field
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np
import torch

BK = 64


def round_up(x: int, m: int) -> int:
    return (x + m - 1) // m * m


_BN_CACHE: dict = {}


def choose_bn(n_values: Sequence[int], multiple: int = 32, geglu: bool = False, k: int = 0) -> int:
    """Cached front end of _choose_bn (a re-structured forward asks ~170 times, mostly with the same arguments)."""
    import os
    key = (tuple(int(n) for n in n_values), multiple, bool(geglu), int(k), os.environ.get("APTP_BN_MODEL"),
           os.environ.get("APTP_BN_OVERHEAD"), os.environ.get("APTP_BALANCED_TILES"))
    bn = _BN_CACHE.get(key)
    if bn is None:
        if len(_BN_CACHE) > 4096:
            _BN_CACHE.clear()
        bn = _BN_CACHE[key] = _choose_bn(n_values, multiple, geglu, k)
    return bn


def _choose_bn(n_values: Sequence[int], multiple: int = 32, geglu: bool = False, k: int = 0) -> int:
    """Accumulator width for one launch from the shared-memory traffic of its tiles (DESIGN.md section 9a: the GEMM main
    loop is bound by the ~128 B/clk the TMA writes and the tensor core's operand reads share). Per K step a 128-row
    tile writes A + the weight box (bn rows; half of it per CTA in the 2-SM scheme, K*taps >= 1280; a quarter of A with
    the conv halo tile) and reads A + the weight rows its MMAs really use -- the last column tile of a bucket is ragged
    and runs with N = its 32-column-rounded remainder (`tile_mma_n` in gemm_sm100.cu), so wide tiles cost little padding.
    Units: rows of 128 B. `k` = reduction length incl. taps (0: unknown, 1-SM assumed). APTP_BN_MODEL=0 restores the
    round-1 rule (fewest padded columns)."""
    import os
    cands = [256, 224, 192, 160, 128, 96, 64]
    if geglu:
        cands = [256, 192, 128]
    if os.environ.get("APTP_BN_MODEL", "1") != "1":
        best, best_cost = None, None
        for bn in cands:
            cols = bn // 2 if geglu else bn
            pen = 1.0 if bn >= 160 else (1.08 if bn >= 128 else (1.25 if bn >= 96 else 1.5))
            cost = sum(((n + cols - 1) // cols) * cols for n in n_values if n > 0) * pen
            if best_cost is None or cost < best_cost - 1e-9:
                best, best_cost = bn, cost
        return best or 128
    two_sm = k >= 1280
    a_write = 128.0 if k < 2880 else 40.0          # 3x3 convs: one halo tile per 9 taps (36 KB / 9 = 4 KB per K step)
    a_write = float(os.environ.get("APTP_BN_OVERHEAD", a_write))
    best, best_cost = None, None
    for bn in cands:
        cols = bn // 2 if geglu else bn
        cost = 0.0
        for n in n_values:
            if n <= 0:
                continue
            w_box = bn / 2.0 if two_sm else float(bn)
            if geglu or os.environ.get("APTP_BALANCED_TILES", "1") == "0":
                full, rem = divmod(n, cols)
                cost += full * (a_write + w_box + 128.0 + bn)
                if rem:
                    n_mma = bn if geglu else min(bn, (rem + 31) // 32 * 32)
                    cost += a_write + w_box + 128.0 + n_mma
            else:  # balanced column tiles (kernels.build_schedule): nt tiles of the 32-rounded N / nt
                nt = (n + bn - 1) // bn
                width = min(bn, ((n + nt - 1) // nt + 31) // 32 * 32)
                cost += nt * (a_write + w_box + 128.0 + width)
        if best_cost is None or cost < best_cost - 1e-9:
            best, best_cost = bn, cost
    return best or 128


@dataclass
class ExpertSet:
    """Distinct architecture codes of the current batch and the sample -> expert assignment."""
    codes: np.ndarray            # [E, dim] uint8 (0/1)
    sample_expert: np.ndarray    # [Bg] expert id of each gate row
    width_starts: List[int]      # arch column of each width gate (len n_gates + 1)
    n_width: int
    # [E] weight source of each expert (PrunedExpertMixture: the fine-tuned model it runs on; two experts may share a
    # code and still differ here). None: one source for every expert, the model being run.
    source: Optional[np.ndarray] = None

    @property
    def n_experts(self) -> int:
        return self.codes.shape[0]

    def width_bits(self, gate_idx: int) -> np.ndarray:
        s, e = self.width_starts[gate_idx], self.width_starts[gate_idx + 1]
        return self.codes[:, s:e]

    def depth_bits(self, depth_idx: int) -> np.ndarray:
        return self.codes[:, self.n_width + depth_idx]

    def sources(self) -> np.ndarray:
        return self.source if self.source is not None else np.zeros(self.n_experts, dtype=np.int64)

    def key(self) -> bytes:
        return self.codes.tobytes() + (b"" if self.source is None else self.source.astype(np.int64).tobytes())


@dataclass
class BatchLayout:
    """Sample order used inside the engine: sorted by expert (stable), contiguous per expert."""
    perm: np.ndarray          # internal position -> original sample index
    inv_perm: np.ndarray
    expert_of_pos: np.ndarray  # expert id per internal position
    starts: np.ndarray        # [E+1] first internal position of each expert
    batch: int

    @staticmethod
    def build(sample_expert: np.ndarray, n_experts: int, batch: int) -> "BatchLayout":
        bg = len(sample_expert)
        assert batch % bg == 0, f"batch {batch} is not a multiple of the gate batch {bg}"
        # CFG: gates repeat along the batch (pdm/models/unet/gates.py:18-19) -> sample b uses row b % bg
        eid = np.asarray([sample_expert[b % bg] for b in range(batch)], dtype=np.int64)
        perm = np.argsort(eid, kind="stable")
        inv = np.empty_like(perm)
        inv[perm] = np.arange(batch)
        counts = np.bincount(eid, minlength=n_experts)
        starts = np.concatenate([[0], np.cumsum(counts)])
        return BatchLayout(perm=perm, inv_perm=inv, expert_of_pos=eid[perm], starts=starts, batch=batch)


def kept_variants(bits: np.ndarray, source: Optional[np.ndarray] = None) -> Tuple[List[np.ndarray], np.ndarray]:
    """bits [E, w] 0/1 -> (list of distinct kept-index arrays, variant id per expert). With `source` [E], experts of
    different weight sources never share a variant (their compacted blocks hold different weights)."""
    variants: Dict[tuple, int] = {}
    kept: List[np.ndarray] = []
    vid = np.zeros(bits.shape[0], dtype=np.int64)
    for e in range(bits.shape[0]):
        k = (int(source[e]) if source is not None else 0, bits[e].tobytes())
        if k not in variants:
            variants[k] = len(kept)
            kept.append(np.nonzero(bits[e])[0])
        vid[e] = variants[k]
    return kept, vid


def expand_groups(kept_groups: np.ndarray, group_size: int) -> np.ndarray:
    return (kept_groups[:, None] * group_size + np.arange(group_size)[None, :]).reshape(-1)


# --------------------------------------------------------------------------------------------------
# weight packing (runs on the GPU with torch indexing; results are cached per ExpertSet)
# --------------------------------------------------------------------------------------------------
def pack_conv_weight(w: torch.Tensor) -> torch.Tensor:
    """[Cout, Cin, 3, 3] -> K-major [Cout, 9*Cin] with K index = (dy*3+dx)*Cin + c."""
    cout, cin = w.shape[0], w.shape[1]
    return w.permute(0, 2, 3, 1).reshape(cout, 9 * cin)


def pack_conv_weight_dgrad(w: torch.Tensor) -> torch.Tensor:
    """Weights of the conv dgrad expressed as a forward 3x3 conv of the output gradient:
    dX[y,x,c] = sum_{tap,n} dY[y+1-dy, x+1-dx, n] W[n,c,dy,dx]  ->  [Cin, 9*Cout] with K index =
    (tap')*Cout + n and tap' = 8 - tap (taps flipped, channels transposed)."""
    cout, cin = w.shape[0], w.shape[1]
    return w.flip(2, 3).permute(1, 2, 3, 0).reshape(cin, 9 * cout).contiguous()


def pack_rows(w2d: torch.Tensor, kept_rows: List[np.ndarray], n_pad: int) -> torch.Tensor:
    """N compaction: one [n_pad, K] block per variant, kept rows first, zero rows after."""
    out = torch.zeros(len(kept_rows) * n_pad, w2d.shape[1], device=w2d.device, dtype=torch.bfloat16)
    for v, rows in enumerate(kept_rows):
        idx = torch.as_tensor(rows, device=w2d.device, dtype=torch.long)
        out[v * n_pad: v * n_pad + len(rows)] = w2d.index_select(0, idx).to(torch.bfloat16)
    return out


def pack_cols(w: torch.Tensor, kept_cols: List[np.ndarray], taps: int) -> torch.Tensor:
    """K compaction: w [N, taps*C] (tap-major); per variant keep the columns `kept` of every tap,
    moved to the front of the tap's C-wide slot, zeros after (slot pitch stays C)."""
    n, kc = w.shape
    c = kc // taps
    out = torch.zeros(len(kept_cols) * n, kc, device=w.device, dtype=torch.bfloat16)
    w3 = w.reshape(n, taps, c)
    for v, cols in enumerate(kept_cols):
        idx = torch.as_tensor(cols, device=w.device, dtype=torch.long)
        blk = out[v * n:(v + 1) * n].reshape(n, taps, c)
        blk[:, :, :len(cols)] = w3.index_select(2, idx).to(torch.bfloat16)
    return out


def border_table(w_conv2: torch.Tensor, beta: torch.Tensor, pruned_cols: List[np.ndarray]) -> torch.Tensor:
    """Contribution of zero-gated norm2 groups to conv2 under *gated* semantics: those channels enter
    conv2 as the constant silu(beta_c) wherever the 3x3 window is inside the image.
    Returns [V, 9 classes (ycls*3+xcls), Cout] fp32."""
    cout = w_conv2.shape[0]
    V = len(pruned_cols)
    tab = torch.zeros(V, 9, cout, device=w_conv2.device, dtype=torch.float32)
    sb = torch.nn.functional.silu(beta.float())
    # taps valid per border class along one axis: class 0 (first row/col): d in {1,2}; 1 (interior): all; 2 (last): {0,1}
    valid = {0: (1, 2), 1: (0, 1, 2), 2: (0, 1)}
    for v, cols in enumerate(pruned_cols):
        if len(cols) == 0:
            continue
        idx = torch.as_tensor(cols, device=w_conv2.device, dtype=torch.long)
        # per-tap vector v_t[o] = sum_c W[o, c, dy, dx] * silu(beta_c) over pruned c
        vt = (w_conv2.float().index_select(1, idx) * sb.index_select(0, idx)[None, :, None, None]).sum(1)  # [Cout,3,3]
        for yc in range(3):
            for xc in range(3):
                acc = torch.zeros(cout, device=w_conv2.device)
                for dy in valid[yc]:
                    for dx in valid[xc]:
                        acc = acc + vt[:, dy, dx]
                tab[v, yc * 3 + xc] = acc
    return tab
