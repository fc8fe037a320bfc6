"""Host-side launchers for the sm_100a kernels: torch tensors in, C-ABI calls out (ctypes).

PyTorch is only plumbing here (device memory, the current stream); every op below runs a
hand-written kernel from libaptp_sm100.so and raises if the library is missing.
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass
from typing import List, Optional, Sequence

import numpy as np
import torch

from . import _lib
from ._lib import (A_CONV3X3, A_CONV3X3_S2, A_LINEAR, EPI_GEGLU, EPI_SILU, OUT_BF16, OUT_F32, OUT_F32_NCHW, GemmArgs,
                   check, load)

BM = 128
BK = 64
TILE_PLACEHOLDER, TILE_A_FIRST, TILE_A_LAST, TILE_SKIP = 1, 2, 4, 8  # APTP_TILE_*
A_STAT_MAX_CHUNKS = 6
_MAX_PAIRS = {}


def gemm_max_pairs() -> int:
    """Co-resident CTA pairs of the GEMM kernel on the current device (aptp_gemm_max_pairs), cached."""
    dev = torch.cuda.current_device() if torch.cuda.is_available() else -1
    v = _MAX_PAIRS.get(dev)
    if v is None:
        v = int(load().aptp_gemm_max_pairs()) if dev >= 0 else 74
        _MAX_PAIRS[dev] = v
    return v


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def check_abort() -> None:
    rc = load().aptp_check_abort(_stream())
    if rc != 0:
        check(rc, "aptp_check_abort")


def poll_abort() -> None:
    """Non-blocking mbarrier-timeout check, called once per U-Net forward / train step: raises if a pipelined kernel of
    an EARLIER launch timed out (the flag makes later pipelined kernels unwind early, so their results are invalid)."""
    rc = load().aptp_poll_abort(_stream())
    if rc != 0:
        check(rc, "aptp_poll_abort")


# --------------------------------------------------------------------------------------------
# GEMM schedule (segments = expert buckets, tiles = 128-row x bn-column work items)
# --------------------------------------------------------------------------------------------
@dataclass
class Segment:
    row_begin: int
    row_end: int
    n_valid: int
    k_chunks: int
    w_row_off: int = 0
    vec_off: int = 0
    tab_off: int = 0
    n_store: int = -1  # default: n_valid rounded up to 8
    out_col_off: int = 0
    active: bool = True
    w2_row_off: int = 0  # first row of the bucket's block in the second operand pair's weights (fused shortcut)


@dataclass
class Schedule:
    segs: torch.Tensor   # int32 [n_segs, 12] on device
    tiles: torch.Tensor  # int32 [n_tiles, 4] on device
    n_segs: int
    n_tiles: int
    bn: int
    box: tuple           # (bw, bh, bb)
    a_stat: int = 0      # > 0: A-stationary tile list (resident A chunk slots = max k_chunks), see build_schedule
    a_pairs: int = 0     # CTA pairs that list was laid out for
    flops: float = 0.0   # 2 * kept MACs of this launch (for roofline accounting)
    bytes_in: float = 0.0   # algorithmic operand bytes: kept A rows x kept K + kept weight block (bf16), read once
    out_elems: float = 0.0  # output elements written (x2 / x4 bytes by output type; same count for a residual read)


class _Stager:
    """Pinned staging ring for the small host -> device uploads of schedule / table arrays: one asynchronous copy per
    array instead of a synchronous pageable copy (a forward for a NEW prompt -> expert assignment uploads ~500 of them)."""

    def __init__(self, nbytes: int = 32 << 20):
        self.buf = None
        self.cap = nbytes
        self.off = 0
        self.slabs = {}

    def upload(self, arr: np.ndarray, device) -> torch.Tensor:
        device = torch.device(device)
        t = torch.from_numpy(np.ascontiguousarray(arr))
        if device.type != "cuda" or torch.cuda.is_current_stream_capturing() or t.numel() == 0:
            return t.to(device)
        n = (t.numel() * t.element_size() + 63) // 64 * 64
        if n > self.cap // 4:
            return t.to(device)
        if self.buf is None:
            self.buf = torch.empty(self.cap, dtype=torch.uint8).pin_memory()
        if self.off + n > self.cap:  # ring wrap: every copy issued so far must have left the staging area
            torch.cuda.synchronize()
            self.off = 0
        view = self.buf[self.off:self.off + t.numel() * t.element_size()].view(t.dtype).view(t.shape)
        self.off += n
        view.copy_(t)
        dev = self._device_view(t, n, device)
        dev.copy_(view, non_blocking=True)
        return dev

    def _device_view(self, t: torch.Tensor, n: int, device) -> torch.Tensor:
        """Device memory for one uploaded array, carved out of a 4 MB slab: a forward for a new assignment uploads ~500
        arrays of a few hundred bytes, and 500 separate allocations mean cudaMalloc calls of new small-pool segments in
        the middle of an asynchronously queued forward (each waits for the GPU: 3 - 250 ms per re-structuring, measured).
        The views keep their slab alive; it is freed when the schedules of an evicted state die."""
        key = (device.type, device.index)
        slab = self.slabs.get(key)
        if slab is None or slab[1] + n > slab[0].numel():
            slab = [torch.empty(4 << 20, dtype=torch.uint8, device=device), 0]
            self.slabs[key] = slab
        off = slab[1]
        slab[1] = off + (n + 255) // 256 * 256
        return slab[0][off:off + t.numel() * t.element_size()].view(t.dtype).view(t.shape)


_STAGER = _Stager()


def upload(arr: np.ndarray, device) -> torch.Tensor:
    return _STAGER.upload(arr, device)


def conv_box(W: int, H: int) -> tuple:
    """Pick the 128-pixel output box (bw, bh, bb) that tiles a W x H image."""
    for bw in (128, 64, 32, 16, 8, 4, 2, 1):
        if bw <= W and W % bw == 0:
            rest = BM // bw
            for bh in (rest, rest // 2, rest // 4, rest // 8, rest // 16, rest // 32, rest // 64, rest // 128):
                if bh >= 1 and bh <= H and H % bh == 0 and rest % bh == 0:
                    return bw, bh, rest // bh
    raise ValueError(f"no 128-pixel box tiles a {W}x{H} image")


def build_schedule(segments: Sequence[Segment], bn: int, device, mode: int = A_LINEAR, Ho: int = 1, Wo: int = 1,
                   geglu: bool = False, taps: Optional[int] = None) -> Schedule:
    """Enumerate tiles (m outer, n inner so concurrently running CTAs share the A tile in L2)."""
    segs = np.zeros((max(len(segments), 1), 12), dtype=np.int32)
    runs: List[np.ndarray] = []
    by_rows = {}
    kc_max = 0
    box = (BM, 1, 1) if mode == A_LINEAR else conv_box(Wo, Ho)
    if mode == _lib.A_CONV3X3 and Wo % 8 == 0 and Ho % 16 == 0 and os.environ.get("APTP_CONV_HALO", "1") != "0":
        # 8 x 16 pixel boxes: the kernel then loads ONE 18 x 16 halo tile per K chunk and derives the nine taps from it
        # (aptp_grouped_gemm_fwd, halo mode) instead of nine shifted boxes
        box = (8, 16, 1)
    bw, bh, bb = box
    hw = Ho * Wo
    cols_per_tile = bn // 2 if geglu else bn
    if taps is None:
        taps = 1 if mode == A_LINEAR else 9
    flops = 0.0
    bytes_in = 0.0
    out_elems = 0.0
    for si, s in enumerate(segments):
        n_store = s.n_store if s.n_store >= 0 else (s.n_valid + 7) // 8 * 8
        segs[si, :10] = (s.row_begin, s.row_end, s.n_valid, n_store, s.k_chunks, s.w_row_off, s.vec_off, s.tab_off,
                         s.out_col_off, s.w2_row_off)
        if not s.active or s.row_end <= s.row_begin or s.n_valid <= 0 or s.k_chunks <= 0:
            continue
        n_tiles_n = (max(s.n_valid, n_store) + cols_per_tile - 1) // cols_per_tile
        rows = s.row_end - s.row_begin
        flops += 2.0 * rows * s.n_valid * (2 if geglu else 1) * s.k_chunks * BK * taps
        bytes_in += 2.0 * rows * s.k_chunks * BK + 2.0 * s.n_valid * (2 if geglu else 1) * s.k_chunks * BK * taps
        out_elems += float(rows) * n_store
        if mode == A_LINEAR:
            m_bases = np.arange(s.row_begin, s.row_end, BM, dtype=np.int64)
        else:
            assert s.row_begin % hw == 0 and s.row_end % hw == 0, "conv segments must cover whole samples"
            img = np.arange(s.row_begin // hw, s.row_end // hw, bb, dtype=np.int64)
            oy = np.arange(0, Ho, bh, dtype=np.int64)
            ox = np.arange(0, Wo, bw, dtype=np.int64)
            m_bases = ((img[:, None, None] * Ho + oy[None, :, None]) * Wo + ox[None, None, :]).reshape(-1)
        # tiles go in PAIRS (2i, 2i+1) = two row tiles that share the weight tile: a cluster of two CTAs
        # multicasts it. An odd row-tile count is padded with a placeholder that repeats its partner.
        # (vectorised: a level-0 launch has 10-20 k tiles and a forward ~250 schedules; Python loops over them
        # dominated the cost of re-structuring for a new prompt -> expert assignment)
        nm = len(m_bases)
        if nm == 0:
            continue
        odd = nm % 2
        mb = np.concatenate([m_bases, m_bases[-1:]]) if odd else m_bases
        n_pairs = len(mb) // 2
        m_pair = mb.reshape(n_pairs, 2)                                        # [pair, which]
        # column tiles of a bucket are BALANCED: N = 320 under bn = 224 becomes 160 + 160 rather than 224 + 96 (a narrow
        # ragged tile moves the whole A tile through shared memory for a fraction of the work); width in flags bits 8..15
        width, wflag = bn, 0
        if not geglu and os.environ.get("APTP_BALANCED_TILES", "1") != "0":
            ncols = max(s.n_valid, n_store)
            width = min(bn, ((ncols + n_tiles_n - 1) // n_tiles_n + 31) // 32 * 32)
            wflag = (width // 32) << 8 if width != bn else 0
        n0 = (np.arange(n_tiles_n, dtype=np.int64) * width)                    # [nt]
        blk = np.empty((n_pairs, n_tiles_n, 2, 4), dtype=np.int32)
        blk[..., 0] = si
        blk[..., 1] = m_pair[:, None, :]
        blk[..., 2] = n0[None, :, None]
        blk[..., 3] = wflag
        if odd:
            blk[n_pairs - 1, :, 1, 3] |= TILE_PLACEHOLDER
        # segments over the SAME rows (the q | k | v blocks of one expert bucket) share their A row tiles: their N tiles
        # are walked back to back per pair of row tiles, so A is fetched from DRAM once instead of once per block
        key = (s.row_begin, s.row_end) if mode == A_LINEAR else None
        prev = by_rows.get(key) if key is not None else None
        if prev is not None and runs[prev].shape[0] == blk.shape[0]:
            runs[prev] = np.concatenate([runs[prev], blk], axis=1)
        else:
            if key is not None:
                by_rows[key] = len(runs)
            runs.append(blk)
        kc_max = max(kc_max, s.k_chunks)
    a_stat = a_pairs = 0
    # (opt-in: measured neutral on B200 -- 53.6 ms per step either way, profiles/README.md round 2: the K = 320 layers
    # are bound by the per-tile hand-offs of the issuing warp, not by the L2 -> shared-memory fill)
    if (mode == A_LINEAR and runs and 0 < kc_max <= A_STAT_MAX_CHUNKS and os.environ.get("APTP_A_STAT", "0") != "0"
            and max(r.shape[1] for r in runs) >= 2
            and (torch.device(device).type == "cuda" or os.environ.get("APTP_A_STAT") == "force")):
        # A-stationary layout: the K <= 384 projections are bound by the L2 -> shared-memory fill, so every CTA pair
        # walks ALL N tiles of one pair of row tiles back to back and keeps the A row tile resident. Runs are dealt
        # round-robin to the S pairs of the grid; pair c consumes entries c, c + S, c + 2S, ...
        n_n = np.concatenate([np.full(r.shape[0], r.shape[1], dtype=np.int64) for r in runs])   # N tiles per run
        n_runs = len(n_n)
        S = min(n_runs, gemm_max_pairs())
        R = (n_runs + S - 1) // S
        nn_pad = np.zeros(R * S, dtype=np.int64)
        nn_pad[:n_runs] = n_n
        off = (np.cumsum(nn_pad.reshape(R, S), axis=0) - nn_pad.reshape(R, S)).reshape(-1)[:n_runs]  # entries before it
        max_len = int((np.cumsum(nn_pad.reshape(R, S), axis=0)[-1]).max())
        ent = np.concatenate([r.reshape(-1, 2, 4) for r in runs], 0)            # [entries, 2, 4] in run-major order
        run_of = np.repeat(np.arange(n_runs), n_n)
        first_ent = np.cumsum(n_n) - n_n
        nt = np.arange(len(run_of)) - first_ent[run_of]
        ent[nt == 0, :, 3] |= TILE_A_FIRST
        ent[nt == n_n[run_of] - 1, :, 3] |= TILE_A_LAST
        out_t = np.zeros((max_len * S, 2, 4), dtype=np.int32)
        out_t[:, :, 3] = TILE_SKIP
        out_t[(off[run_of] + nt) * S + (run_of % S)] = ent
        tl = out_t.reshape(-1, 4)
        a_stat, a_pairs = int(kc_max), int(S)
    else:
        tl = np.concatenate([r.reshape(-1, 4) for r in runs], 0) if runs else np.zeros((0, 4), dtype=np.int32)
    # one upload per schedule: [segs | tiles] as a single int32 array, the two tables are views of it
    n_seg_words = segs.size
    both = upload(np.concatenate([segs.reshape(-1), np.ascontiguousarray(tl, dtype=np.int32).reshape(-1)]), device)
    return Schedule(segs=both[:n_seg_words].view(segs.shape), tiles=both[n_seg_words:].view(-1, 4),
                    n_segs=len(segments), n_tiles=int(tl.shape[0]), bn=bn, box=box, a_stat=a_stat, a_pairs=a_pairs,
                    flops=flops, bytes_in=bytes_in, out_elems=out_elems)


def grouped_gemm(a: torch.Tensor, w: torch.Tensor, out: torch.Tensor, sched: Schedule, *, a_ld: int, a_k: int,
                 a_rows: int, mode: int = A_LINEAR, batch: int = 1, H: int = 1, W: int = 1, k_tap_pitch: int = 0,
                 out_ld: int, out_mode: int = OUT_BF16, bias: Optional[torch.Tensor] = None,
                 rowvec: Optional[torch.Tensor] = None, rowvec_ld: int = 0, rows_per_sample: int = 1,
                 residual: Optional[torch.Tensor] = None, res_ld: int = 0, gate: Optional[torch.Tensor] = None,
                 gate_ld: int = 0, gate_group: int = 1, border_tab: Optional[torch.Tensor] = None, tab_ld: int = 0,
                 flags: int = 0, ln_colsum: Optional[torch.Tensor] = None, ln_rowstats: Optional[torch.Tensor] = None,
                 rowstat_out: Optional[torch.Tensor] = None, colstat=None, a2: Optional[torch.Tensor] = None,
                 a2_ld: int = 0, a2_k: int = 0, w2: Optional[torch.Tensor] = None) -> None:
    """out = epilogue(A @ W^T) through aptp_grouped_gemm_fwd. `a`, `w`, `out` may be views: only
    data_ptr() and the explicit pitches are used."""
    if sched.n_tiles == 0:
        return
    args = GemmArgs()
    args.a, args.a_mode, args.a_ld, args.a_k, args.a_rows = a.data_ptr(), mode, a_ld, a_k, a_rows
    args.batch, args.H, args.W = batch, H, W
    args.w, args.w_rows, args.w_ld, args.k_tap_pitch = w.data_ptr(), w.shape[0], w.shape[1], k_tap_pitch
    args.out, args.out_ld, args.out_mode = out.data_ptr(), out_ld, out_mode
    args.bn = sched.bn
    args.bw, args.bh, args.bb = sched.box
    args.bias = _ptr(bias)
    args.rowvec, args.rowvec_ld, args.rows_per_sample = _ptr(rowvec), rowvec_ld, rows_per_sample
    args.residual, args.res_ld = _ptr(residual), res_ld
    args.gate, args.gate_ld, args.gate_group = _ptr(gate), gate_ld, gate_group
    args.border_tab, args.tab_ld = _ptr(border_tab), tab_ld
    if colstat is not None:   # (sum plane, sumsq plane) [batch * blocks, ld] fp32, blocks = rows_per_sample / 32
        cs_sum, cs_sq = colstat
        args.gn_stats, args.gn_stats_sq = cs_sum.data_ptr(), cs_sq.data_ptr()
        args.gn_ld, args.gn_blocks = cs_sum.shape[1], rows_per_sample // 32
        flags |= _lib.EPI_GN_STATS
    else:
        args.gn_stats, args.gn_stats_sq, args.gn_ld, args.gn_blocks = None, None, 0, 0
    args.flags = flags | (_lib.EPI_LN_FOLD if ln_rowstats is not None else 0)
    args.ln_colsum, args.ln_rowstats = _ptr(ln_colsum), _ptr(ln_rowstats)   # ln_rowstats: [rows, 2] fp32 (mean, rstd)
    args.rowstat_out = _ptr(rowstat_out)                                     # [rows, C/32, 2] fp32 (sum, sumsq)
    args.rowstat_chunks = rowstat_out.shape[1] if rowstat_out is not None else 0
    args.a_stat_chunks, args.a_stat_pairs = sched.a_stat, sched.a_pairs
    # second operand pair accumulated into the same tiles (the ResNet's 1x1 shortcut inside conv2; halo-mode convs only)
    args.a2, args.a2_ld, args.a2_k = _ptr(a2), a2_ld, a2_k
    args.w2, args.w2_rows, args.w2_ld = _ptr(w2), (w2.shape[0] if w2 is not None else 0), (w2.shape[1] if w2 is not None else 0)
    args.segs, args.n_segs = sched.segs.data_ptr(), sched.n_segs
    args.tiles, args.n_tiles = sched.tiles.data_ptr(), sched.n_tiles
    check(load().aptp_grouped_gemm_fwd(C.byref(args), _stream()), "aptp_grouped_gemm_fwd")


# --------------------------------------------------------------------------------------------
# norms / elementwise
# --------------------------------------------------------------------------------------------
_GN_WS = {}  # device index -> zero-initialised workspace of aptp_groupnorm_stats (ticket counters + partials)


def _gn_workspace(device, need: int) -> torch.Tensor:
    """Workspace of the deterministic GroupNorm statistics reduction: one per device (the engine issues its kernels
    on one stream at a time; CUDA-graph replays run on that stream too), allocated once with room to spare (its first
    bytes are ticket counters that every launch leaves at zero) and grown only outside CUDA-graph capture."""
    key = torch.device(device).index
    ws = _GN_WS.get(key)
    if ws is None or ws.numel() < need:
        if torch.cuda.is_current_stream_capturing():
            raise RuntimeError("aptp_groupnorm_stats workspace must be sized before CUDA-graph capture "
                               "(run one eager forward of the same shapes first)")
        ws = torch.zeros(max(need, 8 << 20), dtype=torch.uint8, device=device)
        _GN_WS[key] = ws
    return ws


def groupnorm_stats(x0, c0, ld0, x1, c1, ld1, batch, hw, group_size, sample_channels, stats, stats_groups,
                    x_f32: bool = False):
    lib = load()
    need = int(lib.aptp_groupnorm_stats_workspace(batch, hw, stats_groups))
    ws = _gn_workspace(stats.device, need)
    check(lib.aptp_groupnorm_stats(_ptr(x0), c0, ld0, _ptr(x1), c1, ld1, int(x_f32), batch, hw, group_size,
                                   _ptr(sample_channels), _ptr(stats), stats_groups, ws.data_ptr(), ws.numel(),
                                   _stream()), "aptp_groupnorm_stats")


def groupnorm_stats_from_partials(cs0, c0, cs1, c1, blocks, batch, group_size, sample_channels, stats, stats_groups):
    """cs0 / cs1: (sum plane, sumsq plane) written by GEMM epilogues (grouped_gemm(colstat=...)); cs1 None = one source."""
    check(load().aptp_groupnorm_stats_from_partials(
        _ptr(cs0[0]), _ptr(cs0[1]), c0, cs0[0].shape[1], _ptr(cs1[0]) if cs1 else None, _ptr(cs1[1]) if cs1 else None,
        c1, cs1[0].shape[1] if cs1 else 0, blocks, batch, group_size, _ptr(sample_channels), _ptr(stats), stats_groups,
        _stream()), "aptp_groupnorm_stats_from_partials")


def groupnorm_apply(x0, c0, ld0, x1, c1, ld1, y, ldy, batch, hw, group_size, eps, stats, stats_groups, gamma, beta,
                    affine_ld, sample_seg, sample_channels, gate, gate_ld, silu, x_f32: bool = False, raw_out=None,
                    raw_ld: int = 0):
    """`raw_out` (optional bf16 [rows, raw_ld]): also write the un-normalised input (both sources) as bf16 rows."""
    check(load().aptp_groupnorm_apply_raw(_ptr(x0), c0, ld0, _ptr(x1), c1, ld1, int(x_f32), _ptr(y), ldy, batch, hw,
                                          group_size, float(eps), _ptr(stats), stats_groups, _ptr(gamma), _ptr(beta),
                                          affine_ld, _ptr(sample_seg), _ptr(sample_channels), _ptr(gate), gate_ld,
                                          int(silu), _ptr(raw_out), raw_ld, _stream()), "aptp_groupnorm_apply_raw")


def ln_rowstats(partial, rows, C_, eps, out, sample_active=None, rows_per_sample=1):
    """partial [rows, C/32, 2] (sum, sumsq per 32-column chunk, from a GEMM's rowstat_out) -> out [rows, 2] (mean, rstd)."""
    check(load().aptp_ln_rowstats(_ptr(partial), partial.shape[1], rows, C_, float(eps), _ptr(out), _ptr(sample_active),
                                  rows_per_sample, _stream()), "aptp_ln_rowstats")


def layernorm(x, ldx, y, ldy, rows, C_, eps, gamma, beta, sample_active=None, rows_per_sample=1):
    check(load().aptp_layernorm(_ptr(x), ldx, _ptr(y), ldy, rows, C_, float(eps), _ptr(gamma), _ptr(beta),
                                _ptr(sample_active), rows_per_sample, _stream()), "aptp_layernorm")


def depth_lerp(x, ldx, y, ldy, out, ldo, rows, C_, d, rows_per_sample):
    check(load().aptp_depth_lerp(_ptr(x), ldx, _ptr(y), ldy, _ptr(out), ldo, rows, C_, _ptr(d), rows_per_sample,
                                 _stream()), "aptp_depth_lerp")


def copy_rows(src, lds, dst, ldd, rows, C_, sample_mask=None, rows_per_sample=1):
    check(load().aptp_copy_rows(_ptr(src), lds, _ptr(dst), ldd, rows, C_, _ptr(sample_mask), rows_per_sample,
                                _stream()), "aptp_copy_rows")


def copy_rows_cvt(src, lds, dst, ldd, rows, C_, sample_mask=None, rows_per_sample=1):
    """Row copy with conversion: src / dst are bf16 or fp32 tensors (dtype decides)."""
    check(load().aptp_copy_rows_cvt(_ptr(src), int(src.dtype == torch.float32), lds, _ptr(dst),
                                    int(dst.dtype == torch.float32), ldd, rows, C_, _ptr(sample_mask), rows_per_sample,
                                    _stream()), "aptp_copy_rows_cvt")


def depth_lerp_f32(x, ldx, y, ldy, out, ldo, rows, C_, d, rows_per_sample):
    check(load().aptp_depth_lerp_f32(_ptr(x), ldx, _ptr(y), ldy, _ptr(out), ldo, rows, C_, _ptr(d), rows_per_sample,
                                     _stream()), "aptp_depth_lerp_f32")


def upsample2x_cvt(src, dst, batch, H, W, C_):
    check(load().aptp_upsample2x_cvt(_ptr(src), int(src.dtype == torch.float32), _ptr(dst), batch, H, W, C_, _stream()),
          "aptp_upsample2x_cvt")


def upsample2x(src, dst, batch, H, W, C_):
    check(load().aptp_upsample2x(_ptr(src), _ptr(dst), batch, H, W, C_, _stream()), "aptp_upsample2x")


def im2col_input(sample_nchw, dst, batch, cin, H, W):
    check(load().aptp_im2col_input(_ptr(sample_nchw), _ptr(dst), batch, cin, H, W, _stream()), "aptp_im2col_input")


def timestep_embedding(t, dst, batch, dim):
    check(load().aptp_timestep_embedding(_ptr(t), _ptr(dst), batch, dim, _stream()), "aptp_timestep_embedding")


def cast_f32_bf16(src, dst, n):
    check(load().aptp_cast_f32_bf16(_ptr(src), _ptr(dst), n, _stream()), "aptp_cast_f32_bf16")


def silu_bf16(src, dst, n):
    check(load().aptp_silu_bf16(_ptr(src), _ptr(dst), n, _stream()), "aptp_silu_bf16")


def cfg_ddim_step(pred, x, x_out, n, guidance, alpha_t, alpha_prev, v_prediction=True):
    check(load().aptp_cfg_ddim_step(_ptr(pred), _ptr(x), _ptr(x_out), n, float(guidance), float(alpha_t),
                                    float(alpha_prev), int(v_prediction), _stream()), "aptp_cfg_ddim_step")


SAMPLER_STAT_CHUNKS = 16  # APTP_SAMPLER_STAT_CHUNKS


def cfg_pred_stats(pred, n_per_sample, batch, guidance, partials):
    """partials [batch, SAMPLER_STAT_CHUNKS, 4] fp64: chunk sums of m_text, m_text^2, m, m^2 (guidance rescale)."""
    check(load().aptp_cfg_pred_stats(_ptr(pred), n_per_sample, batch, float(guidance), _ptr(partials), _stream()),
          "aptp_cfg_pred_stats")


def cfg_sampler_step(pred, x, x_out, n_per_sample, batch, guidance, rescale, partials, coeffs, x0_hist_in=None,
                     x0_hist_out=None, noise=None, noise_ld=0, v_prediction=True):
    """One CFG (+ rescale) scheduler step; coeffs = (sa, sb, c_x, c_0, c_h, c_e, c_n) of sampling.sampler_plan."""
    c = _lib.SamplerCoeffs(*[float(v) for v in coeffs])
    check(load().aptp_cfg_sampler_step(_ptr(pred), _ptr(x), _ptr(x_out), n_per_sample, batch, float(guidance),
                                       float(rescale), _ptr(partials), C.byref(c), _ptr(x0_hist_in), _ptr(x0_hist_out),
                                       _ptr(noise), noise_ld, int(v_prediction), _stream()), "aptp_cfg_sampler_step")


def cfg_sampler_step_masked(pred, x, x_out, n_per_sample, batch, guidance, rescale, partials, coeffs, image, mask,
                            plane_size, init_noise, a_next, s_next, x0_hist_in=None, x0_hist_out=None, noise=None,
                            noise_ld=0, v_prediction=True):
    """cfg_sampler_step, then x_out = (1 - m) (a_next image + s_next init_noise) + m x_out in the same pass; mask is one
    plane of plane_size floats per sample, broadcast over the channels (inpainting, 1 = regenerate)."""
    c = _lib.SamplerCoeffs(*[float(v) for v in coeffs])
    check(load().aptp_cfg_sampler_step_masked(_ptr(pred), _ptr(x), _ptr(x_out), n_per_sample, batch, float(guidance),
                                              float(rescale), _ptr(partials), C.byref(c), _ptr(x0_hist_in),
                                              _ptr(x0_hist_out), _ptr(noise), noise_ld, int(v_prediction), _ptr(image),
                                              _ptr(mask), plane_size, _ptr(init_noise), float(a_next), float(s_next),
                                              _stream()), "aptp_cfg_sampler_step_masked")


def attention(q, ldq, k, ldk, v, ldv, out, ldo, batch, n_q, n_kv, sample_heads, max_heads, scale, lse2=None):
    check(load().aptp_attention_fwd(_ptr(q), ldq, _ptr(k), ldk, _ptr(v), ldv, _ptr(out), ldo, batch, n_q, n_kv,
                                    _ptr(sample_heads), max_heads, float(scale), _ptr(lse2), _stream()),
          "aptp_attention_fwd")


def attention_bwd(q, ldq, k, ldk, v, ldv, o, ldo, dout, lddo, lse2, delta, dq, lddq, dk, lddk, dv, lddv, batch, n_q,
                  n_kv, sample_heads, max_heads, scale):
    check(load().aptp_attention_bwd(_ptr(q), ldq, _ptr(k), ldk, _ptr(v), ldv, _ptr(o), ldo, _ptr(dout), lddo,
                                    _ptr(lse2), _ptr(delta), _ptr(dq), lddq, _ptr(dk), lddk, _ptr(dv), lddv, batch,
                                    n_q, n_kv, _ptr(sample_heads), max_heads, float(scale), _stream()),
          "aptp_attention_bwd")


# --------------------------------------------------------------------------------------------
# backward of the gated ops (K5)
# --------------------------------------------------------------------------------------------
def scale_cols(u, ldu, y, ldy, batch, hw, C_, gate, gate_ld, group):
    check(load().aptp_scale_cols_fwd(_ptr(u), ldu, _ptr(y), ldy, batch, hw, C_, _ptr(gate), gate_ld, group, _stream()),
          "aptp_scale_cols_fwd")


def scale_cols_bwd(u, ldu, dy, lddy, du, lddu, batch, hw, C_, gate, gate_ld, group, dgate):
    check(load().aptp_scale_cols_bwd(_ptr(u), ldu, _ptr(dy), lddy, _ptr(du), lddu, batch, hw, C_, _ptr(gate), gate_ld,
                                     group, _ptr(dgate), _stream()), "aptp_scale_cols_bwd")


def geglu(hg, ld, out, ldo, batch, hw, inner, gate, gate_ld, group):
    check(load().aptp_geglu_fwd(_ptr(hg), ld, _ptr(out), ldo, batch, hw, inner, _ptr(gate), gate_ld, group, _stream()),
          "aptp_geglu_fwd")


def geglu_bwd(hg, ld, df, lddf, dhg, lddhg, batch, hw, inner, gate, gate_ld, group, dgate):
    check(load().aptp_geglu_bwd(_ptr(hg), ld, _ptr(df), lddf, _ptr(dhg), lddhg, batch, hw, inner, _ptr(gate), gate_ld,
                                group, _ptr(dgate), _stream()), "aptp_geglu_bwd")


def groupnorm_bwd(x, ldx, da, ldda, dx, lddx, accumulate, batch, hw, C_, group_size, eps, stats, stats_groups, gamma,
                  beta, gate, gate_ld, silu, bstats, dgate):
    check(load().aptp_groupnorm_bwd(_ptr(x), ldx, _ptr(da), ldda, _ptr(dx), lddx, int(accumulate), batch, hw, C_,
                                    group_size, float(eps), _ptr(stats), stats_groups, _ptr(gamma), _ptr(beta),
                                    _ptr(gate), gate_ld, int(silu), _ptr(bstats), _ptr(dgate), _stream()),
          "aptp_groupnorm_bwd")


def layernorm_bwd(x, ldx, dy, lddy, dx, lddx, accumulate, rows, C_, eps, gamma):
    check(load().aptp_layernorm_bwd(_ptr(x), ldx, _ptr(dy), lddy, _ptr(dx), lddx, int(accumulate), rows, C_,
                                    float(eps), _ptr(gamma), _stream()), "aptp_layernorm_bwd")


def depth_lerp_bwd(dout, lddo, x, ldx, y, ldy, dy, lddy, dx, lddx, accumulate, batch, hw, C_, d, dd):
    check(load().aptp_depth_lerp_bwd(_ptr(dout), lddo, _ptr(x), ldx, _ptr(y), ldy, _ptr(dy), lddy, _ptr(dx), lddx,
                                     int(accumulate), batch, hw, C_, _ptr(d), _ptr(dd), _stream()),
          "aptp_depth_lerp_bwd")


def add_rows(src, lds, dst, ldd, rows, C_):
    check(load().aptp_add_rows(_ptr(src), lds, _ptr(dst), ldd, rows, C_, _stream()), "aptp_add_rows")


def upsample2x_bwd(dy, dx, batch, H, W, C_):
    check(load().aptp_upsample2x_bwd(_ptr(dy), _ptr(dx), batch, H, W, C_, _stream()), "aptp_upsample2x_bwd")


def zero_insert2x(src, dst, batch, H, W, C_):
    check(load().aptp_zero_insert2x(_ptr(src), _ptr(dst), batch, H, W, C_, _stream()), "aptp_zero_insert2x")


# --------------------------------------------------------------------------------------------
# router
# --------------------------------------------------------------------------------------------
def gumbel_gate(z, u, out, batch, n_width, n_depth, width_starts, n_gates, depth_order, temperature, base,
                non_zero_width):
    check(load().aptp_gumbel_gate_fwd(_ptr(z), _ptr(u), _ptr(out), batch, n_width, n_depth, _ptr(width_starts),
                                      n_gates, _ptr(depth_order), float(temperature), float(base),
                                      int(non_zero_width), _stream()), "aptp_gumbel_gate_fwd")


def gumbel_gate_bwd(z, u, dy, dz, batch, n_width, n_depth, depth_order, temperature, base):
    check(load().aptp_gumbel_gate_bwd(_ptr(z), _ptr(u), _ptr(dy), _ptr(dz), batch, n_width, n_depth, _ptr(depth_order),
                                      float(temperature), float(base), _stream()), "aptp_gumbel_gate_bwd")


def arch_normalize(gates, out, batch, dim, col_depth, col_scale, l2=True):
    check(load().aptp_arch_normalize(_ptr(gates), _ptr(out), batch, dim, _ptr(col_depth), _ptr(col_scale), int(l2),
                                     _stream()), "aptp_arch_normalize")


def arch_normalize_bwd(gates, dy, dx, batch, dim, col_depth, col_scale):
    check(load().aptp_arch_normalize_bwd(_ptr(gates), _ptr(dy), _ptr(dx), batch, dim, _ptr(col_depth),
                                         _ptr(col_scale), _stream()), "aptp_arch_normalize_bwd")


def route_cosine(a_norm, codes_norm, scores, indices, batch, dim, n_codes):
    check(load().aptp_route_cosine(_ptr(a_norm), _ptr(codes_norm), _ptr(scores), _ptr(indices), batch, dim, n_codes,
                                   _stream()), "aptp_route_cosine")


def sinkhorn_phase(phase, Q, scores, partial, indices, batch_local, batch_global, n_codes, epsilon, first_iter):
    check(load().aptp_sinkhorn_phase(phase, _ptr(Q), _ptr(scores), _ptr(partial), _ptr(indices), batch_local,
                                     batch_global, n_codes, float(epsilon), int(first_iter), _stream()),
          "aptp_sinkhorn_phase")


def route_sinkhorn(scores, Q, partial, indices, batch, n_codes, epsilon, iterations):
    check(load().aptp_route_sinkhorn(_ptr(scores), _ptr(Q), _ptr(partial), _ptr(indices), batch, n_codes,
                                     float(epsilon), iterations, _stream()), "aptp_route_sinkhorn")


# --------------------------------------------------------------------------------------------
# K6: loss front/back end of the pruning train step
# --------------------------------------------------------------------------------------------
def add_noise_velocity(latents, noise, timesteps, sqrt_acp, sqrt_1m_acp, noisy, target, batch, per_sample,
                       v_prediction=True):
    check(load().aptp_add_noise_velocity(_ptr(latents), _ptr(noise), _ptr(timesteps), _ptr(sqrt_acp), _ptr(sqrt_1m_acp),
                                         _ptr(noisy), _ptr(target), batch, per_sample, int(v_prediction), _stream()),
          "aptp_add_noise_velocity")


def mse_rows_fwd(a, lda, b, ldb, rows, C_, partial):
    check(load().aptp_mse_rows_fwd(_ptr(a), lda, _ptr(b), ldb, rows, C_, _ptr(partial), partial.numel(), _stream()),
          "aptp_mse_rows_fwd")


def mse_rows_bwd(a, lda, b, ldb, da, ldda, rows, C_, coef, scale):
    check(load().aptp_mse_rows_bwd(_ptr(a), lda, _ptr(b), ldb, _ptr(da), ldda, rows, C_, _ptr(coef), float(scale),
                                   _stream()), "aptp_mse_rows_bwd")


def pred_losses_fwd(pred, target, teacher, batch, per_sample, chunks, partial):
    check(load().aptp_pred_losses_fwd(_ptr(pred), _ptr(target), _ptr(teacher), batch, per_sample, chunks, _ptr(partial),
                                      _stream()), "aptp_pred_losses_fwd")


def pred_losses_bwd(pred, target, teacher, weight, g, dpred, batch, per_sample):
    check(load().aptp_pred_losses_bwd(_ptr(pred), _ptr(target), _ptr(teacher), _ptr(weight), _ptr(g), _ptr(dpred), batch,
                                      per_sample, _stream()), "aptp_pred_losses_bwd")


# --------------------------------------------------------------------------------------------
# K7: closed-form MAC accounting
# --------------------------------------------------------------------------------------------
MACS_GATE_DTYPE = np.dtype([("col", np.int32), ("width", np.int32), ("macs", np.float64)])
MACS_SUB_DTYPE = np.dtype([("first_gate", np.int32), ("n_gates", np.int32), ("depth_col", np.int32),
                           ("reserved", np.int32), ("fixed", np.float64)])


def macs_ratio_fwd(arch, gates_dev, n_gates, subs_dev, n_subs, fixed_total, cur_prunable, cur_total):
    check(load().aptp_macs_ratio_fwd(_ptr(arch), arch.stride(0), arch.shape[0], _ptr(gates_dev), n_gates, _ptr(subs_dev),
                                     n_subs, float(fixed_total), _ptr(cur_prunable), _ptr(cur_total), _stream()),
          "aptp_macs_ratio_fwd")


def macs_ratio_bwd(arch, gates_dev, n_gates, subs_dev, n_subs, dcur, darch):
    check(load().aptp_macs_ratio_bwd(_ptr(arch), arch.stride(0), arch.shape[0], _ptr(gates_dev), n_gates, _ptr(subs_dev),
                                     n_subs, _ptr(dcur), _ptr(darch), darch.stride(0), darch.shape[1], _stream()),
          "aptp_macs_ratio_bwd")


# --------------------------------------------------------------------------------------------
# K8: weight gradients
# --------------------------------------------------------------------------------------------
def wgrad(dy, ld_dy, a, ld_a, dw, dbias, rows, n_out, k_in, conv=None, splits=0, stride=1):
    """dw [n_out, taps * k_in] fp32 (+)= dy^T a over the rows; conv = (batch, H, W) of the INPUT selects the 3x3 taps
    (OHWI layout), stride 1 or 2. splits = 0 picks a split-K factor that fills the GPU."""
    taps = 9 if conv is not None else 1
    if conv is not None:
        batch, H, W = conv
        Ho, Wo = H // stride, W // stride
        bw, bh, bb = conv_box(Wo, Ho)
        n_stages = (Wo // bw) * (Ho // bh) * ((batch + bb - 1) // bb)
    else:
        batch = H = W = bw = bh = bb = 1
        n_stages = (rows + 127) // 128
    if splits <= 0:
        tiles = ((n_out + 127) // 128) * ((k_in + 127) // 128) * taps
        splits = max(1, min(n_stages, (4 * 148 + tiles - 1) // tiles))
    check(load().aptp_wgrad(_ptr(dy), ld_dy, _ptr(a), ld_a, _ptr(dw), dw.stride(0), _ptr(dbias), rows, n_out, k_in,
                            (stride if conv is not None else 0), batch, H, W, bw, bh, bb, splits, _stream()), "aptp_wgrad")


def col_sum_groups(dy, ld, groups, rows_per_group, n_out, out):
    check(load().aptp_col_sum_groups(_ptr(dy), ld, groups, rows_per_group, n_out, _ptr(out), out.stride(0), _stream()),
          "aptp_col_sum_groups")


def groupnorm_bwd_affine(x, ldx, da, ldda, dx, lddx, accumulate, batch, hw, C_, group_size, eps, stats, stats_groups, gamma,
                         beta, gate, gate_ld, silu, bstats, dgate, daffine):
    """groupnorm_bwd that also accumulates daffine [C, 2] = (dgamma, dbeta)."""
    check(load().aptp_groupnorm_bwd_affine(_ptr(x), ldx, _ptr(da), ldda, _ptr(dx), lddx, int(accumulate), batch, hw, C_,
                                           group_size, eps, _ptr(stats), stats_groups, _ptr(gamma), _ptr(beta), _ptr(gate),
                                           gate_ld, int(silu), _ptr(bstats), _ptr(dgate), _ptr(daffine), _stream()),
          "aptp_groupnorm_bwd_affine")


def layernorm_affine_bwd(x, ldx, dy, lddy, rows, C_, eps, daffine):
    check(load().aptp_layernorm_affine_bwd(_ptr(x), ldx, _ptr(dy), lddy, rows, C_, eps, _ptr(daffine), _stream()),
          "aptp_layernorm_affine_bwd")


# --------------------------------------------------------------------------------------------
# K9: fp32 hypernet linear, contrastive loss
# --------------------------------------------------------------------------------------------
def linear_f32_fwd(x, w, bias, y, B, K_, N):
    check(load().aptp_linear_f32_fwd(_ptr(x), _ptr(w), _ptr(bias), _ptr(y), B, K_, N, _stream()), "aptp_linear_f32_fwd")


def linear_f32_bwd(x, w, dy, dx, dw, db, B, K_, N):
    check(load().aptp_linear_f32_bwd(_ptr(x), _ptr(w), _ptr(dy), _ptr(dx), _ptr(dw), _ptr(db), B, K_, N, _stream()),
          "aptp_linear_f32_bwd")


def contrastive_fwd(arch, prompt, arch_temp, prompt_temp, inv_a, inv_p, Sa, Sp, row_loss, loss):
    M = arch.shape[0]
    check(load().aptp_contrastive_fwd(_ptr(arch), arch.shape[1], _ptr(prompt), prompt.shape[1], M, float(arch_temp),
                                      float(prompt_temp), _ptr(inv_a), _ptr(inv_p), _ptr(Sa), _ptr(Sp), _ptr(row_loss),
                                      _ptr(loss), _stream()), "aptp_contrastive_fwd")


def contrastive_bwd(arch, arch_temp, inv_a, Sa, Sp, grad_loss, dG, dhat, darch):
    M = arch.shape[0]
    check(load().aptp_contrastive_bwd(_ptr(arch), arch.shape[1], M, float(arch_temp), _ptr(inv_a), _ptr(Sa), _ptr(Sp),
                                      _ptr(grad_loss), _ptr(dG), _ptr(dhat), _ptr(darch), _stream()),
          "aptp_contrastive_bwd")
