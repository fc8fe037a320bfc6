"""TEST INFRASTRUCTURE: a torch-on-CPU emulation of the C-ABI kernels' *contract* (segments, tiles,
pitches, column offsets, zero padding), monkey-patched over diffusion_pruning_b200.kernels so the
engine's host logic (expert bucketing, weight compaction, schedules, layer wiring) can be checked
against the oracle in the GPU-less build container. It is never imported by the product; the product
path has no fallback and raises without the CUDA library / a CUDA device.

The same functions are the per-launch references of tests/launch_replay.py: they run on the operands'
device, compute in the dtype set by reference_mode() (float32 by default, which is what the CPU tests use)
and, inside reference_mode(), report every region they write together with its unrounded value."""
from __future__ import annotations

import contextlib
import math

import numpy as np
import torch
import torch.nn.functional as F

from diffusion_pruning_b200 import kernels as K
from diffusion_pruning_b200._lib import A_CONV3X3, A_CONV3X3_S2, A_LINEAR, EPI_GEGLU, EPI_SILU, OUT_BF16, OUT_F32, OUT_F32_NCHW


_CDT = torch.float32   # compute dtype of the emulation
_WRITES = None         # list of (destination view, unrounded value, meta) inside reference_mode()


@contextlib.contextmanager
def reference_mode(dtype=torch.float64):
    """Compute in `dtype` and collect the written regions: yields the list that _put() appends to."""
    global _CDT, _WRITES
    old = (_CDT, _WRITES)
    _CDT, _WRITES = dtype, []
    try:
        yield _WRITES
    finally:
        _CDT, _WRITES = old


def _put(dst: torch.Tensor, val: torch.Tensor, **meta) -> None:
    """dst[...] = val rounded to dst's dtype. meta: k = reduction length behind each value (fp32 tolerance),
    blocks = n (dst rows are per-sample groups of n partial-sum blocks whose order is not part of the contract),
    exact = the contract fixes these values exactly (zero padding),
    floor = absolute error the operation's contract allows on top of rounding its result,
    stored = (region, power): dst holds per-32-row sums of region ** power as stored in the output,
    seg / row0 / col0 = grouped-GEMM segment and the output (row, column) of dst[0, 0]."""
    dst.copy_(val.to(dst.dtype) if val.dtype != dst.dtype else val)
    if _WRITES is not None:
        _WRITES.append((dst, val.detach().clone(), meta))


def _put_cols(O, rb, re, oco, nv, nst, acc, k, loc):
    """Output columns [oco, oco + nv) of rows [rb, re) with the result, [oco + nv, oco + nst) with exact zeros."""
    _put(O[rb:re, oco:oco + nv], acc[:, :nv], k=k, **loc)
    if nst > nv:
        _put(O[rb:re, oco + nv:oco + nst], acc[:, nv:nst], exact=True, **dict(loc, col0=oco + nv))


def _c(t: torch.Tensor) -> torch.Tensor:
    return t.to(_CDT)


def _view(t: torch.Tensor, rows: int, cols: int, ld: int) -> torch.Tensor:
    return torch.as_strided(t, (rows, cols), (ld, 1), t.storage_offset())


def _check_tiles(sched: K.Schedule, mode, Ho, Wo, geglu):
    """Every active segment must be exactly covered by its tiles."""
    segs = sched.segs.cpu().numpy()
    tiles = sched.tiles.cpu().numpy()
    tiles = tiles[(tiles[:, 3] & 8) == 0]  # APTP_TILE_SKIP: padding entries of an A-stationary list
    bw, bh, bb = sched.box
    cols = sched.bn // 2 if geglu else sched.bn
    for si in range(sched.n_segs):
        rb, re, nv, ns = segs[si][:4]
        mine = tiles[tiles[:, 0] == si]
        if len(mine) == 0:
            continue
        nt = (max(nv, ns) + cols - 1) // cols
        w32 = int(mine[0, 3] >> 8) & 0xFF
        width = w32 * 32 if w32 else sched.bn  # balanced tiles: narrower than bn, same count
        assert width <= sched.bn and nt * (width // 2 if geglu else width) >= max(nv, ns)
        assert set(mine[:, 2].tolist()) == {i * width for i in range(nt)}
        covered = np.zeros(re - rb, dtype=np.int32)
        for m in np.unique(mine[:, 1]):
            if mode == A_LINEAR:
                r = np.arange(m, m + 128)
            else:
                hw = Ho * Wo
                img0, rem = divmod(int(m), hw)
                oy0, ox0 = divmod(rem, Wo)
                rr = np.arange(128)
                ix, iy, ib = rr % bw, (rr // bw) % bh, rr // (bw * bh)
                r = ((img0 + ib) * Ho + oy0 + iy) * Wo + ox0 + ix
            r = r[(r >= rb) & (r < re)]
            covered[r - rb] += 1
        assert (covered == 1).all(), "tiles must cover each segment row exactly once"


def grouped_gemm(a, w, out, sched, *, a_ld, a_k, a_rows, mode=A_LINEAR, batch=1, H=1, W=1, k_tap_pitch=0, out_ld,
                 out_mode=OUT_BF16, bias=None, rowvec=None, rowvec_ld=0, rows_per_sample=1, residual=None, res_ld=0,
                 gate=None, gate_ld=0, gate_group=1, border_tab=None, tab_ld=0, flags=0, ln_colsum=None, ln_rowstats=None,
                 rowstat_out=None, colstat=None, a2=None, a2_ld=0, a2_k=0, w2=None):
    if sched.n_tiles == 0:
        return
    geglu = bool(flags & EPI_GEGLU)
    stride = 2 if mode == A_CONV3X3_S2 else 1
    Ho, Wo = (H // stride, W // stride) if mode != A_LINEAR else (1, 1)
    _check_tiles(sched, mode, Ho, Wo, geglu)
    segs = sched.segs.cpu().numpy()
    tiles = sched.tiles.cpu().numpy()
    tiles = tiles[(tiles[:, 3] & 8) == 0]
    A = _c(_view(a, a_rows, a_ld, a_ld))
    if A.data_ptr() == a.data_ptr():
        A = A.clone()
    A[:, a_k:] = 0  # reads beyond the tensor-map extent are zero-filled
    Wm = _c(w)
    dev = out.device
    for si in range(sched.n_segs):
        rb, re, nv, ns, kch, wro, voff, toff, oco = [int(v) for v in segs[si][:9]]
        if not (tiles[:, 0] == si).any():
            continue
        kk = kch * 64
        kdepth = kk * (1 if mode == A_LINEAR else 9) + (a2_k if a2 is not None else 0)
        if mode == A_LINEAR:
            Ae = A[rb:re, :kk] if kk <= a_ld else F.pad(A[rb:re], (0, kk - a_ld))
            if geglu:
                half = sched.bn // 2
                nt = (max(nv, ns) + half - 1) // half
                blk = Wm[wro:wro + nt * sched.bn, :kk].reshape(nt, 2, half, kk)
                wh = blk[:, 0].reshape(nt * half, kk)
                wg = blk[:, 1].reshape(nt * half, kk)
                acc_h, acc_g = Ae @ wh.t(), Ae @ wg.t()
                if ln_rowstats is not None:  # APTP_EPI_LN_FOLD: rstd * (acc - mean * colsum), per row
                    mu, rstd = ln_rowstats[rb:re, 0], ln_rowstats[rb:re, 1]
                    cs = ln_colsum[voff:voff + nt * sched.bn].reshape(nt, 2, half)
                    acc_h = rstd[:, None] * (acc_h - mu[:, None] * cs[:, 0].reshape(-1)[None])
                    acc_g = rstd[:, None] * (acc_g - mu[:, None] * cs[:, 1].reshape(-1)[None])
                if bias is not None:
                    bb_ = bias[voff:voff + nt * sched.bn].reshape(nt, 2, half)
                    acc_h = acc_h + bb_[:, 0].reshape(-1)
                    acc_g = acc_g + bb_[:, 1].reshape(-1)
                acc = None
            else:
                ncols = max(nv, ns)
                acc = Ae @ Wm[wro:wro + ncols, :kk].t()
        else:
            hw = Ho * Wo
            b0, b1 = rb // hw, re // hw
            x = A.reshape(batch, H, W, a_ld)[b0:b1, :, :, :kk].permute(0, 3, 1, 2)
            ncols = max(nv, ns)
            wk = Wm[wro:wro + ncols].reshape(ncols, 9, k_tap_pitch)[:, :, :kk].reshape(ncols, 3, 3, kk).permute(0, 3, 1, 2)
            acc = F.conv2d(x, wk, None, stride=stride, padding=1).permute(0, 2, 3, 1).reshape(-1, ncols)
            if a2 is not None:  # second operand pair: 1x1 conv over a second tensor into the same tiles
                assert mode == A_CONV3X3
                A2 = _c(_view(a2, a_rows, a2_k, a2_ld))
                acc = acc + A2[rb:re] @ _c(w2)[:ncols, :a2_k].t()
        rows = torch.arange(rb, re, device=dev)
        sample = rows // rows_per_sample
        if geglu:
            cols = torch.arange(acc_h.shape[1], device=dev)
            if gate is not None:
                gsel = gate[sample][:, (cols // gate_group).clamp(max=gate_ld - 1)]
                acc_h, acc_g = acc_h * gsel, acc_g * gsel
            acc = acc_h * F.gelu(acc_g)
        else:
            cols = torch.arange(acc.shape[1], device=dev)
            if ln_rowstats is not None:
                mu, rstd = ln_rowstats[rb:re, 0], ln_rowstats[rb:re, 1]
                nb = min(nv, acc.shape[1])
                acc[:, :nb] = rstd[:, None] * (acc[:, :nb] - mu[:, None] * ln_colsum[voff:voff + nb][None])
            if bias is not None:
                nb = min(nv, acc.shape[1])
                acc[:, :nb] += bias[voff:voff + nb]
            if rowvec is not None:
                rv = _view(rowvec, int(sample.max()) + 1, acc.shape[1], rowvec_ld)
                acc = acc + rv[sample]
            if border_tab is not None:
                pix = rows % (Ho * Wo)
                oy, ox = pix // Wo, pix % Wo
                yc = torch.where(oy == 0, 0, torch.where(oy == Ho - 1, 2, 1))
                xc = torch.where(ox == 0, 0, torch.where(ox == Wo - 1, 2, 1))
                tab = border_tab.reshape(-1)[toff:toff + 9 * tab_ld].reshape(9, tab_ld)[:, :acc.shape[1]]
                acc = acc + tab[yc * 3 + xc]
            if gate is not None:
                acc = acc * gate[sample][:, (cols // gate_group).clamp(max=gate_ld - 1)]
            if flags & EPI_SILU:
                acc = F.silu(acc)
        if residual is not None:
            R = _c(_view(residual, re, res_ld, res_ld))
            nb = min(nv, acc.shape[1])
            acc[:, :nb] += R[rb:re, oco:oco + nb]
        acc[:, nv:] = 0
        nst = max(ns, nv) if out_mode != OUT_F32_NCHW else nv
        loc = dict(seg=si, row0=rb, col0=oco)
        if out_mode == OUT_BF16:
            O = _view(out, re, out_ld, out_ld)
            _put_cols(O, rb, re, oco, nv, nst, acc, kdepth, loc)
            if colstat is not None:  # statistics of the STORED (bf16-rounded) values
                assert rows_per_sample % 128 == 0 and rb % rows_per_sample == 0
                a32 = _c(acc[:, :nst].to(torch.bfloat16)).reshape((re - rb) // 32, 32, nst)
                nblk = rows_per_sample // 32
                st = O[rb:re, oco:oco + nst]  # (a replay recomputes these sums from the values the device stored there)
                _put(colstat[0][rb // 32: re // 32, oco:oco + nst], a32.sum(1), k=32, blocks=nblk,
                     stored=(st, 1), **loc)
                _put(colstat[1][rb // 32: re // 32, oco:oco + nst], (a32 * a32).sum(1), k=32, blocks=nblk,
                     stored=(st, 2), **loc)
            if rowstat_out is not None:  # per-row (sum, sumsq) per 32-column chunk of the stored values
                assert oco % 32 == 0 and nst % 32 == 0
                a32 = acc[:, :nst].reshape(re - rb, nst // 32, 32)
                _put(rowstat_out[rb:re, oco // 32: oco // 32 + nst // 32, 0], a32.sum(-1), k=32, part="rowstat", **loc)
                _put(rowstat_out[rb:re, oco // 32: oco // 32 + nst // 32, 1], (a32 * a32).sum(-1), k=32, part="rowstat", **loc)
        elif out_mode == OUT_F32:
            O = _view(out, re, out_ld, out_ld)
            _put_cols(O, rb, re, oco, nv, nst, acc, kdepth, loc)
            if colstat is not None:  # per-channel partial sums of every 32-row block (block order differs from the
                # device's tile / quadrant order for conv boxes; the consumer only sums over the blocks of a sample)
                assert rows_per_sample % 128 == 0 and rb % rows_per_sample == 0
                a32 = acc[:, :nst].reshape((re - rb) // 32, 32, nst)
                nblk = rows_per_sample // 32
                _put(colstat[0][rb // 32: re // 32, oco:oco + nst], a32.sum(1), k=32, blocks=nblk, **loc)
                _put(colstat[1][rb // 32: re // 32, oco:oco + nst], (a32 * a32).sum(1), k=32, blocks=nblk,
                     **loc)
        else:
            nb = re // rows_per_sample
            O = torch.as_strided(out, (nb, out_ld, rows_per_sample), (out_ld * rows_per_sample, rows_per_sample, 1),
                                 out.storage_offset())
            _put(O[rb // rows_per_sample:nb, :nv], acc[:, :nv].reshape(-1, rows_per_sample, nv).permute(0, 2, 1),
                 k=kdepth, seg=si)


def groupnorm_stats(x0, c0, ld0, x1, c1, ld1, batch, hw, group_size, sample_channels, stats, stats_groups,
                    x_f32=False):
    X = _c(_view(x0, batch * hw, c0, ld0))
    if c1:
        X = torch.cat([X, _c(_view(x1, batch * hw, c1, ld1))], 1)
    st = stats.view(batch, stats_groups, 2)
    chans = sample_channels.cpu() if sample_channels is not None else None
    for b in range(batch):
        ct = int(chans[b]) if chans is not None else c0 + c1
        if ct <= 0:
            continue
        xb = X[b * hw:(b + 1) * hw, :ct]
        g = (ct + group_size - 1) // group_size
        xg = xb.reshape(hw, g, group_size)
        _put(st[b, :g, 0], xg.sum((0, 2)), k=hw * group_size)  # overwritten, not accumulated (deterministic reduction)
        _put(st[b, :g, 1], (xg * xg).sum((0, 2)), k=hw * group_size)


def groupnorm_stats_from_partials(cs0, c0, cs1, c1, blocks, batch, group_size, sample_channels, stats, stats_groups):
    S = _c(cs0[0].view(batch, blocks, -1)[:, :, :c0]).sum(1)
    Q = _c(cs0[1].view(batch, blocks, -1)[:, :, :c0]).sum(1)
    if cs1 is not None:
        S = torch.cat([S, _c(cs1[0].view(batch, blocks, -1)[:, :, :c1]).sum(1)], 1)
        Q = torch.cat([Q, _c(cs1[1].view(batch, blocks, -1)[:, :, :c1]).sum(1)], 1)
    st = stats.view(batch, stats_groups, 2)
    chans = sample_channels.cpu() if sample_channels is not None else None
    for b in range(batch):
        ct = int(chans[b]) if chans is not None else S.shape[1]
        if ct <= 0:
            continue
        g = (ct + group_size - 1) // group_size
        _put(st[b, :g, 0], S[b, :ct].reshape(g, group_size).sum(1), k=blocks * group_size)
        _put(st[b, :g, 1], Q[b, :ct].reshape(g, group_size).sum(1), k=blocks * group_size)


def groupnorm_apply(x0, c0, ld0, x1, c1, ld1, y, ldy, batch, hw, group_size, eps, stats, stats_groups, gamma, beta,
                    affine_ld, sample_seg, sample_channels, gate, gate_ld, silu, x_f32=False, raw_out=None, raw_ld=0):
    X = _c(_view(x0, batch * hw, c0, ld0))
    if c1:
        X = torch.cat([X, _c(_view(x1, batch * hw, c1, ld1))], 1)
    chans = sample_channels.cpu() if sample_channels is not None else None
    segs = sample_seg.cpu() if sample_seg is not None else None
    if raw_out is not None:
        R = _view(raw_out, batch * hw, raw_ld, raw_ld)
        for b in range(batch):
            ct = int(chans[b]) if chans is not None else c0 + c1
            if ct > 0:
                _put(R[b * hw:(b + 1) * hw, :ct], X[b * hw:(b + 1) * hw, :ct])
    Y = _view(y, batch * hw, ldy, ldy)
    st = _c(stats.view(batch, stats_groups, 2))
    G = _c(gamma.reshape(-1, affine_ld))
    Bt = _c(beta.reshape(-1, affine_ld))
    for b in range(batch):
        ct = int(chans[b]) if chans is not None else c0 + c1
        if ct <= 0:
            continue
        seg = int(segs[b]) if segs is not None else 0
        g = ct // group_size
        n = hw * group_size
        mean = st[b, :g, 0] / n
        var = (st[b, :g, 1] / n - mean * mean).clamp(min=0)
        gt = _c(gate[b, :g]) if gate is not None else torch.ones(g, dtype=X.dtype, device=X.device)
        rstd = torch.rsqrt(gt * gt * var + eps)
        w = G[seg, :ct] * (rstd * gt).repeat_interleave(group_size)
        sh = Bt[seg, :ct] - mean.repeat_interleave(group_size) * w
        o = X[b * hw:(b + 1) * hw, :ct] * w + sh
        if silu:
            o = F.silu(o)
        cs = min((ct + 63) // 64 * 64, ldy)
        _put(Y[b * hw:(b + 1) * hw, :ct], o)
        _put(Y[b * hw:(b + 1) * hw, ct:cs], torch.zeros(hw, cs - ct, dtype=o.dtype, device=o.device), exact=True)


def ln_rowstats(partial, rows, C_, eps, out, sample_active=None, rows_per_sample=1):
    ps = _c(partial[:rows]).sum(1)
    mu = ps[:, 0] / C_
    _put(out[:rows, 0], mu, k=C_)
    _put(out[:rows, 1], torch.rsqrt((ps[:, 1] / C_ - mu * mu).clamp(min=0) + eps), k=C_)


def layernorm(x, ldx, y, ldy, rows, C_, eps, gamma, beta, sample_active=None, rows_per_sample=1):
    X = _c(_view(x, rows, C_, ldx))
    Y = _view(y, rows, C_, ldy)
    o = F.layer_norm(X, (C_,), _c(gamma), _c(beta), eps)
    _put_rows(Y, o, sample_active, rows_per_sample)


def _put_rows(D, S, sample_mask, rows_per_sample):
    """D[r] = S[r] for the rows of the samples whose mask entry is set (every row without a mask)."""
    if sample_mask is None:
        _put(D, S)
        return
    m = sample_mask.cpu().bool().tolist()
    b = 0
    while b < len(m):  # runs of consecutive selected samples as one region
        if not m[b]:
            b += 1
            continue
        e = b
        while e < len(m) and m[e]:
            e += 1
        _put(D[b * rows_per_sample:e * rows_per_sample], S[b * rows_per_sample:e * rows_per_sample])
        b = e


def depth_lerp(x, ldx, y, ldy, out, ldo, rows, C_, d, rows_per_sample):
    X = _c(_view(x, rows, C_, ldx))
    Yv = _c(_view(y, rows, C_, ldy))
    dd = _c(d).repeat_interleave(rows_per_sample)[:, None]
    _put(_view(out, rows, C_, ldo), (1 - dd) * X + dd * Yv)


def copy_rows(src, lds, dst, ldd, rows, C_, sample_mask=None, rows_per_sample=1):
    _put_rows(_view(dst, rows, C_, ldd), _view(src, rows, C_, lds).clone(), sample_mask, rows_per_sample)


def copy_rows_cvt(src, lds, dst, ldd, rows, C_, sample_mask=None, rows_per_sample=1):
    _put_rows(_view(dst, rows, C_, ldd), _view(src, rows, C_, lds).to(dst.dtype, copy=True), sample_mask,
              rows_per_sample)


def depth_lerp_f32(x, ldx, y, ldy, out, ldo, rows, C_, d, rows_per_sample):
    X = _c(_view(x, rows, C_, ldx))
    Yv = _c(_view(y, rows, C_, ldy)).clone()
    dd = _c(d).repeat_interleave(rows_per_sample)[:, None]
    _put(_view(out, rows, C_, ldo), (1 - dd) * X + dd * Yv)


def upsample2x_cvt(src, dst, batch, H, W, C_):
    upsample2x(src.to(torch.bfloat16), dst, batch, H, W, C_)


def upsample2x(src, dst, batch, H, W, C_):
    s = src.view(batch, H, W, C_)
    _put(dst.view(batch, 2 * H, 2 * W, C_), s.repeat_interleave(2, 1).repeat_interleave(2, 2))


def im2col_input(sample_nchw, dst, batch, cin, H, W):
    cols = F.unfold(_c(sample_nchw), 3, padding=1).reshape(batch, cin, 9, H * W).permute(0, 3, 2, 1).reshape(batch * H * W, 9 * cin)
    full = torch.zeros(dst.shape, dtype=cols.dtype, device=cols.device)
    full[:, :9 * cin] = cols
    _put(dst, full)


def timestep_embedding(t, dst, batch, dim):
    half = dim // 2
    f = torch.exp(-math.log(10000.0) * torch.arange(half, dtype=_CDT, device=t.device) / half)
    arg = _c(t)[:, None] * f[None]
    _put(dst, torch.cat([torch.cos(arg), torch.sin(arg)], 1))


def cast_f32_bf16(src, dst, n):
    _put(dst.view(-1)[:n], src.reshape(-1)[:n].clone())


def silu_bf16(src, dst, n):
    _put(dst.view(-1)[:n], F.silu(_c(src.reshape(-1)[:n])))


def attention(q, ldq, k, ldk, v, ldv, out, ldo, batch, n_q, n_kv, sample_heads, max_heads, scale, lse2=None):
    heads = sample_heads.cpu()
    for b in range(batch):
        nh = int(heads[b])
        if nh == 0:
            continue
        Q = _c(_view(q, (b + 1) * n_q, nh * 64, ldq)[b * n_q:]).reshape(n_q, nh, 64).transpose(0, 1)
        Kk = _c(_view(k, (b + 1) * n_kv, nh * 64, ldk)[b * n_kv:]).reshape(n_kv, nh, 64).transpose(0, 1)
        V = _c(_view(v, (b + 1) * n_kv, nh * 64, ldv)[b * n_kv:]).reshape(n_kv, nh, 64).transpose(0, 1)
        s = Q @ Kk.transpose(1, 2) * scale
        p = torch.softmax(s, -1)
        o = (p @ V).transpose(0, 1).reshape(n_q, nh * 64)
        # floor: the kernel rounds the probabilities to bf16 for the P @ V product (half an ulp of each weight on V)
        _put(_view(out, (b + 1) * n_q, nh * 64, ldo)[b * n_q:], o, k=n_kv, floor=2.0 ** -8 * float(V.pow(2).mean().sqrt()))
        if lse2 is not None:  # [batch, max_heads, n_q]: log-sum-exp of the scaled scores in the log2 domain
            _put(lse2.view(batch, max_heads, n_q)[b, :nh], torch.logsumexp(s, -1) / math.log(2.0), k=n_kv,
                 part="lse")


def attention_bwd(q, ldq, k, ldk, v, ldv, o, ldo, dout, lddo, lse2, delta, dq, lddq, dk, lddk, dv, lddv, batch, n_q,
                  n_kv, sample_heads, max_heads, scale):
    """dq, dk, dv of attention() for the kept heads of each sample (P from the scores, delta = rowsum(dout * o) with
    the forward output `o` as given); delta [batch, max_heads, n_q] is written too."""
    heads = sample_heads.cpu()
    for b in range(batch):
        nh = int(heads[b])
        if nh == 0:
            continue

        def rows(t, ld, n):
            return _c(_view(t, (b + 1) * n, nh * 64, ld)[b * n:]).reshape(n, nh, 64).transpose(0, 1)
        Q, Kk, V = rows(q, ldq, n_q), rows(k, ldk, n_kv), rows(v, ldv, n_kv)
        O, dO = rows(o, ldo, n_q), rows(dout, lddo, n_q)
        p = torch.softmax(Q @ Kk.transpose(1, 2) * scale, -1)
        dlt = (dO * O).sum(-1)
        dS = p * (dO @ V.transpose(1, 2) - dlt[..., None])
        # floor: the kernel forms dS = P * (dP - delta) after a cancellation and rounds it (and P) to bf16 for its
        # products: a few percent of each gradient's rms (2^-5; measured up to ~3 % on a B200)
        for t, ld, n, g in ((dq, lddq, n_q, dS @ Kk * scale), (dk, lddk, n_kv, dS.transpose(1, 2) @ Q * scale),
                            (dv, lddv, n_kv, p.transpose(1, 2) @ dO)):
            _put(_view(t, (b + 1) * n, nh * 64, ld)[b * n:], g.transpose(0, 1).reshape(n, nh * 64), k=n_kv,
                 floor=2.0 ** -5 * float(g.pow(2).mean().sqrt()), part="grad")
        _put(delta.view(batch, max_heads, n_q)[b, :nh], dlt, k=64, part="delta")


def wgrad(dy, ld_dy, a, ld_a, dw, dbias, rows, n_out, k_in, conv=None, splits=0, stride=1):
    """dw [n_out, taps * k_in] (OHWI) += dy^T a over the rows (3x3 taps, zero padding, stride 1 / 2 for conv =
    (batch, H, W) of the input); dbias += column sums of dy."""
    DY = _c(_view(dy, rows, n_out, ld_dy))
    if conv is None:
        g = DY.t() @ _c(_view(a, rows, k_in, ld_a))
        taps = 1
    else:
        batch, H, W = conv
        X = _c(_view(a, batch * H * W, k_in, ld_a)).reshape(batch, H, W, k_in).permute(0, 3, 1, 2)
        cols = F.unfold(X, 3, padding=1, stride=stride)                       # [batch, k_in * 9, Ho * Wo]
        g = torch.einsum("bln,bkl->nk", DY.reshape(batch, -1, n_out), cols)  # [n_out, k_in * 9], (c, tap) order
        g = g.reshape(n_out, k_in, 9).transpose(1, 2).reshape(n_out, 9 * k_in)
        taps = 9
    D = torch.as_strided(dw, (n_out, taps * k_in), (dw.stride(0), 1), dw.storage_offset())
    _put(D, _c(D) + g, k=rows)
    if dbias is not None:
        _put(dbias[:n_out], _c(dbias[:n_out]) + DY.sum(0), k=rows, part="bias")


def check_abort():
    return None


def install(monkeypatch):
    for name in ("grouped_gemm", "groupnorm_stats", "groupnorm_stats_from_partials", "groupnorm_apply", "layernorm", "ln_rowstats", "depth_lerp", "copy_rows",
                 "copy_rows_cvt", "depth_lerp_f32", "upsample2x_cvt",
                 "upsample2x", "im2col_input", "timestep_embedding", "cast_f32_bf16", "silu_bf16", "attention",
                 "check_abort"):
        monkeypatch.setattr(K, name, globals()[name])


# ------------------------------------------------------------------------------------------------
# router kernels (contract of csrc/router.cu), so the quantizer's HOST logic -- uniform draw order, phase
# protocol of the sharded Sinkhorn with its all-reduces -- can run under gloo in the GPU-less container
# ------------------------------------------------------------------------------------------------
def gumbel_gate(z, u, out, batch, n_width, n_depth, width_starts, n_gates, depth_order, temperature, base,
                non_zero_width):
    g = -torch.log(-torch.log(u + 1e-20) + 1e-20)
    y = torch.sigmoid((z[:, :n_width] + g[:, :n_width] + base) / temperature)
    ws = width_starts.tolist()
    if non_zero_width:
        y = y.clone()
        for i in range(n_gates):
            s, e = ws[i], ws[i + 1]
            dead = (y[:, s:e] >= 0.5).sum(1) == 0
            y[dead, s] += 0.5
    out[:, :n_width] = y
    if n_depth:
        x = torch.flip(torch.cumsum(torch.softmax(z[:, n_width:], 1), 1), dims=[1])
        x = torch.log(x + 1e-6) - torch.log1p(-(x - 1e-6))
        yd = torch.sigmoid((x + g[:, n_width:] + base) / temperature)
        out[:, n_width + depth_order.long()] = yd


def arch_normalize(gates, out, batch, dim, col_depth, col_scale, l2=True):
    cd = col_depth.long()
    hard = (gates >= 0.5).float()
    dep = gates[:, cd.clamp_min(0)]
    v = torch.where(cd[None, :] >= 0, gates * dep, hard) * col_scale[None, :]
    out.copy_(v / v.norm(dim=1, keepdim=True) if l2 else v)


def route_cosine(a_norm, codes_norm, scores, indices, batch, dim, n_codes):
    s = (a_norm.double() @ codes_norm.double().t()).float()
    scores.copy_(s)
    indices.copy_(torch.argmax(s, dim=1))


def sinkhorn_phase(phase, Q, scores, partial, indices, batch_local, batch_global, n_codes, epsilon, first_iter):
    if phase == 0:
        Q.copy_(torch.exp(scores / epsilon))
        partial[0] = Q.double().sum()
    elif phase == 1:
        if first_iter:
            Q.div_(partial[0].float())
        partial[1:1 + n_codes] = Q.double().sum(0)
    elif phase == 2:
        Q.div_(partial[1:1 + n_codes].float()[None, :])
        Q.div_(float(n_codes))
        Q.div_(Q.sum(1, keepdim=True))
        Q.div_(float(batch_global))
    else:
        Q.mul_(float(batch_global))
        indices.copy_(torch.argmax(Q, dim=1))


def route_sinkhorn(scores, Q, partial, indices, batch, n_codes, epsilon, iterations):
    sinkhorn_phase(0, Q, scores, partial, indices, batch, batch, n_codes, epsilon, 0)
    for it in range(iterations):
        sinkhorn_phase(1, Q, scores, partial, indices, batch, batch, n_codes, epsilon, it == 0)
        sinkhorn_phase(2, Q, scores, partial, indices, batch, batch, n_codes, epsilon, 0)
    sinkhorn_phase(3, Q, scores, partial, indices, batch, batch, n_codes, epsilon, 0)


def install_router(setattr_fn):
    """setattr_fn(obj, name, value): monkeypatch.setattr or plain setattr (spawned workers)."""
    from diffusion_pruning_b200.quantizer import StructureVectorQuantizer
    for name in ("gumbel_gate", "arch_normalize", "route_cosine", "sinkhorn_phase", "route_sinkhorn"):
        setattr_fn(K, name, globals()[name])
    setattr_fn(StructureVectorQuantizer, "_require_cuda", staticmethod(lambda t, what: None))
