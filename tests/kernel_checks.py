"""Per-kernel numerics checks: each hand-written CUDA kernel against a plain PyTorch fp32 reference of
the same op on the same (bf16-rounded) inputs. Used by tests/test_kernels_gpu.py and by
tools/kernel_check.py (which runs all of them without stopping at the first failure)."""
from __future__ import annotations

import math

import torch
import torch.nn.functional as F

from diffusion_pruning_b200 import kernels as K
from diffusion_pruning_b200._lib import (A_CONV3X3, A_CONV3X3_S2, A_LINEAR, EPI_GEGLU, EPI_RES_F32, EPI_SILU, OUT_BF16,
                                         OUT_F32, OUT_F32_NCHW)

DEV = "cuda"


def _rand(*shape, scale=1.0, seed=0):
    g = torch.Generator(device="cpu").manual_seed(seed)
    return (torch.randn(*shape, generator=g) * scale).to(DEV)


def _close(got, ref, atol, rtol, what):
    got = got.float()
    ref = ref.float()
    err = (got - ref).abs()
    tol = atol + rtol * ref.abs()
    bad = (err > tol).sum().item()
    assert bad == 0, f"{what}: {bad}/{err.numel()} mismatches, max err {err.max().item():.4g}, ref max {ref.abs().max().item():.4g}"


def _conv_ref(x, w, b, stride):
    """3x3 / pad 1 conv as unfold + matmul (keeps cuDNN, whose first load takes minutes on a cold box, out)."""
    B, Cin, H, W = x.shape
    cols = F.unfold(x, 3, padding=1, stride=stride)  # [B, Cin*9, L]
    y = w.reshape(w.shape[0], -1) @ cols + b[None, :, None]
    return y.reshape(B, w.shape[0], H // stride, W // stride)


def _sdpa_ref(q, k, v, scale):
    p = torch.softmax((q @ k.transpose(-1, -2)) * scale, dim=-1)
    return p @ v


def check_gemm_linear(M=1000, Kd=320, N=320, bn=160, bias=True, residual=True, silu=False, seed=0):
    a = _rand(M, Kd, seed=seed).bfloat16()
    w = _rand(N, Kd, scale=Kd ** -0.5, seed=seed + 1).bfloat16()
    b = _rand(N, seed=seed + 2) if bias else None
    res = _rand(M, N, seed=seed + 3).bfloat16() if residual else None
    out = torch.full((M, N), float("nan"), device=DEV, dtype=torch.bfloat16)
    sched = K.build_schedule([K.Segment(0, M, N, (Kd + 63) // 64)], bn, DEV)
    K.grouped_gemm(a, w, out, sched, a_ld=Kd, a_k=Kd, a_rows=M, out_ld=N, bias=b, residual=res, res_ld=N,
                   flags=EPI_SILU if silu else 0)
    K.check_abort()
    ref = a.float() @ w.float().t()
    if bias:
        ref = ref + b
    if silu:
        ref = F.silu(ref)
    if residual:
        ref = ref + res.float()
    _close(out, ref, 2e-2, 1e-2, f"gemm_linear M{M} K{Kd} N{N} bn{bn}")


def check_gemm_grouped(seed=0, HW=256, C=320, N=320, samples=(3, 2, 4), n_valid=(250, 320, 130), k_valid=(192, 320, 70),
                       active=(True, True, False)):
    """3 expert buckets: different kept N / kept K, one depth-dropped; compacted weight blocks. With C >= 1280 the
    launch takes the 2-SM scheme; HW not a multiple of 128 puts bucket starts off the 128-row grid."""
    M = sum(samples) * HW
    a = torch.zeros(M, C, device=DEV, dtype=torch.bfloat16)
    w = torch.zeros(3 * N, C, device=DEV, dtype=torch.bfloat16)
    bias = torch.zeros(3 * N, device=DEV)
    out = torch.full((M, N), 7.0, device=DEV, dtype=torch.bfloat16)
    segs, refs = [], []
    r0 = 0
    for e in range(3):
        rows = samples[e] * HW
        ae = _rand(rows, k_valid[e], seed=seed + 10 * e).bfloat16()
        we = _rand(n_valid[e], k_valid[e], scale=k_valid[e] ** -0.5, seed=seed + 10 * e + 1).bfloat16()
        be = _rand(n_valid[e], seed=seed + 10 * e + 2)
        a[r0:r0 + rows, :k_valid[e]] = ae
        w[e * N:e * N + n_valid[e], :k_valid[e]] = we
        bias[e * N:e * N + n_valid[e]] = be
        segs.append(K.Segment(r0, r0 + rows, n_valid[e], (k_valid[e] + 63) // 64, w_row_off=e * N, vec_off=e * N,
                              n_store=min((n_valid[e] + 63) // 64 * 64, N), active=active[e]))
        refs.append((r0, rows, ae.float() @ we.float().t() + be))
        r0 += rows
    sched = K.build_schedule(segs, 128, DEV)
    K.grouped_gemm(a, w, out, sched, a_ld=C, a_k=C, a_rows=M, out_ld=N, bias=bias, rows_per_sample=HW)
    K.check_abort()
    for e, (r0, rows, ref) in enumerate(refs):
        blk = out[r0:r0 + rows].float()
        if not active[e]:
            assert (blk == 7.0).all(), "inactive bucket must not be written"
            continue
        _close(blk[:, :n_valid[e]], ref, 2e-2, 1e-2, f"grouped bucket {e}")
        ns = min((n_valid[e] + 63) // 64 * 64, N)
        assert (blk[:, n_valid[e]:ns] == 0).all(), f"bucket {e}: K padding columns must be zero"
        assert (blk[:, ns:] == 7.0).all(), f"bucket {e}: columns past n_store must be untouched"


def check_conv3x3(B=3, H=16, W=16, Cin=128, Cout=96, bn=96, stride=1, border=False, temb=True, seed=0):
    x = _rand(B, Cin, H, W, seed=seed).bfloat16()
    w = _rand(Cout, Cin, 3, 3, scale=(9 * Cin) ** -0.5, seed=seed + 1).bfloat16()
    b = _rand(Cout, seed=seed + 2)
    Ho, Wo = H // stride, W // stride
    x_nhwc = x.permute(0, 2, 3, 1).contiguous()
    w_packed = w.permute(0, 2, 3, 1).reshape(Cout, 9 * Cin).contiguous()
    out = torch.full((B * Ho * Wo, Cout), float("nan"), device=DEV, dtype=torch.bfloat16)
    rv = _rand(B, Cout, seed=seed + 3) if temb else None
    tab = _rand(9, Cout, seed=seed + 4) if border else None
    mode = A_CONV3X3 if stride == 1 else A_CONV3X3_S2
    sched = K.build_schedule([K.Segment(0, B * Ho * Wo, Cout, (Cin + 63) // 64)], bn, DEV, mode=mode, Ho=Ho, Wo=Wo)
    K.grouped_gemm(x_nhwc, w_packed, out, sched, a_ld=Cin, a_k=Cin, a_rows=B * H * W, mode=mode, batch=B, H=H, W=W,
                   k_tap_pitch=Cin, out_ld=Cout, bias=b, rowvec=rv, rowvec_ld=Cout, rows_per_sample=Ho * Wo,
                   border_tab=tab, tab_ld=Cout)
    K.check_abort()
    ref = _conv_ref(x.float(), w.float(), b, stride)
    if temb:
        ref = ref + rv[:, :, None, None]
    if border:
        ys = torch.tensor([0 if y == 0 else (2 if y == Ho - 1 else 1) for y in range(Ho)], device=DEV)
        xs = torch.tensor([0 if x_ == 0 else (2 if x_ == Wo - 1 else 1) for x_ in range(Wo)], device=DEV)
        cls = ys[:, None] * 3 + xs[None, :]
        ref = ref + tab[cls].permute(2, 0, 1)[None]
    ref = ref.permute(0, 2, 3, 1).reshape(B * Ho * Wo, Cout)
    _close(out, ref, 2e-2, 1e-2, f"conv3x3 s{stride} B{B} {H}x{W} {Cin}->{Cout}")


def check_conv3x3_fused_shortcut(B=2, H=32, W=32, Cin=320, Cout=320, C2=448, bn=160, seed=0):
    """3x3 conv (halo-tile scheme: 8 x 16 boxes, 2-SM) with the ResNet's 1x1 conv_shortcut over a second tensor accumulated
    into the same tiles (aptp_gemm_args.a2 / w2), fp32 rows out with the border table and both biases."""
    x = _rand(B, Cin, H, W, seed=seed).bfloat16()
    w = _rand(Cout, Cin, 3, 3, scale=(9 * Cin) ** -0.5, seed=seed + 1).bfloat16()
    b = _rand(Cout, seed=seed + 2)
    x2 = _rand(B * H * W, C2, seed=seed + 3).bfloat16()
    w2 = _rand(Cout, C2, scale=C2 ** -0.5, seed=seed + 4).bfloat16()
    x_nhwc = x.permute(0, 2, 3, 1).contiguous()
    w_packed = w.permute(0, 2, 3, 1).reshape(Cout, 9 * Cin).contiguous()
    out = torch.full((B * H * W, Cout), float("nan"), device=DEV, dtype=torch.float32)
    sched = K.build_schedule([K.Segment(0, B * H * W, Cout, (Cin + 63) // 64)], bn, DEV, mode=A_CONV3X3, Ho=H, Wo=W)
    assert sched.box == (8, 16, 1)
    K.grouped_gemm(x_nhwc, w_packed, out, sched, a_ld=Cin, a_k=Cin, a_rows=B * H * W, mode=A_CONV3X3, batch=B, H=H, W=W,
                   k_tap_pitch=Cin, out_ld=Cout, out_mode=OUT_F32, bias=b, rows_per_sample=H * W, a2=x2, a2_ld=C2, a2_k=C2,
                   w2=w2)
    K.check_abort()
    ref = _conv_ref(x.float(), w.float(), b, 1).permute(0, 2, 3, 1).reshape(B * H * W, Cout) + x2.float() @ w2.float().t()
    _close(out, ref, 2e-2, 1e-2, "conv3x3 + fused 1x1 shortcut")


def check_geglu(M=512, Kd=320, inner=1280, n_keep=1000, bn=256, seed=0):
    """Packed rows interleave [bn/2 h | bn/2 g] per tile; output = h * gelu(g) compacted."""
    a = _rand(M, Kd, seed=seed).bfloat16()
    w = _rand(2 * inner, Kd, scale=Kd ** -0.5, seed=seed + 1).bfloat16()
    b = _rand(2 * inner, seed=seed + 2)
    keep = torch.arange(n_keep, device=DEV)  # keep first n_keep hidden columns
    half = bn // 2
    n_tiles = (n_keep + half - 1) // half
    wp = torch.zeros(n_tiles * bn, Kd, device=DEV, dtype=torch.bfloat16)
    bp = torch.zeros(n_tiles * bn, device=DEV)
    for t in range(n_tiles):
        cols = keep[t * half:(t + 1) * half]
        wp[t * bn:t * bn + len(cols)] = w[cols]
        wp[t * bn + half:t * bn + half + len(cols)] = w[inner + cols]
        bp[t * bn:t * bn + len(cols)] = b[cols]
        bp[t * bn + half:t * bn + half + len(cols)] = b[inner + cols]
    n_store = (n_keep + 63) // 64 * 64
    out = torch.full((M, n_store), float("nan"), device=DEV, dtype=torch.bfloat16)
    sched = K.build_schedule([K.Segment(0, M, n_keep, (Kd + 63) // 64, n_store=n_store)], bn, DEV, geglu=True)
    K.grouped_gemm(a, wp, out, sched, a_ld=Kd, a_k=Kd, a_rows=M, out_ld=n_store, bias=bp, flags=EPI_GEGLU)
    K.check_abort()
    proj = a.float() @ w.float().t() + b
    ref = proj[:, :inner][:, :n_keep] * F.gelu(proj[:, inner:][:, :n_keep])
    _close(out[:, :n_keep], ref, 2e-2, 1e-2, "geglu")
    assert (out[:, n_keep:].float() == 0).all(), "geglu: padding must be zero"



def check_gemm_epilogue_mix(seed=0):
    """Soft-gate multiplier, column offset into a fused [q|k|v]-style output, residual aliasing the output
    (in-place token stream update), ragged last tile."""
    M, Kd, N, HW, gg = 1000, 320, 320, 250, 64
    B = M // HW
    a = _rand(M, Kd, seed=seed).bfloat16()
    w = _rand(N, Kd, scale=Kd ** -0.5, seed=seed + 1).bfloat16()
    b = _rand(N, seed=seed + 2)
    gate = torch.rand(B, N // gg, device=DEV) * 0.8 + 0.1
    out = torch.full((M, 3 * N), 3.0, device=DEV, dtype=torch.bfloat16)
    sched = K.build_schedule([K.Segment(0, M, N, (Kd + 63) // 64, out_col_off=N)], 160, DEV)
    K.grouped_gemm(a, w, out, sched, a_ld=Kd, a_k=Kd, a_rows=M, out_ld=3 * N, bias=b, rows_per_sample=HW, gate=gate,
                   gate_ld=N // gg, gate_group=gg)
    K.check_abort()
    ref = (a.float() @ w.float().t() + b) * gate.repeat_interleave(HW, 0).repeat_interleave(gg, 1)
    _close(out[:, N:2 * N], ref, 2e-2, 1e-2, "epilogue gate + out_col_off")
    assert (out[:, :N].float() == 3.0).all() and (out[:, 2 * N:].float() == 3.0).all(), "neighbour columns touched"
    tok = _rand(M, N, seed=seed + 5).bfloat16()
    tok0 = tok.clone()
    sched = K.build_schedule([K.Segment(0, M, N, (Kd + 63) // 64)], 128, DEV)
    K.grouped_gemm(a, w, tok, sched, a_ld=Kd, a_k=Kd, a_rows=M, out_ld=N, bias=b, residual=tok, res_ld=N)
    K.check_abort()
    _close(tok, a.float() @ w.float().t() + b + tok0.float(), 2e-2, 1e-2, "in-place residual")


def check_conv_residual(B=3, H=16, W=16, Cin=128, Cout=128, bn=128, seed=0):
    """conv2 of a ResNet: bias + border table + residual read through a different row pitch."""
    x = _rand(B, Cin, H, W, seed=seed).bfloat16()
    w = _rand(Cout, Cin, 3, 3, scale=(9 * Cin) ** -0.5, seed=seed + 1).bfloat16()
    b = _rand(Cout, seed=seed + 2)
    res = _rand(B * H * W, Cout + 64, seed=seed + 3).bfloat16()
    x_nhwc = x.permute(0, 2, 3, 1).contiguous()
    w_packed = w.permute(0, 2, 3, 1).reshape(Cout, 9 * Cin).contiguous()
    out = torch.full((B * H * W, Cout), float("nan"), device=DEV, dtype=torch.bfloat16)
    sched = K.build_schedule([K.Segment(0, B * H * W, Cout, (Cin + 63) // 64)], bn, DEV, mode=A_CONV3X3, Ho=H, Wo=W)
    K.grouped_gemm(x_nhwc, w_packed, out, sched, a_ld=Cin, a_k=Cin, a_rows=B * H * W, mode=A_CONV3X3, batch=B, H=H,
                   W=W, k_tap_pitch=Cin, out_ld=Cout, bias=b, rows_per_sample=H * W, residual=res, res_ld=Cout + 64)
    K.check_abort()
    ref = _conv_ref(x.float(), w.float(), b, 1).permute(0, 2, 3, 1).reshape(B * H * W, Cout) + res[:, :Cout].float()
    _close(out, ref, 2e-2, 1e-2, "conv3x3 + residual")


def check_geglu_gate(seed=0):
    M, Kd, inner, HW, gw = 512, 320, 1280, 256, 32
    a = _rand(M, Kd, seed=seed).bfloat16()
    w = _rand(2 * inner, Kd, scale=Kd ** -0.5, seed=seed + 1).bfloat16()
    b = _rand(2 * inner, seed=seed + 2)
    gate = torch.rand(M // HW, gw, device=DEV) * 0.9 + 0.05
    bn, half = 256, 128
    nt = inner // half
    wp = torch.stack([w[:inner].view(nt, half, Kd), w[inner:].view(nt, half, Kd)], 1).reshape(nt * bn, Kd).contiguous()
    bp = torch.stack([b[:inner].view(nt, half), b[inner:].view(nt, half)], 1).reshape(nt * bn).contiguous()
    out = torch.full((M, inner), float("nan"), device=DEV, dtype=torch.bfloat16)
    sched = K.build_schedule([K.Segment(0, M, inner, (Kd + 63) // 64)], bn, DEV, geglu=True)
    K.grouped_gemm(a, wp, out, sched, a_ld=Kd, a_k=Kd, a_rows=M, out_ld=inner, bias=bp, flags=EPI_GEGLU,
                   rows_per_sample=HW, gate=gate, gate_ld=gw, gate_group=inner // gw)
    K.check_abort()
    proj = a.float() @ w.float().t() + b
    gfull = gate.repeat_interleave(HW, 0).repeat_interleave(inner // gw, 1)
    ref = (proj[:, :inner] * gfull) * F.gelu(proj[:, inner:] * gfull)
    _close(out, ref, 2e-2, 1e-2, "geglu + soft gate")


def check_out_modes(seed=0):
    B, HW, Kd, N = 2, 256, 320, 4
    a = _rand(B * HW, Kd, seed=seed).bfloat16()
    w = torch.zeros(32, Kd, device=DEV, dtype=torch.bfloat16)
    w[:N] = _rand(N, Kd, scale=Kd ** -0.5, seed=seed + 1).bfloat16()
    out = torch.full((B, N, HW), float("nan"), device=DEV, dtype=torch.float32)
    sched = K.build_schedule([K.Segment(0, B * HW, N, Kd // 64)], 32, DEV)
    K.grouped_gemm(a, w, out, sched, a_ld=Kd, a_k=Kd, a_rows=B * HW, out_ld=N, out_mode=OUT_F32_NCHW,
                   rows_per_sample=HW)
    K.check_abort()
    ref = (a.float() @ w[:N].float().t()).reshape(B, HW, N).permute(0, 2, 1)
    _close(out, ref, 1e-3, 1e-3, "out f32 nchw")
    out2 = torch.full((B * HW, 32), float("nan"), device=DEV, dtype=torch.float32)
    sched = K.build_schedule([K.Segment(0, B * HW, 32, Kd // 64)], 32, DEV)
    K.grouped_gemm(a, w, out2, sched, a_ld=Kd, a_k=Kd, a_rows=B * HW, out_ld=32, out_mode=OUT_F32)
    K.check_abort()
    _close(out2, a.float() @ w.float().t(), 1e-3, 1e-3, "out f32")


def check_groupnorm(B=3, HW=256, C0=320, C1=0, groups=32, silu=True, gate=False, compact=False, seed=0, f32=False):
    C = C0 + C1
    gs = C // groups
    x0 = _rand(B * HW, C0, seed=seed).bfloat16() * 2 + 0.5
    x1 = _rand(B * HW, C1, seed=seed + 1).bfloat16() if C1 else None
    if f32:  # fp32 residual-stream rows (values that bf16 cannot represent exactly)
        x0 = x0.float() + _rand(B * HW, C0, seed=seed + 7) * 1e-3
        x1 = (x1.float() + _rand(B * HW, C1, seed=seed + 8) * 1e-3) if C1 else None
    gamma = _rand(2, C, seed=seed + 2) * 0.2 + 1
    beta = _rand(2, C, seed=seed + 3) * 0.2
    sample_seg = torch.tensor([i % 2 for i in range(B)], device=DEV, dtype=torch.int32)
    if compact:
        ch = torch.tensor([gs * (groups - 3 * (i % 3)) for i in range(B)], device=DEV, dtype=torch.int32)
    else:
        ch = None
    g = (torch.rand(B, groups, device=DEV) * 0.8 + 0.2) if gate else None
    stats = torch.zeros(B, groups, 2, device=DEV)
    y = torch.full((B * HW, C), float("nan"), device=DEV, dtype=torch.bfloat16)
    stats.fill_(float("nan"))  # the statistics pass overwrites (no zeroing contract any more)
    K.groupnorm_stats(x0, C0, C0, x1, C1, C1, B, HW, gs, ch, stats, groups, x_f32=f32)
    K.groupnorm_apply(x0, C0, C0, x1, C1, C1, y, C, B, HW, gs, 1e-5, stats, groups, gamma, beta, C, sample_seg, ch, g,
                      groups, silu, x_f32=f32)
    torch.cuda.synchronize()
    # deterministic reduction: a second pass gives bit-identical statistics
    stats2 = torch.full_like(stats, float("nan"))
    K.groupnorm_stats(x0, C0, C0, x1, C1, C1, B, HW, gs, ch, stats2, groups, x_f32=f32)
    torch.cuda.synchronize()
    for b in range(B):
        ng = (int(ch[b]) if compact else C) // gs
        assert torch.equal(stats[b, :ng], stats2[b, :ng]), "groupnorm statistics are not bit-reproducible"
        xs = (torch.cat([x0.float(), x1.float()], 1) if C1 else x0.float())[b * HW:(b + 1) * HW, :ng * gs]
        ref_sum = xs.double().reshape(HW, ng, gs).sum(dim=(0, 2))
        ref_sq = (xs.double() ** 2).reshape(HW, ng, gs).sum(dim=(0, 2))
        _close(stats[b, :ng, 0], ref_sum, 1e-2, 1e-5, "groupnorm sum")
        _close(stats[b, :ng, 1], ref_sq, 1e-2, 1e-5, "groupnorm sumsq")
    xf = torch.cat([x0.float(), x1.float()], 1) if C1 else x0.float()
    for b in range(B):
        cb = int(ch[b]) if compact else C
        xb = xf[b * HW:(b + 1) * HW, :cb].t().reshape(1, cb, HW)
        if gate:
            xb = xb * g[b].repeat_interleave(gs)[:cb].reshape(1, cb, 1)
        ref = F.group_norm(xb, cb // gs, gamma[b % 2, :cb], beta[b % 2, :cb], 1e-5)
        if silu:
            ref = F.silu(ref)
        ref = ref[0].t()
        _close(y[b * HW:(b + 1) * HW, :cb], ref, 3e-2, 1e-2, f"groupnorm sample {b}")
        if compact:
            pad = min((cb + 63) // 64 * 64, C)
            assert (y[b * HW:(b + 1) * HW, cb:pad].float() == 0).all(), "groupnorm: K padding must be zero"


def check_layernorm(rows=1000, C=640, seed=0):
    x = (_rand(rows, C, seed=seed) * 3 + 1).bfloat16()
    gamma = _rand(C, seed=seed + 1) * 0.2 + 1
    beta = _rand(C, seed=seed + 2) * 0.2
    y = torch.empty_like(x)
    K.layernorm(x, C, y, C, rows, C, 1e-5, gamma, beta)
    torch.cuda.synchronize()
    _close(y, F.layer_norm(x.float(), (C,), gamma, beta, 1e-5), 3e-2, 1e-2, "layernorm")


def check_elementwise(seed=0):
    B, H, W, C = 2, 8, 8, 64
    x = _rand(B * H * W, C, seed=seed).bfloat16()
    y = _rand(B * H * W, C, seed=seed + 1).bfloat16()
    d = torch.tensor([0.25, 1.0], device=DEV)
    out = torch.empty_like(x)
    K.depth_lerp(x, C, y, C, out, C, B * H * W, C, d, H * W)
    dd = d.repeat_interleave(H * W)[:, None]
    _close(out, (1 - dd) * x.float() + dd * y.float(), 1e-2, 1e-2, "depth_lerp")
    up = torch.empty(B * 4 * H * W, C, device=DEV, dtype=torch.bfloat16)
    K.upsample2x(x, up, B, H, W, C)
    ref = F.interpolate(x.reshape(B, H, W, C).permute(0, 3, 1, 2).float(), scale_factor=2.0, mode="nearest")
    _close(up, ref.permute(0, 2, 3, 1).reshape(-1, C), 0, 0, "upsample2x")
    dst = torch.full((B * H * W, 2 * C), 5.0, device=DEV, dtype=torch.bfloat16)
    mask = torch.tensor([0, 1], device=DEV, dtype=torch.uint8)
    K.copy_rows(x, C, dst[:, C:], 2 * C, B * H * W, C, mask, H * W)
    torch.cuda.synchronize()
    assert (dst[:H * W].float() == 5.0).all() and (dst[H * W:, :C].float() == 5.0).all()
    assert torch.equal(dst[H * W:, C:], x[H * W:])
    s = torch.randn(B, 4, H, W, device=DEV)
    col = torch.empty(B * H * W, 64, device=DEV, dtype=torch.bfloat16)
    K.im2col_input(s, col, B, 4, H, W)
    ref = F.unfold(s, 3, padding=1)  # [B, C*9, HW] with index c*9 + tap
    ref = ref.reshape(B, 4, 9, H * W).permute(0, 3, 2, 1).reshape(B * H * W, 36)
    _close(col[:, :36], ref, 1e-2, 1e-2, "im2col")
    assert (col[:, 36:].float() == 0).all()
    t = torch.tensor([981.0, 21.0], device=DEV)
    emb = torch.empty(B, 320, device=DEV, dtype=torch.bfloat16)
    K.timestep_embedding(t, emb, B, 320)
    k = torch.arange(160, device=DEV, dtype=torch.float32)
    f = torch.exp(-math.log(10000.0) * k / 160)
    ref = torch.cat([torch.cos(t[:, None] * f), torch.sin(t[:, None] * f)], 1)
    _close(emb, ref, 1e-2, 1e-2, "timestep_embedding")


def check_stream_f32(seed=0):
    """fp32 residual-stream helpers: converting row copies, fp32 depth lerp (in place), upsample from fp32, vector cast."""
    B, H, W, C = 2, 8, 8, 64
    M = B * H * W
    x = _rand(M, C, seed=seed)
    y = _rand(M, C, seed=seed + 1)
    d = torch.tensor([0.25, 1.0], device=DEV)
    dd = d.repeat_interleave(H * W)[:, None]
    out = y.clone()
    K.depth_lerp_f32(x, C, out, C, out, C, M, C, d, H * W)
    _close(out, (1 - dd) * x + dd * y, 1e-6, 1e-6, "depth_lerp_f32")
    mask = torch.tensor([0, 1], device=DEV, dtype=torch.uint8)
    for sdt in (torch.float32, torch.bfloat16):
        for ddt in (torch.float32, torch.bfloat16):
            src = x.to(sdt)
            dst = torch.full((M, 2 * C), 5.0, device=DEV, dtype=ddt)
            K.copy_rows_cvt(src, C, dst[:, C:], 2 * C, M, C, mask, H * W)
            torch.cuda.synchronize()
            assert (dst[:H * W].float() == 5.0).all() and (dst[H * W:, :C].float() == 5.0).all()
            assert torch.equal(dst[H * W:, C:], src[H * W:].to(ddt)), f"copy_rows_cvt {sdt} -> {ddt}"
    up = torch.empty(B * 4 * H * W, C, device=DEV, dtype=torch.bfloat16)
    K.upsample2x_cvt(x, up, B, H, W, C)
    ref = F.interpolate(x.reshape(B, H, W, C).permute(0, 3, 1, 2), scale_factor=2.0, mode="nearest")
    assert torch.equal(up, ref.permute(0, 2, 3, 1).reshape(-1, C).bfloat16()), "upsample2x_cvt"
    c16 = torch.empty(M, C, device=DEV, dtype=torch.bfloat16)
    K.cast_f32_bf16(x, c16, M * C)
    assert torch.equal(c16, x.bfloat16()), "cast_f32_bf16 (vector path)"
    c16b = torch.empty(M * C - 3, device=DEV, dtype=torch.bfloat16)
    K.cast_f32_bf16(x.reshape(-1)[3:], c16b, M * C - 3)
    assert torch.equal(c16b, x.reshape(-1)[3:].bfloat16()), "cast_f32_bf16 (scalar path)"


def check_gemm_res_f32(conv=False, seed=0):
    """fp32 output + fp32 residual (APTP_EPI_RES_F32), in place: the block outputs of the fp32 residual stream."""
    if conv:
        B, H, W, Cin, Cout, bn = 2, 16, 16, 128, 192, 192
        x = _rand(B, Cin, H, W, seed=seed).bfloat16()
        w = _rand(Cout, Cin, 3, 3, scale=(9 * Cin) ** -0.5, seed=seed + 1).bfloat16()
        b = _rand(Cout, seed=seed + 2)
        M = B * H * W
        a = x.permute(0, 2, 3, 1).reshape(M, Cin).contiguous()
        wp = w.permute(0, 2, 3, 1).reshape(Cout, 9 * Cin).contiguous()
        res = _rand(M, Cout, seed=seed + 3)
        out = res.clone()
        sched = K.build_schedule([K.Segment(0, M, Cout, (Cin + 63) // 64)], bn, DEV, mode=A_CONV3X3, Ho=H, Wo=W)
        K.grouped_gemm(a, wp, out, sched, a_ld=Cin, a_k=Cin, a_rows=M, mode=A_CONV3X3, batch=B, H=H, W=W,
                       k_tap_pitch=Cin, out_ld=Cout, out_mode=OUT_F32, bias=b, residual=out, res_ld=Cout,
                       flags=EPI_RES_F32, rows_per_sample=H * W)
        K.check_abort()
        ref = _conv_ref(x.float(), w.float(), b, 1).permute(0, 2, 3, 1).reshape(M, Cout) + res
    else:
        M, Kd, N, bn = 1000, 320, 320, 160
        a = _rand(M, Kd, seed=seed).bfloat16()
        w = _rand(N, Kd, scale=Kd ** -0.5, seed=seed + 1).bfloat16()
        b = _rand(N, seed=seed + 2)
        res = _rand(M, N, seed=seed + 3) * 3
        out = torch.full((M, N), float("nan"), device=DEV, dtype=torch.float32)
        sched = K.build_schedule([K.Segment(0, M, N, (Kd + 63) // 64)], bn, DEV)
        K.grouped_gemm(a, w, out, sched, a_ld=Kd, a_k=Kd, a_rows=M, out_ld=N, out_mode=OUT_F32, bias=b, residual=res,
                       res_ld=N, flags=EPI_RES_F32)
        K.check_abort()
        ref = a.float() @ w.float().t() + b + res
    _close(out, ref, 2e-3, 1e-4, "gemm fp32 out + fp32 residual")


def check_gemm_ln_fold(geglu=False, seed=0, C=320):
    """LayerNorm folded into the consumer GEMM (APTP_EPI_LN_FOLD) with the row statistics written by the producer GEMM's
    epilogue (rowstat_out): producer = Linear + residual -> x (bf16); consumer = Linear(LayerNorm(x)) [or GEGLU].
    C = 1280 runs producer and consumer in the 2-SM scheme."""
    M, N = 1000, 640
    a0 = _rand(M, C, seed=seed).bfloat16()
    w0 = _rand(C, C, scale=C ** -0.5, seed=seed + 1).bfloat16()
    res = (_rand(M, C, seed=seed + 2) * 2 + 0.7).bfloat16()
    x = res.clone()
    part = torch.full((M, C // 32, 2), float("nan"), device=DEV)
    sched = K.build_schedule([K.Segment(0, M, C, C // 64)], 160, DEV)
    K.grouped_gemm(a0, w0, x, sched, a_ld=C, a_k=C, a_rows=M, out_ld=C, residual=x, res_ld=C, rowstat_out=part)
    K.check_abort()
    xr = (a0.float() @ w0.float().t() + res.float())
    _close(x, xr, 3e-2, 1e-2, "producer output")
    ref_p = torch.stack([xr.reshape(M, C // 32, 32).sum(-1), (xr ** 2).reshape(M, C // 32, 32).sum(-1)], -1)
    _close(part, ref_p, 2e-2, 2e-3, "row-stat partials")
    gamma = _rand(C, seed=seed + 3) * 0.2 + 1
    beta = _rand(C, seed=seed + 4) * 0.2
    rs = torch.full((M, 2), float("nan"), device=DEV)
    K.ln_rowstats(part, M, C, 1e-5, rs)
    _close(rs[:, 0], xr.mean(1), 1e-3, 1e-3, "ln mean")
    _close(rs[:, 1], torch.rsqrt(xr.var(1, unbiased=False) + 1e-5), 1e-3, 2e-3, "ln rstd")
    xs = x.float()  # what the consumer reads
    ln = F.layer_norm(xs, (C,), gamma, beta, 1e-5)
    if not geglu:
        w = _rand(N, C, scale=C ** -0.5, seed=seed + 5)
        b = _rand(N, seed=seed + 6)
        wf = (w * gamma[None]).bfloat16()
        colsum = wf.float().sum(1).contiguous()
        bias = (w @ beta + b).contiguous()
        out = torch.full((M, N), float("nan"), device=DEV, dtype=torch.bfloat16)
        sched = K.build_schedule([K.Segment(0, M, N, C // 64)], 160, DEV)
        K.grouped_gemm(x, wf, out, sched, a_ld=C, a_k=C, a_rows=M, out_ld=N, bias=bias, ln_colsum=colsum,
                       ln_rowstats=rs)
        K.check_abort()
        _close(out, ln @ w.t() + b, 4e-2, 2e-2, "ln-fold linear")
    else:
        inner, bn = 640, 256
        half = bn // 2
        w = _rand(2 * inner, C, scale=C ** -0.5, seed=seed + 5)
        b = _rand(2 * inner, seed=seed + 6) * 0.1
        nt = inner // half
        wg = w * gamma[None]
        wp = torch.stack([wg[:inner].reshape(nt, half, C), wg[inner:].reshape(nt, half, C)], 1).reshape(nt * bn, C).bfloat16()
        bb = w @ beta + b
        bp = torch.stack([bb[:inner].reshape(nt, half), bb[inner:].reshape(nt, half)], 1).reshape(nt * bn).contiguous()
        colsum = wp.float().sum(1).contiguous()
        out = torch.full((M, inner), float("nan"), device=DEV, dtype=torch.bfloat16)
        sched = K.build_schedule([K.Segment(0, M, inner, C // 64)], bn, DEV, geglu=True)
        K.grouped_gemm(x, wp, out, sched, a_ld=C, a_k=C, a_rows=M, out_ld=inner, bias=bp, flags=EPI_GEGLU,
                       ln_colsum=colsum, ln_rowstats=rs)
        K.check_abort()
        hg = ln @ w.t() + b
        _close(out, hg[:, :inner] * F.gelu(hg[:, inner:]), 5e-2, 3e-2, "ln-fold geglu")


def check_conv_colstat_bf16(B=2, H=32, W=32, Cin=320, Cout=288, bn=160, seed=0):
    """APTP_EPI_GN_STATS on a bf16 conv output (ResNet conv1 -> norm2): the partial planes hold the column sums of the
    STORED (bf16-rounded) values; halo-tile boxes (8 x 16), ragged last column tile."""
    hw, M = H * W, B * H * W
    x = _rand(B, Cin, H, W, seed=seed).bfloat16()
    a = x.permute(0, 2, 3, 1).reshape(M, Cin).contiguous()
    w = _rand(Cout, Cin, 3, 3, scale=(9 * Cin) ** -0.5, seed=seed + 1).bfloat16()
    wp = w.permute(0, 2, 3, 1).reshape(Cout, 9 * Cin).contiguous()
    b = _rand(Cout, seed=seed + 2)
    out = torch.full((M, Cout), float("nan"), device=DEV, dtype=torch.bfloat16)
    cs = (torch.full((M // 32, Cout), float("nan"), device=DEV), torch.full((M // 32, Cout), float("nan"), device=DEV))
    sched = K.build_schedule([K.Segment(0, M, Cout, Cin // 64)], bn, DEV, mode=A_CONV3X3, Ho=H, Wo=W)
    K.grouped_gemm(a, wp, out, sched, a_ld=Cin, a_k=Cin, a_rows=M, mode=A_CONV3X3, batch=B, H=H, W=W, k_tap_pitch=Cin,
                   out_ld=Cout, bias=b, rows_per_sample=hw, colstat=cs)
    K.check_abort()
    ref = _conv_ref(x.float(), w.float(), b, 1).permute(0, 2, 3, 1).reshape(M, Cout)
    _close(out, ref, 2e-2, 1e-2, "conv3x3 bf16 with column statistics")
    o3 = out.float().reshape(B, hw, Cout)
    _close(cs[0].reshape(B, hw // 32, Cout).sum(1), o3.sum(1), 2e-3, 1e-4, "bf16 column sums")
    _close(cs[1].reshape(B, hw // 32, Cout).sum(1), (o3 * o3).sum(1), 2e-3, 1e-4, "bf16 column sums of squares")


def check_gemm_colstat(conv=False, seed=0):
    """APTP_EPI_GN_STATS: per-channel (sum, sumsq) partials of the fp32 output gathered in the GEMM epilogue, then reduced
    per (sample, group) by aptp_groupnorm_stats_from_partials -- vs torch on the stored output (two-source cat case too)."""
    B, H, W, Cin, Cout, bn = 3, 16, 16, 128, 320, 160
    hw, M = H * W, 3 * 16 * 16
    x = _rand(B, Cin, H, W, seed=seed).bfloat16()
    a = x.permute(0, 2, 3, 1).reshape(M, Cin).contiguous()
    res = _rand(M, Cout, seed=seed + 3) + 0.3
    out = res.clone()
    cs = (torch.full((B * hw // 32, Cout), float("nan"), device=DEV), torch.full((B * hw // 32, Cout), float("nan"), device=DEV))
    b = _rand(Cout, seed=seed + 2)
    if conv:
        w = _rand(Cout, Cin, 3, 3, scale=(9 * Cin) ** -0.5, seed=seed + 1).bfloat16()
        wp = w.permute(0, 2, 3, 1).reshape(Cout, 9 * Cin).contiguous()
        sched = K.build_schedule([K.Segment(0, M, Cout, Cin // 64)], bn, DEV, mode=A_CONV3X3, Ho=H, Wo=W)
        K.grouped_gemm(a, wp, out, sched, a_ld=Cin, a_k=Cin, a_rows=M, mode=A_CONV3X3, batch=B, H=H, W=W, k_tap_pitch=Cin,
                       out_ld=Cout, out_mode=OUT_F32, bias=b, residual=out, res_ld=Cout, flags=EPI_RES_F32,
                       rows_per_sample=hw, colstat=cs)
    else:
        w = _rand(Cout, Cin, scale=Cin ** -0.5, seed=seed + 1).bfloat16()
        # two expert buckets with different kept widths are not needed here: the planes are per output column
        sched = K.build_schedule([K.Segment(0, 2 * hw, Cout, Cin // 64), K.Segment(2 * hw, M, Cout, Cin // 64)], bn, DEV)
        K.grouped_gemm(a, w, out, sched, a_ld=Cin, a_k=Cin, a_rows=M, out_ld=Cout, out_mode=OUT_F32, bias=b, residual=out,
                       res_ld=Cout, flags=EPI_RES_F32, rows_per_sample=hw, colstat=cs)
    K.check_abort()
    o3 = out.reshape(B, hw, Cout)
    _close(cs[0].reshape(B, hw // 32, Cout).sum(1), o3.sum(1), 2e-3, 1e-5, "column sums")
    _close(cs[1].reshape(B, hw // 32, Cout).sum(1), (o3 * o3).sum(1), 2e-3, 1e-5, "column sums of squares")
    # consumer side: one source, then [out | skip] as an up-block cat with groups straddling the boundary
    groups = 32
    stats = torch.full((B, groups, 2), float("nan"), device=DEV)
    K.groupnorm_stats_from_partials(cs, Cout, None, 0, hw // 32, B, Cout // groups, None, stats, groups)
    ref = torch.stack([o3.reshape(B, hw, groups, -1).sum((1, 3)), (o3 * o3).reshape(B, hw, groups, -1).sum((1, 3))], -1)
    _close(stats, ref, 1e-2, 1e-5, "group statistics from partials")
    skip = _rand(M, 160, seed=seed + 9)
    s3 = skip.reshape(B, hw, 160)
    cs1 = (s3.reshape(B, hw // 32, 32, 160).sum(2).reshape(-1, 160).contiguous(),
           (s3 * s3).reshape(B, hw // 32, 32, 160).sum(2).reshape(-1, 160).contiguous())
    gs = (Cout + 160) // groups   # 15: groups straddle the 320 | 160 boundary
    ch = torch.tensor([Cout + 160, 0, Cout + 160], device=DEV, dtype=torch.int32)
    stats2 = torch.full((B, groups, 2), -7.0, device=DEV)
    K.groupnorm_stats_from_partials(cs, Cout, cs1, 160, hw // 32, B, gs, ch, stats2, groups)
    cat = torch.cat([o3, s3], 2)
    ref2 = torch.stack([cat.reshape(B, hw, groups, gs).sum((1, 3)), (cat * cat).reshape(B, hw, groups, gs).sum((1, 3))], -1)
    _close(stats2[0], ref2[0], 1e-2, 1e-5, "two-source group statistics")
    _close(stats2[2], ref2[2], 1e-2, 1e-5, "two-source group statistics")
    assert (stats2[1] == -7.0).all(), "samples with zero channels are skipped"


def check_conv_grouped(H=32, W=32, Cin=320, N=320, bn=160, samples=(2, 1, 3), n_valid=(320, 250, 130),
                       k_valid=(320, 192, 64), active=(True, False, True), seed=0):
    """3x3 conv over three expert buckets (whole samples each) with different kept Cin / Cout, one depth-dropped, in
    one launch: 32 x 32 images take the 2-SM halo scheme (8 x 16 boxes), 4 x 4 images 4 x 4 x 8 boxes whose batch
    extent runs past the bucket (and the batch)."""
    B = sum(samples)
    hw = H * W
    x = torch.zeros(B, H, W, Cin, device=DEV, dtype=torch.bfloat16)
    wp = torch.zeros(3 * N, 9 * Cin, device=DEV, dtype=torch.bfloat16)
    bias = torch.zeros(3 * N, device=DEV)
    out = torch.full((B * hw, N), 7.0, device=DEV, dtype=torch.bfloat16)
    segs, refs, b0 = [], [], 0
    for e in range(3):
        nb, kv, nv = samples[e], k_valid[e], n_valid[e]
        xe = _rand(nb, kv, H, W, seed=seed + 10 * e).bfloat16()
        we = _rand(nv, kv, 3, 3, scale=(9 * kv) ** -0.5, seed=seed + 10 * e + 1).bfloat16()
        be = _rand(nv, seed=seed + 10 * e + 2)
        x[b0:b0 + nb, :, :, :kv] = xe.permute(0, 2, 3, 1)
        wp[e * N:e * N + nv].view(nv, 9, Cin)[:, :, :kv] = we.permute(0, 2, 3, 1).reshape(nv, 9, kv)
        bias[e * N:e * N + nv] = be
        ns = min((nv + 63) // 64 * 64, N)
        segs.append(K.Segment(b0 * hw, (b0 + nb) * hw, nv, (kv + 63) // 64, w_row_off=e * N, vec_off=e * N, n_store=ns,
                              active=active[e]))
        refs.append((b0 * hw, nb * hw, nv, ns, _conv_ref(xe.float(), we.float(), be, 1)))
        b0 += nb
    sched = K.build_schedule(segs, bn, DEV, mode=A_CONV3X3, Ho=H, Wo=W)
    K.grouped_gemm(x.reshape(B * hw, Cin), wp, out, sched, a_ld=Cin, a_k=Cin, a_rows=B * hw, mode=A_CONV3X3, batch=B,
                   H=H, W=W, k_tap_pitch=Cin, out_ld=N, bias=bias, rows_per_sample=hw)
    K.check_abort()
    for e, (r0, rows, nv, ns, ref) in enumerate(refs):
        blk = out[r0:r0 + rows].float()
        if not active[e]:
            assert (blk == 7.0).all(), f"conv bucket {e}: inactive bucket must not be written"
            continue
        _close(blk[:, :nv], ref.permute(0, 2, 3, 1).reshape(rows, nv), 2e-2, 1e-2, f"conv bucket {e} box {sched.box}")
        assert (blk[:, nv:ns] == 0).all(), f"conv bucket {e}: padding columns must be zero"
        assert (blk[:, ns:] == 7.0).all(), f"conv bucket {e}: columns past n_store must be untouched"


def check_attention(B=2, heads=3, kept=(3, 1), Nq=256, Nkv=256, seed=0):
    C = heads * 64
    q = _rand(B * Nq, C, seed=seed).bfloat16()
    k = _rand(B * Nkv, C, seed=seed + 1).bfloat16()
    v = _rand(B * Nkv, C, seed=seed + 2).bfloat16()
    out = torch.full((B * Nq, C), 9.0, device=DEV, dtype=torch.bfloat16)
    sh = torch.tensor(list(kept), device=DEV, dtype=torch.int32)
    K.attention(q, C, k, C, v, C, out, C, B, Nq, Nkv, sh, heads, 0.125)
    K.check_abort()
    qf = q.float().reshape(B, Nq, heads, 64).transpose(1, 2)
    kf = k.float().reshape(B, Nkv, heads, 64).transpose(1, 2)
    vf = v.float().reshape(B, Nkv, heads, 64).transpose(1, 2)
    ref = _sdpa_ref(qf, kf, vf, 0.125).transpose(1, 2).reshape(B, Nq, heads, 64)
    got = out.reshape(B, Nq, heads, 64).float()
    for b in range(B):
        _close(got[b, :, :kept[b]], ref[b, :, :kept[b]], 2e-2, 2e-2, f"attention sample {b} Nq{Nq} Nkv{Nkv}")
        assert (got[b, :, kept[b]:] == 9.0).all(), "pruned heads must not be written"


def check_attention_rescale(B=2, heads=2, Nq=256, Nkv=640, seed=3):
    """Scores whose row maximum keeps growing from key tile to key tile (and jumps by far more than the 2^8
    lazy-rescale window), plus a ragged last key tile: exercises the optimistic-exponential redo path and the
    polynomial exp2 clamp of the softmax."""
    C = heads * 64
    q = (_rand(B * Nq, C, seed=seed) * 3.0).bfloat16()
    k = _rand(B * Nkv, C, seed=seed + 1)
    ramp = torch.linspace(0.2, 6.0, Nkv, device=DEV).repeat(B).unsqueeze(1)   # later keys score (much) higher
    k = (k * ramp).bfloat16()
    v = _rand(B * Nkv, C, seed=seed + 2).bfloat16()
    out = torch.zeros(B * Nq, C, device=DEV, dtype=torch.bfloat16)
    sh = torch.full((B,), heads, device=DEV, dtype=torch.int32)
    K.attention(q, C, k, C, v, C, out, C, B, Nq, Nkv, sh, heads, 0.125)
    K.check_abort()
    qf = q.float().reshape(B, Nq, heads, 64).transpose(1, 2)
    kf = k.float().reshape(B, Nkv, heads, 64).transpose(1, 2)
    vf = v.float().reshape(B, Nkv, heads, 64).transpose(1, 2)
    ref = _sdpa_ref(qf, kf, vf, 0.125).transpose(1, 2).reshape(B, Nq, heads, 64)
    got = out.reshape(B, Nq, heads, 64).float()
    assert torch.isfinite(got).all(), "attention produced non-finite values"
    _close(got, ref, 3e-2, 3e-2, f"attention rescale Nq{Nq} Nkv{Nkv}")


ALL = [
    ("gemm_linear_small", lambda: check_gemm_linear()),
    ("gemm_linear_bn256", lambda: check_gemm_linear(M=4096, Kd=1280, N=1280, bn=256)),
    ("gemm_linear_bn64_silu", lambda: check_gemm_linear(M=64, Kd=320, N=1280, bn=64, residual=False, silu=True)),
    ("gemm_linear_bn128_k1024", lambda: check_gemm_linear(M=154, Kd=1024, N=640, bn=128, bias=False, residual=False)),
    ("gemm_grouped", check_gemm_grouped),
    ("conv3x3_16", lambda: check_conv3x3()),
    ("conv3x3_64", lambda: check_conv3x3(B=2, H=64, W=64, Cin=64, Cout=64, bn=64)),
    ("conv3x3_8_border", lambda: check_conv3x3(B=5, H=8, W=8, Cin=192, Cout=160, bn=160, border=True)),
    ("conv3x3_32", lambda: check_conv3x3(B=1, H=32, W=32, Cin=320, Cout=320, bn=160)),
    ("conv3x3_fused_shortcut", check_conv3x3_fused_shortcut),
    ("conv3x3_fused_shortcut_ragged", lambda: check_conv3x3_fused_shortcut(B=1, H=16, W=16, Cin=640, Cout=608, C2=1920, bn=224)),
    ("conv3x3_s2_16", lambda: check_conv3x3(stride=2, temb=False)),
    ("conv3x3_s2_64", lambda: check_conv3x3(B=2, H=64, W=64, Cin=64, Cout=64, bn=64, stride=2, temb=False)),
    ("geglu", check_geglu),
    ("geglu_gate", check_geglu_gate),
    ("gemm_epilogue_mix", check_gemm_epilogue_mix),
    ("conv_residual", check_conv_residual),
    ("conv_residual_8", lambda: check_conv_residual(B=5, H=8, W=8, Cin=192, Cout=320, bn=160)),
    ("out_modes", check_out_modes),
    ("groupnorm", lambda: check_groupnorm()),
    ("groupnorm_two_src", lambda: check_groupnorm(C0=640, C1=320, silu=False)),
    ("groupnorm_wide", lambda: check_groupnorm(B=2, HW=64, C0=1280, C1=1280)),
    ("groupnorm_gate_compact", lambda: check_groupnorm(gate=True, compact=True)),
    ("groupnorm_tiny_groups", lambda: check_groupnorm(C0=64, HW=64)),
    ("groupnorm_f32", lambda: check_groupnorm(f32=True)),
    ("groupnorm_f32_two_src", lambda: check_groupnorm(C0=640, C1=320, silu=False, f32=True)),
    ("groupnorm_f32_wide", lambda: check_groupnorm(B=2, HW=64, C0=1280, C1=1280, f32=True)),
    ("groupnorm_f32_compact", lambda: check_groupnorm(compact=True, f32=True, HW=4096)),
    ("groupnorm_big", lambda: check_groupnorm(B=8, HW=4096, C0=320)),
    ("stream_f32", check_stream_f32),
    ("gemm_res_f32", check_gemm_res_f32),
    ("gemm_colstat", check_gemm_colstat),
    ("conv_colstat", lambda: check_gemm_colstat(conv=True)),
    ("conv_colstat_bf16", check_conv_colstat_bf16),
    ("conv_colstat_bf16_8x8box", lambda: check_conv_colstat_bf16(B=3, H=16, W=8, Cin=128, Cout=160, bn=160)),
    ("gemm_ln_fold", check_gemm_ln_fold),
    ("gemm_ln_fold_geglu", lambda: check_gemm_ln_fold(geglu=True)),
    ("conv_res_f32", lambda: check_gemm_res_f32(conv=True)),
    ("layernorm", lambda: check_layernorm()),
    ("layernorm_1280", lambda: check_layernorm(rows=77, C=1280)),
    ("elementwise", check_elementwise),
    # 2-SM scheme (taps * K >= 1280) with the features the full-width U-Net combines with it
    ("geglu_2sm_k1280", lambda: check_geglu(M=600, Kd=1280, inner=1280, n_keep=1000)),
    ("gemm_ln_fold_2sm", lambda: check_gemm_ln_fold(C=1280)),
    ("gemm_ln_fold_geglu_2sm", lambda: check_gemm_ln_fold(geglu=True, C=1280)),
    ("gemm_grouped_2sm_unaligned", lambda: check_gemm_grouped(HW=200, C=1280, N=640, samples=(3, 2, 1),
                                                               n_valid=(600, 640, 330), k_valid=(1280, 704, 1000),
                                                               active=(True, False, True))),
    ("conv3x3_s2_2sm_cin320", lambda: check_conv3x3(B=3, H=32, W=32, Cin=320, Cout=320, bn=160, stride=2, temb=False)),
    ("conv_grouped_halo", lambda: check_conv_grouped()),
    ("conv_grouped_4x4x8", lambda: check_conv_grouped(H=4, W=4, Cin=640, N=640, bn=224, samples=(5, 2, 6),
                                                       n_valid=(640, 600, 320), k_valid=(640, 448, 192))),
    ("attention_self", lambda: check_attention()),
    ("attention_rescale", lambda: check_attention_rescale()),
    ("attention_rescale_ragged", lambda: check_attention_rescale(Nq=384, Nkv=600, seed=5)),
    ("attention_cross77", lambda: check_attention(Nkv=77)),
    ("attention_small_q", lambda: check_attention(B=3, heads=2, kept=(2, 0, 1), Nq=64, Nkv=64)),
    ("attention_long", lambda: check_attention(B=1, heads=1, kept=(1,), Nq=1024, Nkv=1024)),
]
