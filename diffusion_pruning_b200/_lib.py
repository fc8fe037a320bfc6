"""ctypes binding of libaptp_sm100.so (C ABI: include/aptp_sm100.h).

There is deliberately no fallback: if the shared library is missing or a call fails, we raise.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

_PKG = Path(__file__).resolve().parent
LIB_PATH = _PKG / "libaptp_sm100.so"

c_void_p, c_int, c_int64, c_float = C.c_void_p, C.c_int32, C.c_int64, C.c_float


class GemmSeg(C.Structure):
    _fields_ = [(n, C.c_int32) for n in
                ("row_begin", "row_end", "n_valid", "n_store", "k_chunks", "w_row_off", "vec_off", "tab_off",
                 "out_col_off", "w2_row_off", "pad1", "pad2")]


class GemmTile(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("seg", "m_base", "n0", "flags")]


class GemmArgs(C.Structure):
    _fields_ = [
        ("a", c_void_p), ("a_mode", c_int), ("a_ld", c_int), ("a_k", c_int), ("a_rows", c_int64),
        ("batch", c_int), ("H", c_int), ("W", c_int),
        ("w", c_void_p), ("w_rows", c_int64), ("w_ld", c_int), ("k_tap_pitch", c_int),
        ("out", c_void_p), ("out_ld", c_int), ("out_mode", c_int),
        ("bn", c_int), ("bw", c_int), ("bh", c_int), ("bb", c_int),
        ("bias", c_void_p), ("rowvec", c_void_p), ("rowvec_ld", c_int), ("rows_per_sample", c_int),
        ("residual", c_void_p), ("res_ld", c_int),
        ("gate", c_void_p), ("gate_ld", c_int), ("gate_group", c_int),
        ("border_tab", c_void_p), ("tab_ld", c_int),
        ("gn_stats", c_void_p), ("gn_ld", c_int), ("gn_blocks", c_int),
        ("flags", c_int),
        ("segs", c_void_p), ("n_segs", c_int), ("tiles", c_void_p), ("n_tiles", c_int),
        ("ln_colsum", c_void_p), ("ln_rowstats", c_void_p), ("ln_reserved0", c_int), ("ln_reserved1", c_int),
        ("ln_reserved2", c_float),
        ("rowstat_out", c_void_p), ("rowstat_chunks", c_int),
        ("gn_stats_sq", c_void_p), ("a_stat_chunks", c_int), ("a_stat_pairs", c_int),
        ("a2", c_void_p), ("a2_ld", c_int), ("a2_k", c_int), ("w2", c_void_p), ("w2_rows", c_int64), ("w2_ld", c_int),
    ]


A_LINEAR, A_CONV3X3, A_CONV3X3_S2 = 0, 1, 2
OUT_BF16, OUT_F32, OUT_F32_NCHW = 0, 1, 2
EPI_GEGLU, EPI_SILU, EPI_GN_STATS, EPI_RES_F32, EPI_LN_FOLD = 1, 2, 4, 8, 16

# name -> (restype, argtypes); must list every symbol declared in include/aptp_sm100.h
SIGNATURES = {
    "aptp_version": (c_int, []),
    "aptp_last_error": (C.c_char_p, []),
    "aptp_check_abort": (c_int, [c_void_p]),
    "aptp_poll_abort": (c_int, [c_void_p]),
    "aptp_grouped_gemm_fwd": (c_int, [C.POINTER(GemmArgs), c_void_p]),
    "aptp_gemm_max_pairs": (c_int, []),
    "aptp_groupnorm_stats_workspace": (c_int64, [c_int, c_int, c_int]),
    "aptp_groupnorm_stats": (c_int, [c_void_p, c_int, c_int, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int,
                                     c_void_p, c_void_p, c_int, c_void_p, c_int64, c_void_p]),
    "aptp_groupnorm_stats_from_partials": (c_int, [c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p, c_int, c_int,
                                                   c_int, c_int, c_int, c_void_p, c_void_p, c_int, c_void_p]),
    "aptp_groupnorm_apply": (c_int, [c_void_p, c_int, c_int, c_void_p, c_int, c_int, c_int, c_void_p, c_int, c_int,
                                     c_int, c_int, c_float, c_void_p, c_int, c_void_p, c_void_p, c_int, c_void_p,
                                     c_void_p, c_void_p, c_int, c_int, c_void_p]),
    "aptp_groupnorm_apply_raw": (c_int, [c_void_p, c_int, c_int, c_void_p, c_int, c_int, c_int, c_void_p, c_int, c_int,
                                         c_int, c_int, c_float, c_void_p, c_int, c_void_p, c_void_p, c_int, c_void_p,
                                         c_void_p, c_void_p, c_int, c_int, c_void_p, c_int, c_void_p]),
    "aptp_copy_rows_cvt": (c_int, [c_void_p, c_int, c_int, c_void_p, c_int, c_int, c_int64, c_int, c_void_p, c_int,
                                   c_void_p]),
    "aptp_depth_lerp_f32": (c_int, [c_void_p, c_int, c_void_p, c_int, c_void_p, c_int, c_int64, c_int, c_void_p, c_int,
                                    c_void_p]),
    "aptp_upsample2x_cvt": (c_int, [c_void_p, c_int, c_void_p, c_int, c_int, c_int, c_int, c_void_p]),
    "aptp_ln_rowstats": (c_int, [c_void_p, c_int, c_int64, c_int, c_float, c_void_p, c_void_p, c_int, c_void_p]),
    "aptp_layernorm": (c_int, [c_void_p, c_int, c_void_p, c_int, c_int64, c_int, c_float, c_void_p, c_void_p,
                               c_void_p, c_int, c_void_p]),
    "aptp_depth_lerp": (c_int, [c_void_p, c_int, c_void_p, c_int, c_void_p, c_int, c_int64, c_int, c_void_p, c_int,
                                c_void_p]),
    "aptp_copy_rows": (c_int, [c_void_p, c_int, c_void_p, c_int, c_int64, c_int, c_void_p, c_int, c_void_p]),
    "aptp_upsample2x": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p]),
    "aptp_im2col_input": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p]),
    "aptp_timestep_embedding": (c_int, [c_void_p, c_void_p, c_int, c_int, c_void_p]),
    "aptp_cast_f32_bf16": (c_int, [c_void_p, c_void_p, c_int64, c_void_p]),
    "aptp_silu_bf16": (c_int, [c_void_p, c_void_p, c_int64, c_void_p]),
    "aptp_cfg_ddim_step": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_float, c_float, c_float, c_int, c_void_p]),
    "aptp_attention_fwd": (c_int, [c_void_p, c_int, c_void_p, c_int, c_void_p, c_int, c_void_p, c_int, c_int, c_int,
                                   c_int, c_void_p, c_int, c_float, c_void_p, c_void_p]),
    "aptp_attention_bwd": (c_int, [c_void_p, c_int, c_void_p, c_int, c_void_p, c_int, c_void_p, c_int, c_void_p, c_int,
                                   c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_int, c_void_p, c_int, c_int, c_int,
                                   c_int, c_void_p, c_int, c_float, c_void_p]),
    "aptp_gumbel_gate_fwd": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_int, c_void_p,
                                     c_float, c_float, c_int, c_void_p]),
    "aptp_gumbel_gate_bwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_float,
                                     c_float, c_void_p]),
    "aptp_arch_normalize": (c_int, [c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p, c_int, c_void_p]),
    "aptp_arch_normalize_bwd": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "aptp_route_cosine": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p]),
    "aptp_sinkhorn_phase": (c_int, [c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_float,
                                    c_int, c_void_p]),
    "aptp_scale_cols_fwd": (c_int, [c_void_p, c_int, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_int, c_int,
                                    c_void_p]),
    "aptp_scale_cols_bwd": (c_int, [c_void_p, c_int, c_void_p, c_int, c_void_p, c_int, c_int, c_int, c_int, c_void_p,
                                    c_int, c_int, c_void_p, c_void_p]),
    "aptp_geglu_fwd": (c_int, [c_void_p, c_int, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_int, c_int, c_void_p]),
    "aptp_geglu_bwd": (c_int, [c_void_p, c_int, c_void_p, c_int, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_int,
                               c_int, c_void_p, c_void_p]),
    "aptp_groupnorm_bwd": (c_int, [c_void_p, c_int, c_void_p, c_int, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int,
                                   c_float, c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p,
                                   c_void_p, c_void_p]),
    "aptp_layernorm_bwd": (c_int, [c_void_p, c_int, c_void_p, c_int, c_void_p, c_int, c_int, c_int64, c_int, c_float,
                                   c_void_p, c_void_p]),
    "aptp_depth_lerp_bwd": (c_int, [c_void_p, c_int, c_void_p, c_int, c_void_p, c_int, c_void_p, c_int, c_void_p, c_int,
                                    c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "aptp_add_rows": (c_int, [c_void_p, c_int, c_void_p, c_int, c_int64, c_int, c_void_p]),
    "aptp_upsample2x_bwd": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p]),
    "aptp_zero_insert2x": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p]),
    "aptp_route_sinkhorn": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_float, c_int, c_void_p]),
    "aptp_add_noise_velocity": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int,
                                        c_int, c_int, c_void_p]),
    "aptp_mse_rows_fwd": (c_int, [c_void_p, c_int, c_void_p, c_int, c_int64, c_int, c_void_p, c_int, c_void_p]),
    "aptp_mse_rows_bwd": (c_int, [c_void_p, c_int, c_void_p, c_int, c_void_p, c_int, c_int64, c_int, c_void_p, c_float,
                                  c_void_p]),
    "aptp_pred_losses_fwd": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p]),
    "aptp_macs_ratio_fwd": (c_int, [c_void_p, c_int, c_int, c_void_p, c_int, c_void_p, c_int, C.c_double, c_void_p,
                                    c_void_p, c_void_p]),
    "aptp_macs_ratio_bwd": (c_int, [c_void_p, c_int, c_int, c_void_p, c_int, c_void_p, c_int, c_void_p, c_void_p, c_int,
                                    c_int, c_void_p]),
    "aptp_groupnorm_bwd_affine": (c_int, [c_void_p, c_int, c_void_p, c_int, c_void_p, c_int, c_int, c_int, c_int, c_int,
                                          c_int, c_float, c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_int, c_int,
                                          c_void_p, c_void_p, c_void_p, c_void_p]),
    "aptp_layernorm_affine_bwd": (c_int, [c_void_p, c_int, c_void_p, c_int, c_int64, c_int, c_float, c_void_p, c_void_p]),
    "aptp_col_sum_groups": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_int, c_void_p]),
    "aptp_wgrad": (c_int, [c_void_p, c_int, c_void_p, c_int, c_void_p, c_int64, c_void_p, c_int64, c_int, c_int, c_int,
                           c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "aptp_linear_f32_fwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p]),
    "aptp_linear_f32_bwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int,
                                    c_void_p]),
    "aptp_contrastive_fwd": (c_int, [c_void_p, c_int, c_void_p, c_int, c_int, c_float, c_float, c_void_p, c_void_p,
                                     c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "aptp_contrastive_bwd": (c_int, [c_void_p, c_int, c_int, c_float, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                     c_void_p, c_void_p, c_void_p]),
    "aptp_pred_losses_bwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int,
                                     c_void_p]),
}

_lib = None


class AptpError(RuntimeError):
    pass


def load() -> C.CDLL:
    """Load the CUDA extension; raise loudly if it is not built (no CPU / eager fallback exists)."""
    global _lib
    if _lib is not None:
        return _lib
    path = Path(os.environ.get("APTP_LIB") or LIB_PATH)  # APTP_LIB: kernel-tuning builds of the same library (tools/)
    if not path.exists():
        raise AptpError(
            f"{path} is missing: build it with `python -m diffusion_pruning_b200.build` "
            "(the product path has no fallback implementation)")
    lib = C.CDLL(os.fspath(path))
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the .so does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        msg = load().aptp_last_error().decode("utf-8", "replace")
        raise AptpError(f"{what or 'libaptp_sm100'} failed (status {rc}): {msg}")
