"""ctypes binding of `libaptai_b200.so` (the C ABI declared in include/aptai_b200.h).

There is deliberately no fallback of any kind: if the shared library is missing, or a compute entry point is
called on a device that is not sm_100, a RuntimeError is raised.
"""
from __future__ import annotations

import ctypes as C
from pathlib import Path

_PKG = Path(__file__).resolve().parent
import os as _os

# APTAI_LIB_ALT: another build of the same library (same-box A/B of a kernel change against the previous build;
# profiling only — the product library is the one next to this file)
LIB_PATH = Path(_os.environ["APTAI_LIB_ALT"]).resolve() if _os.environ.get("APTAI_LIB_ALT") else _PKG / "libaptai_b200.so"

c_void_p, c_int, c_i64, c_float, c_size_t = C.c_void_p, C.c_int, C.c_int64, C.c_float, C.c_size_t


class GemmArgs(C.Structure):
    """struct aptai_gemm_args (include/aptai_b200.h)."""
    _fields_ = [
        ("a", c_void_p), ("a_row_stride", c_i64), ("a_seg_stride", c_i64),
        ("a_rows", C.c_int32), ("a_cols", C.c_int32), ("P", C.c_int32), ("taps", C.c_int32),
        ("kb_per_tap", C.c_int32), ("a_col_per_nblk", C.c_int32),
        ("w", c_void_p), ("N", C.c_int32), ("block_n", C.c_int32), ("segs", C.c_int32), ("rows_per_seg", C.c_int32),
        ("bias", c_void_p), ("gamma", c_void_p), ("beta", c_void_p), ("residual", c_void_p),
        ("out_f32", c_void_p), ("out_bf16", c_void_p), ("ldo", c_i64), ("out_seg_stride", c_i64),
        ("seg_valid_rows", c_void_p), ("mask_seg_rows", C.c_int32), ("act", C.c_int32), ("ln", C.c_int32), ("ln_eps", c_float), ("cta_pair", C.c_int32), ("half_fmt", C.c_int32),
        ("aux", c_void_p), ("out_pre", c_void_p),
    ]


class PrepEntry(C.Structure):
    """struct aptai_prep_entry (include/aptai_b200.h), 64 bytes."""
    _fields_ = [("src", c_void_p), ("dst", c_void_p), ("dst_t", c_void_p), ("dst_f32", c_void_p),
                ("rows", C.c_int32), ("cols", C.c_int32), ("dst_ld", C.c_int32), ("dst_t_ld", C.c_int32),
                ("scale", c_float), ("scale_t", c_float), ("tile0", C.c_int32), ("tiles_x", C.c_int32)]


# name -> (restype, argtypes); every symbol include/aptai_b200.h declares
PROTOTYPES = {
    "aptai_version": (c_int, []),
    "aptai_last_error_string": (C.c_char_p, []),
    "aptai_launch_count": (c_i64, []),
    "aptai_gemm_bf16": (c_int, [C.POINTER(GemmArgs), c_void_p]),
    "aptai_set_traversal": (None, [c_int]),
    "aptai_conv0_workspace_bytes": (c_size_t, [c_int, c_int]),
    "aptai_conv0_norm_gelu": (c_int, [c_void_p, c_int, c_i64, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_float,
                                      c_void_p, c_int, c_void_p, c_int, c_void_p]),
    "aptai_layernorm": (c_int, [c_void_p, c_int, c_i64, c_int, c_void_p, c_void_p, c_float, c_void_p, c_void_p,
                                c_int, c_void_p]),
    "aptai_cast_pad_bf16": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    "aptai_cast_pad_h16": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_int, c_void_p]),
    "aptai_posconv_fold": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "aptai_posconv_fold_fmt": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_int,
                                       c_void_p]),
    "aptai_attention_fwd_fmt": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p]),
    "aptai_attention_fwd": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p]),
    "aptai_attention_fwd_v3": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p]),
    "aptai_heads": (c_int, [c_void_p, c_i64, c_int, c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p,
                            c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "aptai_pr_head_wide_workspace_bytes": (c_size_t, [c_i64, c_int, c_int, c_int]),
    "aptai_pr_head_wide": (c_int, [c_void_p, c_i64, c_int, c_void_p, c_void_p, c_int, c_void_p, c_i64, c_void_p,
                                   c_size_t, c_void_p]),
    "aptai_logits_rows": (c_int, [c_void_p, c_i64, c_int, c_i64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "aptai_pr_head_wide_bwd": (c_int, [c_void_p, c_i64, c_int, c_void_p, c_int, c_void_p, c_i64, c_void_p, c_void_p,
                                       c_void_p, c_void_p, c_size_t, c_void_p]),
    "aptai_lowpass_fir": (c_int, [c_void_p, c_int, c_int, c_int, c_void_p, c_int, c_void_p, c_void_p]),
    "aptai_softmax_rows": (c_int, [c_void_p, c_i64, c_int, c_int, c_void_p, c_void_p]),
    "aptai_tail": (c_int, [c_void_p, c_i64, c_int, c_void_p, c_void_p, c_float, c_void_p, c_void_p, c_int, c_int, c_void_p,
                           c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "aptai_posconv_slab": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p]),
    "aptai_posconv_slab_fmt": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p]),
    "aptai_frame_lengths": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p]),
    "aptai_cross_attention": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p,
                                      c_void_p, c_void_p, c_void_p, c_float, c_int, c_int, c_void_p, c_void_p,
                                      c_void_p, c_void_p]),
    "aptai_masked_mse_ce": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_i64, c_int, c_int, c_void_p, c_void_p,
                                    c_void_p]),
    "aptai_ctc_workspace_bytes": (c_size_t, [c_int, c_int, c_int]),
    "aptai_logsoftmax_ctc": (c_int, [c_void_p, c_int, c_int, c_int, c_void_p, c_int, c_void_p, c_void_p, c_int, c_int,
                                     c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "aptai_logsoftmax_ctc_ex": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_float, c_void_p, c_void_p, c_int,
                                        c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p,
                                        c_void_p, c_void_p, c_size_t, c_void_p]),
    "aptai_viterbi_workspace_bytes": (c_size_t, [c_int, c_int, c_int]),
    "aptai_ctc_viterbi_f32": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int,
                                      c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "aptai_ctc_greedy": (c_int, [c_void_p, c_int, c_int, c_int, c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_int,
                                 c_void_p]),
    "aptai_ctc_decode_ref": (c_int, [c_void_p, c_int, c_int, c_int, c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p,
                                     c_int, c_void_p]),
    "aptai_split3_bf16": (c_int, [c_void_p, c_i64, c_int, c_i64, c_int, c_float, c_void_p, c_void_p]),
    "aptai_rowop_split3": (c_int, [c_void_p, c_i64, c_int, c_void_p, c_void_p, c_float, c_int, c_int, c_void_p,
                                   c_void_p, c_void_p]),
    "aptai_conv0_accurate": (c_int, [c_void_p, c_int, c_i64, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_float,
                                     c_void_p, c_int, c_void_p, c_void_p]),
    "aptai_gelu_add_f32": (c_int, [c_void_p, c_void_p, c_i64, c_void_p, c_void_p]),
    "aptai_cast_pad_split": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "aptai_posconv_fold_split": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p,
                                         c_void_p]),
    "aptai_attention_fwd_f32": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p]),
    "aptai_cross_attention_bwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                          c_float, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                          c_void_p, c_void_p]),
    "aptai_bilstm_256": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p]),
    "aptai_bilstm_256_train": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p,
                                       c_void_p, c_void_p]),
    "aptai_bilstm_256_bwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int,
                                     c_void_p, c_void_p]),
    # ---- training step
    "aptai_attention_fwd_lse": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p]),
    "aptai_attention_bwd_dot": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p]),
    "aptai_attention_bwd_dot_zero": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "aptai_attention_bwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p,
                                    c_void_p, c_void_p]),
    "aptai_attention_fwd_dropout": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_float,
                                            C.c_uint64, c_void_p]),
    "aptai_attention_bwd_dropout": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int,
                                            c_void_p, c_void_p, c_float, C.c_uint64, c_void_p]),
    "aptai_attention_dropout_mask": (c_int, [c_int, c_int, c_int, c_float, C.c_uint64, c_void_p, c_void_p]),
    "aptai_scale_cast_bf16": (c_int, [c_void_p, c_i64, c_int, c_float, c_void_p, c_i64, c_void_p]),
    "aptai_gemm_wgrad_bf16": (c_int, [c_void_p, c_i64, c_void_p, c_i64, c_i64, c_int, c_int, c_float, c_void_p, c_i64,
                                      c_void_p]),
    "aptai_posconv_wgrad_bf16": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    "aptai_conv_wgrad_bf16": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    "aptai_ln_gelu_fwd_512": (c_int, [c_void_p, c_i64, c_void_p, c_void_p, c_float, c_void_p, c_void_p]),
    "aptai_ln_gelu_bwd_512": (c_int, [c_void_p, c_i64, c_i64, c_void_p, c_void_p, c_i64, c_void_p, c_void_p, c_i64,
                                      c_void_p, c_void_p, c_float, c_void_p, c_void_p, c_void_p, c_void_p]),
    "aptai_gelu_bwd_rows_512": (c_int, [c_void_p, c_i64, c_i64, c_void_p, c_i64, c_void_p, c_void_p]),
    "aptai_conv0_groupnorm_bwd": (c_int, [c_void_p, c_i64, c_void_p, c_int, c_i64, c_int, c_void_p, c_void_p, c_void_p,
                                          c_void_p, c_void_p, c_void_p]),
    "aptai_conv0_im2col_bf16": (c_int, [c_void_p, c_int, c_i64, c_i64, c_void_p, c_void_p]),
    "aptai_posconv_weightnorm_bwd": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p,
                                             c_void_p, c_void_p, c_void_p]),
    "aptai_gelu_bwd": (c_int, [c_void_p, c_void_p, c_i64, c_void_p, c_void_p]),
    "aptai_colsum": (c_int, [c_void_p, c_int, c_i64, c_int, c_i64, c_float, c_void_p, c_void_p]),
    "aptai_layernorm_bwd": (c_int, [c_void_p, c_void_p, c_i64, c_int, c_void_p, c_float, c_void_p, c_void_p, c_void_p,
                                    c_void_p, c_void_p, c_void_p]),
    "aptai_layernorm_bwd_colsum": (c_int, [c_void_p, c_void_p, c_i64, c_int, c_void_p, c_float, c_void_p, c_void_p,
                                           c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "aptai_heads_bwd": (c_int, [c_void_p, c_i64, c_int, c_void_p, c_int, c_void_p, c_int, c_void_p, c_void_p,
                                c_void_p, c_int, c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p]),
    "aptai_masked_mse_ce_bwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_i64, c_int, c_int, c_void_p, c_void_p,
                                        c_void_p, c_void_p, c_void_p]),
    "aptai_dropout": (c_int, [c_void_p, c_int, c_void_p, c_i64, c_float, C.c_uint64, c_void_p, c_void_p, c_void_p]),
    "aptai_prepare_weights": (c_int, [c_void_p, c_int, c_int, c_void_p]),
    "aptai_prepare_weights_fmt": (c_int, [c_void_p, c_int, c_int, c_int, c_void_p]),
    "aptai_adam_step": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p,
                                c_float, c_float, c_float, c_float, c_float, c_int, c_float, c_void_p]),
    # ---- callers' data formats
    "aptai_collate_pad": (c_int, [c_void_p, c_int, c_void_p, c_int, c_i64, c_void_p, c_void_p, c_void_p]),
    "aptai_resample_fir": (c_int, [c_void_p, c_void_p, c_int, c_i64, c_void_p, c_int, c_int, c_int, c_void_p, c_i64,
                                   c_void_p]),
    "aptai_interp_linear_f64": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    "aptai_frames_to_segments": (c_int, [c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p,
                                         c_int, c_void_p]),
    "aptai_tv_metrics": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "aptai_boundary_stats": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, C.c_double, c_void_p,
                                     c_void_p]),
    "aptai_frame_overlap": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p]),
}

_lib = None


def load() -> C.CDLL:
    """Load the shared library (building is the job of `aptai_b200.build` / `__graft_entry__.build()`)."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise RuntimeError(
            f"{LIB_PATH} not found: the CUDA extension is not built. Run `python -m aptai_b200.build` "
            "(aptai_b200 has no CPU or PyTorch fallback).")
    lib = C.CDLL(str(LIB_PATH))
    for name, (res, args) in PROTOTYPES.items():
        fn = getattr(lib, name)   # AttributeError if a declared symbol is missing
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def last_error() -> str:
    return load().aptai_last_error_string().decode("utf-8", "replace")


def check(rc: int, what: str) -> None:
    if rc != 0:
        raise RuntimeError(f"aptai_b200.{what} failed (status {rc}): {last_error()}")


def launch_count() -> int:
    return int(load().aptai_launch_count())
