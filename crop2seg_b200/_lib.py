"""ctypes binding of the C ABI declared in ``include/crop2seg_b200.h``.

The library is the product: if it is missing or fails to load, every operator raises.  There is
no PyTorch / CPU fallback anywhere in this package.
"""
from __future__ import annotations

import ctypes
import os
import threading

from .build import LIB_PATH

C2S_ABI_VERSION = 12

# enum c2s_dtype / c2s_agg_mode / c2s_pe_mode / c2s_ltae_flags
F32, BF16 = 0, 1
AGG_ATT_GROUP, AGG_ATT_MEAN, AGG_MEAN = 0, 1, 2
PE_NONE, PE_SINUSOID, PE_SINUSOID_LINEAR, PE_DOY_TABLE = 0, 1, 2, 3
LTAE_ATTN_ONLY, LTAE_SKIP_ATTN_STORE, LTAE_ZERO_PADDED, LTAE_BN_BATCH_STATS, LTAE_REUSE_FOLDED = 1, 2, 4, 8, 16
# enum c2s_option / c2s_ltae_kernel (kernel-selection switches for parity tests and A/B measurements)
OPT_LTAE_KERNEL, OPT_AGG_KERNEL, OPT_AGG_TAPS, OPT_LTAE_BWD_KERNEL = 0, 1, 2, 3
LTAE_KERNEL_AUTO, LTAE_KERNEL_GENERAL, LTAE_KERNEL_SLAB, LTAE_KERNEL_TEAM = 0, 1, 2, 3

EXPORTS = (
    "c2s_abi_version", "c2s_last_error", "c2s_launch_count", "c2s_reset_launch_count", "c2s_last_kernel",
    "c2s_last_ltae_kernel", "c2s_set_option", "c2s_get_option",
    "c2s_agg_workspace_bytes", "c2s_agg_forward", "c2s_agg_backward_workspace_bytes", "c2s_agg_backward",
    "c2s_agg_skipconv_workspace_bytes", "c2s_agg_skipconv_forward", "c2s_agg_skipconv_backward_workspace_bytes",
    "c2s_agg_skipconv_backward", "c2s_agg_skipconv_bstats_workspace_bytes", "c2s_agg_skipconv_bstats_forward",
    "c2s_agg_skipconv_bstats_backward_workspace_bytes", "c2s_agg_skipconv_bstats_backward", "c2s_pad_mask",
    "c2s_ltae_workspace_bytes", "c2s_ltae_forward", "c2s_ltae_backward_workspace_bytes", "c2s_ltae_backward",
    "c2s_ltae_mlp_backward_workspace_bytes", "c2s_ltae_mlp_backward", "c2s_ltae_inconv_grad", "c2s_ltae_fold_backward",
    "c2s_ltae_rows_forward",
    "c2s_conv2d_supported", "c2s_conv2d_workspace_bytes", "c2s_conv2d_forward", "c2s_group_stats", "c2s_group_norm_relu",
    "c2s_tile_patchify", "c2s_tile_classmap", "c2s_frame_index", "c2s_frames_gather", "c2s_frames_scatter",
    "c2s_boundary_target", "c2s_seg_loss_workspace_bytes", "c2s_seg_loss_forward", "c2s_seg_loss_backward",
)
LOSS_CROSS_ENTROPY, LOSS_FOCAL = 0, 1  # enum c2s_loss_kind
RAW_I16, RAW_U16, RAW_F32 = 0, 1, 2  # enum c2s_raw_dtype


class AggDesc(ctypes.Structure):
    _fields_ = [(n, ctypes.c_int32) for n in ("B", "T", "C", "H", "W", "n_heads", "ha", "wa", "mode", "dtype")]


class SkipConvParams(ctypes.Structure):
    _fields_ = [(n, ctypes.c_void_p) for n in ("conv_weight", "conv_bias", "bn_weight", "bn_bias", "bn_running_mean",
                                               "bn_running_var")] + [("bn_eps", ctypes.c_float)]


SKIPCONV_BWD_IO_FIELDS = ("grad_x", "grad_attn", "grad_conv_weight", "grad_conv_bias", "grad_bn_weight", "grad_bn_bias")


class SkipConvBwdIo(ctypes.Structure):
    _fields_ = [(n, ctypes.c_void_p) for n in SKIPCONV_BWD_IO_FIELDS]


class TileDesc(ctypes.Structure):
    _fields_ = [(n, ctypes.c_int32) for n in ("T", "T_pad", "C", "H", "W", "patch", "grid_h", "grid_w", "patch_begin",
                                              "patch_count", "src_dtype", "dst_dtype")] + [("pad_value", ctypes.c_float)]


class LossDesc(ctypes.Structure):
    _fields_ = [(n, ctypes.c_int32) for n in ("B", "K", "H", "W", "dtype", "kind", "ignore_index", "size_average")] + \
               [("gamma", ctypes.c_float), ("label_smoothing", ctypes.c_float)]


class LtaeDesc(ctypes.Structure):
    _fields_ = [(n, ctypes.c_int32) for n in (
        "B", "T", "C", "H", "W", "n_head", "d_k", "d_model", "c_out", "has_inconv", "pe_mode", "pe_abs",
        "pos_dtype", "dtype", "flags")] + [(n, ctypes.c_float) for n in (
        "gn_eps", "bn_eps", "attn_keep_scale", "mlp_keep_scale")]


LTAE_PARAM_FIELDS = (
    "in_norm_weight", "in_norm_bias", "inconv_weight", "inconv_bias", "query", "key_weight", "key_bias",
    "mlp_weight", "mlp_bias", "bn_weight", "bn_bias", "bn_running_mean", "bn_running_var",
    "out_norm_weight", "out_norm_bias", "pe_denom", "pe_fc_weight", "pe_fc_bias", "pe_abs_fc_weight",
    "pe_abs_fc_bias",
)
LTAE_MASK_FIELDS = ("attn_keep", "mlp_keep")  # uint8 dropout keep masks (training only)


class LtaeParams(ctypes.Structure):
    _fields_ = [(n, ctypes.c_void_p) for n in LTAE_PARAM_FIELDS + LTAE_MASK_FIELDS + ("save_o", "save_y")]


LTAE_BWD_IO_FIELDS = ("grad_o", "grad_attn", "grad_x", "grad_u", "grad_cpos", "grad_gamma", "grad_beta", "zn_rows",
                      "sa_rows", "grad_pe")


class LtaeBwdIo(ctypes.Structure):
    _fields_ = [(n, ctypes.c_void_p) for n in LTAE_BWD_IO_FIELDS]


LTAE_MLP_BWD_IO_FIELDS = ("o_rows", "y_rows", "grad_out", "bn_mean", "bn_var", "grad_o", "grad_mlp_weight", "grad_mlp_bias",
                          "grad_bn_weight", "grad_bn_bias", "grad_out_norm_weight", "grad_out_norm_bias")


LTAE_FOLD_BWD_IO_FIELDS = ("grad_u", "grad_cpos", "grad_gamma_direct", "grad_beta_direct", "grad_in_norm_weight",
                           "grad_in_norm_bias", "grad_inconv_weight", "grad_inconv_bias", "grad_query", "grad_key_weight",
                           "grad_key_bias", "grad_pe")


class LtaeFoldBwdIo(ctypes.Structure):
    _fields_ = [(n, ctypes.c_void_p) for n in LTAE_FOLD_BWD_IO_FIELDS]


class LtaeMlpBwdIo(ctypes.Structure):
    _fields_ = [(n, ctypes.c_void_p) for n in LTAE_MLP_BWD_IO_FIELDS]


class ConvDesc(ctypes.Structure):
    _fields_ = [(n, ctypes.c_int32) for n in ("frames", "c_in", "c_out", "H", "W", "kernel", "stride", "padding", "dtype")]


class ConvInputNorm(ctypes.Structure):
    _fields_ = [("stats", ctypes.c_void_p), ("gamma", ctypes.c_void_p), ("beta", ctypes.c_void_p),
                ("n_groups", ctypes.c_int32), ("n_sub", ctypes.c_int32), ("relu", ctypes.c_int32), ("eps", ctypes.c_float)]


class C2SError(RuntimeError):
    """A C-ABI call returned a non-zero status (message from ``c2s_last_error``)."""


_lock = threading.Lock()
_lib = None


def load() -> ctypes.CDLL:
    """Load ``libcrop2seg_b200.so`` (once).  Raises if it was not built -- there is no fallback."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            raise C2SError(
                f"{LIB_PATH} not found: build the CUDA library first "
                "(python -m crop2seg_b200.build, or __graft_entry__.build()). crop2seg_b200 has no fallback path.")
        lib = ctypes.CDLL(LIB_PATH)
        vp, sz, i32 = ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int
        lib.c2s_abi_version.restype = i32
        lib.c2s_last_error.restype = ctypes.c_char_p
        lib.c2s_last_kernel.restype = ctypes.c_char_p
        lib.c2s_last_ltae_kernel.restype = ctypes.c_char_p
        lib.c2s_launch_count.restype = ctypes.c_int64
        lib.c2s_reset_launch_count.restype = None
        lib.c2s_set_option.restype = i32
        lib.c2s_set_option.argtypes = [i32, i32]
        lib.c2s_get_option.restype = i32
        lib.c2s_get_option.argtypes = [i32]
        lib.c2s_agg_workspace_bytes.restype = sz
        lib.c2s_agg_workspace_bytes.argtypes = [ctypes.POINTER(AggDesc)]
        lib.c2s_agg_forward.restype = i32
        lib.c2s_agg_forward.argtypes = [ctypes.POINTER(AggDesc), vp, vp, vp, vp, vp, sz, vp]
        lib.c2s_agg_skipconv_workspace_bytes.restype = sz
        lib.c2s_agg_skipconv_workspace_bytes.argtypes = [ctypes.POINTER(AggDesc)]
        lib.c2s_agg_skipconv_forward.restype = i32
        lib.c2s_agg_skipconv_forward.argtypes = [ctypes.POINTER(AggDesc), vp, vp, vp, ctypes.POINTER(SkipConvParams), vp,
                                                 vp, sz, vp]
        lib.c2s_agg_skipconv_backward_workspace_bytes.restype = sz
        lib.c2s_agg_skipconv_backward_workspace_bytes.argtypes = [ctypes.POINTER(AggDesc)]
        lib.c2s_agg_skipconv_backward.restype = i32
        lib.c2s_agg_skipconv_backward.argtypes = [ctypes.POINTER(AggDesc), vp, vp, vp, ctypes.POINTER(SkipConvParams), vp,
                                                  vp, ctypes.POINTER(SkipConvBwdIo), vp, sz, vp]
        lib.c2s_agg_skipconv_bstats_workspace_bytes.restype = sz
        lib.c2s_agg_skipconv_bstats_workspace_bytes.argtypes = [ctypes.POINTER(AggDesc)]
        lib.c2s_agg_skipconv_bstats_forward.restype = i32
        lib.c2s_agg_skipconv_bstats_forward.argtypes = [ctypes.POINTER(AggDesc), vp, vp, vp, ctypes.POINTER(SkipConvParams),
                                                        vp, vp, vp, vp, vp, sz, vp]
        lib.c2s_agg_skipconv_bstats_backward_workspace_bytes.restype = sz
        lib.c2s_agg_skipconv_bstats_backward_workspace_bytes.argtypes = [ctypes.POINTER(AggDesc)]
        lib.c2s_agg_skipconv_bstats_backward.restype = i32
        lib.c2s_agg_skipconv_bstats_backward.argtypes = [ctypes.POINTER(AggDesc), vp, vp, vp, ctypes.POINTER(SkipConvParams),
                                                         vp, vp, vp, vp, vp, ctypes.POINTER(SkipConvBwdIo), vp, sz, vp]
        lib.c2s_ltae_rows_forward.restype = i32
        lib.c2s_ltae_rows_forward.argtypes = [vp, vp, vp, i32, vp, vp]
        lib.c2s_ltae_inconv_grad.restype = i32
        lib.c2s_ltae_inconv_grad.argtypes = [vp, vp, vp, vp, vp, ctypes.c_int64, i32, i32, i32, vp]
        lib.c2s_pad_mask.restype = i32
        lib.c2s_pad_mask.argtypes = [vp, i32, ctypes.c_int64, ctypes.c_int64, ctypes.c_float, vp, vp]
        lib.c2s_agg_backward_workspace_bytes.restype = sz
        lib.c2s_agg_backward_workspace_bytes.argtypes = [ctypes.POINTER(AggDesc)]
        lib.c2s_agg_backward.restype = i32
        lib.c2s_agg_backward.argtypes = [ctypes.POINTER(AggDesc), vp, vp, vp, vp, vp, vp, vp, sz, vp]
        lib.c2s_ltae_workspace_bytes.restype = sz
        lib.c2s_ltae_workspace_bytes.argtypes = [ctypes.POINTER(LtaeDesc)]
        lib.c2s_ltae_forward.restype = i32
        lib.c2s_ltae_forward.argtypes = [ctypes.POINTER(LtaeDesc), ctypes.POINTER(LtaeParams), vp, vp, vp, vp, vp,
                                         vp, vp, vp, sz, vp]
        lib.c2s_ltae_backward_workspace_bytes.restype = sz
        lib.c2s_ltae_backward_workspace_bytes.argtypes = [ctypes.POINTER(LtaeDesc)]
        lib.c2s_ltae_backward.restype = i32
        lib.c2s_ltae_backward.argtypes = [ctypes.POINTER(LtaeDesc), ctypes.POINTER(LtaeParams), vp, vp, vp,
                                          ctypes.POINTER(LtaeBwdIo), vp, sz, vp]
        lib.c2s_ltae_mlp_backward_workspace_bytes.restype = sz
        lib.c2s_ltae_mlp_backward_workspace_bytes.argtypes = [ctypes.POINTER(LtaeDesc)]
        lib.c2s_ltae_mlp_backward.restype = i32
        lib.c2s_ltae_mlp_backward.argtypes = [ctypes.POINTER(LtaeDesc), ctypes.POINTER(LtaeParams),
                                              ctypes.POINTER(LtaeMlpBwdIo), vp, sz, vp]
        lib.c2s_tile_patchify.restype = i32
        lib.c2s_tile_patchify.argtypes = [ctypes.POINTER(TileDesc), vp, vp, vp, vp, vp, vp]
        lib.c2s_tile_classmap.restype = i32
        lib.c2s_tile_classmap.argtypes = [ctypes.POINTER(TileDesc), vp, i32, vp, vp, vp]
        lib.c2s_frame_index.restype = i32
        lib.c2s_frame_index.argtypes = [vp, ctypes.c_int64, vp, vp, vp]
        lib.c2s_frames_gather.restype = i32
        lib.c2s_frames_gather.argtypes = [vp, vp, vp, ctypes.c_int64, ctypes.c_int64, i32, vp]
        lib.c2s_frames_scatter.restype = i32
        lib.c2s_frames_scatter.argtypes = [vp, vp, vp, ctypes.c_int64, ctypes.c_int64, i32, ctypes.c_float, vp]
        lib.c2s_boundary_target.restype = i32
        lib.c2s_boundary_target.argtypes = [vp, i32, i32, i32, i32, vp, vp]
        lib.c2s_seg_loss_workspace_bytes.restype = sz
        lib.c2s_seg_loss_workspace_bytes.argtypes = []
        lib.c2s_seg_loss_forward.restype = i32
        lib.c2s_seg_loss_forward.argtypes = [ctypes.POINTER(LossDesc), vp, vp, vp, vp, vp, sz, vp]
        lib.c2s_seg_loss_backward.restype = i32
        lib.c2s_seg_loss_backward.argtypes = [ctypes.POINTER(LossDesc), vp, vp, vp, vp, vp, vp, vp]
        lib.c2s_ltae_fold_backward.restype = i32
        lib.c2s_ltae_fold_backward.argtypes = [ctypes.POINTER(LtaeDesc), ctypes.POINTER(LtaeParams),
                                               ctypes.POINTER(LtaeFoldBwdIo), vp, sz, vp]
        lib.c2s_conv2d_supported.restype = i32
        lib.c2s_conv2d_supported.argtypes = [ctypes.POINTER(ConvDesc)]
        lib.c2s_conv2d_workspace_bytes.restype = sz
        lib.c2s_conv2d_workspace_bytes.argtypes = [ctypes.POINTER(ConvDesc)]
        lib.c2s_conv2d_forward.restype = i32
        lib.c2s_conv2d_forward.argtypes = [ctypes.POINTER(ConvDesc), vp, ctypes.POINTER(ConvInputNorm), vp, vp, vp, vp, vp, sz, vp]
        lib.c2s_group_stats.restype = i32
        lib.c2s_group_stats.argtypes = [vp, i32, ctypes.c_int64, i32, ctypes.c_int64, i32, vp, vp]
        lib.c2s_group_norm_relu.restype = i32
        lib.c2s_group_norm_relu.argtypes = [vp, vp, i32, vp, vp, vp, vp, i32, ctypes.c_int64, i32, ctypes.c_int64, i32,
                                            ctypes.c_float, i32, vp]
        got = lib.c2s_abi_version()
        if got != C2S_ABI_VERSION:
            raise C2SError(f"ABI mismatch: library reports version {got}, binding expects {C2S_ABI_VERSION}")
        _lib = lib
    return _lib


def check(status: int, what: str) -> None:
    if status != 0:
        msg = load().c2s_last_error().decode("utf-8", "replace")
        raise C2SError(f"{what} failed with status {status}: {msg}")


def launch_count() -> int:
    return int(load().c2s_launch_count())


def reset_launch_count() -> None:
    load().c2s_reset_launch_count()


def last_kernel() -> str:
    return load().c2s_last_kernel().decode("utf-8", "replace")


def last_ltae_kernel() -> str:
    """The L-TAE attention kernel that served the last ``c2s_ltae_forward`` call."""
    return load().c2s_last_ltae_kernel().decode("utf-8", "replace")


class option:
    """``with _lib.option(_lib.OPT_LTAE_KERNEL, _lib.LTAE_KERNEL_GENERAL): ...`` -- process-wide kernel-selection
    switch of the library (``c2s_set_option``), restored on exit.  For parity tests and A/B measurements; production
    leaves every option at 0."""

    def __init__(self, which: int, value: int):
        self.which, self.value = which, int(value)

    def __enter__(self):
        lib = load()
        self.old = lib.c2s_get_option(self.which)
        check(lib.c2s_set_option(self.which, self.value), "c2s_set_option")
        return self

    def __exit__(self, *exc):
        load().c2s_set_option(self.which, self.old)
