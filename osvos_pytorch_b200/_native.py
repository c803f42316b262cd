"""ctypes binding of libosvos_b200.so (the C ABI declared in include/osvos_b200.h).

This is the stub a maintainer of the reference would add to call the native hot
path from Python (INTEGRATION.md).  There is deliberately NO fallback: if the
library cannot be loaded, or a call fails, an exception is raised.
"""
import ctypes
import os
from ctypes import (POINTER, Structure, c_char_p, c_double, c_float, c_int, c_int32, c_size_t, c_uint32, c_uint64,
                    c_void_p)

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libosvos_b200.so")

FLAG_RELU = 1
FLAG_FAST = 2
FLAG_RELU_MASK = 4
FLAG_ACCUMULATE = 8
FLAG_DEFER_FINISH = 16
WGRAD_FINISH_MAX = 24


class NativeLibraryError(RuntimeError):
    pass


class Conv3x3Args(Structure):
    _fields_ = [("x_hi", c_void_p), ("x_lo", c_void_p), ("w_packed", c_void_p), ("bias", c_void_p),
                ("y_hi", c_void_p), ("y_lo", c_void_p), ("y_f32", c_void_p), ("mask_hi", c_void_p),
                ("proj_w", c_void_p), ("proj_b", c_void_p), ("pq", c_void_p),
                ("pool_hi", c_void_p), ("pool_lo", c_void_p), ("colsum", c_void_p),
                ("n", c_int), ("h", c_int), ("w", c_int), ("cin", c_int), ("cout", c_int), ("flags", c_int),
                ("k_valid", c_int)]


class Stage1Args(Structure):
    _fields_ = [("x", c_void_p), ("w1", c_void_p), ("b1", c_void_p), ("w2_packed", c_void_p), ("b2", c_void_p),
                ("y_hi", c_void_p), ("y_lo", c_void_p), ("pool_hi", c_void_p), ("pool_lo", c_void_p),
                ("n", c_int), ("h", c_int), ("w", c_int)]


class TailFwdArgs(Structure):
    _fields_ = [("pq", c_void_p * 4), ("fuse_bias", c_void_p), ("out", c_void_p * 5), ("label", c_void_p),
                ("sums", c_void_p), ("losses", c_void_p), ("loss_weights", c_float * 5), ("divisor", c_float),
                ("n", c_int), ("h", c_int), ("w", c_int)]


TAIL_SUMS = 15


class TailLossBwdArgs(Structure):
    _fields_ = [("logits", c_void_p * 5), ("label", c_void_p), ("sums", c_void_p), ("upstream", c_void_p),
                ("loss_weights", c_float * 5), ("divisor", c_float), ("dpq", c_void_p * 4), ("fuse_bias_grad", c_void_p),
                ("n", c_int), ("h", c_int), ("w", c_int)]


class WgradArgs(Structure):
    _fields_ = [("x_hi", c_void_p), ("x_lo", c_void_p), ("dz_hi", c_void_p), ("dz_lo", c_void_p), ("dw", c_void_p),
                ("workspace", c_void_p), ("n", c_int), ("h", c_int), ("w", c_int), ("cin", c_int), ("cout", c_int),
                ("dz_channels", c_int), ("flags", c_int)]


class LaunchPlan(Structure):
    """osvos_launch_plan (include/osvos_b200.h)."""
    _fields_ = [("block_n", c_int), ("planes", c_int), ("split_acc", c_int), ("lean", c_int), ("items", c_int),
                ("grid", c_int), ("tap_mode", c_int), ("pixel_splits", c_int)]


TAP_ROWS, TAP_PAIRS, TAP_NINE = 3, 5, 9


class WgradFinishItem(Structure):
    _fields_ = [("workspace", c_void_p), ("dw", c_void_p), ("cout", c_int), ("cin", c_int), ("dz_channels", c_int),
                ("accumulate", c_int), ("scale", c_float)]


class FoldItem(Structure):
    """osvos_fold_item (include/osvos_b200.h)."""
    _fields_ = [("side_w", c_void_p), ("side_b", c_void_p), ("proj_w", c_void_p), ("proj_b", c_void_p),
                ("packed", c_void_p), ("bias2", c_void_p), ("folded_f32", c_void_p), ("cin", c_int)]


class SideWgradItem(Structure):
    """osvos_side_wgrad_item (include/osvos_b200.h)."""
    _fields_ = [("x_hi", c_void_p), ("x_lo", c_void_p), ("dpq", c_void_p), ("g", c_void_p), ("n", c_int), ("h", c_int),
                ("w", c_int), ("c", c_int)]


class SideGradsItem(Structure):
    """osvos_side_grads_item (include/osvos_b200.h)."""
    _fields_ = [("g", c_void_p), ("side_w", c_void_p), ("side_b", c_void_p), ("proj_w", c_void_p),
                ("d_side_w", c_void_p), ("d_side_b", c_void_p), ("d_score_w", c_void_p), ("d_score_b", c_void_p),
                ("d_fuse_w", c_void_p), ("c", c_int), ("accumulate", c_int)]


class TailBwdArgs(Structure):
    _fields_ = [("grad_out", c_void_p * 5), ("dpq", c_void_p * 4), ("n", c_int), ("h", c_int), ("w", c_int)]


class SgdSegment(Structure):
    """osvos_sgd_segment (include/osvos_b200.h); 80 bytes, uploaded as a device table."""
    _fields_ = [("param", c_void_p), ("grad", c_void_p), ("momentum", c_void_p), ("numel", c_uint64),
                ("lr", c_float), ("weight_decay", c_float), ("momentum_coef", c_float),
                ("cout", c_int32), ("cin", c_int32), ("colp_fwd", c_int32), ("colp_flip", c_int32),
                ("work_items", c_uint32), ("packed_fwd", c_void_p), ("packed_flip", c_void_p)]


U8_PROB, U8_BYTESCALE, U8_MASK = 0, 1, 2
SGD_MAX_SEGMENTS = 64

# name -> (restype, argtypes); mirrors include/osvos_b200.h one to one (tests/test_abi.py checks it)
SIGNATURES = {
    "osvos_version": (c_int, []),
    "osvos_last_error": (c_char_p, []),
    "osvos_packed_weight_bytes": (c_size_t, [c_int, c_int]),
    "osvos_pack_conv3x3_weights": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p]),
    "osvos_nchw_to_act": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p]),
    "osvos_act_to_nchw": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p]),
    "osvos_conv_first_fwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int,
                                     c_void_p]),
    "osvos_conv3x3": (c_int, [POINTER(Conv3x3Args), c_void_p]),
    "osvos_conv3x3_plan": (c_int, [POINTER(Conv3x3Args), POINTER(LaunchPlan)]),
    "osvos_stage1_fused": (c_int, [POINTER(Stage1Args), c_void_p]),
    "osvos_set_pdl": (c_int, [c_int]),
    "osvos_fold_side_weights": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p]),
    "osvos_side_folded_multi": (c_int, [POINTER(Conv3x3Args), c_int, c_void_p]),
    "osvos_fold_side_weights_multi": (c_int, [POINTER(FoldItem), c_int, c_void_p]),
    "osvos_conv3x3_simt": (c_int, [POINTER(Conv3x3Args), c_void_p]),
    "osvos_maxpool2x2_fwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p]),
    "osvos_tail_fwd": (c_int, [POINTER(TailFwdArgs), c_void_p]),
    "osvos_cbce_fwd": (c_int, [c_void_p, c_void_p, c_size_t, c_double, c_void_p, c_void_p, c_void_p]),
    "osvos_cbce_bwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_double, c_size_t, c_void_p, c_void_p]),
    "osvos_wgrad_workspace_bytes": (c_size_t, [c_int, c_int]),
    "osvos_conv3x3_wgrad": (c_int, [POINTER(WgradArgs), c_void_p]),
    "osvos_conv3x3_wgrad_plan": (c_int, [POINTER(WgradArgs), POINTER(LaunchPlan)]),
    "osvos_wgrad_finish": (c_int, [POINTER(WgradFinishItem), c_int, c_void_p]),
    "osvos_tail_bwd": (c_int, [POINTER(TailBwdArgs), c_void_p]),
    "osvos_tail_loss_bwd": (c_int, [POINTER(TailLossBwdArgs), c_void_p]),
    "osvos_sum_f32": (c_int, [c_void_p, c_size_t, c_void_p, c_void_p, c_void_p]),
    "osvos_unpool_add_mask": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                      c_int, c_int, c_int, c_int, c_void_p]),
    "osvos_side_folded_wgrad_floats": (c_size_t, [c_int]),
    "osvos_side_folded_wgrad": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p]),
    "osvos_side_folded_wgrad_multi": (c_int, [POINTER(SideWgradItem), c_int, c_void_p]),
    "osvos_side_grads_finish": (c_int, [POINTER(SideGradsItem), c_int, c_void_p]),
    "osvos_unpool_side_mask": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                       c_void_p, c_int, c_int, c_int, c_int, c_void_p]),
    "osvos_channel_sum": (c_int, [c_void_p, c_void_p, c_void_p, c_size_t, c_int, c_void_p]),
    "osvos_conv_first_bwd_workspace_bytes": (c_size_t, []),
    "osvos_conv_first_bwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int,
                                     c_void_p]),
    "osvos_side_project": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p]),
    "osvos_logits_to_u8": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_size_t, c_int, c_void_p]),
    "osvos_sgd_work_items": (c_uint32, [c_uint64, c_int, c_int]),
    "osvos_sgd_step": (c_int, [c_void_p, c_int, c_uint32, c_int, c_void_p]),
    "osvos_affine_warp": (c_int, [c_void_p, c_void_p, POINTER(c_double), POINTER(c_int), c_int, c_int, c_int, c_int,
                                  c_int, c_void_p]),
}

_lib = None


def load():
    """Load the shared library once; raise NativeLibraryError if it is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise NativeLibraryError(
            f"{LIB_PATH} not found: build it with `python -m osvos_pytorch_b200.build` "
            "(or __graft_entry__.build()).  There is no CPU / PyTorch fallback for the OSVOS hot path.")
    try:
        lib = ctypes.CDLL(LIB_PATH)
    except OSError as e:  # pragma: no cover
        raise NativeLibraryError(f"cannot load {LIB_PATH}: {e}") from e
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(status, what):
    if status != 0:
        msg = load().osvos_last_error()
        raise NativeLibraryError(f"{what} failed with status {status}: {msg.decode() if msg else ''}")


def ptr(t):
    """Device pointer of a tensor (None -> NULL)."""
    return None if t is None else t.data_ptr()
