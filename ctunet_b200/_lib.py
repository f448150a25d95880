"""ctypes binding of the C ABI declared in include/ctunet_b200.h.

The shared library is built in-tree (``ctunet_b200/libctunet_b200.so``) by ``__graft_entry__.build()``
or ``make -C ctunet_b200/csrc``.  There is no CPU fallback: if the library is missing, or a call
fails, a RuntimeError is raised.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import c_char_p, c_double, c_float, c_int, c_longlong, c_ulonglong, c_void_p

import torch  # noqa: F401  (loads libcudart / libcuda into the process before our library)

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("CTUNET_B200_LIB") or os.path.join(_HERE, "libctunet_b200.so")   # override: A/B builds

CTU_F32, CTU_BF16 = 0, 1
CTU_MAX_SRC = 4
CTU_ACCUM_PREZEROED = 0x100   # include/ctunet_b200.h: the caller zeroed the double accumulators
HEAD_SOFTMAX, HEAD_SIGMOID, HEAD_SP, HEAD_SP_SOFTMAX = 1, 2, 4, 8

P = c_void_p
I = c_int
LL = c_longlong
ULL = c_ulonglong
D = c_double
F = c_float

# name -> (restype, argtypes); must list every function of include/ctunet_b200.h
SIGNATURES = {
    "ctu_last_error": (c_char_p, []),
    "ctu_version": (I, []),
    "ctu_has_tensor_path": (I, []),
    "ctu_pack_ncdhw": (I, [P, P, I, I, I, LL, P]),
    "ctu_unpack_ncdhw": (I, [P, P, I, I, I, LL, P]),
    "ctu_pack_patches": (I, [P, P, P, I, I, I, I, I, I, I, P]),
    "ctu_head_labels": (I, [I, P, P, I, P, P, I, I, P, I, I, I, I, P, P, I, LL, P]),
    "ctu_head_accumulate": (I, [I, P, P, I, P, P, I, I, P, I, I, I, I, P, P, I, LL, P]),
    "ctu_window_finalize": (I, [P, I, I, I, I, I, P, P, P, P, P, P]),
    "ctu_conv_wpack_floats": (LL, [I, I, I, P]),
    "ctu_conv_pack_weight": (I, [P, P, I, I, I, P, P]),
    "ctu_conv_wpack_dgrad_floats": (LL, [I, I, I]),
    "ctu_conv_pack_weight_dgrad": (I, [P, P, I, I, I, P, I, P]),
    "ctu_conv_unpack_wgrad": (I, [P, P, I, I, I, P, P]),
    "ctu_conv3d_fprop": (I, [I, P, P, I, P, P, P, P, I, I, I, I, I, I, I, I, P]),
    "ctu_conv_tc_bnred_supported": (I, [I, I, P, I, I, I, I]),
    "ctu_conv3d_dgrad_bnred": (I, [P, P, I, P, P, I, I, I, I, I, I, P, P, P, I, P]),
    "ctu_conv_tc_supported": (I, [I, I, P, I, I, I, I]),
    "ctu_conv_tc_wgrad_supported": (I, [I, I, P, I, I, I, I]),
    "ctu_conv_tc_wimg_bytes": (LL, [I, I, P, I]),
    "ctu_conv_tc_pack_weight": (I, [P, P, I, I, P, I, P]),
    "ctu_conv_wide_supported": (I, [I, I, I, I, I, I, I]),
    "ctu_conv_wide_wimg_bytes": (LL, [I, I, I, I, I, I, I]),
    "ctu_conv_wide_pack_weight": (I, [P, P, I, I, I, I, I, I, I, P]),
    "ctu_conv_wide_wgrad_supported": (I, [I, I, I, I, I, I]),
    "ctu_upfuse_cout": (I, [I]),
    "ctu_upfuse_workspace_floats": (LL, [I, I, I]),
    "ctu_upfuse_compose": (I, [P, P, P, P, P, P, I, I, I, P, P]),
    "ctu_upfuse_decompose": (I, [P, P, P, P, P, P, P, P, P, I, I, I, P, P]),
    "ctu_conv3d_wgrad": (I, [I, P, P, I, P, P, P, I, I, I, I, I, I, I, I, P]),
    "ctu_convt_wpack_floats": (LL, [I, I, P]),
    "ctu_convt_pack_weight": (I, [P, P, I, I, P, P]),
    "ctu_convt_wpack_dgrad_floats": (LL, [I, I]),
    "ctu_convt_pack_weight_dgrad": (I, [P, P, I, I, P, I, P]),
    "ctu_convt_unpack_wgrad": (I, [P, P, I, I, P, P]),
    "ctu_gather_batch": (I, [I, P, P, P, P, P, P]),
    "ctu_convt2_fprop": (I, [I, P, P, I, P, P, P, I, I, I, I, I, P]),
    "ctu_convt2_dgrad": (I, [I, P, P, P, I, I, I, I, I, I, P]),
    "ctu_convt2_wgrad": (I, [I, P, P, I, P, P, P, I, I, I, I, I, P]),
    "ctu_bn_stats": (I, [I, P, I, I, I, LL, P, P]),
    "ctu_bn_finalize": (I, [P, D, P, P, P, P, P, F, F, I, I, I, P, P]),
    "ctu_bn_running_update": (I, [P, D, P, P, P, F, I, I, P]),
    "ctu_bn_relu_fwd": (I, [I, P, P, P, P, I, I, I, I, I, I, P]),
    "ctu_bn_relu_fwd_train": (I, [I, P, P, D, P, P, P, P, P, F, F, I, P, P, P, I, I, I, I, I, I, P]),
    "ctu_bn_relu_bwd_reduce": (I, [I, P, P, P, P, P, I, I, I, I, I, I, P]),
    "ctu_bn_relu_bwd_apply": (I, [I, P, P, P, P, P, P, D, P, P, P, I, I, I, I, I, I, P]),
    "ctu_bn_relu_fwd_drop": (I, [I, P, P, P, P, I, I, I, I, I, I, P, P]),
    "ctu_bn_relu_fwd_train_drop": (I, [I, P, P, D, P, P, P, P, P, F, F, I, P, P, P, I, I, I, I, I, I, P, P]),
    "ctu_bn_relu_bwd_reduce_drop": (I, [I, P, P, P, P, P, I, I, I, I, I, I, P, P]),
    "ctu_bn_relu_bwd_apply_drop": (I, [I, P, P, P, P, P, P, D, P, P, P, I, I, I, I, I, I, P, P]),
    "ctu_dropout3d_keep": (I, [I, P, P, P, I, ULL, P, P, P]),
    "ctu_head_fwd": (I, [I, P, P, I, P, P, I, I, P, P, I, LL, P]),
    "ctu_head_bwd": (I, [I, P, P, I, P, P, I, I, P, P, P, P, P, P, P, I, LL, P]),
    "ctu_head_loss_fwd": (I, [I, P, P, I, P, P, I, I, P, P, I, I, F, F, P, P, P, I, LL, P]),
    "ctu_head_loss_bwd": (I, [I, P, P, I, P, P, I, I, P, P, I, I, F, F, P, P, P, I, LL, P]),
    "ctu_head_param_grad": (I, [I, P, P, I, P, I, P, P, I, LL, P]),
    "ctu_dice_ce_fwd": (I, [P, P, I, I, LL, I, I, P, P, P]),
    "ctu_dice_ce_bwd": (I, [P, P, I, I, LL, I, I, P, P, P, P]),
    "ctu_argmax_channels": (I, [P, P, I, I, LL, P]),
    "ctu_count_nonzero_u8": (I, [P, LL, P, P]),
    "ctu_kth_nonzero_u8": (I, [P, I, I, I, LL, P, P, P]),
    "ctu_flap_mask_u8": (I, [P, P, P, I, I, I, P, D, I, D, P]),
    "ctu_encode_flaprec_u8": (I, [P, P, P, P, P, P, P, I, I, LL, P]),
    "ctu_encode_flaprec_bits": (I, [P, P, P, P, P, P, P, I, I, LL, P]),
    "ctu_hu_window": (I, [P, P, LL, F, F, P]),
    "ctu_hu_threshold": (I, [P, P, LL, I, P]),
    "ctu_resample_nearest_f32": (I, [P, P, I, I, I, I, I, I, P]),
    "ctu_resample_nearest_u8": (I, [P, P, I, I, I, I, I, I, P]),
    "ctu_resample_nearest_index": (I, [P, I, I, P]),
    "ctu_resample_trilinear_f32": (I, [P, P, I, I, I, I, I, I, P]),
    "ctu_components_workspace_bytes": (LL, [I, I, I, I]),
    "ctu_label_components": (I, [I, P, I, I, I, I, I, P, P, P, LL, P]),
    "ctu_filter_components": (I, [I, P, I, I, I, I, I, LL, P, P, LL, P]),
    "ctu_dice_coeff": (I, [P, P, I, I, LL, P, P, P]),
    "ctu_hausdorff_workspace_bytes": (LL, [I, I, I, I, I]),
    "ctu_hausdorff": (I, [P, P, I, I, I, I, I, D, P, LL, P, P]),
    "ctu_surface_metrics_workspace_bytes": (LL, [I, I, I, I, I]),
    "ctu_surface_metrics": (I, [I, P, I, P, I, I, I, I, P, D, D, P, P, LL, P]),
    "ctu_loss_combine": (I, [P, P, I, P, P, P]),
    "ctu_optim_chunk_bytes": (I, []),
    "ctu_optim_chunk_elems": (I, []),
    "ctu_optim_step": (I, [I, P, I, P, P, P, P, P, P, D, D, D, D, D, D, I, D, P]),
    "ctu_optim_post": (I, [P, P, P, I, P]),
    "ctu_peer_flag_bytes": (I, []),
    "ctu_peer_alloc": (I, [LL, P, P]),
    "ctu_peer_open": (I, [P, P]),
    "ctu_peer_close": (I, [P]),
    "ctu_peer_free": (I, [P]),
    "ctu_peer_signal": (I, [P, P, I, I, P]),
    "ctu_peer_wait_done": (I, [P, P, I, I, P]),
    "ctu_optim_step_peer": (I, [I, P, I, P, P, I, I, P, P, P, P, P, D, D, D, D, D, D, I, D, P, LL, I, P]),
    "ctu_peer_error": (I, [P]),
    "ctu_salt_pepper_u8": (I, [P, P, LL, D, D, P, P, ULL, ULL, P]),
    "ctu_affine_draw": (I, [I, I, I, I, P, I, ULL, P, P, P, P]),
    "ctu_affine_encode_flaprec": (I, [I, P, P, P, P, P, P, P, P, I, I, I, I, I, P]),
    "ctu_affine_masks_u8": (I, [I, P, P, P, I, I, I, I, P]),
    "ctu_craniectomy_workspace_bytes": (LL, [I, I, I, I]),
    "ctu_craniectomy_draw": (I, [I, P, I, I, I, I, D, I, I, I, ULL, P, P, P, LL, P]),
    "ctu_craniectomy_encode_flaprec": (I, [I, P, P, P, P, P, P, P, I, I, I, I, I, P]),
    "ctu_craniectomy_masks_u8": (I, [P, P, P, P, P, I, I, I, I, P]),
}

_lib = None
launches = 0   # number of library entry points that enqueued GPU work (bench.py reports it)


def load() -> ctypes.CDLL:
    global _lib
    if _lib is None:
        if not os.path.isfile(LIB_PATH):
            raise RuntimeError(
                "ctunet_b200: %s is missing -- build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(there is no CPU or PyTorch fallback for the hot path)" % LIB_PATH)
        lib = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)      # AttributeError if the build is stale
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def last_error() -> str:
    return load().ctu_last_error().decode("utf-8", "replace")


def call(name: str, *args):
    """Invoke a status-returning entry point; raises RuntimeError on failure."""
    global launches
    rc = getattr(load(), name)(*args)
    if rc != 0:
        raise RuntimeError("%s failed (%d): %s" % (name, rc, last_error()))
    launches += 1


_raw_stream = getattr(torch._C, "_cuda_getCurrentRawStream", None)
_raw_device = getattr(torch._C, "_cuda_getDevice", None)


def stream_ptr() -> int:
    """cudaStream_t of torch's current stream on the current device (what every entry point is enqueued on).  The raw
    accessors cost ~0.3 us; ``torch.cuda.current_stream()`` builds a Stream object (~4 us, 165 times per eager step)."""
    if _raw_stream is not None and _raw_device is not None:
        return _raw_stream(_raw_device())
    return torch.cuda.current_stream().cuda_stream


def int_array(values):
    return (c_int * len(values))(*values)


def ll_array(values):
    return (c_longlong * len(values))(*values)


def ptr_array(values):
    return (c_void_p * len(values))(*values)
