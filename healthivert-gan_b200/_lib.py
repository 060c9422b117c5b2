"""ctypes binding of libhv_b200.so (C ABI declared in include/hv_b200.h).

There is NO CPU fallback: if the library is missing, or a compute entry point is called
without a CUDA device / with CPU tensors, the call raises.
"""
import ctypes
import os
from ctypes import (POINTER, Structure, c_char_p, c_float, c_int, c_int32, c_longlong, c_size_t,
                    c_uint64, c_void_p)

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libhv_b200.so")

HV_ACT = {"none": 0, "elu": 1, "relu": 2, "sigmoid": 3, "lrelu": 4, "clamp1": 5, "heads": 6}
HV_SRC_DIRECT, HV_SRC_UP2, HV_SRC_SUB2, HV_SRC_SCALAR = 0, 1, 2, 3
HV_PREC = {"fp32": 0, "bf16": 1}


class HvError(RuntimeError):
    pass


class hv_conv_src(Structure):
    _fields_ = [("ptr", c_void_p), ("channels", c_int), ("mode", c_int)]


class hv_conv_desc(Structure):
    _fields_ = [("n", c_int), ("cin", c_int), ("cout", c_int), ("hin", c_int), ("win", c_int),
                ("k", c_int), ("stride", c_int), ("pad", c_int), ("dil", c_int), ("act", c_int),
                ("nsrc", c_int), ("src", hv_conv_src * 4)]


# name -> (restype, argtypes); every symbol include/hv_b200.h declares
SIGNATURES = {
    "hv_last_error": (c_char_p, []),
    "hv_version": (c_int, []),
    "hv_launch_count": (c_uint64, []),
    "hv_sn_prepare": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "hv_conv2d_fwd": (c_int, [POINTER(hv_conv_desc), c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "hv_conv2d_bf16": (c_int, [POINTER(hv_conv_desc), c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p]),
    "hv_gap_fc_sigmoid": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p]),
    "hv_ctx_attn_workspace_bytes": (c_size_t, [c_int, c_int, c_int, c_int]),
    "hv_ctx_attn_fwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int,
                                c_float, c_int, c_int, c_void_p, c_void_p]),
    "hv_ctx_attn_fwd_bf16": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int,
                                     c_float, c_int, c_int, c_void_p]),
    "hv_stitch": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_void_p,
                          c_int, c_int, c_int, c_void_p]),
    "hv_threshold": (c_int, [c_void_p, c_void_p, c_void_p, c_float, c_size_t, c_void_p]),
    "hv_sobel": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p]),
    "hv_edge_xor_loss": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p]),
    "hv_column_heights": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p,
                                  c_void_p]),
    "hv_conv2d_dgrad": (c_int, [POINTER(hv_conv_desc), c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "hv_conv2d_wgrad": (c_int, [POINTER(hv_conv_desc), c_void_p, c_void_p, c_void_p, c_void_p]),
    "hv_act_bwd": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_size_t, c_void_p]),
    "hv_upsample2_bwd": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p]),
    "hv_stitch_bwd": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p]),
    "hv_axpby": (c_int, [c_float, c_void_p, c_float, c_void_p, c_size_t, c_void_p]),
    "hv_affine": (c_int, [c_float, c_void_p, c_float, c_void_p, c_size_t, c_void_p]),
    "hv_height_loss": (c_int, [c_void_p, c_void_p, c_void_p, c_float, c_int, c_void_p, c_void_p, c_void_p, c_void_p]),
    "hv_masked_center": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_size_t, c_void_p]),
    "hv_sn_bwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p]),
    "hv_gap_fc_sigmoid_bwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_void_p,
                                      c_int, c_int, c_int, c_void_p]),
    "hv_ctx_attn_bwd_workspace_bytes": (c_size_t, [c_int, c_int, c_int, c_int]),
    "hv_ctx_attn_bwd": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_float, c_int, c_void_p, c_void_p,
                                c_void_p]),
    "hv_ctx_attn_fwd_tc": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int,
                                c_float, c_int, c_int, c_void_p, c_void_p]),
    "hv_ctx_attn_bwd_tc": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_float, c_int, c_void_p, c_void_p,
                                c_void_p]),
    "hv_bn_lrelu_fwd": (c_int, [c_void_p] * 8 + [c_int, c_int, c_int, c_float, c_float, c_float, c_void_p]),
    "hv_bn_lrelu_bwd": (c_int, [c_void_p] * 9 + [c_int, c_int, c_int, c_float, c_void_p]),
    "hv_in_lrelu_fwd": (c_int, [c_void_p] * 5 + [c_int, c_int, c_int, c_float, c_float, c_void_p]),
    "hv_in_lrelu_bwd": (c_int, [c_void_p] * 7 + [c_int, c_int, c_int, c_float, c_void_p]),
    "hv_act_fwd": (c_int, [c_void_p, c_void_p, c_int, c_size_t, c_void_p]),
    "hv_reduce_scalar": (c_int, [c_void_p, c_void_p, c_float, c_int, c_size_t, c_float, c_void_p, c_void_p, c_void_p]),
    "hv_loss_grad": (c_int, [c_void_p, c_void_p, c_float, c_int, c_float, c_void_p, c_int, c_void_p, c_int, c_size_t,
                             c_void_p]),
    "hv_dice_fwd": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_float, c_void_p]),
    "hv_dice_bwd": (c_int, [c_void_p, c_void_p, c_float, c_float, c_void_p, c_int, c_int, c_int, c_void_p]),
    "hv_adam_step": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_float, c_float, c_float, c_float, c_int,
                             c_void_p]),
    "hv_multi_tensor_chunk": (c_int, []),
    "hv_adam_step_multi": (c_int, [c_void_p, c_int, c_longlong, c_float, c_float, c_float, c_float, c_int, c_void_p]),
    "hv_bucket_copy": (c_int, [c_void_p, c_int, c_longlong, c_void_p, c_float, c_int, c_void_p]),
    "hv_debug_conv_trace": (c_int, [c_void_p]),
    "hv_debug_conv_timeline": (c_int, [c_void_p]),
    "hv_act_bwd_bias": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p]),
    "hv_sn_prepare_multi": (c_int, [c_void_p, c_int, c_int, c_void_p]),
    "hv_sn_bwd_multi": (c_int, [c_void_p, c_int, c_void_p]),
    "hv_post_forward": (c_int, [c_void_p] * 12 + [c_int, c_int, c_int] + [c_void_p] * 12 + [c_int, c_int, c_int, c_void_p]),
    "hv_conv2d_wgrad_bf16_workspace_bytes": (c_size_t, [POINTER(hv_conv_desc)]),
    "hv_conv2d_dgrad_bf16_workspace_bytes": (c_size_t, [POINTER(hv_conv_desc)]),
    "hv_conv2d_wgrad_bf16": (c_int, [POINTER(hv_conv_desc), c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "hv_conv2d_dgrad_bf16": (c_int, [POINTER(hv_conv_desc), c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "hv_dconv_workspace_bytes": (c_size_t, [c_int] * 6),
    "hv_dconv_fwd_bf16": (c_int, [c_void_p, c_void_p, c_void_p] + [c_int] * 6 + [c_void_p, c_void_p]),
    "hv_dconv_bwd_bf16": (c_int, [c_void_p] * 5 + [c_int] * 6 + [c_void_p, c_void_p]),
    "hv_pixel_d_workspace_bytes": (c_size_t, [c_int] * 3),
    "hv_pixel_d_fwd_bf16": (c_int, [c_void_p] * 14 + [c_int] * 6 + [c_float] * 3 + [c_void_p, c_void_p]),
    "hv_pixel_d_bwd_bf16": (c_int, [c_void_p] * 21 + [c_int] * 6 + [c_float, c_void_p, c_void_p]),
    "hv_vol_to_u8": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, ctypes.c_double, c_void_p]),
    "hv_slice_id_counts": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    "hv_slice_prepare": (c_int, [c_void_p] * 5 + [c_int, c_int, c_int, c_int] + [c_void_p] * 10 + [c_void_p]),
    "hv_slice_finish": (c_int, [c_void_p] * 7 + [c_int, c_int, c_int] + [c_void_p] * 4 + [c_void_p]),
    "hv_resample_curve": (c_int, [c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_int, c_int, c_int, c_int, ctypes.c_double, c_void_p, c_void_p]),
    "hv_generator_num_layers": (c_int, []),
    "hv_generator_layer_info": (c_int, [c_int, c_char_p] + [POINTER(c_int)] * 7),
    "hv_generator_create": (c_int, [POINTER(c_void_p), c_int, c_int]),
    "hv_generator_destroy": (c_int, [c_void_p]),
    "hv_generator_set_layer": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p]),
    "hv_generator_set_fc": (c_int, [c_void_p, c_int, c_void_p, c_void_p]),
    "hv_generator_prepare": (c_int, [c_void_p, c_int, c_void_p]),
    "hv_generator_forward": (c_int, [c_void_p] + [c_void_p] * 4 + [c_int] + [c_void_p] * 8 + [c_int, c_void_p]),
    "hv_generator_run_layer": (c_int, [c_void_p, c_int, c_int, c_void_p]),
    "hv_generator_run_chain": (c_int, [c_void_p, c_int, c_int, c_int, c_void_p]),
    "hv_pipeline_create": (c_int, [POINTER(c_void_p), c_void_p, c_int, c_int, c_int, c_int]),
    "hv_pipeline_destroy": (c_int, [c_void_p]),
    "hv_pipeline_slot": (c_int, [c_void_p, c_int] + [POINTER(c_void_p)] * 8),
    "hv_pipeline_bytes": (c_size_t, [c_void_p, c_int]),
    "hv_pipeline_stream": (c_void_p, [c_void_p, c_int]),
    "hv_pipeline_submit": (c_int, [c_void_p, c_int, c_int]),
    "hv_pipeline_wait": (c_int, [c_void_p, c_int]),
    "hv_generator_read_tap": (c_longlong, [c_void_p, c_int, c_void_p, c_void_p]),
}

_lib = None


def lib():
    """Load the shared library once; fail loudly when it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise HvError(
                f"{LIB_PATH} is missing: the CUDA extension has not been built "
                "(run `python -c 'import __graft_entry__ as g; g.build()'`). There is no CPU fallback.")
        handle = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(handle, name)
            fn.restype = res
            fn.argtypes = args
        _lib = handle
    return _lib


def check(rc):
    if rc is not None and rc < 0:
        msg = lib().hv_last_error().decode("utf-8", "replace")
        raise HvError(f"hv_b200 error {rc}: {msg}")
    return rc


def ptr(t):
    """Device pointer of a contiguous CUDA tensor (None -> NULL)."""
    if t is None:
        return None
    if not t.is_cuda:
        raise HvError("hv_b200 kernels need CUDA tensors (no CPU fallback)")
    if not t.is_contiguous():
        raise HvError("hv_b200 kernels need contiguous tensors")
    return t.data_ptr()


def stream():
    import torch
    return torch.cuda.current_stream().cuda_stream


def launch_count():
    return int(lib().hv_launch_count())
