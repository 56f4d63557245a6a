"""ctypes binding of libcrowdmod_b200.so (the C ABI declared in include/crowdmod_b200.h).

There is no fallback: if the shared library is missing the import of any compute path raises,
and every entry point that needs a GPU raises when called without one.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libcrowdmod_b200.so")

CM_MAX_LEVELS = 8


class UNetConfig(C.Structure):
    """struct cm_unet_config (include/crowdmod_b200.h)."""

    _fields_ = [
        ("in_channels", C.c_int32),
        ("out_channels", C.c_int32),
        ("num_res_blocks", C.c_int32),
        ("base_channels", C.c_int32),
        ("num_levels", C.c_int32),
        ("mult", C.c_int32 * CM_MAX_LEVELS),
        ("attn", C.c_int32 * CM_MAX_LEVELS),
        ("time_multiple", C.c_int32),
        ("rows", C.c_int32),
        ("cols", C.c_int32),
        ("past_len", C.c_int32),
        ("future_len", C.c_int32),
        ("table_steps", C.c_int32),
        ("weight_terms", C.c_int32),
        ("dgrad_terms", C.c_int32),
        ("train_act_terms", C.c_int32),
    ]


class DitConfig(C.Structure):
    """struct cm_dit_config (include/crowdmod_b200.h)."""

    _fields_ = [(k, C.c_int32) for k in (
        "in_channels", "out_channels", "rows", "cols", "past_len", "future_len", "t_patch", "patch", "hidden", "depth",
        "heads", "mlp_hidden", "time_multiple", "table_steps", "t_max_slots")]


class ChainArgs(C.Structure):
    """struct cm_chain_args (include/crowdmod_b200.h)."""

    _fields_ = [
        ("past", C.c_void_p),
        ("x", C.c_void_p),
        ("n", C.c_int32),
        ("nsteps", C.c_int32),
        ("tsteps", C.c_void_p),
        ("coef", C.c_void_p),
        ("mode", C.c_int32),
        ("noise", C.c_void_p),
        ("seed", C.c_uint64),
        ("sample_offset", C.c_int64),
        ("history", C.c_void_p),
        ("use_graph", C.c_int32),
    ]


# name -> (restype, argtypes); must list EVERY function include/crowdmod_b200.h declares
# (tests/test_abi.py checks the two against each other).
SIGNATURES = {
    "cm_version": (C.c_int, []),
    "cm_last_error": (C.c_char_p, []),
    "cm_device_error": (C.c_int, []),
    "cm_unet_create": (C.c_int, [C.POINTER(UNetConfig), C.POINTER(C.c_void_p)]),
    "cm_unet_destroy": (C.c_int, [C.c_void_p]),
    "cm_unet_param_count": (C.c_int, [C.c_void_p]),
    "cm_unet_param_info": (C.c_int, [C.c_void_p, C.c_int, C.c_char_p, C.c_int,
                                     C.POINTER(C.c_int64), C.POINTER(C.c_int)]),
    "cm_unet_set_param": (C.c_int, [C.c_void_p, C.c_char_p, C.c_void_p, C.c_int64]),
    "cm_unet_bind_params": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p), C.c_int]),
    "cm_unet_pack": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p]),
    "cm_unet_reserve": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_int64)]),
    "cm_unet_forward": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                  C.c_int, C.c_void_p]),
    "cm_unet_launches_per_forward": (C.c_int, [C.c_void_p]),
    "cm_unet_flops_per_sample": (C.c_double, [C.c_void_p]),
    "cm_unet_op_count": (C.c_int, [C.c_void_p]),
    "cm_unet_op_info": (C.c_int, [C.c_void_p, C.c_int, C.c_char_p, C.c_int, C.POINTER(C.c_int),
                                  C.POINTER(C.c_double)]),
    "cm_unet_debug_op_tensor": (C.c_int, [C.c_void_p, C.c_int]),
    "cm_unet_debug_tensor_read": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int64,
                                            C.POINTER(C.c_int), C.POINTER(C.c_int), C.c_void_p]),
    "cm_unet_op_exec_flops": (C.c_double, [C.c_void_p, C.c_int]),
    "cm_unet_profile_forward": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                          C.c_int, C.c_void_p, C.POINTER(C.c_float), C.c_int]),
    "cm_ddpm_sample": (C.c_int, [C.c_void_p, C.POINTER(ChainArgs), C.c_void_p]),
    "cm_last_chain_launches": (C.c_int64, [C.c_void_p]),
    "cm_last_chain_graph_launches": (C.c_int64, [C.c_void_p]),
    "cm_last_chain_graph_rebuilt": (C.c_int, [C.c_void_p]),
    "cm_unet_grad_layout": (C.c_int, [C.c_void_p, C.POINTER(C.c_int64), C.c_int, C.POINTER(C.c_int64)]),
    "cm_unet_dropout_layout": (C.c_int, [C.c_void_p, C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.c_int,
                                         C.POINTER(C.c_int32)]),
    "cm_unet_train_forward": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                        C.c_int, C.c_void_p, C.c_void_p]),
    "cm_unet_backward": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "cm_last_backward_launches": (C.c_int64, [C.c_void_p]),
    "cm_op_conv3d_dgrad": (C.c_int, [C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                     C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "cm_op_conv3d_dgrad_f32": (C.c_int, [C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                         C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "cm_op_conv3d_wgrad": (C.c_int, [C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                     C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p,
                                     C.c_int, C.c_void_p]),
    "cm_op_conv3d": (C.c_int, [C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                               C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int,
                               C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    "cm_op_gn_silu": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p,
                                C.c_int, C.c_int, C.c_float, C.c_int, C.c_void_p, C.c_void_p,
                                C.c_void_p]),
    "cm_op_attn_core": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int,
                                  C.c_void_p]),
    "cm_op_attn_core_backward": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int,
                                           C.c_void_p]),
    "cm_op_attn_block": (C.c_int, [C.c_void_p] * 9 + [C.c_int, C.c_int, C.c_int, C.c_int, C.c_float, C.c_void_p]),
    "cm_op_first_conv": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                   C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                   C.c_void_p]),
    "cm_op_final_conv": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int,
                                   C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                   C.c_void_p]),
    "cm_op_gn_backward": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int] + [C.c_void_p] * 6
                          + [C.c_int] * 4 + [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p,
                                             C.c_int, C.c_void_p]),
    "cm_op_cast_colsum": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p,
                                    C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "cm_op_rowsum_all": (C.c_int, [C.c_void_p, C.POINTER(C.c_int64), C.c_int, C.c_int, C.c_void_p, C.c_void_p]),
    "cm_op_final_conv_backward": (C.c_int, [C.c_void_p, C.c_float, C.c_void_p, C.c_int, C.c_int] + [C.c_void_p] * 4
                                  + [C.c_int] * 7 + [C.c_void_p, C.c_void_p]),
    "cm_op_first_conv_wgrad": (C.c_int, [C.c_void_p] * 5 + [C.c_int] * 7 + [C.c_void_p]),
    "cm_op_temb_backward": (C.c_int, [C.c_void_p] * 4 + [C.c_int] * 4
                            + [C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.c_int,
                               C.c_void_p, C.POINTER(C.c_int64), C.POINTER(C.c_int64)] + [C.c_void_p] * 7),
    "cm_op_loss_scale": (C.c_int, [C.c_void_p, C.c_int64, C.c_float, C.c_void_p, C.c_void_p]),
    "cm_dit_create": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p)]),
    "cm_dit_destroy": (C.c_int, [C.c_void_p]),
    "cm_dit_param_count": (C.c_int, [C.c_void_p]),
    "cm_dit_param_info": (C.c_int, [C.c_void_p, C.c_int, C.c_char_p, C.c_int, C.POINTER(C.c_int64), C.POINTER(C.c_int)]),
    "cm_dit_bind_params": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p), C.c_int]),
    "cm_dit_pack": (C.c_int, [C.c_void_p, C.c_void_p]),
    "cm_dit_forward": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    "cm_dit_sample": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "cm_dit_flops_per_sample": (C.c_double, [C.c_void_p]),
    "cm_dit_last_launches": (C.c_int64, [C.c_void_p]),
    "cm_window_gather": (C.c_int, [C.c_void_p, C.c_int64, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p,
                                   C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "cm_metrics_reduce": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p,
                                    C.c_void_p]),
}
CM_METRICS_PER_FRAME = 21

_lib = None


class NativeError(RuntimeError):
    pass


def lib() -> C.CDLL:
    """Load the shared library (once).  Raises if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise NativeError(
                f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; "
                "g.build()'` (there is no CPU or PyTorch fallback for the hot path)")
        l = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(l, name)
            fn.restype = res
            fn.argtypes = args
        _lib = l
    return _lib


def check(rc: int) -> None:
    if rc != 0:
        msg = lib().cm_last_error()
        raise NativeError(f"crowdmod_b200 error {rc}: {msg.decode() if msg else '?'}")


DEVICE_ERRORS = {
    301: "a loss-scaled fp16 gradient operand saturated (the value was clamped): the gradients of that step are "
         "not trustworthy",
}


def check_device_error(where: str = "") -> None:
    """Reads and clears the device-side error flag (synchronises) and raises on a non-zero code.  Kernels
    never hang or trap on a protocol error (bounded mbarrier waits) or on a saturated gradient: they set the
    flag and carry on, so the production loops poll it -- once per epoch in training, once per chain in
    sampling -- instead of silently stepping on corrupt data."""
    code = lib().cm_device_error()
    if code != 0:
        what = DEVICE_ERRORS.get(code, "a kernel pipeline wait timed out: partial outputs" if code > 0
                                 else "the device could not be queried")
        raise NativeError(f"crowdmod_b200 device error {code}{' in ' + where if where else ''}: {what}")


def ptr(t):
    """Device/host pointer of a torch tensor (or None)."""
    return None if t is None else C.c_void_p(t.data_ptr())


def current_stream():
    import torch
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)
