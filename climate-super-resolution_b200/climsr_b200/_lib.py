"""ctypes binding of include/climsr_b200.h (the C-ABI drop-in boundary).  Fails loudly if the .so is missing."""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libclimsr_b200.so")

CSR_OK = 0
CSR_ERR_BAD_ARG = -1            # CsrStatus in include/climsr_b200.h
NUM_METRICS = 18
METRIC_KEYS = ("acc@0.1", "acc@0.25", "acc@0.5", "acc@0.75", "acc@1", "acc@01.25", "acc@1.5", "acc@2", "psnr", "ssim", "mae",
               "mse", "rmse", "mape", "smape", "r2", "l1_loss", "mse_loss")   # key names of core/task.py:318-334 (typo kept)


class CsrError(RuntimeError):
    pass


class NetDesc(C.Structure):
    _fields_ = [("in_channels", C.c_int32), ("out_channels", C.c_int32), ("nf", C.c_int32), ("nb", C.c_int32),
                ("gc", C.c_int32), ("scale", C.c_int32)]


class ConvDesc(C.Structure):
    _fields_ = [("n", C.c_int32), ("h", C.c_int32), ("w", C.c_int32), ("cin", C.c_int32), ("cout", C.c_int32),
                ("kh", C.c_int32), ("kw", C.c_int32), ("in_c", C.c_int32), ("in_coff", C.c_int32), ("out_c", C.c_int32),
                ("out_coff", C.c_int32), ("act", C.c_int32), ("out_mode", C.c_int32), ("in_up2", C.c_int32),
                ("transposed", C.c_int32), ("scale1", C.c_float), ("scale2", C.c_float),
                ("res1_c", C.c_int32), ("res1_coff", C.c_int32), ("res2_c", C.c_int32), ("res2_coff", C.c_int32),
                ("gate_c", C.c_int32), ("gate_coff", C.c_int32), ("gate_from", C.c_int32), ("gate_neg", C.c_float),
                ("act_slope", C.c_float)]


class View(C.Structure):
    """CsrView: the real outputs of a layer inside its (N, hs, ws, c) buffer - pixel (i, j) at (off + step*i, off + step*j)."""
    _fields_ = [("hs", C.c_int32), ("ws", C.c_int32), ("c", C.c_int32), ("off", C.c_int32), ("step", C.c_int32),
                ("hl", C.c_int32), ("wl", C.c_int32)]


class WgradDesc(C.Structure):
    _fields_ = [("n", C.c_int32), ("h", C.c_int32), ("w", C.c_int32), ("cin", C.c_int32), ("cout", C.c_int32),
                ("kh", C.c_int32), ("kw", C.c_int32), ("x_c", C.c_int32), ("x_coff", C.c_int32), ("g_c", C.c_int32),
                ("g_coff", C.c_int32), ("in_up2", C.c_int32), ("scale", C.c_float)]


def _load():
    if not os.path.exists(LIB_PATH):
        raise CsrError(f"{LIB_PATH} is missing: build it with `python climate-super-resolution_b200/build.py` "
                       "(no CPU fallback exists for this path)")
    L = C.CDLL(LIB_PATH)
    vp, i32, sz, f32 = C.c_void_p, C.c_int32, C.c_size_t, C.c_float
    nd, cd, wd = C.POINTER(NetDesc), C.POINTER(ConvDesc), C.POINTER(WgradDesc)
    sig = {
        "csr_abi_version": (C.c_int, []),
        "csr_last_error": (C.c_char_p, []),
        "csr_device_check": (C.c_int, []),
        "csr_set_option": (C.c_int, [i32, i32]),
        "csr_kernel_launch_count": (C.c_int64, []),
        "csr_has_experiments": (C.c_int, []),
        "csr_debug_set_trace": (C.c_int, [vp]),
        "csr_debug_set_timeline": (C.c_int, [vp, i32]),
        "csr_num_layers": (C.c_int, [nd]),
        "csr_layer_shape": (C.c_int, [nd, i32, C.POINTER(i32 * 4), C.c_char_p, sz]),
        "csr_packed_weight_bytes": (sz, [nd]),
        "csr_pack_weights": (C.c_int, [nd, C.POINTER(vp), C.POINTER(vp), vp, sz, vp]),
        "csr_workspace_bytes": (sz, [nd, i32, i32, i32]),
        "csr_plan_create": (C.c_int, [nd, i32, i32, i32, vp, sz, C.POINTER(vp)]),
        "csr_plan_forward": (C.c_int, [vp, vp, vp, vp, vp, vp, vp]),
        "csr_plan_num_launches": (C.c_int, [vp]),
        "csr_plan_destroy": (None, [vp]),
        "csr_train_workspace_bytes": (sz, [nd, i32, i32, i32]),
        "csr_train_plan_create": (C.c_int, [nd, i32, i32, i32, vp, sz, C.POINTER(vp)]),
        "csr_packed_weight_bytes_bwd": (sz, [nd]),
        "csr_pack_weights_bwd": (C.c_int, [nd, C.POINTER(vp), vp, sz, vp]),
        "csr_plan_backward": (C.c_int, [vp, vp, vp, C.POINTER(vp), C.POINTER(vp), vp]),
        "csr_plan_num_backward_ops": (C.c_int, [vp]),
        "csr_plan_buffer": (C.c_int, [vp, i32, i32, C.POINTER(sz), C.POINTER(i32 * 4)]),
        "csr_plan_grad_floats": (sz, [vp]),
        "csr_plan_graph_status": (C.c_int, [vp, i32]),
        "csr_plan_grad_offset": (C.c_int, [vp, i32, i32, C.POINTER(sz)]),
        "csr_plan_backward_flat": (C.c_int, [vp, vp, vp, vp, vp]),
        "csr_plan_backward_segments": (C.c_int, [vp, i32]),
        "csr_plan_backward_flat_seg": (C.c_int, [vp, vp, vp, vp, i32, C.POINTER(sz), C.POINTER(sz), vp]),
        "csr_generator_forward": (C.c_int, [nd, vp, vp, vp, vp, vp, vp, sz, i32, i32, i32, vp]),
        "csr_conv2d_scratch_bytes": (sz, [cd]),
        "csr_conv2d_nhwc": (C.c_int, [cd, vp, vp, vp, vp, vp, vp, vp, vp, sz, vp]),
        "csr_conv2d_pack": (C.c_int, [cd, vp, vp, vp, sz, vp]),
        "csr_conv2d_wgrad_scratch_bytes": (sz, [wd]),
        "csr_conv2d_wgrad": (C.c_int, [wd, vp, vp, vp, vp, vp, sz, vp]),
        "csr_nchw_f32_to_nhwc_bf16": (C.c_int, [vp, vp, i32, i32, i32, i32, i32, i32, vp]),
        "csr_nhwc_bf16_to_nchw_f32": (C.c_int, [vp, vp, i32, i32, i32, i32, i32, i32, vp]),
        "csr_nchw_f32_to_nhwc_split": (C.c_int, [vp, vp, i32, i32, i32, i32, i32, vp]),
        "csr_maxpool2x2_split": (C.c_int, [vp, vp, i32, i32, i32, i32, vp]),
        "csr_pixel_loss_scratch_bytes": (sz, [C.c_int64]),
        "csr_l1_loss": (C.c_int, [vp, vp, vp, C.c_int64, vp, vp, sz, vp]),
        "csr_mse_loss": (C.c_int, [vp, vp, vp, C.c_int64, vp, vp, sz, vp]),
        "csr_metrics_scratch_bytes": (sz, [i32, i32, i32]),
        "csr_masked_metrics": (C.c_int, [vp, vp, vp, vp, vp, vp, f32, f32, C.c_double, C.c_double, C.c_double, i32, i32, i32, vp, vp, sz, vp]),
        "csr_minmax_normalize": (C.c_int, [vp, i32, i32, i32, vp, vp, C.c_double, C.c_double, C.c_double, f32, vp, vp, vp, vp]),
        "csr_minmax_denormalize_mask": (C.c_int, [vp, vp, i32, i32, i32, i32, vp, vp, C.c_double, C.c_double, C.c_double, vp, vp]),
        "csr_disc_gather": (C.c_int, [vp, C.POINTER(View), i32, vp, i32, vp, vp, vp]),
        "csr_disc_collect": (C.c_int, [vp, C.POINTER(View), i32, i32, vp, f32, vp, vp]),
        "csr_disc_bn_scratch_bytes": (sz, [i32]),
        "csr_disc_bn_forward": (C.c_int, [vp, C.POINTER(View), i32, vp, vp, f32, f32, vp, vp, i32, vp, vp, vp, vp, vp, sz, vp]),
        "csr_disc_bn_backward": (C.c_int, [vp, C.POINTER(View), i32, i32, vp, f32, vp, vp, vp, vp, vp, sz, vp, vp, vp, vp]),
        "csr_disc_flatten": (C.c_int, [vp, C.POINTER(View), i32, vp, vp]),
        "csr_disc_unflatten": (C.c_int, [vp, C.POINTER(View), i32, vp, vp]),
        "csr_linear_forward": (C.c_int, [vp, vp, vp, vp, i32, i32, i32, vp]),
        "csr_linear_backward": (C.c_int, [vp, vp, vp, vp, vp, vp, i32, i32, i32, vp]),
        "csr_channel_attention": (C.c_int, [vp, vp, vp, vp, vp, vp, vp, vp, i32, i32, i32, i32, i32, vp]),
        "csr_channel_attention_backward_scratch_bytes": (sz, [i32, i32]),
        "csr_channel_attention_backward": (C.c_int, [vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, sz, i32, i32, i32, i32, i32, vp]),
        "csr_pixel_shuffle2": (C.c_int, [vp, vp, i32, i32, i32, i32, vp]),
        "csr_pixel_unshuffle2": (C.c_int, [vp, vp, i32, i32, i32, i32, vp]),
        "csr_grad_pack_bf16": (C.c_int, [vp, vp, sz, f32, vp]),
        "csr_grad_unpack_bf16": (C.c_int, [vp, vp, sz, f32, vp]),
        "csr_lr_input_from_hr": (C.c_int, [vp, vp, vp, i32, i32, i32, i32, vp, vp, vp, vp, vp, vp]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(L, name)
        fn.restype = res
        fn.argtypes = args
    return L


lib = _load()
EXPORTS = ("csr_abi_version", "csr_last_error", "csr_device_check", "csr_set_option", "csr_kernel_launch_count", "csr_has_experiments", "csr_debug_set_trace", "csr_debug_set_timeline", "csr_num_layers",
           "csr_layer_shape", "csr_packed_weight_bytes", "csr_pack_weights", "csr_workspace_bytes", "csr_plan_create",
           "csr_plan_forward", "csr_plan_num_launches", "csr_plan_destroy", "csr_train_workspace_bytes", "csr_train_plan_create",
           "csr_packed_weight_bytes_bwd", "csr_pack_weights_bwd", "csr_plan_backward", "csr_plan_num_backward_ops", "csr_plan_buffer", "csr_plan_grad_floats", "csr_plan_graph_status", "csr_plan_grad_offset",
           "csr_plan_backward_flat", "csr_plan_backward_segments", "csr_plan_backward_flat_seg", "csr_generator_forward", "csr_conv2d_scratch_bytes",
           "csr_conv2d_nhwc", "csr_conv2d_pack", "csr_conv2d_wgrad_scratch_bytes", "csr_conv2d_wgrad", "csr_nchw_f32_to_nhwc_bf16", "csr_nhwc_bf16_to_nchw_f32",
           "csr_nchw_f32_to_nhwc_split", "csr_maxpool2x2_split", "csr_pixel_loss_scratch_bytes", "csr_l1_loss", "csr_mse_loss",
           "csr_metrics_scratch_bytes", "csr_masked_metrics", "csr_minmax_normalize", "csr_minmax_denormalize_mask", "csr_disc_gather", "csr_disc_collect", "csr_disc_bn_scratch_bytes", "csr_disc_bn_forward",
           "csr_disc_bn_backward", "csr_disc_flatten", "csr_disc_unflatten", "csr_linear_forward", "csr_linear_backward",
           "csr_channel_attention", "csr_channel_attention_backward_scratch_bytes", "csr_channel_attention_backward", "csr_pixel_shuffle2",
           "csr_pixel_unshuffle2", "csr_grad_pack_bf16", "csr_grad_unpack_bf16", "csr_lr_input_from_hr")


def check(rc: int, what: str = "") -> None:
    if rc != CSR_OK:
        msg = lib.csr_last_error().decode("utf-8", "replace")
        raise CsrError(f"{what or 'climsr_b200'} failed (status {rc}): {msg}")


def device_check() -> None:
    """Raise unless an sm_100 (B200) device is current and usable."""
    check(lib.csr_device_check(), "csr_device_check")


def kernel_launch_count() -> int:
    return int(lib.csr_kernel_launch_count())


def current_stream_ptr() -> int:
    import torch
    return int(torch.cuda.current_stream().cuda_stream)
