"""ctypes binding of libstep_b200.so (the C ABI declared in include/step_b200.h).

PyTorch only supplies device memory and the current CUDA stream; every compute call below goes
through the C ABI.  There is no fallback: if the library is missing or a tensor is not on a CUDA
device the call raises (north_star: "no CPU fallback").
"""
import ctypes
import os

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libstep_b200.so")

F32, F16 = 0, 1
EXT_NONE, EXT_PREDICT, EXT_EXTRAPOLATE, EXT_MEAN = 0, 1, 2, 3
A_AUTO, A_LINEAR, A_BOX, A_IM2COL, A_HALO, A_BEST, A_SIMT = 0, 1, 2, 3, 4, 5, 9

_lib = None

c_int, c_float, c_void_p, c_size_t = ctypes.c_int, ctypes.c_float, ctypes.c_void_p, ctypes.c_size_t


class ConvParams(ctypes.Structure):
    """mirror of step_conv_params (include/step_b200.h)"""
    _fields_ = [(n, c_int) for n in
                ("dtype", "N", "T", "H", "W", "Cin", "in_ld", "Cout", "out_ld", "out_coff", "KT", "KH", "KW",
                 "ST", "SH", "SW", "PT", "PH", "PW", "OT", "OH", "OW", "relu", "w_ld")] + \
               [("x", c_void_p), ("w", c_void_p), ("scale", c_void_p), ("shift", c_void_p),
                ("residual", c_void_p), ("res_ld", c_int), ("res_coff", c_int), ("y", c_void_p),
                ("a_mode", c_int), ("n_splits", c_int), ("split", c_int * 2), ("y_extra", c_void_p * 2),
                ("ld_extra", c_int * 2), ("coff_extra", c_int * 2), ("zero_cin_last_kt", c_int)]


def _declare(lib):
    P, I, Fl, S = c_void_p, c_int, c_float, c_void_p  # S = stream
    sigs = {
        "step_version": ([], c_int),
        "step_last_error": ([], ctypes.c_char_p),
        "step_launch_count": ([], ctypes.c_uint64),
        "step_nms_workspace_bytes": ([I], c_size_t),
        "step_nms_f32": ([P, P, I, Fl, I, P, P, P, c_size_t, S], c_int),
        "step_nms_segmented_f32": ([P, P, P, I, Fl, I, Fl, P, S], c_int),
        "step_nms_segmented_max_rows": ([], c_int),
        "step_detect_f32": ([P, I, P, I, P, I, I, I, I, Fl, Fl, I, Fl, Fl, Fl, Fl, I, I, P, P, P, P, P, S], c_int),
        "step_roi_align_fwd_nchw_f32": ([P, I, I, I, I, P, I, Fl, I, I, I, P, S], c_int),
        "step_roi_align_bwd_nchw_f32": ([P, P, I, Fl, I, I, I, I, I, I, I, P, S], c_int),
        "step_roi_pool_fwd_nchw_f32": ([P, I, I, I, I, P, I, Fl, I, I, P, P, S], c_int),
        "step_roi_pool_bwd_nchw_f32": ([P, P, P, I, I, I, I, I, I, I, P, S], c_int),
        "step_roi_align_fwd_nhwc": ([P, I, I, I, I, I, I, P, I, Fl, I, I, I, P, I, I, I, I, I, S], c_int),
        "step_roi_pool_fwd_nhwc": ([P, I, I, I, I, I, I, P, I, Fl, I, I, P, I, I, I, I, S], c_int),
        "step_tube_decode_f32": ([P, I, P, I, P, S], c_int),
        "step_tube_encode_f32": ([P, P, I, I, P, S], c_int),
        "step_tube_valid_f32": ([P, I, Fl, Fl, S], c_int),
        "step_tube_extrapolate_f32": ([P, I, I, I, Fl, Fl, P, S], c_int),
        "step_tube_extend_f32": ([P, I, Fl, Fl, Fl, P, S], c_int),
        "step_tube_update_f32": ([P, P, P, P, P, I, I, I, I, I, Fl, Fl, P, P, P, P, S], c_int),
        "step_clip_to_ndhwc": ([P, I, I, I, I, I, P, I, I, S], c_int),
        "step_clip_to_s2d_f16": ([P, I, I, I, I, I, P, I, S], c_int),
        "step_frames_to_clip_f32": ([P, P, I, I, I, I, I, I, I, Fl, Fl, Fl, Fl, Fl, Fl, P, S], c_int),
        "step_frames_to_s2d_f16": ([P, P, I, I, I, I, I, I, I, Fl, Fl, Fl, Fl, Fl, Fl, P, S], c_int),
        "step_nhwc_to_nchw_f32": ([P, I, I, I, I, I, P, S], c_int),
        "step_nchw_to_nhwc": ([P, I, I, I, P, I, I, S], c_int),
        "step_conv3d_fwd": ([ctypes.POINTER(ConvParams), S], c_int),
        "step_maxpool3d_fwd": ([P, I] + [I] * 21 + [P, I, S], c_int),
        "step_mean_mid": ([P, I, I, I, I, I, I, P, I, S], c_int),
        "step_linear_small_n_workspace_bytes": ([I, I, I], c_size_t),
        "step_linear_small_n": ([P, I, I, I, I, P, P, I, P, I, I, I, P, P, c_size_t, S], c_int),
        "step_head_regress": ([P, I, I, I, I, I, P, P, I, I, I, I, P, P, P, P, c_size_t, S], c_int),
        "step_bottleneck_exit_f16": ([P, ctypes.c_longlong, P, P, ctypes.c_longlong, P, P, I, P, ctypes.c_longlong, P, ctypes.c_longlong,
                                     ctypes.c_longlong, I, I, I, S], c_int),
        "step_head_losses_f32": ([P, P, P, P, P, P, I, I, I, I, I, Fl, Fl, P, P, P, P, P, P, P, P, P, S], c_int),
        "step_roi_align_bwd_nhwc": ([P, I, I, P, I, Fl, I, I, I, I, I, I, I, P, I, S], c_int),
        "step_linear_small_n_bwd": ([P, I, I, I, I, P, P, I, P, I, P, P, S], c_int),
        "step_conv1x1_wgrad_workspace_bytes": ([I, I, I], c_size_t),
        "step_conv1x1_wgrad_f16": ([P, I, P, I, I, I, I, Fl, P, I, I, P, c_size_t, S], c_int),
        "step_conv_wgrad_workspace_bytes": ([I, I, I, I], c_size_t),
        "step_conv_wgrad_f16": ([P, I, P, I, I, I, I, I, I, I, I, I, I, I, I, I, Fl, P, I, I, P, c_size_t, S], c_int),
        "step_act_bwd_f16": ([P, I, P, I, P, I, ctypes.c_longlong, I, P, I, P, I, S], c_int),
        "step_colsum_f16": ([P, I, ctypes.c_longlong, I, Fl, P, P, S], c_int),
        "step_mean_mid_bwd": ([P, I, I, I, I, Fl, P, I, S], c_int),
        "step_f32_accum_f16": ([P, ctypes.c_longlong, I, Fl, P, I, S], c_int),
        "step_maxpool3d_bwd_f16": ([P, I, P, I] + [I] * 20 + [P, I, P, S], c_int),
        "step_debug_tma_tile": ([ctypes.POINTER(ConvParams), I, I, I, I, I, P, P, P, S], c_int),
    }
    for name, (argtypes, restype) in sigs.items():
        fn = getattr(lib, name)  # AttributeError here == header / library mismatch
        fn.argtypes = argtypes
        fn.restype = restype
    return sigs


def lib():
    """Load (once) and return the shared library.  Raises if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError("step_b200: %s not found -- run `python -m step_b200.build` (there is no "
                               "CPU / PyTorch fallback for the hot path)" % LIB_PATH)
        l = ctypes.CDLL(LIB_PATH)
        _declare(l)
        _lib = l
    return _lib


def exported_symbols():
    return sorted(_declare(lib()).keys())


def check(rc):
    if rc != 0:
        raise RuntimeError("step_b200 [%d]: %s" % (rc, lib().step_last_error().decode("utf-8", "replace")))


def stream(device=None):
    """The launch stream: torch's current stream of `device` (default: the current device).  Callers working on
    tensors of another GPU wrap their launches in `torch.cuda.device(dev)` (kernels must run on the device that owns
    their pointers; test.py:85-87 places det_net i on cuda:(i+1) % gpu_count)."""
    return c_void_p(torch.cuda.current_stream(device).cuda_stream)


def same_device(*tensors):
    """All CUDA tensors of one launch must live on one device; returns it."""
    dev = None
    for t in tensors:
        if t is None:
            continue
        need_cuda(t)
        if dev is None:
            dev = t.device
        elif t.device != dev:
            raise RuntimeError("step_b200: tensors of one launch on different devices (%s vs %s)" % (dev, t.device))
    return dev


def ptr(t):
    return c_void_p(t.data_ptr()) if t is not None else c_void_p(0)


def need_cuda(*tensors):
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise RuntimeError("step_b200: expected a CUDA tensor (no CPU fallback on the hot path), got device %s"
                               % t.device)


def dt(t):
    if t.dtype == torch.float32:
        return F32
    if t.dtype == torch.float16:
        return F16
    raise RuntimeError("step_b200: unsupported dtype %s (float32 / float16 only)" % t.dtype)


def launch_count():
    return int(lib().step_launch_count())
