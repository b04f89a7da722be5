"""ctypes binding of libfvfi.so (C-ABI declared in include/fvfi.h).

The reference hands raw ``tensor.data_ptr()`` values and torch's current stream to
CuPy-launched kernels (src/adacof/cupy_module/adacof.py:337-354); this module keeps that
convention.  The library is built in-tree by ../build.py; a missing library is a hard error
when an op is called -- there is no fallback path.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None

c_fp = ctypes.c_void_p
c_int = ctypes.c_int
c_size = ctypes.c_size_t


class FvfiError(RuntimeError):
    pass


def lib_path():
    return os.path.join(_HERE, "libfvfi.so")


_PROTOS = {
    "fvfi_version": (c_int, []),
    "fvfi_last_error": (ctypes.c_char_p, []),
    "fvfi_device_sm_count": (c_int, []),
    "fvfi_launch_count": (ctypes.c_ulonglong, []),
    "fvfi_adacof_forward": (c_int, [c_fp] * 5 + [c_int] * 9 + [c_fp]),
    "fvfi_adacof_backward": (c_int, [c_fp] * 9 + [c_int] * 10 + [c_fp]),
    "fvfi_adacofnet_tail": (c_int, [c_fp] * 11 + [c_int] * 5 + [c_fp]),
    "fvfi_adacofnet_warp_blend": (c_int, [c_fp] * 13 + [c_int] * 7 + [c_fp]),
    "fvfi_adacofnet_warp_blend_rows": (c_int, [c_fp] * 11 + [c_int] * 8 + [c_fp]),
    "fvfi_fusion_blend": (c_int, [c_fp] * 3 + [c_size, c_fp]),
    "fvfi_rgb2lab": (c_int, [c_fp, c_fp, c_int, c_int, c_int, c_fp]),
    "fvfi_lab2rgb": (c_int, [c_fp, c_fp, c_int, c_int, c_int, c_fp]),
    "fvfi_gaussian_filter": (c_int, [c_fp, c_fp, c_fp, c_int, c_int, c_int, ctypes.c_float, c_fp]),
    "fvfi_median_filter": (c_int, [c_fp, c_fp, c_int, c_int, c_int, c_int, c_fp]),
    "fvfi_conv2d_packed_weight_floats": (c_size, [c_int] * 5),
    "fvfi_conv2d_pack_weights": (c_int, [c_fp, c_fp, c_int, c_int, c_int, c_int, c_int, c_fp]),
    "fvfi_conv2d_nhwc": (c_int, [c_fp, c_int, c_fp, c_fp, c_fp, c_int] + [c_int] * 11 + [c_fp]),
    "fvfi_conv2d_nhwc_residual": (c_int, [c_fp, c_int, c_fp, c_fp, c_fp, c_int, c_fp, c_int] + [c_int] * 11 + [c_fp]),
    "fvfi_conv2d_nhwc_upsampled": (c_int, [c_fp, c_int, c_int, c_int, c_int, c_fp, c_int, c_int, c_fp, c_fp, c_fp, c_int, c_fp, c_int]
                                   + [c_int] * 11 + [c_fp]),
    "fvfi_conv2d_overflow_count": (c_int, []),
    "fvfi_conv2d_grad_act_workspace_floats": (c_size, [c_int] * 5),
    "fvfi_conv2d_grad_act": (c_int, [c_fp, c_int, c_fp, c_int, c_fp] + [c_int] * 6 + [c_fp, c_fp, c_fp]),
    "fvfi_reflect_pad_backward_nhwc": (c_int, [c_fp, c_int, c_fp, c_int] + [c_int] * 5 + [c_fp]),
    "fvfi_conv2d_wgrad_workspace_floats": (c_size, [c_int] * 6),
    "fvfi_conv2d_wgrad_nhwc": (c_int, [c_fp, c_int, c_fp, c_int, ctypes.c_longlong, ctypes.c_longlong, c_fp] + [c_int] * 7 + [c_fp, c_fp]),
    "fvfi_max_pool2_backward_nhwc": (c_int, [c_fp, c_int, c_fp, c_int, c_fp, c_int] + [c_int] * 4 + [c_fp]),
    "fvfi_avg_pool2_backward_nhwc": (c_int, [c_fp, c_int, c_fp, c_int] + [c_int] * 4 + [c_fp]),
    "fvfi_resize_bilinear_backward_nhwc": (c_int, [c_fp, c_int, c_fp, c_int, c_fp, c_int] + [c_int] * 8 + [c_fp]),
    "fvfi_fusion_blend_backward": (c_int, [c_fp] * 5 + [c_size, c_fp]),
    "fvfi_planar_concat_nhwc": (c_int, [c_fp, c_fp, c_int, c_fp, c_int, c_int, c_int, c_int, c_fp]),
    "fvfi_nchw_to_nhwc_slice": (c_int, [c_fp, c_fp, c_int, c_int, c_int, c_int, c_int, c_fp]),
    "fvfi_conv1x1_nhwc": (c_int, [c_fp, c_int, c_fp, c_fp, c_fp, c_int, c_size, c_int, c_int, c_int, c_fp]),
    "fvfi_upsample2_tapsum": (c_int, [c_fp, c_int, c_fp, c_fp, c_int, c_int, c_int, c_int, c_fp]),
    "fvfi_phasenet_assemble": (c_int, [c_fp, c_fp, c_fp, c_fp, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_fp]),
    "fvfi_phasenet_outputs": (c_int, [c_fp, c_int, c_fp, c_fp, c_fp, c_int, c_int, c_int, c_int, c_int, c_int, c_fp]),
    "fvfi_phasenet_assemble_offset": (c_int, [c_fp, c_fp, c_fp, c_fp] + [c_int] * 9 + [c_fp]),
    "fvfi_phasenet_outputs_offset": (c_int, [c_fp, c_int, c_fp, c_fp, c_fp] + [c_int] * 8 + [c_fp]),
    "fvfi_rgb8_to_rgb_lab": (c_int, [c_fp, c_fp, c_fp, c_int, c_int, c_int, c_fp]),
    "fvfi_fusion_blend_rgb8": (c_int, [c_fp, c_fp, c_fp, c_int, c_int, c_int, c_fp]),
    "fvfi_max_pool2_nhwc": (c_int, [c_fp, c_int, c_fp, c_int, c_int, c_int, c_int, c_int, c_fp]),
    "fvfi_adacofnet_prep": (c_int, [c_fp, c_fp, c_fp, c_fp, c_fp, c_int, c_int, c_int, c_int, c_int, c_int, c_fp, c_fp]),
    "fvfi_avg_pool2_nhwc": (c_int, [c_fp, c_int, c_fp, c_int, c_int, c_int, c_int, c_int, c_fp]),
    "fvfi_resize_bilinear_nhwc": (c_int, [c_fp, c_int, c_fp, c_int] + [c_int] * 7 + [c_fp]),
    "fvfi_resize_bilinear_nhwc_fused": (c_int, [c_fp, c_int, c_fp, c_int, c_fp, c_int] + [c_int] * 8 + [c_fp]),
    "fvfi_adacof_forward_host": (c_int, [c_fp] * 5 + [c_int] * 8),
    "fvfi_adacof_backward_host": (c_int, [c_fp] * 8 + [c_int] * 8),
    "fvfi_pyr_plan_create": (c_int, [c_int, c_int, c_int, c_int, ctypes.c_double, ctypes.POINTER(c_fp)]),
    "fvfi_pyr_plan_destroy": (None, [c_fp]),
    "fvfi_pyr_num_levels": (c_int, [c_fp]),
    "fvfi_pyr_level_shape": (c_int, [c_fp, c_int, ctypes.POINTER(c_int), ctypes.POINTER(c_int)]),
    "fvfi_pyr_next_size": (c_int, [c_int, ctypes.c_double]),
    "fvfi_pyr_workspace_bytes": (c_size, [c_fp, c_int]),
    "fvfi_pyr_decompose": (c_int, [c_fp, c_fp, c_int, c_fp, c_fp, c_fp, c_fp, c_fp, c_fp, c_fp]),
    "fvfi_pyr_reconstruct": (c_int, [c_fp, c_fp, c_fp, c_fp, c_fp, c_int, c_fp, c_fp, c_fp]),
    "fvfi_pyr_highband_filter": (c_int, [c_fp, c_fp, c_int, c_fp, c_fp, c_fp]),
    "fvfi_pyr_reconstruct_backward": (c_int, [c_fp, c_fp, c_int, c_fp, c_fp, c_fp, c_fp, c_fp, c_fp, c_fp, c_fp]),
    "fvfi_pyr_build_complex": (c_int, [c_fp, c_fp, c_int, c_fp, c_fp, c_fp, c_fp, c_fp]),
    "fvfi_pyr_reconstruct_complex": (c_int, [c_fp, c_fp, c_fp, c_fp, c_int, c_fp, c_fp, c_fp]),
}


def lib():
    """Load libfvfi.so (once).  Raises FvfiError if it has not been built."""
    global _LIB
    if _LIB is None:
        path = lib_path()
        if not os.path.exists(path):
            raise FvfiError(
                "libfvfi.so not found at %s -- build it with "
                "`python fusion-method-for-video-frame-interpolation_b200/build.py`; "
                "there is no CPU / PyTorch fallback for the hot path" % path)
        L = ctypes.CDLL(path)
        missing = []
        for name, (res, args) in _PROTOS.items():
            try:
                fn = getattr(L, name)
            except AttributeError:
                missing.append(name)
                continue
            fn.restype = res
            fn.argtypes = args
        if missing:
            raise FvfiError("libfvfi.so at %s is stale: missing symbols %s -- rebuild with build.py" % (path, missing))
        _LIB = L
    return _LIB


def check(rc):
    if rc != 0:
        raise FvfiError("libfvfi error %d: %s" % (rc, lib().fvfi_last_error().decode()))


def ptr(t):
    """data_ptr of a tensor or None -> NULL."""
    return None if t is None else t.data_ptr()


def stream_ptr():
    import torch
    return torch.cuda.current_stream().cuda_stream
