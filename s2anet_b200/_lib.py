"""ctypes binding of libs2a_b200.so (the C ABI declared in include/s2a_b200.h).

There is NO fallback: if the library is missing this module raises at first use, and every op
refuses CPU tensors.  torch is used only for device memory, streams and dtype bookkeeping.
"""
import ctypes as C
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "csrc", "libs2a_b200.so")

S2A_F32, S2A_BF16, S2A_F16 = 0, 1, 2
S2A_IOU_NO_REJECT = 1
_DTYPES = {torch.float32: S2A_F32, torch.bfloat16: S2A_BF16, torch.float16: S2A_F16}

_vp, _i64, _i32, _f32, _f64, _sz = C.c_void_p, C.c_int64, C.c_int, C.c_float, C.c_double, C.c_size_t

# name -> (restype, argtypes); must list every symbol include/s2a_b200.h declares
PROTOTYPES = {
    "s2a_version": (_i32, []),
    "s2a_last_error": (C.c_char_p, []),
    "s2a_measure_fp32_fma_tflops": (_i32, [_vp, _i32, _vp]),
    "s2a_transpose_planes": (_i32, [_vp, _vp, _i64, _i64, _i64, _i32, _vp]),
    "s2a_box_iou_rotated": (_i32, [_vp, _i64, _vp, _i64, _i64, _vp, _i64, _i64, _i64, _i32, _vp]),
    "s2a_box_iou_rotated_tiles": (_i32, [_vp, _i64, _vp, _i64, _i64, _vp, _i64, _i64, _i32, _i32, _i32, _i32, _i32, _vp]),
    "s2a_nms_rotated_workspace_bytes": (_sz, [_i64]),
    "s2a_nms_rotated": (_i32, [_vp, _i64, _vp, _i64, _vp, _i64, _f32, _vp, _vp, _vp, _sz, _vp]),
    "s2a_multiclass_nms_rotated_workspace_bytes": (_sz, [_i64, _i64, _i64]),
    "s2a_multiclass_nms_rotated": (_i32, [_vp, _vp, _i64, _i64, _i64, _f32, _f32, _i64, _vp, _vp, _vp, _i64, _vp,
                                          _sz, _vp]),
    "s2a_multiclass_nms_rotated_packed": (_i32, [_vp, _vp, _i64, _i64, _i64, _f32, _f32, _i64, _vp, _i32, _i64, _i64, _vp, _sz,
                                                 _vp]),
    "s2a_arf_forward": (_i32, [_vp, _vp, _vp] + [_i32] * 7 + [_vp]),
    "s2a_arf_backward": (_i32, [_vp, _vp, _vp] + [_i32] * 7 + [_vp]),
    "s2a_ri_pool_forward": (_i32, [_vp, _vp, _i64, _i64, _i64, _i32, _i32, _vp]),
    "s2a_deform_conv_forward_f32": (_i32, [_vp, _vp, _vp, _vp] + [_i32] * 16 + [_vp]),
    "s2a_alignconv_forward_f32": (_i32, [_vp, _vp, _vp, _vp] + [_i32] * 5 + [_f32, _vp]),
    "s2a_orconv_forward_f32": (_i32, [_vp, _vp, _vp, _vp, _vp, _vp] + [_i32] * 7 + [_vp]),
    "s2a_conv_pack_weight": (_i32, [_vp, _i32, _vp, _vp, _i32, _i32, _i32, _i32, _i32, _vp]),
    "s2a_alignconv_forward_tc": (_i32, [_vp, _vp, _vp, _vp] + [_i32] * 5 + [_f32, _i32, _vp]),
    "s2a_deform_conv_forward_tc": (_i32, [_vp, _vp, _i32, _vp, _vp] + [_i32] * 8 + [_vp]),
    "s2a_deform_conv_dgrad_tc": (_i32, [_vp, _vp, _i32, _vp, _vp, _vp, _vp] + [_i32] * 6 + [_vp]),
    "s2a_deform_conv_wgrad_tc": (_i32, [_vp, _vp, _i32, _vp, _vp] + [_i32] * 6 + [_vp]),
    "s2a_conv_pack_weight_tf32": (_i32, [_vp, _vp, _vp, _vp, _i32, _i32, _i32, _i32, _vp]),
    "s2a_conv_forward_tf32x3": (_i32, [_vp, _vp, _i32, _vp, _vp, _vp, _vp, _vp] + [_i32] * 5 + [_f32, _i32, _vp]),
    "s2a_orconv_forward_tc": (_i32, [_vp, _vp, _vp, _vp, _vp] + [_i32] * 6 + [_vp]),
    "s2a_alignconv_forward_tc_multi": (_i32, [_i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp] + [_i32] * 4 + [_vp]),
    "s2a_orconv_forward_tc_multi": (_i32, [_i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp] + [_i32] * 4 + [_vp]),
    "s2a_conv2d_pack_weight": (_i32, [_vp, _i32, _vp, _i32, _i32, _i32, _i32, _vp]),
    "s2a_conv2d_forward_tc_multi": (_i32, [_i32, _vp, _vp, _vp, _vp, _vp, _vp] + [_i32] * 6 + [_vp]),
    "s2a_conv2d_forward_tc_multi2": (_i32, [_i32, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp] + [_i32] * 6 + [_vp]),
    "s2a_conv2d_forward_tc_fam_decode": (_i32, [_i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp] + [_i32] * 3 +
                                         [_f32, _f32, _f64, _i32, _vp]),
    "s2a_deform_im2col_f32": (_i32, [_vp, _vp, _vp] + [_i32] * 13 + [_vp]),
    "s2a_deform_col2im_f32": (_i32, [_vp, _vp, _vp, _vp, _vp] + [_i32] * 13 + [_vp]),
    "s2a_assign_labels_workspace_bytes": (_sz, [_i64, _i64, _i64]),
    "s2a_assign_labels": (_i32, [_vp, _vp, _vp, _i64, _i64, _i64, _f32, _f32, _f32, _f32, _f32, _i32, _i32, _vp, _vp, _sz, _vp]),
    "s2a_poly_nms_workspace_bytes": (_sz, [_i64]),
    "s2a_poly_nms": (_i32, [_vp, _i64, _i64, _f64, _vp, _vp, _vp, _sz, _vp]),
    "s2a_poly_iou_pairs": (_i32, [_vp, _vp, _i64, _vp, _vp]),
    "s2a_fam_decode": (_i32, [_i32, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _f32, _f32, _f64, _i32, _vp]),
    "s2a_select_decode_workspace_bytes": (_sz, [_i32, _vp, _vp, _i32]),
    "s2a_select_decode": (_i32, [_i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i32, _i32, _i32, _f64, _i32, _vp, _vp, _vp,
                                 _i64, _vp, _sz, _vp]),
}

_lib = None


def load():
    """Load the shared library (once).  Raises RuntimeError if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                "libs2a_b200.so is missing (%s). Build it with `python -m s2anet_b200.build`; "
                "s2anet_b200 has no CPU or PyTorch fallback." % LIB_PATH)
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in PROTOTYPES.items():
            fn = getattr(lib, name)
            fn.restype, fn.argtypes = res, args
        _lib = lib
    return _lib


# kernels of THIS library launched by one successful C call (library sorts inside are not counted)
KERNELS_PER_CALL = {
    "transpose_planes": 1, "box_iou_rotated": 1, "box_iou_rotated_batched": 1, "box_iou_rotated_tiles": 1, "nms_rotated": 4, "multiclass_nms_rotated": 6, "multiclass_nms_rotated_packed": 6,
    "arf_forward": 1, "arf_backward": 1, "ri_pool": 1, "deform_conv_forward_cuda": 1, "alignconv_forward": 1,
    "orconv_forward": 1, "conv_pack_weight": 1, "alignconv_forward_tc": 1, "orconv_forward_tc": 1, "deform_conv_forward_tc": 1, "deform_conv_dgrad_tc": 9, "deform_conv_wgrad_tc": 1, "conv_pack_weight_tf32": 1, "conv_forward_tf32x3": 1,
    "alignconv_forward_tc_multi": 1, "orconv_forward_tc_multi": 1, "fam_decode": 1, "select_decode": 3, "conv2d_pack_weight": 1,
    "conv2d_forward_tc_multi": 1, "conv2d_forward_tc_multi2": 1, "conv2d_forward_tc_fam_decode": 1,
    "assign_labels": 2, "deform_im2col": 1, "deform_col2im": 1,
    "poly_nms": 4, "poly_iou_pairs": 1,
}
launches = 0          # running count, read by bench.py for "gpu_launches"


def check(rc, what):
    global launches
    launches += KERNELS_PER_CALL.get(what, 0)
    if rc != 0:
        msg = load().s2a_last_error().decode("utf-8", "replace")
        raise RuntimeError("%s failed (status %d): %s" % (what, rc, msg))


def ptr(t):
    return None if t is None else C.c_void_p(t.data_ptr())


def stream_ptr(device):
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def dtype_code(t):
    try:
        return _DTYPES[t.dtype]
    except KeyError:
        raise TypeError("unsupported dtype %s (float32, bfloat16, float16 only)" % t.dtype)


def require_cuda(*tensors):
    dev = None
    for t in tensors:
        if t is None:
            continue
        if not t.is_cuda:
            raise NotImplementedError("s2anet_b200 ops are CUDA (sm_100a) only; got a %s tensor" % t.device.type)
        if dev is None:
            dev = t.device
        elif t.device != dev:
            raise RuntimeError("all tensors must be on the same CUDA device (%s vs %s)" % (dev, t.device))
    return dev
