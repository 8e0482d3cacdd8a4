"""ctypes binding of libepb.so (include/epb.h).  There is NO fallback: if the
library is missing or a call fails, the product path raises."""
import ctypes
import os

HERE = os.path.dirname(os.path.abspath(__file__))
# EPB_LIB_PATH: a probe build of the same library (tools/build_variant.py); never a fallback
LIB_PATH = os.environ.get("EPB_LIB_PATH") or os.path.join(HERE, "libepb.so")

EPB_MAX_TAPS = 64

c_int, c_i64, c_f, c_d, c_p = (ctypes.c_int, ctypes.c_int64, ctypes.c_float,
                               ctypes.c_double, ctypes.c_void_p)


class ConvGeom(ctypes.Structure):
    """epb_conv_geom (include/epb.h)."""
    _fields_ = [("N", c_int), ("Hi", c_int), ("Wi", c_int), ("Cin", c_int),
                ("Ho", c_int), ("Wo", c_int), ("Cout", c_int),
                ("Hp", c_int), ("Wp", c_int),
                ("os", c_int), ("ph", c_int), ("pw", c_int), ("is_", c_int),
                ("T", c_int),
                ("dh", c_int * EPB_MAX_TAPS), ("dw", c_int * EPB_MAX_TAPS),
                ("wt", c_int * EPB_MAX_TAPS), ("Tw", c_int),
                ("in_relu", c_int), ("accumulate", c_int), ("precision", c_int)]


_PROTOS = {
    "epb_version": (c_int, []),
    "epb_last_error": (ctypes.c_char_p, []),
    "epb_device_check": (c_int, []),
    "epb_conv_fprop": (c_int, [ctypes.POINTER(ConvGeom), c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p]),
    "epb_conv_wgrad": (c_int, [ctypes.POINTER(ConvGeom), c_p, c_p, c_p, c_p, c_p, c_p]),
    "epb_pack_weight": (c_int, [c_p, c_p, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_p]),
    "epb_pack_weight_batch": (c_int, [c_p, c_int, ctypes.c_longlong, c_p]),
    "epb_im2col": (c_int, [c_p, c_p] + [c_int] * 12 + [c_p]),
    "epb_nchw_to_nhwc": (c_int, [c_p, c_p, c_int, c_int, c_int, c_int, c_int, c_p]),
    "epb_nhwc_to_nchw": (c_int, [c_p, c_p, c_int, c_int, c_int, c_int, c_int, c_p]),
    "epb_channel_stats": (c_int, [c_p, c_i64, c_int, c_p, c_p]),
    "epb_bn_finalize": (c_int, [c_p, c_i64, c_int, c_p, c_p, c_f, c_f, c_p, c_p, c_p, c_p, c_p, c_p, c_p]),
    "epb_bn_eval_affine": (c_int, [c_int, c_p, c_p, c_p, c_p, c_f, c_p, c_p, c_p]),
    "epb_bn_act": (c_int, [c_p, c_p, c_p, c_p, c_p, c_p, c_int, c_p, c_i64, c_int, c_p]),
    "epb_bn_relu_maxpool": (c_int, [c_p, c_p, c_p, c_p, c_p, c_int, c_int, c_int, c_int, c_p]),
    "epb_maxpool_bwd": (c_int, [c_p, c_p, c_p, c_int, c_int, c_int, c_int, c_p]),
    "epb_bn_bwd_reduce": (c_int, [c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_int, c_i64, c_int, c_p, c_p]),
    "epb_bn_bwd_apply": (c_int, [c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_int, c_p, c_i64, c_int, c_p, c_p, c_p, c_p]),
    "epb_add_masked": (c_int, [c_p, c_p, c_p, c_p, c_i64, c_p]),
    "epb_avgpool": (c_int, [c_p, c_p, c_int, c_int, c_int, c_p]),
    "epb_avgpool_bwd": (c_int, [c_p, c_p, c_int, c_int, c_int, c_int, c_p]),
    "epb_colsum": (c_int, [c_p, c_i64, c_int, c_p, c_p]),
    "epb_softargmax_fwd": (c_int, [c_p, c_int, c_int, c_int, c_int, c_int, c_int, c_p, c_p, c_p]),
    "epb_softargmax_bwd": (c_int, [c_p, c_int, c_int, c_int, c_int, c_int, c_int, c_p, c_p, c_p, c_p, c_p]),
    "epb_jointloss_fwd_bwd": (c_int, [c_p, c_p, c_p, c_int, c_int, c_int, c_f, c_p, c_p, c_p]),
    "epb_heatmap_joint_loss": (c_int, [c_p, c_p, c_p, c_int, c_int, c_f, c_p, c_p, c_p, c_int, c_int, c_f, c_f,
                                       c_p, c_p, c_p, c_p]),
    "epb_argmax2d": (c_int, [c_p, c_int, c_int, c_int, c_p, c_p, c_p, c_p]),
    "epb_final_preds": (c_int, [c_p, c_int, c_int, c_int, c_int, c_p, c_p, c_int, c_p, c_p, c_p]),
    "epb_patch_to_image": (c_int, [c_p, c_p, c_int, c_int, c_d, c_d, c_d, c_p, c_p]),
    "epb_triangulate": (c_int, [c_p, c_p, c_int, c_p, c_p, c_int, c_int, c_int, c_d, c_p, c_p, c_p]),
    "epb_triangulate_nview": (c_int, [c_p, c_int, c_p, c_int, c_int, c_int, c_p, c_p, c_p]),
    "epb_project_labels": (c_int, [c_p, c_p, c_p, c_int, c_int, c_d, c_d, c_d, c_p, c_p, c_p]),
    "epb_h36m_eval": (c_int, [c_p, c_p, c_p, c_int, c_int, c_int, ctypes.c_uint32, c_d, c_p, c_p, c_p, c_p, c_p]),
    "epb_add3": (c_int, [c_p, c_p, c_p, c_p, c_i64, c_p]),
    "epb_mask_scale": (c_int, [c_p, c_p, c_f, c_p, c_i64, c_p]),
    "epb_patch_sample": (c_int, [c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_int, c_int, c_int, c_p, c_p, c_p]),
    "epb_patch_sample_occ": (c_int, [c_p] * 7 + [c_int, c_int, c_int] + [c_p] * 5 + [c_p]),
    "epb_patch_joints": (c_int, [c_p, c_p, c_p, c_int, c_int, c_d, c_d, c_d, c_int, c_p, c_p]),
    "epb_bn_finalize_scale": (c_int, [c_p, c_i64, c_int, c_p, c_p, c_f, c_f] + [c_p] * 12),
    "epb_softargmax_bwd_split": (c_int, [c_p] + [c_int] * 5 + [c_p] * 6 + [c_int, c_p]),
    "epb_act_scale": (c_int, [c_p, c_p, c_p, c_i64, c_int, c_p, c_p, c_p, c_p, c_p, c_p]),
    # split-fp16 family: the int before the stream is the plane count (1 or 2)
    "epb_bn_act_split": (c_int, [c_p] * 8 + [c_int, c_i64, c_int, c_p, c_p, c_p, c_int, c_p]),
    "epb_bn_relu_maxpool_split": (c_int, [c_p] * 6 + [c_int] * 5 + [c_p]),
    "epb_im2col_split": (c_int, [c_p] * 3 + [c_int] * 12 + [c_p]),
    "epb_split16": (c_int, [c_p, ctypes.c_longlong, c_p, c_p, c_p, c_int, c_p]),
    "epb_split16_batch": (c_int, [c_p, c_int, ctypes.c_longlong, c_p, c_int, c_p]),
    "epb_conv16_fprop": (c_int, [ctypes.POINTER(ConvGeom)] + [c_p] * 7 + [c_int, c_p]),
    "epb_conv16_wgrad": (c_int, [ctypes.POINTER(ConvGeom)] + [c_p] * 6 + [ctypes.c_longlong, c_int, c_p]),
    "epb_bn_bwd_reduce_mx": (c_int, [c_p] * 7 + [c_int, c_i64, c_int, c_p, c_p, c_p]),
    "epb_bn_bwd_apply_split": (c_int, [c_p] * 8 + [c_int, c_p, c_p, c_i64, c_int] + [c_p] * 5 + [c_int, c_p]),
    "epb_bn_bwd_split": (c_int, [c_p] * 9 + [c_int, c_i64, c_int] + [c_p] * 5 + [c_int, c_p]),
    "epb_debug_conv16_trace": (c_int, [c_p, c_int]),
    "epb_avgpool_split": (c_int, [c_p, c_p, c_p, c_int, c_int, c_int, c_int, c_p]),
    "epb_sumsq": (c_int, [c_p, c_i64, c_p, c_p]),
    "epb_clip_scale": (c_int, [c_p, c_i64, c_p, c_d, c_p]),
    "epb_adam_step": (c_int, [c_p, c_p, c_p, c_p, c_i64, c_f, c_f, c_f, c_f, c_f, c_int, c_f, c_p]),
    "epb_sgd_step": (c_int, [c_p, c_p, c_p, c_i64, c_f, c_f, c_f, c_int, c_int, c_f, c_p]),
    "epb_adam_step_dev": (c_int, [c_p, c_p, c_p, c_p, c_i64, c_p, c_p, c_p]),
    "epb_sgd_step_dev": (c_int, [c_p, c_p, c_p, c_i64, c_p, c_p, c_p]),
}

EXPORTS = tuple(_PROTOS)


class EpbError(RuntimeError):
    pass


_lib = None


def lib():
    """Load libepb.so (once).  Raises if it was not built -- no CPU fallback."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise EpbError("libepb.so not built (%s); run `python -c 'import __graft_entry__ as g; "
                           "g.build()'`. There is no CPU fallback." % LIB_PATH)
        L = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in _PROTOS.items():
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def check(rc):
    if rc != 0:
        raise EpbError("libepb call failed (%d): %s" % (rc, lib().epb_last_error().decode()))


def call(name, *args):
    check(getattr(lib(), name)(*args))
