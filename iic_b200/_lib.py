"""ctypes binding of libiic_b200.so (include/iic_b200.h).

There is no CPU path and no fallback: if the library is missing, or a call
returns an error, this module raises.  `python -m iic_b200.build` (or
`__graft_entry__.build()`) compiles it with nvcc for sm_100a.
"""
import ctypes
import os
from ctypes import POINTER, Structure, c_char_p, c_double, c_float, c_int, c_longlong, c_void_p

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libiic_b200.so")

F32, BF16 = 0, 1
TF32, TF32X3 = 2, 3  # conv compute modes on F32 storage (include/iic_b200.h)
PHASE_FUSED, PHASE_PARTIAL, PHASE_FINISH = 0, 1, 2


class ConvGeom(Structure):
  _fields_ = [(n, c_int) for n in ("n", "h", "w", "cin", "oh", "ow", "cout", "kh", "kw", "stride", "pad", "dil")]


class PackJob(Structure):
  _fields_ = [("w", c_void_p), ("dst", c_void_p)] + [(n, c_int) for n in ("kind", "cout", "cin", "kh", "kw", "reserved")]


_P = c_void_p
_SIGS = {
  "iic_abi_version": (c_int, []),
  "iic_last_error": (c_char_p, []),
  "iic_launch_count": (c_longlong, [c_int]),
  "iic_get_option": (c_int, [c_char_p]),
  "iic_set_option": (c_int, [c_char_p, c_int]),
  "iic_iid_loss": (c_int, [_P, _P, c_int, c_int, c_int, c_float, c_double, _P, _P, _P, _P, _P, c_int, _P]),
  "iic_joint_mi": (c_int, [_P, c_int, c_int, c_float, c_double, c_int, _P, _P, _P]),
  "iic_seg_kp": (c_int, [c_int]),
  "iic_seg_prepare": (c_int, [_P, _P, _P, _P, _P, _P, c_int, c_int, c_int, c_int, _P]),
  "iic_seg_unprepare": (c_int, [_P, _P, _P, _P, _P, _P, c_int, c_int, c_int, c_int, _P]),
  "iic_seg_prepare_shift": (c_int, [_P, _P, _P, _P, _P, _P, c_int, c_int, c_int, c_int, c_int, c_int, _P]),
  "iic_seg_unprepare_shift": (c_int, [_P, _P, _P, _P, _P, _P, c_int, c_int, c_int, c_int, c_int, c_int, _P]),
  "iic_seg_joint_workspace": (c_longlong, [c_int, c_int, c_int]),
  "iic_seg_joint": (c_int, [_P, _P, _P, _P, c_int, c_int, c_int, c_int, c_int, _P]),
  "iic_seg_joint_tc_workspace": (c_longlong, [c_int, c_int, c_int, c_int, c_int]),
  "iic_seg_joint_tc": (c_int, [_P, _P, _P, _P, c_int, c_int, c_int, c_int, c_int, _P]),
  "iic_seg_corr_tc_workspace": (c_longlong, [c_int, c_int, c_int, c_int, c_int]),
  "iic_seg_corr_tc": (c_int, [_P, _P, _P, _P, c_int, c_int, c_int, c_int, c_int, c_int, c_float, _P]),
  "iic_seg_corr_bwd": (c_int, [_P, _P, _P, c_int, c_int, c_int, c_int, c_int, c_int, c_float, _P]),
  "iic_box_filter": (c_int, [_P, _P, _P, c_int, c_int, c_int, c_int, c_int, _P]),
  "iic_sobel": (c_int, [_P, _P, c_int, c_int, c_int, c_int, c_int, c_int, _P]),
  "iic_grey_sobel": (c_int, [_P, c_int, _P, c_int, c_int, c_int, _P]),
  "iic_nchw_to_nhwc": (c_int, [_P, _P, c_int, c_int, c_int, c_int, c_int, _P]),
  "iic_nhwc_to_nchw": (c_int, [_P, c_int, _P, c_int, c_int, c_int, c_int, _P]),
  "iic_cast": (c_int, [_P, c_int, _P, c_int, c_longlong, _P]),
  "iic_pack_weight": (c_int, [_P, _P, c_int, c_int, c_int, c_int, c_int, c_int, _P]),
  "iic_unpack_wgrad": (c_int, [_P, _P, c_int, c_int, c_int, c_int, c_int, _P]),
  "iic_conv_fprop": (c_int, [_P, _P, _P, POINTER(ConvGeom), c_int, _P]),
  "iic_conv_fprop_stats_blocks": (c_int, [POINTER(ConvGeom), c_int]),
  "iic_conv_fprop_stats": (c_int, [_P, _P, _P, POINTER(ConvGeom), c_int, c_int, _P, _P]),
  "iic_bn_stats_from_partials": (c_int, [_P, c_int, c_int, c_int, c_longlong, c_int, _P, _P, c_float, c_float, _P, _P, _P,
                                         _P, _P, _P]),
  "iic_conv_dgrad": (c_int, [_P, _P, _P, _P, POINTER(ConvGeom), c_int, _P]),
  "iic_conv_dgrad_masked": (c_int, [_P, _P, _P, _P, _P, POINTER(ConvGeom), c_int, _P]),
  "iic_conv_wgrad_workspace": (c_longlong, [POINTER(ConvGeom), c_int]),
  "iic_conv_wgrad": (c_int, [_P, _P, _P, _P, POINTER(ConvGeom), c_int, _P]),
  "iic_conv_wgrad_oihw_workspace": (c_longlong, [POINTER(ConvGeom), c_int]),
  "iic_conv_wgrad_oihw": (c_int, [_P, _P, _P, c_int, _P, POINTER(ConvGeom), c_int, _P]),
  "iic_stem_fprop": (c_int, [_P, _P, _P, POINTER(ConvGeom), c_int, _P]),
  "iic_stem_wgrad": (c_int, [_P, _P, _P, c_int, _P, c_longlong, POINTER(ConvGeom), c_int, _P]),
  "iic_stem_fprop_stats_tc_blocks": (c_int, [POINTER(ConvGeom), c_int]),
  "iic_stem_fprop_stats_tc": (c_int, [_P, _P, _P, POINTER(ConvGeom), c_int, _P, _P]),
  "iic_stem_wgrad_tc_workspace": (c_longlong, [POINTER(ConvGeom)]),
  "iic_stem_wgrad_tc": (c_int, [_P, _P, _P, c_int, _P, POINTER(ConvGeom), _P]),
  "iic_bn_stats": (c_int, [_P, c_int, c_longlong, c_int, _P, _P, c_float, c_float, _P, _P, c_int, _P, _P, _P, _P]),
  "iic_bn_apply": (c_int, [_P, _P, _P, _P, _P, c_int, c_longlong, c_int, c_int, _P]),
  "iic_bn_relu_maxpool": (c_int, [_P, _P, _P, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int, _P]),
  "iic_bn_relu_maxpool_bwd": (c_int, [_P, _P, _P, _P, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int, _P]),
  "iic_bn_bwd_reduce": (c_int, [_P, _P, _P, _P, _P, c_int, c_longlong, c_int, _P, _P]),
  "iic_bn_bwd_apply": (c_int, [_P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, c_int, c_int, c_longlong, c_int, _P]),
  "iic_bn_bwd_fused": (c_int, [_P, _P, _P, c_int, _P, _P, _P, _P, _P, _P, _P, _P, _P, c_int, c_int, c_longlong, c_int, _P]),
  "iic_bn_apply_views": (c_int, [_P, _P, _P, _P, _P, c_int, c_longlong, c_int, c_int, c_int, _P]),
  "iic_bn_apply_views_mask": (c_int, [_P, _P, _P, _P, _P, _P, c_int, c_longlong, c_int, c_int, _P]),
  "iic_bn_bwd_fused_bits": (c_int, [_P, _P, _P, c_int, _P, _P, _P, _P, _P, _P, _P, c_int, c_int, c_longlong, c_int, _P]),
  "iic_bn_stats_from_partials_views": (c_int, [_P, c_int, c_int, c_int, c_longlong, c_int, _P, _P, c_float, c_float, _P, _P, _P, _P, _P]),
  "iic_pack_weights_batched": (c_int, [_P, c_int, c_int, _P]),
  "iic_stem_bwd_fused_workspace": (c_longlong, [POINTER(ConvGeom), c_int, c_int, c_int]),
  "iic_stem_bwd_fused": (c_int, [_P, _P, _P, _P, _P, _P, _P, _P, c_int, _P, c_int, POINTER(ConvGeom), c_int, c_int, c_int, _P,
                                 c_longlong, _P]),
  "iic_stem_bwd_dy": (c_int, [_P, _P, _P, _P, _P, _P, _P, c_int, _P, POINTER(ConvGeom), c_int, c_int, c_int, _P, c_longlong, _P]),
  "iic_stem_fprop_stats_blocks": (c_int, [POINTER(ConvGeom), c_int, c_int]),
  "iic_stem_fprop_stats": (c_int, [_P, _P, _P, POINTER(ConvGeom), c_int, c_int, _P, _P]),
  "iic_argmax_rows": (c_int, [_P, c_longlong, c_int, _P, _P]),
  "iic_argmax_channels": (c_int, [_P, c_int, c_int, c_longlong, _P, _P]),
  "iic_confusion_counts": (c_int, [_P, _P, _P, c_int, c_longlong, c_int, c_int, _P, c_int, _P]),
  "iic_avgpool": (c_int, [_P, c_int, _P, c_int, c_int, c_int, _P]),
  "iic_avgpool_bwd": (c_int, [_P, _P, c_int, c_int, c_int, c_int, _P]),
  "iic_heads_fwd": (c_int, [_P, _P, _P, _P, _P, c_int, c_int, c_int, c_int, _P]),
  "iic_heads_bwd": (c_int, [_P, _P, _P, _P, _P, _P, _P, _P, c_int, c_int, c_int, c_int, _P]),
  "iic_cross_entropy": (c_int, [_P, _P, c_int, c_int, _P, _P, _P]),
  "iic_linear_fwd": (c_int, [_P, _P, _P, _P, c_int, c_int, c_int, _P]),
  "iic_linear_bwd": (c_int, [_P, _P, _P, _P, _P, _P, c_int, c_int, c_int, c_int, _P]),
  "iic_col_sum": (c_int, [_P, c_int, c_longlong, c_int, _P, c_int, _P]),
  "iic_seg_head_workspace":(c_longlong, [c_int, c_int, c_int, c_int, c_int]),
  "iic_seg_head_fwd": (c_int, [_P, c_int, _P, _P, _P, _P, c_int, c_int, c_int, c_int, c_int, c_int, c_int, _P]),
  "iic_seg_head_bwd": (c_int, [_P, c_int, _P, _P, _P, _P, _P, _P, _P, _P, c_int, c_int, c_int, c_int, c_int, c_int,
                               c_int, c_int, _P]),
  "iic_adam_step": (c_int, [POINTER(c_void_p), POINTER(c_longlong), c_int, c_float, c_float, c_float, c_float,
                            c_float, c_int, _P]),
  "iic_adam_step_dev": (c_int, [POINTER(c_void_p), POINTER(c_longlong), c_int, c_float, c_float, c_float, c_float,
                                c_float, _P, _P]),
}

_lib = None


def declared_symbols():
  return sorted(_SIGS)


def lib():
  """Loads the shared library once; raises (never falls back) if it is absent."""
  global _lib
  if _lib is None:
    if not os.path.exists(LIB_PATH):
      raise RuntimeError(
        "iic_b200: %s not found. The CUDA extension is mandatory (there is no CPU or PyTorch "
        "fallback); build it with `python -m iic_b200.build`." % LIB_PATH)
    l = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in _SIGS.items():
      fn = getattr(l, name)  # AttributeError if the library does not export a declared symbol
      fn.restype = res
      fn.argtypes = args
    _lib = l
  return _lib


class IICError(RuntimeError):
  pass


def check(rc, what=""):
  if rc != 0:
    msg = lib().iic_last_error().decode("utf-8", "replace")
    if rc == -1:
      # the reference signals shape / argument problems with `assert` (IID_losses.py:10,40)
      raise AssertionError("%s: %s" % (what, msg))
    raise IICError("%s failed (%d): %s" % (what, rc, msg))
