"""Thin typed wrappers: torch CUDA tensors -> raw pointers -> libiic_b200.so.

Each function enqueues its kernel(s) on ``torch.cuda.current_stream()`` and
returns immediately.  Inputs must be contiguous CUDA tensors; nothing here
touches the CPU path (there is none).
"""
import ctypes

import torch

from . import _lib
from ._lib import BF16, F32, TF32, TF32X3, ConvGeom, check

# storage dtype per mode (TF32 / TF32X3 are compute modes of the convolutions on fp32 storage)
_TORCH_DT = {F32: torch.float32, BF16: torch.bfloat16, TF32: torch.float32, TF32X3: torch.float32}


def torch_dtype(dt):
  return _TORCH_DT[dt]


def iic_dtype(t):
  if t.dtype == torch.float32:
    return F32
  if t.dtype == torch.bfloat16:
    return BF16
  raise AssertionError("unsupported dtype %s" % t.dtype)


def _stream():
  return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _p(t):
  if t is None:
    return None
  assert t.is_cuda, "iic_b200 runs on CUDA tensors only (no CPU fallback)"
  assert t.is_contiguous(), "iic_b200 kernels need contiguous tensors"
  return ctypes.c_void_p(t.data_ptr())


def conv_geom(n, h, w, cin, cout, kh, kw, stride, pad, dil):
  oh = (h + 2 * pad - dil * (kh - 1) - 1) // stride + 1
  ow = (w + 2 * pad - dil * (kw - 1) - 1) // stride + 1
  return ConvGeom(n, h, w, cin, oh, ow, cout, kh, kw, stride, pad, dil)


# ---- optional per-launch timing of the convolution kernels (bench.py roofline leg) ---------------
_conv_timing = {"on": False, "records": []}


def conv_timing(enable):
  _conv_timing["on"] = bool(enable)
  _conv_timing["records"] = []


def conv_timing_summary():
  """-> dict kind -> (launches, algorithmic FLOPs, device ms); call after torch.cuda.synchronize()."""
  out = {}
  for kind, flops, e0, e1 in (r[:4] for r in _conv_timing["records"]):
    n, f, ms = out.get(kind, (0, 0.0, 0.0))
    out[kind] = (n + 1, f + flops, ms + e0.elapsed_time(e1))
  return out


def conv_timing_by_layer():
  """-> dict "kind KxK sS CIN->COUT @H xN" -> (launches, algorithmic FLOPs, device ms): the live per-geometry table."""
  out = {}
  for rec in _conv_timing["records"]:
    if len(rec) < 5 or rec[4] is None:
      continue
    kind, flops, e0, e1, g = rec
    key = "%s %dx%d s%d %d->%d @%d n%d" % (kind, g.kh, g.kw, g.stride, g.cin, g.cout, g.h, g.n)
    n, f, ms = out.get(key, (0, 0.0, 0.0))
    out[key] = (n + 1, f + flops, ms + e0.elapsed_time(e1))
  return out


class _timed(object):
  def __init__(self, kind, g):
    self.kind, self.g = kind, g

  def __enter__(self):
    if _conv_timing["on"]:
      self.e0, self.e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
      self.e0.record()
    return self

  def __exit__(self, *exc):
    if _conv_timing["on"]:
      self.e1.record()
      g = self.g
      flops = 2.0 * g.n * g.oh * g.ow * g.cout * g.kh * g.kw * g.cin  # 2*MAC, identical for fprop/dgrad/wgrad
      _conv_timing["records"].append((self.kind, flops, self.e0, self.e1, g))
    return False


def _cat(name):
  """Times a whole wrapper under category `name` when conv_timing is on (bench.py breakdown)."""
  def deco(fn):
    def wrapped(*a, **kw):
      if not _conv_timing["on"]:
        return fn(*a, **kw)
      e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
      e0.record()
      r = fn(*a, **kw)
      e1.record()
      _conv_timing["records"].append((name, 0.0, e0, e1))
      return r
    wrapped.__name__ = fn.__name__
    wrapped.__doc__ = fn.__doc__
    return wrapped
  return deco


def launch_count(reset=False):
  return int(_lib.lib().iic_launch_count(1 if reset else 0))


def get_option(name):
  """Kernel-variant switch of the library (include/iic_b200.h: iic_get_option)."""
  v = _lib.lib().iic_get_option(name.encode())
  if v < 0:
    _lib.check(v, "iic_get_option")
  return v


def set_option(name, value):
  """Sets a kernel-variant switch; returns the previous value."""
  v = _lib.lib().iic_set_option(name.encode(), int(value))
  if v < 0:
    _lib.check(v, "iic_set_option")
  return v


class options:
  """`with kernels.options(conv_halo=2): ...` -- scoped override of kernel-variant switches (tests, A/B runs)."""

  def __init__(self, **kw):
    self.kw, self.prev = kw, {}

  def __enter__(self):
    for k, v in self.kw.items():
      self.prev[k] = set_option(k, v)
    return self

  def __exit__(self, *exc):
    for k, v in self.prev.items():
      set_option(k, v)
    return False


# ---- losses ---------------------------------------------------------------------------------
@_cat("iid_loss")
def iid_loss(z, zt, lamb, eps, want_grad, phase=_lib.PHASE_FUSED, joint_ws=None, want_joint=False):
  """z, zt: [S, n, k] fp32.  Returns (loss[S,2] | None, dz | None, dzt | None, joint_out | None)."""
  S, n, k = z.shape
  assert zt.shape == z.shape and z.dtype == torch.float32 and zt.dtype == torch.float32
  loss = None if phase == _lib.PHASE_PARTIAL else torch.empty((S, 2), device=z.device, dtype=torch.float32)
  dz = torch.empty_like(z) if (want_grad and phase != _lib.PHASE_PARTIAL) else None
  dzt = torch.empty_like(zt) if (want_grad and phase != _lib.PHASE_PARTIAL) else None
  jout = torch.empty((S, k, k), device=z.device, dtype=torch.float32) if want_joint else None
  check(_lib.lib().iic_iid_loss(_p(z), _p(zt), S, n, k, float(lamb), float(eps), _p(loss), _p(dz), _p(dzt),
                                _p(joint_ws), _p(jout), phase, _stream()), "iic_iid_loss")
  return loss, dz, dzt, jout


def joint_mi(joint, lamb, eps, detached, want_h):
  """joint [S,k,k] raw -> (loss [S,2], H [S,k,k] | None)"""
  S, k, _ = joint.shape
  loss = torch.empty((S, 2), device=joint.device, dtype=torch.float32)
  H = torch.empty_like(joint) if want_h else None
  check(_lib.lib().iic_joint_mi(_p(joint), S, k, float(lamb), float(eps), int(bool(detached)), _p(loss), _p(H),
                                _stream()), "iic_joint_mi")
  return loss, H


# ---- segmentation objective -------------------------------------------------------------------
def seg_kp(k):
  kp = int(_lib.lib().iic_seg_kp(int(k)))
  assert kp > 0, "segmentation losses support k <= 48"
  return kp


def seg_prepare(x1, x2, theta, mask, shift=(0, 0)):
  n, k, h, w = x1.shape
  kp = seg_kp(k)
  x1m = torch.empty((n, h, w, kp), device=x1.device, dtype=torch.float32)
  x2m = torch.empty_like(x1m)
  check(_lib.lib().iic_seg_prepare_shift(_p(x1), _p(x2), _p(theta), _p(mask), _p(x1m), _p(x2m), n, k, h, w, int(shift[0]),
                                         int(shift[1]), _stream()), "iic_seg_prepare")
  return x1m, x2m


def seg_unprepare(dx1m, dx2m, theta, mask, k, shift=(0, 0)):
  n, h, w, _ = dx1m.shape
  dx1 = torch.empty((n, k, h, w), device=dx1m.device, dtype=torch.float32)
  dx2 = torch.empty_like(dx1)
  check(_lib.lib().iic_seg_unprepare_shift(_p(dx1m), _p(dx2m), _p(theta), _p(mask), _p(dx1), _p(dx2), n, k, h, w,
                                           int(shift[0]), int(shift[1]), _stream()), "iic_seg_unprepare")
  return dx1, dx2


# host-side switches of the tensor-core segmentation kernels (csrc/seg_joint_tc.cu):
#   SEG_CORR_TC   backward contractions (kind::tf32, K-major overlapped operand): validated on a B200 in round 2
#                 (tests/test_gpu_parity_seg.py::test_seg_corr_tensor_core_matches_simt), ON
#   SEG_JOINT_TC  forward joint (kind::f16 on bf16 three-term operands, MN-major Toeplitz operand): validated on a B200 in
#                 round 2 (test_seg_joint_tensor_core_matches_simt_and_oracle, the reference golden of the loss), ON
SEG_CORR_TC = {"on": __import__("os").environ.get("IIC_SEG_CORR_TC", "1") != "0"}
SEG_JOINT_TC = {"on": __import__("os").environ.get("IIC_SEG_JOINT_TC", "1") != "0"}


def seg_joint_tc(x1m, x2m, k, T):
  """Tensor-core joint; returns None when the geometry is not supported."""
  n, h, w, kp = x1m.shape
  if kp != 16:
    return None
  nbytes = int(_lib.lib().iic_seg_joint_tc_workspace(n, k, h, w, T))
  if nbytes <= 0:
    return None
  V = 2 * T + 1
  ws = torch.empty(nbytes // 4, device=x1m.device, dtype=torch.float32)
  joint = torch.empty((V * V, k, k), device=x1m.device, dtype=torch.float32)
  check(_lib.lib().iic_seg_joint_tc(_p(x1m), _p(x2m), _p(joint), _p(ws), n, k, h, w, T, _stream()), "iic_seg_joint_tc")
  return joint


def seg_joint(x1m, x2m, k, T, allow_tc=True):
  if allow_tc and SEG_JOINT_TC["on"] and T > 0:
    j = seg_joint_tc(x1m, x2m, k, T)
    if j is not None:
      return j
  n, h, w, _ = x1m.shape
  V = 2 * T + 1
  nbytes = int(_lib.lib().iic_seg_joint_workspace(n, k, T))
  ws = torch.empty(max(nbytes // 4, 1), device=x1m.device, dtype=torch.float32)
  joint = torch.empty((V * V, k, k), device=x1m.device, dtype=torch.float32)
  check(_lib.lib().iic_seg_joint(_p(x1m), _p(x2m), _p(joint), _p(ws), n, k, h, w, T, _stream()), "iic_seg_joint")
  return joint


def seg_corr_tc(inp, H, k, T, sgn, scale):
  """Tensor-core version of seg_corr_bwd; None when the geometry is not supported."""
  n, h, w, kp = inp.shape
  if kp != 16:
    return None
  nbytes = int(_lib.lib().iic_seg_corr_tc_workspace(n, k, h, w, T))
  if nbytes <= 0:
    return None
  ws = torch.empty(nbytes // 4, device=inp.device, dtype=torch.float32)
  out = torch.empty_like(inp)
  check(_lib.lib().iic_seg_corr_tc(_p(inp), _p(H), _p(out), _p(ws), n, k, h, w, T, sgn, float(scale), _stream()),
        "iic_seg_corr_tc")
  return out


def seg_corr_bwd(inp, H, k, T, sgn, scale, allow_tc=True):
  if allow_tc and SEG_CORR_TC["on"] and T > 0:
    o = seg_corr_tc(inp, H, k, T, sgn, scale)
    if o is not None:
      return o
  n, h, w, _ = inp.shape
  out = torch.empty_like(inp)
  check(_lib.lib().iic_seg_corr_bwd(_p(inp), _p(H), _p(out), n, k, h, w, T, sgn, float(scale), _stream()),
        "iic_seg_corr_bwd")
  return out


def box_filter(x, k, T):
  n, h, w, _ = x.shape
  tmp, out = torch.empty_like(x), torch.empty_like(x)
  check(_lib.lib().iic_box_filter(_p(x), _p(tmp), _p(out), n, k, h, w, T, _stream()), "iic_box_filter")
  return out


@_cat("sobel")
def sobel(imgs, include_rgb, using_ir):
  n, c, h, w = imgs.shape
  cout = (3 if include_rgb else 0) + 2 + (1 if using_ir else 0)
  out = torch.empty((n, cout, h, w), device=imgs.device, dtype=torch.float32)
  check(_lib.lib().iic_sobel(_p(imgs), _p(out), n, c, h, w, int(bool(include_rgb)), int(bool(using_ir)), _stream()),
        "iic_sobel")
  return out


@_cat("sobel")
def grey_sobel(rgb):
  """rgb [n,3,h,w] uint8 or fp32 -> [n,2,h,w] sobel of the grey image (dataloader tail + sobel_process fused)."""
  n, c, h, w = rgb.shape
  assert c == 3 and rgb.dtype in (torch.uint8, torch.float32)
  out = torch.empty((n, 2, h, w), device=rgb.device, dtype=torch.float32)
  check(_lib.lib().iic_grey_sobel(_p(rgb), int(rgb.dtype == torch.uint8), _p(out), n, h, w, _stream()), "iic_grey_sobel")
  return out


# ---- layout ---------------------------------------------------------------------------------
def nchw_to_nhwc(x, dt):
  n, c, h, w = x.shape
  out = torch.empty((n, h, w, c), device=x.device, dtype=_TORCH_DT[dt])
  check(_lib.lib().iic_nchw_to_nhwc(_p(x), _p(out), dt, n, c, h, w, _stream()), "iic_nchw_to_nhwc")
  return out


def nhwc_to_nchw(x):
  n, h, w, c = x.shape
  out = torch.empty((n, c, h, w), device=x.device, dtype=torch.float32)
  check(_lib.lib().iic_nhwc_to_nchw(_p(x), iic_dtype(x), _p(out), n, c, h, w, _stream()), "iic_nhwc_to_nchw")
  return out


def cast(x, dt):
  out = torch.empty(x.shape, device=x.device, dtype=_TORCH_DT[dt])
  check(_lib.lib().iic_cast(_p(x), iic_dtype(x), _p(out), dt, x.numel(), _stream()), "iic_cast")
  return out


# ---- convolution ----------------------------------------------------------------------------
def weight_dtype(dt, cdt):
  """dtype to hand to pack_weight for storage dtype `dt` and compute dtype `cdt`: 3xTF32 convolutions take their
  weights pre-split ([2][...] fp32: raw plane + lo plane, include/iic_b200.h: iic_pack_weight)."""
  return TF32X3 if cdt == TF32X3 else dt


def _packed_shape(w, dt, kind):
  cout, cin, kh, kw = w.shape
  shape = (cout, kh, kw, cin) if kind == 0 else (cin, kh, kw, cout)
  return (2,) + shape if dt == TF32X3 else shape


@_cat("pack_weight")
def pack_weight(w, dt, kind):
  cout, cin, kh, kw = w.shape
  out = torch.empty(_packed_shape(w, dt, kind), device=w.device, dtype=_TORCH_DT[dt])
  check(_lib.lib().iic_pack_weight(_p(w), _p(out), dt, kind, cout, cin, kh, kw, _stream()), "iic_pack_weight")
  return out


class PackPlan(object):
  """Device job table + persistent destination buffers for iic_pack_weights_batched.  Built once per set of
  weight tensors (keyed by their storage addresses) and replayed every step: one launch instead of one per
  convolution and layout."""

  def __init__(self, weights, kinds, dt):
    import numpy as np
    self.key = PackPlan.make_key(weights, kinds, dt)
    self.dt = dt
    self.out = {}
    jobs = (_lib.PackJob * (len(weights) * len(kinds)))()
    i = 0
    for wi, w in enumerate(weights):
      assert w.is_cuda and w.is_contiguous() and w.dtype == torch.float32
      cout, cin, kh, kw = w.shape
      for kind in kinds:
        dst = torch.empty(_packed_shape(w, dt, kind), device=w.device, dtype=_TORCH_DT[dt])
        self.out[(wi, kind)] = dst
        jobs[i] = _lib.PackJob(w.data_ptr(), dst.data_ptr(), kind, cout, cin, kh, kw, 0)
        i += 1
    self.njobs = i
    raw = np.frombuffer(bytes(jobs), dtype=np.uint8).copy()
    self.table = torch.from_numpy(raw).to(weights[0].device)

  @staticmethod
  def make_key(weights, kinds, dt):
    return (tuple(w.data_ptr() for w in weights), tuple(kinds), dt)

  @_cat("pack_weight")
  def run(self):
    check(_lib.lib().iic_pack_weights_batched(_p(self.table), self.njobs, self.dt, _stream()), "iic_pack_weights_batched")
    return self.out


def _check_packed(wp, g, dt):
  want = (2 if dt == TF32X3 else 1) * g.cout * g.cin * g.kh * g.kw
  assert wp.numel() == want, "weights for dtype %d must be packed with pack_weight(w, weight_dtype(store, %d), kind): %d elements, expected %d" % (dt, dt, wp.numel(), want)


def conv_fprop(x, wp, g, dt):
  _check_packed(wp, g, dt)
  y = torch.empty((g.n, g.oh, g.ow, g.cout), device=x.device, dtype=_TORCH_DT[dt])
  with _timed("fprop", g):
    check(_lib.lib().iic_conv_fprop(_p(x), _p(wp), _p(y), ctypes.byref(g), dt, _stream()), "iic_conv_fprop")
  return y


def conv_fprop_stats(x, wp, g, dt, views):
  """fprop + fused per-view BN statistics partials.  Returns (y, partial, nblk) or None if unsupported."""
  nblk = int(_lib.lib().iic_conv_fprop_stats_blocks(ctypes.byref(g), dt))
  if nblk <= 0:
    return None
  y = torch.empty((g.n, g.oh, g.ow, g.cout), device=x.device, dtype=_TORCH_DT[dt])
  partial = torch.empty((nblk, 2, 2, g.cout), device=x.device, dtype=torch.float32)  # rows are always [2 views][2][C]
  with _timed("fprop", g):
    check(_lib.lib().iic_conv_fprop_stats(_p(x), _p(wp), _p(y), ctypes.byref(g), dt, views, _p(partial), _stream()),
          "iic_conv_fprop_stats")
  return y, partial, nblk


@_cat("bn_stats")
def bn_stats_from_partials(partial, nblk, views, view, M, gamma, beta, eps, momentum, running_mean, running_var):
  C = gamma.numel()
  dev = partial.device
  ws = torch.empty(2 * C, device=dev, dtype=torch.float64)
  ss = torch.empty(2 * C, device=dev, dtype=torch.float32)
  mi = torch.empty(2 * C, device=dev, dtype=torch.float32)
  check(_lib.lib().iic_bn_stats_from_partials(_p(partial), nblk, views, view, M, C, _p(gamma), _p(beta), float(eps),
                                              float(momentum), _p(running_mean), _p(running_var), _p(ws), _p(ss), _p(mi),
                                              _stream()), "iic_bn_stats_from_partials")
  return ss, mi


def conv_dgrad(dy, wpt, g, dt, addend=None, addend_mask=None):
  """addend_mask (uint8 [pixels][cin / 8], bn_apply_views_mask's bits): the addend passes only where its bit is set."""
  _check_packed(wpt, g, dt)
  dx = torch.empty((g.n, g.h, g.w, g.cin), device=dy.device, dtype=_TORCH_DT[dt])
  with _timed("dgrad", g):
    if addend_mask is not None:
      assert addend is not None and addend_mask.dtype == torch.uint8 and addend_mask.numel() * 8 == addend.numel()
      check(_lib.lib().iic_conv_dgrad_masked(_p(dy), _p(wpt), _p(addend), _p(addend_mask), _p(dx), ctypes.byref(g), dt,
                                             _stream()), "iic_conv_dgrad_masked")
    else:
      check(_lib.lib().iic_conv_dgrad(_p(dy), _p(wpt), _p(addend), _p(dx), ctypes.byref(g), dt, _stream()),
            "iic_conv_dgrad")
  return dx


# host-side switch: wgrad writes the torch-layout gradient itself (iic_conv_wgrad_oihw) instead of wgrad + unpack
# (validated on a B200 in round 2: bit-identical in 12 geometries; 350 launches per step less)
WGRAD_FUSED_UNPACK = {"on": __import__("os").environ.get("IIC_WGRAD_FUSED", "1") != "0"}


def conv_wgrad(x, dy, g, dt, grad_out, accumulate):
  """Accumulates (or writes) the torch-layout [cout][cin][kh][kw] fp32 gradient into grad_out."""
  if WGRAD_FUSED_UNPACK["on"]:
    nbytes = int(_lib.lib().iic_conv_wgrad_oihw_workspace(ctypes.byref(g), dt))
    ws = torch.empty((max(nbytes, 4) + 3) // 4, device=x.device, dtype=torch.float32)
    with _timed("wgrad", g):
      check(_lib.lib().iic_conv_wgrad_oihw(_p(x), _p(dy), _p(grad_out), int(bool(accumulate)), _p(ws), ctypes.byref(g), dt,
                                           _stream()), "iic_conv_wgrad_oihw")
    return grad_out
  nbytes = int(_lib.lib().iic_conv_wgrad_workspace(ctypes.byref(g), dt))
  ws = torch.empty((max(nbytes, 4) + 3) // 4, device=x.device, dtype=torch.float32)
  dwp = torch.empty((g.cout, g.kh, g.kw, g.cin), device=x.device, dtype=torch.float32)
  with _timed("wgrad", g):
    check(_lib.lib().iic_conv_wgrad(_p(x), _p(dy), _p(dwp), _p(ws), ctypes.byref(g), dt, _stream()), "iic_conv_wgrad")
  check(_lib.lib().iic_unpack_wgrad(_p(dwp), _p(grad_out), int(bool(accumulate)), g.cout, g.cin, g.kh, g.kw, _stream()),
        "iic_unpack_wgrad")
  return grad_out


@_cat("stem_fprop")
def stem_fprop(x_nchw, w, g, dt):
  y = torch.empty((g.n, g.oh, g.ow, g.cout), device=x_nchw.device, dtype=_TORCH_DT[dt])
  check(_lib.lib().iic_stem_fprop(_p(x_nchw), _p(w), _p(y), ctypes.byref(g), dt, _stream()), "iic_stem_fprop")
  return y


# stem convolution (+ statistics) on tcgen05 in bf16 mode (csrc/stem_tc.cu); written after the last GPU session: off
STEM_FPROP_TC = {"on": __import__("os").environ.get("IIC_STEM_FPROP_TC", "0") != "0"}


def stem_fprop_stats_tc(x_nchw, w, g, views):
  """-> (y bf16, partial, nblk) or None if the geometry is unsupported (include/iic_b200.h: iic_stem_fprop_stats_tc)."""
  nblk = int(_lib.lib().iic_stem_fprop_stats_tc_blocks(ctypes.byref(g), views))
  if nblk <= 0:
    return None
  y = torch.empty((g.n, g.oh, g.ow, g.cout), device=x_nchw.device, dtype=torch.bfloat16)
  partial = torch.empty((nblk, 2, 2, g.cout), device=x_nchw.device, dtype=torch.float32)
  check(_lib.lib().iic_stem_fprop_stats_tc(_p(x_nchw), _p(w), _p(y), ctypes.byref(g), views, _p(partial), _stream()),
        "iic_stem_fprop_stats_tc")
  return y, partial, nblk


@_cat("stem_fprop")
def stem_fprop_stats(x_nchw, w, g, dt, views):
  """Stem conv + fused per-view BN statistics partials.  Returns (y, partial, nblk) or None if unsupported."""
  if STEM_FPROP_TC["on"] and dt == BF16:
    r = stem_fprop_stats_tc(x_nchw, w, g, views)
    if r is not None:
      return r
  nblk = int(_lib.lib().iic_stem_fprop_stats_blocks(ctypes.byref(g), dt, views))
  if nblk <= 0:
    return None
  y = torch.empty((g.n, g.oh, g.ow, g.cout), device=x_nchw.device, dtype=_TORCH_DT[dt])
  partial = torch.empty((nblk, 2, 2, g.cout), device=x_nchw.device, dtype=torch.float32)
  check(_lib.lib().iic_stem_fprop_stats(_p(x_nchw), _p(w), _p(y), ctypes.byref(g), dt, views, _p(partial), _stream()),
        "iic_stem_fprop_stats")
  return y, partial, nblk


def stem_bwd_fused_workspace(g, pool_pad, views, dt):
  """Scratch bytes of iic_stem_bwd_fused, 0 if the geometry is not supported."""
  return int(_lib.lib().iic_stem_bwd_fused_workspace(ctypes.byref(g), pool_pad, views, dt))


@_cat("stem_bwd_dy")
def stem_bwd_dy(y, dpool, ss, mi, gamma, dgamma, dbeta, bn_accumulate, g, pool_pad, dt):
  """Max-pool routing + ReLU + BatchNorm backward of the stem in two passes over (y, dpool) -> dy (csrc/stem_bwd.cu:
  iic_stem_bwd_dy).  ss, mi: [views, 128] stacked per-view BN coefficients.  Returns None if the geometry is unsupported."""
  views = ss.shape[0]
  nbytes = stem_bwd_fused_workspace(g, pool_pad, views, dt)
  if nbytes <= 0:
    return None
  assert ss.is_contiguous() and mi.is_contiguous() and ss.shape == mi.shape == (views, 128)
  assert y.is_contiguous() and dpool.is_contiguous() and iic_dtype(y) == dt == iic_dtype(dpool)
  ws = torch.empty(nbytes, device=y.device, dtype=torch.uint8)
  dy = torch.empty_like(y)
  check(_lib.lib().iic_stem_bwd_dy(_p(y), _p(dpool), _p(ss), _p(mi), _p(gamma), _p(dgamma), _p(dbeta), int(bool(bn_accumulate)),
                                   _p(dy), ctypes.byref(g), pool_pad, views, dt, _p(ws), nbytes, _stream()), "iic_stem_bwd_dy")
  return dy


@_cat("stem_bwd_fused")
def stem_bwd_fused(x_nchw, y, dpool, ss, mi, gamma, dgamma, dbeta, bn_accumulate, grad_w, w_accumulate, g, pool_pad, dt):
  """Backward of conv3x3 -> BN -> ReLU -> MaxPool(2,2,pool_pad) of the stem in two passes (csrc/stem_bwd.cu).
  ss, mi: [views, 128] stacked per-view BN coefficients.  Returns False (nothing done) if the geometry is unsupported."""
  views = ss.shape[0]
  nbytes = stem_bwd_fused_workspace(g, pool_pad, views, dt)
  if nbytes <= 0:
    return False
  assert ss.is_contiguous() and mi.is_contiguous() and ss.shape == mi.shape == (views, 128)
  assert y.is_contiguous() and dpool.is_contiguous() and x_nchw.is_contiguous() and iic_dtype(y) == dt == iic_dtype(dpool)
  ws = torch.empty(nbytes, device=y.device, dtype=torch.uint8)
  check(_lib.lib().iic_stem_bwd_fused(_p(x_nchw), _p(y), _p(dpool), _p(ss), _p(mi), _p(gamma), _p(dgamma), _p(dbeta),
                                      int(bool(bn_accumulate)), _p(grad_w), int(bool(w_accumulate)), ctypes.byref(g),
                                      pool_pad, views, dt, _p(ws), nbytes, _stream()), "iic_stem_bwd_fused")
  return True


# host-side switch: stem wgrad as im2col + the tcgen05 1x1 wgrad kernel (bf16 mode; OFF until validated on hardware)
STEM_WGRAD_TC = {"on": __import__("os").environ.get("IIC_STEM_WGRAD_TC", "1") != "0"}


STEM_WGRAD_TC64 = {"on": __import__("os").environ.get("IIC_STEM_WGRAD_TC64", "1") != "0"}


def stem_wgrad_tc(x_nchw, dy, g, grad_out, accumulate):
  """bf16 tcgen05 stem wgrad (include/iic_b200.h: iic_stem_wgrad_tc); returns False if the geometry is unsupported."""
  K = g.cin * g.kh * g.kw
  # (33..64 taps -- SegmentationNet10a: validated in the last GPU call of round 2, profiles/r02_session_u.md; its effect on the
  # c5 step was not measured any more: IIC_STEM_WGRAD_TC64=0 returns those stems to the SIMT kernel)
  kmax = 64 if STEM_WGRAD_TC64["on"] else 32
  if not (K <= kmax and g.cout == 64 and g.stride == 1 and g.dil == 1 and g.oh == g.h and g.ow == g.w and dy.dtype == torch.bfloat16):
    return False
  nbytes = int(_lib.lib().iic_stem_wgrad_tc_workspace(ctypes.byref(g)))
  ws = torch.empty(nbytes // 4, device=dy.device, dtype=torch.float32)
  check(_lib.lib().iic_stem_wgrad_tc(_p(x_nchw), _p(dy), _p(grad_out), int(bool(accumulate)), _p(ws), ctypes.byref(g), _stream()),
        "iic_stem_wgrad_tc")
  return True


@_cat("stem_wgrad")
def stem_wgrad(x_nchw, dy, g, dt, grad_out, accumulate):
  if STEM_WGRAD_TC["on"] and dt == BF16 and stem_wgrad_tc(x_nchw, dy, g, grad_out, accumulate):
    return grad_out
  ws = torch.empty(2 * 1024 * 1024, device=dy.device, dtype=torch.float32)  # 8 MB of per-block partials
  check(_lib.lib().iic_stem_wgrad(_p(x_nchw), _p(dy), _p(grad_out), int(bool(accumulate)), _p(ws), ws.numel() * 4,
                                  ctypes.byref(g), dt, _stream()), "iic_stem_wgrad")
  return grad_out


# ---- batch norm / pooling ----------------------------------------------------------------------
@_cat("bn_stats")
def bn_stats(y, gamma, beta, eps, momentum, running_mean, running_var, use_running, ss=None, mi=None):
  C = y.shape[-1]
  M = y.numel() // C
  dev = y.device
  ws = torch.empty(2 * C, device=dev, dtype=torch.float64)
  ss = torch.empty(2 * C, device=dev, dtype=torch.float32) if ss is None else ss
  mi = torch.empty(2 * C, device=dev, dtype=torch.float32) if mi is None else mi
  check(_lib.lib().iic_bn_stats(_p(y), iic_dtype(y), M, C, _p(gamma), _p(beta), float(eps), float(momentum),
                                _p(running_mean), _p(running_var), int(bool(use_running)), _p(ws), _p(ss), _p(mi),
                                _stream()), "iic_bn_stats")
  return ss, mi


@_cat("bn_stats")
def bn_stats_from_partials_views(partial, nblk, slots, views, M, gamma, beta, eps, momentum, running_mean, running_var):
  """All views in one launch -> (scale_shift [views, 2C], mean_invstd [views, 2C])."""
  C = gamma.numel()
  ss = torch.empty((views, 2 * C), device=partial.device, dtype=torch.float32)
  mi = torch.empty((views, 2 * C), device=partial.device, dtype=torch.float32)
  check(_lib.lib().iic_bn_stats_from_partials_views(_p(partial), nblk, slots, views, M, C, _p(gamma), _p(beta), float(eps),
                                                    float(momentum), _p(running_mean), _p(running_var), _p(ss), _p(mi),
                                                    _stream()), "iic_bn_stats_from_partials_views")
  return ss, mi


@_cat("bn_apply")
def bn_apply_views(y, ss, relu, views, res=None, rss=None, out=None):
  """y: `views` stacked batches; ss / rss: [views, 2C] contiguous."""
  C = y.shape[-1]
  M = y.numel() // C
  assert M % views == 0 and ss.is_contiguous() and (rss is None or rss.is_contiguous())
  if out is None:
    out = torch.empty_like(y)
  check(_lib.lib().iic_bn_apply_views(_p(y), _p(ss), _p(res), _p(rss), _p(out), iic_dtype(y), M // views, C,
                                      int(bool(relu)), views, _stream()), "iic_bn_apply_views")
  return out


@_cat("bn_apply")
def bn_apply_views_mask(y, ss, views, res=None, rss=None):
  """relu(bn(y) + residual term) for `views` stacked batches plus its ReLU mask, one byte per 8 channels.
  Returns (out, mask_bits [rows, C / 8] uint8)."""
  C = y.shape[-1]
  M = y.numel() // C
  assert M % views == 0 and ss.is_contiguous() and (rss is None or rss.is_contiguous())
  out = torch.empty_like(y)
  mbits = torch.empty((M, C // 8), device=y.device, dtype=torch.uint8)
  check(_lib.lib().iic_bn_apply_views_mask(_p(y), _p(ss), _p(res), _p(rss), _p(out), _p(mbits), iic_dtype(y), M // views, C,
                                           views, _stream()), "iic_bn_apply_views_mask")
  return out, mbits


@_cat("bn_bwd")
def bn_bwd_fused_bits(g_in, mbits, y, mis, gamma, dgamma, dbeta, accumulate, want_g_out):
  """bn_bwd_fused with the ReLU mask given as bits (bn_apply_views_mask) instead of the activation."""
  views = len(mis)
  assert views in (1, 2)
  C = y.shape[-1]
  M = y.numel() // C
  assert M % views == 0 and mbits.dtype == torch.uint8 and mbits.numel() == M * (C // 8) and mbits.is_contiguous()
  dy = torch.empty_like(y)
  g_out = torch.empty_like(y) if want_g_out else None
  mi1 = mis[1] if views == 2 else None
  check(_lib.lib().iic_bn_bwd_fused_bits(_p(g_in), _p(mbits), _p(y), views, _p(mis[0]), _p(mi1), _p(gamma), _p(dy), _p(g_out),
                                         _p(dgamma), _p(dbeta), int(bool(accumulate)), iic_dtype(y), M // views, C,
                                         _stream()), "iic_bn_bwd_fused_bits")
  return dy, g_out


@_cat("bn_bwd")
def bn_bwd_fused(g_in, act, y, mis, gamma, dgamma, dbeta, accumulate, want_g_out, mask_sss=None):
  """BatchNorm backward of 1 or 2 stacked views in one cooperative launch.  mis / mask_sss: per-view tensors."""
  views = len(mis)
  assert views in (1, 2)
  C = y.shape[-1]
  M = y.numel() // C
  assert M % views == 0 and (act is None or mask_sss is None)
  dy = torch.empty_like(y)
  g_out = torch.empty_like(y) if want_g_out else None
  ms = list(mask_sss) if mask_sss is not None else [None] * views
  mi1 = mis[1] if views == 2 else None
  ms1 = ms[1] if views == 2 else None
  check(_lib.lib().iic_bn_bwd_fused(_p(g_in), _p(act), _p(y), views, _p(mis[0]), _p(mi1), _p(ms[0]), _p(ms1), _p(gamma),
                                    _p(dy), _p(g_out), _p(dgamma), _p(dbeta), int(bool(accumulate)), iic_dtype(y),
                                    M // views, C, _stream()), "iic_bn_bwd_fused")
  return dy, g_out


@_cat("bn_apply")
def bn_apply(y, ss, relu, res=None, rss=None, out=None):
  C = y.shape[-1]
  M = y.numel() // C
  if out is None:
    out = torch.empty_like(y)
  check(_lib.lib().iic_bn_apply(_p(y), _p(ss), _p(res), _p(rss), _p(out), iic_dtype(y), M, C, int(bool(relu)),
                                _stream()), "iic_bn_apply")
  return out


def pooled_shape(y, pad):
  n, h, w, C = y.shape
  return (n, (h + 2 * pad - 2) // 2 + 1, (w + 2 * pad - 2) // 2 + 1, C)


@_cat("bn_pool")
def bn_relu_maxpool(y, ss, pad, out=None):
  n, h, w, C = y.shape
  oh, ow = (h + 2 * pad - 2) // 2 + 1, (w + 2 * pad - 2) // 2 + 1
  if out is None:
    out = torch.empty((n, oh, ow, C), device=y.device, dtype=y.dtype)
  check(_lib.lib().iic_bn_relu_maxpool(_p(y), _p(ss), _p(out), iic_dtype(y), n, h, w, C, pad, oh, ow, _stream()),
        "iic_bn_relu_maxpool")
  return out


@_cat("bn_pool_bwd")
def bn_relu_maxpool_bwd(y, ss, dpool, pad, out=None):
  n, h, w, C = y.shape
  _, oh, ow, _ = dpool.shape
  g = torch.empty_like(y) if out is None else out
  check(_lib.lib().iic_bn_relu_maxpool_bwd(_p(y), _p(ss), _p(dpool), _p(g), iic_dtype(y), n, h, w, C, pad, oh, ow,
                                           _stream()), "iic_bn_relu_maxpool_bwd")
  return g


@_cat("bn_bwd")
def bn_bwd(g_in, act, y, mi, gamma, dgamma, dbeta, accumulate, want_g_out, dy=None, g_out=None, mask_ss=None):
  """Returns (dy, g_masked | None); writes/accumulates dgamma, dbeta."""
  C = y.shape[-1]
  M = y.numel() // C
  dt = iic_dtype(y)
  sums = torch.empty(2 * C, device=y.device, dtype=torch.float64)
  assert act is None or mask_ss is None
  check(_lib.lib().iic_bn_bwd_reduce(_p(g_in), _p(act), _p(mask_ss), _p(y), _p(mi), dt, M, C, _p(sums), _stream()),
        "iic_bn_bwd_reduce")
  if dy is None:
    dy = torch.empty_like(y)
  if want_g_out and g_out is None:
    g_out = torch.empty_like(y)
  if not want_g_out:
    g_out = None
  check(_lib.lib().iic_bn_bwd_apply(_p(g_in), _p(act), _p(mask_ss), _p(y), _p(mi), _p(gamma), _p(sums), _p(dy), _p(g_out),
                                    _p(dgamma), _p(dbeta), int(bool(accumulate)), dt, M, C, _stream()),
        "iic_bn_bwd_apply")
  return dy, g_out


@_cat("avgpool")
def avgpool(x):
  n, h, w, C = x.shape
  feat = torch.empty((n, C), device=x.device, dtype=torch.float32)
  check(_lib.lib().iic_avgpool(_p(x), iic_dtype(x), _p(feat), n, h * w, C, _stream()), "iic_avgpool")
  return feat


@_cat("avgpool")
def avgpool_bwd(dfeat, shape, dt):
  n, h, w, C = shape
  dx = torch.empty(shape, device=dfeat.device, dtype=_TORCH_DT[dt])
  check(_lib.lib().iic_avgpool_bwd(_p(dfeat), _p(dx), dt, n, h * w, C, _stream()), "iic_avgpool_bwd")
  return dx


# ---- heads ----------------------------------------------------------------------------------
@_cat("heads")
def heads_fwd(feat, w, b, S, k):
  n, F = feat.shape
  logits = torch.empty((n, S * k), device=feat.device, dtype=torch.float32)
  z = torch.empty((S, n, k), device=feat.device, dtype=torch.float32)
  check(_lib.lib().iic_heads_fwd(_p(feat), _p(w), _p(b), _p(logits), _p(z), n, F, S, k, _stream()), "iic_heads_fwd")
  return z


@_cat("heads")
def heads_bwd(feat, w, z, dz, S, k, want_dfeat):
  n, F = feat.shape
  dlog = torch.empty((n, S * k), device=feat.device, dtype=torch.float32)
  dw = torch.empty_like(w)
  db = torch.empty(S * k, device=feat.device, dtype=torch.float32)
  dfeat = torch.empty_like(feat) if want_dfeat else None
  check(_lib.lib().iic_heads_bwd(_p(feat), _p(w), _p(z), _p(dz), _p(dlog), _p(dw), _p(db), _p(dfeat), n, F, S, k,
                                 _stream()), "iic_heads_bwd")
  return dw, db, dfeat


# ---- semi-supervised finetuning (csrc/semisup.cu) ------------------------------------------------
@_cat("cross_entropy")
def cross_entropy(logits, targets):
  """logits [n, k] fp32, targets [n] int64 -> (mean NLL as a 0-dim fp32 tensor, dlogits [n, k] = (softmax - onehot) / n)."""
  n, k = logits.shape
  assert logits.dtype == torch.float32 and targets.dtype == torch.int64 and targets.shape == (n,)
  loss = torch.empty((), device=logits.device, dtype=torch.float32)
  dlogits = torch.empty_like(logits)
  check(_lib.lib().iic_cross_entropy(_p(logits), _p(targets), n, k, _p(loss), _p(dlogits), _stream()), "iic_cross_entropy")
  return loss, dlogits


@_cat("linear")
def linear_fwd(x, w, b):
  """x [n, K], w [N, K], b [N] | None (fp32) -> y [n, N] = x w^T + b."""
  n, K = x.shape
  N = w.shape[0]
  assert w.shape == (N, K) and x.dtype == w.dtype == torch.float32
  y = torch.empty((n, N), device=x.device, dtype=torch.float32)
  check(_lib.lib().iic_linear_fwd(_p(x), _p(w), _p(b), _p(y), n, K, N, _stream()), "iic_linear_fwd")
  return y


@_cat("linear")
def linear_bwd(x, w, dy, dw, db, accumulate, want_dx):
  """Writes (accumulate=False) or adds to dw [N, K] and db [N] | None; returns dx [n, K] or None."""
  n, K = x.shape
  N = w.shape[0]
  assert dy.shape == (n, N) and dw.shape == (N, K)
  dx = torch.empty_like(x) if want_dx else None
  check(_lib.lib().iic_linear_bwd(_p(x), _p(w), _p(dy), _p(dw), _p(db), _p(dx), int(bool(accumulate)), n, K, N, _stream()),
        "iic_linear_bwd")
  return dx


def col_sum(x, out, accumulate):
  """out [C] (=|+=) column sums of x [..., C] (fp32 or bf16)."""
  C = x.shape[-1]
  check(_lib.lib().iic_col_sum(_p(x), iic_dtype(x), x.numel() // C, C, _p(out), int(bool(accumulate)), _stream()),
        "iic_col_sum")
  return out


# ---- segmentation sub-head --------------------------------------------------------------------
def seg_head_fwd(feat, w, H, W):
  """feat NHWC [n,hf,wf,C]; w [k,C] fp32 -> (out NCHW [n,k,H,W] fp32, zlow)"""
  n, hf, wf, C = feat.shape
  k = w.shape[0]
  dev = feat.device
  logits = torch.empty((n * hf * wf, k), device=dev, dtype=torch.float32)
  zlow = torch.empty((n, hf + 2, wf + 2, k), device=dev, dtype=torch.float32)
  out = torch.empty((n, k, H, W), device=dev, dtype=torch.float32)
  check(_lib.lib().iic_seg_head_fwd(_p(feat), iic_dtype(feat), _p(w), _p(logits), _p(zlow), _p(out), n, hf, wf, C, k,
                                    H, W, _stream()), "iic_seg_head_fwd")
  return out, zlow


def seg_head_bwd(feat, w, zlow, dout, dfeat, accumulate):
  """Returns dw [k,C]; writes (or accumulates) the feature gradient into dfeat (same dtype as feat)."""
  n, hf, wf, C = feat.shape
  k = w.shape[0]
  H, W = dout.shape[2], dout.shape[3]
  dev = feat.device
  dzlow = torch.empty_like(zlow)
  dlog = torch.empty((n * hf * wf, k), device=dev, dtype=torch.float32)
  dw = torch.empty_like(w)
  nbytes = int(_lib.lib().iic_seg_head_workspace(n, hf, wf, C, k))
  ws = torch.empty(max(nbytes // 4, 1), device=dev, dtype=torch.float32)
  check(_lib.lib().iic_seg_head_bwd(_p(feat), iic_dtype(feat), _p(w), _p(zlow), _p(dout), _p(dzlow), _p(dlog), _p(dw),
                                    _p(ws), _p(dfeat), int(bool(accumulate)), n, hf, wf, C, k, H, W, _stream()),
        "iic_seg_head_bwd")
  return dw


# ---- optimiser ------------------------------------------------------------------------------
@_cat("adam")
def adam_step(params, grads, exp_avgs, exp_avg_sqs, lr, beta1, beta2, eps, weight_decay, step, step_dev=None):
  """step_dev: float32 device scalar holding the step count (graph-replayable form, iic_adam_step_dev)."""
  T = len(params)
  ptrs = (ctypes.c_void_p * (4 * T))()
  sizes = (ctypes.c_longlong * T)()
  for i, (p, g, m, v) in enumerate(zip(params, grads, exp_avgs, exp_avg_sqs)):
    for t in (p, g, m, v):
      assert t.is_cuda and t.is_contiguous() and t.dtype == torch.float32
    ptrs[4 * i], ptrs[4 * i + 1], ptrs[4 * i + 2], ptrs[4 * i + 3] = p.data_ptr(), g.data_ptr(), m.data_ptr(), v.data_ptr()
    sizes[i] = p.numel()
  if step_dev is not None:
    assert step_dev.is_cuda and step_dev.dtype == torch.float32 and step_dev.numel() == 1
    check(_lib.lib().iic_adam_step_dev(ptrs, sizes, T, float(lr), float(beta1), float(beta2), float(eps),
                                       float(weight_decay), _p(step_dev), _stream()), "iic_adam_step_dev")
    return
  check(_lib.lib().iic_adam_step(ptrs, sizes, T, float(lr), float(beta1), float(beta2), float(eps),
                                 float(weight_decay), int(step), _stream()), "iic_adam_step")


# ---- evaluation (SURVEY S8f row 4) ---------------------------------------------------------------------
def argmax_rows(z):
  """z [..., k] fp32 -> int32 [...]: torch.argmax(dim=-1) semantics (first maximum)."""
  assert z.dtype == torch.float32
  k = z.shape[-1]
  rows = z.numel() // k
  out = torch.empty(z.shape[:-1], device=z.device, dtype=torch.int32)
  z = z.contiguous()  # bound to a local: the pointer must outlive the enqueue
  check(_lib.lib().iic_argmax_rows(_p(z), rows, k, _p(out), _stream()), "iic_argmax_rows")
  return out


def argmax_channels(x):
  """x [n, k, h, w] fp32 -> int32 [n, h, w]: torch.argmax(dim=1) semantics."""
  assert x.dtype == torch.float32 and x.dim() == 4
  n, k, h, w = x.shape
  out = torch.empty((n, h, w), device=x.device, dtype=torch.int32)
  x = x.contiguous()
  check(_lib.lib().iic_argmax_channels(_p(x), n, k, h * w, _p(out), _stream()), "iic_argmax_channels")
  return out


def confusion_counts(preds, targets, preds_k, targets_k, mask=None, counts=None):
  """preds [S, n] (or [n]) int32, targets [n] int32, mask [n] uint8 | None -> counts [S, preds_k, targets_k] int64
  (accumulated into `counts` if given)."""
  if preds.dim() == 1:
    preds = preds.unsqueeze(0)
  S, n = preds.shape
  assert preds.dtype == torch.int32 and targets.dtype == torch.int32 and targets.shape == (n,)
  assert mask is None or (mask.dtype == torch.uint8 and mask.shape == (n,))
  acc = counts is not None
  if counts is None:
    counts = torch.empty((S, preds_k, targets_k), device=preds.device, dtype=torch.int64)
  assert counts.shape == (S, preds_k, targets_k) and counts.dtype == torch.int64
  preds, targets = preds.contiguous(), targets.contiguous()
  check(_lib.lib().iic_confusion_counts(_p(preds), _p(targets), _p(mask), S, n, preds_k,
                                        targets_k, _p(counts), int(acc), _stream()), "iic_confusion_counts")
  return counts
