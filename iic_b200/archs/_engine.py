"""Execution engine shared by the iic_b200 networks.

The nn.Module classes in this package hold parameters under the SAME state_dict
keys / shapes as the reference (so its checkpoints load), but never call a
torch op to compute: ``forward`` hands raw device pointers to the sm_100a
kernels of libiic_b200.so, and one ``torch.autograd.Function`` per trunk /
head group runs the hand-written backward.

Precision modes (``net.precision``):
  "bf16" (default): NHWC bf16 activations, tcgen05 bf16 MMA with fp32 TMEM accumulation;
                    BN statistics, parameters, heads and losses stay fp32.
  "tf32":           NHWC fp32 activations, tcgen05 kind::tf32 convolutions (conv_tf32.cu).
  "tf32x3":         the same kernel with the 3xTF32 error-compensated operand split: fp32-grade results from the
                    tensor cores -- the mode that meets the fp32 tolerance of the reference (DESIGN.md S4).
  "fp32":           NHWC fp32 activations, fp32 SIMT convolutions (reference precision; slow, the on-device checker).
"""
import math

import os

import torch
import torch.nn as nn

from .. import kernels as K
from .._lib import BF16, F32, TF32, TF32X3

# precision -> (storage dtype of the activations, compute mode of the convolutions)
_PRECISIONS = {"bf16": (BF16, BF16), "fp32": (F32, F32), "tf32": (F32, TF32), "tf32x3": (F32, TF32X3)}


# ---------------------------------------------------------------------------------------------
# parameter containers (state_dict-compatible with nn.Conv2d / nn.BatchNorm2d / nn.Linear)
# ---------------------------------------------------------------------------------------------
class ConvParams(nn.Module):
  """Holds ``weight`` [cout, cin, kh, kw] like nn.Conv2d(bias=False); no forward."""

  def __init__(self, cin, cout, ksize, stride=1, padding=0, dilation=1):
    super().__init__()
    self.cin, self.cout, self.ksize, self.stride, self.padding, self.dilation = cin, cout, ksize, stride, padding, dilation
    self.weight = nn.Parameter(torch.empty(cout, cin, ksize, ksize))

  def geom(self, n, h, w):
    return K.conv_geom(n, h, w, self.cin, self.cout, self.ksize, self.ksize, self.stride, self.padding, self.dilation)

  def extra_repr(self):
    return "%d, %d, kernel_size=%d, stride=%d, padding=%d, dilation=%d" % (
      self.cin, self.cout, self.ksize, self.stride, self.padding, self.dilation)


class BNParams(nn.Module):
  """Holds weight/bias (+ running stats when tracking) like nn.BatchNorm2d; no forward."""

  def __init__(self, c, track_running_stats=True, eps=1e-5, momentum=0.1):
    super().__init__()
    self.num_features, self.eps, self.momentum = c, eps, momentum
    self.track_running_stats = track_running_stats
    self.weight = nn.Parameter(torch.ones(c))
    self.bias = nn.Parameter(torch.zeros(c))
    if track_running_stats:
      self.register_buffer("running_mean", torch.zeros(c))
      self.register_buffer("running_var", torch.ones(c))
      self.register_buffer("num_batches_tracked", torch.tensor(0, dtype=torch.long))
    else:
      self.register_buffer("running_mean", None)
      self.register_buffer("running_var", None)
      self.register_buffer("num_batches_tracked", None)


class LinearParams(nn.Module):
  def __init__(self, fin, fout):
    super().__init__()
    self.in_features, self.out_features = fin, fout
    self.weight = nn.Parameter(torch.empty(fout, fin))
    self.bias = nn.Parameter(torch.empty(fout))


class Identity(nn.Module):
  """Placeholder keeping Sequential indices identical to the reference (e.g. the Softmax at
  heads.{i}.1, the ReLU / MaxPool entries of the VGG ``features`` list)."""


def init_conv_kaiming(w, mode):
  # nn.init.kaiming_normal_(w, mode=mode, nonlinearity='relu') -- residual.py:77-78, vgg.py:45
  cout, cin, kh, kw = w.shape
  fan = (cout if mode == "fan_out" else cin) * kh * kw
  with torch.no_grad():
    w.normal_(0, math.sqrt(2.0 / fan))


def initialize_weights(net, mode):
  """residual.py:75-85 (mode fan_out) / vgg.py:42-54 (mode fan_in)."""
  for m in net.modules():
    if isinstance(m, ConvParams):
      init_conv_kaiming(m.weight, mode)
    elif isinstance(m, BNParams):
      assert m.track_running_stats == net.batchnorm_track
      m.weight.data.fill_(1)
      m.bias.data.zero_()
    elif isinstance(m, LinearParams):
      m.weight.data.normal_(0, 0.01)
      m.bias.data.zero_()


# ---------------------------------------------------------------------------------------------
# forward / backward building blocks (all activations NHWC)
# ---------------------------------------------------------------------------------------------
class _Ctx(object):
  """Per-forward record of what backward needs."""

  def __init__(self, dt, training, need_grad, groups=1, cdt=None):
    self.dt, self.training, self.need_grad = dt, training, need_grad
    self.cdt = dt if cdt is None else cdt  # compute mode of the convolutions (TF32 / TF32X3 on F32 storage)
    # groups > 1: the batch is the concatenation of `groups` views (x, x_tf) pushed through the trunk in
    # ONE pass; BatchNorm statistics stay per view, exactly as in the reference's two separate forward
    # calls (cluster_sobel_twohead.py:320-321), everything else sees one batch of groups*n images.
    self.groups = groups
    self.saved = []
    self.wcache = {}
    self.mbits = {}  # id(block output) -> its ReLU mask as bits (option bn_bitmask)
    self.nbt = {}    # num_batches_tracked buffers to advance, by increment: one multi-tensor add per forward

  def count_batch(self, bn, k):
    """nn.BatchNorm2d's `num_batches_tracked += 1` per forward call, deferred: 72 one-element add kernels per step of
    ClusterNet5g become one `torch._foreach_add_`."""
    inc = self.nbt.setdefault(id(bn), [bn.num_batches_tracked, 0])
    inc[1] += k

  def flush_batch_counts(self):
    by_k = {}
    for t, k in self.nbt.values():
      by_k.setdefault(k, []).append(t)
    for k, ts in by_k.items():
      torch._foreach_add_(ts, k)
    self.nbt = {}

  def split(self, t):
    if t is None:
      return [None] * self.groups
    if self.groups == 1:
      return [t]
    n = t.shape[0] // self.groups
    return [t[i * n:(i + 1) * n] for i in range(self.groups)]

  def packed(self, conv, kind):
    key = (id(conv), kind)
    if key not in self.wcache:
      self.wcache[key] = K.pack_weight(conv.weight.detach(), K.weight_dtype(self.dt, self.cdt), kind)
    return self.wcache[key]


class _ViewStats(list):
  """Per-view [2C] coefficient tensors that are rows of one contiguous [views, 2C] tensor (`stacked`), so the
  multi-view kernels take one base pointer."""

  def __init__(self, stacked):
    super(_ViewStats, self).__init__(stacked[i] for i in range(stacked.shape[0]))
    self.stacked = stacked


# Host-side variant switches (A/B measurement; defaults from the environment, tests may flip them in place):
#   bn_merged    one launch per BatchNorm pass for all views (0: one launch chain per view, the first implementation)
#   stem_stats   BatchNorm statistics of the stem accumulated inside the stem conv kernel (0: separate pass over y)
#   pack_batched all tensor-core weight layouts of a trunk repacked by one launch (0: one launch per conv and layout)
#   stem_bwd_fused  backward of the 5g stem (conv3x3 -> BN -> ReLU -> MaxPool) in two passes over (y, dpool) instead of
#                max-pool backward, BatchNorm backward and stem wgrad as separate passes.  Correct (tests) but OFF by
#                default: its first version is latency bound (7.6 ms against 4.4 ms for the chain at the bench shape,
#                profiles/r01_bench_v10_variants.md)
#   bn_bitmask   the ReLU of a residual block's output is kept as a 1-bit mask by the forward apply and read by the bn2
#                backward instead of the block output (16 -> 12.25 B per element).  Validated on a B200 in round 2;
#                on the final build of the round: bn_bwd 8.66 -> 7.81 ms, bn_apply 2.76 -> 3.02 ms, c4 step
#                40.50 / 40.30 -> 39.63 / 39.29 ms (profiles/r02_session_j.md): ON
OPTIONS = {
  "bn_merged": os.environ.get("IIC_BN_MERGED", "1") != "0",
  "stem_stats": os.environ.get("IIC_STEM_STATS", "1") != "0",
  "pack_batched": os.environ.get("IIC_PACK_BATCHED", "1") != "0",
  "stem_bwd_fused": os.environ.get("IIC_STEM_BWD_FUSED", "0") != "0",
  "bn_bitmask": os.environ.get("IIC_BN_BITMASK", "1") != "0",
  # wgrad_stream: weight-gradient convolutions run on a second stream.  A wgrad depends on (x, dy) only and nothing in
  # the backward depends on it, while the critical chain alternates tensor-bound dgrads with HBM-bound BatchNorm passes:
  # with the dgrad enqueued first, the (persistent, one CTA per SM) wgrad starts when the dgrad drains and then shares the
  # SMs with the BatchNorm backward of the next stage (tensor pipe + HBM busy at the same time).  Needs BatchNorm kernels
  # that fit beside a resident conv CTA: library option bn_bwd_ctas = 1.
  "wgrad_stream": os.environ.get("IIC_WGRAD_STREAM", "0") != "0",
  # masked_addend (needs bn_bitmask): the bn2 backward of a residual block does not write d_out * (out > 0) for the residual
  # branch; conv1's dgrad epilogue (iic_conv_dgrad_masked) or the downsample BatchNorm backward read d_out and the mask bits.
  # 3.1 GB less written per c4 step.  Validated on a B200 in round 2 (bit-identical block backward in 45 kernel / option
  # combinations, step / precision / net suites and smoke green with it; bn_bwd 7.95 -> 7.50 ms, profiles/r02_session_k.md).
  "masked_addend": os.environ.get("IIC_MASKED_ADDEND", "1") != "0",
  # stem_bwd_dy: max-pool routing + ReLU + BatchNorm backward of the 5g stem in two passes over (y, dpool) that write dy for
  # the (tensor-core) stem wgrad: the routed gradient and the BatchNorm reduce sweep never touch memory (7.5 GB instead of
  # 13.7 GB at the c4 shape).  The first two passes of stem_bwd_fused, whose SIMT wgrad pass was what made it slow.
  # Written after the last GPU session: off until it has run on hardware.
  "stem_bwd_dy": os.environ.get("IIC_STEM_BWD_DY", "0") != "0",
}
_WSTREAMS = {}


def _wgrad_stream(device):
  s = _WSTREAMS.get(device)
  if s is None:
    s = _WSTREAMS[device] = torch.cuda.Stream(device=device)
  return s


def _bn_stats(ctx, bn, y):
  """Per-view batch statistics -> ([scale_shift per view], [mean_invstd per view])."""
  use_running = (not ctx.training) and bn.track_running_stats
  update = ctx.training and bn.track_running_stats
  rm = bn.running_mean if (update or use_running) else None
  rv = bn.running_var if (update or use_running) else None
  C = y.shape[-1]
  sss = _ViewStats(torch.empty((ctx.groups, 2 * C), device=y.device, dtype=torch.float32))
  mis = _ViewStats(torch.empty((ctx.groups, 2 * C), device=y.device, dtype=torch.float32))
  for yg, ss, mi in zip(ctx.split(y), sss, mis):  # running statistics are updated view by view, in call order
    if update:
      ctx.count_batch(bn, 1)
    K.bn_stats(yg, bn.weight.detach(), bn.bias.detach(), bn.eps, bn.momentum, rm, rv, use_running, ss=ss, mi=mi)
  return sss, mis


def _conv_bn(ctx, conv, bn, x, g):
  """y = conv(x) and the per-view BN statistics of y.  On the tensor-core path in training mode the
  statistics are accumulated in the conv epilogue (no separate pass over y)."""
  fused = None
  if ctx.dt == BF16 and (ctx.training or not bn.track_running_stats):
    fused = K.conv_fprop_stats(x, ctx.packed(conv, 0), g, ctx.dt, ctx.groups)
  if fused is None:
    y = K.conv_fprop(x, ctx.packed(conv, 0), g, ctx.cdt)
    ss, mi = _bn_stats(ctx, bn, y)
    return y, ss, mi
  y, partial, nblk = fused
  ss, mi = _stats_from_partials(ctx, bn, y, partial, nblk)
  return y, ss, mi


def _stats_from_partials(ctx, bn, y, partial, nblk):
  """Per-CTA partial sums written by a producing kernel's epilogue -> per-view scale/shift and mean/invstd."""
  update = ctx.training and bn.track_running_stats
  rm = bn.running_mean if update else None
  rv = bn.running_var if update else None
  M = (y.numel() // y.shape[-1]) // ctx.groups
  if OPTIONS["bn_merged"]:
    if update:
      ctx.count_batch(bn, ctx.groups)
    ss, mi = K.bn_stats_from_partials_views(partial, nblk, 2, ctx.groups, M, bn.weight.detach(), bn.bias.detach(),
                                            bn.eps, bn.momentum, rm, rv)
    return _ViewStats(ss), _ViewStats(mi)
  sss, mis = [], []
  for v in range(ctx.groups):
    if update:
      ctx.count_batch(bn, 1)
    ss, mi = K.bn_stats_from_partials(partial, nblk, 2, v, M, bn.weight.detach(), bn.bias.detach(), bn.eps,
                                      bn.momentum, rm, rv)
    sss.append(ss)
    mis.append(mi)
  return sss, mis


def _bn_apply_block_out(ctx, y, ss, res, rss=None):
  """relu(bn2(y) + residual) of a BasicBlock; with `bn_bitmask` the ReLU mask is also kept as bits for the backward."""
  if (OPTIONS["bn_bitmask"] and OPTIONS["bn_merged"] and ctx.need_grad and ctx.groups <= 2 and hasattr(ss, "stacked")
      and (rss is None or hasattr(rss, "stacked"))):
    out, mbits = K.bn_apply_views_mask(y, ss.stacked, ctx.groups, res=res, rss=None if rss is None else rss.stacked)
    ctx.mbits[id(out)] = mbits
    return out
  return _bn_apply(ctx, y, ss, True, res=res, rss=rss)


def _bn_apply(ctx, y, ss, relu, res=None, rss=None):
  out = torch.empty_like(y)
  if OPTIONS["bn_merged"] and hasattr(ss, "stacked") and (rss is None or hasattr(rss, "stacked")):
    return K.bn_apply_views(y, ss.stacked, relu, ctx.groups, res=res, rss=None if rss is None else rss.stacked, out=out)
  for yg, og, sg, rg, rsg in zip(ctx.split(y), ctx.split(out), ss, ctx.split(res), rss if rss is not None else [None] * ctx.groups):
    K.bn_apply(yg, sg, relu, res=rg, rss=rsg, out=og)
  return out


def _bn_relu_maxpool(ctx, y, ss, pad):
  shape = K.pooled_shape(y, pad)
  out = torch.empty(shape, device=y.device, dtype=y.dtype)
  for yg, og, sg in zip(ctx.split(y), ctx.split(out), ss):
    K.bn_relu_maxpool(yg, sg, pad, out=og)
  return out


def _bn_relu_maxpool_bwd(ctx, y, ss, dpool, pad):
  g = torch.empty_like(y)
  for yg, gg, sg, dg in zip(ctx.split(y), ctx.split(g), ss, ctx.split(dpool)):
    K.bn_relu_maxpool_bwd(yg, sg, dg, pad, out=gg)
  return g


class GradSink(object):
  """Collects parameter gradients produced by a trunk backward, keyed by parameter object.

  A parameter whose ``.grad`` is a view of a ``GradArena`` (iic_b200/arena.py) is accumulated in place -- the kernels
  add into the arena, autograd gets ``None`` for it -- and reported to the arena once the kernels of the current
  backward record are enqueued (``commit``), which is what lets the arena all-reduce a bucket while the backward of
  the earlier layers is still running."""

  def __init__(self):
    self.g = {}
    self.direct = {}
    self._touched = []
    self.wstream = None  # side stream that produced some of the gradients (OPTIONS["wgrad_stream"])

  def buf(self, p):
    if id(p) in self.direct:
      return p.grad, True
    if id(p) not in self.g:
      arena = getattr(p, "_iic_arena", None)
      if arena is not None and arena.holds(p):
        self.direct[id(p)] = arena
        self._touched.append(p)
        return p.grad, True
      self.g[id(p)] = torch.empty_like(p, dtype=torch.float32)
      return self.g[id(p)], False
    return self.g[id(p)], True

  def commit(self):
    for p in self._touched:
      self.direct[id(p)].mark(p, producer=self.wstream)
    self._touched = []

  def get(self, p):
    return None if id(p) in self.direct else self.g.get(id(p))


def _bn_backward(ctx, sink, bn, g_in, act, y, mi, want_g_out, mask_ss=None):
  """act: activation whose sign is the ReLU mask (residual blocks); mask_ss: per-view scale/shift when the
  ReLU directly follows the BN (the mask is then recomputed from y instead of reading the activation)."""
  dg, acc1 = sink.buf(bn.weight)
  db, acc2 = sink.buf(bn.bias)
  assert acc1 == acc2
  if OPTIONS["bn_merged"] and ctx.groups <= 2:
    return K.bn_bwd_fused(g_in, act, y, mi, bn.weight.detach(), dg, db, acc1, want_g_out, mask_sss=mask_ss)
  dy = torch.empty_like(y)
  g_out = torch.empty_like(y) if want_g_out else None
  acc = acc1
  mss = mask_ss if mask_ss is not None else [None] * ctx.groups
  for gg, ag, yg, mg, dyg, gog, ms in zip(ctx.split(g_in), ctx.split(act), ctx.split(y), mi, ctx.split(dy),
                                          ctx.split(g_out), mss):
    K.bn_bwd(gg, ag, yg, mg, bn.weight.detach(), dg, db, acc, want_g_out, dy=dyg, g_out=gog, mask_ss=ms)
    acc = True  # later views add to the same dgamma / dbeta
  return dy, g_out


def _conv_wgrad(ctx, sink, conv, x, dy, g):
  gw, acc = sink.buf(conv.weight)
  if not (OPTIONS["wgrad_stream"] and x.is_cuda):
    K.conv_wgrad(x, dy, g, ctx.cdt, gw, acc)
    return
  cur = torch.cuda.current_stream(x.device)
  ws = _wgrad_stream(x.device)
  ws.wait_stream(cur)  # x, dy (and the gradient buffer's previous contents) are ready on the compute stream
  with torch.cuda.stream(ws):
    K.conv_wgrad(x, dy, g, ctx.cdt, gw, acc)
  for t in (x, dy, gw):
    t.record_stream(ws)  # the allocator must not hand this memory out again before the side stream is done with it
  sink.wstream = ws


# ---- stem: conv(NCHW input) + BN + ReLU [+ MaxPool(2,2,pad)] -----------------------------------
def stem_forward(ctx, conv, bn, x_nchw, pool_pad):
  n, c, h, w = x_nchw.shape
  g = conv.geom(n, h, w)
  fused = None
  if OPTIONS["stem_stats"] and ctx.dt == BF16 and (ctx.training or not bn.track_running_stats):
    # statistics in the conv kernel, like _conv_bn
    fused = K.stem_fprop_stats(x_nchw, conv.weight.detach(), g, ctx.dt, ctx.groups)
  if fused is None:
    y = K.stem_fprop(x_nchw, conv.weight.detach(), g, ctx.dt)
    ss, mi = _bn_stats(ctx, bn, y)
  else:
    y, partial, nblk = fused
    ss, mi = _stats_from_partials(ctx, bn, y, partial, nblk)
  out = _bn_relu_maxpool(ctx, y, ss, pool_pad) if pool_pad is not None else _bn_apply(ctx, y, ss, True)
  if ctx.need_grad:
    ctx.saved.append(("stem", conv, bn, x_nchw, g, y, ss, mi, None, pool_pad))
  return out


def stem_backward(ctx, sink, rec, d_out):
  _, conv, bn, x_nchw, g, y, ss, mi, act, pool_pad = rec
  if (pool_pad is not None and OPTIONS["stem_bwd_fused"] and hasattr(ss, "stacked") and hasattr(mi, "stacked")
      and d_out.is_contiguous() and K.stem_bwd_fused_workspace(g, pool_pad, ss.stacked.shape[0], ctx.dt) > 0):
    dg, acc1 = sink.buf(bn.weight)
    db, acc2 = sink.buf(bn.bias)
    gw, accw = sink.buf(conv.weight)
    assert acc1 == acc2
    done = K.stem_bwd_fused(x_nchw, y, d_out, ss.stacked, mi.stacked, bn.weight.detach(), dg, db, acc1, gw, accw, g,
                            pool_pad, ctx.dt)
    assert done
    return None
  dy = None
  if (pool_pad is not None and OPTIONS["stem_bwd_dy"] and hasattr(ss, "stacked") and hasattr(mi, "stacked")
      and d_out.is_contiguous() and K.stem_bwd_fused_workspace(g, pool_pad, ss.stacked.shape[0], ctx.dt) > 0):
    dg, acc1 = sink.buf(bn.weight)
    db, acc2 = sink.buf(bn.bias)
    assert acc1 == acc2
    dy = K.stem_bwd_dy(y, d_out, ss.stacked, mi.stacked, bn.weight.detach(), dg, db, acc1, g, pool_pad, ctx.dt)
  if dy is None:
    if pool_pad is not None:
      gmask = _bn_relu_maxpool_bwd(ctx, y, ss, d_out, pool_pad)
      dy, _ = _bn_backward(ctx, sink, bn, gmask, None, y, mi, False)
    else:
      dy, _ = _bn_backward(ctx, sink, bn, d_out, None, y, mi, False, mask_ss=ss)
  gw, acc = sink.buf(conv.weight)
  K.stem_wgrad(x_nchw, dy, g, ctx.dt, gw, acc)
  return None


# ---- VGG unit: conv + BN + ReLU [+ MaxPool(2,2)] (vgg.py:8-35) -----------------------------------
def convbn_forward(ctx, conv, bn, x, pool_pad):
  n, h, w, _ = x.shape
  g = conv.geom(n, h, w)
  y, ss, mi = _conv_bn(ctx, conv, bn, x, g)
  out = _bn_relu_maxpool(ctx, y, ss, pool_pad) if pool_pad is not None else _bn_apply(ctx, y, ss, True)
  if ctx.need_grad:
    ctx.saved.append(("convbn", conv, bn, x, g, y, ss, mi, None, pool_pad))
  return out


def convbn_backward(ctx, sink, rec, d_out):
  _, conv, bn, x, g, y, ss, mi, act, pool_pad = rec
  if pool_pad is not None:
    gmask = _bn_relu_maxpool_bwd(ctx, y, ss, d_out, pool_pad)
    dy, _ = _bn_backward(ctx, sink, bn, gmask, None, y, mi, False)
  else:
    dy, _ = _bn_backward(ctx, sink, bn, d_out, None, y, mi, False, mask_ss=ss)
  dx = K.conv_dgrad(dy, ctx.packed(conv, 1), g, ctx.cdt)
  _conv_wgrad(ctx, sink, conv, x, dy, g)
  return dx


# ---- residual BasicBlock (residual.py:10-43) -----------------------------------------------------
def block_forward(ctx, blk, x):
  n, h, w, _ = x.shape
  g1 = blk.conv1.geom(n, h, w)
  y1, ss1, mi1 = _conv_bn(ctx, blk.conv1, blk.bn1, x, g1)
  a1 = _bn_apply(ctx, y1, ss1, True)
  g2 = blk.conv2.geom(n, g1.oh, g1.ow)
  y2, ss2, mi2 = _conv_bn(ctx, blk.conv2, blk.bn2, a1, g2)
  if blk.downsample is not None:
    dconv, dbn = blk.downsample[0], blk.downsample[1]
    gd = dconv.geom(n, h, w)
    yd, ssd, mid = _conv_bn(ctx, dconv, dbn, x, gd)
    out = _bn_apply_block_out(ctx, y2, ss2, yd, ssd)
  else:
    gd = yd = mid = None
    out = _bn_apply_block_out(ctx, y2, ss2, x)
  if ctx.need_grad:
    ctx.saved.append(("block", blk, x, g1, y1, mi1, a1, g2, y2, mi2, gd, yd, mid, out, ss1))
  return out


def block_backward(ctx, sink, rec, d_out):
  _, blk, x, g1, y1, mi1, a1, g2, y2, mi2, gd, yd, mid, out, ss1 = rec
  # out = relu(bn2(y2) + r): g = d_out * (out > 0) goes both into bn2 and the residual branch
  mbits = ctx.mbits.get(id(out))
  # masked_addend: the masked copy of d_out for the residual branch is never written -- its consumers (the dgrad epilogue of
  # conv1, or the BatchNorm backward of the downsample branch) apply the mask bits to d_out themselves
  lazy = mbits is not None and OPTIONS["masked_addend"] and ctx.cdt == K.BF16  # (iic_conv_dgrad_masked: bf16 tensor cores)
  if mbits is not None:
    dg, acc1 = sink.buf(blk.bn2.weight)
    db, acc2 = sink.buf(blk.bn2.bias)
    assert acc1 == acc2
    dy2, gres = K.bn_bwd_fused_bits(d_out, mbits, y2, mi2, blk.bn2.weight.detach(), dg, db, acc1, not lazy)
  else:
    dy2, gres = _bn_backward(ctx, sink, blk.bn2, d_out, out, y2, mi2, True)
  # (the dgrad -- critical path -- is enqueued before the wgrad of the same layer: with OPTIONS["wgrad_stream"] the wgrad
  # then starts when the dgrad drains and overlaps the BatchNorm backward that follows)
  da1 = K.conv_dgrad(dy2, ctx.packed(blk.conv2, 1), g2, ctx.cdt)
  _conv_wgrad(ctx, sink, blk.conv2, a1, dy2, g2)
  dy1, _ = _bn_backward(ctx, sink, blk.bn1, da1, None, y1, mi1, False, mask_ss=ss1)  # a1 = relu(bn1(y1))
  if blk.downsample is not None:
    dconv, dbn = blk.downsample[0], blk.downsample[1]
    if lazy:
      dgd, accd1 = sink.buf(dbn.weight)
      dbd, accd2 = sink.buf(dbn.bias)
      assert accd1 == accd2
      dyd, _ = K.bn_bwd_fused_bits(d_out, mbits, yd, mid, dbn.weight.detach(), dgd, dbd, accd1, False)
    else:
      dyd, _ = _bn_backward(ctx, sink, dbn, gres, None, yd, mid, False)
    dxd = K.conv_dgrad(dyd, ctx.packed(dconv, 1), gd, ctx.cdt)
    dx = K.conv_dgrad(dy1, ctx.packed(blk.conv1, 1), g1, ctx.cdt, addend=dxd)
    _conv_wgrad(ctx, sink, dconv, x, dyd, gd)
    _conv_wgrad(ctx, sink, blk.conv1, x, dy1, g1)
    return dx
  if lazy:
    dx = K.conv_dgrad(dy1, ctx.packed(blk.conv1, 1), g1, ctx.cdt, addend=d_out, addend_mask=mbits)
  else:
    dx = K.conv_dgrad(dy1, ctx.packed(blk.conv1, 1), g1, ctx.cdt, addend=gres)
  _conv_wgrad(ctx, sink, blk.conv1, x, dy1, g1)
  return dx


def _prepack(trunk, ectx):
  """All tensor-core weight layouts of the trunk (fprop, and dgrad when a backward follows) in one launch.  The
  job table and the destination buffers persist on the module; they are rebuilt if a weight was re-allocated."""
  if not OPTIONS["pack_batched"]:
    return
  convs = [m for m in trunk.modules() if isinstance(m, ConvParams) and m.cin % 8 == 0]  # (the stem reads fp32 weights)
  if not convs:
    return
  weights = [c.weight.detach() for c in convs]
  kinds = (0, 1) if ectx.need_grad else (0,)
  wdt = K.weight_dtype(ectx.dt, ectx.cdt)
  key = K.PackPlan.make_key(weights, kinds, wdt)
  plans = trunk.__dict__.setdefault("_iic_pack_plans", {})
  plan = plans.get((kinds, wdt))
  if plan is None or plan.key != key:
    plan = plans[(kinds, wdt)] = K.PackPlan(weights, kinds, wdt)
  out = plan.run()
  for wi, c in enumerate(convs):
    for kind in kinds:
      ectx.wcache[(id(c), kind)] = out[(wi, kind)]


_BACKWARD = {"stem": stem_backward, "convbn": convbn_backward, "block": block_backward}


class TrunkFunction(torch.autograd.Function):
  """x (NCHW fp32, no grad) -> trunk feature (fp32).  ``run(ctx_, x)`` executes the forward plan
  and returns (feature, finisher) where finisher maps d_feature -> gradient w.r.t. the last
  NHWC activation."""

  @staticmethod
  def forward(ctx, trunk, run, need_grad, groups, x, *params):
    ectx = _Ctx(_PRECISIONS[trunk.precision][0], trunk.training, need_grad, groups, cdt=_PRECISIONS[trunk.precision][1])
    # the packed dgrad weights live in per-module buffers that the next forward overwrites: remember the versions
    ectx.wversions = [(p, p._version) for p in params if p.dim() == 4] if need_grad else []
    _prepack(trunk, ectx)
    feat, finisher = run(ectx, x)
    ectx.flush_batch_counts()
    ctx.ectx, ctx.finisher, ctx.params = ectx, finisher, params
    return feat

  @staticmethod
  def backward(ctx, dfeat):
    ectx = ctx.ectx
    if ectx.saved is None:
      raise RuntimeError("iic_b200: this trunk forward has already been differentiated once; its saved activations "
                         "were released (retain_graph / double backward are not supported -- run the forward again)")
    for p, v in ectx.wversions:
      if p._version != v:
        raise RuntimeError("iic_b200: a convolution weight was modified in place between this forward and its backward; "
                           "the packed tensor-core copies of the weights belong to the old values (run forward -> "
                           "backward -> optimiser.step() in that order)")
    sink = GradSink()
    d = ctx.finisher(dfeat)
    for rec in reversed(ectx.saved):
      d = _BACKWARD[rec[0]](ectx, sink, rec, d)
      sink.commit()
    if sink.wstream is not None:  # every weight gradient is complete before autograd / the optimiser sees it
      torch.cuda.current_stream(dfeat.device).wait_stream(sink.wstream)
    ectx.saved = None
    ectx.wcache = {}
    grads = tuple(sink.get(p) for p in ctx.params)
    return (None, None, None, None, None) + grads


def run_trunk(trunk, run, x, groups=1):
  if not x.is_cuda:
    raise RuntimeError("iic_b200 networks run on CUDA tensors only (no CPU fallback; the CPU restatement in "
                       "oracle/ is a test checker)")
  assert trunk.precision in _PRECISIONS, "precision must be one of %s" % sorted(_PRECISIONS)
  params = [p for p in trunk.parameters()]
  # (inside Function.forward grad mode is off and needs_input_grad ignores torch.no_grad())
  need_grad = torch.is_grad_enabled() and any(p.requires_grad for p in params)
  assert x.shape[0] % groups == 0
  return TrunkFunction.apply(trunk, run, need_grad, groups, x.detach().float().contiguous(), *params)


# ---------------------------------------------------------------------------------------------
# sub-heads: S x (Linear + Softmax)   (net5g_two_head.py:11-39)
# ---------------------------------------------------------------------------------------------
class HeadsFunction(torch.autograd.Function):
  @staticmethod
  def forward(ctx, feat, w, b, S, k):
    feat = feat.contiguous()
    z = K.heads_fwd(feat, w.contiguous(), b.contiguous(), S, k)
    ctx.save_for_backward(feat, w, z)
    ctx.S, ctx.k = S, k
    return z

  @staticmethod
  def backward(ctx, dz):
    feat, w, z = ctx.saved_tensors
    dw, db, dfeat = K.heads_bwd(feat, w.contiguous(), z, dz.contiguous(), ctx.S, ctx.k, ctx.needs_input_grad[0])
    return dfeat, dw, db, None, None


class LinearFunction(torch.autograd.Function):
  """nn.Linear (fp32) without an activation: the `semisup` head of the TwoHead nets (net5g_two_head.py:22-24) and the last
  Linear of SupHead5 (sup_head5.py:20) -- csrc/semisup.cu iic_linear_fwd / iic_linear_bwd."""

  @staticmethod
  def forward(ctx, x, w, b):
    if not x.is_cuda:
      raise RuntimeError("iic_b200 Linear heads run on CUDA tensors only (no CPU fallback)")
    x = x.float().contiguous()
    ctx.save_for_backward(x, w)
    return K.linear_fwd(x, w.contiguous(), b.contiguous())

  @staticmethod
  def backward(ctx, dy):
    x, w = ctx.saved_tensors
    dw = torch.empty_like(w)
    db = torch.empty(w.shape[0], device=w.device, dtype=torch.float32)
    dx = K.linear_bwd(x, w.contiguous(), dy.contiguous().float(), dw, db, False, ctx.needs_input_grad[0])
    return dx, dw, db


class SubHeads(nn.Module):
  """num_sub_heads x (Linear(F -> k) + Softmax(dim=1)); parameters live at
  ``heads.{i}.0.{weight,bias}`` exactly like the reference's nn.Sequential(Linear, Softmax)."""

  def __init__(self, nfeat, output_k, num_sub_heads):
    super().__init__()
    self.num_sub_heads, self.output_k, self.nfeat = num_sub_heads, output_k, nfeat
    self.heads = nn.ModuleList([nn.Sequential(LinearParams(nfeat, output_k), Identity())
                                for _ in range(num_sub_heads)])

  def forward_stacked(self, x):
    w = torch.cat([h[0].weight for h in self.heads], dim=0)
    b = torch.cat([h[0].bias for h in self.heads], dim=0)
    return HeadsFunction.apply(x, w, b, self.num_sub_heads, self.output_k)  # [S, bn, k]

  def forward(self, x, kmeans_use_features=False):
    if kmeans_use_features:
      return [x for _ in range(self.num_sub_heads)]  # duplicates (net5g_two_head.py:31-34)
    return list(self.forward_stacked(x).unbind(0))
