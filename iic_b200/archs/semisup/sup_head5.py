"""SupHead5 -- drop-in for code/archs/semisup/sup_head5.py:9-40: a clustering network's trunk features (512, or the
layer3 output with ``penultimate_features``) -> Linear(dlen, 2048) -> BatchNorm1d(2048) -> ReLU -> Linear(2048, gt_k), logits
without a softmax.

One ``torch.autograd.Function`` runs the head forward and backward (as HeadsFunction does for the sub-heads):
  * the first Linear is a 1x1 convolution over n images of 1x1 pixels on the convolution engine, in the trunk's precision
    mode (bf16: tcgen05 kind::f16; tf32 / tf32x3: kind::tf32; fp32: SIMT).  Its weight [2048][dlen] is the
    [cout][cin][1][1] layout of a convolution weight, so fprop / dgrad / wgrad are iic_conv_fprop / iic_conv_dgrad /
    iic_conv_wgrad_oihw unchanged;
  * BatchNorm1d(2048) + ReLU are the BatchNorm kernels with M = n rows and C = 2048 channels;
  * the first Linear's bias never enters the product: in train mode BatchNorm removes it, and it is folded into the
    running-mean update and the eval-mode shift instead (running_mean keeps torch's meaning, the mean of x W^T + b).  Its
    gradient is the batch sum of the BatchNorm input gradient (analytically zero), as autograd computes it;
  * the last Linear is iic_linear_fwd / iic_linear_bwd (fp32).
"""
import torch
import torch.nn as nn

from .. import _engine as E
from ... import kernels as K
from ..._lib import F32

__all__ = ["SupHead5"]

HIDDEN = 2048


class _SupHeadFunction(torch.autograd.Function):
  @staticmethod
  def forward(ctx, head, precision, training, feat, w1, b1, gamma, beta, w2, b2):
    if not feat.is_cuda:
      raise RuntimeError("iic_b200 SupHead5 runs on CUDA tensors only (no CPU fallback)")
    dt, cdt = E._PRECISIONS[precision]
    bn = head[1]
    n, dlen = feat.shape
    C = w1.shape[0]
    feat = feat.float().contiguous()
    x = (feat if dt == F32 else K.cast(feat, dt)).view(n, 1, 1, dlen)
    g = K.conv_geom(n, 1, 1, dlen, C, 1, 1, 1, 0, 1)
    wdt = K.weight_dtype(dt, cdt)
    w4 = w1.detach().view(C, dlen, 1, 1)
    use_running = (not training) and bn.track_running_stats
    update = training and bn.track_running_stats
    # running mean of the bias-free product x W^T: torch's running_mean minus the bias
    rm = torch.sub(bn.running_mean, b1.detach()) if (update or use_running) else None
    rv = bn.running_var if (update or use_running) else None
    # (no statistics fused into the convolution epilogue: its per-CTA partial buffer for 2048 channels would exceed the
    # shared memory of conv_tc2; the separate statistics pass reads a [n][2048] tensor)
    y = K.conv_fprop(x, K.pack_weight(w4, wdt, 0), g, cdt)
    ss, mi = K.bn_stats(y, gamma.detach(), beta.detach(), bn.eps, bn.momentum, rm, rv, use_running)
    if update:
      torch.add(rm, b1.detach(), out=bn.running_mean)
      bn.num_batches_tracked.add_(1)
    a = K.bn_apply(y, ss, True)
    a32 = a.view(n, C) if dt == F32 else K.cast(a, F32).view(n, C)
    logits = K.linear_fwd(a32, w2.detach().contiguous(), b2.detach().contiguous())
    ctx.save_for_backward(w1, w2)
    ctx.head_params = (head[0].weight, head[0].bias, head[1].weight, head[1].bias, head[3].weight, head[3].bias)
    ctx.inter = (x, y, ss, mi, a32, g, dt, cdt, wdt, training)
    return logits

  @staticmethod
  def backward(ctx, dlogits):
    if ctx.inter is None:
      raise RuntimeError("iic_b200: this SupHead5 forward has already been differentiated once (retain_graph / double "
                         "backward are not supported -- run the forward again)")
    w1, w2 = ctx.saved_tensors  # (raises if either weight was modified in place since the forward)
    x, y, ss, mi, a32, g, dt, cdt, wdt, training = ctx.inter
    ctx.inter = None
    if not training:
      raise RuntimeError("iic_b200 SupHead5: backward through an eval-mode forward is not supported")
    head = ctx.head_params
    w1p, b1p, gammap, betap, w2p, b2p = head
    ctx.head_params = None
    n, C = a32.shape
    sink = E.GradSink()
    dw2, acc = sink.buf(w2p)
    db2, acc2 = sink.buf(b2p)
    assert acc == acc2
    da = K.linear_bwd(a32, w2.detach().contiguous(), dlogits.contiguous().float(), dw2, db2, acc, True)
    da = (da if dt == F32 else K.cast(da, dt)).view(n, 1, 1, C)
    dgam, accg = sink.buf(gammap)
    dbet, accb = sink.buf(betap)
    assert accg == accb
    dy, _ = K.bn_bwd(da, None, y, mi, gammap.detach(), dgam, dbet, accg, False, mask_ss=ss)  # a = relu(bn(y))
    db1, acc1 = sink.buf(b1p)
    K.col_sum(dy, db1, acc1)
    gw1, accw = sink.buf(w1p)
    K.conv_wgrad(x, dy, g, cdt, gw1.view(C, -1, 1, 1), accw)
    dfeat = None
    if ctx.needs_input_grad[3]:
      dx = K.conv_dgrad(dy, K.pack_weight(w1.detach().view(C, -1, 1, 1), wdt, 1), g, cdt)
      dfeat = (dx if dt == F32 else K.cast(dx, F32)).view(n, -1)
    sink.commit()
    return (None, None, None, dfeat) + tuple(sink.get(p) for p in head)


class SupHead5(nn.Module):
  def __init__(self, net_features, dlen=None, gt_k=None):
    super().__init__()
    self.trunk = net_features
    # nn.Sequential(Linear(dlen, 2048), BatchNorm1d(2048), ReLU(), Linear(2048, gt_k)): same state_dict keys
    net_head = nn.Sequential(E.LinearParams(dlen, HIDDEN), E.BNParams(HIDDEN), E.Identity(), E.LinearParams(HIDDEN, gt_k))
    if torch.cuda.is_available():
      net_head.cuda()
    self.head = net_head
    for m in self.head.modules():
      if isinstance(m, E.BNParams):
        m.weight.data.fill_(1)
        m.bias.data.zero_()
      elif isinstance(m, E.LinearParams):
        m.weight.data.normal_(0, 0.01)
        m.bias.data.zero_()

  @property
  def precision(self):
    return self.trunk.trunk.precision

  def forward(self, x, penultimate_features=False):
    x = self.trunk(x, trunk_features=True, penultimate_features=penultimate_features)
    return self.forward_head(x)

  def forward_head(self, feat):
    """The head alone on trunk features [n, dlen] (fp32, CUDA): logits [n, gt_k]."""
    h = self.head
    return _SupHeadFunction.apply(h, self.precision, self.training, feat, h[0].weight, h[0].bias, h[1].weight, h[1].bias,
                                  h[3].weight, h[3].bias)
