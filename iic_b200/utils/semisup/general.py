"""Drop-in for xu-ji/IIC ``code/utils/semisup/general.py`` and the criterion of IID_semisup_STL10.py:201.

  get_dlen          :9-20    feature length from the trunk's geometry and the batch shape (the reference runs a CPU forward;
                             there is no CPU path here, and none is needed to count)
  assess_acc        :23-45   arg-max of the logits on the device (iic_argmax_rows), one host copy at the end
  assess_acc_block  :48-99   mean of every `contiguous_sz` consecutive rows (the ten crops of one test image) through
                             iic_avgpool, then iic_argmax_rows, one host copy at the end
  CrossEntropyLoss           nn.CrossEntropyLoss() with mean reduction on iic_cross_entropy (loss and gradient, one launch)
"""
import numpy as np
import torch
import torch.nn as nn

from ... import kernels
from ..cluster.transforms import sobel_process

__all__ = ["get_dlen", "assess_acc", "assess_acc_block", "CrossEntropyLoss"]


def _trunk_of(net_features):
  return getattr(net_features, "trunk", net_features)


def trunk_dlen(net_features, h, w, penultimate_features=False):
  """Length of the flattened trunk feature for inputs of h x w pixels."""
  from ...archs.cluster.net5g import ClusterNet5gTrunk
  from ...archs.cluster.net6c import ClusterNet6cTrunk
  trunk = _trunk_of(net_features)
  if isinstance(trunk, ClusterNet5gTrunk):
    if not penultimate_features:
      return 512
    # stem conv 3x3 / pad 1, MaxPool2d(2, 2, padding=1), then the stride-2 first blocks of layer2 and layer3 (3x3 / pad 1)
    h, w = h // 2 + 1, w // 2 + 1
    for _ in range(2):
      h, w = (h - 1) // 2 + 1, (w - 1) // 2 + 1
    return 256 * h * w
  if isinstance(trunk, ClusterNet6cTrunk):
    assert not penultimate_features, "penultimate_features: not needed/implemented for this arch"
    return 512 * (h // 8) * (w // 8)  # 5x5 / pad 2 convolutions, three MaxPool2d(2, 2)
  raise AssertionError("get_dlen: unsupported trunk %s" % type(trunk).__name__)


def get_dlen(net_features, dataloader, include_rgb=None, penultimate_features=False):
  for imgs, _ in dataloader:
    return trunk_dlen(net_features, imgs.shape[-2], imgs.shape[-1], penultimate_features=penultimate_features)
  raise AssertionError("get_dlen: empty dataloader")


def _logits(net, imgs, include_rgb, penultimate_features):
  imgs = sobel_process(imgs.cuda(), include_rgb)
  with torch.no_grad():
    x_out = net(imgs, penultimate_features=penultimate_features)
  assert x_out.dim() == 2 and x_out.dtype == torch.float32
  return x_out.contiguous()


def assess_acc(net, test_loader, gt_k=None, include_rgb=None, penultimate_features=False):
  preds, targets = [], []
  for imgs, t in test_loader:
    x_out = _logits(net, imgs, include_rgb, penultimate_features)
    assert x_out.shape[1] <= gt_k  # (the reference's preds.max() < gt_k)
    preds.append(kernels.argmax_rows(x_out))
    targets.append(np.asarray(t).astype("int"))
  preds = torch.cat(preds).cpu().numpy().astype("int")
  targets = np.concatenate(targets)
  assert (preds.min() >= 0 and preds.max() < gt_k)
  assert (targets.min() >= 0 and targets.max() < gt_k)
  assert (preds.shape == targets.shape)
  return (preds == targets).sum() / float(preds.shape[0])


def assess_acc_block(net, test_loader, gt_k=None, include_rgb=None, penultimate_features=False, contiguous_sz=None):
  outs, targets = [], []
  for imgs, t in test_loader:
    outs.append(_logits(net, imgs, include_rgb, penultimate_features))
    targets.append(np.asarray(t))
  all_out = torch.cat(outs) if len(outs) > 1 else outs[0]
  all_targets = np.concatenate(targets)
  total, dlen = all_out.shape
  num_orig, leftover = divmod(total, contiguous_sz)
  assert (leftover == 0)
  # mean over each run of contiguous_sz rows: AvgPool over "hw" = contiguous_sz, "C" = dlen
  avg = kernels.avgpool(all_out.view(num_orig, 1, contiguous_sz, dlen))
  preds = kernels.argmax_rows(avg).cpu().numpy().astype("int")
  all_targets = all_targets.reshape((num_orig, contiguous_sz))
  all_targets_avg = all_targets.astype("int").sum(axis=1) / contiguous_sz  # sanity check
  all_targets = all_targets[:, 0].astype("int")
  assert (np.array_equal(all_targets_avg, all_targets))
  assert (preds.min() >= 0 and preds.max() < gt_k)
  assert (all_targets.min() >= 0 and all_targets.max() < gt_k)
  assert (preds.shape == all_targets.shape == (num_orig,))
  correct = (preds == all_targets).sum()
  return correct / float(num_orig)


class _CrossEntropy(torch.autograd.Function):
  @staticmethod
  def forward(ctx, logits, target):
    loss, dlogits = kernels.cross_entropy(logits, target)
    ctx.save_for_backward(dlogits)
    return loss

  @staticmethod
  def backward(ctx, g):
    dlogits, = ctx.saved_tensors
    return dlogits * g, None


class CrossEntropyLoss(nn.Module):
  """nn.CrossEntropyLoss() as IID_semisup_STL10.py:201 builds it: no class weights, mean reduction.  A target outside
  [0, k) gives a NaN loss instead of a device assert."""

  def __init__(self, weight=None, size_average=None, ignore_index=-100, reduce=None, reduction="mean"):
    super().__init__()
    assert weight is None and size_average is None and reduce is None and reduction == "mean", \
      "iic_b200 CrossEntropyLoss: mean reduction without class weights only"
    self.ignore_index = ignore_index

  def forward(self, input, target):
    if not input.is_cuda:
      raise RuntimeError("iic_b200 CrossEntropyLoss: CUDA tensors only (no CPU fallback)")
    assert input.dim() == 2 and target.shape == (input.shape[0],)
    return _CrossEntropy.apply(input.float().contiguous(), target.to(input.device, torch.int64).contiguous())
