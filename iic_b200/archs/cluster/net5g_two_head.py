"""ClusterNet5gTwoHead -- drop-in for code/archs/cluster/net5g_two_head.py:11-81."""
import torch.nn as nn

from .. import _engine as E
from .net5g import ClusterNet5gTrunk
from .residual import BasicBlock, ResNet

__all__ = ["ClusterNet5gTwoHead"]


class ClusterNet5gTwoHeadHead(E.SubHeads):
  def __init__(self, config, output_k, semisup=False):
    nfeat = 512 * BasicBlock.expansion
    super().__init__(nfeat, output_k, 0 if semisup else config.num_sub_heads)
    self.batchnorm_track = config.batchnorm_track
    self.semisup = semisup
    if semisup:
      del self.heads
      self.head = E.LinearParams(nfeat, output_k)

  def forward(self, x, kmeans_use_features=False):
    if not self.semisup:
      return super().forward(x, kmeans_use_features=kmeans_use_features)
    return E.LinearFunction.apply(x, self.head.weight, self.head.bias)  # logits, no softmax (the loss is cross-entropy)


class ClusterNet5gTwoHead(ResNet):
  def __init__(self, config):
    super().__init__()
    self.batchnorm_track = config.batchnorm_track
    self.trunk = ClusterNet5gTrunk(config)
    self.head_A = ClusterNet5gTwoHeadHead(config, output_k=config.output_k_A)
    semisup = (hasattr(config, "semisup") and config.semisup)
    self.head_B = ClusterNet5gTwoHeadHead(config, output_k=config.output_k_B, semisup=semisup)
    self._initialize_weights()

  def forward(self, x, head="B", kmeans_use_features=False, trunk_features=False, penultimate_features=False):
    # default is "B" for use by eval code; the training script switches between A and B
    x = self.trunk(x, penultimate_features=penultimate_features)
    if trunk_features:  # for semisup
      return x
    if head == "A":
      x = self.head_A(x, kmeans_use_features=kmeans_use_features)
    elif head == "B":
      x = self.head_B(x, kmeans_use_features=kmeans_use_features)
    else:
      assert (False)
    return x

  def forward_stacked(self, x, head="B"):
    """Same as forward but returns the [S, bn, k] tensor (no unbind) for IID_loss_subheads."""
    feat = self.trunk(x)
    return (self.head_A if head == "A" else self.head_B).forward_stacked(feat)

  def forward_stacked_pair(self, x, x_tf, head="B"):
    """Both views in ONE pass through the trunk (BatchNorm statistics per view, identical to two
    forward calls); returns the two [S, bn, k] softmax stacks."""
    import torch
    n = x.shape[0]
    feat = self.trunk(torch.cat([x, x_tf], dim=0), groups=2)
    z = (self.head_A if head == "A" else self.head_B).forward_stacked(feat)  # [S, 2n, k]
    return z[:, :n], z[:, n:]
