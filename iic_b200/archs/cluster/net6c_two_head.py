"""ClusterNet6cTwoHead -- drop-in for code/archs/cluster/net6c_two_head.py:9-98."""
from .. import _engine as E
from .net6c import ClusterNet6c, ClusterNet6cTrunk, _feat_size
from .vgg import VGGNet

__all__ = ["ClusterNet6cTwoHead"]


class ClusterNet6cTwoHeadHead(E.SubHeads):
  def __init__(self, config, output_k, semisup=False):
    nfeat = _feat_size(config, ClusterNet6c.cfg)
    super().__init__(nfeat, output_k, 0 if semisup else config.num_sub_heads)
    self.batchnorm_track = config.batchnorm_track
    self.cfg = ClusterNet6c.cfg
    self.semisup = semisup
    if semisup:
      del self.heads
      self.head = E.LinearParams(nfeat, output_k)

  def forward(self, x, kmeans_use_features=False):
    if not self.semisup:
      return super().forward(x, kmeans_use_features=kmeans_use_features)
    return E.LinearFunction.apply(x, self.head.weight, self.head.bias)  # logits, no softmax (the loss is cross-entropy)


class ClusterNet6cTwoHead(VGGNet):
  cfg = [(64, 1), ('M', None), (128, 1), ('M', None), (256, 1), ('M', None), (512, 1)]

  def __init__(self, config):
    super().__init__()
    self.batchnorm_track = config.batchnorm_track
    self.trunk = ClusterNet6cTrunk(config)
    self.head_A = ClusterNet6cTwoHeadHead(config, output_k=config.output_k_A)
    semisup = (hasattr(config, "semisup") and config.semisup)
    self.head_B = ClusterNet6cTwoHeadHead(config, output_k=config.output_k_B, semisup=semisup)
    self._initialize_weights()

  def forward(self, x, head="B", kmeans_use_features=False, trunk_features=False, penultimate_features=False):
    if penultimate_features:
      print("Not needed/implemented for this arch")
      exit(1)
    # default is "B" for use by eval code; the training script switches between A and B
    x = self.trunk(x)
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
