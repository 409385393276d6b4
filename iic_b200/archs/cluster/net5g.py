"""ClusterNet5g -- drop-in for code/archs/cluster/net5g.py:10-103 (ResNet-34-shaped trunk,
num_sub_heads x (Linear 512->k + Softmax)), executed by hand-written sm_100a kernels."""
import torch.nn as nn

from .. import _engine as E
from ... import kernels as K
from .residual import BasicBlock, ResNet, ResNetTrunk

__all__ = ["ClusterNet5g"]


class ClusterNet5gTrunk(ResNetTrunk):
  def __init__(self, config):
    super().__init__()
    self.batchnorm_track = config.batchnorm_track
    self.precision = getattr(config, "precision", "bf16")
    block, layers = BasicBlock, [3, 4, 6, 3]
    self.inplanes = 64
    self.conv1 = E.ConvParams(config.in_channels, 64, 3, 1, 1)
    self.bn1 = E.BNParams(64, self.batchnorm_track)
    self.layer1 = self._make_layer(block, 64, layers[0])
    self.layer2 = self._make_layer(block, 128, layers[1], stride=2)
    self.layer3 = self._make_layer(block, 256, layers[2], stride=2)
    self.layer4 = self._make_layer(block, 512, layers[3], stride=2)
    if config.input_sz == 96:
      avg_pool_sz = 7
    elif config.input_sz == 64:
      avg_pool_sz = 5
    elif config.input_sz == 32:
      avg_pool_sz = 3
    self.avg_pool_sz = avg_pool_sz  # nn.AvgPool2d(avg_pool_sz, stride=1) on an avg_pool_sz^2 map

  def forward(self, x, penultimate_features=False, groups=1):
    def run(ctx, xin):
      a = E.stem_forward(ctx, self.conv1, self.bn1, xin, pool_pad=1)  # conv1,bn1,relu,maxpool(2,2,1)
      for layer in (self.layer1, self.layer2, self.layer3):
        for blk in layer:
          a = E.block_forward(ctx, blk, a)
      if penultimate_features:
        # layer3 output flattened in NCHW order (net5g.py:58-60 of the reference); its fp32 gradient goes back to NHWC in
        # the storage type, and the backward of the layer3 blocks runs unchanged (semisup finetuning, SupHead5)
        n, h, w, c = a.shape
        dt = ctx.dt
        return (K.nhwc_to_nchw(a).reshape(n, -1),
                (lambda dfeat: K.nchw_to_nhwc(dfeat.contiguous().float().reshape(n, c, h, w), dt)))
      for blk in self.layer4:
        a = E.block_forward(ctx, blk, a)
      n, h, w, c = a.shape
      assert h == self.avg_pool_sz and w == self.avg_pool_sz, "input_sz does not match the input"
      shape, dt = tuple(a.shape), ctx.dt
      return K.avgpool(a), (lambda dfeat: K.avgpool_bwd(dfeat.contiguous().float(), shape, dt))

    return E.run_trunk(self, run, x, groups)


class ClusterNet5gHead(E.SubHeads):
  def __init__(self, config):
    super().__init__(512 * BasicBlock.expansion, config.output_k, config.num_sub_heads)
    self.batchnorm_track = config.batchnorm_track


class ClusterNet5g(ResNet):
  def __init__(self, config):
    super().__init__()
    self.batchnorm_track = config.batchnorm_track
    self.trunk = ClusterNet5gTrunk(config)
    self.head = ClusterNet5gHead(config)
    self._initialize_weights()

  def forward(self, x, kmeans_use_features=False, trunk_features=False, penultimate_features=False):
    x = self.trunk(x, penultimate_features=penultimate_features)
    if trunk_features:  # for semisup
      return x
    return self.head(x, kmeans_use_features=kmeans_use_features)  # returns list
