"""CPU oracle (test infrastructure only) of the semi-supervised head: code/archs/semisup/sup_head5.py:9-40 restated as a
plain ``torch.nn`` module with the reference's state_dict keys, over the oracle trunks of oracle/nets.py.  Pinned against
the unmodified reference by tests/golden/semisup.npz (tests/golden/make_golden_semisup.py, tests/test_semisup_host.py)."""
import torch.nn as nn
import torch.nn.functional as F

from oracle.nets import _ROUND, q, qw


class SupHead5(nn.Module):
  """trunk features -> Linear(dlen, 2048) -> BatchNorm1d(2048) -> ReLU -> Linear(2048, gt_k) (logits).  Under
  ``oracle.nets.bf16_rounding`` the storage points of the product are rounded: the feature and the first Linear's weight
  (tensor-core operands), its bias-free product (the bias is folded into the BatchNorm, which removes it in train mode) and
  the ReLU output; the last Linear is fp32 in every mode."""

  def __init__(self, net_features, dlen=None, gt_k=None):
    super().__init__()
    self.trunk = net_features
    self.head = nn.Sequential(nn.Linear(dlen, 2048), nn.BatchNorm1d(2048), nn.ReLU(), nn.Linear(2048, gt_k))
    for m in self.head.modules():
      if isinstance(m, nn.BatchNorm1d):
        m.weight.data.fill_(1)
        m.bias.data.zero_()
      elif isinstance(m, nn.Linear):
        m.weight.data.normal_(0, 0.01)
        m.bias.data.zero_()

  def forward(self, x, penultimate_features=False):
    x = self.trunk(x, trunk_features=True, penultimate_features=penultimate_features)
    h = self.head
    if _ROUND["on"]:
      y = q(F.linear(q(x), qw(h[0].weight))) + h[0].bias
    else:
      y = h[0](x)
    return h[3](q(F.relu(h[1](y))))
