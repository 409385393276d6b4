"""GPU: the semi-supervised finetune (SupHead5 + cross-entropy + two Adams, IID_semisup_STL10.py:241-256) against what the
unmodified reference computed (tests/golden/semisup.npz) and against the CPU oracle.

Stated tolerances, and where they come from:
  precision="fp32": those of test_gpu_parity_nets.py (a randomly initialised 34-layer BN ResNet at batch 8 is a chaotic map),
      with the two that were stated for softmax outputs (values <= 1) taken relative to the scale of what is compared here:
      logits 2e-4 x max|logit| (logits reach ~8; BatchNorm1d over 8 rows amplifies feature differences), loss 2e-5 x loss;
      gradient norms 1e-2 relative, stored head gradients 5e-2 relative L2; head.1 running statistics 1e-4 relative,
      eval-mode logits 2e-3 x max|logit|.
      head.0.bias has an analytically zero gradient (BatchNorm1d removes the bias): both sides hold rounding noise, bounded
      in absolute terms.  After one Adam step an element moves by ~lr * sign(grad): elements whose gradient is noise (most
      of some BatchNorm vectors) may move the other way, so parameters after the step are compared within 2 lr.
  Three steps of iic_semisup_step against the oracle stepped by torch.optim.Adam: the fp32 oracle against the fp64 oracle
      over the same three steps differs by 9.7e-3 relative in the third loss, by up to 5.75 learning rates in a parameter,
      by 1.0e-2 in head.1.running_mean and 7.2e-3 relative in running_var; the product may differ by twice that.
  precision="tf32x3": the same checks at twice the fp32 tolerances (3xTF32 convolutions are fp32-grade, DESIGN.md S4).
  precision="bf16": the CPU oracle run with bf16 rounding at the product's storage points (oracle.nets.bf16_rounding) is
      compared with the fp32 oracle IN THE TEST, and the product's logits and loss may deviate from the fp32 golden by at
      most twice that.  Gradients are not compared at this configuration: at batch 8 the random 34-layer trunk is chaotic
      under bf16 rounding (two bf16 emulations that differ only in accumulation order disagree by ~45 % in the gradients,
      test_gpu_parity_nets.py), and the head's weight gradient is a sum over those 8 feature rows.  The bf16 gradients are
      checked at the paper's shape (test_paper_shape_bf16_one_step).
  The paper's shape (batch 700, input 64, layer3 features, bf16), head weight gradients against the fp32 mode: the CPU
      oracle with bf16 rounding against the fp32 oracle, at this shape with these weights and inputs, gives cosine 0.9725
      for head.0.weight (the rounding of the 20736-long feature rows and of the weight operand, summed over 700 rows) and
      0.99975 for head.3.weight; the product must stay within twice the oracle's 1 - cos: > 0.945 and > 0.9995.  (A fixed
      0.99 for head.0.weight would be stricter than the bf16 storage format allows.)"""
import os
import sys
from argparse import Namespace

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

sys.path.insert(0, os.path.join(os.path.dirname(__file__), "golden"))
import make_golden_semisup as mgs  # noqa: E402
from oracle import nets as oracle_nets  # noqa: E402
from oracle import weights  # noqa: E402
from tests import semisup_oracle  # noqa: E402
from tests.conftest import load_golden  # noqa: E402
from tests.test_semisup_host import oracle_step  # noqa: E402

CASES = sorted(mgs.SEMISUP_CASES)


@pytest.fixture(scope="module")
def golden_semisup():
  return load_golden("semisup.npz")


def _build(name, precision, input_sz=None, dlen=None):
  import iic_b200.archs as archs
  cfg = dict(mgs.SEMISUP_CFG)
  if input_sz is not None:
    cfg["input_sz"] = input_sz
  pen = mgs.SEMISUP_CASES[name]
  trunk = archs.ClusterNet5g(Namespace(precision=precision, **cfg))
  net = archs.SupHead5(trunk, dlen=dlen or mgs.semisup_dlen(pen), gt_k=mgs.SEMISUP_GT_K)
  weights.fill_state_dict(net)
  return net.cuda().train(), pen


def _opts(net):
  from iic_b200.optim import FusedAdam
  return FusedAdam(net.trunk.parameters(), lr=mgs.SEMISUP_LR[0]), FusedAdam(net.head.parameters(), lr=mgs.SEMISUP_LR[1])


def _run(name, precision):
  """forward, loss, backward, eval logits, one step of the two FusedAdams (the golden's sequence)."""
  from iic_b200.utils.semisup.general import CrossEntropyLoss
  net, pen = _build(name, precision)
  x, t = mgs.semisup_inputs(name)
  x, t = x.cuda(), t.cuda()
  opt_trunk, opt_head = _opts(net)
  opt_trunk.zero_grad(set_to_none=False)
  opt_head.zero_grad(set_to_none=False)
  logits = net(x, penultimate_features=pen)
  loss = CrossEntropyLoss()(logits, t)
  loss.backward()
  out = {"logits": logits.detach().cpu().numpy(), "loss": loss.item(),
         "grads": {n: p.grad.detach().cpu().clone() for n, p in net.named_parameters() if p.grad is not None},
         "buf": {k: getattr(net.head[1], k).cpu().numpy() for k in ("running_mean", "running_var")},
         "names": [n for n, _ in net.named_parameters()]}
  net.eval()
  with torch.no_grad():
    out["eval_logits"] = net(x, penultimate_features=pen).cpu().numpy()
  net.train()
  opt_trunk.step()
  opt_head.step()
  out["params"] = {n: p.detach().cpu().clone() for n, p in net.named_parameters()}
  return out


def _head_grad(c, o, key):
  want = c["grad/" + key].astype(np.float64)
  got = o["grads"][key].numpy().astype(np.float64)
  return (got[:want.shape[0]] if key == "head.0.weight" else got).ravel(), want.ravel()


def _check_fp32_grade(c, o, scale):
  np.testing.assert_allclose(o["logits"], c["logits"], rtol=0, atol=2e-4 * scale * float(np.abs(c["logits"]).max()))
  assert abs(o["loss"] - float(c["loss"])) < 2e-5 * scale * float(c["loss"])
  assert o["names"] == [str(s) for s in c["grad_names"]]
  for pn, norm in zip(c["grad_names"], c["grad_norms"]):
    g = o["grads"].get(str(pn))
    mine = 0.0 if g is None else float(g.double().norm())
    if str(pn) == "head.0.bias":
      assert mine < 1e-5, mine
      continue
    assert abs(mine - norm) <= 1e-2 * scale * norm + 1e-7, (str(pn), mine, norm)
  for key in c.sub("grad"):
    if key == "head.0.bias":
      continue
    got, want = _head_grad(c, o, key)
    assert np.linalg.norm(got - want) <= 5e-2 * scale * np.linalg.norm(want), key
  for key in ("running_mean", "running_var"):
    want = c["buf/head.1." + key]
    np.testing.assert_allclose(o["buf"][key], want, rtol=0, atol=1e-4 * scale * float(np.abs(want).max()))
  # (eval mode runs the trunk on running statistics that have seen one batch: logits reach ~200, compared relative to that)
  np.testing.assert_allclose(o["eval_logits"], c["eval_logits"], rtol=0,
                             atol=2e-3 * scale * max(1.0, float(np.abs(c["eval_logits"]).max())))
  lrs = mgs.SEMISUP_LR
  for key in c.sub("param"):
    want = c["param/" + key]
    got = o["params"][key].numpy()
    got = got[:want.shape[0]] if key == "head.0.weight" else got
    lr = lrs[1] if key.startswith("head.") else lrs[0]
    d = np.abs(got - want)
    assert d.max() <= 2 * lr + 1e-6, (key, d.max())


@pytest.mark.parametrize("name", CASES)
def test_fp32_mode_matches_reference_golden(name, golden_semisup):
  _check_fp32_grade(golden_semisup.sub("semisup/" + name), _run(name, "fp32"), 1.0)


@pytest.mark.parametrize("name", CASES)
def test_tf32x3_mode_matches_reference_golden(name, golden_semisup):
  _check_fp32_grade(golden_semisup.sub("semisup/" + name), _run(name, "tf32x3"), 2.0)


@pytest.mark.parametrize("name", CASES)
def test_bf16_mode_within_the_oracles_bf16_deviation(name, golden_semisup):
  c = golden_semisup.sub("semisup/" + name)
  ref, rnd = oracle_step(name), oracle_step(name, rounding=True)
  o = _run(name, "bf16")
  assert np.isfinite(o["logits"]).all() and np.isfinite(o["loss"])
  assert all(torch.isfinite(g).all() for g in o["grads"].values())
  assert np.abs(o["logits"] - c["logits"]).max() <= 2 * np.abs(rnd["logits"] - ref["logits"]).max()
  assert abs(o["loss"] - float(c["loss"])) <= 2 * abs(rnd["loss"] - ref["loss"])


def test_cross_entropy_matches_torch():
  import torch.nn.functional as F
  from iic_b200 import kernels
  g = torch.Generator().manual_seed(7)
  for n, k in [(700, 10), (700, 70), (37, 10), (5, 70)]:
    logits = (80.0 * torch.randn(n, k, generator=g)).cuda()
    t = torch.randint(0, k, (n,), generator=g).cuda()
    loss, d = kernels.cross_entropy(logits, t)
    lt = logits.clone().requires_grad_(True)
    ref = F.cross_entropy(lt, t)
    ref.backward()
    assert abs(loss.item() - ref.item()) <= 1e-6 * abs(ref.item()), (n, k, loss.item(), ref.item())
    assert (d - lt.grad).abs().max().item() <= 1e-6, (n, k)
    loss2, d2 = kernels.cross_entropy(logits, t)  # deterministic
    assert torch.equal(loss, loss2) and torch.equal(d, d2)
  # an out-of-range target: NaN, no trap; the next call is clean
  bad = t.clone()
  bad[3] = k
  loss, d = kernels.cross_entropy(logits, bad)
  torch.cuda.synchronize()
  assert torch.isnan(loss).item() and torch.isnan(d[3]).all().item() and torch.isfinite(d[4]).all().item()
  loss, d = kernels.cross_entropy(logits, t)
  assert torch.isfinite(loss).item() and abs(loss.item() - F.cross_entropy(logits, t).item()) <= 1e-6 * loss.item()


def test_cross_entropy_module_and_autograd():
  from iic_b200.utils.semisup.general import CrossEntropyLoss
  g = torch.Generator().manual_seed(3)
  logits = torch.randn(64, 10, generator=g).cuda().requires_grad_(True)
  t = torch.randint(0, 10, (64,), generator=g).cuda()
  loss = CrossEntropyLoss()(logits, t)
  (3.0 * loss).backward()
  ref = logits.detach().clone().requires_grad_(True)
  (3.0 * torch.nn.functional.cross_entropy(ref, t)).backward()
  assert (logits.grad - ref.grad).abs().max().item() <= 1e-6


@pytest.mark.parametrize("arch", ["ClusterNet5gTwoHead", "ClusterNet6cTwoHead"])
def test_semisup_twohead_head_vs_oracle(arch):
  import iic_b200.archs as archs
  if arch == "ClusterNet5gTwoHead":
    cfg = dict(in_channels=2, input_sz=32, num_sub_heads=3, output_k_A=20, output_k_B=10, batchnorm_track=True)
  else:
    cfg = dict(in_channels=1, input_sz=24, num_sub_heads=3, output_k_A=20, output_k_B=10, batchnorm_track=True)
  net = archs.__dict__[arch](Namespace(precision="fp32", semisup=True, **cfg))
  weights.fill_state_dict(net)
  net.cuda().train()
  orc = getattr(oracle_nets, arch)(Namespace(**cfg))
  orc.trunk.load_state_dict({k: v.cpu() for k, v in net.trunk.state_dict().items()})
  orc.train()
  x = weights.normal("semisup.twohead." + arch, (6, cfg["in_channels"], cfg["input_sz"], cfg["input_sz"]))
  r = weights.normal("semisup.twohead.r." + arch, (6, 10))
  out = net(x.cuda(), head="B")
  assert out.shape == (6, 10)
  (out * r.cuda()).sum().backward()
  w = net.head_B.head.weight.detach().cpu().clone().requires_grad_(True)
  b = net.head_B.head.bias.detach().cpu().clone().requires_grad_(True)
  ref = torch.nn.functional.linear(orc.trunk(x), w, b)
  (ref * r).sum().backward()
  np.testing.assert_allclose(out.detach().cpu().numpy(), ref.detach().numpy(), rtol=0, atol=2e-4 * max(1.0, ref.abs().max().item()))
  for got, want in [(net.head_B.head.weight.grad, w.grad), (net.head_B.head.bias.grad, b.grad)]:
    assert (got.cpu() - want).norm() <= 5e-2 * want.norm()
  for (n1, p1), (n2, p2) in zip(net.trunk.named_parameters(), orc.trunk.named_parameters()):
    assert n1 == n2
    if p2.grad is not None:
      a, e = float(p1.grad.double().norm()), float(p2.grad.double().norm())
      assert abs(a - e) <= 1e-2 * e + 1e-7, (n1, a, e)


@pytest.mark.parametrize("use_arena", [False, True])
def test_semisup_step_three_steps_vs_oracle_adam(use_arena):
  from iic_b200.arena import GradArena
  from iic_b200.step import iic_semisup_step
  name = "avg"
  net, pen = _build(name, "fp32")
  opts = _opts(net)
  arena = GradArena(net) if use_arena else None
  orc = semisup_oracle.SupHead5(oracle_nets.ClusterNet5g(Namespace(**mgs.SEMISUP_CFG)), dlen=512,
                                gt_k=mgs.SEMISUP_GT_K)
  orc.load_state_dict({k: v.cpu() for k, v in net.state_dict().items()})
  orc.train()
  o_trunk = torch.optim.Adam(orc.trunk.parameters(), lr=mgs.SEMISUP_LR[0])
  o_head = torch.optim.Adam(orc.head.parameters(), lr=mgs.SEMISUP_LR[1])
  for step in range(3):
    x, t = mgs.semisup_inputs("step%d" % step)
    loss = iic_semisup_step(net, opts, x.cuda(), t.cuda(), penultimate_features=pen, sobel=False, arena=arena)
    assert loss.dim() == 0 and loss.is_cuda
    o_trunk.zero_grad()
    o_head.zero_grad()
    lo = torch.nn.CrossEntropyLoss()(orc(x, penultimate_features=pen), t)
    lo.backward()
    o_trunk.step()
    o_head.step()
    assert abs(loss.item() - lo.item()) <= 2e-2 * abs(lo.item()), (step, loss.item(), lo.item())
  assert all(p.grad is None or not p.grad.any() for n, p in net.named_parameters() if ".head.heads." in n)
  orc_params = dict(orc.named_parameters())
  for n, p in net.named_parameters():
    lr = mgs.SEMISUP_LR[1 if n.startswith("head.") else 0]
    d = (p.detach().cpu() - orc_params[n].detach()).abs()
    if ".head.heads." in n:  # never trained: untouched on both sides
      assert d.max().item() == 0.0, n
      continue
    assert d.max().item() <= 12 * lr, (n, d.max().item())
  np.testing.assert_allclose(net.head[1].running_mean.cpu().numpy(), orc.head[1].running_mean.numpy(), rtol=0, atol=2e-2)
  np.testing.assert_allclose(net.head[1].running_var.cpu().numpy(), orc.head[1].running_var.numpy(), rtol=1.5e-2, atol=0)


def _block_restatement(all_logits, all_targets, contiguous_sz, gt_k):
  """assess_acc_block's numpy tail (code/utils/semisup/general.py:77-99)."""
  total, dlen = all_logits.shape
  num_orig = total // contiguous_sz
  a = all_logits.astype(np.float64).reshape((num_orig, contiguous_sz, dlen)).sum(axis=1) / float(contiguous_sz)
  preds = np.argmax(a, axis=1).astype("int")
  tg = all_targets.reshape((num_orig, contiguous_sz))[:, 0].astype("int")
  return (preds == tg).sum() / float(num_orig)


class _Replay(torch.nn.Module):
  """Stands in for the network: returns the next recorded batch of logits."""

  def __init__(self, batches):
    super().__init__()
    self.batches = [b.cuda() for b in batches]
    self.i = 0

  def forward(self, x, penultimate_features=False):
    out = self.batches[self.i]
    self.i += 1
    assert out.shape[0] == x.shape[0]
    return out


def test_assess_acc_block_and_assess_acc_vs_reference_restatement():
  from iic_b200.utils.semisup.general import assess_acc, assess_acc_block
  gt_k, csz, nimg, bsz = 10, 10, 70, 140
  g = np.random.default_rng(5)
  labels = g.integers(0, gt_k, nimg)
  targets = np.repeat(labels, csz)
  logits = g.standard_normal((nimg * csz, gt_k)).astype(np.float32) + 1.5 * np.eye(gt_k, dtype=np.float32)[targets]
  batches = [torch.from_numpy(logits[i:i + bsz]) for i in range(0, len(logits), bsz)]
  loader = [(torch.rand(bsz, 1, 8, 8), torch.from_numpy(targets[i:i + bsz])) for i in range(0, len(logits), bsz)]
  acc = assess_acc_block(_Replay(batches), loader, gt_k=gt_k, include_rgb=False, contiguous_sz=csz)
  assert acc == _block_restatement(logits, targets, csz, gt_k)
  acc1 = assess_acc(_Replay(batches), loader, gt_k=gt_k, include_rgb=False)
  assert acc1 == (np.argmax(logits, axis=1) == targets).sum() / float(len(targets))
  assert 0.0 < acc1 < 1.0


def test_paper_shape_bf16_one_step():
  """ClusterNet5g at input 64, 2 sobel channels from uint8 RGB, batch 700, layer3 features (dlen 20736), gt_k 10: the first
  Linear (20736 -> 2048) runs as a 1x1 convolution over 700 images of 1x1 pixels on the tcgen05 path."""
  from iic_b200 import kernels
  from iic_b200.step import iic_semisup_step
  net16, pen = _build("pen", "bf16", input_sz=64, dlen=20736)
  net32, _ = _build("pen", "fp32", input_sz=64, dlen=20736)
  net32.load_state_dict(net16.state_dict())
  x = torch.from_numpy((weights.uniform("semisup.paper.rgb", (700, 3, 64, 64)).numpy() * 255).astype(np.uint8))
  t = torch.from_numpy((weights.uniform("semisup.paper.t", (700,)).numpy() * 10).astype(np.int64))
  g = kernels.conv_geom(700, 1, 1, 20736, 2048, 1, 1, 1, 0, 1)
  assert kernels._lib.lib().iic_conv_fprop_stats_blocks(kernels.ctypes.byref(g), kernels.BF16) > 0  # tensor-core path
  grads = {}
  for net in (net16, net32):
    opts = _opts(net)
    loss = iic_semisup_step(net, opts, x.cuda(), t.cuda(), penultimate_features=True, sobel=True)
    assert torch.isfinite(loss).item()
    grads[net.precision] = {n: p.grad.detach().double().clone() for n, p in net.named_parameters()
                            if p.grad is not None and ".head.heads." not in n}
    assert all(torch.isfinite(v).all().item() for v in grads[net.precision].values())
  for key, bound in (("head.0.weight", 0.945), ("head.3.weight", 0.9995)):
    a, b = grads["bf16"][key].ravel(), grads["fp32"][key].ravel()
    cos = float(a @ b / (a.norm() * b.norm()))
    print("paper shape: %s bf16 vs fp32 gradient cosine %.6f" % (key, cos))
    assert cos > bound, (key, cos)


def test_errors():
  from iic_b200.utils.semisup.general import CrossEntropyLoss
  net, pen = _build("avg", "fp32")
  x, t = mgs.semisup_inputs("avg")
  with pytest.raises(RuntimeError):
    net(x, penultimate_features=pen)  # CPU input
  with pytest.raises(RuntimeError):
    net.forward_head(torch.zeros(8, 512))
  with pytest.raises(RuntimeError):
    CrossEntropyLoss()(torch.zeros(8, 10), t)
  loss = CrossEntropyLoss()(net(x.cuda(), penultimate_features=pen), t.cuda())
  loss.backward(retain_graph=True)
  with pytest.raises(RuntimeError):
    loss.backward()  # a second backward
  loss = CrossEntropyLoss()(net(x.cuda(), penultimate_features=pen), t.cuda())
  with torch.no_grad():
    net.head[0].weight.add_(1.0)  # in-place weight change between forward and backward
  with pytest.raises(RuntimeError):
    loss.backward()
