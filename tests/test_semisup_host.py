"""CPU: the semi-supervised finetune (SupHead5, IID_semisup_STL10.py) -- the oracle against what the unmodified reference
computed (tests/golden/semisup.npz), the product's state_dict layout and registry entry, get_dlen without a forward, and
the new C-ABI symbols."""
import io
import os
import re
import subprocess
import sys
from argparse import Namespace

import numpy as np
import pytest
import torch

sys.path.insert(0, os.path.join(os.path.dirname(__file__), "golden"))
import make_golden_semisup as mgs  # noqa: E402
from oracle import nets as oracle_nets  # noqa: E402
from oracle import weights  # noqa: E402
from tests import semisup_oracle  # noqa: E402
from tests.conftest import load_golden  # noqa: E402

NEW_SYMBOLS = ("iic_cross_entropy", "iic_linear_fwd", "iic_linear_bwd", "iic_col_sum")


@pytest.fixture(scope="module")
def golden_semisup():
  return load_golden("semisup.npz")


def oracle_step(name, rounding=False):
  """The reference's training step (IID_semisup_STL10.py:241-256) on the oracle: returns what semisup.npz records."""
  pen = mgs.SEMISUP_CASES[name]
  net = semisup_oracle.SupHead5(oracle_nets.ClusterNet5g(Namespace(**mgs.SEMISUP_CFG)),
                                dlen=mgs.semisup_dlen(pen), gt_k=mgs.SEMISUP_GT_K)
  weights.fill_state_dict(net)
  net.train()
  x, t = mgs.semisup_inputs(name)
  opt_trunk = torch.optim.Adam(net.trunk.parameters(), lr=mgs.SEMISUP_LR[0])
  opt_head = torch.optim.Adam(net.head.parameters(), lr=mgs.SEMISUP_LR[1])
  with oracle_nets.bf16_rounding(rounding):
    logits = net(x, penultimate_features=pen)
    loss = torch.nn.CrossEntropyLoss()(logits, t)
    loss.backward()
    out = {"logits": logits.detach().numpy(), "loss": loss.item(),
           "grads": {n: p.grad.clone() for n, p in net.named_parameters() if p.grad is not None},
           "buf": {k: getattr(net.head[1], k).clone().numpy() for k in ("running_mean", "running_var")}}
    with torch.no_grad():
      net.eval()
      out["eval_logits"] = net(x, penultimate_features=pen).numpy()
      net.train()
  opt_trunk.step()
  opt_head.step()
  out["params"] = {n: p.detach().clone() for n, p in net.named_parameters()}
  out["names"] = [n for n, _ in net.named_parameters()]
  return out


@pytest.mark.parametrize("name", sorted(mgs.SEMISUP_CASES))
def test_oracle_sup_head5_matches_reference_golden(name, golden_semisup):
  c = golden_semisup.sub("semisup/" + name)
  o = oracle_step(name)
  np.testing.assert_allclose(o["logits"], c["logits"], rtol=0, atol=1e-5)
  assert abs(o["loss"] - float(c["loss"])) < 1e-5
  assert o["names"] == [str(s) for s in c["grad_names"]]
  for pn, norm in zip(c["grad_names"], c["grad_norms"]):
    g = o["grads"].get(str(pn))
    mine = 0.0 if g is None else float(g.double().norm())
    if str(pn) == "head.0.bias":  # analytically zero (BatchNorm removes the bias): rounding noise on both sides
      assert mine < 1e-5 and norm < 1e-5
      continue
    assert abs(mine - norm) <= 1e-4 * norm + 1e-9, (str(pn), mine, norm)
  for key in c.sub("grad"):
    if key == "head.0.bias":
      continue
    g = o["grads"][key].numpy()
    want = c["grad/" + key]
    got = g[:want.shape[0]] if key == "head.0.weight" else g
    assert np.linalg.norm(got - want) <= 1e-4 * np.linalg.norm(want), key
  for key in ("running_mean", "running_var"):
    np.testing.assert_allclose(o["buf"][key], c["buf/head.1." + key], rtol=1e-5, atol=1e-6)
  np.testing.assert_allclose(o["eval_logits"], c["eval_logits"], rtol=0, atol=1e-4)
  lr_head = mgs.SEMISUP_LR[1]
  for key in c.sub("param"):
    want = c["param/" + key]
    got = o["params"][key].numpy()
    got = got[:want.shape[0]] if key == "head.0.weight" else got
    # (the first Linear's bias moves by Adam-normalised rounding noise: up to one learning rate either way)
    tol = 2 * lr_head if key == "head.0.bias" else 1e-6
    np.testing.assert_allclose(got, want, rtol=0, atol=tol, err_msg=key)


def _product_sup_head5(dlen, input_sz=32):
  import iic_b200.archs as archs
  cfg = dict(mgs.SEMISUP_CFG, input_sz=input_sz)
  trunk = archs.__dict__["ClusterNet5g"](Namespace(precision="fp32", **cfg))
  return archs.__dict__["SupHead5"](trunk, dlen=dlen, gt_k=mgs.SEMISUP_GT_K)


def _layout(sd):
  return ([str(k) for k in sd], [",".join(map(str, v.shape)) for v in sd.values()],
          [str(v.dtype).replace("torch.", "") for v in sd.values()])


@pytest.mark.parametrize("name", sorted(mgs.SEMISUP_CASES))
def test_sup_head5_state_dict_layout_matches_reference(name, golden_semisup):
  c = golden_semisup.sub("semisup/" + name)
  want = ([str(s) for s in c["keys"]], [str(s) for s in c["shapes"]], [str(s) for s in c["dtypes"]])
  net = _product_sup_head5(mgs.semisup_dlen(mgs.SEMISUP_CASES[name]))
  assert _layout(net.state_dict()) == want
  # a checkpoint with the reference's layout loads, and what is saved again has that layout
  ckpt = {}
  for k, shape, dt in zip(*want):
    dims = tuple(int(s) for s in shape.split(",")) if shape else ()
    ckpt[k] = torch.full(dims, 3, dtype=getattr(torch, dt)) if dims == () else torch.ones(dims, dtype=getattr(torch, dt))
  net.load_state_dict(ckpt)
  buf = io.BytesIO()
  torch.save(net.state_dict(), buf)
  buf.seek(0)
  assert _layout(torch.load(buf)) == want
  assert int(net.head[1].num_batches_tracked) == 3


def test_registry_has_sup_head5():
  import iic_b200.archs as archs
  from iic_b200.archs.semisup.sup_head5 import SupHead5
  assert archs.__dict__["SupHead5"] is SupHead5


def test_get_dlen_from_geometry_without_a_forward():
  import iic_b200.archs as archs
  from iic_b200.utils.semisup.general import get_dlen
  for input_sz, pen, want in [(64, False, 512), (32, True, 6400), (64, True, 20736)]:
    cfg = dict(mgs.SEMISUP_CFG, input_sz=input_sz)
    net = archs.ClusterNet5g(Namespace(precision="bf16", **cfg))  # CPU tensors: any forward would raise
    loader = [(torch.zeros(4, 2, input_sz, input_sz), torch.zeros(4, dtype=torch.long))]
    assert get_dlen(net, loader, include_rgb=False, penultimate_features=pen) == want
  cfg6 = dict(in_channels=1, input_sz=64, num_sub_heads=2, output_k=10, batchnorm_track=True)
  net6 = archs.ClusterNet6c(Namespace(precision="bf16", **cfg6))
  assert get_dlen(net6, [(torch.zeros(2, 1, 64, 64), None)]) == net6.head.nfeat


def test_library_exports_semisup_symbols():
  from iic_b200 import _lib, build
  lib = build.build()
  out = subprocess.run(["nm", "-D", "--defined-only", lib], capture_output=True, text=True, check=True).stdout
  exported = set(re.findall(r" T (iic_[a-z0-9_]+)", out))
  for s in NEW_SYMBOLS:
    assert s in exported and s in _lib.declared_symbols(), s
