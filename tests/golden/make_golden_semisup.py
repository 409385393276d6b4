"""Generate tests/golden/semisup.npz FROM THE REFERENCE ITSELF: one training step of the semi-supervised finetune
(code/scripts/semisup/IID_semisup_STL10.py:241-256) through the unmodified SupHead5 (code/archs/semisup/sup_head5.py) over
the unmodified ClusterNet5g, on the CPU.

Run in the build container (needs the reference tree, as make_golden.py does):
    python tests/golden/make_golden_semisup.py

The reference networks are loaded through oracle/refshim.py; sup_head5.py, which the shim does not cover, is loaded here
under the same alias package.  Its constructor calls ``net_head.cuda()`` (sup_head5.py:23): ``Module.cuda`` is a no-op while
it runs.  Inputs are rebuilt by name from oracle/weights.py, so the tests recreate them without this file's reference access.
"""
import importlib
import os
import sys
from argparse import Namespace

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

from oracle import refshim, weights  # noqa: E402


def load_reference_sup_head5():
  """-> (reference namespace of oracle/refshim.py, a SupHead5 constructor that never touches a device)."""
  import torch.nn as nn
  ref = refshim.load()
  refshim._pkg("iicref.archs.semisup", os.path.join(refshim.REF, "code", "archs", "semisup"))
  cls = importlib.import_module("iicref.archs.semisup.sup_head5").SupHead5

  def make(*a, **k):
    cuda = nn.Module.cuda
    nn.Module.cuda = lambda self, *aa, **kk: self
    try:
      return cls(*a, **k)
    finally:
      nn.Module.cuda = cuda
  return ref, make


# semi-supervised finetune (IID_semisup_STL10.py): SupHead5 over ClusterNet5g, one training step
SEMISUP_CFG = dict(in_channels=2, input_sz=32, num_sub_heads=5, output_k=10, batchnorm_track=True)
SEMISUP_BATCH, SEMISUP_GT_K = 8, 10
SEMISUP_LR = (1e-4, 1e-3)  # (trunk_lr, head_lr) of the two torch.optim.Adam
SEMISUP_CASES = {"pen": True, "avg": False}  # name -> penultimate_features (dlen 6400 / 512)
SEMISUP_W1_ROWS = 8  # head.0.weight (2048 x dlen) and its gradient are recorded for these first rows only


def semisup_inputs(name):
  x = weights.normal("semisup.%s.x" % name, (SEMISUP_BATCH, SEMISUP_CFG["in_channels"], SEMISUP_CFG["input_sz"],
                                             SEMISUP_CFG["input_sz"]))
  t = torch.from_numpy((weights.uniform("semisup.%s.t" % name, (SEMISUP_BATCH,)).numpy() * SEMISUP_GT_K).astype(np.int64))
  return x, t


def semisup_dlen(pen):
  return 256 * 5 * 5 if pen else 512


def gen_semisup(ref, out):
  """SupHead5(ClusterNet5g) of the unmodified reference at input 32, batch 8, gt_k 10, named weights: one training step
  (IID_semisup_STL10.py:241-256) with and without penultimate features."""
  for name, pen in SEMISUP_CASES.items():
    dlen = semisup_dlen(pen)
    net = ref.SupHead5(ref.ClusterNet5g(Namespace(**SEMISUP_CFG)), dlen=dlen, gt_k=SEMISUP_GT_K)
    weights.fill_state_dict(net)
    net.train()
    x, t = semisup_inputs(name)
    opt_trunk = torch.optim.Adam(net.trunk.parameters(), lr=SEMISUP_LR[0])
    opt_head = torch.optim.Adam(net.head.parameters(), lr=SEMISUP_LR[1])
    logits = net(x, penultimate_features=pen)
    loss = torch.nn.CrossEntropyLoss()(logits, t)
    opt_trunk.zero_grad()
    opt_head.zero_grad()
    loss.backward()
    p = "semisup/%s/" % name
    out[p + "logits"] = logits.detach().numpy()
    out[p + "loss"] = np.float32(loss.item())
    names, norms = [], []
    for pn, pp in net.named_parameters():
      g = pp.grad
      names.append(pn)
      norms.append(0.0 if g is None else float(g.double().norm()))
      if pn.startswith("head."):
        out[p + "grad/" + pn] = (g[:SEMISUP_W1_ROWS] if pn == "head.0.weight" else g).numpy().copy()
    out[p + "grad_names"] = np.array(names)
    out[p + "grad_norms"] = np.array(norms)
    for key in ("running_mean", "running_var"):
      out[p + "buf/head.1." + key] = getattr(net.head[1], key).numpy().copy()
    with torch.no_grad():
      net.eval()
      out[p + "eval_logits"] = net(x, penultimate_features=pen).numpy()
      net.train()
    opt_trunk.step()
    opt_head.step()
    for pn, pp in net.named_parameters():
      if pn.startswith("head.") or pp.numel() <= 4096:
        out[p + "param/" + pn] = (pp[:SEMISUP_W1_ROWS] if pn == "head.0.weight" else pp).detach().numpy().copy()
    sd = net.state_dict()
    out[p + "keys"] = np.array(list(sd))
    out[p + "shapes"] = np.array([",".join(map(str, v.shape)) for v in sd.values()])
    out[p + "dtypes"] = np.array([str(v.dtype).replace("torch.", "") for v in sd.values()])
    print("semisup", name, dlen, loss.item())


def main():
  assert refshim.available(), "needs the reference tree"
  torch.set_num_threads(8)
  ref, sup_head5 = load_reference_sup_head5()
  ref = Namespace(ClusterNet5g=ref.ClusterNet5g, SupHead5=sup_head5)
  out = {}
  gen_semisup(ref, out)
  path = os.path.join(HERE, "semisup.npz")
  np.savez_compressed(path, **{k.replace("/", "|"): v for k, v in out.items()})
  print("wrote", path, os.path.getsize(path) // 1024, "KiB")


if __name__ == "__main__":
  main()
