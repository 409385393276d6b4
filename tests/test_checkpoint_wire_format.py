"""SURVEY.md S8f row 3: a checkpoint written by the reference's own modules (state_dict of the unmodified reference net,
optimiser state of torch.optim.Adam) loads into the iic_b200 network / FusedAdam with the reference's own calls, and
back.  The reference nets' state_dict layouts (key order, shapes, dtypes) are recorded in tests/golden/
reference_calls.npz.  CPU only (modules hold parameters; no kernel runs)."""
import collections
import os
import sys
from argparse import Namespace

import pytest
import torch

sys.path.insert(0, os.path.join(os.path.dirname(__file__), "golden"))
import make_golden  # noqa: E402
from tests.conftest import load_golden  # noqa: E402


def _reference_checkpoint(name):
  """A state_dict with the layout the reference net saves, filled with seeded values a fresh net does not hold."""
  g = load_golden("reference_calls.npz").sub("checkpoint/" + name)
  gen = torch.Generator().manual_seed(3)
  sd = collections.OrderedDict()
  for key, shape, dtype in zip(g["keys"], g["shapes"], g["dtypes"]):
    shape, dtype = tuple(int(s) for s in str(shape).split(",") if s), getattr(torch, str(dtype))
    if dtype.is_floating_point:
      sd[str(key)] = torch.randn(shape, generator=gen).to(dtype)
    else:
      sd[str(key)] = torch.randint(1, 1000, shape, generator=gen).to(dtype)
  return sd


@pytest.mark.parametrize("name", sorted(make_golden.CHECKPOINT_SPECS))
def test_reference_checkpoint_round_trip(name, tmp_path):
  import iic_b200.archs as archs
  from iic_b200.utils.checkpoint import load_into, load_reference_state_dict
  cfg = make_golden.CHECKPOINT_SPECS[name]
  want = _reference_checkpoint(name)
  path = os.path.join(str(tmp_path), "latest_net.pytorch")
  torch.save(want, path)  # cluster_sobel_twohead.py:429
  net = archs.__dict__[name](Namespace(**cfg))
  net.load_state_dict(torch.load(path, map_location=lambda storage, loc: storage))  # :176-178, verbatim
  got = net.state_dict()
  assert list(got.keys()) == list(want.keys())
  for k in want:
    assert got[k].dtype == want[k].dtype and torch.equal(got[k], want[k]), k
  # saved from a DataParallel wrapper: keys carry a "module." prefix
  path2 = os.path.join(str(tmp_path), "dp.pytorch")
  torch.save(collections.OrderedDict(("module." + k, v) for k, v in want.items()), path2)
  net2 = archs.__dict__[name](Namespace(**cfg))
  load_into(net2, path2)
  assert all(torch.equal(net2.state_dict()[k], want[k]) for k in want)
  assert list(load_reference_state_dict(path2).keys()) == list(want.keys())
  # and back: what iic_b200 saves has the reference's layout (what its strict load_state_dict checks) and values
  torch.save(net.state_dict(), path)
  back = torch.load(path, map_location=lambda storage, loc: storage)
  assert list(back.keys()) == list(want.keys())
  for k in want:
    assert back[k].shape == want[k].shape and back[k].dtype == want[k].dtype and torch.equal(back[k], want[k]), k


def test_adam_state_interchanges_with_torch():
  from iic_b200.optim import FusedAdam
  ps = [torch.nn.Parameter(torch.randn(4, 3)), torch.nn.Parameter(torch.randn(5))]
  ref = torch.optim.Adam(ps, lr=1e-4)
  for p in ps:
    p.grad = torch.randn_like(p)
  ref.step()
  sd = ref.state_dict()
  ours = FusedAdam(ps, lr=1e-4)
  ours.load_state_dict(sd)  # cluster_sobel_twohead.py:187
  out = ours.state_dict()
  assert out["param_groups"][0]["lr"] == 1e-4 and out["param_groups"][0]["betas"] == (0.9, 0.999)
  for i in range(2):
    for key in ("exp_avg", "exp_avg_sq"):
      assert torch.equal(out["state"][i][key], sd["state"][i][key])
    assert float(out["state"][i]["step"]) == 1.0
  back = torch.optim.Adam(ps, lr=1e-4)
  back.load_state_dict(out)


def test_adam_state_written_by_torch_0_4_1_loads():
  """ADVICE r1: the reference's optimiser checkpoints (torch 0.4.1) keep `step` as a Python int and an `amsgrad`
  key in the param groups; FusedAdam.load_state_dict must accept them (resume path, cluster_sobel_twohead.py:187)."""
  from iic_b200.optim import FusedAdam
  ps = [torch.nn.Parameter(torch.randn(4, 3)), torch.nn.Parameter(torch.randn(5))]
  legacy = {"state": {i: {"step": 7, "exp_avg": torch.randn_like(p), "exp_avg_sq": torch.rand_like(p)}
                      for i, p in enumerate(ps)},
            "param_groups": [{"lr": 1e-4, "betas": (0.9, 0.999), "eps": 1e-8, "weight_decay": 0, "amsgrad": False,
                              "params": [0, 1]}]}
  ours = FusedAdam(ps, lr=1e-3)
  ours.load_state_dict(legacy)
  for p in ps:
    st = ours.state[p]
    assert torch.is_tensor(st["step"]) and float(st["step"]) == 7.0
  assert ours.param_groups[0]["lr"] == 1e-4
  # a pickled optimiser (torch.save(optimiser)) goes through __setstate__ as well
  import pickle
  again = pickle.loads(pickle.dumps(ours))
  assert all(torch.is_tensor(again.state[p]["step"]) for p in again.param_groups[0]["params"])
