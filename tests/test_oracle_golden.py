"""CPU: pin the oracle (oracle/) against the golden vectors produced by the
reference itself (tests/golden/make_golden.py), and against analytic known
answers (SURVEY.md S8c "Analytic facts usable as KATs")."""
import math
import os
import sys
from argparse import Namespace

import numpy as np
import pytest
import torch

sys.path.insert(0, os.path.join(os.path.dirname(__file__), "golden"))
import make_golden  # noqa: E402  (specs + named input builders; imports no reference code)
from oracle import iid_losses, nets, seg_losses, transforms, weights  # noqa: E402
from tests.conftest import load_golden  # noqa: E402


def test_iid_oracle_matches_reference_goldens(golden_iid):
  g = golden_iid
  for name in g.names("iid/"):
    c = g.sub("iid/" + name)
    z, zt, lamb = torch.from_numpy(c["z"]), torch.from_numpy(c["zt"]), float(c["lamb"])
    l, l1 = iid_losses.IID_loss(z, zt, lamb=lamb)
    # bit-exact forward vs the unmodified reference (same torch build, fp32)
    assert np.float32(l.item()) == c["ref_loss"], name
    assert np.float32(l1.item()) == c["ref_loss_no_lamb"], name
    assert np.array_equal(iid_losses.compute_joint(z, zt).numpy(), c["ref_joint"]), name
    cf = iid_losses.iid_loss_closed_form(c["z"], c["zt"], lamb=lamb)
    assert abs(cf["loss"] - c["orc_loss_f64"]) < 1e-12
    assert abs(cf["loss"] - float(c["ref_loss"])) < 2e-6
    np.testing.assert_allclose(cf["dz"], c["orc_dz_f64"], rtol=0, atol=1e-12)
    np.testing.assert_allclose(cf["dzt"], c["orc_dzt_f64"], rtol=0, atol=1e-12)


def test_iid_known_answers():
  k = 10
  oh = torch.eye(k).repeat(70, 1)
  l, l1 = iid_losses.IID_loss(oh, oh.clone())
  assert abs(l.item() + math.log(k)) < 1e-5 and l.item() == l1.item()
  z, zt = make_golden.softmax_pair("kat", 300, 7, corr=0.7)
  a = iid_losses.IID_loss(z, zt, lamb=1.3)
  b = iid_losses.IID_loss(zt, z, lamb=1.3)  # symmetric in its arguments
  assert abs(a[0].item() - b[0].item()) < 1e-6
  assert iid_losses.IID_loss(z, zt, lamb=1.0)[0].item() == iid_losses.IID_loss(z, zt, lamb=1.0)[1].item()
  # independent views -> MI ~ 0
  zi, zti = make_golden.softmax_pair("kat2", 4096, 5)
  assert abs(iid_losses.IID_loss(zi, zti)[0].item()) < 5e-3


def test_iid_oracle_vs_live_reference():
  """One IID_loss call of the unmodified reference (recorded in tests/golden/reference_calls.npz): bit-identical."""
  g = load_golden("reference_calls.npz").sub("iid_live")
  z, zt, lamb = make_golden.live_iid_inputs()
  o = iid_losses.IID_loss(z, zt, lamb=lamb)
  assert float(g["ref_loss"]) == float(o[0]) and float(g["ref_loss_no_lamb"]) == float(o[1])


def test_seg_oracle_matches_reference_goldens(golden_seg):
  g = golden_seg
  for name in g.names("seg/"):
    c = g.sub("seg/" + name)
    n, k, h, T, lamb = c["meta"]
    T = int(T)
    for variant, fn in [("collapsed", seg_losses.IID_segmentation_loss),
                        ("uncollapsed", seg_losses.IID_segmentation_loss_uncollapsed)]:
      x1 = torch.from_numpy(c["x1"]).requires_grad_(True)
      x2 = torch.from_numpy(c["x2"]).requires_grad_(True)
      l, l1 = fn(x1, x2, torch.from_numpy(c["theta"]), torch.from_numpy(c["mask"]), float(lamb), T, 0, 0)
      g1, g2 = torch.autograd.grad(l, [x1, x2])
      v = c.sub(variant)
      # align_corners=True (reference-era) vs the False default the fixture was made with:
      # agree to ~4e-6 on square, translation-free affines (SURVEY S8c)
      assert abs(l.item() - float(v["ref_loss"])) < 2e-5, (name, variant)
      assert abs(l1.item() - float(v["ref_loss_no_lamb"])) < 2e-5, (name, variant)
      scale = max(1e-12, np.abs(v["ref_dx1"]).max())
      assert np.abs(g1.numpy() - v["ref_dx1"]).max() < 2e-3 * scale, (name, variant)
      assert np.abs(g2.numpy() - v["ref_dx2"]).max() < 2e-3 * max(1e-12, np.abs(v["ref_dx2"]).max())
      # identical convention -> tight
      x1b = torch.from_numpy(c["x1"]).requires_grad_(True)
      x2b = torch.from_numpy(c["x2"]).requires_grad_(True)
      lb, _ = fn(x1b, x2b, torch.from_numpy(c["theta"]), torch.from_numpy(c["mask"]), float(lamb), T, 0, 0,
                 align_corners=False)
      assert abs(lb.item() - float(v["ref_loss"])) < 1e-6, (name, variant)
      gb = torch.autograd.grad(lb, [x1b])[0]
      assert np.abs(gb.numpy() - v["ref_dx1"]).max() < 1e-5 * scale + 1e-9


def test_seg_box_filter_identity(golden_seg):
  c = golden_seg.sub("seg/small_n3_k4_16_T3")
  x1, x2 = torch.from_numpy(c["x1"]).double(), torch.from_numpy(c["x2"]).double()
  m = torch.from_numpy(c["mask"]).double()[:, None]
  a = seg_losses.seg_joint_displacements(x1 * m, x2 * m, 3).sum(dim=(2, 3))
  b = seg_losses.collapsed_joint_box_filter(x1 * m, x2 * m, 3)
  assert (a - b).abs().max() < 1e-9


def test_sobel_known_answers():
  h = w = 8
  ramp = torch.arange(w, dtype=torch.float32).view(1, 1, 1, w).expand(2, 1, h, w).contiguous()
  o = transforms.sobel_process(ramp, include_rgb=False)
  assert o.shape == (2, 2, h, w)
  # interior: dx = (1+2+1)*(x-1) - (1+2+1)*(x+1) = -8 ; dy = 0
  assert torch.all(o[:, 0, 1:-1, 1:-1] == -8.) and torch.all(o[:, 1, 1:-1, 1:-1] == 0.)
  x = weights.uniform("sobel.x", (3, 5, 9, 9))
  o = transforms.sobel_process(x, include_rgb=True, using_IR=True)
  assert o.shape == (3, 6, 9, 9)
  assert torch.equal(o[:, :3], x[:, :3]) and torch.equal(o[:, 5], x[:, 4])
  o4 = transforms.sobel_process(x[:, :4], include_rgb=True)
  assert torch.equal(o4[:, 3:5], o[:, 3:5])


def _run_net(name, g):
  ctor, cfg, batch, head, lamb = make_golden.NET_SPECS[name]
  net = getattr(nets, ctor)(Namespace(**cfg))
  weights.fill_state_dict(net)
  net.train()
  x, xt = make_golden.net_input("net." + name, cfg, batch)
  kw = {} if head is None else {"head": head}
  o, ot = net(x, **kw), net(xt, **kw)
  loss = sum(iid_losses.IID_loss(a, b, lamb=lamb)[0] for a, b in zip(o, ot)) / len(o)
  loss.backward()
  return net, o, ot, loss


@pytest.mark.parametrize("name", ["5g2h_32_A", "5g2h_32_B", "5g_64", "6c2h_24_A", "6c_24"])
def test_net_oracle_matches_reference_goldens(name, golden_nets):
  c = golden_nets.sub("net/" + name)
  net, o, ot, loss = _run_net(name, c)
  np.testing.assert_allclose(torch.stack(o).detach().numpy(), c["ref_out"], rtol=0, atol=2e-6)
  np.testing.assert_allclose(torch.stack(ot).detach().numpy(), c["ref_out_tf"], rtol=0, atol=2e-6)
  assert abs(loss.item() - float(c["loss"])) < 1e-6
  params = dict(net.named_parameters())
  assert list(params) == list(c["grad_names"])  # same state_dict key order as the reference
  for pn, norm in zip(c["grad_names"], c["grad_norms"]):
    g = params[str(pn)].grad
    mine = 0.0 if g is None else float(g.double().norm())
    assert abs(mine - norm) <= 2e-4 * max(norm, 1e-6) + 1e-9, (pn, mine, norm)
  for key in c.sub("grad"):
    np.testing.assert_allclose(params[key].grad.numpy(), c["grad/" + key], rtol=2e-3, atol=1e-7)
  sd = net.state_dict()
  for key in c.sub("buf"):
    np.testing.assert_allclose(sd[key].numpy(), c["buf/" + key], rtol=1e-5, atol=1e-6)


def test_grey_from_rgb_is_pil_L():
  """oracle.transforms.grey_from_rgb restates custom_greyscale_to_tensor (code/utils/cluster/transforms.py:12-16);
  pinned against PIL itself (what tf.to_grayscale calls) and against the documented luma weights."""
  import numpy as np
  import torch
  from oracle.transforms import grey_from_rgb
  PIL = pytest.importorskip("PIL.Image")
  rng = np.random.default_rng(0)
  a = rng.integers(0, 256, (3, 17, 23, 3), dtype=np.uint8)
  for img in a:
    want = np.asarray(PIL.fromarray(img).convert("L")).astype(np.float32) / 255.0
    got = grey_from_rgb(torch.from_numpy(img).permute(2, 0, 1)[None])[0, 0].numpy()
    assert np.array_equal(got, want)
  f = torch.rand(2, 3, 5, 5)
  assert torch.allclose(grey_from_rgb(f), (0.299 * f[:, 0] + 0.587 * f[:, 1] + 0.114 * f[:, 2])[:, None])


def test_sparse_displacement_oracle_matches_reference_under_seed():
  """random_translation_multiple (seg transforms.py:146-166) and the losses that call it (seg IID_losses.py:29-32,
  :101-104): the oracle draws from numpy's global generator with the reference's calls, so the same seed gives the
  same displacement, loss and gradients as the reference did (tests/golden/reference_calls.npz)."""
  g = load_golden("reference_calls.npz").sub("sparse")
  x, (x1, x2, theta, mask) = make_golden.sparse_inputs()
  for i, seed in enumerate(make_golden.SPARSE_SEEDS):
    np.random.seed(seed)
    b = seg_losses.random_translation_multiple(x, 2, 4)
    assert torch.equal(torch.from_numpy(g["ref_translated"][i]), b)
  for fn_name in ("IID_segmentation_loss", "IID_segmentation_loss_uncollapsed"):
    want = g.sub(fn_name)
    np.random.seed(make_golden.SPARSE_LOSS_SEED)
    a, b = x1.clone().requires_grad_(True), x2.clone().requires_grad_(True)
    l, l1 = getattr(seg_losses, fn_name)(a, b, all_affine2_to_1=theta, all_mask_img1=mask, **make_golden.SPARSE_LOSS_KW)
    ga, gb = torch.autograd.grad(l, [a, b])
    assert abs(float(want["ref_loss"]) - l.item()) < 1e-6 and abs(float(want["ref_loss_no_lamb"]) - l1.item()) < 1e-6
    assert torch.allclose(torch.from_numpy(want["ref_dx1"]), ga, rtol=1e-4, atol=1e-8)
    assert torch.allclose(torch.from_numpy(want["ref_dx2"]), gb, rtol=1e-4, atol=1e-8)


def test_precision_fixture_oracle_matches_reference_golden():
  """The oracle at the well-conditioned operating point (tests/precision_fixture.py) against the golden produced by
  the unmodified reference network: same loss to fp32 rounding, same outputs, same gradients."""
  sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
  from tests import precision_fixture as fx
  from tests.conftest import load_golden
  g = load_golden("precision.npz").sub("wc/32_64_B")
  f = fx.Fixture(32, 64, "B")
  r = f.oracle(torch.float32)
  assert np.allclose(f.trunk_mean.numpy(), g["trunk_mean"], rtol=1e-5, atol=1e-6)
  assert abs(r["loss"] - float(g["loss"])) < 1e-6
  assert np.abs(r["out"].numpy() - g["ref_out"]).max() < 1e-5
  for pn, norm in zip(g["grad_names"], g["grad_norms"]):
    if str(pn) in r["grads"]:
      assert abs(float(r["grads"][str(pn)].norm()) - norm) <= 1e-3 * norm + 1e-9, pn
  for key in g.sub("grad"):
    want = torch.from_numpy(g["grad/" + key]).double()
    assert float((r["grads"][key] - want).norm() / want.norm()) < 5e-3, key
