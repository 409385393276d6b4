"""Generate the golden fixtures in this directory FROM THE REFERENCE ITSELF.

Run in the build container (needs /root/reference):
    python tests/golden/make_golden.py

The reference (xu-ji/IIC) has no tests and no golden vectors (SURVEY.md S4), so
these fixtures are the pin: every tensor tagged ``ref_*`` below was produced by
the UNMODIFIED reference modules imported through oracle/refshim.py (torch
2.11 CPU, fp32).  Gradients of the clustering loss are tagged ``orc_*``: the
reference's IID_loss backward cannot run on torch>=1.x (in-place writes into
expanded views, IID_losses.py:17-19), so those come from the clone-restated
oracle, whose forward is asserted bit-identical to the reference here.

Inputs are rebuilt by name from oracle/weights.py (numpy PCG64), so only small
arrays are stored.
"""
import os
import sys
from argparse import Namespace

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

from oracle import iid_losses, refshim, weights  # noqa: E402

torch.set_num_threads(8)


def softmax_pair(name, n, k, corr=None, salt=0):
  l = weights.normal(name + ".l", (n, k), salt=salt)
  if corr is None:
    lt = weights.normal(name + ".lt", (n, k), salt=salt)
  else:
    lt = l * 3.0 + corr * weights.normal(name + ".lt", (n, k), salt=salt)
    l = l * 3.0
  return torch.softmax(l, 1), torch.softmax(lt, 1)


def iid_cases():
  cases = {}
  cases["c1_indep_256x10"] = softmax_pair("c1", 256, 10) + (1.0,)
  cases["corr_704x10"] = softmax_pair("c2", 704, 10, corr=0.5) + (1.0,)
  cases["corr_704x70"] = softmax_pair("c3", 704, 70, corr=0.5) + (1.0,)
  cases["corr_140x10_lamb1p5"] = softmax_pair("c4", 140, 10, corr=0.5) + (1.5,)
  cases["ragged_37x3_lamb2"] = softmax_pair("c5", 37, 3, corr=1.0) + (2.0,)
  # a cluster that is never used by either view: its row/col of P is < EPS and
  # hits all three clamps of IID_losses.py:17-19
  z, zt = softmax_pair("c6", 200, 10, corr=0.5)
  z[:, 3] = 0.
  zt[:, 3] = 0.
  z = z / z.sum(1, keepdim=True)
  zt = zt / zt.sum(1, keepdim=True)
  cases["zero_cluster_200x10"] = (z, zt, 1.0)
  # perfectly balanced one-hot, identical views: loss = -log k
  oh = torch.eye(10).repeat(70, 1)
  cases["onehot_700x10"] = (oh.clone(), oh.clone(), 1.0)
  return cases


def gen_iid(ref, out):
  for name, (z, zt, lamb) in iid_cases().items():
    with torch.no_grad():
      rl, rl1 = ref.IID_loss(z.clone(), zt.clone(), lamb=lamb)
      rj = ref.compute_joint(z.clone(), zt.clone())
    ol, ol1 = iid_losses.IID_loss(z, zt, lamb=lamb)
    assert float(rl) == float(ol) and float(rl1) == float(ol1), (name, rl, ol)
    zd = z.double().requires_grad_(True)
    ztd = zt.double().requires_grad_(True)
    l64, l64_1 = iid_losses.IID_loss(zd, ztd, lamb=lamb)
    gz, gzt = torch.autograd.grad(l64, [zd, ztd])
    cf = iid_losses.iid_loss_closed_form(z.numpy(), zt.numpy(), lamb=lamb)
    assert abs(cf["loss"] - float(l64)) < 1e-12
    assert np.abs(cf["dz"] - gz.numpy()).max() < 1e-12 * max(1.0, np.abs(cf["dz"]).max())
    out["iid/%s/z" % name] = z.numpy()
    out["iid/%s/zt" % name] = zt.numpy()
    out["iid/%s/lamb" % name] = np.float64(lamb)
    out["iid/%s/ref_loss" % name] = np.float32(rl)
    out["iid/%s/ref_loss_no_lamb" % name] = np.float32(rl1)
    out["iid/%s/ref_joint" % name] = rj.numpy()
    out["iid/%s/orc_loss_f64" % name] = np.float64(l64)
    out["iid/%s/orc_loss_no_lamb_f64" % name] = np.float64(l64_1)
    out["iid/%s/orc_dz_f64" % name] = gz.numpy()
    out["iid/%s/orc_dzt_f64" % name] = gzt.numpy()
    print("iid", name, float(rl), float(rl1))


def seg_inputs(name, n, k, h, flips=True, affine=False):
  x1 = torch.softmax(2.0 * weights.normal(name + ".x1", (n, k, h, h)), 1)
  x2 = torch.softmax(2.0 * weights.normal(name + ".x2", (n, k, h, h)) +
                     2.0 * torch.log(x1), 1)
  theta = torch.zeros(n, 2, 3)
  theta[:, 0, 0] = 1.
  theta[:, 1, 1] = 1.
  if flips:
    theta[::2, 0, 0] = -1.  # h-flip, as cocostuff.py:208-220 generates
  if affine:  # inverse rot/shear/scale without translation (seg transforms.py:115-121)
    a, sh, sc = np.radians(20.), np.radians(5.), 1.1
    m = np.array([[np.cos(a) * sc, -np.sin(a + sh) * sc, 0.], [np.sin(a) * sc, np.cos(a + sh) * sc, 0.],
                  [0., 0., 1.]], dtype=np.float32)
    theta[1] = torch.from_numpy(np.linalg.inv(m).astype(np.float32)[:2])
  mask = (weights.uniform(name + ".mask", (n, h, h)) < 0.7).float()
  return x1, x2, theta, mask


def gen_seg(ref, out):
  specs = {"small_n3_k4_16_T3": (3, 4, 16, 3, 1.5, True, False),
           "k15_n2_32_T10": (2, 15, 32, 10, 1.0, True, False),
           "k3_n4_24_T5_affine": (4, 3, 24, 5, 1.5, True, True)}
  for name, (n, k, h, T, lamb, flips, affine) in specs.items():
    x1, x2, theta, mask = seg_inputs("seg." + name, n, k, h, flips, affine)
    for variant, fn in [("collapsed", ref.IID_segmentation_loss),
                        ("uncollapsed", ref.IID_segmentation_loss_uncollapsed)]:
      a = x1.clone().requires_grad_(True)
      b = x2.clone().requires_grad_(True)
      l, l1 = fn(a, b, all_affine2_to_1=theta, all_mask_img1=mask, lamb=lamb, half_T_side_dense=T,
                 half_T_side_sparse_min=0, half_T_side_sparse_max=0)
      ga, gb = torch.autograd.grad(l, [a, b])
      p = "seg/%s/%s/" % (name, variant)
      out[p + "ref_loss"] = np.float32(l.item())
      out[p + "ref_loss_no_lamb"] = np.float32(l1.item())
      out[p + "ref_dx1"] = ga.numpy()
      out[p + "ref_dx2"] = gb.numpy()
      print("seg", name, variant, l.item(), l1.item())
    out["seg/%s/x1" % name] = x1.numpy()
    out["seg/%s/x2" % name] = x2.numpy()
    out["seg/%s/theta" % name] = theta.numpy()
    out["seg/%s/mask" % name] = mask.numpy()
    out["seg/%s/meta" % name] = np.array([n, k, h, T, lamb], dtype=np.float64)


NET_SPECS = {
  # name: (ctor, config, batch, head, lamb)
  "5g2h_32_A": ("ClusterNet5gTwoHead", dict(in_channels=2, input_sz=32, num_sub_heads=5, output_k_A=70,
                                           output_k_B=10, batchnorm_track=True), 6, "A", 1.0),
  "5g2h_32_B": ("ClusterNet5gTwoHead", dict(in_channels=2, input_sz=32, num_sub_heads=5, output_k_A=70,
                                           output_k_B=10, batchnorm_track=False), 6, "B", 1.0),
  "5g2h_96_B": ("ClusterNet5gTwoHead", dict(in_channels=2, input_sz=96, num_sub_heads=5, output_k_A=70,
                                           output_k_B=10, batchnorm_track=True), 3, "B", 1.0),
  "5g_64": ("ClusterNet5g", dict(in_channels=2, input_sz=64, num_sub_heads=3, output_k=10,
                                 batchnorm_track=True), 3, None, 1.0),
  "6c2h_24_A": ("ClusterNet6cTwoHead", dict(in_channels=1, input_sz=24, num_sub_heads=5, output_k_A=50,
                                           output_k_B=10, batchnorm_track=False), 8, "A", 1.0),
  "6c_24": ("ClusterNet6c", dict(in_channels=1, input_sz=24, num_sub_heads=2, output_k=10,
                                 batchnorm_track=True), 5, None, 1.0),
}


def net_input(name, cfg, batch):
  x = weights.normal(name + ".x", (batch, cfg["in_channels"], cfg["input_sz"], cfg["input_sz"]))
  xt = x + 0.3 * weights.normal(name + ".xt", tuple(x.shape))
  return x, xt


def gen_nets(ref, out):
  for name, (ctor, cfg, batch, head, lamb) in NET_SPECS.items():
    net = getattr(ref, ctor)(Namespace(**cfg))
    weights.fill_state_dict(net)
    net.train()
    x, xt = net_input("net." + name, cfg, batch)
    kw = {} if head is None else {"head": head}
    o = net(x, **kw)
    ot = net(xt, **kw)
    feat = None
    loss = 0.
    for a, b in zip(o, ot):
      l, _ = iid_losses.IID_loss(a, b, lamb=lamb)
      loss = loss + l
    loss = loss / len(o)
    loss.backward()
    p = "net/%s/" % name
    out[p + "ref_out"] = torch.stack(o).detach().numpy()
    out[p + "ref_out_tf"] = torch.stack(ot).detach().numpy()
    out[p + "loss"] = np.float32(loss.item())
    net.zero_grad(set_to_none=False) if False else None
    names, norms = [], []
    for pn, pp in net.named_parameters():
      g = pp.grad
      names.append(pn)
      norms.append(0.0 if g is None else float(g.double().norm()))
      if g is not None and (g.numel() <= 4096 or pn.endswith("conv1.weight") and "layer" not in pn):
        out[p + "grad/" + pn] = g.numpy().copy()
    out[p + "grad_names"] = np.array(names)
    out[p + "grad_norms"] = np.array(norms)
    if cfg["batchnorm_track"]:
      sd = net.state_dict()
      for key in sd:
        if key.endswith("running_mean") or key.endswith("running_var"):
          if sd[key].numel() <= 64 or "layer4.2.bn2" in key:
            out[p + "buf/" + key] = sd[key].numpy().copy()
    with torch.no_grad():
      net.eval()
      f = net(x, trunk_features=True, **kw)
      out[p + "ref_trunk_eval"] = f.numpy() if f.numel() <= 65536 else f[:, :512].numpy()
    print("net", name, loss.item())


def gen_seg_nets(ref, out):
  cfg = dict(in_channels=5, input_sz=32, num_sub_heads=1, output_k_A=15, output_k_B=3, batchnorm_track=True)
  net = ref.SegmentationNet10aTwoHead(Namespace(**cfg))
  weights.fill_state_dict(net, head_gain=20.0)
  net.train()
  name = "10a2h_32"
  x, xt = net_input("net." + name, cfg, 2)
  theta = torch.zeros(2, 2, 3)
  theta[:, 0, 0] = 1.
  theta[:, 1, 1] = 1.
  theta[1, 0, 0] = -1.
  mask = (weights.uniform("net.%s.mask" % name, (2, 32, 32)) < 0.7).float()
  for head, lamb in [("A", 1.0), ("B", 1.5)]:
    net.zero_grad()
    o = net(x, head=head)[0]
    ot = net(xt, head=head)[0]
    l, l1 = ref.IID_segmentation_loss_uncollapsed(o, ot, all_affine2_to_1=theta, all_mask_img1=mask, lamb=lamb,
                                                  half_T_side_dense=4, half_T_side_sparse_min=0,
                                                  half_T_side_sparse_max=0)
    l.backward()
    p = "net/%s_%s/" % (name, head)
    out[p + "ref_out"] = o.detach().numpy()
    out[p + "ref_out_tf"] = ot.detach().numpy()
    out[p + "loss"] = np.float32(l.item())
    out[p + "loss_no_lamb"] = np.float32(l1.item())
    names, norms = [], []
    for pn, pp in net.named_parameters():
      g = pp.grad
      names.append(pn)
      norms.append(0.0 if g is None else float(g.double().norm()))
      if g is not None and g.numel() <= 8192:
        out[p + "grad/" + pn] = g.numpy().copy()
    out[p + "grad_names"] = np.array(names)
    out[p + "grad_norms"] = np.array(norms)
    print("segnet", head, l.item(), l1.item())
  out["net/%s/theta" % name] = theta.numpy()
  out["net/%s/mask" % name] = mask.numpy()


def gen_precision(ref, out):
  """The well-conditioned end-to-end fixture (tests/precision_fixture.py) evaluated by the UNMODIFIED reference
  network: ClusterNet5gTwoHead 32x32, 64 pairs, centred sub-head biases, head gain 200.  It pins the oracle at the
  operating point where the tensor-core modes are given their stated tolerances (tests/test_gpu_precision.py)."""
  sys.path.insert(0, os.path.dirname(HERE))
  import precision_fixture as fx
  for sz, pairs, head in [(32, 64, "B")]:
    net = ref.ClusterNet5gTwoHead(Namespace(**fx.config(sz)))
    trunk_mean = fx.prepare(net, sz, pairs, head)
    net.train()
    x, xt = fx.inputs(sz, pairs)
    o, ot = net(x, head=head), net(xt, head=head)
    loss = sum(iid_losses.IID_loss(a, b)[0] for a, b in zip(o, ot)) / len(o)
    loss.backward()
    p = "wc/%d_%d_%s/" % (sz, pairs, head)
    out[p + "trunk_mean"] = trunk_mean.numpy()
    out[p + "ref_out"] = torch.stack(o).detach().numpy()
    out[p + "ref_out_tf"] = torch.stack(ot).detach().numpy()
    out[p + "loss"] = np.float64(loss.item())
    names, norms = [], []
    for pn, pp in net.named_parameters():
      g = pp.grad
      names.append(pn)
      norms.append(0.0 if g is None else float(g.double().norm()))
      if g is not None and (g.numel() <= 4096 or pn in ("trunk.layer1.0.conv1.weight", "trunk.layer2.0.downsample.0.weight")):
        out[p + "grad/" + pn] = g.numpy().copy()
    out[p + "grad_names"] = np.array(names)
    out[p + "grad_norms"] = np.array(norms)
    print("precision fixture", sz, pairs, head, loss.item())


def live_iid_inputs():
  z, zt = softmax_pair("live", 333, 13, corr=0.4)
  return z, zt, 1.2


def sparse_inputs():
  """Input of random_translation_multiple, and inputs of the segmentation losses with a sparse displacement window."""
  return weights.normal("sparse.x", (2, 3, 12, 12)), seg_inputs("seg.sparse", 3, 4, 16, flips=True)


SPARSE_SEEDS = range(6)  # np.random.seed before each random_translation_multiple(x, 2, 4)
SPARSE_LOSS_SEED = 11  # np.random.seed before each loss call
SPARSE_LOSS_KW = dict(lamb=1.2, half_T_side_dense=2, half_T_side_sparse_min=1, half_T_side_sparse_max=3)

# networks whose reference state_dict layout (key order, shapes, dtypes) a checkpoint carries
CHECKPOINT_SPECS = {
  "ClusterNet5gTwoHead": dict(in_channels=2, input_sz=32, num_sub_heads=3, output_k_A=20, output_k_B=5, batchnorm_track=True),
  "ClusterNet6cTwoHead": dict(in_channels=1, input_sz=24, num_sub_heads=2, output_k_A=12, output_k_B=4, batchnorm_track=False),
  "SegmentationNet10aTwoHead": dict(in_channels=5, input_sz=32, num_sub_heads=1, output_k_A=6, output_k_B=3, batchnorm_track=True),
}


def gen_calls(ref, out):
  """Single calls into the reference whose results the oracle must reproduce exactly: IID_loss, the seeded sparse
  displacement of the segmentation losses, and the state_dict layout a reference checkpoint has."""
  from oracle import seg_losses
  z, zt, lamb = live_iid_inputs()
  with torch.no_grad():
    r = ref.IID_loss(z.clone(), zt.clone(), lamb=lamb)
  out["iid_live/ref_loss"] = np.float32(r[0])
  out["iid_live/ref_loss_no_lamb"] = np.float32(r[1])
  o = iid_losses.IID_loss(z, zt, lamb=lamb)
  assert float(r[0]) == float(o[0]) and float(r[1]) == float(o[1])
  x, (x1, x2, theta, mask) = sparse_inputs()
  shifted = []
  for seed in SPARSE_SEEDS:
    np.random.seed(seed)
    shifted.append(ref.random_translation_multiple(x, 2, 4))
    np.random.seed(seed)
    assert torch.equal(shifted[-1], seg_losses.random_translation_multiple(x, 2, 4))
  out["sparse/ref_translated"] = torch.stack(shifted).numpy()
  for fn_name in ("IID_segmentation_loss", "IID_segmentation_loss_uncollapsed"):
    np.random.seed(SPARSE_LOSS_SEED)
    a, b = x1.clone().requires_grad_(True), x2.clone().requires_grad_(True)
    l, l1 = getattr(ref, fn_name)(a, b, all_affine2_to_1=theta, all_mask_img1=mask, **SPARSE_LOSS_KW)
    ga, gb = torch.autograd.grad(l, [a, b])
    p = "sparse/%s/" % fn_name
    out[p + "ref_loss"] = np.float32(l.item())
    out[p + "ref_loss_no_lamb"] = np.float32(l1.item())
    out[p + "ref_dx1"] = ga.numpy()
    out[p + "ref_dx2"] = gb.numpy()
    print("sparse", fn_name, l.item(), l1.item())
  for name, cfg in CHECKPOINT_SPECS.items():
    sd = getattr(ref, name)(Namespace(**cfg)).state_dict()
    p = "checkpoint/%s/" % name
    out[p + "keys"] = np.array(list(sd))
    out[p + "shapes"] = np.array([",".join(map(str, v.shape)) for v in sd.values()])
    out[p + "dtypes"] = np.array([str(v.dtype).replace("torch.", "") for v in sd.values()])
    print("checkpoint", name, len(sd), "entries")


def main():
  assert refshim.available(), "needs /root/reference"
  ref = refshim.load()
  only = sys.argv[1:]
  for fname, gens in [("iid_loss.npz", [gen_iid]), ("seg_loss.npz", [gen_seg]),
                      ("nets.npz", [gen_nets, gen_seg_nets]), ("precision.npz", [gen_precision]),
                      ("reference_calls.npz", [gen_calls])]:
    if only and fname not in only:
      continue
    out = {}
    for g in gens:
      g(ref, out)
    path = os.path.join(HERE, fname)
    np.savez_compressed(path, **{k.replace("/", "|"): v for k, v in out.items()})
    print("wrote", path, os.path.getsize(path) // 1024, "KiB")


if __name__ == "__main__":
  main()
