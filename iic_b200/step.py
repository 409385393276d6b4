"""The per-batch training step of the reference's scripts, written against the drop-in API.

Clustering (code/scripts/cluster/cluster_sobel_twohead.py:286-355):
    zero_grad -> sobel_process(x), sobel_process(x_tf) -> net(x, head), net(x_tf, head)
    -> IID_loss per sub-head, mean -> backward -> (all-reduce of gradients) -> optimiser.step()
Segmentation (code/scripts/segmentation/segmentation_twohead.py:262-361):
    zero_grad -> sobel_process(x, include_rgb), ... -> net(x, head), net(x_tf, head)
    -> IID_segmentation_loss(_uncollapsed) per sub-head with the batch's affine2_to_1 / mask, mean -> backward -> step
Semi-supervised finetune (code/scripts/semisup/IID_semisup_STL10.py:241-256):
    sobel_process(x) -> SupHead5 logits -> cross-entropy -> zero_grad (trunk, head) -> backward -> two Adam steps

Inputs are the image batches the dataloaders hand to the script (host or device tensors; host tensors are copied on
the current stream).  ``set_to_none=False`` is the reference's behaviour (torch 0.4.1 ``zero_grad`` zero-fills, so the
head that is not being trained keeps receiving Adam moment decay once it has been trained); pass ``arena=GradArena(net)``
to keep all gradients in one flat buffer (one memset, gradients written in place by the backward, bucketed all-reduce
overlapped with the backward under torch.distributed)."""
import torch

from . import distributed
from .utils.cluster.IID_losses import IID_loss_subheads
from .utils.cluster.transforms import rgb_sobel_process, sobel_process


def _zero(net, optimiser, arena, set_to_none, overlap):
  if arena is not None:
    arena.begin_step(overlap=overlap)
    if optimiser is not None and hasattr(optimiser, "grad_filter"):
      optimiser.grad_filter = arena.is_live
  elif optimiser is not None:
    optimiser.zero_grad(set_to_none=set_to_none)
  else:
    net.zero_grad(set_to_none=set_to_none)


def _finish(net, optimiser, arena):
  if arena is not None:
    arena.flush()
  else:
    distributed.allreduce_gradients(net.parameters())
  if optimiser is not None:
    optimiser.step()


def _to_net_input(imgs, sobel, include_rgb):
  """Dataloader tensor -> network input: sobel_process as the scripts call it; an RGB (n,3,h,w) batch (uint8 or fp32)
  with include_rgb=False takes the fused grey + sobel kernel (the grey conversion the reference does on the CPU)."""
  if not sobel:
    return imgs
  if imgs.shape[1] == 3 and not include_rgb:
    return rgb_sobel_process(imgs)
  return sobel_process(imgs, include_rgb)


def iic_cluster_step(net, optimiser, imgs, imgs_tf, head="B", lamb=1.0, include_rgb=False, sobel=True,
                     set_to_none=False, pair_batched=True, arena=None, repeats=1):
  """Returns (avg_loss, avg_loss_no_lamb) as 0-dim device tensors (no host sync).

  ``repeats`` = R > 1 (SURVEY S8f row 2): the reference builds view 1 by copying the SAME tf1 mini-batch into every one
  of its ``num_dataloaders`` slabs (cluster_sobel_twohead.py:303-306), so each image is pushed through the net R times.
  Here ``imgs`` holds the n unique images and ``imgs_tf`` the R*n transformed ones (slab order); the trunk runs once on
  the unique images and their softmax rows are repeated.  Loss and all parameter gradients equal the reference's
  slab-assembled step (BatchNorm's batch mean / biased variance do not change when every sample appears R times, and
  its backward is linear in the incoming gradient); only the running_var's unbiased correction differs,
  m/(m-1) with m = n*h*w instead of R*n*h*w.  An algorithmic saving outside the roofline accounting: 2R -> R+1 trunk
  passes per unique image."""
  pair = hasattr(net, "forward_stacked_pair") and pair_batched and repeats == 1
  _zero(net, optimiser, arena, set_to_none, overlap=pair)
  dev = next(net.parameters()).device
  if not imgs.is_cuda:
    imgs = imgs.to(dev, non_blocking=True)
    imgs_tf = imgs_tf.to(dev, non_blocking=True)
  assert imgs_tf.shape[0] == repeats * imgs.shape[0], "imgs_tf must hold `repeats` transformed copies of every image"
  imgs = _to_net_input(imgs, sobel, include_rgb)
  imgs_tf = _to_net_input(imgs_tf, sobel, include_rgb)
  if repeats > 1:
    assert hasattr(net, "forward_stacked"), "repeats needs a network with forward_stacked"
    x_outs = net.forward_stacked(imgs, head=head).repeat(1, repeats, 1)  # [S, R*n, k] in slab order
    x_tf_outs = net.forward_stacked(imgs_tf, head=head)
  elif pair:
    x_outs, x_tf_outs = net.forward_stacked_pair(imgs, imgs_tf, head=head)
  elif hasattr(net, "forward_stacked"):
    x_outs = net.forward_stacked(imgs, head=head)
    x_tf_outs = net.forward_stacked(imgs_tf, head=head)
  else:
    x_outs, x_tf_outs = net(imgs), net(imgs_tf)
  loss, loss_no_lamb = IID_loss_subheads(x_outs, x_tf_outs, lamb=lamb)
  avg_loss, avg_loss_no_lamb = loss.mean(), loss_no_lamb.mean()
  avg_loss.backward()
  _finish(net, optimiser, arena)
  return avg_loss.detach(), avg_loss_no_lamb.detach()


def assemble_slabs(imgs, imgs_tf_list, device=None):
  """The slab assembly of cluster_sobel_twohead.py:290-318 without its zero-filled staging tensors: returns
  (all_imgs, all_imgs_tf) with the tf1 batch copied into every slab and the d-th transformed batch into slab d
  (host tensors are uploaded straight into their slab, non-blocking)."""
  R, n = len(imgs_tf_list), imgs.shape[0]
  device = device or (imgs.device if imgs.is_cuda else torch.device("cuda", torch.cuda.current_device()))
  all_imgs = torch.empty((R * n,) + tuple(imgs.shape[1:]), device=device, dtype=imgs.dtype)
  all_tf = torch.empty((R * n,) + tuple(imgs_tf_list[0].shape[1:]), device=device, dtype=imgs_tf_list[0].dtype)
  for d, t in enumerate(imgs_tf_list):
    assert t.shape[0] == n
    all_imgs[d * n:(d + 1) * n].copy_(imgs, non_blocking=True)
    all_tf[d * n:(d + 1) * n].copy_(t, non_blocking=True)
  return all_imgs, all_tf


def iic_seg_step(net, optimiser, imgs, imgs_tf, affine2_to_1, mask_img1, head="B", lamb=1.0, half_T_side_dense=10,
                 half_T_side_sparse_min=0, half_T_side_sparse_max=0, uncollapsed=True, include_rgb=True, sobel=True,
                 set_to_none=False, arena=None):
  """One batch of segmentation_twohead.py:262-361.  ``imgs`` are the (n, 4, h, w) rgb+grey batches of the dataloader
  when ``sobel`` (-> 5 channels, utils/segmentation/general.py:5-11 of the reference), else the network input itself.
  Returns (avg_loss, avg_loss_no_lamb) as 0-dim device tensors."""
  from .utils.segmentation.IID_losses import IID_segmentation_loss, IID_segmentation_loss_uncollapsed
  loss_fn = IID_segmentation_loss_uncollapsed if uncollapsed else IID_segmentation_loss
  _zero(net, optimiser, arena, set_to_none, overlap=False)
  dev = next(net.parameters()).device
  if not imgs.is_cuda:
    imgs, imgs_tf = imgs.to(dev, non_blocking=True), imgs_tf.to(dev, non_blocking=True)
    affine2_to_1, mask_img1 = affine2_to_1.to(dev, non_blocking=True), mask_img1.to(dev, non_blocking=True)
  imgs = _to_net_input(imgs, sobel, include_rgb)
  imgs_tf = _to_net_input(imgs_tf, sobel, include_rgb)
  x_outs = net(imgs, head=head)
  x_tf_outs = net(imgs_tf, head=head)
  avg_loss = avg_loss_no_lamb = None
  for i in range(len(x_outs)):
    loss, loss_no_lamb = loss_fn(x_outs[i], x_tf_outs[i], all_affine2_to_1=affine2_to_1, all_mask_img1=mask_img1,
                                 lamb=lamb, half_T_side_dense=half_T_side_dense,
                                 half_T_side_sparse_min=half_T_side_sparse_min,
                                 half_T_side_sparse_max=half_T_side_sparse_max)
    avg_loss = loss if avg_loss is None else avg_loss + loss
    avg_loss_no_lamb = loss_no_lamb if avg_loss_no_lamb is None else avg_loss_no_lamb + loss_no_lamb
  avg_loss = avg_loss / len(x_outs)
  avg_loss_no_lamb = avg_loss_no_lamb / len(x_outs)
  avg_loss.backward()
  _finish(net, optimiser, arena)
  return avg_loss.detach(), avg_loss_no_lamb.detach()


def iic_semisup_step(net, optimisers, imgs, targets, penultimate_features=False, include_rgb=False, sobel=True, arena=None):
  """One batch of the semi-supervised finetune (code/scripts/semisup/IID_semisup_STL10.py:241-256): sobel_process ->
  net(imgs, penultimate_features) -> nn.CrossEntropyLoss() -> zero_grad of both optimisers -> backward -> opt_trunk.step(),
  opt_head.step().  ``net`` is a SupHead5, ``optimisers`` the (opt_trunk, opt_head) pair of FusedAdam over
  ``net.trunk.parameters()`` and ``net.head.parameters()``.  The sub-heads inside the trunk receive no gradient and are not
  stepped, as in the reference.  Returns the loss as a 0-dim device tensor (no host sync)."""
  from .utils.semisup.general import CrossEntropyLoss
  opt_trunk, opt_head = optimisers
  _zero(net, opt_trunk, arena, False, overlap=True)  # (every parameter gets its gradient from one backward node)
  if arena is not None:
    opt_head.grad_filter = arena.is_live
  else:
    opt_head.zero_grad(set_to_none=False)
  dev = next(net.parameters()).device
  if not imgs.is_cuda:
    imgs = imgs.to(dev, non_blocking=True)
  if not targets.is_cuda:
    targets = targets.to(dev, non_blocking=True)
  imgs = _to_net_input(imgs, sobel, include_rgb)
  x_out = net(imgs, penultimate_features=penultimate_features)
  loss = CrossEntropyLoss()(x_out, targets)
  loss.backward()
  _finish(net, opt_trunk, arena)
  opt_head.step()
  return loss.detach()
