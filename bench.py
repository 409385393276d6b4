#!/usr/bin/env python
"""Benchmark of the IIC training hot path (BASELINE.json metric): img-pairs/s through
ClusterNet5gTwoHead + IID_loss (k=10 head B, 5 sub-heads) on synthetic 96x96 batches.

    python bench.py --gpus N --steps K --warmup W            # this repo's sm_100a path, default workload c4
    python bench.py --config {c2,c3,c4,c4-strong,c5}         # the other BASELINE.json configurations
    python bench.py --impl reference ...                     # the reference algorithm on the host CPUs
    torchrun ... bench.py --gpus N                           # N > 1 also checks N-rank result == one-device sharded
                                                             # emulation (parity_ok; --no-verify to skip, --verify at N = 1)

A step = one pass of the reference's per-batch loop (cluster_sobel_twohead.py:286-355 / segmentation_twohead.py:
262-361): zero_grad, (grey+)sobel x2, net(x), net(x_tf), IID loss over the sub-heads, backward, gradient all-reduce
(N>1, overlapped with the backward), Adam step.  `value` times it with the image batches already resident in HBM;
`e2e` times the same call with PINNED HOST batches (H2D inside the timed region, loss read back).
Prints ONE JSON line on rank 0.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "img-pairs/s through ClusterNet5g+IID_loss at 1/2/4/8 B200 vs CPU ref"

# BASELINE.json configs (SURVEY.md S8 "Config shorthand"); flop = algorithmic conv FLOPs per image pair (2*MAC,
# fprop + dgrad + wgrad, both views; SURVEY.md S8d).  scaling "weak": `batch` pairs per GPU; "strong": `batch` global.
CONFIGS = {
  "c2": dict(net="ClusterNet6cTwoHead", cfg=dict(in_channels=1, input_sz=24, num_sub_heads=5, output_k_A=50, output_k_B=10,
                                                 batchnorm_track=False),
             batch=700, scaling="weak", flop=1.069e9 + 0.0, kind="cluster", sobel=False, rgb=False, cpu_pairs=256,
             desc="MNIST-shape ClusterNet6cTwoHead(24x24 grey, 5 sub-heads, k_A=50/k_B=10)"),
  "c3": dict(net="ClusterNet5gTwoHead", cfg=dict(in_channels=2, input_sz=32, num_sub_heads=5, output_k_A=70, output_k_B=10,
                                                 batchnorm_track=False),
             batch=660, scaling="strong", flop=5.32e9, kind="cluster", sobel=True, rgb=True, cpu_pairs=128,
             desc="CIFAR10-shape ClusterNet5gTwoHead(32x32, sobel 2ch, 5 sub-heads, k_A=70/k_B=10)"),
  "c4": dict(net="ClusterNet5gTwoHead", cfg=dict(in_channels=2, input_sz=96, num_sub_heads=5, output_k_A=70, output_k_B=10,
                                                 batchnorm_track=True),
             batch=704, scaling="weak", flop=36342890496.0, kind="cluster", sobel=True, rgb=True, cpu_pairs=32,
             desc="STL10-shape ClusterNet5gTwoHead(96x96, sobel 2ch, 5 sub-heads, k_A=70/k_B=10)"),
  "c4-strong": dict(net="ClusterNet5gTwoHead", cfg=dict(in_channels=2, input_sz=96, num_sub_heads=5, output_k_A=70,
                                                        output_k_B=10, batchnorm_track=True),
                    batch=704, scaling="strong", flop=36342890496.0, kind="cluster", sobel=True, rgb=True, cpu_pairs=32,
                    desc="STL10-shape ClusterNet5gTwoHead(96x96, sobel 2ch, 5 sub-heads, k_A=70/k_B=10), 704 pairs GLOBAL"),
  "c5": dict(net="SegmentationNet10aTwoHead", cfg=dict(in_channels=5, input_sz=128, num_sub_heads=1, output_k_A=15,
                                                       output_k_B=3, batchnorm_track=True),
             batch=120, scaling="strong", flop=215.05e9, kind="seg", sobel=True, rgb=True, cpu_pairs=4,
             desc="COCO-Stuff-3-shape SegmentationNet10aTwoHead(128x128, rgb+sobel 5ch, k_A=15/k_B=3), "
                  "IID_segmentation_loss half_T_side_dense=10"),
}


# Defaults that depend on code having run on a B200 (flipped by hand after tools/gpu_r2_a.sh passes): until then the
# default command line takes round 1's validated path, so that the driver's round-end run cannot be broken by a kernel
# that has never executed.  Every item stays selectable from the command line.
VALIDATED = {"arena": True, "rgb_input": True, "also": "tf32x3"}  # arena / rgb: gpurun_out/a_tests.log, a_bench.json (round 2, session A)


def parse():
  ap = argparse.ArgumentParser()
  ap.add_argument("--gpus", type=int, default=1)
  ap.add_argument("--steps", type=int, default=10)
  ap.add_argument("--warmup", type=int, default=3)
  ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
  ap.add_argument("--config", default="c4", choices=sorted(CONFIGS))
  ap.add_argument("--pairs-per-gpu", type=int, default=0, help="override the configuration's batch (per GPU)")
  ap.add_argument("--precision", default="bf16", choices=["bf16", "tf32", "tf32x3", "fp32"])
  ap.add_argument("--also", default=VALIDATED["also"], help="comma list of further precision modes measured briefly at N=1 "
                                                   "(reported under precision_modes); '' for none")
  ap.add_argument("--head", default=None, help="A | B (default: B for clustering, A for segmentation)")
  ap.add_argument("--seg-collapsed", action="store_true", help="c5: IID_segmentation_loss instead of _uncollapsed")
  ap.add_argument("--grey-input", dest="grey_input", action="store_true", default=not VALIDATED["rgb_input"],
                  help="clustering: feed 1-channel grey batches (round-1 bench input) instead of RGB -> grey -> sobel")
  ap.add_argument("--rgb-input", dest="grey_input", action="store_false", help="clustering: RGB batches, fused grey + sobel")
  ap.add_argument("--cpu-pairs", type=int, default=0, help="bounded CPU sample: image pairs per reference step")
  ap.add_argument("--no-cpu-baseline", action="store_true")
  ap.add_argument("--no-roofline", action="store_true")
  ap.add_argument("--no-arena", dest="no_arena", action="store_true", default=not VALIDATED["arena"],
                  help="round-1 gradient path (autograd accumulation, cat + all-reduce)")
  ap.add_argument("--arena", dest="no_arena", action="store_false",
                  help="flat in-place gradients, bucketed all-reduce overlapped with the backward")
  ap.add_argument("--graph", action="store_true", help="capture the step into a CUDA graph and replay it (needs --arena): "
                                                       "removes the ~4 ms of host launch work per step that bounds small per-GPU batches")
  ap.add_argument("--verify", action="store_true", help="check the N-rank loss / gradient checksum against the one-device "
                                                        "emulation of the sharded algorithm; adds parity_ok to the line "
                                                        "(on by default for N > 1; untimed, ~2 s)")
  ap.add_argument("--no-verify", action="store_true")
  ap.add_argument("--layer-table", action="store_true", help="add the live per-geometry conv table to roofline.by_layer")
  ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                  help="write what the last timed step returned and left in the network (losses, parameters, buffers, "
                       "gradients) as DIR/<name>.npy, to compare two builds output for output")
  a = ap.parse_args()
  if a.dump_outputs and a.impl != "ours":
    ap.error("--dump-outputs records this repo's timed path (--impl ours)")
  if a.head is None:
    a.head = "A" if CONFIGS[a.config]["kind"] == "seg" else "B"
  return a


def net_config(cname, precision=None):
  from argparse import Namespace
  cfg = dict(CONFIGS[cname]["cfg"])
  if precision is not None:
    cfg["precision"] = precision
  return Namespace(**cfg)


def peaks(precision="bf16"):
  path = os.path.join(ROOT, "MEASURED_PEAKS.json")
  if os.path.exists(path):
    with open(path) as f:
      p = json.load(f)
    bf16, src = float(p["bf16_tflops_sustained"]), "measured (MEASURED_PEAKS.json, sustained bf16 cuBLAS)"
    hbm = float(p["hbm_gbs"])
  else:
    bf16, hbm, src = 1400.0, 6650.0, "fallback (B200_PROFILING.md)"
  # tcgen05 kind::tf32 runs at half the kind::f16 rate; 3xTF32 issues three MMAs per product; the SIMT mode's ceiling
  # is the fp32 FMA rate (148 SMs x 128 lanes x 2 x 1.965 GHz)
  scale = {"bf16": 1.0, "tf32": 0.5, "tf32x3": 1.0 / 6.0}
  if precision == "fp32":
    return dict(tflops=148 * 128 * 2 * 1.965e9 / 1e12, hbm=hbm, src="fp32 FMA peak (148 SMs x 128 x 2 x 1.965 GHz)")
  tag = {"bf16": "", "tf32": " / 2 (kind::tf32)", "tf32x3": " / 6 (kind::tf32, three MMAs per product)"}[precision]
  return dict(tflops=bf16 * scale[precision], hbm=hbm, src=src + tag)


class ClockSampler(object):
  """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

  def __init__(self, index):
    self.index, self.rows, self.proc = index, [], None

  def start(self):
    q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    try:
      self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits",
                                    "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
      threading.Thread(target=self._read, daemon=True).start()
    except Exception:
      self.proc = None

  def _read(self):
    for line in self.proc.stdout:
      self.rows.append([c.strip() for c in line.split(",")])

  def stop(self):
    if self.proc is None:
      return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
    time.sleep(0.15)
    self.proc.terminate()
    sm, mx, reasons = [], None, set()
    names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
    for r in self.rows:
      try:
        sm.append(float(r[0]))
        mx = float(r[1])
        for nme, v in zip(names, r[3:7]):
          if v.lower().startswith("active"):
            reasons.add(nme)
      except Exception:
        pass
    sm.sort()
    return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


def host_threads():
  """One thread per PHYSICAL core this process may run on.  torch.distributed.run exports OMP_NUM_THREADS=1, which would
  otherwise pin the CPU arm to one thread (VERDICT r1: 4.3 pairs/s 'reference' numbers at N >= 2); one thread per logical
  CPU (128 on the B200 hosts) oversubscribes the 64 cores and is 5x slower than 64 threads (measured: 3.2 vs 16 pairs/s)."""
  try:
    logical = len(os.sched_getaffinity(0))
  except AttributeError:
    logical = os.cpu_count() or 1
  physical = None
  try:
    import psutil
    physical = psutil.cpu_count(logical=False)
  except Exception:
    pass
  if not physical:
    physical = max(1, logical // 2)
  return max(1, min(logical, physical))


def workload_config(args, pairs_per_gpu, n):
  c = CONFIGS[args.config]
  if c["kind"] == "seg":
    inp = "128x128 rgb+grey (4ch) pair -> sobel -> 5ch, per-image flip matrices, Bernoulli(0.7) masks"
    loss = "IID_segmentation_loss%s T=10" % ("" if args.seg_collapsed else "_uncollapsed")
  else:
    sz = c["cfg"]["input_sz"]
    if not c["sobel"]:
      inp = "%dx%dx1 grey pair" % (sz, sz)
    elif args.grey_input:
      inp = "%dx%dx1 grey pair -> sobel" % (sz, sz)
    else:
      inp = "%dx%dx3 uint8 rgb pair -> grey (PIL 'L' formula) -> sobel, fused on device" % (sz, sz)
    loss = "IID_loss lamb=1"
  return {"workload": "%s: %s head %s, %s, Adam" % (args.config, c["desc"], args.head, loss), "name": args.config,
          "pairs_per_gpu": pairs_per_gpu, "global_batch": pairs_per_gpu * n, "input": inp,
          "parallelism": "dp%d (pairs sharded, per-rank BN, all-reduce of the joint + weight grads%s)%s" % (
            n, "" if args.no_arena else ", bucketed in place and overlapped with the backward",
            ", step replayed from a CUDA graph" if args.graph else ""),
          "l2": "per-step working set far exceeds the 126 MB L2 (activations of one step: GBs); no explicit flush"}


def pairs_for(args, world):
  c = CONFIGS[args.config]
  if args.pairs_per_gpu:
    return args.pairs_per_gpu
  if c["scaling"] == "weak":
    return c["batch"]
  assert c["batch"] % world == 0, "%s: global batch %d does not divide over %d GPUs" % (args.config, c["batch"], world)
  return c["batch"] // world


def make_host_batch(args, B, seed, pin=True):
  """Synthetic dataloader output for one rank: the tensors the reference's loop receives (pinned host memory)."""
  import torch
  c = CONFIGS[args.config]
  g = torch.Generator().manual_seed(seed)
  sz = c["cfg"]["input_sz"]
  if c["kind"] == "seg":
    imgs = [torch.rand(B, 4, sz, sz, generator=g) for _ in range(2)]
    theta = torch.zeros(B, 2, 3)
    theta[:, 0, 0] = 1.
    theta[:, 1, 1] = 1.
    theta[torch.rand(B, generator=g) < 0.5, 0, 0] = -1.  # horizontal flip (cocostuff.py:208-220)
    mask = (torch.rand(B, sz, sz, generator=g) < 0.7).float()
    batch = imgs + [theta, mask]
  else:
    if c["sobel"] and c["rgb"] and not args.grey_input:
      # RGB as the dataloader holds it (PIL images are uint8); the grey conversion + sobel run fused on the device
      batch = [torch.randint(0, 256, (B, 3, sz, sz), generator=g, dtype=torch.uint8) for _ in range(2)]
    else:
      batch = [torch.rand(B, 1, sz, sz, generator=g) for _ in range(2)]
  return [t.pin_memory() for t in batch] if pin else batch


# ---------------------------------------------------------------------------------------------
# reference arm: the reference algorithm (oracle port of xu-ji/IIC) on the host cores
# ---------------------------------------------------------------------------------------------
def cpu_reference_step_fn(args, pairs):
  import torch

  from oracle import iid_losses as oracle_iid
  from oracle import nets as oracle_nets
  from oracle import seg_losses as oracle_seg
  from oracle import transforms as oracle_tf
  torch.set_num_threads(host_threads())
  c = CONFIGS[args.config]
  torch.manual_seed(0)
  net = getattr(oracle_nets, c["net"])(net_config(args.config))
  net.train()
  opt = torch.optim.Adam(net.parameters(), lr=1e-4)
  batch = make_host_batch(args, pairs, 7, pin=False)
  head = args.head

  def grey(x):  # custom_greyscale_to_tensor (code/utils/cluster/transforms.py:12-16)
    return x if x.shape[1] == 1 else oracle_tf.grey_from_rgb(x)

  def step():
    opt.zero_grad(set_to_none=False)
    if c["kind"] == "seg":
      x, xt = oracle_tf.sobel_process(batch[0], True), oracle_tf.sobel_process(batch[1], True)
      o, ot = net(x, head=head), net(xt, head=head)
      fn = oracle_seg.IID_segmentation_loss if args.seg_collapsed else oracle_seg.IID_segmentation_loss_uncollapsed
      loss = sum(fn(a, b, all_affine2_to_1=batch[2], all_mask_img1=batch[3], lamb=1.0, half_T_side_dense=10,
                    half_T_side_sparse_min=0, half_T_side_sparse_max=0)[0] for a, b in zip(o, ot)) / len(o)
    else:
      x, xt = grey(batch[0]), grey(batch[1])
      if c["sobel"]:
        x, xt = oracle_tf.sobel_process(x, False), oracle_tf.sobel_process(xt, False)
      o, ot = net(x, head=head), net(xt, head=head)
      loss = sum(oracle_iid.IID_loss(a, b)[0] for a, b in zip(o, ot)) / len(o)
    loss.backward()
    opt.step()
    return float(loss)

  return step


def time_cpu_reference(args, pairs, steps, warmup):
  """`steps` timed steps of `pairs` image pairs (fixed counts: the same sample on every box and at every N)."""
  import torch
  step = cpu_reference_step_fn(args, pairs)
  for _ in range(max(1, warmup)):
    step()
  t0 = time.time()
  for _ in range(steps):
    step()
  dt = (time.time() - t0) / steps
  c = CONFIGS[args.config]
  return dict(value=pairs / dt, unit="img-pairs/s", cores=torch.get_num_threads(), kind="port",
              sample="%d steps (+%d warm-up) of %d img-pairs of workload %s, oracle port of the reference (torch CPU fp32, "
                     "%d threads): %ssobel + net x2 + loss + backward + Adam" % (
                       steps, max(1, warmup), pairs, args.config, torch.get_num_threads(), "" if c["sobel"] else "no ")), dt


def run_reference(args):
  rank = int(os.environ.get("RANK", "0"))
  if rank != 0:
    return
  pairs = args.cpu_pairs or CONFIGS[args.config]["cpu_pairs"]
  base, dt = time_cpu_reference(args, pairs, args.steps, args.warmup)
  line = {"impl": "reference", "metric": METRIC, "value": base["value"], "unit": "img-pairs/s", "n_gpus": args.gpus,
          "steps": args.steps, "warmup": max(1, args.warmup), "ms_per_step": dt * 1e3, "higher_is_better": True,
          "scaling": CONFIGS[args.config]["scaling"], "vs_baseline": None, "dtype": "f32", "data": "synthetic",
          "config": workload_config(args, pairs, 1), "cpu_baseline": base,
          "e2e": {"value": base["value"], "unit": "img-pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
          "gpu_launches": 0}
  print(json.dumps(line))


# ---------------------------------------------------------------------------------------------
# this repo's arm
# ---------------------------------------------------------------------------------------------
class Job(object):
  """Network + optimiser + gradient arena of one precision mode, and the step the bench times."""

  def __init__(self, args, precision, dev):
    import iic_b200.archs as archs
    from iic_b200.arena import GradArena
    from iic_b200.optim import FusedAdam
    import torch
    self.args, self.c, self.precision = args, CONFIGS[args.config], precision
    torch.manual_seed(0)
    self.net = getattr(archs, self.c["net"])(net_config(args.config, precision)).to(dev)
    self.net.train()
    self.opt = FusedAdam(self.net.parameters(), lr=1e-4)
    self.arena = None if args.no_arena else GradArena(self.net)
    self.gstep = None

  def step(self, batch):
    from iic_b200.step import iic_cluster_step, iic_seg_step
    a, c = self.args, self.c
    if a.graph:
      if self.gstep is None:
        from iic_b200.graph import GraphedStep
        assert self.arena is not None, "--graph needs --arena"
        if c["kind"] == "seg":
          self.gstep = GraphedStep(self.net, self.opt, self.arena, batch, kind="seg", head=a.head, lamb=1.0,
                                   half_T_side_dense=10, uncollapsed=not a.seg_collapsed)
        else:
          self.gstep = GraphedStep(self.net, self.opt, self.arena, batch, kind="cluster", head=a.head, lamb=1.0,
                                   sobel=c["sobel"])
      return self.gstep(*batch)
    if c["kind"] == "seg":
      return iic_seg_step(self.net, self.opt, batch[0], batch[1], batch[2], batch[3], head=a.head, lamb=1.0,
                          half_T_side_dense=10, uncollapsed=not a.seg_collapsed, arena=self.arena)
    return iic_cluster_step(self.net, self.opt, batch[0], batch[1], head=a.head, lamb=1.0, sobel=c["sobel"],
                            arena=self.arena)


DUMP_SAMPLE = 1 << 15  # entries kept of a larger tensor by --dump-outputs
DUMP_LIMIT = 64 << 20  # bytes --dump-outputs may write


def dump_outputs(job, out, path):
  """Writes what a step handed its caller: the returned (loss, loss_no_lamb), and the parameters, buffers and gradients
  it left in the network, as float32 (integer buffers: float64) .npy files.  A tensor of more than DUMP_SAMPLE entries
  is reduced to DUMP_SAMPLE of its flat entries, at sorted indices drawn by a generator seeded with the tensor's name,
  so the sample is the same in every run and every build."""
  import zlib

  import numpy as np
  import torch
  arrays = {"loss": out[0], "loss_no_lamb": out[1]}
  for n, p in job.net.named_parameters():
    arrays["param." + n] = p
    if p.grad is not None:
      arrays["grad." + n] = p.grad
  for n, b in job.net.named_buffers():
    arrays["buffer." + n] = b
  os.makedirs(path, exist_ok=True)
  total = 0
  for name, t in arrays.items():
    a = t.detach().reshape(-1)
    if a.numel() > DUMP_SAMPLE:
      rng = np.random.default_rng(zlib.crc32(name.encode()))
      idx = np.sort(rng.choice(a.numel(), DUMP_SAMPLE, replace=False))
      a = a[torch.from_numpy(idx).to(a.device)]
    a = (a.float() if t.is_floating_point() else a.double()).cpu().numpy()
    if t.numel() <= DUMP_SAMPLE:
      a = a.reshape(tuple(t.shape))
    total += a.nbytes
    assert total <= DUMP_LIMIT, "--dump-outputs: more than %d bytes" % DUMP_LIMIT
    np.save(os.path.join(path, name + ".npy"), a)


def measure(job, resident, host, steps, warmup, world, dev, sampler=None, dump=None):
  """-> dict(sec, sec_e2e, launches, loss, clocks): device-timed (CUDA events, max over ranks) resident and e2e legs.
  ``dump``: directory for dump_outputs of the last resident step (rank 0)."""
  import torch
  import torch.distributed as dist

  from iic_b200 import kernels

  def barrier():
    if world > 1:
      dist.barrier()
    torch.cuda.synchronize()

  def timed(src, read_back):
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.time()
    e0.record()
    last = None
    for _ in range(steps):
      last = job.step(src)
      if read_back:
        last = (last[0].item(), last[1].item())  # device -> host read of the step's result
    e1.record()
    barrier()
    wall = time.time() - t0
    ms = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
    if world > 1:
      dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    return ms.item() / 1e3, wall, last

  for _ in range(warmup):
    job.step(resident)
  if sampler is not None:
    sampler.start()
  kernels.launch_count(reset=True)
  sec, wall, last = timed(resident, False)
  launches = kernels.launch_count()
  if getattr(job, "gstep", None) is not None:  # replays do not pass through the host-side counter
    launches += steps * job.gstep.launches_per_replay
  clocks = sampler.stop() if sampler is not None else None
  if dump is not None:
    dump_outputs(job, last, dump)
  job.step(host)
  sec_e, _, _ = timed(host, True)
  return dict(sec=sec, sec_e2e=sec_e, launches=launches, loss=float(last[0]), clocks=clocks, wall=wall)


def roofline(job, resident, sec_per_step, pairs, flop_per_pair, precision):
  import torch

  from iic_b200 import kernels
  kernels.conv_timing(True)
  for _ in range(2):
    job.step(resident)
  torch.cuda.synchronize()
  summ = kernels.conv_timing_summary()
  layers = kernels.conv_timing_by_layer() if getattr(job.args, "layer_table", False) else None
  kernels.conv_timing(False)
  pk = peaks(precision)
  other = {k: {"launches": v[0] // 2, "ms_per_step": v[2] / 2} for k, v in summ.items() if v[1] == 0.0}
  summ = {k: v for k, v in summ.items() if v[1] > 0.0}
  flops = sum(v[1] for v in summ.values())
  ms = sum(v[2] for v in summ.values())
  nl = sum(v[0] for v in summ.values())
  ach = flops / (ms * 1e-3) / 1e12 if ms > 0 else 0.0
  kernel = {"bf16": "conv_tc2_kernel / conv_halo_kernel (tcgen05 kind::f16 implicit-GEMM fprop/dgrad/wgrad)",
            "tf32": "conv_tf32_kernel<.,.,1> (tcgen05 kind::tf32 implicit GEMM on fp32 activations)",
            "tf32x3": "conv_tf32_kernel<.,.,3> (tcgen05 kind::tf32, 3xTF32 split: three MMAs per product)",
            "fp32": "simt conv kernels (fp32 FMA)"}[precision]
  traffic, tsrc = None, "not captured for this build / workload"
  tpath = os.path.join(ROOT, "profiles", "r02_traffic.json")
  if os.path.exists(tpath):
    try:
      with open(tpath) as f:
        t = json.load(f).get("%s/%s" % (job.args.config, precision))
      if t and t.get("pairs_per_gpu") == pairs:
        traffic, tsrc = t["dram_bytes_per_launch"], t["source"]
    except Exception:
      pass
  extra = {}
  if layers:
    extra["by_layer"] = {k: {"launches": v[0] // 2, "ms_per_step": round(v[2] / 2, 4),
                             "tflops": round(v[1] / (v[2] * 1e-3) / 1e12, 1)} for k, v in sorted(layers.items())}
  return {**extra, "bound": "tensor", "kernel": kernel, "achieved": ach, "peak": pk["tflops"], "unit": "TFLOP/s",
          "frac": ach / pk["tflops"], "traffic": traffic, "traffic_source": tsrc, "peak_source": pk["src"],
          "launches_timed": nl, "flop_per_launch_avg": flops / max(nl, 1), "ms_per_launch_avg": ms / max(nl, 1),
          "by_kind": {k: {"launches": v[0], "tflops": v[1] / (v[2] * 1e-3) / 1e12 if v[2] > 0 else 0.0,
                          "ms_per_step": v[2] / 2} for k, v in summ.items()},
          "conv_share_of_step": (ms / 2) / (sec_per_step * 1e3), "other_kernels_ms_per_step": other,
          "whole_step_frac": pairs / sec_per_step * flop_per_pair / 1e12 / pk["tflops"]}


def _verify_batch(args, B, seed, dev):
  """A pair of CORRELATED views (view 2 = view 1 + a few grey levels of noise): with the bench's independent random views
  the mutual information is zero whatever the network does."""
  import torch
  x = make_host_batch(args, B, seed, pin=False)[0]
  g = torch.Generator().manual_seed(seed + 77)
  if x.dtype == torch.uint8:
    xt = (x.int() + torch.randint(-6, 7, x.shape, generator=g)).clamp_(0, 255).to(torch.uint8)
  else:
    xt = (x + 0.03 * torch.randn(x.shape, generator=g)).clamp_(0, 1)
  return [x.to(dev), xt.to(dev)]


def _condition_for_verify(net, args, x):
  """The conditioning of tests/precision_fixture.py, applied on the device: head gain 200 and sub-head biases centred on
  the mean trunk feature of ``x``.  A randomly initialised IIC network has collapsed (all images in one cluster, loss
  ~ 1e-9): loss and gradients are then rounding noise and no cross-rank comparison means anything.  Deterministic, so
  every rank and the emulation end up with bit-identical parameters."""
  import torch

  from iic_b200.step import _to_net_input
  c = CONFIGS[args.config]
  heads = (net.head_A if args.head == "A" else net.head_B).heads if hasattr(net, "head_B") else net.head.heads
  with torch.no_grad():
    f = net(_to_net_input(x, c["sobel"], False), trunk_features=True).float().mean(0)
    for h in heads:
      h[0].weight.mul_(200.0)
      h[0].bias.copy_(-(h[0].weight.float() @ f).to(h[0].bias.dtype))
    for m in net.modules():  # undo the probe forward's running-statistics update
      if getattr(m, "track_running_stats", False) and getattr(m, "running_mean", None) is not None:
        m.running_mean.zero_()
        m.running_var.fill_(1.)


def verify(args, world, rank, dev):
  """N ranks (bucketed overlapped all-reduce, phased joint) against the one-device emulation of the same sharded
  algorithm (per-chunk BatchNorm, summed partial joints): loss and the fp64 checksum of ALL gradients."""
  import torch
  import torch.distributed as dist

  from iic_b200 import distributed as iicd
  c = CONFIGS[args.config]
  if c["kind"] != "cluster":
    return {"parity_ok": None, "why": "verify covers the clustering workloads"}
  B = min(pairs_for(args, world), 48)
  import copy
  args = copy.copy(args)
  args.graph = False  # (a graphed step runs warm-up optimiser steps before its capture: the check compares ONE eager step)
  job = Job(args, args.precision, dev)
  batches = [_verify_batch(args, B, 5000 + r, dev) for r in range(world)]
  _condition_for_verify(job.net, args, batches[0][0])
  loss, _ = job.step(batches[rank])  # includes the Adam step: compare the gradients it consumed
  if job.arena is not None:
    gsum, gsq = job.arena.grad_checksum()
  else:
    gs = [p.grad.double() for p in job.net.parameters() if p.grad is not None]
    gsum, gsq = float(sum(g.sum() for g in gs)), float(sum((g * g).sum() for g in gs))
  got = torch.tensor([float(loss), gsum, gsq], dtype=torch.float64, device=dev)
  allv = [torch.zeros_like(got) for _ in range(world)]
  if world > 1:
    dist.all_gather(allv, got)
  else:
    allv = [got]
  if rank != 0:
    return None
  same = all(torch.allclose(v, allv[0], rtol=1e-9, atol=0) for v in allv)
  # one-device emulation on rank 0 (fresh identical network: same seed)
  was = iicd._group["enabled"]
  iicd._group["enabled"] = False
  try:
    emu = Job(args, args.precision, dev)
    emu.arena = None
    _condition_for_verify(emu.net, args, batches[0][0])
    el = iicd.emulate_sharded_backward(emu.net, [b[0] for b in batches], [b[1] for b in batches], head=args.head, lamb=1.0,
                                       sobel=c["sobel"])
    gs = [p.grad.double() for p in emu.net.parameters() if p.grad is not None]
    esum, esq = float(sum(g.sum() for g in gs)), float(sum((g * g).sum() for g in gs))
  finally:
    iicd._group["enabled"] = was
  rel = lambda a, b: abs(a - b) / max(abs(b), 1e-30)  # noqa: E731
  tol = 1e-3 if args.precision == "bf16" else 1e-4
  out = {"ranks_agree": bool(same), "pairs_per_rank": B, "loss": float(allv[0][0]), "loss_emulated": float(el),
         "grad_sq_rel_err": rel(float(allv[0][2]), esq), "grad_sum_abs_err": abs(float(allv[0][1]) - esum),
         "grad_norm": esq ** 0.5, "tolerance": tol}
  out["parity_ok"] = bool(same and rel(out["loss"], out["loss_emulated"]) < tol and out["grad_sq_rel_err"] < 10 * tol)
  return out


def run_ours(args):
  import torch
  import torch.distributed as dist

  from iic_b200 import distributed as iicd
  from iic_b200 import kernels

  world = int(os.environ.get("WORLD_SIZE", "1"))
  rank = int(os.environ.get("RANK", "0"))
  local = int(os.environ.get("LOCAL_RANK", "0"))
  assert torch.cuda.is_available(), "bench.py needs a GPU (there is no CPU fallback)"
  torch.cuda.set_device(local)
  dev = torch.device("cuda", local)
  if world > 1:
    dist.init_process_group("nccl", device_id=dev)
    iicd.enable()
  assert world == args.gpus, "--gpus %d but WORLD_SIZE=%d (launch with torch.distributed.run)" % (args.gpus, world)
  c = CONFIGS[args.config]
  B = pairs_for(args, world)

  host = make_host_batch(args, B, 1000 + rank)
  resident = [h.to(dev) for h in host]
  job = Job(args, args.precision, dev)
  m = measure(job, resident, host, args.steps, args.warmup, world, dev, ClockSampler(local) if rank == 0 else None,
              args.dump_outputs if rank == 0 else None)
  value = B * world * args.steps / m["sec"]
  e2e = B * world * args.steps / m["sec_e2e"]

  roof = None
  if not args.no_roofline and not args.graph:  # (per-launch events do not exist inside a graph replay)
    roof = roofline(job, resident, m["sec"] / args.steps, B, c["flop"], args.precision)

  modes = {}
  if world == 1 and args.also:
    for mode in [x for x in args.also.split(",") if x and x != args.precision]:
      del job
      torch.cuda.empty_cache()
      job = Job(args, mode, dev)
      ks, kw = (3, 3) if mode != "fp32" else (1, 1)
      mm = measure(job, resident, host, ks, kw, world, dev)
      entry = {"value": B * ks / mm["sec"], "unit": "img-pairs/s", "ms_per_step": mm["sec"] / ks * 1e3, "steps": ks,
               "warmup": kw, "e2e": B * ks / mm["sec_e2e"], "loss": mm["loss"], "gpu_launches": mm["launches"]}
      if not args.no_roofline:
        r = roofline(job, resident, mm["sec"] / ks, B, c["flop"], mode)
        entry["roofline"] = {k: r[k] for k in ("achieved", "peak", "frac", "unit", "peak_source", "kernel", "by_kind",
                                               "conv_share_of_step", "whole_step_frac")}
      modes[mode] = entry

  ver = None
  if args.verify or (world > 1 and not args.no_verify):
    try:
      ver = verify(args, world, rank, dev)
    except Exception as e:  # the check is a collective: every rank raises together or none does
      if args.verify:
        raise
      ver = {"parity_ok": None, "why": "verify failed to run: %r" % (e,)}

  overlap = None
  if world > 1 and job.arena is not None and not args.graph:
    job.arena.profile = True
    job.step(resident)
    torch.cuda.synchronize()
    overlap = job.arena.timeline()
    job.arena.profile = False

  cpu = None
  if rank == 0 and not args.no_cpu_baseline and world == 1:
    cpu, _ = time_cpu_reference(args, args.cpu_pairs or c["cpu_pairs"], 3, 1)

  if rank == 0:
    from iic_b200.archs import _engine
    variants = {k: kernels.get_option(k) for k in ("conv_halo", "conv_halo_wgrad", "conv_halo_store", "stem_quad",
                                                   "dgrad_prefetch", "tc2_mt2", "conv_halo_stats", "bn_bwd_ctas",
                                                   "tf32x3_raw_hi", "wgrad_mt", "halo_addend_tma", "dgrad_s2_mt")}
    variants.update({k: int(v) for k, v in _engine.OPTIONS.items()})
    variants.update({"stem_wgrad_tc": int(kernels.STEM_WGRAD_TC["on"]), "wgrad_fused_unpack": int(kernels.WGRAD_FUSED_UNPACK["on"]),
                     "seg_joint_tc": int(kernels.SEG_JOINT_TC["on"]), "seg_corr_tc": int(kernels.SEG_CORR_TC["on"])})
    h2d = sum(t.numel() * t.element_size() for t in host) * world
    line = {"metric": METRIC, "value": value, "unit": "img-pairs/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": m["sec"] / args.steps * 1e3, "higher_is_better": True,
            "scaling": c["scaling"] if not args.pairs_per_gpu else "weak",
            "vs_baseline": None, "dtype": {"bf16": "bf16", "tf32": "tf32", "tf32x3": "tf32x3 (fp32-grade)", "fp32": "f32"}[args.precision],
            "data": "synthetic", "config": workload_config(args, B, world), "clocks": m["clocks"],
            "e2e": {"value": e2e, "unit": "img-pairs/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 8 * world,
                    "ms_per_step": m["sec_e2e"] / args.steps * 1e3},
            "gpu_launches": m["launches"], "loss": m["loss"], "wall_s": m["wall"], "kernel_variants": variants}
    if roof is not None:
      line["roofline"] = roof
    if modes:
      line["precision_modes"] = modes
    if overlap is not None:
      line["allreduce_timeline"] = overlap
    if ver is not None:
      line["verify"] = ver
      line["parity_ok"] = ver.get("parity_ok")
    if cpu is not None:
      line["cpu_baseline"] = cpu
    print(json.dumps(line))
  if world > 1:
    # captured graphs hold NCCL work: destroy them (and everything else that references the communicator's streams) before
    # the process group, or the teardown hangs (seen at N = 2 with --graph)
    job.gstep = None
    del job
    torch.cuda.synchronize()
    dist.barrier()
    dist.destroy_process_group()


def main():
  # keep stdout to the single JSON line: NCCL prints its version banner there at NCCL_DEBUG=VERSION
  if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
    os.environ["NCCL_DEBUG"] = "WARN"
  args = parse()
  if args.impl == "reference":
    run_reference(args)
  else:
    run_ours(args)


if __name__ == "__main__":
  main()
