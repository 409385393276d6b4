"""Timing of the semi-supervised finetune step at the paper's configuration (IID_semisup_STL10.py with
--penultimate_features, examples/commands.txt:52): ClusterNet5g at input 64, 2 sobel channels computed from uint8 RGB on the
device, batch 700, layer3 features (dlen 20736), gt_k 10, bf16, two FusedAdam.

Prints one JSON line: median step time over >= 30 event-timed steps after warm-up and img/s; the head alone (both Linears,
BatchNorm1d, cross-entropy, forward + backward) timed the same way on fixed trunk features; the head's GEMM FLOP and
achieved TFLOP/s; the device name and power limit read in the same run; the kernel names of the head GEMMs from a
separate torch.profiler pass.

    python tools/semisup_bench.py [--steps 30] [--warmup 5] [--batch 700] [--precision bf16]
"""
import argparse
import json
import os
import subprocess
import sys
from argparse import Namespace

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def _power():
  try:
    return subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                          capture_output=True, text=True, timeout=60).stdout.strip()
  except Exception as e:  # noqa: BLE001
    return "unavailable (%s)" % e


def _median(xs):
  xs = sorted(xs)
  return xs[len(xs) // 2]


def _timed(fn, steps, warmup):
  for _ in range(warmup):
    fn()
  torch.cuda.synchronize()
  ms = []
  for _ in range(steps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    e1.synchronize()
    ms.append(e0.elapsed_time(e1))
  return ms


def main():
  ap = argparse.ArgumentParser()
  ap.add_argument("--steps", type=int, default=30)
  ap.add_argument("--warmup", type=int, default=5)
  ap.add_argument("--batch", type=int, default=700)
  ap.add_argument("--precision", default="bf16")
  a = ap.parse_args()
  assert torch.cuda.is_available(), "semisup_bench measures on the GPU; there is no CPU timing"
  import iic_b200.archs as archs
  from iic_b200.optim import FusedAdam
  from iic_b200.step import iic_semisup_step
  from iic_b200.utils.semisup.general import CrossEntropyLoss
  from oracle import weights

  n, sz, dlen, gt_k, hidden = a.batch, 64, 20736, 10, 2048
  cfg = dict(in_channels=2, input_sz=sz, num_sub_heads=5, output_k=70, batchnorm_track=True, precision=a.precision)
  net = archs.SupHead5(archs.ClusterNet5g(Namespace(**cfg)), dlen=dlen, gt_k=gt_k)
  weights.fill_state_dict(net)
  net.cuda().train()
  opts = (FusedAdam(net.trunk.parameters(), lr=1e-4), FusedAdam(net.head.parameters(), lr=1e-3))
  g = torch.Generator().manual_seed(0)
  imgs = torch.randint(0, 256, (n, 3, sz, sz), generator=g, dtype=torch.uint8).cuda()
  targets = torch.randint(0, gt_k, (n,), generator=g).cuda()

  step_ms = _timed(lambda: iic_semisup_step(net, opts, imgs, targets, penultimate_features=True), a.steps, a.warmup)

  feat = torch.randn(n, dlen, generator=g).cuda().requires_grad_(True)
  crit = CrossEntropyLoss()

  def head_only():
    crit(net.forward_head(feat), targets).backward()
  head_ms = _timed(head_only, a.steps, a.warmup)

  # GEMM FLOP of the head per step: first Linear fprop + dgrad + wgrad, last Linear fprop + dgrad + wgrad
  flop = 3 * 2.0 * n * dlen * hidden + 3 * 2.0 * n * hidden * gt_k
  from torch.profiler import ProfilerActivity, profile
  with profile(activities=[ProfilerActivity.CUDA]) as prof:
    head_only()
    torch.cuda.synchronize()
  kernels = sorted({e.key for e in prof.key_averages() if "conv_tc2" in e.key or "conv_tf32" in e.key or "simt_gemm" in e.key
                    or "wgrad" in e.key})
  step, head = _median(step_ms), _median(head_ms)
  print(json.dumps({
    "workload": "semisup SupHead5(ClusterNet5g) input 64, 2 sobel channels from uint8 RGB, batch %d, penultimate features "
                "(dlen %d), gt_k %d, %s" % (n, dlen, gt_k, a.precision),
    "device": torch.cuda.get_device_name(0), "power_limit_and_max_sm_clock": _power(),
    "steps": a.steps, "warmup": a.warmup,
    "step_ms_median": round(step, 3), "step_ms_min": round(min(step_ms), 3), "img_per_s": round(n / step * 1e3, 1),
    "head_ms_median": round(head, 3), "head_share_of_step": round(head / step, 4),
    "head_gemm_gflop": round(flop / 1e9, 2), "head_tflops_achieved": round(flop / (head * 1e-3) / 1e12, 1),
    "head_gemm_kernels": kernels}))


if __name__ == "__main__":
  main()
