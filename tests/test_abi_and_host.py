"""CPU-only: the C-ABI library loads and exports every symbol include/iic_b200.h declares, the
Python mirror keeps the reference's interface, and the product has no CPU fallback."""
import os
import re
import subprocess
import sys
from argparse import Namespace

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def built():
  from iic_b200 import build
  return build.build()


def test_library_exports_every_declared_symbol(built):
  header = open(os.path.join(ROOT, "include", "iic_b200.h")).read()
  declared = set(re.findall(r"\b(iic_[a-z0-9_]+)\s*\(", header))
  declared -= {"iic_conv_geom"}
  out = subprocess.run(["nm", "-D", "--defined-only", built], capture_output=True, text=True, check=True).stdout
  exported = set(re.findall(r" T (iic_[a-z0-9_]+)", out))
  assert declared, "no declarations parsed"
  assert declared <= exported, sorted(declared - exported)
  from iic_b200 import _lib
  assert set(_lib.declared_symbols()) == declared, sorted(set(_lib.declared_symbols()) ^ declared)
  l = _lib.lib()  # dlopen + prototype binding (no compute: there is no GPU here)
  assert l.iic_abi_version() == 1
  assert l.iic_launch_count(0) == 0


def test_sm100a_tensor_core_and_async_copy_sass(built):
  from iic_b200 import build
  cuobjdump = os.path.join(os.path.dirname(build.NVCC), "cuobjdump")  # the toolkit that built the library
  sass = subprocess.run([cuobjdump, "-sass", built], capture_output=True, text=True, check=True).stdout
  assert "UTCHMMA" in sass, "tcgen05.mma missing from the SASS"
  assert "LDTM" in sass and "UTMALDG" in sass and "UTMASTG" in sass  # TMEM read-out, TMA loads (tiled + im2col) and stores
  assert "UTMALDG.4D.IM2COL" in sass
  assert "sm_100a" in sass or "SM100a" in sass.upper()


def test_state_dict_keys_match_reference_layout():
  import iic_b200.archs as archs
  from oracle import nets as oracle_nets
  for name, cfg in [("ClusterNet5gTwoHead", dict(in_channels=2, input_sz=96, num_sub_heads=5, output_k_A=70,
                                                 output_k_B=10, batchnorm_track=True)),
                    ("ClusterNet5g", dict(in_channels=2, input_sz=64, num_sub_heads=5, output_k=10,
                                          batchnorm_track=False)),
                    ("ClusterNet6cTwoHead", dict(in_channels=1, input_sz=24, num_sub_heads=5, output_k_A=50,
                                                 output_k_B=10, batchnorm_track=False)),
                    ("ClusterNet6c", dict(in_channels=1, input_sz=24, num_sub_heads=5, output_k=10,
                                          batchnorm_track=True))]:
    a = archs.__dict__[name](Namespace(**cfg)).state_dict()
    b = getattr(oracle_nets, name)(Namespace(**cfg)).state_dict()  # key-compatible with the reference (golden-pinned)
    assert list(a.keys()) == list(b.keys())
    assert all(a[k].shape == b[k].shape for k in a)


def test_no_cpu_fallback_and_product_never_imports_oracle():
  from iic_b200.utils.cluster.IID_losses import IID_loss
  from iic_b200.utils.cluster.transforms import sobel_process
  z = torch.softmax(torch.randn(8, 3), 1)
  with pytest.raises(RuntimeError):
    IID_loss(z, z)
  with pytest.raises(RuntimeError):
    sobel_process(torch.zeros(1, 1, 4, 4), False)
  for dirpath, _, files in os.walk(os.path.join(ROOT, "iic_b200")):
    for f in files:
      if f.endswith((".py", ".cu", ".cuh", ".h")):
        src = open(os.path.join(dirpath, f)).read()
        assert not re.search(r"^\s*(from|import)\s+oracle", src, re.M), os.path.join(dirpath, f)


def test_missing_library_fails_loudly(monkeypatch):
  from iic_b200 import _lib
  monkeypatch.setattr(_lib, "_lib", None)
  monkeypatch.setattr(_lib, "LIB_PATH", "/nonexistent/libiic_b200.so")
  with pytest.raises(RuntimeError, match="no CPU or PyTorch fallback"):
    _lib.lib()


def test_default_kernel_variants_are_the_validated_set(built):
  """The defaults that ship are the set measured fastest on a B200 with the whole GPU suite green
  (profiles/r01_bench_v10_variants.md); variants written after the last GPU session must stay off until they have run
  on hardware (DESIGN.md S8)."""
  import os
  import subprocess
  import sys
  code = ("import json, iic_b200.kernels as K, iic_b200.archs._engine as E;"
          "print(json.dumps([{n: K.get_option(n) for n in ('conv_halo','conv_halo_wgrad','conv_halo_store','tc2_mt2',"
          "'dgrad_prefetch','stem_quad','stem_bwd_v2','conv_halo_stats','bn_bwd_ctas','tf32x3_raw_hi','wgrad_mt','halo_addend_tma','dgrad_s2_mt')}, E.OPTIONS]))")
  env = {k: v for k, v in os.environ.items() if not k.startswith("IIC_")}
  out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=env, cwd=ROOT, check=True).stdout
  import json
  lib_opts, host_opts = json.loads(out.strip().splitlines()[-1])
  assert lib_opts == {"conv_halo": 1, "conv_halo_wgrad": 1, "conv_halo_store": 1, "tc2_mt2": 1, "dgrad_prefetch": 1,
                      "stem_quad": 2, "stem_bwd_v2": 0, "conv_halo_stats": 1, "bn_bwd_ctas": 2, "tf32x3_raw_hi": 1, "wgrad_mt": 1, "halo_addend_tma": 1, "dgrad_s2_mt": 0}
  assert host_opts == {"bn_merged": True, "stem_stats": True, "pack_batched": True, "stem_bwd_fused": False, "bn_bitmask": True,
                       "wgrad_stream": False, "masked_addend": True, "stem_bwd_dy": False}


def test_weight_packing_contract_of_the_precision_modes():
  """Host side of the packed-weight contract (include/iic_b200.h: iic_pack_weight): 3xTF32 convolutions take their
  weights pre-split as [raw plane | lo plane]; every other mode packs in the storage dtype; the conv wrappers refuse a
  buffer packed for another mode before any pointer reaches the library."""
  from iic_b200 import kernels as K
  from iic_b200._lib import BF16, F32, TF32, TF32X3
  assert K.weight_dtype(F32, TF32X3) == TF32X3 and K.weight_dtype(F32, TF32) == F32
  assert K.weight_dtype(BF16, BF16) == BF16 and K.weight_dtype(F32, F32) == F32
  w = torch.zeros(128, 64, 3, 3)
  assert K._packed_shape(w, F32, 0) == (128, 3, 3, 64) and K._packed_shape(w, BF16, 1) == (64, 3, 3, 128)
  assert K._packed_shape(w, TF32X3, 0) == (2, 128, 3, 3, 64) and K._packed_shape(w, TF32X3, 1) == (2, 64, 3, 3, 128)
  g = K.conv_geom(1, 8, 8, 64, 128, 3, 3, 1, 1, 1)
  K._check_packed(torch.empty(K._packed_shape(w, TF32X3, 0)), g, TF32X3)
  K._check_packed(torch.empty(K._packed_shape(w, F32, 0)), g, TF32)
  with pytest.raises(AssertionError, match="pack_weight"):
    K._check_packed(torch.empty(K._packed_shape(w, F32, 0)), g, TF32X3)
  with pytest.raises(AssertionError, match="pack_weight"):
    K._check_packed(torch.empty(K._packed_shape(w, TF32X3, 0)), g, BF16)
