"""Import shim that loads the UNMODIFIED reference modules (xu-ji/IIC, Python-2.7 /
torch-0.4.1 code; a checkout named by $IIC_REFERENCE) under Python 3 / torch 2.x.
Used only by tests/golden/make_golden.py, which records what the reference
computes as the golden fixtures the tests compare against.  Recipe: SURVEY.md
Appendix A.
"""
import builtins
import importlib
import os
import sys
import types

REF = os.environ.get("IIC_REFERENCE", "/root/reference")


def available():
  return os.path.isdir(os.path.join(REF, "code", "utils", "cluster"))


def _stub_matplotlib():
  if "matplotlib" in sys.modules:
    return
  m = types.ModuleType("matplotlib")
  m.use = lambda *a, **k: None
  mp = types.ModuleType("matplotlib.pyplot")
  m.pyplot = mp
  sys.modules["matplotlib"] = m
  sys.modules["matplotlib.pyplot"] = mp


def _pkg(name, path):
  mod = types.ModuleType(name)
  mod.__path__ = [path]
  sys.modules[name] = mod
  return mod


_loaded = {}


def load():
  """Returns a namespace with the reference's hot-path callables."""
  if _loaded:
    return types.SimpleNamespace(**_loaded)
  assert available(), "reference tree not present"
  builtins.xrange = range
  _stub_matplotlib()
  code = os.path.join(REF, "code")
  # the reference package is literally called `code` (would shadow the stdlib
  # module pdb/pytest use); its hot-path modules only use relative imports, so
  # the tree is mounted under the alias package `iicref` instead.
  for name, path in [("iicref", code), ("iicref.utils", code + "/utils"),
                     ("iicref.utils.cluster", code + "/utils/cluster"),
                     ("iicref.utils.segmentation", code + "/utils/segmentation"),
                     ("iicref.archs", code + "/archs"),
                     ("iicref.archs.cluster", code + "/archs/cluster"),
                     ("iicref.archs.segmentation", code + "/archs/segmentation")]:
    _pkg(name, path)
  sys.path.insert(0, code + "/archs/cluster")  # py2 implicit-relative imports
  cl = importlib.import_module("iicref.utils.cluster.IID_losses")
  sg = importlib.import_module("iicref.utils.segmentation.IID_losses")
  tf = importlib.import_module("iicref.utils.segmentation.transforms")
  n5 = importlib.import_module("net5g")
  n5t = importlib.import_module("net5g_two_head")
  n6 = importlib.import_module("net6c")
  n6t = importlib.import_module("net6c_two_head")
  n10 = importlib.import_module("iicref.archs.segmentation.net10a")
  sys.modules["net10a"] = n10
  n10t = importlib.import_module("iicref.archs.segmentation.net10a_twohead")
  _loaded.update(IID_loss=cl.IID_loss, compute_joint=cl.compute_joint,
                 IID_segmentation_loss=sg.IID_segmentation_loss,
                 IID_segmentation_loss_uncollapsed=sg.IID_segmentation_loss_uncollapsed,
                 perform_affine_tf=tf.perform_affine_tf,
                 random_translation_multiple=tf.random_translation_multiple,
                 ClusterNet5g=n5.ClusterNet5g, ClusterNet5gTwoHead=n5t.ClusterNet5gTwoHead,
                 ClusterNet6c=n6.ClusterNet6c, ClusterNet6cTwoHead=n6t.ClusterNet6cTwoHead,
                 SegmentationNet10a=n10.SegmentationNet10a,
                 SegmentationNet10aTwoHead=n10t.SegmentationNet10aTwoHead)
  return types.SimpleNamespace(**_loaded)
