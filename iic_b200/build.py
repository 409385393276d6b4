"""Builds iic_b200/lib/libiic_b200.so (the C-ABI library) with nvcc for sm_100a.

nvcc cross-compiles without a GPU.  Objects are cached under build/ keyed by source mtime.  Every output is written
under a temporary name and renamed into place, so processes building at the same time (e.g. test workers) never
read a half-written object or library.
"""
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(HERE, "csrc")
LIBDIR = os.path.join(HERE, "lib")
OBJDIR = os.path.join(ROOT, "build", "obj")
LIB = os.path.join(LIBDIR, "libiic_b200.so")

NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17", "-Xcompiler", "-fPIC",
         "-Xptxas", "-v", "--expt-relaxed-constexpr"]


def sources():
  return sorted(f for f in os.listdir(CSRC) if f.endswith(".cu"))


def _newer(a, b):
  return (not os.path.exists(b)) or os.path.getmtime(a) > os.path.getmtime(b)


def _compile(src):
  s = os.path.join(CSRC, src)
  o = os.path.join(OBJDIR, src[:-3] + ".o")
  deps = [s, os.path.join(ROOT, "include", "iic_b200.h")] + [os.path.join(CSRC, h) for h in os.listdir(CSRC) if h.endswith(".cuh")]
  if not any(_newer(d, o) for d in deps):
    return o, ""
  tmp = "%s.%d.tmp" % (o, os.getpid())
  r = subprocess.run([NVCC] + FLAGS + ["-c", s, "-o", tmp], capture_output=True, text=True)
  if r.returncode != 0:
    raise RuntimeError("nvcc failed for %s:\n%s\n%s" % (src, r.stdout, r.stderr))
  os.replace(tmp, o)
  return o, r.stderr


def build(verbose=False):
  os.makedirs(LIBDIR, exist_ok=True)
  os.makedirs(OBJDIR, exist_ok=True)
  with ThreadPoolExecutor(max_workers=8) as ex:
    res = list(ex.map(_compile, sources()))
  objs = [o for o, _ in res]
  if verbose:
    for _, log in res:
      if log:
        print(log)
  if any(_newer(o, LIB) for o in objs):
    tmp = "%s-%d.so" % (LIB[:-3], os.getpid())
    r = subprocess.run([NVCC, "-shared", "-o", tmp] + objs + ["-lcudart"], capture_output=True, text=True)
    if r.returncode != 0:
      raise RuntimeError("link failed:\n%s\n%s" % (r.stdout, r.stderr))
    os.replace(tmp, LIB)
  return LIB


if __name__ == "__main__":
  print(build(verbose="-v" in sys.argv))
