"""Builds libhge_b200.so (the C-ABI library of include/hge_b200.h) in-tree with nvcc for
sm_100a.  nvcc cross-compiles without a GPU, so this runs in the dev container too.

    python -m hypergraphembedding_b200.build [--force] [--verbose]
"""
import argparse
import glob
import os
import shutil
import subprocess
import sys

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(PKG_DIR, "csrc")
LIB_NAME = "libhge_b200.so"
LIB_PATH = os.path.join(PKG_DIR, LIB_NAME)

# host-only sources (.cpp) go through g++ directly: they use x86 intrinsics with per-function
# target attributes, which nvcc's front end does not take
CXX_FLAGS = ["-O3", "-std=c++17", "-fPIC", "-Wall", "-Wno-unused-function", "-Wno-psabi", "-pthread"]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC,-O3,-Wall,-Wno-unused-function", "-Xptxas", "-v",
]


def find_nvcc():
  for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
    if cand and os.path.exists(cand):
      return cand
  raise RuntimeError("nvcc not found; libhge_b200.so cannot be built")


def sources():
  return sorted(glob.glob(os.path.join(CSRC, "*.cu")) + glob.glob(os.path.join(CSRC, "*.cpp")))


def needs_build():
  if not os.path.exists(LIB_PATH):
    return True
  built = os.path.getmtime(LIB_PATH)
  deps = sources() + glob.glob(os.path.join(CSRC, "*.cuh")) + glob.glob(
      os.path.join(PKG_DIR, "..", "include", "*.h")) + [os.path.abspath(__file__)]
  return any(os.path.getmtime(d) > built for d in deps)


def build(force=False, verbose=False):
  """Compiles every CUDA / C++ source under csrc/ into one shared library."""
  if not force and not needs_build():
    return LIB_PATH
  nvcc = find_nvcc()
  objs = []
  obj_dir = os.path.join(CSRC, "_obj")
  os.makedirs(obj_dir, exist_ok=True)
  procs = []
  for src in sources():
    obj = os.path.join(obj_dir, os.path.basename(src) + ".o")
    objs.append(obj)
    if src.endswith(".cpp"):
      cuda_inc = os.path.join(os.path.dirname(os.path.dirname(nvcc)), "include")
      cmd = [os.environ.get("CXX", "g++")] + CXX_FLAGS + ["-I", cuda_inc, "-c", src, "-o", obj]
    else:
      cmd = [nvcc] + NVCC_FLAGS + ["-x", "cu", "-c", src, "-o", obj]
    procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT,
                                        text=True)))
  log = []
  failed = False
  for src, p in procs:
    text, _ = p.communicate()
    log.append("== %s\n%s" % (os.path.basename(src), text))
    failed |= p.returncode != 0
  with open(os.path.join(obj_dir, "build.log"), "w") as f:
    f.write("\n".join(log))
  if failed or verbose:
    sys.stderr.write("\n".join(log) + "\n")
  if failed:
    raise RuntimeError("nvcc failed; see the log above")
  tmp = LIB_PATH + ".tmp"
  subprocess.check_call([nvcc, "-shared", "-o", tmp] + objs + ["-gencode",
                                                               "arch=compute_100a,code=sm_100a",
                                                               "-Xlinker", "-lpthread"])
  os.replace(tmp, LIB_PATH)
  return LIB_PATH


if __name__ == "__main__":
  ap = argparse.ArgumentParser()
  ap.add_argument("--force", action="store_true")
  ap.add_argument("--verbose", action="store_true")
  args = ap.parse_args()
  print(build(force=args.force, verbose=args.verbose))
