"""Builds libpclseg.so (the C-ABI CUDA library) in-tree with nvcc for sm_100a.

    python -m pclsegmentation_b200.build [--force]

nvcc cross-compiles without a GPU.  The .so stays next to this file (git-ignored, but it travels to the
GPU box with the repo snapshot).
"""
import hashlib
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
# PCLS_LIB_SUFFIX=_dbg builds a second library next to the product one (development builds with extra flags)
_SUFFIX = os.environ.get("PCLS_LIB_SUFFIX", "")
LIB = os.path.join(HERE, "libpclseg%s.so" % _SUFFIX)
OBJ_DIR = os.path.join(HERE, "build%s" % _SUFFIX)
# conv_tc.cu holds ~160 kernel instantiations: it is compiled once per part (-DPCLS_TC_PART=k, see the file) in parallel
TC_PARTS = 13
SOURCES = [("conv_tc.cu", k) for k in range(TC_PARTS)] + ["conv_head.cu", "net.cu", "nn_kernels.cu", "pool_conv.cu", "squeeze_upconv.cu",
           "projection.cu", "point_labels.cu", "point_instances.cu", "tta.cu", "calibration.cu", "mc_dropout.cu", "semantic_map.cu", "dataset_stats.cu", "head.cu", "input_stage.cu", "confusion.cu", "validation.cu", "error.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17", "-Xcompiler", "-fPIC",
              "--expt-relaxed-constexpr"]
# development builds, e.g. PCLS_NVCC_FLAGS="-DPCLS_TC_DEBUG=1" (wait-cycle counters)
NVCC_FLAGS += os.environ.get("PCLS_NVCC_FLAGS", "").split()


def _nvcc():
  for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
    if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
      return cand
  return "nvcc"


def _digest():
  h = hashlib.sha256()
  h.update(" ".join(NVCC_FLAGS).encode())
  names = sorted(os.listdir(CSRC)) + ["../../include/pclseg.h"]
  for n in names:
    p = os.path.join(CSRC, n)
    if os.path.isfile(p):
      h.update(n.encode())
      with open(p, "rb") as f:
        h.update(f.read())
  return h.hexdigest()


def build(force=False, verbose=False):
  os.makedirs(OBJ_DIR, exist_ok=True)
  stamp = os.path.join(OBJ_DIR, "digest.txt")
  dig = _digest()
  if not force and os.path.exists(LIB) and os.path.exists(stamp) and open(stamp).read() == dig:
    return LIB
  nvcc = _nvcc()

  def compile_one(src):
    extra = []
    if isinstance(src, tuple):
      src, part = src
      obj = os.path.join(OBJ_DIR, src.replace(".cu", "_p%d.o" % part))
      extra = ["-DPCLS_TC_PART=%d" % part]
    else:
      obj = os.path.join(OBJ_DIR, src.replace(".cu", ".o"))
    cmd = [nvcc] + NVCC_FLAGS + extra + ["-c", os.path.join(CSRC, src), "-o", obj]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
      raise RuntimeError("nvcc failed for %s:\n%s\n%s" % (src, r.stdout, r.stderr))
    if verbose and (r.stdout or r.stderr):
      print(r.stdout, r.stderr)
    return obj

  with ThreadPoolExecutor(max_workers=min(os.cpu_count() or 8, len(SOURCES))) as ex:
    objs = list(ex.map(compile_one, SOURCES))
  cmd = [nvcc, "-shared", "-o", LIB] + objs + ["-gencode", "arch=compute_100a,code=sm_100a", "-lcudart", "-ldl"]
  r = subprocess.run(cmd, capture_output=True, text=True)
  if r.returncode != 0:
    raise RuntimeError("link failed:\n%s\n%s" % (r.stdout, r.stderr))
  with open(stamp, "w") as f:
    f.write(dig)
  return LIB


if __name__ == "__main__":
  print(build(force="--force" in sys.argv, verbose=True))
