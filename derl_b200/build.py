"""In-tree nvcc build of libderl_b200.so (the C-ABI library, sm_100a only).

No torch headers are involved: the library links only the CUDA runtime, so it builds in
seconds and the resulting .so travels to the GPU box with the repo snapshot.
"""
import hashlib
import os
import shutil
import subprocess
import sys

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
REPO_DIR = os.path.dirname(PKG_DIR)
CSRC = os.path.join(PKG_DIR, "csrc")
INCLUDE = os.path.join(REPO_DIR, "include")
LIB_PATH = os.path.join(PKG_DIR, "libderl_b200.so")
STAMP_PATH = os.path.join(PKG_DIR, ".libderl_b200.stamp")
SOURCES = ("abi.cu", "gae.cu", "gather.cu", "frame_stacks.cu", "frame_pack.cu", "ppo_loss.cu", "frames.cu", "relu_bwd.cu", "stem_tc.cu", "stem_bwd_tc.cu", "mlp_update.cu", "heads.cu",
           "host_api.cu")
NVCC_FLAGS = (
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-std=c++17", "-lineinfo",
    "--fmad=false",  # float32 parity with torch's separately-rounded ops; fp64 uses *_rn anyway
    "-Xcompiler", "-fPIC", "-shared", "-cudart", "static",
)


def find_nvcc():
  nvcc = os.environ.get("NVCC") or shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
  if not os.path.exists(nvcc):
    raise RuntimeError("nvcc not found (set $NVCC); derl_b200 has no prebuilt or CPU fallback")
  return nvcc


def source_digest():
  h = hashlib.sha256()
  names = [os.path.join(CSRC, n) for n in sorted(os.listdir(CSRC))]
  names += [os.path.join(INCLUDE, n) for n in sorted(os.listdir(INCLUDE))]
  for path in names:
    h.update(path.encode())
    with open(path, "rb") as f:
      h.update(f.read())
  h.update(" ".join(NVCC_FLAGS).encode())
  return h.hexdigest()


def is_fresh():
  if not (os.path.exists(LIB_PATH) and os.path.exists(STAMP_PATH)):
    return False
  with open(STAMP_PATH) as f:
    return f.read().strip() == source_digest()


def build(force=False, verbose=False):
  """Compile the library if sources changed; returns the path of the .so."""
  if not force and is_fresh():
    return LIB_PATH
  cmd = [find_nvcc(), *NVCC_FLAGS, "-I", INCLUDE, "-I", CSRC]
  if verbose:
    cmd += ["-Xptxas", "-v"]
  cmd += [os.path.join(CSRC, s) for s in SOURCES]
  cmd += ["-o", LIB_PATH]
  proc = subprocess.run(cmd, capture_output=True, text=True)
  if verbose or proc.returncode != 0:
    sys.stderr.write(proc.stdout + proc.stderr)
  if proc.returncode != 0:
    raise RuntimeError("nvcc failed building libderl_b200.so:\n" + proc.stderr[-4000:])
  with open(STAMP_PATH, "w") as f:
    f.write(source_digest())
  return LIB_PATH


if __name__ == "__main__":
  print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
