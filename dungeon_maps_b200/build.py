"""Builds the C-ABI CUDA library in-tree: dungeon_maps_b200/libdungeon_maps_b200.so.

nvcc cross-compiles for sm_100a without a GPU.  --fmad=false keeps nvcc from
contracting a*b+c (the reference's float32 op order is part of the contract;
the kernels use explicit __f*_rn intrinsics on top of that).  -lineinfo so ncu's
source page maps back to the .cu files.  cudart is linked statically so the
library has no dependency on torch or on a system libcudart.
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
# $DM_B200_LIB points the binding at another build of the same ABI (kernel experiments, scripts/exp_build.sh)
LIB = os.environ.get("DM_B200_LIB") or os.path.join(HERE, "libdungeon_maps_b200.so")
SOURCES = ["dm_api.cu", "dm_project.cu", "dm_labels.cu", "dm_flow.cu", "dm_fuse.cu", "dm_points.cu", "dm_builder.cu", "dm_params.cu", "dm_ordered.cu",
           "dm_geodesic.cu", "dm_components.cu", "dm_distance.cu", "dm_match.cu"]
NVCC_FLAGS = [
  "-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "--fmad=false",
  "-Xcompiler", "-fPIC", "-Xcompiler", "-ffp-contract=off", "-shared", "-cudart", "static",
]


def _nvcc() -> str:
  for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
    if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
      return cand
  return "nvcc"


def needs_build() -> bool:
  if not os.path.exists(LIB):
    return True
  t = os.path.getmtime(LIB)
  deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)]
  deps.append(os.path.join(HERE, "..", "include", "dungeon_maps_b200.h"))
  return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
  if not force and not needs_build():
    return LIB
  cmd = [_nvcc()] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else [])
  cmd += ["-o", LIB] + [os.path.join(CSRC, s) for s in SOURCES]
  subprocess.run(cmd, check=True)
  return LIB


if __name__ == "__main__":
  print(build(force=True, verbose="-v" in sys.argv))
