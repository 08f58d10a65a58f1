"""Builds libgsplat_b200.so in-tree with nvcc for sm_100a (no torch headers: the library is a
plain C ABI, see include/gsplat_b200.h).

  python -m taichi_gaussian_rasterizer_b200.csrc.build [--force] [--verbose]

geom_kernels.cu carries the bit-exactness contract (include/gs_numeric.h) and is compiled without
FMA contraction on both its device image (-fmad=false) and its host image (-ffp-contract=off).
"""
import argparse
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path

CSRC = Path(__file__).resolve().parent
PKG = CSRC.parent
ROOT = PKG.parent
OUT = PKG / "libgsplat_b200.so"
OBJ = ROOT / "build" / "obj"

SOURCES = ["api.cu", "geom_kernels.cu", "point_kernels.cu", "scan_sort.cu", "raster_api.cu",
           "raster_generic.cu", "raster_fast_fwd.cu", "raster_fast_bwd.cu", "raster_fast_bwd_wide.cu",
           "optim_kernels.cu", "morton.cu", "multimem_reduce.cu"]
HEADERS = ["common.cuh", "geom_math.cuh", "lookback.cuh", "raster.cuh", "raster_math.cuh", "raster_fast.cuh",
           "../../include/gsplat_b200.h", "../../include/gs_numeric.h"]

ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
COMMON = ["-O3", "-std=c++17", "-lineinfo", "-Xcompiler", "-fPIC", "--expt-relaxed-constexpr"]
PER_FILE = {
  "geom_kernels.cu": ["-fmad=false", "-Xcompiler", "-ffp-contract=off"],
  # gradients and SH colours carry tolerances (1e-4 / 1e-5 relative L2), not bit-exactness: MUFU based division,
  # sqrt and exp instead of the IEEE sequences (projection backward: 1720 -> 1128 SASS instructions)
  "point_kernels.cu": ["--use_fast_math"],
}


def nvcc() -> str:
  cand = os.environ.get("NVCC") or "/usr/local/cuda/bin/nvcc"
  return cand if Path(cand).exists() else "nvcc"


def host_compiler_args():
  # the image exports CXX=/opt/gcc/bin/g++ (a wrapper without libgomp specs); the system g++ is fine
  ccbin = os.environ.get("GS_CCBIN", "/usr/bin/g++")
  return ["-ccbin", ccbin] if Path(ccbin).exists() else []


def _newest_input() -> float:
  files = [CSRC / s for s in SOURCES] + [CSRC / h for h in HEADERS] + [Path(__file__)]
  return max(f.stat().st_mtime for f in files)


def _compile(src: str, verbose: bool, ptxas_info: bool) -> Path:
  obj = OBJ / (src.replace(".cu", ".o"))
  cmd = [nvcc(), *host_compiler_args(), *ARCH, *COMMON, *PER_FILE.get(src, []), "-c", str(CSRC / src), "-o", str(obj)]
  if ptxas_info:
    cmd += ["-Xptxas", "-v"]
  r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
  if r.returncode != 0:
    raise RuntimeError(f"nvcc failed for {src}:\n{' '.join(cmd)}\n{r.stdout}")
  if verbose or ptxas_info:
    print(f"[build] {src}\n{r.stdout}")
  return obj


def build(force: bool = False, verbose: bool = False, ptxas_info: bool = False, precise_point_kernels: bool = False) -> Path:
  """``precise_point_kernels``: a second library, libgsplat_b200_precise.so, whose point_kernels.cu is compiled WITHOUT
  --use_fast_math — only for benchmarks/fast_math_cost.py, which measures what the flag costs in gradient accuracy and
  buys in time (the product library is always the default build)."""
  out = PKG / "libgsplat_b200_precise.so" if precise_point_kernels else OUT
  if not force and out.exists() and out.stat().st_mtime >= _newest_input():
    return out
  OBJ.mkdir(parents=True, exist_ok=True)
  if precise_point_kernels:   # every other object is shared with the default build
    build(force, verbose, ptxas_info)
    obj = OBJ / "point_kernels_precise.o"
    cmd = [nvcc(), *host_compiler_args(), *ARCH, *COMMON, "-c", str(CSRC / "point_kernels.cu"), "-o", str(obj)]
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode != 0:
      raise RuntimeError(f"nvcc failed for point_kernels.cu (precise):\n{r.stdout}")
    objs = [obj if s == "point_kernels.cu" else OBJ / s.replace(".cu", ".o") for s in SOURCES]
  else:
    with ThreadPoolExecutor(max_workers=min(8, len(SOURCES))) as pool:
      objs = list(pool.map(lambda s: _compile(s, verbose, ptxas_info), SOURCES))
  cmd = [nvcc(), *host_compiler_args(), *ARCH, "-shared", "-o", str(out), *[str(o) for o in objs]]
  r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
  if r.returncode != 0:
    raise RuntimeError(f"link failed:\n{' '.join(cmd)}\n{r.stdout}")
  return out


if __name__ == "__main__":
  ap = argparse.ArgumentParser()
  ap.add_argument("--force", action="store_true")
  ap.add_argument("--verbose", action="store_true")
  ap.add_argument("--ptxas-info", action="store_true")
  ap.add_argument("--precise-point-kernels", action="store_true")
  args = ap.parse_args()
  print(build(args.force, args.verbose, args.ptxas_info, args.precise_point_kernels))
