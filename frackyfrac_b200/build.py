"""Builds the native libraries in-tree (sm_100a only).

  frackyfrac_b200/_build/libfrcfrc_cuda.so   CUDA engine + C ABI (include/frcfrc_cuda.h)
  frackyfrac_b200/_build/libfrcfrc_host.so   C++ host side (Newick / table readers, Go %v writer)
  frackyfrac_b200/_build/frcfrc              C++ stand-in for the Go CLI (same flags and output)
  frackyfrac_b200/_build/sprspr              C++ stand-in for the dense -> sparse converter (sprspr/sprspr.go)

nvcc cross-compiles without a GPU, so this runs on the CPU-only build box; the
.so files travel to the GPU box with the repo snapshot.
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
OUT = os.path.join(HERE, "_build")
CSRC = os.path.join(HERE, "csrc")
HOST = os.path.join(HERE, "host")

CUDA_SOURCES = ["job.cu", "plan.cpp", "embed.cu", "exact.cu", "weighted.cu", "unweighted_tc.cu", "comm.cu", "wire.cu"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC", "--expt-relaxed-constexpr", "-Xptxas", "-v",
]


def _nvcc() -> str:
    for cand in (shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: libfrcfrc_cuda cannot be built (there is no CPU fallback)")


def _stale(target: str, sources: list[str]) -> bool:
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(s) > t for s in sources)


def build_cuda(force: bool = False, verbose: bool = False) -> str:
    os.makedirs(OUT, exist_ok=True)
    lib = os.path.join(OUT, "libfrcfrc_cuda.so")
    headers = [os.path.join(CSRC, h) for h in ("frc_internal.h", "ptx.cuh", "host_pool.h", "plan.h", "wire.cuh")]
    headers.append(os.path.join(ROOT, "include", "frcfrc_cuda.h"))
    objs = []
    for src in CUDA_SOURCES:
        s = os.path.join(CSRC, src)
        o = os.path.join(OUT, os.path.splitext(src)[0] + ".o")
        objs.append(o)
        if force or _stale(o, [s] + headers):
            cmd = [_nvcc(), *NVCC_FLAGS, *os.environ.get("FRC_BUILD_DEFS", "").split(), "-c", s, "-o", o]
            r = subprocess.run(cmd, capture_output=True, text=True)
            log = os.path.join(OUT, src + ".ptxas.log")
            with open(log, "w") as f:
                f.write(r.stdout + r.stderr)
            if verbose or r.returncode:
                sys.stderr.write(r.stdout + r.stderr)
            if r.returncode:
                raise RuntimeError(f"nvcc failed on {src}")
    if force or _stale(lib, objs):
        cmd = [_nvcc(), "-shared", "-o", lib, *objs, "-cudart", "shared", "-ldl"]
        subprocess.run(cmd, check=True)
    return lib


def build_host(force: bool = False) -> tuple[str, str]:
    os.makedirs(OUT, exist_ok=True)
    lib = os.path.join(OUT, "libfrcfrc_host.so")
    exe = os.path.join(OUT, "frcfrc")
    srcs = [os.path.join(HOST, f) for f in os.listdir(HOST) if f.endswith((".cpp", ".hpp"))]
    cxx = shutil.which("g++") or "g++"
    common = [cxx, "-O2", "-g", "-std=c++17", "-fPIC", "-Wall", "-Wextra", "-pthread",
              "-I", os.path.join(ROOT, "include")]
    if force or _stale(lib, srcs):
        subprocess.run([*common, "-shared", "-o", lib, os.path.join(HOST, "hostlib.cpp"),
                        os.path.join(HOST, "fileio.cpp"), "-lz", "-ldl"], check=True)
    cuda_lib = os.path.join(OUT, "libfrcfrc_cuda.so")
    if force or _stale(exe, srcs + ([cuda_lib] if os.path.exists(cuda_lib) else [])):
        subprocess.run([*common, "-o", exe, os.path.join(HOST, "frcfrc_main.cpp"),
                        os.path.join(HOST, "hostlib.cpp"), os.path.join(HOST, "fileio.cpp"),
                        "-L", OUT, "-lfrcfrc_cuda", "-lz", "-ldl",
                        "-Wl,-rpath,$ORIGIN"], check=True)
    sprspr = os.path.join(OUT, "sprspr")
    if force or _stale(sprspr, srcs):
        subprocess.run([*common, "-o", sprspr, os.path.join(HOST, "sprspr_main.cpp"),
                        os.path.join(HOST, "hostlib.cpp"), os.path.join(HOST, "fileio.cpp"), "-lz", "-ldl"], check=True)
    return lib, exe


def build_all(force: bool = False, verbose: bool = False) -> None:
    build_cuda(force, verbose)
    build_host(force)


if __name__ == "__main__":
    build_all(force="--force" in sys.argv, verbose="-v" in sys.argv)
    print("built", os.listdir(OUT))
