"""In-tree build of libspx.so (hand-written CUDA for sm_100a behind the C-ABI in include/spx.h).

    python -m sycl_points_b200.build [--force]

nvcc cross-compiles without a GPU; the .so lands next to this file so that it travels to the GPU
box with the repo snapshot (it is git-ignored, not gpurun-ignored)."""
from __future__ import annotations

import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT = os.path.join(HERE, "libspx.so")
SOURCES = ["spx_runtime.cu", "spx_knn.cu", "spx_features.cu", "spx_voxel.cu", "spx_registration.cu", "spx_batch.cu", "spx_voxelmap.cu", "spx_outlier.cu", "spx_cluster.cu", "spx_plane.cu", "spx_fpfh.cu", "spx_ransac.cu"]
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
FLAGS = ["-O3", "-std=c++17", "-lineinfo", "--fmad=true", "-Xcompiler", "-fPIC,-O2,-fvisibility=hidden",
         "-Xptxas", "-v", "--expt-relaxed-constexpr"]


def _nvcc() -> str:
    for c in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if c and (os.path.isabs(c) and os.path.exists(c) or not os.path.isabs(c)):
            return c
    return "nvcc"


def _deps():
    out = [os.path.join(HERE, "..", "include", "spx.h"), os.path.abspath(__file__)]
    for f in os.listdir(CSRC):
        if f.endswith((".cu", ".cuh")):
            out.append(os.path.join(CSRC, f))
    return out


def is_stale() -> bool:
    if not os.path.exists(OUT):
        return True
    t = os.path.getmtime(OUT)
    return any(os.path.getmtime(d) > t for d in _deps())


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not is_stale():
        return OUT
    objs = []
    env = dict(os.environ)
    env.pop("CXX", None)
    env.pop("CC", None)
    host = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
    os.makedirs(os.path.join(HERE, "build"), exist_ok=True)
    log = []
    procs = []
    for src in SOURCES:
        obj = os.path.join(HERE, "build", src.replace(".cu", ".o"))
        cmd = [_nvcc(), "-ccbin", host, *ARCH, *FLAGS, "-c", os.path.join(CSRC, src), "-o", obj]
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, env=env)))
        objs.append(obj)
    for src, p in procs:
        out, _ = p.communicate()
        log.append(f"==== {src}\n{out}")
        if p.returncode != 0:
            sys.stderr.write("\n".join(log))
            raise RuntimeError(f"nvcc failed on {src}")
    cmd = [_nvcc(), "-ccbin", host, *ARCH, "-shared", "-o", OUT, *objs, "-Xlinker", "--exclude-libs,ALL", "-lpthread"]
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, env=env)
    log.append(r.stdout)
    if r.returncode != 0:
        sys.stderr.write("\n".join(log))
        raise RuntimeError("link failed")
    with open(os.path.join(HERE, "build", "ptxas.log"), "w") as f:
        f.write("\n".join(log))
    if verbose:
        print("\n".join(log))
    return OUT


if __name__ == "__main__":
    build(force="--force" in sys.argv, verbose=True)
    print("built", OUT)
