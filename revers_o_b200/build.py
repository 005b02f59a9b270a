"""Build the CUDA library in-tree:  python -m revers_o_b200.build

nvcc cross-compiles sm_100a without a GPU.  Output: revers_o_b200/lib/librevers_o_b200.so (git-ignored,
travels to the GPU box with the gpurun snapshot).  The library links the static CUDA runtime and needs
nothing from torch.
"""
from __future__ import annotations

import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT = os.path.join(HERE, "lib", "librevers_o_b200.so")
SOURCES = ["api.cu", "scan_tc.cu", "scan_tc2.cu", "select.cu", "prep_scan_small.cu", "mask_pool.cu", "mask_pool_tc.cu", "selfjoin.cu", "knn.cu", "kmeans.cu"]
NVCC = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC", "--expt-relaxed-constexpr",
    "-cudart", "static",
]


def _stale() -> bool:
    if not os.path.exists(OUT):
        return True
    t = os.path.getmtime(OUT)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(HERE, "..", "include", "revers_o_b200.h")]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not _stale():
        return OUT
    os.makedirs(os.path.dirname(OUT), exist_ok=True)
    objs = []
    procs = []
    for src in SOURCES:
        obj = os.path.join(HERE, "lib", src.replace(".cu", ".o"))
        cmd = [NVCC, *FLAGS, "-c", os.path.join(CSRC, src), "-o", obj]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(obj)
    failed = False
    for src, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0 or verbose:
            print(f"--- {src} ---\n{out}", file=sys.stderr)
        failed |= p.returncode != 0
    if failed:
        raise RuntimeError("nvcc failed")
    link = [NVCC, "-shared", "-cudart", "static", "-gencode", "arch=compute_100a,code=sm_100a", "-o", OUT, *objs]
    subprocess.run(link, check=True)
    return OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
