"""Build ``libmgd.so`` in-tree with nvcc for sm_100a (B200).

``python -m multigriddet_b200.build`` or ``build()``.  The library is a plain
C-ABI shared object (no Python / torch linkage); it travels to the GPU box with
the repository snapshot.
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libmgd.so")
SOURCES = ("api.cu", "encode.cu", "decode.cu", "nms.cu", "match.cu", "boxes.cu", "loss.cu", "exchange.cu", "map.cu",
           "recall.cu")
HEADERS = ("common.cuh", "decode_math.cuh", "libm_emul.h", "dlpack_abi.h", os.path.join("..", "..", "include", "mgd.h"))

# -fmad=false: integer results (anchor, cell, keep set) depend on IEEE operations in
# the reference's order; nothing may be contracted into an FMA.  No fast-math.
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17", "-fmad=false",
    "-Xcompiler", "-fPIC,-O2,-Wall,-fvisibility=hidden",
    "-Xptxas", "-v",
]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.isfile(cand):
            return cand
    raise RuntimeError("nvcc not found: libmgd cannot be built (there is no CPU fallback)")


def is_stale() -> bool:
    if not os.path.isfile(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, s) for s in SOURCES + HEADERS] + [os.path.abspath(__file__)]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not is_stale():
        return LIB
    nvcc = _nvcc()
    objdir = os.path.join(HERE, "build")
    os.makedirs(objdir, exist_ok=True)
    # one nvcc per source, side by side (the sources are independent translation units)
    from concurrent.futures import ThreadPoolExecutor

    def compile_one(src):
        obj = os.path.join(objdir, src.replace(".cu", ".o"))
        cmd = [nvcc, *NVCC_FLAGS, "-c", os.path.join(CSRC, src), "-o", obj]
        return src, obj, subprocess.run(cmd, capture_output=True, text=True)

    objs = []
    log = []
    with ThreadPoolExecutor(max_workers=min(len(SOURCES), os.cpu_count() or 1)) as pool:
        for src, obj, r in pool.map(compile_one, SOURCES):
            log.append(r.stderr)
            if r.returncode != 0:
                sys.stderr.write(r.stdout + r.stderr)
                raise RuntimeError("nvcc failed on " + src)
            objs.append(obj)
    cmd = [nvcc, "-shared", "-o", LIB, *objs, "-Xcompiler", "-fPIC"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout + r.stderr)
        raise RuntimeError("link failed")
    with open(os.path.join(objdir, "ptxas.log"), "w") as fh:
        fh.write("\n".join(log))
    if verbose:
        sys.stderr.write("\n".join(log))
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
