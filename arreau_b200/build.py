"""In-tree nvcc build of libarreau_b200.so (sm_100a only).

    python -m arreau_b200.build          # rebuild if any source is newer than the library

The library is built next to the sources (arreau_b200/lib/) so that it travels to the GPU box with the
repo snapshot; it is git-ignored.  There is no fallback: without the library the package raises.
"""
from __future__ import annotations

import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(HERE, "csrc")
LIB_DIR = os.path.join(HERE, "lib")
LIB_PATH = os.path.join(LIB_DIR, "libarreau_b200.so")
SOURCES = ["graph.cu", "state.cu", "model_simt.cu", "model_tc.cu", "step.cu", "train_ops.cu", "train_net.cu",
           "metrics.cu"]
HEADERS = [os.path.join(CSRC, "common.cuh"), os.path.join(CSRC, "tc_common.cuh"),
           os.path.join(ROOT, "include", "arreau_b200.h")]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC", "-Xptxas", "-v"]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    raise RuntimeError("nvcc not found")


def needs_build() -> bool:
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    deps = [os.path.join(CSRC, s) for s in SOURCES] + HEADERS + [os.path.abspath(__file__)]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile every .cu for sm_100a into one shared library; returns its path."""
    if not force and not needs_build():
        return LIB_PATH
    os.makedirs(LIB_DIR, exist_ok=True)
    objs = []
    procs = []
    for s in SOURCES:
        obj = os.path.join(LIB_DIR, s.replace(".cu", ".o"))
        objs.append(obj)
        cmd = [_nvcc(), *NVCC_FLAGS, *os.environ.get("ARREAU_NVCC_EXTRA", "").split(), "-c", os.path.join(CSRC, s), "-o", obj]
        procs.append((s, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    log = []
    for s, p in procs:
        out, _ = p.communicate()
        log.append(f"== {s}\n{out}")
        if p.returncode != 0:
            raise RuntimeError(f"nvcc failed on {s}:\n{out}")
    tmp = LIB_PATH + ".tmp"
    link = subprocess.run([_nvcc(), "-shared", "-o", tmp, *objs], stdout=subprocess.PIPE, stderr=subprocess.STDOUT,
                          text=True)
    if link.returncode != 0:
        raise RuntimeError(f"link failed:\n{link.stdout}")
    os.replace(tmp, LIB_PATH)
    with open(os.path.join(LIB_DIR, "build.log"), "w") as f:
        f.write("\n".join(log))
    if verbose:
        print("\n".join(log))
    return LIB_PATH


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
