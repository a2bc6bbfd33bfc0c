"""In-tree build of the C-ABI library (nvcc, sm_100a only).

    python -m autogptq_b200.build        # or: python __graft_entry__.py build

Produces ``autogptq_b200/_C/libautogptq_b200.so``.  The .so is git-ignored but travels to the GPU box
with the repo snapshot; nothing is installed into site-packages.
"""
from __future__ import annotations

import hashlib
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT_DIR = os.path.join(HERE, "_C")
LIB_NAME = "libautogptq_b200.so"
LIB_PATH = os.path.join(OUT_DIR, LIB_NAME)
STAMP = os.path.join(OUT_DIR, "build.stamp")

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-std=c++17", "-lineinfo",
    "-Xcompiler", "-fPIC",
    "-DAGB200_NO_FAST_MATH",
]
# translation units of the library (compiled in parallel, then linked)
UNITS = ["abi.cu", "chain.cu"]
# chain.cu holds only the 576-thread persistent chain kernel: 65536 / 576 = 113 registers per thread at most
UNIT_FLAGS = {"chain.cu": ["-maxrregcount=112"]}


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: the CUDA extension cannot be built (there is no CPU fallback)")


def _sources_digest() -> str:
    h = hashlib.sha256()
    files = sorted(os.listdir(CSRC)) + ["../../include/autogptq_b200.h"]
    for f in files:
        p = os.path.join(CSRC, f)
        if os.path.isfile(p):
            h.update(f.encode())
            h.update(open(p, "rb").read())
    h.update(" ".join(NVCC_FLAGS).encode())
    h.update(repr(sorted(UNIT_FLAGS.items())).encode())
    return h.hexdigest()


def build_extension(force: bool = False, verbose: bool = False) -> str:
    os.makedirs(OUT_DIR, exist_ok=True)
    digest = _sources_digest()
    if not force and os.path.exists(LIB_PATH) and os.path.exists(STAMP) and open(STAMP).read().strip() == digest:
        return LIB_PATH
    nvcc = _nvcc()
    only = os.environ.get("AGB200_BUILD_ONLY")          # developer aid: recompile just these units (comma separated)
    procs = []
    objs = []
    for unit in UNITS:
        obj = os.path.join(OUT_DIR, unit.replace(".cu", ".o"))
        objs.append(obj)
        if only and unit not in only.split(",") and os.path.exists(obj):
            continue
        cmd = [nvcc, *NVCC_FLAGS, *UNIT_FLAGS.get(unit, []), "-c", "-o", obj, os.path.join(CSRC, unit)]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
            print(" ".join(cmd), flush=True)
        procs.append((unit, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)))
    for unit, proc in procs:
        out, err = proc.communicate()
        if proc.returncode != 0:
            sys.stderr.write(out + err)
            raise RuntimeError(f"nvcc failed on {unit} with exit code {proc.returncode}")
        if verbose:
            sys.stderr.write(err)
    link = subprocess.run([nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", LIB_PATH, *objs],
                          capture_output=True, text=True)
    if link.returncode != 0:
        sys.stderr.write(link.stdout + link.stderr)
        raise RuntimeError(f"link failed with exit code {link.returncode}")
    with open(STAMP, "w") as f:
        f.write(digest)
    return LIB_PATH


if __name__ == "__main__":
    print(build_extension(force="--force" in sys.argv, verbose="-v" in sys.argv))
