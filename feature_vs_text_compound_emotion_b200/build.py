"""Compile csrc/*.cu into the in-tree shared library libcer_b200.so for sm_100a.

nvcc cross-compiles without a GPU; the .so is git-ignored but travels to the GPU box.
    python -m feature_vs_text_compound_emotion_b200.build [--force]
"""
from __future__ import annotations

import hashlib
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
INCLUDE = os.path.join(os.path.dirname(HERE), "include")
LIB = os.path.join(HERE, "libcer_b200.so")
STAMP = os.path.join(HERE, ".libcer_b200.stamp")
SOURCES = ["common.cu", "ir50.cu", "vggish.cu", "tcn.cu", "tcn_tc.cu", "fusion.cu", "train.cu", "preproc.cu", "logmel.cu", "heads.cu", "se.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC,-O2"]


def _nvcc() -> str:
    for cand in (shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: cannot build libcer_b200.so")


def _digest() -> str:
    h = hashlib.sha256()
    files = [os.path.join(CSRC, f) for f in sorted(os.listdir(CSRC))] + [os.path.join(INCLUDE, "cer_b200.h")]
    for f in files:
        h.update(f.encode())
        h.update(open(f, "rb").read())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def build(force: bool = False, verbose: bool = False) -> str:
    digest = _digest()
    if not force and os.path.exists(LIB) and os.path.exists(STAMP) and open(STAMP).read().strip() == digest:
        return LIB
    objs = []
    procs = []
    tmp = os.path.join(HERE, "build")
    os.makedirs(tmp, exist_ok=True)
    for src in SOURCES:
        obj = os.path.join(tmp, src.replace(".cu", ".o"))
        cmd = [_nvcc(), *NVCC_FLAGS, "-I", INCLUDE, "-c", os.path.join(CSRC, src), "-o", obj]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(obj)
    for src, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0:
            raise RuntimeError(f"nvcc failed on {src}:\n{out}")
        if verbose:
            print(out)
    link = [_nvcc(), "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", LIB, *objs]
    r = subprocess.run(link, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}")
    open(STAMP, "w").write(digest)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
