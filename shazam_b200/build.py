"""Build the sm_100a shared library IN-TREE (shazam_b200/_lib/libsia_b200.so).

nvcc cross-compiles without a GPU; the built .so travels to the GPU box with the
repo snapshot (it is git-ignored, not gpurun-ignored)."""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIBDIR = os.path.join(HERE, "_lib")
LIB = os.path.join(LIBDIR, "libsia_b200.so")
SOURCES = ["api.cu", "scan.cu", "stft.cu", "peaks.cu", "pairs_sha1.cu", "sort.cu", "index_store.cu", "index_query.cu", "index_apriori.cu", "index_pvote.cu", "index_dist.cu", "noise.cu",
           "stream.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC", "-Xcompiler", "-O3"]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found")


def _stale(target: str, deps) -> bool:
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build_native(force: bool = False, verbose: bool = False) -> str:
    os.makedirs(LIBDIR, exist_ok=True)
    headers = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))]
    headers.append(os.path.join(os.path.dirname(HERE), "include", "sia_b200.h"))
    sources = [s for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]
    nvcc = _nvcc()
    objs, procs = [], []
    for src in sources:
        path = os.path.join(CSRC, src)
        obj = os.path.join(LIBDIR, src.replace(".cu", ".o"))
        objs.append(obj)
        if force or _stale(obj, [path] + headers):
            cmd = [nvcc, *NVCC_FLAGS, "-c", path, "-o", obj]
            if verbose:
                cmd.insert(1, "-Xptxas=-v")
                print(" ".join(cmd), file=sys.stderr)
            procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    failed = []
    for src, p in procs:
        out, _ = p.communicate()
        if verbose and out:
            print(out, file=sys.stderr)
        if p.returncode != 0:
            failed.append(f"{src}:\n{out}")
    if failed:
        raise RuntimeError("nvcc failed:\n" + "\n".join(failed))
    if force or procs or _stale(LIB, objs):
        cmd = [nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", LIB, *objs]
        r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
        if r.returncode != 0:
            raise RuntimeError("link failed:\n" + r.stdout)
    return LIB


if __name__ == "__main__":
    print(build_native(force="--force" in sys.argv, verbose="-v" in sys.argv))
