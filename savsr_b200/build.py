"""Build libsavsr_sm100.so in-tree with nvcc for sm_100a (no torch headers, no JIT cache)."""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB_DIR = os.path.join(HERE, "lib")
LIB_PATH = os.path.join(LIB_DIR, "libsavsr_sm100.so")
SOURCES = ["capi.cu", "conv_igemm.cu", "conv_wgrad.cu", "train_ops.cu", "train_attn.cu", "train_mask.cu", "plan.cu", "small_ops.cu", "satu.cu", "datapath.cu", "colour.cu", "scenes.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC", "-Xcompiler", "-Wall", "--expt-relaxed-constexpr"]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found (set NVCC=/path/to/nvcc)")


def _stale(out: str, deps: list[str]) -> bool:
    if not os.path.exists(out):
        return True
    t = os.path.getmtime(out)
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    os.makedirs(LIB_DIR, exist_ok=True)
    nvcc = _nvcc()
    headers = [os.path.join(CSRC, "common.cuh"), os.path.join(HERE, "..", "include", "savsr_b200.h")]
    objs = []
    procs = []
    for src in SOURCES:
        s = os.path.join(CSRC, src)
        o = os.path.join(LIB_DIR, src.replace(".cu", ".o"))
        objs.append(o)
        if force or _stale(o, [s] + headers):
            cmd = [nvcc, *NVCC_FLAGS, "-c", s, "-o", o] + (["-Xptxas", "-v"] if verbose else [])
            procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    failed = False
    for src, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0 or verbose:
            print(f"--- nvcc {src} (exit {p.returncode})\n{out}", file=sys.stderr)
        failed |= p.returncode != 0
    if failed:
        raise RuntimeError("nvcc failed; see output above")
    if force or procs or _stale(LIB_PATH, objs):
        cmd = [nvcc, "-shared", "-o", LIB_PATH, *objs, "-gencode", "arch=compute_100a,code=sm_100a"]
        subprocess.run(cmd, check=True)
    return LIB_PATH


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
