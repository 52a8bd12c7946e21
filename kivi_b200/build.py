"""nvcc recipe for libkivi_b200.so (sm_100a only, in-tree, no torch headers).

    python -m kivi_b200.build [--force] [--verbose]

The shared object lands next to the sources (kivi_b200/csrc/libkivi_b200.so): git-ignored, but
it travels to the GPU box with gpurun.  nvcc cross-compiles without a GPU.
"""
from __future__ import annotations

import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
SO = os.path.join(CSRC, "libkivi_b200.so")
SOURCES = ["kivi_api.cu", "kivi_pack.cu", "kivi_bgemv.cu", "kivi_bgemv_mma.cu", "kivi_cache.cu", "kivi_decode.cu", "kivi_attn_k2v2.cu",
           "kivi_attn_k4v4.cu", "kivi_attn_k2v4.cu", "kivi_attn_k4v2.cu", "kivi_model.cu", "kivi_sample.cu"]
HEADERS = ["kivi_common.cuh", "kivi_decode.cuh", "kivi_attn.cuh", os.path.join("..", "..", "include", "kivi_b200.h")]
NVCC_FLAGS = ["-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo",
              "-Xcompiler", "-fPIC", "--expt-relaxed-constexpr"]


def _nvcc() -> str:
    return os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", "nvcc")


def _sources():
    return [s for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]


def needs_build() -> bool:
    if not os.path.exists(SO):
        return True
    t = os.path.getmtime(SO)
    deps = [os.path.join(CSRC, s) for s in _sources()] + \
           [os.path.join(CSRC, h) for h in HEADERS if os.path.exists(os.path.join(CSRC, h))]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not needs_build():
        return SO
    objs = []
    procs = []
    for s in _sources():
        obj = os.path.join(CSRC, s.replace(".cu", ".o"))
        cmd = [_nvcc(), "-c", os.path.join(CSRC, s), "-o", obj] + NVCC_FLAGS
        if verbose:
            cmd += ["-Xptxas", "-v"]
        procs.append((cmd, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(obj)
    for cmd, p in procs:
        out, _ = p.communicate()
        if verbose or p.returncode != 0:
            sys.stderr.write(" ".join(cmd) + "\n" + out)
        if p.returncode != 0:
            raise RuntimeError(f"nvcc failed ({p.returncode}) for: {' '.join(cmd)}")
    tmp = SO + ".tmp"
    subprocess.check_call([_nvcc(), "-shared", "-o", tmp] + objs +
                          ["-gencode", "arch=compute_100a,code=sm_100a", "-Xcompiler", "-fPIC", "-lcudart"])
    os.replace(tmp, SO)
    for o in objs:
        os.remove(o)
    return SO


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
