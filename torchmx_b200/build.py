"""Build libmxq.so (hand-written sm_100a CUDA behind the C ABI in include/mxq.h) in-tree.

    python -m torchmx_b200.build [--force]

nvcc cross-compiles without a GPU.  The .so stays next to the sources (git-ignored, but it
travels to the GPU box with the repo snapshot).
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "lib", "libmxq.so")
SOURCES = ["mxq_api.cu", "mxq_quantize.cu", "mxq_dequantize.cu", "mxq_transcode.cu", "mxq_tmap.cu", "mxq_gemm.cu", "mxq_gemm_skinny.cu", "mxq_gemm_dequant.cu", "mxq_softmax.cu", "mxq_flash_attention.cu", "mxq_act_quant.cu", "mxq_glue.cu", "mxq_kv_cache.cu"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-std=c++17", "-lineinfo",
    "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden",
    "--expt-relaxed-constexpr",
    # NO --use_fast_math / -ftz: fp32 subnormals carry real values at the ends of the E8M0 range.
]


if os.environ.get("MXQ_DEV") == "1":  # developer build: the clock64 trace / tile-configuration hooks of the K3 kernels (tools/gemm_trace.py)
    NVCC_FLAGS.append("-DMXQ_DEV")


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: libmxq.so cannot be built (there is no CPU fallback)")


FLAGS_STAMP = os.path.join(HERE, "lib", "nvcc_flags.txt")  # a developer build must not be mistaken for a fresh release build


def _stale() -> bool:
    if not os.path.exists(LIB):
        return True
    if not os.path.exists(FLAGS_STAMP) or open(FLAGS_STAMP).read() != " ".join(NVCC_FLAGS):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(os.path.dirname(HERE), "include", "mxq.h"), __file__]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not _stale():
        return LIB
    os.makedirs(os.path.dirname(LIB), exist_ok=True)
    objdir = os.path.join(HERE, "lib", "obj")
    os.makedirs(objdir, exist_ok=True)
    nvcc = _nvcc()
    procs = []
    objs = []
    for src in SOURCES:
        obj = os.path.join(objdir, src.replace(".cu", ".o"))
        objs.append(obj)
        cmd = [nvcc, *NVCC_FLAGS, "-c", os.path.join(CSRC, src), "-o", obj]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
            print(" ".join(cmd), flush=True)
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    failed = False
    for src, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0 or verbose:
            sys.stderr.write(f"--- {src} ---\n{out}\n")
        failed |= p.returncode != 0
    if failed:
        raise RuntimeError("nvcc failed building libmxq.so")
    tmp = LIB + ".tmp"
    subprocess.check_call([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-o", tmp, *objs,
                           "-Xcompiler", "-fPIC", "-lcudart_static", "-lcuda"])
    os.replace(tmp, LIB)
    with open(FLAGS_STAMP, "w") as f:
        f.write(" ".join(NVCC_FLAGS))
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
