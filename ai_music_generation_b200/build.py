"""Builds libabcgpt.so (the hand-written sm_100a kernels + C ABI) in-tree with nvcc.

No torch.utils.cpp_extension / JIT cache: the shared object lives next to the sources so that it travels to
the GPU box with the repository snapshot.  `python -m ai_music_generation_b200.build` or
`__graft_entry__.build()`.
"""
from __future__ import annotations

import hashlib
import os
import shutil
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJ_DIR = os.path.join(HERE, "build")
LIB_PATH = os.path.join(HERE, "libabcgpt.so")
DEBUG_LIB_PATH = os.path.join(HERE, "libabcgpt_debug.so")  # product objects + instrumentation entry points (tools/ only)
SOURCES = ["common.cu", "gemm.cu", "attn.cu", "attn_pair.cu", "attn_fwd3.cu", "attn_hd.cu", "attn_varlen.cu", "layernorm.cu", "elementwise.cu", "nvls.cu", "sample.cu", "api.cu"]
DEBUG_SOURCES = ["microbench.cu", "debug_api.cu"]  # include/abcgpt_debug.h; never linked into libabcgpt.so
HEADERS = ["common.h", "kernels.h", "ptx.cuh", "dropout.cuh", "attn_helpers.cuh", "attn_hd.cuh", os.path.join("..", "..", "include", "abcgpt.h"),
           os.path.join("..", "..", "include", "abcgpt_debug.h")]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-std=c++17", "-lineinfo",
    "-Xcompiler", "-fPIC",
    "--expt-relaxed-constexpr",
    "-Xptxas", "-v",
]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found; libabcgpt.so cannot be built")


def _digest() -> str:
    h = hashlib.sha256()
    for name in SOURCES + DEBUG_SOURCES + HEADERS:
        with open(os.path.join(CSRC, name), "rb") as f:
            h.update(f.read())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def build(force: bool = False, verbose: bool = False, debug: bool = False) -> str:
    """Compile (if stale) and return the path of libabcgpt.so (debug=True: also libabcgpt_debug.so, returns its path)."""
    stamp = os.path.join(OBJ_DIR, "stamp_debug" if debug else "stamp")
    target = DEBUG_LIB_PATH if debug else LIB_PATH
    digest = _digest()
    if not force and os.path.exists(target) and os.path.exists(stamp):
        with open(stamp) as f:
            if f.read().strip() == digest:
                return target
    os.makedirs(OBJ_DIR, exist_ok=True)
    nvcc = _nvcc()

    def compile_one(src: str) -> str:
        obj = os.path.join(OBJ_DIR, src.replace(".cu", ".o"))
        cmd = [nvcc, *NVCC_FLAGS, "-c", os.path.join(CSRC, src), "-o", obj]
        res = subprocess.run(cmd, capture_output=True, text=True)
        with open(obj + ".log", "w") as f:
            f.write(" ".join(cmd) + "\n" + res.stdout + res.stderr)
        if res.returncode != 0:
            raise RuntimeError(f"nvcc failed for {src}:\n{res.stdout}\n{res.stderr}")
        if verbose:
            sys.stderr.write(res.stderr)
        return obj

    srcs = SOURCES + (DEBUG_SOURCES if debug else [])
    with ThreadPoolExecutor(max_workers=min(len(srcs), os.cpu_count() or 4)) as ex:
        objs = list(ex.map(compile_one, srcs))
    # the product library never contains the instrumentation objects; the debug library is a superset
    links = [(LIB_PATH, objs[:len(SOURCES)], "stamp")]
    if debug:
        links.append((DEBUG_LIB_PATH, objs, "stamp_debug"))
    for path, members, stamp_name in links:
        cmd = [nvcc, "-shared", "-o", path, *members, "-lcudart"]
        res = subprocess.run(cmd, capture_output=True, text=True)
        if res.returncode != 0:
            raise RuntimeError(f"link failed:\n{res.stdout}\n{res.stderr}")
        with open(os.path.join(OBJ_DIR, stamp_name), "w") as f:
            f.write(digest)
    return target


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv, debug="--debug" in sys.argv))
