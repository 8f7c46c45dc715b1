"""Build libmocha_b200.so in-tree with nvcc for sm_100a (cross-compiles without a GPU).

    python -m mocha_sigasia2023_b200.build [--force] [--verbose]

The shared library is git-ignored but travels to the GPU box with the gpurun snapshot.
"""
from __future__ import annotations

import hashlib
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
ROOT = os.path.dirname(HERE)
LIB = os.path.join(HERE, "libmocha_b200.so")
OBJ_DIR = os.path.join(HERE, "build")

SOURCES = ["api.cu", "gemm_f32.cu", "ops.cu", "gemm_tc.cu", "fused_tail.cu", "fused_attn.cu", "match.cu", "networks.cu",
           "networks_bf16.cu", "kinematics.cu", "ingest.cu"]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17",
    "-Xcompiler", "-fPIC",
    "--expt-relaxed-constexpr",
    "-Xptxas", "-v",
]


def _nvcc() -> str:
    cand = os.environ.get("NVCC") or "/usr/local/cuda/bin/nvcc"
    return cand if os.path.exists(cand) else "nvcc"


def _digest(paths) -> str:
    h = hashlib.sha256()
    for p in sorted(paths):
        with open(p, "rb") as f:
            h.update(p.encode())
            h.update(f.read())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def build(force: bool = False, verbose: bool = False, trace: bool = False) -> str:
    """trace=True builds libmocha_b200_trace.so with -DMOCHA_TRACE (in-kernel time lines for tools/tc_trace.py)."""
    lib_path = LIB.replace(".so", "_trace.so") if trace else LIB
    obj_dir = OBJ_DIR + ("_trace" if trace else "")
    flags = NVCC_FLAGS + (["-DMOCHA_TRACE"] if trace else [])
    srcs = [os.path.join(CSRC, s) for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]
    deps = srcs + [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith(".cuh")]
    deps.append(os.path.join(ROOT, "include", "mocha_b200.h"))
    stamp = os.path.join(obj_dir, "stamp")
    digest = _digest(deps)
    if not force and os.path.exists(lib_path) and os.path.exists(stamp) and open(stamp).read() == digest:
        return lib_path
    os.makedirs(obj_dir, exist_ok=True)

    def compile_one(src: str) -> str:
        obj = os.path.join(obj_dir, os.path.basename(src)[:-3] + ".o")
        cmd = [_nvcc(), *flags, "-c", src, "-o", obj]
        r = subprocess.run(cmd, capture_output=True, text=True)
        log = os.path.join(obj_dir, os.path.basename(src)[:-3] + ".ptxas.log")
        with open(log, "w") as f:
            f.write(r.stderr)
        # (nvcc can return 0 after a host-preprocessor error such as a macro arity mismatch: treat any "error:" line as fatal)
        if r.returncode != 0 or ": error:" in r.stderr or " error: " in r.stderr:
            raise RuntimeError(f"nvcc failed for {src}:\n{r.stdout}\n{r.stderr}")
        if verbose:
            sys.stderr.write(r.stderr)
        return obj

    with ThreadPoolExecutor(max_workers=min(8, len(srcs))) as ex:
        objs = list(ex.map(compile_one, srcs))
    cmd = [_nvcc(), "-shared", "-o", lib_path, *objs, "-gencode", "arch=compute_100a,code=sm_100a", "-lcudart"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    with open(stamp, "w") as f:
        f.write(digest)
    return lib_path


if __name__ == "__main__":
    path = build(force="--force" in sys.argv, verbose="--verbose" in sys.argv, trace="--trace" in sys.argv)
    print(path)
