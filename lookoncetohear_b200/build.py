"""Build the in-tree CUDA extension (C-ABI shared library) for sm_100a with nvcc.

    python -m lookoncetohear_b200.build [--force]

The .so lands in lookoncetohear_b200/lib/ (git-ignored, but it travels to the GPU box with the
gpurun snapshot).  nvcc cross-compiles without a GPU.
"""
import hashlib
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIBDIR = os.path.join(HERE, "lib")
LIB = os.path.join(LIBDIR, "liblookonce_b200.so")
SOURCES = ["sep_engine.cu", "embed_engine.cu", "umma_gemm.cu", "eval_metrics.cu", "render.cu", "binaural_metrics.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "--compiler-options", "-fPIC", "-shared", "-Xptxas", "-v"]


def _fingerprint():
    h = hashlib.sha256()
    inc = os.path.join(os.path.dirname(HERE), "include")
    for d in (CSRC, inc):
        for fn in sorted(os.listdir(d)):
            if fn.endswith((".cu", ".cuh", ".h")):
                with open(os.path.join(d, fn), "rb") as f:
                    h.update(fn.encode())
                    h.update(f.read())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def nvcc_path():
    for c in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if c and (os.path.isfile(c) or c == "nvcc"):
            return c
    return "nvcc"


def build(force=False, verbose=False):
    """Compile if sources changed since the last build.  Returns the library path."""
    os.makedirs(LIBDIR, exist_ok=True)
    stamp = LIB + ".sha256"
    fp = _fingerprint()
    if not force and os.path.isfile(LIB) and os.path.isfile(stamp) and open(stamp).read().strip() == fp:
        return LIB
    cmd = [nvcc_path()] + NVCC_FLAGS + ["-o", LIB] + [os.path.join(CSRC, s) for s in SOURCES]
    res = subprocess.run(cmd, capture_output=True, text=True)
    log = res.stdout + res.stderr
    with open(os.path.join(LIBDIR, "build.log"), "w") as f:
        f.write(" ".join(cmd) + "\n" + log)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + log[-4000:])
    if verbose:
        print(log)
    with open(stamp, "w") as f:
        f.write(fp)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
