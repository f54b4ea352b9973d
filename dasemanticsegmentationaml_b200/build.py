"""Builds libb200seg.so (the C-ABI CUDA library) in-tree with nvcc for sm_100a.

Usage: ``python -m dasemanticsegmentationaml_b200.build [--force]``.  The library is compiled from
``csrc/*.cu`` with ``-gencode arch=compute_100a,code=sm_100a -lineinfo`` (tcgen05 / TMA need the
arch-specific ``a`` target) and linked with the static CUDA runtime, so the only run-time
dependency is the driver.  No GPU is needed to build.
"""
import hashlib
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(HERE, "build")
LIB = os.path.join(HERE, "libb200seg.so")

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC", "-I", CSRC,
    "-I", os.path.join(os.path.dirname(HERE), "include"),
]
# --use_fast_math (approximate division / exp / rsqrt, flush-to-zero) only where it pays and is
# covered by a parity test with the flag ON: the GEMM epilogues (igemm.cu: no transcendental at all)
# and the issue-bound up-sampling / softmax / cross-entropy kernels (loss.cu: __expf / __logf per
# pixel and class; tests/test_modules_gpu.py::test_fused_losses_against_torch holds the loss to 1e-4
# and the gradients to 1e-3 against torch).  BatchNorm statistics, optimizers, depthwise convs, metrics
# and the input pipeline are compiled with IEEE division / sqrt.
FAST_MATH_SOURCES = ("igemm.cu", "loss.cu")


def _nvcc():
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    raise RuntimeError("nvcc not found")


def _digest(paths):
    """Hash of the sources and flags with paths relative to the repository, so that a built tree that is
    moved or copied (read-only, say) is not rebuilt."""
    root = os.path.dirname(HERE)
    h = hashlib.sha1()
    for p in sorted(paths):
        with open(p, "rb") as f:
            h.update(os.path.relpath(p, root).encode())
            h.update(f.read())
    h.update(" ".join(NVCC_FLAGS + list(FAST_MATH_SOURCES)).replace(root, "").encode())
    return h.hexdigest()


def sources():
    return sorted(os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith(".cu"))


def headers():
    inc = os.path.join(os.path.dirname(HERE), "include")
    hs = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".h", ".cuh"))]
    if os.path.isdir(inc):
        hs += [os.path.join(inc, f) for f in os.listdir(inc) if f.endswith(".h")]
    return sorted(hs)


def build(force=False, verbose=False):
    """Compile every csrc/*.cu and link libb200seg.so; skipped when sources are unchanged."""
    os.makedirs(OBJ, exist_ok=True)
    stamp = os.path.join(OBJ, "stamp")
    dig = _digest(sources() + headers())
    if not force and os.path.exists(LIB) and os.path.exists(stamp) and open(stamp).read() == dig:
        return LIB
    nvcc = _nvcc()
    objs = []

    def compile_one(src):
        obj = os.path.join(OBJ, os.path.basename(src)[:-3] + ".o")
        cmd = [nvcc] + NVCC_FLAGS + (["--use_fast_math"] if os.path.basename(src) in FAST_MATH_SOURCES else []) + ["-c", src, "-o", obj]
        if verbose:
            cmd.insert(1, "-Xptxas")
            cmd.insert(2, "-v")
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("nvcc failed for %s:\n%s\n%s" % (src, r.stdout, r.stderr))
        if verbose:
            sys.stderr.write(r.stderr)
        return obj

    with ThreadPoolExecutor(max_workers=min(8, os.cpu_count() or 1)) as ex:
        objs = list(ex.map(compile_one, sources()))
    cmd = [nvcc, "-shared", "-o", LIB] + objs + ["-gencode", "arch=compute_100a,code=sm_100a",
                                                  "-cudart", "static", "-Xcompiler", "-fPIC", "-ldl"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("link failed:\n%s\n%s" % (r.stdout, r.stderr))
    with open(stamp, "w") as f:
        f.write(dig)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
