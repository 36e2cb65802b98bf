"""Build the CUDA extension in-tree: gym_lmaze_b200/liblmaze_b200.so (sm_100a only).

The .so is git-ignored but travels to the GPU box with the repo snapshot.  It
links the CUDA runtime statically and has no dependency on torch or Python.
"""
import os
import shutil
import subprocess

_PKG = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(_PKG)
LIB_PATH = os.path.join(_PKG, "liblmaze_b200.so")
SOURCES = [os.path.join(_PKG, "csrc", "lmz_abi.cu")]
HEADERS = [os.path.join(_PKG, "csrc", "lmz_kernels.cuh"), os.path.join(_PKG, "csrc", "lmz_variants.h"),
           os.path.join(_PKG, "csrc", "lmz_v2.cuh"), os.path.join(_PKG, "csrc", "lmz_v5.cuh"), os.path.join(_PKG, "csrc", "lmz_fov.cuh"),
           os.path.join(_PKG, "csrc", "lmz_fov_rollout.cuh"), os.path.join(_PKG, "csrc", "lmz_final.cuh"),
           os.path.join(_ROOT, "include", "lmaze_b200.h"), os.path.join(_ROOT, "include", "lmz_dlpack.h")]


def _nvcc():
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.isfile(cand):
            return cand
    raise RuntimeError("nvcc not found: cannot build the sm_100a extension")


def nvcc_command(out=LIB_PATH, extra=()):
    return [_nvcc(), "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
            "-Xcompiler", "-fPIC", "-shared", "-cudart", "static", "-ccbin", shutil.which("g++") or "g++",
            "-I", os.path.join(_ROOT, "include"), *extra, "-o", out, *SOURCES]


def source_hash():
    """sha256 over the kernel sources and the public headers (path-sorted): what profiles/traffic.json and the
    ncu summaries are keyed by, so that a capture of older kernels cannot pass as evidence for the current ones."""
    import hashlib
    h = hashlib.sha256()
    for f in sorted(SOURCES + HEADERS):
        h.update(os.path.relpath(f, _ROOT).encode())
        h.update(b"\0")
        h.update(open(f, "rb").read())
    return h.hexdigest()[:16]


def is_stale():
    if not os.path.isfile(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    return any(os.path.getmtime(f) > t for f in SOURCES + HEADERS)


def build(force=False, verbose=False):
    """Compile if the .so is missing or older than its sources.  Returns the path."""
    if force or is_stale():
        cmd = nvcc_command(extra=("-Xptxas", "-v") if verbose else ())
        res = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
        if verbose or res.returncode != 0:
            print(res.stdout)
        if res.returncode != 0:
            raise RuntimeError("nvcc failed (exit %d)" % res.returncode)
    return LIB_PATH


if __name__ == "__main__":
    import sys
    build(force=True, verbose="-v" in sys.argv)
    print(LIB_PATH)
