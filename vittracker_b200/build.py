"""In-tree build of libvittrack_b200.so with nvcc for sm_100a (no JIT cache: the .so sits next to the
sources so that it travels with a repo snapshot).

    python -m vittracker_b200.build [--force] [--verbose]
"""
from __future__ import annotations

import hashlib
import os
import shutil
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(PKG_DIR, "csrc")
INCLUDE = os.path.join(os.path.dirname(PKG_DIR), "include")
# VT_LIB_DIR: development builds (cycle traces, experiments) go to a side directory and are loaded from there
LIB_DIR = os.path.abspath(os.environ["VT_LIB_DIR"]) if os.environ.get("VT_LIB_DIR") else os.path.join(PKG_DIR, "lib")
LIB_PATH = os.path.join(LIB_DIR, "libvittrack_b200.so")
STAMP = os.path.join(LIB_DIR, "build.stamp")

SOURCES = ["vt_api.cu", "vt_crop.cu", "vt_stem.cu", "vt_stem_tc.cu", "vt_stem_fused.cu", "vt_block_simt.cu", "vt_block_tc.cu", "vt_head.cu", "vt_generic.cu", "vt_yuv.cu", "vt_slots.cu", "vt_records.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-lineinfo",
              "-Xcompiler", "-fPIC", "-Xcompiler", "-fno-fast-math", "-Xcompiler", "-fopenmp", "--fmad=true", "-I", INCLUDE]


class NvccMissing(RuntimeError):
    pass


def _nvcc() -> str:
    for c in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if c and os.path.isfile(c):
            return c
    raise NvccMissing("nvcc not found: libvittrack_b200.so cannot be built (there is no CPU fallback)")


def _sources():
    return [os.path.join(CSRC, s) for s in SOURCES if os.path.isfile(os.path.join(CSRC, s))]


def _digest() -> str:
    h = hashlib.sha256()
    h.update(" ".join(f for f in NVCC_FLAGS if f != INCLUDE).encode())
    h.update(os.environ.get("NVCC_EXTRA", "").encode())
    files = sorted(os.listdir(CSRC)) + [os.path.join(INCLUDE, f) for f in sorted(os.listdir(INCLUDE))]
    for f in files:
        p = f if os.path.isabs(f) else os.path.join(CSRC, f)
        if os.path.isfile(p):
            h.update(os.path.basename(p).encode())
            with open(p, "rb") as fh:
                h.update(fh.read())
    return h.hexdigest()


def is_fresh() -> bool:
    if not (os.path.isfile(LIB_PATH) and os.path.isfile(STAMP)):
        return False
    with open(STAMP) as fh:
        return fh.read().strip() == _digest()


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile every .cu for sm_100a and link the shared library; returns its path."""
    if not force and is_fresh():
        return LIB_PATH
    nvcc = _nvcc()
    os.makedirs(LIB_DIR, exist_ok=True)
    # one builder at a time (torchrun starts every rank at once): the others wait on the lock and find a fresh library
    import fcntl
    with open(os.path.join(LIB_DIR, ".build.lock"), "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        try:
            if not force and is_fresh():
                return LIB_PATH
            return _build_locked(nvcc, verbose)
        finally:
            fcntl.flock(lock, fcntl.LOCK_UN)


def _build_locked(nvcc: str, verbose: bool) -> str:
    objs = []

    def compile_one(src: str) -> str:
        obj = os.path.join(LIB_DIR, os.path.basename(src)[:-3] + ".o")
        extra = os.environ.get("NVCC_EXTRA", "").split()
        cmd = [nvcc, *NVCC_FLAGS, *extra, "-c", src, "-o", obj] + (["-Xptxas", "-v"] if verbose else [])
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError(f"nvcc failed for {src}:\n{r.stdout}\n{r.stderr}")
        if verbose:
            sys.stderr.write(r.stderr)
        return obj

    with ThreadPoolExecutor(max_workers=min(8, os.cpu_count() or 1)) as ex:
        objs = list(ex.map(compile_one, _sources()))
    cmd = [nvcc, "-shared", "-o", LIB_PATH, *objs, "-gencode", "arch=compute_100a,code=sm_100a", "-lcudart", "-lgomp"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    with open(STAMP, "w") as fh:
        fh.write(_digest())
    return LIB_PATH


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
