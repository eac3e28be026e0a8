"""Build recipe for libcwipc_util_cuda.so (sm_100a only).

The library is plain C++17 + CUDA compiled with nvcc: no PyTorch, no Triton, no CMake.  It is
built IN-TREE (cwipc_util_b200/lib/) so that the .so travels with the repo snapshot to the GPU box.

    python -m cwipc_util_b200.build            # build what is out of date
    python -m cwipc_util_b200.build --force
"""
from __future__ import annotations

import concurrent.futures
import fcntl
import hashlib
import os
import shutil
import subprocess
import sys

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
REPO_DIR = os.path.dirname(PKG_DIR)
CSRC_DIR = os.path.join(PKG_DIR, "csrc")
LIB_DIR = os.path.join(PKG_DIR, "lib")
OBJ_DIR = os.path.join(REPO_DIR, "build", "obj")
INCLUDE_DIR = os.path.join(REPO_DIR, "include")

LIB_NAME = "libcwipc_util_cuda.so"
# Same library under the name python/cwipc/util.py looks up with find_library('cwipc_util').
DROPIN_NAME = "libcwipc_util.so"

SOURCES = [
    "runtime.cu",
    "pointops.cu",
    "radix_sort.cu",
    "downsample.cu",
    "outliers.cu",
    "logging.cpp",
    "pointcloud.cpp",
    "filters.cpp",
    "icp.cpp",
    "slab.cpp",
    "abi.cpp",
    "synthetic.cpp",
    "ply.cpp",
]

NVCC_FLAGS = [
    "-std=c++17",
    "-O3",
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-lineinfo",
    "-fmad=false",  # float parity with the reference's non-contracted x86-64 arithmetic
    "-Xcompiler", "-fPIC,-fvisibility=hidden,-Wall,-Wno-unused-function",
    "-I", INCLUDE_DIR,
    "-I", CSRC_DIR,
]


def _nvcc() -> str:
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        raise RuntimeError("nvcc not found: libcwipc_util_cuda cannot be built")
    return nvcc


def _headers_digest() -> "hashlib._Hash":
    """Content hash of every header + the flags (mtimes do not survive the copy to the GPU box)."""
    h = hashlib.sha1(" ".join(NVCC_FLAGS).encode())
    for d in (CSRC_DIR, INCLUDE_DIR):
        for root, _, files in sorted(os.walk(d)):
            for f in sorted(files):
                if f.endswith((".h", ".hpp", ".cuh")):
                    h.update(f.encode())
                    h.update(open(os.path.join(root, f), "rb").read())
    return h


def _is_current(stamp: str, digest: str, *artefacts: str) -> bool:
    if not all(os.path.exists(a) for a in artefacts) or not os.path.exists(stamp):
        return False
    return open(stamp).read().strip() == digest


def _compile_one(args) -> str:
    src, obj, verbose = args
    tmp = f"{obj}.tmp{os.getpid()}.o"
    cmd = [_nvcc(), *NVCC_FLAGS, "-x", "cu", "-c", src, "-o", tmp]
    if verbose:
        cmd.insert(1, "-Xptxas=-v")
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"nvcc failed on {os.path.basename(src)}:\n{r.stdout}\n{r.stderr}")
    os.replace(tmp, obj)   # never a half-written object under the final name
    return r.stderr if verbose else ""


def _link(objs, target: str, soname: str) -> None:
    tmp = f"{target}.tmp{os.getpid()}"
    cmd = [_nvcc(), "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-Xcompiler", "-fPIC", "-Xlinker", f"-soname={soname}", "-o", tmp, *objs, "-lpthread", "-ldl"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"link failed:\n{r.stdout}\n{r.stderr}")
    os.chmod(tmp, 0o755)
    os.replace(tmp, target)


def lib_path() -> str:
    return os.path.join(LIB_DIR, LIB_NAME)


def build_library(force: bool = False, verbose: bool = False) -> str:
    """Build what is out of date.  Safe to call from several processes at once (every rank of a torchrun launch on a
    fresh checkout does): the whole build runs under an exclusive file lock, the stamp is re-checked once the lock is
    held, and objects / libraries are written under temporary names and renamed into place."""
    os.makedirs(OBJ_DIR, exist_ok=True)
    os.makedirs(LIB_DIR, exist_ok=True)
    hdr = _headers_digest()
    target = lib_path()
    dropin = os.path.join(LIB_DIR, DROPIN_NAME)
    # whole-library stamp first: on the GPU box the prebuilt .so is used as is
    lib_h = hdr.copy()
    digests = {}
    for name in SOURCES:
        h = hdr.copy()
        h.update(open(os.path.join(CSRC_DIR, name), "rb").read())
        digests[name] = h.hexdigest()
        lib_h.update(digests[name].encode())
    lib_stamp = os.path.join(LIB_DIR, ".stamp")
    if not force and _is_current(lib_stamp, lib_h.hexdigest(), target, dropin):
        return target
    with open(os.path.join(LIB_DIR, ".lock"), "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        try:
            if not force and _is_current(lib_stamp, lib_h.hexdigest(), target, dropin):
                return target   # another process built it while we waited
            jobs, objs = [], []
            for name in SOURCES:
                src = os.path.join(CSRC_DIR, name)
                obj = os.path.join(OBJ_DIR, name + ".o")
                objs.append(obj)
                if force or not _is_current(obj + ".stamp", digests[name], obj):
                    jobs.append((src, obj, verbose))
            if jobs:
                with concurrent.futures.ThreadPoolExecutor(max_workers=min(8, len(jobs))) as ex:
                    for out in ex.map(_compile_one, jobs):
                        if out:
                            print(out, file=sys.stderr)
                for src, obj, _ in jobs:
                    open(obj + ".stamp", "w").write(digests[os.path.basename(src)])
            _link(objs, target, LIB_NAME)
            # the drop-in carries its own SONAME: ctypes.util.find_library('cwipc_util') (python/cwipc/util.py:149-161)
            # resolves a library on LD_LIBRARY_PATH through its SONAME
            _link(objs, dropin, DROPIN_NAME)
            tmp = lib_stamp + f".tmp{os.getpid()}"
            open(tmp, "w").write(lib_h.hexdigest())
            os.replace(tmp, lib_stamp)
        finally:
            fcntl.flock(lock, fcntl.LOCK_UN)
    return target


if __name__ == "__main__":
    force = "--force" in sys.argv
    verbose = "--verbose" in sys.argv
    print(build_library(force=force, verbose=verbose))
