"""Build libzenflow_b200.so in-tree with nvcc for sm_100a (no JIT cache, no torch extension).

The library is a plain C-ABI shared object (include/zenflow_b200.h); it links only
against the CUDA runtime.  `python -m zenflow_b200.build` rebuilds when sources changed.
"""
from __future__ import annotations

import hashlib
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB_DIR = os.path.join(HERE, "_native")
LIB_PATH = os.path.join(LIB_DIR, "libzenflow_b200.so")
STAMP = os.path.join(LIB_DIR, "build.stamp")

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17",
    "-Xcompiler", "-fPIC", "-shared",
    "--cudart", "shared",
    "-Xptxas", "-v",
]


EXTRA_FLAGS = [f for f in os.environ.get("ZF_NVCC_EXTRA", "").split() if f]


def _sources():
    return sorted(os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith(".cu"))


def _digest() -> str:
    """Content digest of the sources and flags.  File NAMES only (no absolute paths): the tree is copied to other
    machines and must not look stale there."""
    h = hashlib.sha256()
    inc = os.path.join(os.path.dirname(HERE), "include", "zenflow_b200.h")
    files = [os.path.join(CSRC, f) for f in sorted(os.listdir(CSRC))] + [inc]
    for p in files:
        with open(p, "rb") as f:
            h.update(os.path.basename(p).encode())
            h.update(f.read())
    h.update(" ".join(NVCC_FLAGS + EXTRA_FLAGS).encode())
    return h.hexdigest()


def nvcc_path() -> str:
    p = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(p):
        raise RuntimeError("nvcc not found; zenflow_b200 needs the CUDA toolkit to build its kernels")
    return p


def _fresh(dig: str) -> bool:
    return os.path.exists(LIB_PATH) and os.path.exists(STAMP) and open(STAMP).read().strip() == dig


def is_fresh() -> bool:
    """True when the in-tree library was built from exactly the sources (and flags) in this tree."""
    return _fresh(_digest())


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile every .cu under csrc/ into one shared library. Returns its path.

    Safe under concurrent callers (one process per GPU): an exclusive file lock serialises the build, the library
    is written to a temporary name and renamed into place, and whoever gets the lock second finds it fresh."""
    import fcntl

    os.makedirs(LIB_DIR, exist_ok=True)
    dig = _digest()
    if not force and _fresh(dig):
        return LIB_PATH
    with open(os.path.join(LIB_DIR, "build.lock"), "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        try:
            if not force and _fresh(dig):
                return LIB_PATH
            tmp = LIB_PATH + f".tmp{os.getpid()}"
            # one nvcc per translation unit, in parallel; objects are reused when neither the source nor any
            # header nor the flags changed
            from concurrent.futures import ThreadPoolExecutor

            obj_dir = os.path.join(LIB_DIR, "obj")
            os.makedirs(obj_dir, exist_ok=True)
            hdr = hashlib.sha256()
            inc = os.path.join(os.path.dirname(HERE), "include", "zenflow_b200.h")
            for p in sorted(os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))) + [inc]:
                hdr.update(open(p, "rb").read())
            hdr.update(" ".join(NVCC_FLAGS + EXTRA_FLAGS).encode())
            compile_flags = [f for f in NVCC_FLAGS if f != "-shared"] + EXTRA_FLAGS

            def compile_one(src):
                key = hashlib.sha256(hdr.digest() + open(src, "rb").read()).hexdigest()[:24]
                obj = os.path.join(obj_dir, os.path.basename(src) + "." + key + ".o")
                if os.path.exists(obj):
                    return obj, "", 0
                for old in os.listdir(obj_dir):
                    if old.startswith(os.path.basename(src) + "."):
                        os.remove(os.path.join(obj_dir, old))
                otmp = obj + f".tmp{os.getpid()}"
                r = subprocess.run([nvcc_path()] + compile_flags + ["-c", "-o", otmp, src], capture_output=True, text=True)
                if r.returncode == 0:
                    os.replace(otmp, obj)
                return obj, "# " + os.path.basename(src) + "\n" + r.stdout + r.stderr, r.returncode

            with ThreadPoolExecutor(max_workers=min(8, os.cpu_count() or 1)) as pool:
                results = list(pool.map(compile_one, _sources()))
            log = "".join(r[1] for r in results)
            rc = max(r[2] for r in results)
            cmd = [nvcc_path()] + NVCC_FLAGS + EXTRA_FLAGS + ["-o", tmp] + [r[0] for r in results] + ["-ldl"]
            if rc == 0:
                res = subprocess.run(cmd, capture_output=True, text=True)
                log += res.stdout + res.stderr
                rc = res.returncode
            with open(os.path.join(LIB_DIR, "build.log"), "w") as f:
                f.write(" ".join(cmd).replace(tmp, LIB_PATH) + "\n" + log)
            if rc != 0:
                if os.path.exists(tmp):
                    os.remove(tmp)
                raise RuntimeError("nvcc failed:\n" + log[-8000:])
            if verbose:
                print(log)
            os.replace(tmp, LIB_PATH)
            with open(STAMP + ".tmp", "w") as f:
                f.write(dig)
            os.replace(STAMP + ".tmp", STAMP)
        finally:
            fcntl.flock(lock, fcntl.LOCK_UN)
    return LIB_PATH


if __name__ == "__main__":
    path = build(force="--force" in sys.argv, verbose=True)
    print("built", path)
