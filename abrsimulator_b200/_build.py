"""Builds libabr_b200.so (sm_100a) in-tree with nvcc.

Used by ``__graft_entry__.build()`` and on first import when the library is
missing but a toolchain is present.  The .so is git-ignored but travels to the
GPU box with the repo snapshot.
"""
from __future__ import annotations

import hashlib
import os
import shutil
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
# development only: ABR_LIB_SUFFIX=_x builds/loads lib/libabr_b200_x.so with ABR_EXTRA_NVCC_FLAGS (A/B kernel variants)
_SUFFIX = os.environ.get("ABR_LIB_SUFFIX", "")
LIB = os.path.join(HERE, "lib", f"libabr_b200{_SUFFIX}.so")
STAMP = LIB + ".srchash"
SOURCES = ["abr_step.cu", "abr_mpc.cu", "abr_mpc_scen.cu", "abr_capi.cu", "abr_sort.cu"]
HEADERS = [os.path.join(CSRC, "abr_common.cuh"), os.path.join(CSRC, "abr_mpc_search.cuh"),
           os.path.join(HERE, "..", "include", "abr_b200.h"),
           os.path.join(HERE, "..", "include", "abr_b200_lookahead.h"),
           os.path.join(HERE, "..", "include", "abr_b200_mpc_pred.h"),
           os.path.join(HERE, "..", "include", "abr_b200_mpc_scen.h"),
           os.path.join(HERE, "..", "include", "abr_b200_obs.h")]

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-fmad=false", "-std=c++17",
              "-Xcompiler", "-fPIC", "-shared", "-cudart", "static"] + os.environ.get("ABR_EXTRA_NVCC_FLAGS", "").split()


def _nvcc():
    for c in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if c and os.path.exists(c):
            return c
    return None


def _source_hash() -> str:
    h = hashlib.sha256()
    for d in [os.path.join(CSRC, s) for s in SOURCES] + HEADERS:
        with open(d, "rb") as f:
            h.update(f.read())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def is_stale() -> bool:
    """True when the .so is missing or was built from different sources (content hash, not mtimes: the
    snapshot that travels to the GPU box does not preserve a meaningful mtime order)."""
    if os.environ.get("ABR_NO_REBUILD") and os.path.exists(LIB):
        return False          # development only: A/B of libraries built from other revisions of the sources
    if not os.path.exists(LIB) or not os.path.exists(STAMP):
        return True
    try:
        return open(STAMP).read().strip() != _source_hash()
    except OSError:
        return True


def build_library(force: bool = False, verbose: bool = False) -> str:
    """Builds the library under an exclusive file lock: in a one-process-per-GPU launch every rank may find a stale
    library at import; the first one builds (objects and the link go to a private directory, the finished .so is
    moved into place with os.replace, so no process can ever dlopen a half-written file), the others wait on the lock
    and find it fresh."""
    if not force and not is_stale():
        return LIB
    import fcntl
    os.makedirs(os.path.dirname(LIB), exist_ok=True)
    with open(LIB + ".lock", "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        try:
            if not force and not is_stale():      # another process built it while this one waited
                return LIB
            return _build_locked(verbose)
        finally:
            fcntl.flock(lock, fcntl.LOCK_UN)


def _build_locked(verbose: bool) -> str:
    nvcc = _nvcc()
    if nvcc is None:
        raise RuntimeError("nvcc not found: cannot build libabr_b200.so (set NVCC or add nvcc to PATH)")
    # one nvcc per source, in parallel (abr_step.cu alone holds ~50 kernel instantiations), then one link
    from concurrent.futures import ThreadPoolExecutor
    compile_flags = [f for f in NVCC_FLAGS if f != "-shared"]
    obj_dir = os.path.join(os.path.dirname(LIB), "obj" + _SUFFIX, f"build.{os.getpid()}")
    os.makedirs(obj_dir, exist_ok=True)
    tmp_lib = os.path.join(obj_dir, os.path.basename(LIB))

    def compile_one(src):
        obj = os.path.join(obj_dir, os.path.splitext(src)[0] + ".o")
        cmd = [nvcc] + compile_flags + (["-Xptxas", "-v"] if verbose else []) + ["-c", "-o", obj, os.path.join(CSRC, src)]
        return obj, subprocess.run(cmd, capture_output=True, text=True)

    with ThreadPoolExecutor(max_workers=len(SOURCES)) as pool:
        results = list(pool.map(compile_one, SOURCES))
    log = ""
    try:
        for obj, res in results:
            log += res.stdout + res.stderr
            if res.returncode != 0:
                raise RuntimeError("nvcc failed:\n" + res.stdout + res.stderr)
        res = subprocess.run([nvcc] + NVCC_FLAGS + ["-o", tmp_lib] + [obj for obj, _ in results], capture_output=True, text=True)
        if res.returncode != 0:
            raise RuntimeError("nvcc link failed:\n" + res.stdout + res.stderr)
        if verbose:
            print(log + res.stdout + res.stderr)
        if os.path.exists(STAMP):
            os.remove(STAMP)                      # never a fresh stamp next to an old library
        os.replace(tmp_lib, LIB)
        with open(STAMP + f".{os.getpid()}", "w") as f:
            f.write(_source_hash())
        os.replace(STAMP + f".{os.getpid()}", STAMP)
    finally:
        shutil.rmtree(obj_dir, ignore_errors=True)
    return LIB
