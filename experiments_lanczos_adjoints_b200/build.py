"""Build libb200lanczos.so (sm_100a) in-tree with nvcc.  No torch, no JIT cache:
the .so lives next to the sources so it travels with the repo snapshot.
Each .cu is compiled to an object (in parallel, cached by content hash), then linked."""

from __future__ import annotations

import concurrent.futures
import hashlib
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(HERE, "build")
LIB = os.path.join(HERE, "libb200lanczos.so")
STAMP = LIB + ".stamp"

NVCC_FLAGS = [
    "-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo",
    "-Xcompiler", "-fPIC", "-Xcompiler", "-O3", "--expt-relaxed-constexpr",
]  # fmt: skip
NVCC_FLAGS += os.environ.get("BL_NVCC_EXTRA", "").split()  # e.g. -DBL_STEP_DEBUG (debug builds; part of the stamp)


def sources():
    return sorted(os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith(".cu"))


def _headers_digest():
    h = hashlib.sha256()
    inc = os.path.join(HERE, "..", "include", "b200_lanczos.h")
    for path in sorted(os.listdir(CSRC)):
        if path.endswith((".cuh", ".h")):
            with open(os.path.join(CSRC, path), "rb") as f:
                h.update(path.encode() + f.read())
    with open(inc, "rb") as f:
        h.update(f.read())
    h.update(" ".join(NVCC_FLAGS).encode())
    return h.hexdigest()


def _file_digest(path, headers):
    h = hashlib.sha256(headers.encode())
    with open(path, "rb") as f:
        h.update(f.read())
    return h.hexdigest()


def find_nvcc():
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    return None


def _compile(nvcc, src, obj, verbose):
    cmd = [nvcc, *NVCC_FLAGS, "-c", src, "-o", obj]
    if verbose:
        cmd.insert(1, "-Xptxas=-v")
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError(f"nvcc failed on {os.path.basename(src)}:\n" + res.stdout + res.stderr)
    return res.stderr


def build(force: bool = False, verbose: bool = False) -> str:
    """Build (or reuse) the library.  Safe when several ranks import the package at once: an exclusive
    file lock serialises the builders and the late-comers find the finished library.  A library that is
    up to date is returned without writing to the tree, so a built tree may be read-only."""
    import fcntl

    if not force and _is_current(_digests()[1]):
        return LIB
    os.makedirs(OBJ, exist_ok=True)
    with open(os.path.join(OBJ, ".lock"), "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        try:
            return _build_locked(force, verbose)
        finally:
            fcntl.flock(lock, fcntl.LOCK_UN)


def _digests():
    """Per-source digests and the library's digest over all of them (what STAMP records)."""
    headers = _headers_digest()
    digests = {src: _file_digest(src, headers) for src in sources()}
    return digests, hashlib.sha256("".join(digests[s] for s in sorted(digests)).encode()).hexdigest()


def _is_current(total: str) -> bool:
    if not (os.path.exists(LIB) and os.path.exists(STAMP)):
        return False
    with open(STAMP) as f:
        return f.read().strip() == total


def _build_locked(force: bool, verbose: bool) -> str:
    digests, total = _digests()
    if not force and _is_current(total):
        return LIB
    nvcc = find_nvcc()
    if nvcc is None:
        if os.path.exists(LIB):
            return LIB  # prebuilt library shipped with the snapshot
        raise RuntimeError("nvcc not found and no prebuilt libb200lanczos.so present")
    os.makedirs(OBJ, exist_ok=True)
    jobs, objs = [], []
    with concurrent.futures.ThreadPoolExecutor(max_workers=os.cpu_count() or 4) as pool:
        for src, dig in digests.items():
            obj = os.path.join(OBJ, os.path.basename(src)[:-3] + "." + dig[:16] + ".o")
            objs.append(obj)
            if force or verbose or not os.path.exists(obj):
                jobs.append(pool.submit(_compile, nvcc, src, obj, verbose))
        for j in jobs:
            log = j.result()
            if verbose:
                print(log, file=sys.stderr)
    res = subprocess.run([nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", LIB, *objs, "-ldl"],
                         capture_output=True, text=True)  # fmt: skip
    if res.returncode != 0:
        raise RuntimeError("link failed:\n" + res.stdout + res.stderr)
    keep = set(objs)
    for f in os.listdir(OBJ):  # drop objects of older source versions
        if f.endswith(".o") and os.path.join(OBJ, f) not in keep:
            try:
                os.remove(os.path.join(OBJ, f))
            except FileNotFoundError:
                pass
    with open(STAMP, "w") as f:
        f.write(total)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
