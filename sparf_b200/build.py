"""Build the C-ABI shared library (sparf_b200/lib/libsparf_b200.so) with nvcc for sm_100a.

nvcc cross-compiles without a GPU; the .so is git-ignored but travels to the GPU box with the
working tree.  `python -m sparf_b200.build [--force]`.
"""
from __future__ import annotations

import glob
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB_DIR = os.path.join(HERE, "lib")
LIB_PATH = os.path.join(LIB_DIR, "libsparf_b200.so")
INCLUDE = os.path.join(os.path.dirname(HERE), "include")

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC", "-shared",
    "--expt-relaxed-constexpr",
    "-diag-suppress", "177",
]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: cannot build libsparf_b200.so")


def sources():
    return sorted(glob.glob(os.path.join(CSRC, "*.cu")))


HASH_PATH = LIB_PATH + ".srchash"


def _source_hash() -> str:
    """Content hash of everything the library is built from (+ the flags).  File times are useless here: the tree is
    copied to the GPU box, where every file gets a fresh mtime and N ranks would all decide to rebuild at once."""
    import hashlib
    h = hashlib.sha256(" ".join(NVCC_FLAGS).encode())
    for d in sorted(sources() + glob.glob(os.path.join(CSRC, "*.cuh")) + glob.glob(os.path.join(INCLUDE, "*.h"))):
        h.update(os.path.basename(d).encode())
        with open(d, "rb") as f:
            h.update(f.read())
    return h.hexdigest()


def _stale() -> bool:
    if not os.path.exists(LIB_PATH) or os.path.getsize(LIB_PATH) < 4096:
        return True
    try:
        with open(HASH_PATH) as f:
            return f.read().strip() != _source_hash()
    except OSError:
        return True


TRACE_LIB_PATH = os.path.join(LIB_DIR, "libsparf_b200_trace.so")   # debug build (tools/trace_chain.py), never loaded by default


def build(force: bool = False, verbose: bool = False, trace: bool = False) -> str:
    """Compile every .cu under csrc/ into one shared library.  Returns its path.  trace=True builds the wait-time
    tracing variant (-DSPARF_TC_TRACE, plus any extra -D flags in SPARF_NVCC_DEFINES) next to it;
    `SPARF_B200_LIB=<path>` makes sparf_b200._lib load that instead.  The main library takes no defines from the
    environment: it is built from exactly what _source_hash() covers."""
    out_path = TRACE_LIB_PATH if trace else LIB_PATH
    if not trace and not force and not _stale():
        return LIB_PATH
    os.makedirs(LIB_DIR, exist_ok=True)
    # one builder at a time (several ranks of one job may get here together); whoever waited re-checks first
    import fcntl
    lock = open(os.path.join(LIB_DIR, ".build.lock"), "w")
    fcntl.flock(lock, fcntl.LOCK_EX)
    try:
        if not trace and not force and not _stale():
            return LIB_PATH
        return _build_locked(out_path, verbose, trace)
    finally:
        fcntl.flock(lock, fcntl.LOCK_UN)
        lock.close()


def _build_locked(out_path, verbose, trace):
    srcs = sources()
    defines = ["-DSPARF_WITH_TC"] if os.path.exists(os.path.join(CSRC, "mlp_tc.cu")) else []
    if trace:   # debug build: extra defines (e.g. -DSPARF_TC_TRACE_EVENTS) from the environment
        defines += ["-DSPARF_TC_TRACE"] + os.environ.get("SPARF_NVCC_DEFINES", "").split()
    tmp = "%s.tmp.%d" % (out_path, os.getpid())
    cmd = [_nvcc()] + NVCC_FLAGS + defines + ["-I", INCLUDE, "-o", tmp] + srcs
    if verbose:
        cmd.insert(1, "-Xptxas=-v")
        print(" ".join(cmd))
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        sys.stderr.write(res.stdout + res.stderr)
        raise RuntimeError("nvcc failed building libsparf_b200.so")
    if verbose:
        print(res.stdout + res.stderr)
    os.replace(tmp, out_path)
    if not trace:
        with open(HASH_PATH, "w") as f:
            f.write(_source_hash())
    return out_path


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv, trace="--trace" in sys.argv))
