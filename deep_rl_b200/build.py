"""Builds deep_rl_b200/lib/libdrl_b200.so (sm_100a only) in-tree with nvcc.

    python -m deep_rl_b200.build [--force] [--verbose]

The .so is git-ignored but travels to the GPU box with the repo snapshot.
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

PKG = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(PKG, "csrc")
LIBDIR = os.path.join(PKG, "lib")
OBJDIR = os.path.join(PKG, "build")
SO = os.path.join(LIBDIR, "libdrl_b200.so")

SOURCES = ["abi_misc.cu", "env_ops.cu", "policy_ops.cu", "rollout.cu", "rollout_tc.cu", "gae_ops.cu", "update_ops.cu", "update_tc.cu", "umma_selftest.cu", "update256.cu", "rollout256.cu", "replay_ops.cu", "reinforce_ops.cu"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17", "-fmad=false",
    "-Xcompiler", "-fPIC", "-Xptxas", "-v", "--expt-relaxed-constexpr",
]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: libdrl_b200.so cannot be built")


def _newest_source_mtime() -> float:
    files = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(os.path.dirname(PKG), "include", "drl_b200.h")]
    return max(os.path.getmtime(f) for f in files)


def is_stale() -> bool:
    return not os.path.exists(SO) or os.path.getmtime(SO) < _newest_source_mtime()


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not is_stale():
        return SO
    nvcc = _nvcc()
    os.makedirs(LIBDIR, exist_ok=True)
    os.makedirs(OBJDIR, exist_ok=True)

    def compile_one(src: str):
        obj = os.path.join(OBJDIR, src.replace(".cu", ".o"))
        extra = os.environ.get("DRL_EXTRA_NVCC_FLAGS", "").split()     # e.g. -DDRL_ROLLOUT_STAMPS for profiles/tools/ro_stamps.py
        cmd = [nvcc, *NVCC_FLAGS, *extra, "-c", os.path.join(CSRC, src), "-o", obj]
        res = subprocess.run(cmd, capture_output=True, text=True)
        return src, obj, res

    with ThreadPoolExecutor(max_workers=len(SOURCES)) as ex:
        results = list(ex.map(compile_one, SOURCES))
    log = []
    for src, obj, res in results:
        log.append(f"==== {src} ====\n{res.stderr}")
        if res.returncode != 0:
            sys.stderr.write("\n".join(log))
            raise RuntimeError(f"nvcc failed on {src}")
    with open(os.path.join(OBJDIR, "ptxas.log"), "w") as f:
        f.write("\n".join(log))
    if verbose:
        print("\n".join(log))
    tmp = SO + f".tmp{os.getpid()}"       # link to a private name, then rename: a concurrent dlopen never sees a partial file
    link = [nvcc, "-shared", "-o", tmp, *[obj for _, obj, _ in results], "-gencode", "arch=compute_100a,code=sm_100a"]
    res = subprocess.run(link, capture_output=True, text=True)
    if res.returncode != 0:
        sys.stderr.write(res.stderr)
        raise RuntimeError("nvcc link failed")
    os.replace(tmp, SO)
    return SO


def build_locked() -> str:
    """What the import path calls: returns the library path, rebuilding first if it is missing or stale.  The check and the
    build run under an exclusive file lock (all ranks of a torchrun job import at once).  A stale library without a
    compiler at hand (a stripped deployment may not have one) is used as it is.  An up-to-date library is returned without
    opening the lock file, so that a read-only installation imports."""
    import fcntl
    if not is_stale():
        return SO
    os.makedirs(LIBDIR, exist_ok=True)
    with open(os.path.join(LIBDIR, ".build.lock"), "w") as lk:
        fcntl.flock(lk, fcntl.LOCK_EX)
        try:
            if is_stale():
                try:
                    _nvcc()
                except RuntimeError:
                    if os.path.exists(SO):
                        return SO
                    raise
                build()
        finally:
            fcntl.flock(lk, fcntl.LOCK_UN)
    return SO


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
