"""In-tree build of libilsm_cuda.so (sm_100a only).  nvcc cross-compiles without a GPU; the resulting .so is
git-ignored but travels to the GPU box with the repository snapshot."""
from __future__ import annotations

import os
import shutil
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libilsm_cuda.so")

NVCC_FLAGS = [
    "-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo",
    "-Xcompiler", "-fPIC,-fvisibility=hidden,-ffp-contract=off",
]
# Host code is never contracted either (-ffp-contract=off): fp64 rules a caller restates bit for bit, like the full loop's
# keyframe rule (csrc/ilsm_keyframe.hpp), must not depend on whether the host ISA has FMA (x86-64 baseline has none,
# AArch64 has it and GCC contracts there by default).
# Parity with the reference's x86-64 SSE2 build (CMakeLists.txt:5-6, no FMA): files whose float results are compared
# bit for bit are compiled without a*b+c contraction.  registration.cu keeps its bit-exact parts (pose transform,
# float distances) in explicit round-to-nearest intrinsics and is compared with a tolerance elsewhere (fits, residuals,
# LM), so its fp64 arithmetic may use DFMA.
FMAD = {"registration.cu": "true"}
OBJ = os.path.join(HERE, "build")


def sources():
    return sorted(os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith(".cu"))


STAMP = LIB + ".stamp"
LOCK = os.path.join(HERE, ".build.lock")


def _fingerprint(extra_flags=()):
    """Content hash of every source, header and flag that goes into the library.  mtimes are useless here: the tree is
    copied to the GPU box (fresh mtimes in arbitrary order), and a stale verdict there would make every rank of a
    multi-GPU launch rebuild the library at the same time."""
    import hashlib
    h = hashlib.sha256()
    deps = sorted(os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cu", ".cuh", ".hpp", ".h")))
    deps.append(os.path.join(HERE, "..", "include", "ilsm.h"))
    for d in deps:
        h.update(os.path.basename(d).encode())
        with open(d, "rb") as fh:
            h.update(fh.read())
    h.update(repr((NVCC_FLAGS, sorted(FMAD.items()), list(extra_flags))).encode())
    return h.hexdigest()


def _stale(lib=LIB, extra_flags=()):
    if not os.path.exists(lib) or not os.path.exists(lib + ".stamp"):
        return True
    try:
        return open(lib + ".stamp").read().strip() != _fingerprint(extra_flags)
    except OSError:
        return True


def nvcc_path():
    return shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"


def build(force: bool = False, verbose: bool = False, extra_flags=(), lib: str = LIB, obj_dir: str = OBJ) -> str:
    """One nvcc -c per source (in parallel), then one link into libilsm_cuda.so (or `lib`, for instrumented variants).
    Serialised across processes with a file lock: the ranks of a torchrun launch all call this."""
    if not force and not _stale(lib, extra_flags):
        return lib
    import fcntl
    with open(LOCK, "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        try:
            if not force and not _stale(lib, extra_flags):  # another process built it while we waited
                return lib
            return _build_locked(verbose, extra_flags, lib, obj_dir)
        finally:
            fcntl.flock(lock, fcntl.LOCK_UN)


def _build_locked(verbose, extra_flags, lib, obj_dir):
    os.makedirs(obj_dir, exist_ok=True)
    procs = []
    for src in sources():
        name = os.path.basename(src)
        obj = os.path.join(obj_dir, name[:-3] + ".o")
        cmd = ([nvcc_path()] + NVCC_FLAGS + list(extra_flags) + ["-fmad=" + FMAD.get(name, "false")] +
               (["-Xptxas", "-v"] if verbose else []) + ["-c", src, "-o", obj])
        procs.append((name, obj, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    objs = []
    for name, obj, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0:
            raise RuntimeError(f"nvcc failed on {name}:\n{out}")
        if verbose:
            print(out)
        objs.append(obj)
    tmp = lib + f".tmp{os.getpid()}"
    r = subprocess.run([nvcc_path(), "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", tmp] + objs,
                       capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("link failed:\n" + r.stdout + r.stderr)
    os.replace(tmp, lib)  # atomic: a concurrent dlopen never sees a half-written library
    with open(lib + ".stamp", "w") as fh:
        fh.write(_fingerprint(extra_flags))
    return lib
