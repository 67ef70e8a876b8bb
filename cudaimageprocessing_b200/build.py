"""Builds libgf_b200.so (hand-written CUDA for sm_100a) in-tree with nvcc.

    python -m cudaimageprocessing_b200.build [--force]

The library is the product: C ABI (include/gf_b200.h) + the C++ drop-in shims
(include/guided_filter.h, include/guided_filter_d.h).  nvcc cross-compiles without a GPU.
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

PKG = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(PKG)
CSRC = os.path.join(PKG, "csrc")
LIB = os.path.join(PKG, "libgf_b200.so")

NVCC_FLAGS = [
    "-std=c++17", "-O3", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo",
    "-Xcompiler", "-fPIC", "-shared", "-Xptxas=-v",
]


def _sources():
    return [os.path.join(CSRC, f) for f in sorted(os.listdir(CSRC)) if f.endswith(".cu")]


def _stale() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + \
           [os.path.join(ROOT, "include", f) for f in os.listdir(os.path.join(ROOT, "include"))]
    return any(os.path.getmtime(d) > t for d in deps)


def _compile_and_link(out: str, defines: list[str]) -> tuple[int, str]:
    """Every .cu under csrc/ is one translation unit: compiled to an object file in parallel, then linked."""
    import tempfile
    from concurrent.futures import ThreadPoolExecutor
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        raise RuntimeError("nvcc not found: libgf_b200.so cannot be built (there is no CPU fallback)")
    flags = [f for f in NVCC_FLAGS if f != "-shared"] + ["-I", os.path.join(ROOT, "include"), "-I", CSRC] + list(defines)
    if os.path.exists(os.path.join(CSRC, "gf_fast.cuh")):
        flags.append("-DGF_HAVE_FAST")
    log = []
    with tempfile.TemporaryDirectory(prefix="gfbuild_") as tmp:
        def one(src):
            obj = os.path.join(tmp, os.path.basename(src)[:-3] + ".o")
            res = subprocess.run([nvcc] + flags + ["-c", src, "-o", obj], capture_output=True, text=True)
            return res.returncode, res.stdout + res.stderr, obj
        with ThreadPoolExecutor(max_workers=min(8, os.cpu_count() or 2)) as ex:
            results = list(ex.map(one, _sources()))
        for rc, text, _ in results:
            log.append(text)
            if rc != 0:
                return rc, "".join(log)
        res = subprocess.run([nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", out] + [o for _, _, o in results],
                             capture_output=True, text=True)
        log.append(res.stdout + res.stderr)
        return res.returncode, "".join(log)


def build_variant(name: str, defines: list[str]) -> str:
    """Developer tool: a differently configured build (e.g. -DGF_WS_TIMING) next to the product
    library, for A/B timing through GF_LIB_PATH (bench_tools/ab.py).  Never loaded by default."""
    out = os.path.join(PKG, name)
    rc, text = _compile_and_link(out, defines)
    if rc != 0:
        sys.stderr.write(text)
        raise RuntimeError("nvcc failed building " + name)
    return out


def build(force: bool = False, verbose: bool = False) -> str:
    """Builds the library if it is missing or older than its sources.  Safe when several processes import the package
    at once (one rank per GPU under torchrun): an exclusive file lock serialises the check and the build, the link goes
    to a temporary name and is renamed into place, and whoever gets the lock second finds a fresh library."""
    import fcntl
    if not force and not _stale():
        return LIB
    with open(os.path.join(PKG, ".build.lock"), "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        try:
            if not force and not _stale():
                return LIB
            tmp = LIB + f".tmp{os.getpid()}"
            rc, text = _compile_and_link(tmp, [])
            if verbose or rc != 0:
                sys.stderr.write(text)
            if rc != 0:
                if os.path.exists(tmp):
                    os.remove(tmp)
                raise RuntimeError("nvcc failed building libgf_b200.so")
            os.replace(tmp, LIB)
            with open(os.path.join(PKG, "build_ptxas.log"), "w") as f:
                f.write(text)
        finally:
            fcntl.flock(lock, fcntl.LOCK_UN)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
