"""Builds liblcgs_b200.so (the C-ABI library) in-tree with nvcc for sm_100a.

No torch, no JIT cache: the .so lands next to the sources so that it travels to the GPU box with
the repository snapshot.  Flags that matter:
  -gencode arch=compute_100a,code=sm_100a   B200 only
  --fmad=false                              the arithmetic contract (see csrc/lcgs_math.cuh)
  -lineinfo                                 so ncu's source page maps to our code
"""
from __future__ import annotations

import atexit
import fcntl
import hashlib
import os
import shutil
import subprocess
import sys
import tempfile
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
BUILD = os.path.join(CSRC, "build")
LIB = os.path.join(HERE, "liblcgs_b200.so")
SOURCES = ["capi.cu", "preprocess.cu", "scan.cu", "binning.cu", "sort.cu", "blend.cu", "backward.cu", "ssim.cu"]
HEADERS = ["common.cuh", "frame_plan.cuh", "lcgs_math.cuh", "lcgs_grad.cuh", "lookback.cuh", "blend_walk.cuh", "ssim_math.cuh", os.path.join("..", "..", "include", "lcgs_b200.h")]

NVCC = os.environ.get("LCGS_NVCC", "/usr/local/cuda/bin/nvcc")
NVCC_FLAGS = [
    "-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "--fmad=false",
    "-Xcompiler", "-fPIC,-fvisibility=hidden,-ffp-contract=off", "-Xptxas", "-v", "-ccbin", "g++",
]


STAMP = LIB + ".stamp"  # digest of the sources the shipped .so was built from (travels with it to the GPU box)
# -DLCGS_TUNING build (kernel geometries selectable by environment variable, extra sweep variants): a SEPARATE library
# that only scripts/tune_*.py load (LCGS_TUNING=1); the production library has none of it.
TUNING_LIB = os.path.join(HERE, "liblcgs_b200_tuning.so")


def _mtime(path: str) -> float:
    return os.path.getmtime(path) if os.path.exists(path) else 0.0


def _source_digest() -> str:
    h = hashlib.sha256(" ".join(NVCC_FLAGS).encode())
    for f in SOURCES + HEADERS:
        with open(os.path.join(CSRC, f), "rb") as fh:
            h.update(f.encode() + b"\0" + fh.read())
    return h.hexdigest()


def is_stale() -> bool:
    """Content-based (file times do not survive the copy to another box): the .so is stale iff it is missing
    or its stamp does not match the digest of the sources + flags."""
    if not os.path.exists(LIB) or not os.path.exists(STAMP):
        return True
    with open(STAMP) as fh:
        return fh.read().strip() != _source_digest()


def build_native(force: bool = False, verbose: bool = False) -> str:
    if not force and not is_stale():
        return LIB
    if not os.path.exists(NVCC):
        raise RuntimeError("nvcc not found at %s and %s is missing or stale" % (NVCC, LIB))
    os.makedirs(BUILD, exist_ok=True)
    # several ranks of one job may get here together: one builds, the others wait and find a fresh library
    with open(LIB + ".lock", "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        try:
            if not force and not is_stale():
                return LIB
            return _build_native_locked(verbose)
        finally:
            fcntl.flock(lock, fcntl.LOCK_UN)


def build_tuning(verbose: bool = False) -> str:
    """Always rebuilds liblcgs_b200_tuning.so (-DLCGS_TUNING)."""
    os.makedirs(BUILD, exist_ok=True)
    return _build_native_locked(verbose, tuning=True)


def _build_native_locked(verbose: bool, tuning: bool = False) -> str:
    log_path = os.path.join(BUILD, "ptxas_tuning.log" if tuning else "ptxas.log")
    out_lib = TUNING_LIB if tuning else LIB
    extra = ["-DLCGS_TUNING"] if tuning else []

    def compile_one(src: str):
        obj = os.path.join(BUILD, src.replace(".cu", ".tuning.o" if tuning else ".o"))
        cmd = [NVCC, *NVCC_FLAGS, *extra, "-c", os.path.join(CSRC, src), "-o", obj]
        r = subprocess.run(cmd, capture_output=True, text=True)
        return src, obj, r

    with ThreadPoolExecutor(max_workers=len(SOURCES)) as ex:
        results = list(ex.map(compile_one, SOURCES))
    with open(log_path, "w") as log:
        for src, _, r in results:
            log.write("==== %s ====\n%s\n%s\n" % (src, r.stdout, r.stderr))
    for src, _, r in results:
        if r.returncode != 0:
            sys.stderr.write(r.stdout + r.stderr)
            raise RuntimeError("nvcc failed on %s" % src)
        if verbose:
            sys.stderr.write(r.stderr)
    objs = [o for _, o, _ in results]
    tmp = "%s.tmp.%d" % (out_lib, os.getpid())  # link aside, then rename: nobody ever maps a half-written library
    link = [NVCC, "-shared", "-o", tmp, *objs, "-gencode", "arch=compute_100a,code=sm_100a", "-ccbin", "g++"]
    r = subprocess.run(link, capture_output=True, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout + r.stderr)
        raise RuntimeError("link failed")
    os.replace(tmp, out_lib)
    if tuning:
        return out_lib
    with open(STAMP + ".tmp", "w") as fh:
        fh.write(_source_digest() + "\n")
    os.replace(STAMP + ".tmp", STAMP)
    return LIB


APP_DIR = os.path.join(HERE, "cpp", "app")
APP_BIN = os.path.join(HERE, "lcgs-app")
APP_SOURCES = [os.path.join(APP_DIR, "main.cpp"), os.path.join(APP_DIR, "gaussians.cpp")]
APP_INCLUDES = [os.path.join(HERE, "cpp", "include"), os.path.join(HERE, "..", "include"), APP_DIR,
                "/usr/local/cuda/include"]


def _app_deps():
    deps = list(APP_SOURCES)
    for root, _, files in os.walk(os.path.join(HERE, "cpp")):
        deps += [os.path.join(root, f) for f in files if f.endswith((".h", ".hpp"))]
    return deps


def build_app(force: bool = False) -> str:
    """lcgs-app: the C++ CLI (cpp/app) over the C++ facade (cpp/include) and liblcgs_b200.so."""
    lib = build_native()
    newest = max([_mtime(f) for f in _app_deps()] + [_mtime(lib)])
    if not force and _mtime(APP_BIN) >= newest:
        return APP_BIN
    cmd = ["g++", "-O2", "-std=c++20", "-Wall", "-Wextra", "-Wno-missing-field-initializers"]
    for inc in APP_INCLUDES:
        cmd += ["-I", inc]
    cmd += APP_SOURCES + ["-o", APP_BIN, "-L", HERE, "-llcgs_b200", "-Wl,-rpath,$ORIGIN", "-L/usr/local/cuda/lib64",
                          "-lcudart_static", "-lz", "-ldl", "-lrt", "-lpthread"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout + r.stderr)
        raise RuntimeError("building lcgs-app failed")
    return APP_BIN


FACADE_TEST_SRC = os.path.join(HERE, "..", "tests", "facade", "test_facade.cpp")
FACADE_TEST_BIN = os.path.join(HERE, "..", "tests", "facade", "test_facade")


_facade_tmp = None  # private directory of a facade test built outside a read-only tree


def build_facade_test(force: bool = False) -> str:
    """tests/facade/test_facade: the reference's GSTileSplatter::forward call sequence and a 16-byte-float3 camera
    compiled against the C++ facade (checks that the facade keeps the reference's argument lists).  In a tree the
    tests cannot write to, a stale or missing binary is built into a private temporary directory instead, removed when
    Python exits."""
    global _facade_tmp
    lib = build_native()
    newest = max([_mtime(f) for f in _app_deps()] + [_mtime(lib), _mtime(FACADE_TEST_SRC)])
    out = FACADE_TEST_BIN
    if not force and _mtime(out) >= newest:
        return out
    if not os.access(os.path.dirname(out), os.W_OK) or (os.path.exists(out) and not os.access(out, os.W_OK)):
        if _facade_tmp is None:
            _facade_tmp = tempfile.mkdtemp(prefix="lcgs_b200_facade_")
            atexit.register(shutil.rmtree, _facade_tmp, True)
        out = os.path.join(_facade_tmp, "test_facade")
        if not force and _mtime(out) >= newest:
            return out
    cmd = ["g++", "-O1", "-std=c++20", "-Wall", "-Wextra", "-Wno-missing-field-initializers"]
    for inc in APP_INCLUDES:
        cmd += ["-I", inc]
    cmd += [FACADE_TEST_SRC, os.path.join(APP_DIR, "gaussians.cpp"), "-o", out, "-L", HERE, "-llcgs_b200",
            "-Wl,-rpath," + HERE, "-L/usr/local/cuda/lib64", "-lcudart_static", "-ldl", "-lrt", "-lpthread"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        sys.stderr.write(r.stdout + r.stderr)
        raise RuntimeError("building tests/facade/test_facade failed")
    return out


if __name__ == "__main__":
    if "--tuning" in sys.argv:
        print(build_tuning(verbose=True))
        sys.exit(0)
    print(build_native(force="--force" in sys.argv, verbose=True))
    print(build_app(force="--force" in sys.argv))
