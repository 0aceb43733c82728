"""In-tree build of librayhs_b200.so (sm_100a CUDA + C++ front end), the oracle and the CLI.

    python -m rayhs_b200.build            # build everything that is out of date
    python -m rayhs_b200.build --force

The product library never links or loads anything under oracle/; the oracle is built here
only because tests/, smoke() and bench.py's CPU-baseline legs need the checker.
"""
from __future__ import annotations

import hashlib
import os
import shutil
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "rayhs_b200", "csrc")
OBJ = os.path.join(ROOT, "build", "obj")
LIB = os.path.join(ROOT, "rayhs_b200", "librayhs_b200.so")
CLI = os.path.join(ROOT, "rayhs_b200", "rayhs")
ORACLE_SRC = os.path.join(ROOT, "oracle", "oracle.cpp")
ORACLE_LIB_SRC = os.path.join(ROOT, "oracle", "batch.cpp")  # includes ORACLE_SRC
ORACLE_LIB = os.path.join(ROOT, "oracle", "_build", "liborc.so")

NVCC = os.environ.get("NVCC") or shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
CXX = os.environ.get("CXX") or "g++"

# -fmad=false: the reference (GHC) never fuses a multiply with an add; the kernels keep its
# operation order so that t, u, v, hit points and colours are bit-identical to the oracle's.
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-std=c++17", "-O3", "-lineinfo", "-fmad=false",
    "-Xcompiler", "-fPIC,-ffp-contract=off", "-Xptxas", "-v",
]
CXX_FLAGS = ["-std=c++17", "-O2", "-fPIC", "-ffp-contract=off", "-Wall", "-Wno-unused-function"]

CUDA_SOURCES = ["kernels.cu", "runtime.cu", "setup_kernels.cu"]
CXX_SOURCES = ["frontend.cpp", "host_build.cpp", "light_maps.cpp"]
HEADERS = [os.path.join(CSRC, h) for h in ("device_types.cuh", "common.h", "light_geom.h", "render_plan.h", "scene_update.h")] + [os.path.join(ROOT, "include", "rayhs_b200.h")]


def _digest(deps: list[str], flags: list[str]) -> str:
    h = hashlib.sha256(" ".join(flags).encode())
    for d in deps:
        if os.path.exists(d):
            with open(d, "rb") as f:
                h.update(f.read())
    return h.hexdigest()


def _stale(target: str, deps: list[str], flags: list[str]) -> bool:
    """Content-based: the target's .stamp holds the digest of the sources and flags it was built from
    (mtimes do not survive the copy to the GPU box; the stamp travels with the .so)."""
    if not os.path.exists(target) or not os.path.exists(target + ".stamp"):
        return True
    with open(target + ".stamp") as f:
        return f.read().strip() != _digest(deps, flags)


def _stamp(target: str, deps: list[str], flags: list[str]) -> None:
    with open(target + ".stamp", "w") as f:
        f.write(_digest(deps, flags))


def _run(cmd: list[str], log: str | None = None) -> None:
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if log:
        with open(log, "w") as f:
            f.write(" ".join(cmd) + "\n" + r.stdout)
    if r.returncode != 0:
        sys.stderr.write(r.stdout)
        raise RuntimeError("build step failed: " + " ".join(cmd))


def build_library(force: bool = False) -> str:
    all_src = [os.path.join(CSRC, s) for s in CUDA_SOURCES + CXX_SOURCES] + HEADERS
    all_flags = NVCC_FLAGS + CXX_FLAGS
    if not force and not _stale(LIB, all_src, all_flags):
        return LIB
    os.makedirs(OBJ, exist_ok=True)
    objs = []
    for src in CUDA_SOURCES:
        s, o = os.path.join(CSRC, src), os.path.join(OBJ, src + ".o")
        if force or _stale(o, [s] + HEADERS, NVCC_FLAGS):
            _run([NVCC, *NVCC_FLAGS, "-c", s, "-o", o], log=os.path.join(OBJ, src + ".ptxas.log"))
            _stamp(o, [s] + HEADERS, NVCC_FLAGS)
        objs.append(o)
    for src in CXX_SOURCES:
        s, o = os.path.join(CSRC, src), os.path.join(OBJ, src + ".o")
        if force or _stale(o, [s] + HEADERS, CXX_FLAGS):
            _run([CXX, *CXX_FLAGS, "-c", s, "-o", o])
            _stamp(o, [s] + HEADERS, CXX_FLAGS)
        objs.append(o)
    _run([NVCC, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", LIB, *objs, "-lpthread", "-ldl"])
    _stamp(LIB, all_src, all_flags)
    return LIB


def build_cli(force: bool = False) -> str:
    src = os.path.join(CSRC, "rayhs_main.cpp")
    if os.path.exists(src) and (force or _stale(CLI, [src] + HEADERS, CXX_FLAGS)):
        _run([CXX, *CXX_FLAGS, src, "-o", CLI, "-L" + os.path.dirname(LIB), "-lrayhs_b200", "-Wl,-rpath,$ORIGIN"])
        _stamp(CLI, [src] + HEADERS, CXX_FLAGS)
    return CLI


def build_oracle(force: bool = False) -> str:
    os.makedirs(os.path.dirname(ORACLE_LIB), exist_ok=True)
    flags = ["-std=c++17", "-O2", "-ffp-contract=off", "-fPIC", "-shared"]
    deps = [ORACLE_LIB_SRC, ORACLE_SRC, HEADERS[-1]]
    if force or _stale(ORACLE_LIB, deps, flags):
        _run([CXX, *flags, ORACLE_LIB_SRC, "-o", ORACLE_LIB, "-lpthread"])
        _stamp(ORACLE_LIB, deps, flags)
    return ORACLE_LIB


def build_oracle_ref() -> None:
    """oracle/_ref would hold the reference's own implementation compiled from /root/reference.  The
    reference is pure Haskell (22 .hs files, no C sources) and GHC is not in this image, so there is
    nothing to build; the oracle stays a restatement ("port")."""
    return None


def build_all(force: bool = False) -> None:
    build_library(force)
    build_cli(force)
    build_oracle(force)


if __name__ == "__main__":
    build_all("--force" in sys.argv)
    print(LIB)
