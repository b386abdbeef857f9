"""Build libdfusion.so (hand-written sm_100a CUDA + C ABI) in-tree with nvcc.

No torch extension machinery: the library is a plain C-ABI shared object (include/dfusion.h) that the Python
host side binds with ctypes and a C++ application links directly.
"""
from __future__ import annotations

import os
import subprocess
import sys
from pathlib import Path

HERE = Path(__file__).resolve().parent
ROOT = HERE.parent
CSRC = HERE / "csrc"
LIB = HERE / "libdfusion.so"

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-std=c++17", "-lineinfo",
    # numerics contract: no implicit FMA contraction, IEEE div/sqrt, no FTZ (see df_common.cuh)
    "-fmad=false", "-prec-div=true", "-prec-sqrt=true", "-ftz=false",
    "-Xcompiler", "-fPIC", "-Xcompiler", "-O2",
    "-I", str(ROOT / "include"),
]


def sources() -> list[Path]:
    return sorted(CSRC.glob("*.cu")) + sorted(CSRC.glob("*.cpp"))


def needs_build() -> bool:
    if not LIB.exists():
        return True
    t = LIB.stat().st_mtime
    deps = sources() + sorted(CSRC.glob("*.cuh")) + sorted(CSRC.glob("*.h")) + sorted((ROOT / "include").rglob("*.h*"))
    return any(d.stat().st_mtime > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> Path:
    if not force and not needs_build():
        return LIB
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    objs = []
    objdir = HERE / "build"
    objdir.mkdir(exist_ok=True)
    procs = []
    for src in sources():
        obj = objdir / (src.stem + ".o")
        objs.append(obj)
        cmd = [nvcc, *NVCC_FLAGS, *os.environ.get("DF_NVCC_EXTRA", "").split(), "-x", "cu", "-c", str(src), "-o", str(obj)]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    failed = False
    for src, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0 or verbose:
            sys.stderr.write(f"--- {src.name} ---\n{out}\n")
        failed |= p.returncode != 0
    if failed:
        raise RuntimeError("nvcc failed building libdfusion.so")
    link = [nvcc, "-shared", "-o", str(LIB), *map(str, objs), "-gencode", "arch=compute_100a,code=sm_100a"]
    r = subprocess.run(link, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode != 0:
        raise RuntimeError("link failed:\n" + r.stdout)
    return LIB


MIRROR_LIB = HERE / "libkfusion.so"
MIRROR_SRC = CSRC / "kfusion" / "kfusion_mirror.cpp"
MIRROR_INC = ["-I", str(ROOT / "include"), "-I", str(ROOT / "include" / "cvcompat")]


def build_mirror(force: bool = False) -> Path:
    """libkfusion.so: the C++ mirror of the reference's public classes (include/kfusion) over libdfusion.so"""
    build()
    deps = [MIRROR_SRC, LIB] + sorted((ROOT / "include").rglob("*.h*"))
    if not force and MIRROR_LIB.exists() and all(d.stat().st_mtime <= MIRROR_LIB.stat().st_mtime for d in deps):
        return MIRROR_LIB
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    cmd = [nvcc, "-std=c++17", "-O2", "-Xcompiler", "-fPIC", "-Xcompiler", "-ffp-contract=off", *MIRROR_INC, "-shared", "-o", str(MIRROR_LIB),
           str(MIRROR_SRC), "-L", str(HERE), "-ldfusion", "-Xlinker", "-rpath", "-Xlinker", "$ORIGIN"]
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode != 0:
        raise RuntimeError("building libkfusion.so failed:\n" + r.stdout)
    return MIRROR_LIB


def build_cpp_program(src: Path, out: Path) -> Path:
    """compile + link a C++ program against the mirror (used by tests/test_cpp_mirror.py)"""
    build_mirror()
    out.parent.mkdir(parents=True, exist_ok=True)
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    cmd = [nvcc, "-std=c++17", "-O1", *MIRROR_INC, "-o", str(out), str(src), "-L", str(HERE), "-lkfusion", "-ldfusion",
           "-Xlinker", "-rpath", "-Xlinker", str(HERE)]
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode != 0:
        raise RuntimeError(f"building {src.name} failed:\n" + r.stdout)
    return out


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
    if "--mirror" in sys.argv:
        print(build_mirror(force="--force" in sys.argv))
