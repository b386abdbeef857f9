"""ctypes/numpy binding of the CPU mesh oracle (oracle/orc_mesh.c -> oracle/liborc_mesh.so).  TEST INFRASTRUCTURE ONLY, like orc.py.
The library is built on its own, with liborc.so's compiler flags, from orc_mesh.c and orc_tsdf.c (half conversion); it reuses orc.py's
ctypes structures."""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from pathlib import Path

import numpy as np

from . import orc

HERE = Path(__file__).resolve().parent
LIB = HERE / "liborc_mesh.so"
SRCS = [HERE / "orc_mesh.c", HERE / "orc_tsdf.c"]
DEPS = SRCS + [HERE / "orc_common.h", HERE.parent / "dynamicfusion_b200" / "csrc" / "mc_table.h", Path(__file__)]
CFLAGS = ["-std=gnu11", "-O2", "-fPIC", "-ffp-contract=off", "-fno-fast-math", "-fopenmp", "-march=x86-64-v3", "-Wall", "-Wextra",
          "-Wno-unused-parameter"]
_lib = None


def build(force: bool = False) -> Path:
    if force or not LIB.exists() or any(s.stat().st_mtime > LIB.stat().st_mtime for s in DEPS):
        cc = "/usr/bin/gcc" if os.access("/usr/bin/gcc", os.X_OK) else "gcc"
        tmp = LIB.with_suffix(f".{os.getpid()}.tmp")
        subprocess.run([cc, *CFLAGS, "-shared", "-o", str(tmp), *map(str, SRCS), "-lm"], check=True, stdout=subprocess.PIPE,
                       stderr=subprocess.STDOUT)
        os.replace(tmp, LIB)
    return LIB


def load() -> C.CDLL:
    global _lib
    if _lib is None:
        _lib = C.CDLL(str(build()))
    return _lib


def extract_mesh(vol_data, dims, vs, trunc, mw, pose, vcap=None, tcap=None):
    """orc_extract_mesh: returns (vertices [n, 4] float32, edge keys [n] uint32, triangles [m, 3] int32, (true vertex count, true
    triangle count)); n = min(count, vcap), m = min(count, tcap) and 0 when the vertices overflow.  Capacities default to whatever the
    mesh needs."""
    vol = orc.volume(vol_data, dims, vs, trunc, mw)
    counts = (C.c_longlong * 2)()
    if vcap is None or tcap is None:
        load().orc_extract_mesh(vol, orc.aff(*pose), None, None, C.c_longlong(0), None, C.c_longlong(0), counts)
        vcap = counts[0] if vcap is None else vcap
        tcap = counts[1] if tcap is None else tcap
    verts = np.zeros((max(vcap, 1), 4), np.float32)
    keys = np.zeros(max(vcap, 1), np.uint32)
    tris = np.zeros((max(tcap, 1), 3), np.int32)
    load().orc_extract_mesh(vol, orc.aff(*pose), orc._p(verts), orc._p(keys), C.c_longlong(vcap), orc._p(tris), C.c_longlong(tcap), counts)
    nv, nt = int(counts[0]), int(counts[1])
    n = min(nv, vcap)
    m = min(nt, tcap) if nv <= vcap else 0
    return verts[:n].copy(), keys[:n].copy(), tris[:m].copy(), (nv, nt)
