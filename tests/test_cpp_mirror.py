"""The C++ mirror of the reference's public API (include/kfusion/*.hpp + libkfusion.so): a demo.cpp-like program
(tests/cpp/demo_like.cpp) must compile and link against it on the CPU box, and run green on the GPU."""
import json
import os
import struct
import subprocess
import zlib
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parents[1]
EXE = ROOT / "tests" / "cpp" / "_build" / "demo_like"


def _build():
    from dynamicfusion_b200 import build
    return build.build_cpp_program(ROOT / "tests" / "cpp" / "demo_like.cpp", EXE)


def test_demo_like_program_compiles_and_links():
    exe = _build()
    assert exe.exists()
    # the mirror library exports the reference's class symbols
    out = subprocess.run(["nm", "-DC", str(ROOT / "dynamicfusion_b200" / "libkfusion.so")], capture_output=True, text=True).stdout
    for sym in ("kfusion::KinFu::operator()", "kfusion::KinFuParams::default_params_dynamicfusion", "kfusion::WarpField::warp",
                "kfusion::cuda::TsdfVolume::integrate", "kfusion::cuda::ProjectiveICP::estimateTransform", "kfusion::cuda::computeDists",
                "kfusion::WarpFieldOptimiser::optimiseWarpData", "kfusion::cuda::DeviceMemory2D::upload"):
        assert sym in out, sym


@pytest.mark.gpu
def test_demo_like_program_runs():
    exe = _build()
    r = subprocess.run([str(exe)], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "all checks passed" in r.stdout


# ---------------------------------------------------------------------------------------------------------------------------------
# PNG input of the headless OpenCV stand-ins (include/cvcompat)
def write_png(path, arr):
    """8-bit RGB (H, W, 3) or 16-bit grey (H, W) PNG, filter type 0, one IDAT"""
    h, w = arr.shape[:2]
    if arr.dtype == np.uint16:
        ctype, depth, data, stride = 0, 16, arr.astype(">u2").tobytes(), w * 2
    else:
        ctype, depth, data, stride = 2, 8, np.ascontiguousarray(arr, np.uint8).tobytes(), w * 3
    raw = b"".join(b"\x00" + data[y * stride:(y + 1) * stride] for y in range(h))

    def chunk(t, d):
        return struct.pack(">I", len(d)) + t + d + struct.pack(">I", zlib.crc32(t + d) & 0xffffffff)
    Path(path).write_bytes(b"\x89PNG\r\n\x1a\n" + chunk(b"IHDR", struct.pack(">IIBBBBB", w, h, depth, ctype, 0, 0, 0))
                           + chunk(b"IDAT", zlib.compress(raw, 1)) + chunk(b"IEND", b""))


def test_headless_imread_reads_depth_and_colour_pngs(tmp_path):
    from dynamicfusion_b200 import build
    rng = np.random.default_rng(5)
    depth = rng.integers(0, 6000, (48, 64), dtype=np.uint16)
    color = rng.integers(0, 256, (48, 64, 3), dtype=np.uint8)
    (tmp_path / "depth").mkdir()
    write_png(tmp_path / "depth" / "000.png", depth)
    write_png(tmp_path / "c.png", color)
    exe = tmp_path / "imread_check"
    cmd = ["/usr/bin/g++" if Path("/usr/bin/g++").exists() else "g++", "-std=c++17", "-O1", *build.MIRROR_INC, "-o", str(exe),
           str(ROOT / "tests" / "cpp" / "imread_check.cpp"), "-lz"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    out = subprocess.run([str(exe), str(tmp_path / "depth"), str(tmp_path / "c.png")], capture_output=True, text=True)
    assert out.returncode == 0, out.stderr
    v = [int(x) for x in out.stdout.split()]
    disp = np.clip(np.floor(depth.astype(np.float64) * (255.0 / 4000) + 0.5), 0, 255)
    assert v == [48, 64, 2, int(depth.sum(dtype=np.uint64)), 48, 64, 16, int(color[..., 2].sum()), int(color[..., 1].sum()), int(color[..., 0].sum()),
                 int(disp.sum()), 1]


def test_mirror_exports_every_symbol_the_reference_demo_imports():
    """the reference's own apps/demo.cpp, built unchanged against include/kfusion + the headless OpenCV stand-ins (include/cvcompat),
    imports these symbols (tests/golden/ref_demo_imports.json): the mirror library must define every one of them"""
    from dynamicfusion_b200 import build
    lib = build.build_mirror()
    mirror = subprocess.run(["readelf", "-d", str(lib)], capture_output=True, text=True).stdout
    assert "libdfusion.so" in mirror                          # the mirror binds to the C ABI
    defined = set(subprocess.run(["nm", "-D", "--defined-only", str(lib)], capture_output=True, text=True).stdout.split())
    wanted = json.loads((ROOT / "tests" / "golden" / "ref_demo_imports.json").read_text())["symbols"]
    assert len(wanted) >= 15 and [s for s in wanted if s not in defined] == []


# ---------------------------------------------------------------------------------------------------------------------------------
# PLY export of the canonical cloud (SURVEY 8f(4)): the header-only C++ writer and its Python twin produce the same bytes
def _read_ply(path):
    raw = Path(path).read_bytes()
    head, body = raw.split(b"end_header\n", 1)
    lines = head.decode().splitlines()
    n = int([l for l in lines if l.startswith("element vertex")][0].split()[-1])
    props = [l.split()[-1] for l in lines if l.startswith("property float")]
    return np.frombuffer(body, "<f4").reshape(n, len(props)), props


def test_ply_export_cpp_and_python_agree(tmp_path):
    from dynamicfusion_b200 import build
    exe = tmp_path / "ply_check"
    cmd = ["/usr/bin/g++" if Path("/usr/bin/g++").exists() else "g++", "-std=c++17", "-O1", *build.MIRROR_INC, "-o", str(exe),
           str(ROOT / "tests" / "cpp" / "ply_check.cpp")]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    out = subprocess.run([str(exe), str(tmp_path)], capture_output=True, text=True)
    assert out.returncode == 0 and out.stdout.split() == ["6", "6", "-1"], out.stdout + out.stderr
    data, props = _read_ply(tmp_path / "with_normals.ply")
    assert props == ["x", "y", "z", "nx", "ny", "nz"] and data.shape == (6, 6)
    idx = np.array([0, 1, 2, 4, 5, 6], np.float32)
    assert np.array_equal(data[:, 0], 0.5 * idx) and np.array_equal(data[:, 1], -idx) and np.array_equal(data[:, 2], 2 + idx)
    assert np.array_equal(data[:, 5], [1, 1, 1, 1, 0, 1])                       # the NaN normal became 0 0 0
    pts_only, props2 = _read_ply(tmp_path / "points_only.ply")
    assert props2 == ["x", "y", "z"] and np.array_equal(pts_only, data[:, :3])
    # the Python twin writes the same file byte for byte
    pytest.importorskip("torch")
    from dynamicfusion_b200 import host
    cloud = np.zeros((7, 4), np.float32)
    cloud[:, 0], cloud[:, 1], cloud[:, 2] = 0.5 * np.arange(7), np.float32(-1.0) * np.arange(7, dtype=np.float32), 2 + np.arange(7)   # -1.f * 0 = -0.f
    cloud[3, 0] = np.nan
    nrm = np.zeros((7, 4), np.float32)
    nrm[:, 2] = 1
    nrm[5, 1] = np.nan
    assert host.save_ply(tmp_path / "py.ply", cloud, nrm) == 6
    assert (tmp_path / "py.ply").read_bytes() == (tmp_path / "with_normals.ply").read_bytes()


def test_cmake_package_builds_installs_and_is_consumable(tmp_path):
    """SURVEY 7 step 1: a CMake package for C++ consumers.  Configure + build + install the two libraries with the top-level
    CMakeLists.txt, then build tests/cpp/demo_like.cpp in a separate CMake project through find_package(dynamicfusion_b200)."""
    import shutil
    cmake = shutil.which("cmake")
    if not cmake or not Path("/usr/local/cuda/bin/nvcc").exists():
        pytest.skip("cmake / nvcc not available")
    gen = ["-G", "Ninja"] if shutil.which("ninja") else []
    build, prefix = tmp_path / "build", tmp_path / "prefix"
    env = dict(os.environ, CUDACXX="/usr/local/cuda/bin/nvcc")
    for cmd in ([cmake, "-S", str(ROOT), "-B", str(build), *gen, "-DCMAKE_CUDA_COMPILER=/usr/local/cuda/bin/nvcc"],
                [cmake, "--build", str(build), "-j", "8"], [cmake, "--install", str(build), "--prefix", str(prefix)]):
        r = subprocess.run(cmd, capture_output=True, text=True, env=env, timeout=1500)
        assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert (prefix / "lib" / "libdfusion.so").exists() and (prefix / "lib" / "libkfusion.so").exists()
    assert (prefix / "include" / "dfusion.h").exists() and (prefix / "include" / "kfusion" / "kinfu.hpp").exists()
    # every symbol the header declares is exported by the CMake-built library too
    from dynamicfusion_b200 import capi
    syms = subprocess.run(["nm", "-D", "--defined-only", str(prefix / "lib" / "libdfusion.so")], capture_output=True, text=True).stdout
    assert all(f" T {name}\n" in syms for name in capi.PROTOTYPES), [n for n in capi.PROTOTYPES if f" T {n}\n" not in syms]
    consumer = tmp_path / "consumer"
    consumer.mkdir()
    (consumer / "CMakeLists.txt").write_text(
        "cmake_minimum_required(VERSION 3.24)\nproject(consumer LANGUAGES CXX CUDA)\nset(CMAKE_CXX_STANDARD 17)\n"
        "find_package(dynamicfusion_b200 CONFIG REQUIRED)\nfind_package(CUDAToolkit REQUIRED)\n"
        f"add_executable(demo_like {ROOT / 'tests' / 'cpp' / 'demo_like.cpp'})\n"
        "target_link_libraries(demo_like PRIVATE dynamicfusion_b200::kfusion CUDA::cudart)\n")
    for cmd in ([cmake, "-S", str(consumer), "-B", str(consumer / "b"), *gen, f"-DCMAKE_PREFIX_PATH={prefix}", "-DCMAKE_CUDA_COMPILER=/usr/local/cuda/bin/nvcc",
                 "-DCMAKE_CUDA_ARCHITECTURES=100a"], [cmake, "--build", str(consumer / "b")]):
        r = subprocess.run(cmd, capture_output=True, text=True, env=env, timeout=900)
        assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert (consumer / "b" / "demo_like").exists()
