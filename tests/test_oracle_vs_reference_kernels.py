"""Pins the oracle's TSDF / image / ICP kernels to the REFERENCE's own code.

oracle/ref_shim compiles the reference's kfusion/src/cuda/{tsdf_volume,imgproc,proj_icp}.cu for the host (a CUDA-on-CPU
emulation of the handful of runtime/texture/intrinsic calls they make, oracle/ref_shim/cudahost/cuda_runtime.h) into
oracle/_ref/libkfref.so (and proj_icp.cu once more with the reference's compile-time USE_DEPTH switch into libkfref_usedepth.so).  Bar: BIT-EXACT on every output (u32 voxels, u16 images, f32 vertex/normal maps, f64 ICP sums).

  * test_oracle_matches_reference_digests: oracle outputs vs the committed SHA-256 digests of the reference's outputs
    (tests/golden/kfref_golden.json, written by tests/golden/make_kfref_golden.py);
  * test_oracle_bit_exact_vs_reference_build: the outputs where the reference's host run is racy (kfref_cases.RACY), rebuilt from
    the oracle's and the pixels the reference zeroed (tests/golden/kfref_racy.npz), against the reference's digests.

extract_kernel (tsdf_volume.cu:511-710: warp votes, a warp-synchronous scan over volatile shared memory, shared staging) cannot be
run thread after thread; it runs under the warp-lock-step executor of oracle/ref_shim/cudahost/lockstep.h (32 lanes of a warp as
fibers, min-PC scheduling on every shared-memory access, votes as warp barriers) in oracle/_ref/libkfref_lockstep.so, and the
SORTED point set is compared bit for bit (`*/cloud_sorted`, three volumes incl. ragged dims).

Not covered by the host build (documented in DESIGN.md): the float tree-order of the ICP block reduction (launch-geometry
dependent); the approximate GPU intrinsics (__expf, __fdividef, rsqrt) are taken as their correctly rounded operations on both
sides; extraction into a buffer that fills up (the reference writes out of bounds there, see kfref/extract_tail.inc)."""
import json
from pathlib import Path

import numpy as np
import pytest

import kfref_cases

GOLDEN = json.loads((Path(__file__).parent / "golden" / "kfref_golden.json").read_text())
RACY_PIXELS = np.load(Path(__file__).parent / "golden" / "kfref_racy.npz")


@pytest.fixture(scope="module")
def oracle_outputs(orc):
    return kfref_cases.all_cases(orc, ref=False)


def test_oracle_matches_reference_digests(oracle_outputs):
    assert set(oracle_outputs) == set(GOLDEN)
    checked = 0
    for name, arr in oracle_outputs.items():
        g = GOLDEN[name]
        assert list(arr.shape) == g["shape"] and str(arr.dtype) == g["dtype"], name
        if name.rsplit("/", 1)[1] in kfref_cases.RACY:
            continue                                             # see kfref_cases.RACY; compared element-wise below
        assert kfref_cases.digest(arr) == g["sha256"], f"{name}: oracle output differs from the reference's"
        checked += 1
    assert checked >= 44


def test_scenes_are_meaningful(oracle_outputs):
    o = oracle_outputs
    assert np.count_nonzero(o["tsdf64_tilted/volume"]) > 50_000 and np.count_nonzero(o["tsdf96_identity/volume"]) > 150_000
    assert np.count_nonzero(~np.isnan(o["tsdf64_tilted/ray_points"][..., 0])) > 50_000
    assert len(o["tsdf96_identity/cloud_normals"]) > 5_000 and np.count_nonzero(~np.isnan(o["tsdf96_identity/cloud_normals"][:, 0])) > 2_000
    assert np.count_nonzero(o["tsdf64_tilted/removed_dists"] != o["tsdf64_tilted/dists"]) > 10_000
    for lvl in range(3):
        assert int(o[f"imgproc_icp/icp_inliers_l{lvl}"][0]) > 1000 >> lvl


def test_oracle_bit_exact_vs_reference_build(oracle_outputs):
    for name, a in oracle_outputs.items():
        if name.rsplit("/", 1)[1] not in kfref_cases.RACY:
            continue
        diff = np.unpackbits(RACY_PIXELS[name], count=a.size // a.shape[-1]).astype(bool).reshape(a.shape[:-1])
        assert not np.isnan(a[diff]).any(), name
        b = a.copy()
        # every difference is a pixel whose texel an earlier thread had already zeroed: the reference then read Dp = 0
        b[diff] = 0.0
        assert kfref_cases.digest(b) == GOLDEN[name]["sha256"], f"{name}: oracle != reference kernels outside the racy pixels"
        assert 0 < np.count_nonzero(diff) < 0.7 * np.count_nonzero(~np.isnan(a[..., 0])), name
