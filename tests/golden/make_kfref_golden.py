"""Regenerate tests/golden/kfref_golden.json: SHA-256 digests of what the REFERENCE's own CUDA kernels
(kfusion/src/cuda/{tsdf_volume,imgproc,proj_icp}.cu, compiled for the host by oracle/ref_shim into
oracle/_ref/libkfref.so) produce on the seeded scenes of tests/kfref_cases.py, plus two array files:

  * kfref_racy.npz    -- for each output in kfref_cases.RACY, the pixels where the reference's host run differs from the oracle
                         (np.packbits of the flat pixel mask); the reference holds +0.0 in every channel of each of them;
  * kfref_render.npz  -- the reference's display and depth-path image kernels on kfref_cases.render_scene: the bit-exact outputs
                         as digests, the Phong images (compared to a grey level) on every 4th row and column (SAMPLE).

Needs a checkout of the reference project (REF, default as in oracle/Makefile):

    make -C oracle ref REF=<reference checkout> && python tests/golden/make_kfref_golden.py

tests/test_oracle_vs_reference_kernels.py and tests/test_render_gpu.py compare against these files."""
import ctypes as C
import json
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[2]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))

from oracle import orc  # noqa: E402
import kfref_cases  # noqa: E402

HERE = Path(__file__).resolve().parent
LIGHT = (0.3, -0.2, -0.5)
SAMPLE = (slice(None, None, 4), slice(None, None, 4))      # the display kernels work pixel by pixel: a grid of pixels is a fair sample


def racy(ref_outputs):
    mine = kfref_cases.all_cases(orc, ref=False)
    out = {}
    for name, b in ref_outputs.items():
        if name.rsplit("/", 1)[1] not in kfref_cases.RACY:
            continue
        a = mine[name]
        diff = np.any((a.view(np.uint32) != b.view(np.uint32)) & ~(np.isnan(a) & np.isnan(b)), axis=-1).reshape(-1)
        assert not b.reshape(-1, b.shape[-1])[diff].view(np.uint32).any(), name
        out[name] = np.packbits(diff)
    np.savez_compressed(HERE / "kfref_racy.npz", **out)


def render():
    ref, vp = orc.load_ref(), (lambda a: C.c_void_p(a.ctypes.data))
    s = kfref_cases.render_scene(orc)
    K, light = kfref_cases.K, (C.c_float * 3)(*LIGHT)
    hp, hn = s["points"], s["normals"]
    out = {"volume_sha256": kfref_cases.digest(s["volume"])}
    rimg, rtan = np.zeros((480, 640, 4), np.uint8), np.zeros((480, 640, 4), np.uint8)
    ref.kfref_render_image(vp(hp), C.c_size_t(640 * 16), vp(hn), C.c_size_t(640 * 16), 640, 480, orc.intr(*K), light, vp(rimg), C.c_size_t(640 * 4))
    ref.kfref_render_tangent_colors(vp(hn), C.c_size_t(640 * 16), 640, 480, vp(rtan), C.c_size_t(640 * 4))
    rtan[np.isnan(hn[..., 0])] = 0                           # compared where the normal is defined
    out["render_image"], out["render_tangent_sha256"] = rimg[SAMPLE], kfref_cases.digest(rtan)
    # depth path: computeNormalsAndMaskDepth -> resizeDepthNormals -> renderImage(depth)
    d_ref, n_ref = s["depth"].copy(), np.zeros((480, 640, 4), np.float32)
    ref.kfref_normals_mask_depth(orc.intr(*K), vp(d_ref), C.c_size_t(640 * 2), 640, 480, vp(n_ref), C.c_size_t(640 * 16))
    dd_ref, nd_ref = np.zeros((240, 320), np.uint16), np.zeros((240, 320, 4), np.float32)
    ref.kfref_resize_depth_normals(vp(d_ref), C.c_size_t(640 * 2), vp(n_ref), C.c_size_t(640 * 16), 640, 480, vp(dd_ref), C.c_size_t(320 * 2), vp(nd_ref),
                                   C.c_size_t(320 * 16))
    rimg_d = np.zeros((480, 640, 4), np.uint8)
    ref.kfref_render_image_depth(vp(d_ref), C.c_size_t(640 * 2), vp(n_ref), C.c_size_t(640 * 16), 640, 480, orc.intr(*K), light, vp(rimg_d), C.c_size_t(640 * 4))
    out.update({"masked_depth_sha256": kfref_cases.digest(d_ref), "masked_normals_sha256": kfref_cases.digest(n_ref),
                "resized_depth_sha256": kfref_cases.digest(dd_ref), "resized_normals_sha256": kfref_cases.digest(nd_ref),
                "render_image_depth": rimg_d[SAMPLE]})
    # ray-cast, depth variant, and cloudToDepth of the point map
    c2d = np.zeros((480, 640), np.uint16)
    ref.kfref_cloud_to_depth(vp(hp), C.c_size_t(640 * 16), 640, 480, vp(c2d), C.c_size_t(640 * 2))
    rd, rn = np.zeros((480, 640), np.uint16), np.zeros((480, 640, 4), np.float32)
    ref.kfref_raycast_depth(orc.volume(s["volume"], s["dims"], s["voxel_size"], kfref_cases.TRUNC, kfref_cases.MAXW), orc.aff(*s["cam2vol"]), orc._f9(s["Rinv"]),
                            orc.intr(*K), 640, 480, C.c_float(0.75), C.c_float(0.5), vp(rd), C.c_size_t(640 * 2), vp(rn), C.c_size_t(640 * 16))
    valid = ~np.isnan(hp[..., 2])
    assert np.array_equal(c2d[valid], rd[valid]) and np.all(rd[~valid] == 0), "reference cloudToDepth and depth ray-cast disagree"
    out["raycast_depth_sha256"] = kfref_cases.digest(rd)
    np.savez_compressed(HERE / "kfref_render.npz", **out)


if __name__ == "__main__":
    orc.build()
    assert orc.reference_available(), "oracle/_ref/libkfref.so missing: run `make -C oracle ref REF=<reference checkout>` first"
    ref_outputs = kfref_cases.all_cases(orc, ref=True)
    out = {}
    for name, arr in ref_outputs.items():
        out[name] = {"sha256": kfref_cases.digest(arr), "dtype": str(arr.dtype), "shape": list(arr.shape)}
    (HERE / "kfref_golden.json").write_text(json.dumps(out, indent=1, sort_keys=True) + "\n")
    racy(ref_outputs)
    render()
    print(f"wrote {len(out)} digests, kfref_racy.npz, kfref_render.npz")
