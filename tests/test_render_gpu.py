"""Display kernels (df_render_image, df_render_tangent_colors -- what KinFu::renderImage and the reference's demo show) against the
REFERENCE's own render kernels (kfusion/src/cuda/imgproc.cu:474-583), run on the host by tests/golden/make_kfref_golden.py on the
scene of kfref_cases.render_scene; their outputs are stored in tests/golden/kfref_render.npz.  There is no oracle restatement for
these: the comparison is directly with the reference's code.  Bar: tangent colours identical wherever the normal is defined; the
Phong image within 1 grey level (the reference's __powf / rsqrt are approximate GPU intrinsics)."""
import ctypes as C
from pathlib import Path

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

import kfref_cases  # noqa: E402
from dynamicfusion_b200 import capi, host, synth  # noqa: E402

K = synth.DEFAULT_K
GOLDEN = np.load(Path(__file__).parent / "golden" / "kfref_render.npz")
SAMPLE = (slice(None, None, 4), slice(None, None, 4))      # the pixel grid the Phong images are stored on


@pytest.fixture(scope="module")
def scene(orc):
    s = kfref_cases.render_scene(orc)
    assert kfref_cases.digest(s["volume"]) == str(GOLDEN["volume_sha256"])
    return s


def test_render_kernels_match_the_reference_code(scene):
    hp, hn = scene["points"], scene["normals"]
    assert int((~np.isnan(hp[..., 0])).sum()) > 100_000
    pts, nrm = torch.from_numpy(hp).cuda(), torch.from_numpy(hn).cuda()
    light = (C.c_float * 3)(0.3, -0.2, -0.5)
    lib = capi.load()
    img = torch.zeros((480, 640, 4), dtype=torch.uint8, device="cuda")
    tan = torch.zeros_like(img)
    capi.check(lib.df_render_image(pts.data_ptr(), 640 * 16, nrm.data_ptr(), 640 * 16, 640, 480, light, img.data_ptr(), 640 * 4, None))
    capi.check(lib.df_render_tangent_colors(nrm.data_ptr(), 640 * 16, 640, 480, tan.data_ptr(), 640 * 4, None))
    torch.cuda.synchronize()
    rimg = GOLDEN["render_image"]
    gi, gt = img.cpu().numpy(), tan.cpu().numpy()
    assert np.abs(gi[SAMPLE].astype(np.int16) - rimg.astype(np.int16)).max() <= 1
    assert np.mean(gi[SAMPLE] != rimg) < 0.02
    valid = ~np.isnan(hn[..., 0])
    gt[~valid] = 0
    assert kfref_cases.digest(gt) == str(GOLDEN["render_tangent_sha256"])
    assert len(np.unique(gi[valid][:, 0])) > 50 and len(np.unique(gi[~valid][:, 0])) > 50      # a shaded surface over the gradient background


def test_depth_path_image_ops_match_the_reference_code(scene):
    """cuda/imgproc.hpp functions of the reference's USE_DEPTH path (computeNormalsAndMaskDepth, resizeDepthNormals, cloudToDepth,
    renderImage(depth)) and the depth variant of the ray-cast: bit-exact against the reference's own kernels (Phong image: 1 level)"""
    lib = capi.load()
    depth = scene["depth"]
    # computeNormalsAndMaskDepth
    d_dev = host.u16_to_device(depth)
    n_dev = torch.zeros((480, 640, 4), dtype=torch.float32, device="cuda")
    capi.check(lib.df_normals_mask_depth(capi.make_intr(*K), d_dev.data_ptr(), 640 * 2, 640, 480, n_dev.data_ptr(), 640 * 16, None))
    gd, gn = host.u16_from_device(d_dev), n_dev.cpu().numpy()
    assert kfref_cases.digest(gd) == str(GOLDEN["masked_depth_sha256"]) and np.count_nonzero(gd != depth) > 500
    assert kfref_cases.digest(gn) == str(GOLDEN["masked_normals_sha256"])
    # resizeDepthNormals
    dd = torch.zeros((240, 320), dtype=torch.int16, device="cuda")
    nd = torch.zeros((240, 320, 4), dtype=torch.float32, device="cuda")
    capi.check(lib.df_resize_depth_normals(d_dev.data_ptr(), 640 * 2, n_dev.data_ptr(), 640 * 16, 640, 480, dd.data_ptr(), 320 * 2, nd.data_ptr(), 320 * 16, None))
    assert kfref_cases.digest(host.u16_from_device(dd)) == str(GOLDEN["resized_depth_sha256"])
    assert kfref_cases.digest(nd.cpu().numpy()) == str(GOLDEN["resized_normals_sha256"])
    # renderImage(depth)
    light = (C.c_float * 3)(0.3, -0.2, -0.5)
    img = torch.zeros((480, 640, 4), dtype=torch.uint8, device="cuda")
    capi.check(lib.df_render_image_depth(d_dev.data_ptr(), 640 * 2, n_dev.data_ptr(), 640 * 16, 640, 480, capi.make_intr(*K), light, img.data_ptr(), 640 * 4, None))
    rimg = GOLDEN["render_image_depth"]
    gi = img.cpu().numpy()[SAMPLE]
    assert np.abs(gi.astype(np.int16) - rimg.astype(np.int16)).max() <= 1 and np.mean(gi != rimg) < 0.02
    # ray-cast, depth variant = points variant + cloudToDepth; against the reference's depth ray-cast of the same volume, which
    # tests/golden/make_kfref_golden.py also checked against the reference's cloudToDepth of the scene's point map
    dim = 128
    vol = host.TsdfVolume((dim, dim, dim))
    # the size first: setTruncDist clamps to 2.1 voxels of the current size (3 m by default), and the scene's distance is 0.04
    vol.setSize((1.0, 1.0, 1.0)); vol.setTruncDist(0.04); vol.setMaxWeight(64); vol.setPose(synth.volume_pose(1.0))
    vol.setRaycastStepFactor(0.75); vol.setGradientDeltaFactor(0.5); vol.clear()
    pose = host.identity_pose()
    vol.integrate(host.computeDists(host.u16_to_device(synth.umbrella_depth(0)), K), pose, K)
    assert kfref_cases.digest(vol.data_.cpu().numpy().view(np.uint32)) == str(GOLDEN["volume_sha256"])
    pts, nrm, _ = vol.raycast(pose, K, 640, 480)
    rc = torch.zeros((480, 640), dtype=torch.int16, device="cuda")
    capi.check(lib.df_cloud_to_depth(pts.data_ptr(), 640 * 16, 640, 480, rc.data_ptr(), 640 * 2, None))
    valid = ~np.isnan(pts.cpu().numpy()[..., 2])
    g_rc = host.u16_from_device(rc)
    assert np.all(g_rc[~valid] == 0) and np.count_nonzero(g_rc) > 100_000
    assert kfref_cases.digest(g_rc) == str(GOLDEN["raycast_depth_sha256"])
