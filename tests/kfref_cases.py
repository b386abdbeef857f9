"""Seeded scenes run through the oracle's kernels (oracle/orc_*.c) or -- inside `with orc.reference()` -- through the
REFERENCE's own CUDA kernels compiled for the host (oracle/_ref/libkfref.so, built by oracle/ref_shim from
/root/reference/kfusion/src/cuda/*.cu).  Shared by tests/test_oracle_vs_reference_kernels.py and
tests/golden/make_kfref_golden.py so that the committed digests and the live comparison cover identical inputs."""
import contextlib
import hashlib
import math

import numpy as np

from dynamicfusion_b200 import synth

K = synth.DEFAULT_K
TRUNC, MAXW = 0.04, 64


def _inv(p):
    Ri = np.linalg.inv(np.asarray(p[0], np.float64)).astype(np.float32)
    return Ri, (-(Ri @ np.asarray(p[1], np.float32))).astype(np.float32)


def _mul(a, b):
    return (a[0] @ b[0]).astype(np.float32), (a[0] @ b[1] + a[1]).astype(np.float32)


def _tilted_pose():
    a, b = np.deg2rad(7.0), np.deg2rad(-4.0)
    Rx = np.array([[1, 0, 0], [0, np.cos(a), -np.sin(a)], [0, np.sin(a), np.cos(a)]])
    Ry = np.array([[np.cos(b), 0, np.sin(b)], [0, 1, 0], [-np.sin(b), 0, np.cos(b)]])
    return (Rx @ Ry).astype(np.float32), np.array([0.03, -0.02, 0.05], np.float32)


def _identity():
    return np.eye(3, dtype=np.float32), np.zeros(3, np.float32)


def sort_points(p: np.ndarray) -> np.ndarray:
    """order-independent form of a point list: rows sorted by their bit patterns (the reference appends in warp-completion order,
    the oracle in (z, y, x, axis) order; parity is on the SET of points, bit for bit)"""
    p = np.ascontiguousarray(p, np.float32)
    u = p.view(np.uint32)
    return p[np.lexsort(u.T[::-1])]


def tsdf_case(orc, dim, tilted, ref, dims=None):
    """compute_dists -> 2 x integrate -> raycast -> extract cloud -> extract_normals -> project_and_remove"""
    ctx = orc.reference() if ref else contextlib.nullcontext()
    out = {}
    depth = synth.sphere_wall_depth(seed=dim)
    dims, vs = dims or (dim,) * 3, (1.0 / dim,) * 3
    vol_pose = synth.volume_pose(1.0)
    cam = _tilted_pose() if tilted else _identity()
    with ctx:
        dists = orc.compute_dists(depth, K)
        vol = np.full(dims[0] * dims[1] * dims[2], 0xdeadbeef, np.uint32)
        orc.clear_volume(vol, dims, vs, TRUNC, MAXW)
        for pose in (cam, _mul(cam, (np.eye(3, dtype=np.float32), np.array([0.004, 0.0, 0.002], np.float32)))):
            orc.integrate(vol, dims, vs, TRUNC, MAXW, dists, _mul(_inv(pose), vol_pose), K)
        cam2vol = _mul(_inv(vol_pose), cam)
        pts, nrm, _ = orc.raycast_points(vol, dims, vs, TRUNC, MAXW, cam2vol, _inv(cam2vol)[0], K, 640, 480, 0.75, 0.5)
    out["dists"], out["volume"], out["ray_points"], out["ray_normals"] = dists, vol, pts, nrm
    with ctx:
        # zero-crossing cloud: the oracle's restatement, or the reference's own warp-synchronous extract_kernel (tsdf_volume.cu:511-710)
        # under the warp-lock-step executor (oracle/ref_shim/cudahost/lockstep.h -> libkfref_lockstep.so)
        cloud = sort_points(orc.extract_cloud(vol, dims, vs, TRUNC, MAXW, vol_pose, 400000))
        out["cloud_sorted"] = cloud
        out["cloud_normals"] = orc.extract_normals(vol, dims, vs, TRUNC, MAXW, cloud, vol_pose, _inv(vol_pose)[0], 0.5)
        # raycast points back in the camera frame, projected into the frame's dists (kinfu.cpp:300)
        proj = pts.copy()
        Ri, ti = _inv(cam2vol)
        m = ~np.isnan(proj[..., 0])
        proj[m, :3] = (proj[m, :3] @ Ri.T + ti).astype(np.float32)
        d2 = dists.copy()
        orc.project_and_remove(d2, K, proj)
    out["removed_dists"], out["projected_points"] = d2, proj
    return out


def imgproc_icp_case(orc, ref):
    """bilateral -> truncate -> pyramid -> points/normals per level -> resize -> ICP sums per level"""
    ctx = orc.reference() if ref else contextlib.nullcontext()
    out = {}

    def pyramids(depth):
        b = orc.bilateral(depth, 7, 4.5, 0.04)
        orc.truncate_depth(b, 1.35)
        ds = [b]
        for _ in range(2):
            ds.append(orc.pyr_down(ds[-1], 0.04))
        return ds, [orc.points_normals(tuple(k / (1 << i) for k in K), d) for i, d in enumerate(ds)]

    with ctx:
        da, a = pyramids(synth.umbrella_depth(0))
        db, b = pyramids(synth.umbrella_depth(3, shape_t=0))
        for i, d in enumerate(da):
            out[f"depth_l{i}"] = d
        for i, (v, n) in enumerate(a):
            out[f"points_l{i}"], out[f"normals_l{i}"] = v, n
        rv, rn = orc.resize_points_normals(a[0][0], a[0][1])
        out["resized_points"], out["resized_normals"] = rv, rn
        T = (np.eye(3, dtype=np.float32), np.array([0.002, -0.001, 0.0], np.float32))
        for lvl in range(3):
            Kl = tuple(k / (1 << lvl) for k in K)
            sums, inl = orc.icp_accumulate(b[lvl][0], b[lvl][1], a[lvl][0], a[lvl][1], Kl, T, 0.1 * 0.1, math.cos(30 * 0.017453293))
            out[f"icp_sums_l{lvl}"], out[f"icp_inliers_l{lvl}"] = sums, np.array([inl], np.int64)
            # the reference's compile-time USE_DEPTH alternative: depth pyramids masked where the normal is invalid (what
            # computeNormalsAndMaskDepth leaves, kinfu.cpp:241-243) in place of the vertex maps
            dc, dp = db[lvl].copy(), da[lvl].copy()
            dc[np.isnan(b[lvl][1][..., 0])] = 0
            dp[np.isnan(a[lvl][1][..., 0])] = 0
            sums, inl = orc.icp_accumulate_depth(dc, b[lvl][1], dp, a[lvl][1], Kl, T, 0.1 * 0.1, math.cos(30 * 0.017453293))
            out[f"icp_depth_sums_l{lvl}"], out[f"icp_depth_inliers_l{lvl}"] = sums, np.array([inl], np.int64)
    return out


def all_cases(orc, ref):
    cases = {"tsdf64_tilted": tsdf_case(orc, 64, True, ref), "tsdf96_identity": tsdf_case(orc, 96, False, ref),
             # ragged dims: x not a multiple of the 32-wide block, y not a multiple of its 6 rows (partially and fully idle warps)
             "tsdf_ragged": tsdf_case(orc, 48, True, ref, dims=(48, 50, 40)), "imgproc_icp": imgproc_icp_case(orc, ref)}
    return {f"{c}/{k}": v for c, d in cases.items() for k, v in d.items()}


def render_scene(orc):
    """inputs of the display kernels (tests/test_render_gpu.py): the 128^3 umbrella volume integrated from the identity pose, its
    ray-cast point / normal maps, and the depth frame with a hole of the depth-path image ops.  Poses are formed as
    host.TsdfVolume.integrate / raycast form them, so the volume equals the GPU's bit for bit."""
    from dynamicfusion_b200 import host
    dim = 128
    dims, vs = (dim,) * 3, (1.0 / dim,) * 3
    vol_pose, pose = synth.volume_pose(1.0), host.identity_pose()
    vol = np.zeros(dim ** 3, np.uint32)
    orc.clear_volume(vol, dims, vs, TRUNC, MAXW)
    orc.integrate(vol, dims, vs, TRUNC, MAXW, orc.compute_dists(synth.umbrella_depth(0), K), host.aff_mul(host.aff_inv(pose), vol_pose), K)
    cam2vol = host.aff_mul(host.aff_inv(vol_pose), pose)
    Rinv = np.linalg.inv(cam2vol[0].astype(np.float64)).astype(np.float32)
    pts, nrm, _ = orc.raycast_points(vol, dims, vs, TRUNC, MAXW, cam2vol, Rinv, K, 640, 480, 0.75, 0.5)
    depth = synth.umbrella_depth(2)
    depth[100:140, 200:260] = 0                                              # a hole
    return {"dims": dims, "voxel_size": vs, "volume": vol, "cam2vol": cam2vol, "Rinv": Rinv, "points": np.ascontiguousarray(pts),
            "normals": np.ascontiguousarray(nrm), "depth": depth}


def canonical_bytes(a: np.ndarray) -> bytes:
    """bit pattern with every NaN mapped to one quiet NaN (payloads are not part of the contract)"""
    a = np.ascontiguousarray(a)
    if a.dtype == np.float32:
        u = a.view(np.uint32).copy()
        u[np.isnan(a)] = 0x7fc00000
        return u.tobytes()
    if a.dtype == np.float64:
        u = a.view(np.uint64).copy()
        u[np.isnan(a)] = 0x7ff8000000000000
        return u.tobytes()
    return a.tobytes()


def digest(a: np.ndarray) -> str:
    return hashlib.sha256(canonical_bytes(a)).hexdigest()


# project_kernel (tsdf_volume.cu:114-137) reads the dists texture while other threads zero texels of the same buffer: where two
# source pixels land on one texel the second reader may see 0.  The oracle reads the ORIGINAL dists everywhere; the sequential
# host run of the reference sees the zeros of earlier threads.  `removed_dists` (what integrate consumes) is unaffected.
RACY = ("projected_points",)
