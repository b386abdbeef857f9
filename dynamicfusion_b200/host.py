"""Python host-side mirror of the reference's component API for the hot path, over the C ABI (capi.py).

Names, argument meaning and defaults follow the reference's host classes so parity tests read like the reference:
  TsdfVolume       <- kfusion::cuda::TsdfVolume      (kfusion/include/kfusion/cuda/tsdf_volume.hpp:11-100)
  computeDists ... <- kfusion::cuda::* free functions (kfusion/include/kfusion/cuda/imgproc.hpp:9-33)
  ProjectiveICP    <- kfusion::cuda::ProjectiveICP   (kfusion/include/kfusion/cuda/projective_icp.hpp:9-46)
  WarpField        <- kfusion::WarpField             (kfusion/include/kfusion/warp_field.hpp:41-88)
torch supplies device memory and streams; every compute call goes through libdfusion.so.
Images: depth/dists are torch.int16 (u16 bits) [rows, cols]; vertex/normal maps torch.float32 [rows, cols, 4].
Poses are (R 3x3 float32, t 3 float32) numpy pairs (cv::Affine3f).
"""
from __future__ import annotations

import ctypes as C
import math

import numpy as np
import torch

from . import capi


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _lib():
    if not torch.cuda.is_available():
        raise RuntimeError("dynamicfusion_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
    return capi.load()


def aff_inv(pose):
    """cv::Affine3f::inv(): R^-1 (closed form 3x3), t' = -R^-1 t, in float32"""
    R, t = np.asarray(pose[0], np.float32), np.asarray(pose[1], np.float32)
    Ri = np.linalg.inv(R.astype(np.float64)).astype(np.float32)
    return Ri, (-(Ri @ t)).astype(np.float32)


def aff_mul(A, B):
    RA, tA = np.asarray(A[0], np.float32), np.asarray(A[1], np.float32)
    RB, tB = np.asarray(B[0], np.float32), np.asarray(B[1], np.float32)
    return (RA @ RB).astype(np.float32), (RA @ tB + tA).astype(np.float32)


def identity_pose():
    return np.eye(3, dtype=np.float32), np.zeros(3, np.float32)


def u16_to_device(a: np.ndarray, device="cuda") -> torch.Tensor:
    assert a.dtype == np.uint16
    return torch.from_numpy(a.view(np.int16).copy()).to(device)


def u16_from_device(t: torch.Tensor) -> np.ndarray:
    return t.cpu().numpy().view(np.uint16)


# ------------------------------------------------------------------ imgproc free functions ---------------------------------------------------
def computeDists(depth: torch.Tensor, intr) -> torch.Tensor:
    rows, cols = depth.shape
    dists = torch.empty_like(depth)
    capi.check(_lib().df_compute_dists(depth.data_ptr(), cols * 2, cols, rows, capi.make_intr(*intr), dists.data_ptr(), cols * 2, _stream()))
    return dists


def depthBilateralFilter(depth: torch.Tensor, ksz: int, sigma_spatial: float, sigma_depth: float) -> torch.Tensor:
    rows, cols = depth.shape
    out = torch.empty_like(depth)
    capi.check(_lib().df_bilateral(depth.data_ptr(), cols * 2, cols, rows, out.data_ptr(), cols * 2, ksz, sigma_spatial, sigma_depth, _stream()))
    return out


def depthTruncation(depth: torch.Tensor, threshold: float) -> None:
    rows, cols = depth.shape
    capi.check(_lib().df_truncate_depth(depth.data_ptr(), cols * 2, cols, rows, threshold, _stream()))


def depthBuildPyramid(depth: torch.Tensor, sigma_depth: float) -> torch.Tensor:
    rows, cols = depth.shape
    out = torch.empty((rows // 2, cols // 2), dtype=depth.dtype, device=depth.device)
    capi.check(_lib().df_pyr_down(depth.data_ptr(), cols * 2, cols, rows, out.data_ptr(), (cols // 2) * 2, sigma_depth, _stream()))
    return out


def computePointNormals(intr, depth: torch.Tensor):
    rows, cols = depth.shape
    pts = torch.empty((rows, cols, 4), dtype=torch.float32, device=depth.device)
    nrm = torch.empty_like(pts)
    capi.check(_lib().df_points_normals(capi.make_intr(*intr), depth.data_ptr(), cols * 2, cols, rows, pts.data_ptr(), cols * 16,
                                        nrm.data_ptr(), cols * 16, _stream()))
    return pts, nrm


def resizePointsNormals(points: torch.Tensor, normals: torch.Tensor):
    rows, cols = points.shape[:2]
    vd = torch.empty((rows // 2, cols // 2, 4), dtype=torch.float32, device=points.device)
    nd = torch.empty_like(vd)
    capi.check(_lib().df_resize_points_normals(points.data_ptr(), cols * 16, normals.data_ptr(), cols * 16, cols, rows,
                                               vd.data_ptr(), (cols // 2) * 16, nd.data_ptr(), (cols // 2) * 16, _stream()))
    return vd, nd


def save_ply(path, points, normals=None, triangles=None) -> int:
    """Export of the extracted canonical cloud (SURVEY 8f(4); Report.md "Export the reconstructions to .ply"): the Python twin of
    kfusion::writePly (include/kfusion/io/ply.hpp) -- binary little-endian PLY, float x y z [nx ny nz]; points with a NaN coordinate
    are skipped, NaN normals written as 0.  points / normals: host or device arrays of shape [N, >=3].
    triangles ([M, 3] int32 vertex indices, e.g. from TsdfVolume.fetchMesh / KinFu.mesh): the mesh form, which adds `element face M`
    (`property list uchar int vertex_indices`) and writes every vertex as given -- mesh vertices are finite, and dropping one would shift
    the indices.  Returns the number of vertices written."""
    host = lambda a: np.asarray(a.detach().cpu().numpy() if isinstance(a, torch.Tensor) else a)
    pts = np.asarray(host(points), np.float32)[:, :3]
    keep = ~np.isnan(pts).any(1) if triangles is None else np.ones(len(pts), bool)
    cols = [pts[keep]]
    if normals is not None:
        nrm = np.asarray(host(normals), np.float32)[:, :3][keep].copy()
        nrm[np.isnan(nrm).any(1)] = 0.0
        cols.append(nrm)
    data = np.ascontiguousarray(np.concatenate(cols, 1), "<f4")
    with open(path, "wb") as f:
        what = b"canonical cloud" if triangles is None else b"mesh"
        f.write(b"ply\nformat binary_little_endian 1.0\ncomment dynamicfusion " + what + b"\n")
        f.write(f"element vertex {len(data)}\nproperty float x\nproperty float y\nproperty float z\n".encode())
        if normals is not None:
            f.write(b"property float nx\nproperty float ny\nproperty float nz\n")
        if triangles is not None:
            tri = np.asarray(host(triangles), np.int32).reshape(-1, 3)
            f.write(f"element face {len(tri)}\nproperty list uchar int vertex_indices\n".encode())
        f.write(b"end_header\n")
        f.write(data.tobytes())
        if triangles is not None:
            faces = np.empty(len(tri), np.dtype([("n", "u1"), ("i", "<i4", 3)]))
            faces["n"] = 3
            faces["i"] = tri
            f.write(faces.tobytes())
    return len(data)


def _popcount32(t: torch.Tensor) -> torch.Tensor:
    """per-element population count of an int32 tensor (bit tricks on int64 to stay clear of the sign bit)"""
    v = t.to(torch.int64) & 0xffffffff
    v = v - ((v >> 1) & 0x55555555)
    v = (v & 0x33333333) + ((v >> 2) & 0x33333333)
    v = (v + (v >> 4)) & 0x0f0f0f0f
    return (v * 0x01010101 >> 24) & 0xff


# ------------------------------------------------------------------ TsdfVolume ---------------------------------------------------------------
class TsdfVolume:
    """cuda::TsdfVolume (tsdf_volume.hpp:11-100, tsdf_volume.cpp).  Class defaults as tsdf_volume.cpp:7-14."""

    def __init__(self, dims, device="cuda", track_activity=False):
        self.device = device
        self.track_activity = track_activity      # dfusion.h DF_ACTIVITY_VOXELS: lets fetchCloud skip surface-free stretches
        self.activity_ = None
        self.trunc_dist_ = 0.03
        self.max_weight_ = 128
        self.size_ = np.array([3.0, 3.0, 3.0], np.float32)
        self.pose_ = identity_pose()
        self.gradient_delta_factor_ = 0.75
        self.raycast_step_factor_ = 0.75
        self.cloud_capacity = 0
        self._ws = None
        self._mesh_ws = None
        self._proj_ws = None
        self.create(dims)

    def create(self, dims):
        self.dims_ = np.array(dims, np.int32)
        n = int(self.dims_[0]) * int(self.dims_[1]) * int(self.dims_[2])
        self.data_ = torch.empty(n, dtype=torch.int32, device=self.device)
        if self.track_activity:
            self.activity_ = torch.zeros(int(_lib().df_volume_activity_bytes(self._vol())), dtype=torch.uint8, device=self.device)
        self.setTruncDist(self.trunc_dist_)
        self.clear()

    def getDims(self):
        return self.dims_

    def getVoxelSize(self):
        return (self.size_ / self.dims_.astype(np.float32)).astype(np.float32)

    def getSize(self):
        return self.size_

    def setSize(self, size):
        self.size_ = np.asarray(size, np.float32).reshape(3)
        self.setTruncDist(self.trunc_dist_)

    def getTruncDist(self):
        return self.trunc_dist_

    def setTruncDist(self, distance):
        vsz = self.getVoxelSize()
        self.trunc_dist_ = float(max(np.float32(distance), np.float32(2.1) * vsz.max()))   # tsdf_volume.cpp:68-73

    def setMaxWeight(self, w):
        self.max_weight_ = int(w)

    def getMaxWeight(self):
        return self.max_weight_

    def setPose(self, pose):
        self.pose_ = (np.asarray(pose[0], np.float32), np.asarray(pose[1], np.float32))

    def getPose(self):
        return self.pose_

    def setRaycastStepFactor(self, f):
        self.raycast_step_factor_ = float(f)

    def setGradientDeltaFactor(self, f):
        self.gradient_delta_factor_ = float(f)

    def applyAffine(self, affine):
        self.pose_ = aff_mul(affine, self.pose_)

    def _vol(self) -> capi.Volume:
        return capi.make_volume(self.data_.data_ptr(), self.dims_, self.getVoxelSize(), self.trunc_dist_, self.max_weight_)

    def clear(self):
        capi.check(_lib().df_clear_volume(self._vol(), _stream()))
        if self.activity_ is not None:
            self.activity_.zero_()

    def integrate(self, dists: torch.Tensor, camera_pose, intr, n_updated: torch.Tensor | None = None):
        vol2cam = aff_mul(aff_inv(camera_pose), self.pose_)                           # tsdf_volume.cpp:112
        rows, cols = dists.shape
        capi.check(_lib().df_integrate_tracked(self._vol(), dists.data_ptr(), cols * 2, cols, rows, capi.make_aff(*vol2cam),
                                               capi.make_intr(*intr), n_updated.data_ptr() if n_updated is not None else None,
                                               self.activity_.data_ptr() if self.activity_ is not None else None, None, _stream()))
        return vol2cam

    def integrate_warped(self, depth: torch.Tensor, camera_pose, intr, warp_field, weight_scale: float = 0.0,
                         counters: torch.Tensor | None = None):
        """Per-voxel warped integration (dfusion.h df_integrate_warped; SURVEY 8f(1)): what TsdfVolume::surface_fusion
        (tsdf_volume.cpp:228-254) was written towards.  depth = the u16 millimetre frame; the field's warp_to_live is applied
        before the camera transform, as WarpField::warp does."""
        world2cam = aff_mul(aff_inv(camera_pose), warp_field.warp_to_live_)
        rows, cols = depth.shape
        if warp_field.grid_ is None:
            raise RuntimeError("integrate_warped needs the node grid (WarpField(use_grid=True) + buildKDTree)")
        capi.check(_lib().df_integrate_warped(self._vol(), depth.data_ptr(), cols * 2, cols, rows, capi.make_aff(*self.pose_),
                                              capi.make_aff(*world2cam), capi.make_intr(*intr), warp_field.nodes_.data_ptr(),
                                              warp_field.nodes_.shape[0], warp_field.grid_.data_ptr(), float(weight_scale),
                                              counters.data_ptr() if counters is not None else None,
                                              self.activity_.data_ptr() if self.activity_ is not None else None, None, _stream()))
        return world2cam

    def raycast(self, camera_pose, intr, cols: int, rows: int, dense: bool = False):
        """dense=True forces the plain march (df_raycast_points) on a tracked volume; by default a tracked volume's march skips the
        bricks without negative voxels (df_raycast_points_tracked) -- same maps bit for bit"""
        cam2vol = aff_mul(aff_inv(self.pose_), camera_pose)                           # tsdf_volume.cpp:162
        Rinv = np.linalg.inv(cam2vol[0].astype(np.float64)).astype(np.float32)
        pts = torch.empty((rows, cols, 4), dtype=torch.float32, device=self.device)
        nrm = torch.empty_like(pts)
        if self.activity_ is not None and not dense:
            capi.check(_lib().df_raycast_points_tracked(self._vol(), capi.make_aff(*cam2vol), capi.f9(Rinv), capi.make_intr(*intr), cols, rows,
                                                        self.raycast_step_factor_, self.gradient_delta_factor_, pts.data_ptr(), cols * 16,
                                                        nrm.data_ptr(), cols * 16, self.activity_.data_ptr(), _stream()))
        else:
            capi.check(_lib().df_raycast_points(self._vol(), capi.make_aff(*cam2vol), capi.f9(Rinv), capi.make_intr(*intr), cols, rows,
                                                self.raycast_step_factor_, self.gradient_delta_factor_, pts.data_ptr(), cols * 16,
                                                nrm.data_ptr(), cols * 16, _stream()))
        return pts, nrm, (cam2vol, Rinv)

    def raycast_stats(self, camera_pose, intr, cols: int, rows: int, activity_ptr: int | None = None) -> dict:
        """df_raycast_points_stats: the ray-cast kernel instantiated with counters (measurement only).  Returns the unique voxels the
        launch reads (U of SURVEY 8d), the rays that produced a vertex, the march samples, and the algorithmic bytes 4*U + 32*cols*rows."""
        cam2vol = aff_mul(aff_inv(self.pose_), camera_pose)
        Rinv = np.linalg.inv(cam2vol[0].astype(np.float64)).astype(np.float32)
        pts = torch.empty((rows, cols, 4), dtype=torch.float32, device=self.device)
        nrm = torch.empty_like(pts)
        touched = torch.zeros(int(_lib().df_raycast_touched_bytes(self._vol())) // 4, dtype=torch.int32, device=self.device)
        stats = torch.zeros(2, dtype=torch.int64, device=self.device)
        if activity_ptr is None and self.activity_ is not None:     # activity_ptr = 0 forces the dense march on a tracked volume
            activity_ptr = self.activity_.data_ptr()
        if activity_ptr:
            capi.check(_lib().df_raycast_points_stats_tracked(self._vol(), capi.make_aff(*cam2vol), capi.f9(Rinv), capi.make_intr(*intr), cols, rows,
                                                              self.raycast_step_factor_, self.gradient_delta_factor_, pts.data_ptr(), cols * 16,
                                                              nrm.data_ptr(), cols * 16, touched.data_ptr(), stats.data_ptr(), activity_ptr, _stream()))
        else:
            capi.check(_lib().df_raycast_points_stats(self._vol(), capi.make_aff(*cam2vol), capi.f9(Rinv), capi.make_intr(*intr), cols, rows,
                                                      self.raycast_step_factor_, self.gradient_delta_factor_, pts.data_ptr(), cols * 16,
                                                      nrm.data_ptr(), cols * 16, touched.data_ptr(), stats.data_ptr(), _stream()))
        unique = int(_popcount32(touched).sum().item())
        hits, samples = (int(v) for v in stats.cpu().numpy())
        return {"unique_voxels": unique, "hit_rays": hits, "march_samples": samples, "algorithmic_bytes": 4 * unique + 32 * cols * rows,
                "points": pts, "normals": nrm}

    def project_and_remove(self, dists: torch.Tensor, intr, points: torch.Tensor):
        rows, cols = dists.shape
        prow, pcol = points.shape[:2]
        need = _lib().df_project_workspace_bytes(cols, rows)
        if self._proj_ws is None or self._proj_ws.numel() < need:
            self._proj_ws = torch.zeros(need, dtype=torch.uint8, device=self.device)
        capi.check(_lib().df_project_and_remove(dists.data_ptr(), cols * 2, cols, rows, capi.make_intr(*intr), points.data_ptr(),
                                                pcol * 16, pcol, prow, self._proj_ws.data_ptr(), _stream()))

    def fetchCloud(self, capacity: int = 256 * 256 * 256):
        """returns (points [capacity,4] device tensor, count device int32 tensor) -- no host sync"""
        need = _lib().df_extract_workspace_bytes(self._vol())
        if self._ws is None or self._ws.numel() < need:
            self._ws = torch.empty(need, dtype=torch.uint8, device=self.device)
        out = torch.empty((capacity, 4), dtype=torch.float32, device=self.device)
        count = torch.zeros(1, dtype=torch.int32, device=self.device)
        capi.check(_lib().df_extract_cloud_tracked(self._vol(), capi.make_aff(*self.pose_), out.data_ptr(), capacity, count.data_ptr(),
                                                   self._ws.data_ptr(), self.activity_.data_ptr() if self.activity_ is not None else None,
                                                   _stream()))
        return out, count

    def fetchMesh(self, vcap: int, tcap: int, normals: bool = True):
        """Triangle mesh of the zero level set (dfusion.h df_extract_mesh; marching cubes), through the activity map when the volume
        tracks one.  Returns device tensors (vertices [vcap, 4] float32, normals [vcap, 4] or None, edge keys [vcap] int32 holding the u32
        keys, triangles [tcap, 3] int32, counts [2] int32 = true vertex / triangle totals) -- no host sync.  Only the first
        min(count, cap) rows are written, and no triangle is when the vertices overflow."""
        need = _lib().df_extract_mesh_workspace_bytes(self._vol())
        if self._mesh_ws is None or self._mesh_ws.numel() < need:
            self._mesh_ws = torch.empty(need, dtype=torch.uint8, device=self.device)
        verts = torch.empty((max(vcap, 1), 4), dtype=torch.float32, device=self.device)
        keys = torch.empty(max(vcap, 1), dtype=torch.int32, device=self.device)
        tris = torch.empty((max(tcap, 1), 3), dtype=torch.int32, device=self.device)
        counts = torch.zeros(2, dtype=torch.int32, device=self.device)
        capi.check(_lib().df_extract_mesh(self._vol(), capi.make_aff(*self.pose_), self.activity_.data_ptr() if self.activity_ is not None else None,
                                          verts.data_ptr(), keys.data_ptr(), vcap, tris.data_ptr(), tcap, counts.data_ptr(),
                                          self._mesh_ws.data_ptr(), _stream()))
        nrm = self.fetchNormals(verts, vcap, counts[:1]) if normals and vcap > 0 else None
        return verts[:vcap], nrm, keys[:vcap], tris[:tcap], counts

    def fetchNormals(self, cloud: torch.Tensor, n: int, count_dev: torch.Tensor | None = None):
        Rinv = np.linalg.inv(self.pose_[0].astype(np.float64)).astype(np.float32)
        out = torch.empty((max(n, 1), 4), dtype=torch.float32, device=self.device)
        capi.check(_lib().df_extract_normals(self._vol(), cloud.data_ptr(), n, count_dev.data_ptr() if count_dev is not None else None,
                                             capi.make_aff(*self.pose_), capi.f9(Rinv), self.gradient_delta_factor_, out.data_ptr(), _stream()))
        return out[:n]


# ------------------------------------------------------------------ ProjectiveICP ------------------------------------------------------------
class ProjectiveICP:
    """cuda::ProjectiveICP (projective_icp.hpp:9-46); defaults projective_icp.cpp:68-76"""
    MAX_PYRAMID_LEVELS = 4

    def __init__(self, device="cuda"):
        self.device = device
        self.angle_thres_ = 20.0 * 0.017453293
        self.dist_thres_ = 0.1
        self.iters_ = [10, 5, 4, 0]
        self._T = torch.zeros(12, dtype=torch.float32, device=device)
        self._ok = torch.zeros(1, dtype=torch.int32, device=device)
        self._scratch = torch.zeros(32 + 27 * 1024, dtype=torch.float64, device=device)

    def setDistThreshold(self, d):
        self.dist_thres_ = float(d)

    def setAngleThreshold(self, a):
        self.angle_thres_ = float(a)

    def setIterationsNum(self, iters):
        it = list(iters)[: self.MAX_PYRAMID_LEVELS]
        self.iters_ = it + [0] * (self.MAX_PYRAMID_LEVELS - len(it))

    def getUsedLevelsNum(self):
        i = self.MAX_PYRAMID_LEVELS - 1
        while i >= 0 and not self.iters_[i]:
            i -= 1
        return i + 1

    def accumulate(self, vcurr, ncurr, vprev, nprev, intr_level, T):
        rows, cols = vcurr.shape[:2]
        out = self._scratch
        capi.check(_lib().df_icp_accumulate(vcurr.data_ptr(), cols * 16, ncurr.data_ptr(), cols * 16, vprev.data_ptr(), cols * 16,
                                            nprev.data_ptr(), cols * 16, cols, rows, capi.make_intr(*intr_level), capi.make_aff(*T),
                                            self.dist_thres_ * self.dist_thres_, math.cos(self.angle_thres_), out.data_ptr(), _stream()))
        return out[:27].clone()

    def estimateTransform(self, intr, vcurr, ncurr, vprev, nprev):
        """returns (ok, (R, t)) -- syncs to read the result (the fused pipeline never does)"""
        L = self.getUsedLevelsNum()
        vp = lambda xs: (C.c_void_p * L)(*[x.data_ptr() for x in xs[:L]])
        cols = (C.c_int * L)(*[x.shape[1] for x in vcurr[:L]])
        rows = (C.c_int * L)(*[x.shape[0] for x in vcurr[:L]])
        pitch = (C.c_size_t * L)(*[x.shape[1] * 16 for x in vcurr[:L]])
        it = (C.c_int * L)(*self.iters_[:L])
        capi.check(_lib().df_icp_estimate(vp(vcurr), vp(ncurr), vp(vprev), vp(nprev), cols, rows, pitch, L, it, capi.make_intr(*intr),
                                          self.dist_thres_, self.angle_thres_, self._T.data_ptr(), self._ok.data_ptr(),
                                          self._scratch.data_ptr(), _stream()))
        T = self._T.cpu().numpy()
        return bool(self._ok.item()), (T[:9].reshape(3, 3).copy(), T[9:].copy())


    def accumulateDepth(self, dcurr, ncurr, dprev, nprev, intr_level, T):
        """the reference's USE_DEPTH alternative of the association pass: u16 (rows, cols) depth maps in place of the vertex maps"""
        rows, cols = dcurr.shape[:2]
        out = self._scratch
        capi.check(_lib().df_icp_accumulate_depth(dcurr.data_ptr(), cols * 2, ncurr.data_ptr(), cols * 16, dprev.data_ptr(), cols * 2,
                                                  nprev.data_ptr(), cols * 16, cols, rows, capi.make_intr(*intr_level), capi.make_aff(*T),
                                                  self.dist_thres_ * self.dist_thres_, math.cos(self.angle_thres_), out.data_ptr(),
                                                  _stream()))
        return out[:27].clone()

    def estimateTransformDepth(self, intr, dcurr, ncurr, dprev, nprev):
        """estimateTransform(affine, intr, DepthPyr, NormalsPyr, DepthPyr, NormalsPyr) (projective_icp.hpp:38)"""
        L = self.getUsedLevelsNum()
        vp = lambda xs: (C.c_void_p * L)(*[x.data_ptr() for x in xs[:L]])
        cols = (C.c_int * L)(*[x.shape[1] for x in dcurr[:L]])
        rows = (C.c_int * L)(*[x.shape[0] for x in dcurr[:L]])
        dpitch = (C.c_size_t * L)(*[x.shape[1] * 2 for x in dcurr[:L]])
        npitch = (C.c_size_t * L)(*[x.shape[1] * 16 for x in dcurr[:L]])
        it = (C.c_int * L)(*self.iters_[:L])
        capi.check(_lib().df_icp_estimate_depth(vp(dcurr), vp(ncurr), vp(dprev), vp(nprev), cols, rows, dpitch, npitch, L, it,
                                                capi.make_intr(*intr), self.dist_thres_, self.angle_thres_, self._T.data_ptr(),
                                                self._ok.data_ptr(), self._scratch.data_ptr(), _stream()))
        T = self._T.cpu().numpy()
        return bool(self._ok.item()), (T[:9].reshape(3, 3).copy(), T[9:].copy())


# ------------------------------------------------------------------ WarpField ----------------------------------------------------------------
NODE_STRIDE = 12
KNN_NEIGHBOURS = 8


class WarpField:
    """kfusion::WarpField (warp_field.hpp:41-88).  Nodes live on the device as [M, 12] float32 (see dfusion.h).
    `use_grid` selects the uniform node grid (buildKDTree's replacement) or the exhaustive shared-memory scan; both give
    identical neighbours."""

    def __init__(self, device="cuda", use_grid=True):
        self.device = device
        self.nodes_ = torch.zeros((0, NODE_STRIDE), dtype=torch.float32, device=device)
        self.warp_to_live_ = identity_pose()
        self.use_grid = use_grid
        self.grid_ = None
        self._ws = None

    def init(self, first_frame):
        """WarpField::init(std::vector<Vec3f>) (warp_field.cpp:70-88): every non-NaN point becomes a node with the
        identity DualQuaternion() (rot (1,0,0,0), dual (1,0,0,0)) and weight 3*voxel_size with voxel_size forced to 1."""
        v = np.asarray(first_frame, np.float32).reshape(-1, 3)
        v = v[~np.isnan(v[:, 0])]
        n = np.zeros((len(v), NODE_STRIDE), np.float32)
        n[:, 0:3] = v
        n[:, 3] = 1.0
        n[:, 7] = 1.0
        n[:, 11] = 3.0
        self.setNodes(torch.from_numpy(n).to(self.device))

    def setNodes(self, nodes: torch.Tensor):
        self.nodes_ = nodes
        self.buildKDTree()

    def buildKDTree(self):
        """WarpField::buildKDTree (warp_field.cpp:275-282) -> df_build_node_grid"""
        M = self.nodes_.shape[0]
        self.grid_ = None
        if self.use_grid and M > 0:
            self.grid_ = torch.empty(_lib().df_node_grid_bytes(M), dtype=torch.uint8, device=self.device)
            capi.check(_lib().df_build_node_grid(self.nodes_.data_ptr(), M, self.grid_.data_ptr(), _stream()))

    def _grid(self):
        return self.grid_.data_ptr() if self.grid_ is not None else None

    def setWarpToLive(self, pose):
        self.warp_to_live_ = pose

    def getNodes(self):
        return self.nodes_

    def KNN(self, points: torch.Tensor):
        N, stride = points.shape
        idx = torch.empty((N, 8), dtype=torch.int32, device=self.device)
        d2 = torch.empty((N, 8), dtype=torch.float32, device=self.device)
        capi.check(_lib().df_knn8(self.nodes_.data_ptr(), self.nodes_.shape[0], self._grid(), points.data_ptr(), N, stride, idx.data_ptr(),
                                  d2.data_ptr(), _stream()))
        return idx, d2

    def warp(self, points: torch.Tensor, normals: torch.Tensor, flags: int = 0, want_knn: bool = False):
        N, stride = points.shape
        idx = w = None
        if want_knn:
            idx = torch.empty((N, 8), dtype=torch.int32, device=self.device)
            w = torch.empty((N, 8), dtype=torch.float32, device=self.device)
        capi.check(_lib().df_warp(self.nodes_.data_ptr(), self.nodes_.shape[0], self._grid(), points.data_ptr(), normals.data_ptr(), N, stride,
                                  capi.make_aff(*self.warp_to_live_), flags, idx.data_ptr() if want_knn else None,
                                  w.data_ptr() if want_knn else None, _stream()))
        return idx, w

    def extend(self, cloud: torch.Tensor, radius: float, step: int = 50, max_nodes: int = 4096, count_dev: torch.Tensor | None = None) -> int:
        """Extending the warp field (dfusion.h df_extend_field; SURVEY 8f(3), Report.md step 4): append a node for every step-th point of
        the canonical cloud whose nearest node is farther than `radius`; rebuilds the node grid when nodes were added.  Returns the count."""
        M = self.nodes_.shape[0]
        cap, stride = cloud.shape
        table = torch.zeros((max_nodes, NODE_STRIDE), dtype=torch.float32, device=self.device)
        table[:M] = self.nodes_
        ws = torch.empty(_lib().df_extend_field_workspace_bytes(cap), dtype=torch.uint8, device=self.device)
        m_out = torch.zeros(1, dtype=torch.int32, device=self.device)
        capi.check(_lib().df_extend_field(table.data_ptr(), M, max_nodes, self._grid(), cloud.data_ptr(), cap,
                                          count_dev.data_ptr() if count_dev is not None else None, stride, float(radius), int(step),
                                          m_out.data_ptr(), ws.data_ptr(), _stream()))
        Mn = int(m_out.item())
        if Mn != M:
            self.setNodes(table[:Mn].clone())
        return Mn

    def optimiseWarpData(self, canonical: torch.Tensor, live: torch.Tensor, nonlinear_iters=5, linear_iters=100, flags=0):
        """WarpFieldOptimiser::optimiseWarpData (warp_field_optimiser.cpp:7-16) -> device LM/PCG"""
        N, stride = canonical.shape
        M = self.nodes_.shape[0]
        need = _lib().df_solve_workspace_bytes(M, N)
        if self._ws is None or self._ws.numel() < need:
            self._ws = torch.empty(need, dtype=torch.uint8, device=self.device)
        stats = torch.zeros(8, dtype=torch.float64, device=self.device)
        capi.check(_lib().df_solve_data_term(self.nodes_.data_ptr(), M, self._grid(), canonical.data_ptr(), live.data_ptr(), N, stride,
                                             nonlinear_iters, linear_iters, flags, stats.data_ptr(), self._ws.data_ptr(), _stream()))
        return stats

    def optimiseWarpF2(self, canonical: torch.Tensor, live: torch.Tensor, reg_lambda=0.0, tukey_c=0.01, huber_delta=1e-4, lm_mu=1e-4,
                       gn_iters=3, reg_k=4, flags=0, lin_iters=200):
        """df_solve_f2 (SURVEY 8f(2), opt-in): robust data term over 6-DoF node increments + regularisation; flags = DF_F2_TWIST (1) |
        DF_F2_TUKEY (2) | DF_F2_HUBER (4).  Nodes (rotation + dual part) are updated in place; returns the 16 stats (device tensor)."""
        import ctypes as C
        N, stride = canonical.shape
        M = self.nodes_.shape[0]
        prm = capi.F2Params(float(reg_lambda), float(tukey_c), float(huber_delta), float(lm_mu), int(gn_iters), int(reg_k), int(flags), int(lin_iters))
        ws = torch.empty(_lib().df_solve_f2_workspace_bytes(M, N, int(reg_k)), dtype=torch.uint8, device=self.device)
        stats = torch.zeros(16, dtype=torch.float64, device=self.device)
        capi.check(_lib().df_solve_f2(self.nodes_.data_ptr(), M, self._grid(), canonical.data_ptr(), live.data_ptr(), N, stride, C.byref(prm),
                                      stats.data_ptr(), ws.data_ptr(), _stream()))
        return stats
