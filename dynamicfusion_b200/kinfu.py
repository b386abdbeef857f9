"""KinFu / KinFuParams: Python host-side mirror of kfusion::KinFu (kfusion/include/kfusion/kinfu.hpp:15-97) over the
C ABI handle df_kinfu_* (include/dfusion.h).  The per-frame loop itself lives in libdfusion.so (csrc/pipeline.cu)."""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import capi

BUF = {"volume": 0, "dists": 1, "curr_depth": 2, "curr_points": 3, "curr_normals": 4, "prev_points": 5, "prev_normals": 6,
       "canonical": 7, "canonical_normals": 8, "cloud": 9, "cloud_normals": 10, "nodes": 11, "canonical_visible": 12,
       "solve_stats": 13, "activity": 14}
STAGES = ["preprocess", "icp", "raycast_canonical", "warp1", "solve", "warp2", "project_remove", "integrate", "extract", "raycast_prev"]

RIGID_ONLY = 1
STAGE_TIMING = 2
REF_GRAPH_QUIRK = 4
EXTEND_FIELD = 16         # DF_KINFU_EXTEND_FIELD: grow the warp field over unsupported canonical surface (SURVEY 8f(3))
F2_SOLVE = 32             # DF_KINFU_F2_SOLVE: robust 6-DoF data term + regulariser instead of the translation-only solve (SURVEY 8f(2))
USE_DEPTH = 64            # DF_KINFU_USE_DEPTH: the reference's compile-time USE_DEPTH frame loop (depth-pyramid ICP)
WARPED_INTEGRATE = 8      # DF_KINFU_WARPED_INTEGRATE: per-voxel warped fusion (SURVEY 8f(1)) instead of the rigid fallback
MESH_LIVE = 1             # DF_MESH_LIVE: df_kinfu_extract_mesh carries the mesh through the current warp field


class KinFuParams:
    """KinFuParams::default_params_dynamicfusion() / default_params() (kinfu.cpp:14-89)"""

    @staticmethod
    def default_params_dynamicfusion() -> capi.KinfuParams:
        p = capi.KinfuParams()
        capi.load().df_kinfu_default_params(C.byref(p), 0)
        return p

    @staticmethod
    def default_params() -> capi.KinfuParams:
        p = capi.KinfuParams()
        capi.load().df_kinfu_default_params(C.byref(p), 1)
        return p

    @staticmethod
    def set_volume(p: capi.KinfuParams, dim: int, size: float) -> None:
        for i in range(3):
            p.volume_dims[i] = dim
            p.volume_size[i] = size
        p.volume_pose.t[0] = -size / 2
        p.volume_pose.t[1] = -size / 2
        p.volume_pose.t[2] = 0.5


class KinFu:
    def __init__(self, params: capi.KinfuParams):
        if not torch.cuda.is_available():
            raise RuntimeError("dynamicfusion_b200.KinFu needs a CUDA device (sm_100a); there is no CPU fallback")
        self.lib = capi.load()
        self.params = params
        self.h = self.lib.df_kinfu_create(C.byref(params))
        if not self.h:
            raise RuntimeError("df_kinfu_create failed")
        self.lib.df_kinfu_set_stream(self.h, torch.cuda.current_stream().cuda_stream)

    def close(self):
        if getattr(self, "h", None):
            self.lib.df_kinfu_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def reset(self):
        capi.check(-self.lib.df_kinfu_reset(self.h))

    def __call__(self, depth) -> bool:
        """KinFu::operator()(depth).  depth: HOST numpy uint16 [rows, cols] (uploaded inside the call) or a DEVICE
        torch.int16 tensor [rows, cols]."""
        if isinstance(depth, np.ndarray):
            assert depth.dtype == np.uint16 and depth.flags.c_contiguous
            r = self.lib.df_kinfu_process_host(self.h, depth.ctypes.data, depth.strides[0])
        else:
            r = self.lib.df_kinfu_process_device(self.h, depth.data_ptr(), depth.stride(0) * 2)
        if r < 0:
            capi.check(-r)
        return bool(r)

    def process_host_ptr(self, ptr: int, pitch: int) -> int:
        return self.lib.df_kinfu_process_host(self.h, ptr, pitch)

    def getCameraPose(self, time: int = -1):
        out = (C.c_float * 12)()
        self.lib.df_kinfu_get_pose(self.h, time, out)
        a = np.array(list(out), np.float32)
        return a[:9].reshape(3, 3), a[9:]

    def info(self) -> dict:
        v = (C.c_longlong * 12)()
        self.lib.df_kinfu_get_info(self.h, v, 12)
        keys = ["frame_counter", "nodes", "cloud_points", "poses", "icp_ok", "launches", "resets", "lm_iters", "n_updated", "pcg_iters",
                "n_warped", "solve_overflows"]
        return dict(zip(keys, [int(x) for x in v]))

    def set_overrides(self, bilateral_depth=None, pose=None, nodes=None) -> None:
        """df_kinfu_set_overrides (lock-step parity hook): numpy u16 [rows, cols] / (R 3x3, t 3) / float32 [M, 12] for the next frame"""
        keep = []
        d = p12 = n = None
        M = 0
        if bilateral_depth is not None:
            b = np.ascontiguousarray(bilateral_depth, np.uint16); keep.append(b); d = b.ctypes.data
        if pose is not None:
            a = np.concatenate([np.asarray(pose[0], np.float32).reshape(9), np.asarray(pose[1], np.float32).reshape(3)]); keep.append(a); p12 = a.ctypes.data
        if nodes is not None:
            t = np.ascontiguousarray(nodes, np.float32); keep.append(t); n = t.ctypes.data; M = len(t)
        capi.check(self.lib.df_kinfu_set_overrides(self.h, d, (self.params.cols * 2), p12, n, M))

    def state_digest(self) -> list:
        """df_kinfu_state_digest: [volume checksum, node-table checksum, cloud points, pose-chain hash] (u64 each)"""
        v = (C.c_ulonglong * 4)()
        capi.check(self.lib.df_kinfu_state_digest(self.h, v))
        return [int(x) for x in v]

    def mesh(self, live: bool = False, normals: bool = True):
        """The current model as a triangle mesh (df_kinfu_extract_mesh): canonical, or carried into the live frame through the warp field
        (live=True; a rigid-only object, or one whose field does not exist yet, raises).  Leaves the object's state untouched.  Returns
        numpy (vertices [n, 3] float32, normals [n, 3] float32 or None, triangles [m, 3] int32, edge keys [n] uint32)."""
        vcap = max(int(self.params.cloud_capacity), 1024)
        tcap = 2 * vcap
        counts = (C.c_int * 2)()
        while True:
            v = torch.empty((vcap, 4), dtype=torch.float32, device="cuda")
            n = torch.empty((vcap, 4), dtype=torch.float32, device="cuda") if normals else None
            k = torch.empty(vcap, dtype=torch.int32, device="cuda")
            t = torch.empty((tcap, 3), dtype=torch.int32, device="cuda")
            capi.check(self.lib.df_kinfu_extract_mesh(self.h, MESH_LIVE if live else 0, v.data_ptr(), n.data_ptr() if normals else None,
                                                      k.data_ptr(), vcap, t.data_ptr(), tcap, counts))
            if counts[0] <= vcap and counts[1] <= tcap:
                break
            vcap, tcap = max(vcap, counts[0]), max(tcap, counts[1])     # the counts are true totals: one more call fits
        nv, nt = counts[0], counts[1]
        return (v[:nv, :3].cpu().numpy(), n[:nv, :3].cpu().numpy() if normals else None, t[:nt].cpu().numpy(),
                k[:nv].cpu().numpy().view(np.uint32))

    def stage_ms(self) -> dict:
        v = (C.c_float * 10)()
        n = self.lib.df_kinfu_get_stage_ms(self.h, v, 10)
        return dict(zip(STAGES[:n], [float(x) for x in v][:n]))

    def buffer(self, name: str) -> np.ndarray:
        """copy a device buffer of the current state to the host as numpy (tests/diagnostics)"""
        ptr, pitch, cols, rows = C.c_void_p(), C.c_size_t(), C.c_int(), C.c_int()
        capi.check(self.lib.df_kinfu_get_buffer(self.h, BUF[name], C.byref(ptr), C.byref(pitch), C.byref(cols), C.byref(rows)))
        nbytes = pitch.value * rows.value
        if nbytes == 0:
            return np.zeros(0, np.uint8)
        raw = np.empty(nbytes, np.uint8)
        capi.check(self.lib.df_kinfu_read_buffer(self.h, BUF[name], raw.ctypes.data, nbytes))
        p = self.params
        if name == "volume":
            return raw.view(np.uint32)
        if name in ("dists", "curr_depth"):
            return raw.view(np.uint16).reshape(p.rows, p.cols)
        if name in ("cloud", "cloud_normals"):
            n = self.info()["cloud_points"]
            return raw.view(np.float32).reshape(-1, 4)[:n].copy()
        if name == "nodes":
            return raw.view(np.float32).reshape(-1, 12)
        if name == "solve_stats":
            return raw.view(np.float64)
        return raw.view(np.float32).reshape(p.rows, p.cols, 4)
