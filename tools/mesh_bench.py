"""Mesh extraction cost on the flagship model (one B200): runs bench.py's synthetic sequence (512^3 TSDF over 1 m^3, 640x480 depth,
2048 warp nodes) to bench.py's last default frame, then times with CUDA events (warm-up, then the median of --reps repetitions):
  cloud     df_extract_cloud_tracked + df_extract_normals (what the frame loop extracts; the baseline)
  mesh      df_extract_mesh (no normals)
  mesh_n    df_extract_mesh + df_extract_normals at the vertices
each with and without the volume's activity map, and
  kinfu_canonical / kinfu_live   df_kinfu_extract_mesh (normals on; synchronous: includes its count read-back, and the warp for live).
Prints one JSON line with the device name and power limit, the vertex / triangle counts and the bytes the algorithm reads: the voxels
of the stretches it scans, each once (every stretch without the map, the active ones with it), plus the map.

    python tools/mesh_bench.py [--frames 70] [--reps 60] [--out FILE]
"""
from __future__ import annotations

import argparse
import json
import subprocess
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))

DIM, SIZE, COLS, ROWS, MAX_NODES = 512, 1.0, 640, 480, 2048     # bench.py's configuration


def gpu_identity():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clock = [s.strip() for s in out.split(",")]
        return {"device": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:                                         # the device name from torch is still recorded
        return {"nvidia_smi_error": str(e)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--frames", type=int, default=70, help="frames of the sequence to run first (bench.py's defaults end at frame 69)")
    ap.add_argument("--reps", type=int, default=60)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", type=Path)
    args = ap.parse_args()
    assert args.reps >= 50

    import torch
    from dynamicfusion_b200 import capi, kinfu as kf, synth
    assert torch.cuda.is_available(), "mesh_bench.py needs a CUDA device"
    lib = capi.load()

    p = kf.KinFuParams.default_params_dynamicfusion()
    kf.KinFuParams.set_volume(p, DIM, SIZE)
    p.max_nodes = MAX_NODES
    p.cloud_capacity = 4_000_000
    k = kf.KinFu(p)
    for t in range(args.frames):
        depth = torch.from_numpy(synth.umbrella_depth(t, seed=0).view(np.int16).copy()).cuda()
        lib.df_kinfu_process_device(k.h, depth.data_ptr(), COLS * 2)
    info = k.info()                                                # waits for the frame's extraction
    torch.cuda.synchronize()

    import ctypes as C
    ptr, pitch, cols, rows = C.c_void_p(), C.c_size_t(), C.c_int(), C.c_int()
    capi.check(lib.df_kinfu_get_buffer(k.h, 0, C.byref(ptr), C.byref(pitch), C.byref(cols), C.byref(rows)))
    vol_ptr = ptr.value
    capi.check(lib.df_kinfu_get_buffer(k.h, 14, C.byref(ptr), C.byref(pitch), C.byref(cols), C.byref(rows)))
    act_ptr, act_bytes = ptr.value, cols.value
    vs = SIZE / DIM
    vol = capi.make_volume(vol_ptr, (DIM,) * 3, (vs,) * 3, max(p.tsdf_trunc_dist, 2.1 * vs), p.tsdf_max_weight)
    pose = p.volume_pose
    Rinv = capi.f9(np.linalg.inv(np.array(pose.R, np.float64).reshape(3, 3)).astype(np.float32))
    stream = torch.cuda.current_stream().cuda_stream

    cap = 4_000_000
    cloud = torch.empty((cap, 4), dtype=torch.float32, device="cuda")
    cloud_n = torch.empty_like(cloud)
    count = torch.zeros(1, dtype=torch.int32, device="cuda")
    ews = torch.empty(lib.df_extract_workspace_bytes(vol), dtype=torch.uint8, device="cuda")
    verts = torch.empty((cap, 4), dtype=torch.float32, device="cuda")
    vnrm = torch.empty_like(verts)
    keys = torch.empty(cap, dtype=torch.int32, device="cuda")
    tcap = 2 * cap
    tris = torch.empty((tcap, 3), dtype=torch.int32, device="cuda")
    counts = torch.zeros(2, dtype=torch.int32, device="cuda")
    mws = torch.empty(lib.df_extract_mesh_workspace_bytes(vol), dtype=torch.uint8, device="cuda")

    def cloud_call(act):
        capi.check(lib.df_extract_cloud_tracked(vol, pose, cloud.data_ptr(), cap, count.data_ptr(), ews.data_ptr(), act, stream))
        capi.check(lib.df_extract_normals(vol, cloud.data_ptr(), cap, count.data_ptr(), pose, Rinv, p.gradient_delta_factor, cloud_n.data_ptr(), stream))

    def mesh_call(act, normals=False):
        capi.check(lib.df_extract_mesh(vol, pose, act, verts.data_ptr(), keys.data_ptr(), cap, tris.data_ptr(), tcap, counts.data_ptr(),
                                       mws.data_ptr(), stream))
        if normals:
            capi.check(lib.df_extract_normals(vol, verts.data_ptr(), cap, counts.data_ptr(), pose, Rinv, p.gradient_delta_factor,
                                              vnrm.data_ptr(), stream))

    host_counts = (C.c_int * 2)()

    def kinfu_call(flags):
        capi.check(lib.df_kinfu_extract_mesh(k.h, flags, verts.data_ptr(), vnrm.data_ptr(), keys.data_ptr(), cap, tris.data_ptr(), tcap, host_counts))

    def time_ms(fn):
        for _ in range(args.warmup):
            fn()
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2 * args.reps)]
        for i in range(args.reps):
            ev[2 * i].record()
            fn()
            ev[2 * i + 1].record()
        torch.cuda.synchronize()
        t = np.array([ev[2 * i].elapsed_time(ev[2 * i + 1]) for i in range(args.reps)])
        return {"median_ms": float(np.median(t)), "min_ms": float(t.min()), "max_ms": float(t.max())}

    cases = {}
    for tag, act in (("tracked", act_ptr), ("full", None)):       # alternate the variants inside one process
        cases[f"cloud_{tag}"] = time_ms(lambda: cloud_call(act))
        cases[f"mesh_{tag}"] = time_ms(lambda: mesh_call(act))
        cases[f"mesh_n_{tag}"] = time_ms(lambda: mesh_call(act, True))
    cases["kinfu_canonical"] = time_ms(lambda: kinfu_call(0))
    cases["kinfu_live"] = time_ms(lambda: kinfu_call(1))

    mesh_call(act_ptr)
    torch.cuda.synchronize()
    nv, nt = (int(c) for c in counts.cpu().numpy())
    npts = int(count.item())
    act_host = np.empty(act_bytes, np.uint8)
    capi.check(lib.df_kinfu_read_buffer(k.h, 14, act_host.ctypes.data, act_bytes))
    nvox = DIM ** 3
    nstretch = (nvox + 1023) // 1024
    active = int(np.count_nonzero(act_host[:nstretch]))
    bytes_full = 4 * nvox
    bytes_tracked = 4 * 1024 * active + nstretch
    line = {
        "tool": "tools/mesh_bench.py", "workload": f"bench.py sequence to frame {args.frames - 1}: {DIM}^3 TSDF / {SIZE} m^3, {COLS}x{ROWS} depth",
        "torch_device": torch.cuda.get_device_name(0), **gpu_identity(), "reps": args.reps, "nodes": info["nodes"],
        "cloud_points": npts, "mesh_vertices": nv, "mesh_triangles": nt, "active_stretches": active, "stretches": nstretch,
        "algorithmic_read_bytes": {"full": bytes_full, "tracked": bytes_tracked},
        "write_bytes": {"cloud+normals": 32 * npts, "mesh": 20 * nv + 12 * nt, "mesh+normals": 36 * nv + 12 * nt},
        "times": cases,
        "ratio_mesh_over_cloud_tracked": cases["mesh_tracked"]["median_ms"] / cases["cloud_tracked"]["median_ms"],
        "ratio_mesh_n_over_cloud_tracked": cases["mesh_n_tracked"]["median_ms"] / cases["cloud_tracked"]["median_ms"],
    }
    k.close()
    text = json.dumps(line)
    print(text, flush=True)
    if args.out:
        args.out.parent.mkdir(parents=True, exist_ok=True)
        args.out.write_text(text + "\n")


if __name__ == "__main__":
    main()
