#!/usr/bin/env python
"""bench.py -- frames/s of the DynamicFusion per-frame hot path at BASELINE.json's quoted configuration
(configs[1]: synthetic "umbrella" sequence, 640x480 depth, 512^3 TSDF over 1 m^3, ~2k warp nodes, full
preprocess -> ICP -> raycast -> k-NN/DQB warp -> data-term solve -> warp -> project/remove -> integrate -> extract ->
raycast loop on one B200).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

A "step" is one frame.  N > 1 (under torchrun, one rank per GPU): every rank runs an independent sequence (seed = rank,
config 5): weak scaling, no data-path collective; timing is the max over ranks.

One JSON line is printed by rank 0.  `value` = frames/s with the depth frames already resident in HBM; `e2e` = the same
through the reference-facing call with HOST depth buffers (df_kinfu_process_host: H2D of the frame and D2H of the
ICP status + pose inside the timed region); `roofline` = the integrate kernel's algorithmic bytes / its CUDA-event
duration against the measured HBM copy bandwidth; `cpu_baseline` = the CPU oracle's restated loop on the same workload.
--impl reference times that CPU restatement (the reference itself cannot be built here: CUDA 12.9 dropped texture
references, OpenCV/Opt/Terra/Ceres are absent -- see DESIGN.md) with all host threads.
"""
from __future__ import annotations

import os
# OpenMP (the CPU oracle of the cpu_baseline / --impl reference legs): idle workers sleep instead of spinning -- on a box whose
# cgroup CPU quota is smaller than the visible CPU count, spinning workers burn the quota and the run thrashes (round 1:
# 0.08 frames/s on 128 threads vs 0.36 on ONE).  Must be in the environment before libgomp is loaded.
os.environ.setdefault("OMP_WAIT_POLICY", "passive")
os.environ.setdefault("OMP_PROC_BIND", "false")
os.environ.setdefault("OMP_DYNAMIC", "false")

import argparse
import json
import statistics
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

DIM, SIZE, COLS, ROWS, MAX_NODES = 512, 1.0, 640, 480, 2048
WORKLOAD = "C2 synthetic umbrella sequence: 640x480 u16 depth, 512^3 TSDF / 1 m^3, ~2k warp nodes, full per-frame loop"
METRIC = "frames/sec @512^3 TSDF, 640x480 depth (full warp+integrate+raycast loop)"


def measured_peaks():
    f = ROOT / "MEASURED_PEAKS.json"
    if f.exists():
        try:
            return float(json.loads(f.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region"""
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None
        self.t0 = self.t1 = None

    def mark_begin(self):
        self.t0 = time.perf_counter()

    def mark_end(self):
        self.t1 = time.perf_counter()

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "10"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), [c.strip() for c in line.split(",")]))

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        # the sampler is started before the warm-up frames (nvidia-smi needs ~0.3 s to emit its first line); only the samples that
        # arrived between mark_begin() and mark_end() -- i.e. while the timed frames were executing -- are reported.  A timed
        # region shorter than the sampling period falls back to the samples within 0.25 s around it and says so.
        inside = [r for (t, r) in self.rows if self.t0 is not None and self.t0 <= t <= (self.t1 or t)]
        note = None
        if not inside and self.t0 is not None:
            inside = [r for (t, r) in self.rows if self.t0 - 0.25 <= t <= (self.t1 or t) + 0.25]
            note = "timed region shorter than the sampling period: samples within 0.25 s of it"
        sm = [float(r[0]) for r in inside if len(r) >= 6 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in inside if len(r) >= 6 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in inside if len(r) >= 6 for n, v in zip(names, r[2:6]) if v.lower().startswith("active")})
        out = {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons, "samples": len(sm)}
        if note:
            out["note"] = note
        return out


def dram_traffic_probe(frames: int, timeout_s: float = 240.0):
    """DRAM bytes per launch of the integrate and ray-cast kernels, measured NOW on this GPU: one extra process runs the same sequence
    (tools/traffic_probe.py) under `ncu --metrics dram__bytes_read.sum,dram__bytes_write.sum` restricted to those kernels; the launches of
    the last three frames are averaged.  Returns {kernel_name: {"read": B, "write": B, "launches": n}} or {"error": ...}."""
    import csv
    import shutil
    import tempfile
    ncu = shutil.which("ncu") or ("/usr/local/cuda/bin/ncu" if Path("/usr/local/cuda/bin/ncu").exists() else None)
    if not ncu:
        return {"error": "ncu not found"}
    with tempfile.TemporaryDirectory() as td:
        log = Path(td) / "traffic.csv"
        cmd = [ncu, "--metrics", "dram__bytes_read.sum,dram__bytes_write.sum", "--clock-control", "none", "--print-units", "base", "--csv",
               "--kernel-name", "regex:integrate_kernel|raycast_points_kernel", "--log-file", str(log),
               sys.executable, str(ROOT / "tools" / "traffic_probe.py"), "--frames", str(frames), "--dim", str(DIM), "--max-nodes", str(MAX_NODES)]
        try:
            r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=timeout_s, cwd=str(ROOT))
        except Exception as e:
            return {"error": repr(e)}
        if r.returncode != 0 or not log.exists():
            return {"error": f"ncu rc {r.returncode}: {r.stdout[-300:]}"}
        rows = [l for l in log.read_text().splitlines() if l.startswith('"')]
        per = {}                                                 # (id, kernel) -> {metric: value}
        for rec in csv.DictReader(rows):
            try:
                key = (int(rec["ID"]), rec["Kernel Name"].split("(")[0].split("<")[0].strip())
                per.setdefault(key, {})[rec["Metric Name"]] = float(rec["Metric Value"].replace(",", ""))
            except Exception:
                continue
        out = {}
        for name in sorted({k[1] for k in per}):
            launches = [per[k] for k in sorted(per) if k[1] == name]
            tail = launches[-(3 if "integrate" in name else 6):]  # last three frames: 1 integrate, 2 ray-casts per frame
            out[name] = {"read": sum(x.get("dram__bytes_read.sum", 0.0) for x in tail) / len(tail),
                         "write": sum(x.get("dram__bytes_write.sum", 0.0) for x in tail) / len(tail), "launches": len(launches)}
        return out or {"error": "no matching kernel in the ncu log"}


def make_frames(n: int, seed: int):
    from dynamicfusion_b200 import synth
    return np.stack([synth.umbrella_depth(t, seed=seed) for t in range(n)])


def cpu_params():
    from oracle import orc_pipe
    p = orc_pipe.default_params(0, dim=DIM, size=SIZE)
    p.max_nodes = MAX_NODES
    p.cloud_capacity = 4_000_000
    return p


def run_cpu(frames: np.ndarray, lead: int, steps: int, calibrate=None):
    """the oracle's restated per-frame loop on the host cores; frame 0 initialises, then `lead` untimed frames (lead-in + warm-up),
    then `steps` timed.  calibrate: optional list of OpenMP thread counts tried on the first untimed frames (one each); the fastest is
    kept for the rest of the run.  Returns (seconds, info, per-frame seconds, threads used, calibration record)."""
    from oracle import orc, orc_pipe
    orc.build()
    k = orc_pipe.KinFu(cpu_params())
    k(frames[0])
    calib, used = {}, None
    cands = list(calibrate or [])
    if cands:
        set_omp_threads(cands[0])
    preroll = 1 if lead > len(cands) else 0        # frame 1 pays first-touch page faults: keep it out of the calibration when there is room
    for t in range(1, 1 + lead):
        if cands and t > preroll:
            c = cands.pop(0)
            set_omp_threads(c)
            t0 = time.perf_counter()
            k(frames[t])
            calib[c] = time.perf_counter() - t0
            if not cands:
                used = min(calib, key=calib.get)
                set_omp_threads(used)
        else:
            k(frames[t])
    per = []
    t0 = time.perf_counter()
    for t in range(1 + lead, 1 + lead + steps):
        t1 = time.perf_counter()
        k(frames[t])
        per.append(time.perf_counter() - t1)
    dt = time.perf_counter() - t0
    info = k.info()
    k.close()
    return dt, info, per, used, calib


_gomp = None


def set_omp_threads(n: int):
    """omp_set_num_threads on the libgomp the oracle links (also overrides torchrun's OMP_NUM_THREADS=1); per calling thread"""
    global _gomp
    import ctypes
    if _gomp is None:
        _gomp = ctypes.CDLL("libgomp.so.1")
    _gomp.omp_set_num_threads(int(max(1, n)))


def host_cpus():
    """(CPUs in the affinity mask, cgroup CPU quota in cores or None): the quota, not the mask, is what the process can use"""
    try:
        aff = len(os.sched_getaffinity(0))
    except Exception:
        aff = os.cpu_count() or 1
    quota = None
    try:                                            # cgroup v2
        q, per = Path("/sys/fs/cgroup/cpu.max").read_text().split()[:2]
        if q != "max":
            quota = float(q) / float(per)
    except Exception:
        pass
    if quota is None:
        try:                                        # cgroup v1
            q = int(Path("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read_text())
            per = int(Path("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read_text())
            if q > 0 and per > 0:
                quota = q / per
        except Exception:
            pass
    return aff, quota


def host_threads():
    """threads the CPU legs start from: the cgroup quota capped by the affinity mask (then refined by calibration)"""
    aff, quota = host_cpus()
    n = aff if quota is None else max(1, min(aff, int(quota + 0.999)))
    return n


def thread_candidates():
    """thread counts tried on the first untimed frames: quota/affinity-derived count, then halves -- a box that lies about its CPUs
    (affinity 128, real share far smaller) shows up as the smaller counts being FASTER, and the fastest is used"""
    n = host_threads()
    c = [n]
    while c[-1] > 4 and len(c) < 4:
        c.append(max(4, c[-1] // 2))
    return c


def frame_stats_ms(per_s):
    v = sorted(1000.0 * x for x in per_s)
    return {"min": v[0], "median": v[len(v) // 2], "max": v[-1]} if v else None


def integrate_kernel_name():
    """the integrate kernel the frame loop's last call launched (df_integrate_last_kernel: the packed-arithmetic kernel falls back to
    the scalar culling kernel when a launch is outside its checked domain)"""
    from dynamicfusion_b200 import capi
    code = capi.load().df_integrate_last_kernel()
    return {5: "integrate_kernel_v5", 3: "integrate_kernel_v3"}.get(code, "integrate_kernel<4>")


def dump_outputs(k, out_dir: Path, max_points: int = 1 << 20, volume_samples: int = 1 << 20):
    """what the last timed frame left for a caller of the frame loop, as DIR/<name>.npy (float32, under 64 MB in all): the camera
    pose [R | t], the ray-cast point / normal maps, the warp nodes, the canonical cloud and its normals (rows sorted by their bit
    patterns, since extraction appends in no fixed order; a seeded sample of `max_points` rows if larger) and a seeded sample of
    `volume_samples` voxels of the TSDF (value and weight).  The ray-cast maps and the cloud normals mark "no hit" / "no normal"
    with NaN: they are written with 0 in place of every non-finite value, and <name>_valid.npy holds 1 for each row (pixel, point)
    whose values are all finite, 0 otherwise.  Same arguments, same inputs, same sample: two builds compare output for output."""
    out_dir.mkdir(parents=True, exist_ok=True)
    R, t = k.getCameraPose()
    arrays = {"camera_pose": np.concatenate([R, t[:, None]], axis=1), "raycast_points": k.buffer("prev_points"),
              "raycast_normals": k.buffer("prev_normals"), "warp_nodes": k.buffer("nodes")[: k.info()["nodes"]]}
    cloud, normals = k.buffer("cloud"), k.buffer("cloud_normals")
    order = np.lexsort(np.ascontiguousarray(cloud).view(np.uint32).T[::-1])
    if len(order) > max_points:
        order = order[np.sort(np.random.default_rng(0).choice(len(order), max_points, replace=False))]
    arrays["cloud_points"], arrays["cloud_normals"] = cloud[order], normals[order]
    vol = k.buffer("volume")
    vox = np.sort(np.random.default_rng(1).integers(0, vol.size, volume_samples))
    arrays["volume_tsdf_sample"] = (vol[vox] & 0xFFFF).astype(np.uint16).view(np.float16).astype(np.float32)
    arrays["volume_weight_sample"] = (vol[vox] >> 16).astype(np.float32)
    for name in ("raycast_points", "raycast_normals", "cloud_normals"):
        finite = np.isfinite(arrays[name])
        arrays[f"{name}_valid"] = finite.all(axis=-1)
        arrays[name] = np.where(finite, arrays[name], np.float32(0))
    for name, a in arrays.items():
        a = np.ascontiguousarray(a, np.float32)
        if not np.isfinite(a).all():
            raise ValueError(f"--dump-outputs: {name} holds non-finite values")
        np.save(out_dir / f"{name}.npy", a)


def bench_config(world: int, first: int, K: int):
    """the SAME dict in both arms (the driver compares them): workload + the timed window, nothing measured"""
    return {"workload": WORKLOAD, "node_cap": MAX_NODES, "knn": 8, "solver": "LM 5 x PCG 100 (early-out)", "sequences": world,
            "parallelism": f"{world} independent sequences" if world > 1 else "single sequence",
            "timed_frames": [first, first + K],
            "l2": "working set (512 MiB volume, re-read every frame) exceeds the 126 MB L2; no explicit flush"}


def reference_arm(args, rank, world):
    """--impl reference: the reference's CPU implementation of the path = the oracle port (the reference itself cannot be built here,
    DESIGN.md 5) on the box's host cores.  Same frames, same timed window, same --steps/--warmup as the GPU arm.  At N > 1 rank 0 runs
    N sequences concurrently (seeds 0..N-1, the host threads split between them), so that `value` counts the same N*K frames as
    the GPU arm's."""
    if rank != 0:
        return
    K, W = args.steps, args.warmup
    first = max(args.frames_from, 1 + W)
    lead = first - 1
    aff, quota = host_cpus()
    cands = thread_candidates()
    if lead < len(cands):
        cands = cands[:max(lead, 1)]
    t_wall0 = time.perf_counter()
    passes = []
    if world == 1:
        frames = make_frames(1 + lead + K, 0)
        dt, info, per, used, calib = run_cpu(frames, lead, K, calibrate=cands)
        passes.append((dt, per))
        # second pass of the same frames (best + spread) if the first left room in the few-minutes budget
        if time.perf_counter() - t_wall0 < 100.0:
            dt2, info, per2, _, _ = run_cpu(frames, lead, K, calibrate=[used])
            passes.append((dt2, per2))
        nseq = 1
    else:
        # N concurrent sequences: calibrate the total thread count on sequence 0's first frames, then one host thread per sequence
        import threading as th
        frames0 = make_frames(1 + len(cands), 0)
        _, _, _, used_total, calib = run_cpu(frames0, len(cands), 0, calibrate=cands)
        per_seq = max(1, used_total // world)
        results = [None] * world

        def one(i):
            set_omp_threads(per_seq)
            fr = make_frames(1 + lead + K, i)
            results[i] = (fr,)
        ts = [th.Thread(target=one, args=(i,)) for i in range(world)]
        [t.start() for t in ts]; [t.join() for t in ts]
        start = th.Barrier(world)

        def run(i):
            set_omp_threads(per_seq)
            from oracle import orc_pipe
            k = orc_pipe.KinFu(cpu_params())
            fr = results[i][0]
            for t in range(0, 1 + lead):
                k(fr[t])
            start.wait()
            t0 = time.perf_counter()
            per = []
            for t in range(1 + lead, 1 + lead + K):
                t1 = time.perf_counter(); k(fr[t]); per.append(time.perf_counter() - t1)
            results[i] = (time.perf_counter() - t0, per, k.info())
            k.close()
        ts = [th.Thread(target=run, args=(i,)) for i in range(world)]
        [t.start() for t in ts]; [t.join() for t in ts]
        dt = max(r[0] for r in results)
        per = [x for r in results for x in r[1]]
        info = results[0][2]
        passes.append((dt, per))
        used, nseq = per_seq, world
    best_dt, best_per = min(passes, key=lambda q: q[0])
    fps = nseq * K / best_dt
    all_fps = [nseq * K / q[0] for q in passes]
    spread = (max(all_fps) - min(all_fps)) / max(all_fps) if len(all_fps) > 1 else None
    sample = (f"{K} timed frames per sequence x {nseq} sequence(s) (+1 init, +{lead} untimed incl. {W} warm-up) of the same 512^3 workload, "
              f"OpenMP {used} threads per sequence, best of {len(passes)} pass(es)")
    line = {"impl": "reference", "metric": METRIC, "value": fps, "unit": "frames/s", "n_gpus": args.gpus, "steps": K, "warmup": W,
            "ms_per_step": 1000.0 * best_dt / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32 (f16/u16 volume)",
            "data": "synthetic", "config": bench_config(world, first, K),
            "note": "CPU restatement (oracle port, OpenMP): the reference's own CUDA/Opt/OpenCV build is not possible in this image (DESIGN.md 5)",
            "run_info": {"nodes": info["nodes"], "cloud_points": info["cloud_points"]},
            "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": used * nseq, "kind": "port", "sample": sample,
                             "affinity_cpus": aff, "cgroup_quota_cpus": quota, "thread_calibration_s_per_frame": {str(c): v for c, v in calib.items()},
                             "passes_fps": all_fps, "spread": spread, "per_sequence_fps": fps / nseq},
            "frame_ms": frame_stats_ms(best_per),
            "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=60)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--roofline-frames", type=int, default=12)
    ap.add_argument("--no-warped", action="store_true", help="skip the short pass through the per-voxel warped fusion variant (SURVEY 8f(1))")
    ap.add_argument("--frames-from", type=int, default=10, help="first TIMED frame of the sequence (SURVEY 8d: steady state = frames 10-99): frame 0 "
                    "initialises, frames 1..F-1 are untimed (the last W of them are the warm-up steps), frames F..F+K-1 are timed")
    ap.add_argument("--no-traffic-probe", action="store_true", help="do not run the one-launch ncu pass that measures the integrate / ray-cast DRAM bytes")
    ap.add_argument("--dump-outputs", metavar="DIR", type=Path, help="write what the last timed frame computed (device-resident arm, rank 0) "
                    "as DIR/<name>.npy")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3)

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        reference_arm(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    from dynamicfusion_b200 import distrib, kinfu as kf

    assert torch.cuda.is_available(), "bench.py needs a CUDA device"
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    distrib.init("nccl", device)

    def barrier():
        distrib.barrier(device)

    K, W = args.steps, args.warmup
    first = max(args.frames_from, 1 + W)                              # first timed frame; frames 1..first-1 untimed (lead-in + W warm-up)
    nframes = first + K
    frames = make_frames(nframes, seed=distrib.sequence_seed(rank))   # independent sequence per rank (config 5)
    frames_i16 = torch.from_numpy(frames.view(np.int16))
    frames_dev = frames_i16.cuda()
    frames_pinned = frames_i16.pin_memory()

    def params(flags=0):
        p = kf.KinFuParams.default_params_dynamicfusion()
        kf.KinFuParams.set_volume(p, DIM, SIZE)
        p.max_nodes = MAX_NODES
        p.cloud_capacity = 4_000_000
        p.flags = flags
        return p

    def timed(run_frame, dump_dir=None):
        """frame 0 + the untimed frames 1..first-1 (the last W = warm-up), then exactly K frames between barrier+sync, CUDA events on the
        launching stream (one event per frame: the whole-region time is ev[0] -> ev[K], the per-frame spread comes for free)"""
        sampler = ClockSampler(local_rank)
        sampler.start()
        k = kf.KinFu(params())
        ok = 0
        for t in range(first):
            run_frame(k, t)
        barrier()
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(K + 1)]
        sampler.mark_begin()
        k.lib.df_kinfu_join(k.h)                                  # the warm-up's overlapped extraction ends before the timed region starts
        ev[0].record()
        for i, t in enumerate(range(first, first + K)):
            ok += run_frame(k, t)
            if i == K - 1:
                k.lib.df_kinfu_join(k.h)                          # ... and the last timed frame's extraction ends inside it
            ev[i + 1].record()
        barrier()
        sampler.mark_end()
        clocks = sampler.stop()
        ms = ev[0].elapsed_time(ev[K])
        per = [ev[i].elapsed_time(ev[i + 1]) * 1e-3 for i in range(K)]
        info = k.info()
        Rf, tf = k.getCameraPose()
        digest = {"digest": k.state_digest(), "pose": [float(x) for x in Rf.reshape(9)] + [float(x) for x in tf]}
        if dump_dir is not None and rank == 0:
            dump_outputs(k, dump_dir)
        k.close()
        ms, _total, ok = distrib.aggregate(ms, ok, device)       # max time over ranks; ok = fewest fused frames on any rank
        return ms, ok, info, clocks, per, digest

    pitch = COLS * 2
    # value: inputs already resident in HBM
    ms_dev, ok_dev, info, clocks, per_dev, digest_dev = timed(lambda k, t: k.lib.df_kinfu_process_device(k.h, frames_dev[t].data_ptr(), pitch),
                                                              args.dump_outputs)
    # e2e: the reference-facing call with HOST buffers (pinned), H2D + D2H inside the timed region
    ms_e2e, ok_e2e, _, clocks_e2e, per_e2e, digest_e2e = timed(lambda k, t: k.lib.df_kinfu_process_host(k.h, frames_pinned[t].data_ptr(), pitch))
    assert ok_dev == K and ok_e2e == K, f"tracking was lost during the timed region ({ok_dev}/{ok_e2e} of {K} frames fused)"

    # roofline of the dominant kernel (integrate): per-stage CUDA events + voxels written, on a separate short pass
    k = kf.KinFu(params(kf.STAGE_TIMING))
    stage_acc, nupd_acc, nroof = {}, 0, 0
    for t in range(min(nframes, first + args.roofline_frames)):          # the stage times are those of the timed window's frames
        k.lib.df_kinfu_process_device(k.h, frames_dev[t].data_ptr(), pitch)
        if t >= first:
            for name, v in k.stage_ms().items():
                stage_acc[name] = stage_acc.get(name, 0.0) + v
            nupd_acc += k.info()["n_updated"]
            nroof += 1
    # ray-cast roofline (the metric names integrate + ray-cast): re-run the frame's last ray-cast on the final volume with the counting
    # instantiation of the kernel (df_raycast_points_stats) to get U = unique voxels read; its time is the stage's CUDA-event time
    raycast_info = None
    try:
        import ctypes as C
        from dynamicfusion_b200 import capi, host
        ptr, pitch_, c_, r_ = C.c_void_p(), C.c_size_t(), C.c_int(), C.c_int()
        capi.check(k.lib.df_kinfu_get_buffer(k.h, kf.BUF["volume"], C.byref(ptr), C.byref(pitch_), C.byref(c_), C.byref(r_)))
        view = host.TsdfVolume.__new__(host.TsdfVolume)
        view.device, view.activity_, view._ws, view._proj_ws = device, None, None, None
        view.dims_ = np.array([DIM] * 3, np.int32)
        view.size_ = np.array([SIZE] * 3, np.float32)
        view.trunc_dist_ = max(0.04, 2.1 * SIZE / DIM)
        view.max_weight_ = 64
        view.pose_ = (np.eye(3, dtype=np.float32), np.array([-SIZE / 2, -SIZE / 2, 0.5], np.float32))
        view.raycast_step_factor_, view.gradient_delta_factor_ = 0.75, 0.5
        view._vol = lambda: capi.make_volume(ptr.value, view.dims_, view.getVoxelSize(), view.trunc_dist_, view.max_weight_)
        st = view.raycast_stats(k.getCameraPose(), (570.342, 570.342, 320.0, 240.0), COLS, ROWS, activity_ptr=0)
        raycast_info = {kk: st[kk] for kk in ("unique_voxels", "hit_rays", "march_samples", "algorithmic_bytes")}
        # what the frame loop's brick-skipping march (df_raycast_points_tracked) actually fetches, same maps
        aptr = C.c_void_p()
        capi.check(k.lib.df_kinfu_get_buffer(k.h, kf.BUF["activity"], C.byref(aptr), C.byref(pitch_), C.byref(c_), C.byref(r_)))
        st2 = view.raycast_stats(k.getCameraPose(), (570.342, 570.342, 320.0, 240.0), COLS, ROWS, activity_ptr=aptr.value)
        raycast_info["unique_voxels_tracked"] = st2["unique_voxels"]
    except Exception as e:                                                      # informational: never lose the headline line
        raycast_info = {"error": repr(e)}
    k.close()
    stage_ms = {n: v / max(nroof, 1) for n, v in stage_acc.items()}
    n_upd = nupd_acc / max(nroof, 1)
    peak, peak_src = measured_peaks()
    alg_bytes = 8.0 * n_upd + 2.0 * COLS * ROWS                # SURVEY 8d: 4 B read + 4 B write per updated voxel + the fp16 dists image
    integ_ms = stage_ms.get("integrate", float("nan"))
    achieved = alg_bytes / (integ_ms * 1e-3) / 1e9 if integ_ms and integ_ms > 0 else float("nan")
    # DRAM traffic of the two kernels, measured in THIS run (one ncu pass over the same sequence, rank 0 at N = 1); the committed
    # capture (profiles/integrate_traffic.json) is only the fallback when ncu is unavailable
    traffic, traffic_rc, traffic_src, probe = None, None, None, None
    if rank == 0 and world == 1 and not args.no_traffic_probe:
        probe = dram_traffic_probe(min(nframes, first + 3))
        for name, v in probe.items():
            if isinstance(v, dict) and "integrate" in name:
                traffic, traffic_src = v["read"] + v["write"], f"live ncu pass ({name}, dram__bytes_read.sum + dram__bytes_write.sum, mean of the last 3 launches)"
            if isinstance(v, dict) and "raycast" in name:
                traffic_rc = v["read"] + v["write"]
    if traffic is None:
        tf = ROOT / "profiles" / "integrate_traffic.json"
        if tf.exists():
            try:
                traffic = json.loads(tf.read_text()).get("dram_bytes_per_launch")
                traffic_src = "committed capture profiles/integrate_traffic.json (live probe unavailable: %s)" % ((probe or {}).get("error", "not run"))
            except Exception:
                traffic = None

    total_frames = K * world
    fps = total_frames / (ms_dev * 1e-3)
    fps_e2e = total_frames / (ms_e2e * 1e-3)
    line = {
        "metric": METRIC, "value": fps, "unit": "frames/s", "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": ms_dev / K,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32 (f16/u16 volume)", "data": "synthetic",
        "config": bench_config(world, first, K),
        "run_info": {"nodes": info["nodes"], "cloud_points": info["cloud_points"]},
        "frame_ms": frame_stats_ms(per_dev),
        "e2e": {"value": fps_e2e, "unit": "frames/s", "h2d_bytes_per_step": COLS * ROWS * 2, "d2h_bytes_per_step": 52,
                "ms_per_step": ms_e2e / K, "frame_ms": frame_stats_ms(per_e2e)},
        "gpu_launches": int(info["launches"]) * K,
        "clocks": clocks,
        "roofline": {"kernel": integrate_kernel_name(), "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                     "frac": achieved / peak if peak else None, "traffic": traffic, "traffic_source": traffic_src,
                     "traffic_over_algorithmic": (traffic / alg_bytes) if (traffic and alg_bytes) else None, "peak_source": peak_src,
                     "algorithmic_bytes_per_launch": alg_bytes, "voxels_written_per_launch": n_upd, "kernel_ms": integ_ms,
                     "dense_upper_bound_bytes": 8.0 * DIM ** 3 + 2.0 * COLS * ROWS},
        "stage_ms": stage_ms,
    }
    if raycast_info and "error" not in raycast_info:
        rc_ms = stage_ms.get("raycast_prev", float("nan"))
        rc_ach = raycast_info["algorithmic_bytes"] / (rc_ms * 1e-3) / 1e9 if rc_ms and rc_ms > 0 else float("nan")
        line["roofline_raycast"] = {"kernel": "raycast_points_kernel", "bound": "hbm", "achieved": rc_ach, "peak": peak, "unit": "GB/s",
                                    "frac": rc_ach / peak if peak else None, "traffic": traffic_rc, "kernel_ms": rc_ms,
                                    "algorithmic_bytes_per_launch": raycast_info["algorithmic_bytes"], "unique_voxels_read": raycast_info["unique_voxels"],
                                    "unique_voxels_fetched_by_the_brick_skipping_march": raycast_info.get("unique_voxels_tracked"),
                                    "hit_rays": raycast_info["hit_rays"], "march_samples": raycast_info["march_samples"],
                                    "uncached_upper_bound_bytes": 4 * (raycast_info["march_samples"] + 64 * raycast_info["hit_rays"]) + 32 * COLS * ROWS,
                                    "note": "U = unique voxels the reference's (dense) march touches, counted by the counting instantiation of the kernel on the last "
                                            "frame's volume and pose (SURVEY 8d definition); the frame loop's brick-skipping march fetches fewer (second count) and its "
                                            "measured DRAM traffic is `traffic`; kernel_ms = the stage's CUDA-event time averaged over the roofline frames"}
    elif raycast_info:
        line["roofline_raycast"] = raycast_info
    if rank == 0 and world == 1 and not args.no_warped:
        # SURVEY 8f(1), reported beside the headline (never part of it): the same sequence with the fusion step of every frame done by
        # df_integrate_warped (DF_KINFU_WARPED_INTEGRATE) instead of the reference's rigid fallback.  Short separate pass.
        try:
            p = params(kf.STAGE_TIMING | kf.WARPED_INTEGRATE)
            p.fusion_weight_scale = 100.0
            kw = kf.KinFu(p)
            nw = min(nframes, 3 + 8)
            acc, n_upd_w, n_warped, cnt = {}, 0, 0, 0
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            for t in range(nw):
                if t == 3:
                    torch.cuda.synchronize()
                    e0.record()
                kw.lib.df_kinfu_process_device(kw.h, frames_dev[t].data_ptr(), pitch)
                if t >= 3:
                    for name, v in kw.stage_ms().items():
                        acc[name] = acc.get(name, 0.0) + v
                    i = kw.info()
                    n_upd_w += i["n_updated"]; n_warped += i["n_warped"]; cnt += 1
            e1.record()
            torch.cuda.synchronize()
            kw.close()
            line["warped_fusion"] = {"what": "same workload, fusion step = per-voxel warped integration (df_integrate_warped, weight_scale 100)",
                                     "frames": cnt, "ms_per_frame_incl_stage_readback": e0.elapsed_time(e1) / max(cnt, 1),
                                     "stage_ms": {n: v / max(cnt, 1) for n, v in acc.items()},
                                     "voxels_warped_per_frame": n_warped / max(cnt, 1), "voxels_written_per_frame": n_upd_w / max(cnt, 1),
                                     "volume_voxels": DIM ** 3}
        except Exception as e:                                                  # informational only: never lose the headline line
            line["warped_fusion"] = {"error": repr(e)}
    # ---- multi-GPU correctness record (SURVEY 8e): every rank's end state (volume checksum, node-table checksum, cloud points, pose-chain
    # hash) is all-gathered; rank 0 then re-runs every other rank's sequence on ITS GPU and requires bit-identical digests -- the proof
    # that ranks 1..N-1 fused the right volumes, not just that they were busy.  Also at N = 1: device-resident and host-buffer runs agree.
    def same_state(a, b):
        """(exact, close): exact = volume checksum, cloud count and pose-chain hash identical (the node-table checksum is reported but not
        required: the row assembly's double sums depend on the order an atomic cursor hands out, so a translation's last bit can
        differ between runs, DESIGN 4); close = final pose within 1e-4 and cloud count within 0.1 %"""
        da, db = a["digest"], b["digest"]
        exact = da[0] == db[0] and da[2] == db[2] and da[3] == db[3]
        close = max(abs(x - y) for x, y in zip(a["pose"], b["pose"])) < 1e-4 and abs(da[2] - db[2]) <= 1e-3 * max(db[2], 1)
        return exact, close

    ex, cl = same_state(digest_dev, digest_e2e)
    check = {"device_vs_host_path_identical": ex, "device_vs_host_path_close": cl, "node_table_identical": digest_dev["digest"][1] == digest_e2e["digest"][1]}
    if world > 1:
        u64 = lambda d: d - (1 << 64) if d >= (1 << 63) else d
        mine = torch.tensor([u64(d) for d in digest_dev["digest"]] + [ok_dev], dtype=torch.int64, device=device)
        pose = torch.tensor(digest_dev["pose"], dtype=torch.float64, device=device)
        allv = [torch.zeros_like(mine) for _ in range(world)]
        allp = [torch.zeros_like(pose) for _ in range(world)]
        dist.all_gather(allv, mine)
        dist.all_gather(allp, pose)
        if rank == 0:
            got = [{"digest": [int(x) & ((1 << 64) - 1) for x in v[:4].tolist()], "pose": p_.tolist()} for v, p_ in zip(allv, allp)]
            mism, soft = [], []
            for r in range(1, world):
                fr = torch.from_numpy(make_frames(nframes, seed=distrib.sequence_seed(r)).view(np.int16)).cuda()
                kr = kf.KinFu(params())
                for t in range(nframes):
                    kr.lib.df_kinfu_process_device(kr.h, fr[t].data_ptr(), pitch)
                Rr, tr_ = kr.getCameraPose()
                want = {"digest": kr.state_digest(), "pose": [float(x) for x in Rr.reshape(9)] + [float(x) for x in tr_]}
                kr.close()
                del fr
                exact, close = same_state(got[r], want)
                if not exact:
                    (soft if close else mism).append(r)
            check.update({"ranks": world, "rank_digests": [[f"{x:016x}" for x in g["digest"]] for g in got], "ranks_recomputed_on_gpu0": world - 1,
                          "ranks_matching_to_rounding_only": soft, "mismatching_ranks": mism, "all_ranks_match_single_gpu_run": not mism and not soft,
                          "all_ranks_ok": not mism})
            if mism:
                print(f"[bench] WARNING: ranks {mism} ended in a state that differs from a single-GPU run of the same sequence", file=sys.stderr, flush=True)
        barrier()
    line["state_check"] = check
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        # bounded sample: 1 init + the calibration frames + 10 timed frames of the same sequence (about 15-25 s of CPU work)
        steps_cpu = min(10, K)
        cands = thread_candidates()
        aff, quota = host_cpus()
        dt, cinfo, per_cpu, used, calib = run_cpu(frames[: 1 + len(cands) + steps_cpu], len(cands), steps_cpu, calibrate=cands)
        line["cpu_baseline"] = {"value": steps_cpu / dt, "unit": "frames/s", "cores": used, "kind": "port",
                                "sample": f"{steps_cpu} timed frames (+1 init, +{len(cands)} untimed thread-count calibration frames) of the same sequence "
                                          f"through the CPU oracle (OpenMP, {used} threads)",
                                "affinity_cpus": aff, "cgroup_quota_cpus": quota,
                                "thread_calibration_s_per_frame": {str(c): v for c, v in calib.items()}, "frame_ms": frame_stats_ms(per_cpu)}
        # SURVEY 8d also asks for the single-thread figure (the reference's own warp / k-NN loops are serial): 2 frames, 1 OpenMP thread
        try:
            set_omp_threads(1)
            dt1 = run_cpu(frames[:3], 0, 2)[0]
            set_omp_threads(used)
            line["cpu_baseline"]["single_thread_value"] = 2 / dt1
        except Exception as e:                                                  # informational only
            line["cpu_baseline"]["single_thread_value"] = None
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
