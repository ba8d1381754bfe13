#!/usr/bin/env python
"""bench.py -- scans/sec of the ImMesh localization + meshing hot path on synthetic LiDAR scans.

One "step" = one LiDAR scan through the whole path: constant-velocity prediction, all IESKF iterations (voxel-hash
lookup, point-to-plane residual selection, Jacobian, H^T R^-1 H reduction, 6x6 IESKF update), VoxelMap update, transform
of the full-resolution scan, vertex append, per-voxel dilation / Delaunay / pull-commit, push.

  python bench.py --gpus 1 --steps K --warmup W               our CUDA path (N>1: launched under torchrun)
  python bench.py --impl reference --gpus 1 --steps K ...     the reference algorithm on the host cores (oracle port)
  python bench.py --config C1|C2|C3|C4|C5|C5s1                the other BASELINE.json configurations (default: the 100k metric config)
  python bench.py ... --dump-outputs DIR                      also write what the timed path returned after its last step as DIR/*.npy

Prints ONE JSON line (rank 0).  `value` = scans/s with the scans already resident in HBM (device-event time, L2
flushed between scans); `e2e` = scans/s through the C ABI with pinned HOST buffers (H2D of both clouds and D2H of the
state + frame counters inside the timed region); `roofline` = the dominant kernel's algorithmic bytes / CUDA-event
time against the measured HBM peak; `cpu_baseline` = the CPU oracle on a bounded sample of the same stream (pipelined and
serial, all cores and the reference's 4 threads).  Before anything is timed a prefix of the stream goes through the timed
(pipelined, graph-replayed) path AND the oracle: `value` is only printed when state, VoxelMap and mesh are identical.
"""
from __future__ import annotations

import argparse
import dataclasses
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

# Seven CUDA streams per scan pipeline (localization + upload, mesh + 2 side + upload, front-end) next to torch's and NCCL's own:
# with the default of 8 hardware work queues two of them can alias and serialise the localization and the mesh pipeline of a rank
# (seen as one rank of eight running at the blocking-call rate).  Must be set before the CUDA context exists.
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

METRIC = "scans/sec (synthetic 100k-pt scans) loc+mesh"


# --------------------------------------------------------------------------------------------- workloads
def workloads():
    from immesh_b200 import api
    velodyne = dataclasses.replace(api.VELODYNE, calib_laser=1)      # config/velodyne.yaml as shipped (calib_laser: true)
    c5_lio = dataclasses.replace(api.AVIA, voxel_size=0.2, filter_size_surf=0.2, hash_capacity_log2=23, max_nodes=8 << 20, max_chunks=8 << 20)
    c5_mesh = api.MeshConfig(points_minimum_scale=0.05, voxel_resolution=0.2, number_of_pts_append_to_map=10000)
    c5s1_mesh = api.MeshConfig(points_minimum_scale=0.05, voxel_resolution=0.2, number_of_pts_append_to_map=2000000,
                               max_vertices=48 << 20, max_triangles=128 << 20, max_voxels=8 << 20)
    return {
        "C100k": dict(kind="avia100k", lio=api.AVIA, mesh=api.MeshConfig(), map_warm=8, steps=30, gate=3, cpu_sample=8,
                      workload="synthetic 100k-pt scan stream (Livox-Avia-shape FoV, 10 Hz, 1 m/s), avia.yaml parameters: leaf 0.4 m, root voxel 0.5 m, max_layer 2, 4 IESKF iterations, mesh voxel 0.4 m, xi 0.1 m, 10000 pts appended/frame"),
        "C1": dict(kind="avia", lio=api.AVIA, mesh=api.MeshConfig(), map_warm=0, steps=20, gate=4, cpu_sample=8,
                   workload="BASELINE C1: synthetic Livox-Avia-shape scans, 24k pts, config/avia.yaml (0.5 m root voxel, 0.4 m leaf), the first scans after map initialisation (cold map)"),
        "C2": dict(kind="avia", lio=api.AVIA, mesh=api.MeshConfig(), map_warm=20, steps=100, gate=6, cpu_sample=10,
                   workload="BASELINE C2: synthetic Livox-Avia stream, 24k pts/scan @100 Hz, 0.4 m leaf / mesh voxel (config/avia.yaml), consumed back to back on a warm map"),
        "C3": dict(kind="hdl64", lio=velodyne, mesh=api.MeshConfig(), map_warm=4, steps=20, gate=3, cpu_sample=6,
                   workload="BASELINE C3: Velodyne HDL-64 KITTI-shape synthetic stream, 131072 pts/scan @10 Hz, config/velodyne.yaml (3 m root voxel, max_layer 4, max_points 1000, leaf 0.5 m, 3 iterations, calib_laser true)"),
        "C4": dict(kind="hdl64loop", lio=velodyne, mesh=api.MeshConfig(), map_warm=4, steps=40, gate=3, cpu_sample=6,
                   workload="BASELINE C4: KITTI-odometry-seq-00-shape synthetic stream (HDL-64, 131072 pts/scan, closed loop revisited lap after lap; the first scans of the 4541-scan trajectory), config/velodyne.yaml"),
        "C5": dict(kind="ouster1m", lio=c5_lio, mesh=c5_mesh, map_warm=2, steps=6, gate=1, cpu_sample=2,
                   workload="BASELINE C5: dense Ouster-128-aggregate synthetic, 1M pts/scan, 0.2 m root voxel / leaf / mesh voxel (xi 0.05 m), 10000 pts appended/frame (step 100)"),
        "C5s1": dict(kind="ouster1m", lio=c5_lio, mesh=c5s1_mesh, map_warm=1, steps=4, gate=1, cpu_sample=1,
                     workload="BASELINE C5 with number_of_pts_append_to_map raised so that every point is an append candidate (step 1): 1M candidates/frame"),
    }


def _gen_one(args):
    kind, k, seed, leaf, ext_T = args
    from immesh_b200 import synth
    sensor = synth.make_sensor(kind)
    body, R, t = synth.make_scan(sensor, k, seed, None, ext_T)
    return dict(body_full=body, body_ds=synth.voxel_grid_downsample(body, leaf), R_true=R, t_true=t, dt=1.0 / sensor.hz)


def get_stream(wl, n_scans, seed=0):
    """Deterministic scans 0..n_scans-1 of the workload's stream (ray-casting is numpy on the host: generated in parallel)."""
    cfg = wl["lio"]
    jobs = [(wl["kind"], k, seed, cfg.filter_size_surf, cfg.ext_T) for k in range(n_scans)]
    big = wl["kind"] in ("ouster1m",)
    nproc = min(len(jobs), 8 if big else 16, max(1, (os.cpu_count() or 2) // 2))
    if nproc > 1 and n_scans > 4:
        import multiprocessing as mp
        with mp.get_context("fork").Pool(nproc) as pool:
            return pool.map(_gen_one, jobs, chunksize=1)
    return [_gen_one(j) for j in jobs]


def init_state_vec(scans):
    s = np.zeros(348)
    s[0:9] = scans[0]["R_true"].reshape(9)
    s[9:12] = scans[0]["t_true"]
    s[12:15] = (scans[1]["t_true"] - scans[0]["t_true"]) / scans[0]["dt"]
    for i in range(18):
        s[24 + i * 18 + i] = 1e-7
    return s


def config_block(name, wl, scans):
    """Identical in both arms (the driver compares the two `config` objects)."""
    return {"workload": wl["workload"], "name": name,
            "points_per_scan_raw": int(np.mean([s["body_full"].shape[0] for s in scans[1:5]])),
            "points_per_scan_downsampled": int(np.mean([s["body_ds"].shape[0] for s in scans[1:5]])),
            "map_warm_scans": wl["map_warm"],
            "pipeline": "localization(k+1) overlaps meshing(k) (GPU arm: two CUDA streams; CPU arm: 1/max(t_loc, t_mesh)), as the reference's LIO thread || mesh threads",
            "l2": "GPU arm: flushed by a 256 MB write queued before every scan, INSIDE the timed region"}


# --------------------------------------------------------------------------------------------- clocks
class ClockSampler:
    """SM clock + throttle reasons sampled DURING the timed regions.  NVML in a thread (about 2 ms per sample: the timed
    region of a default run is only ~15 ms, too short for `nvidia-smi -lms`), nvidia-smi as the fallback."""
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
    BITS = {"sw_power_cap": 0x4, "hw_slowdown": 0x8, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40}

    def __init__(self, index=0, uuid=None):
        self.index, self.uuid, self.rows, self.proc = index, uuid, [], None
        self.samples, self.max_mhz, self.mask, self.stop_flag, self.thread, self.how = [], None, 0, False, None, None

    def _nvml_handle(self):
        import pynvml as nv
        nv.nvmlInit()
        h = None
        if self.uuid:
            for cand in (self.uuid, "GPU-" + self.uuid):
                try:
                    h = nv.nvmlDeviceGetHandleByUUID(cand.encode() if isinstance(cand, str) else cand)
                    break
                except Exception:
                    h = None
        if h is None:
            vis = os.environ.get("CUDA_VISIBLE_DEVICES", "")
            idx = self.index
            if vis and all(x.strip().isdigit() for x in vis.split(",")) and self.index < len(vis.split(",")):
                idx = int(vis.split(",")[self.index])
            h = nv.nvmlDeviceGetHandleByIndex(idx)
        return nv, h

    def start(self):
        try:
            nv, h = self._nvml_handle()
            self.max_mhz = float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
            reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or getattr(nv, "nvmlDeviceGetCurrentClocksThrottleReasons")
            nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)

            def loop():
                while not self.stop_flag:
                    try:
                        self.samples.append(float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)))
                        self.mask |= int(reasons(h))
                    except Exception:
                        pass
                    time.sleep(0.002)
            self.thread = threading.Thread(target=loop, daemon=True)
            self.thread.start()
            self.how = "nvml"
            return
        except Exception:
            self.thread = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
            self.how = "nvidia-smi"
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.thread is not None:
            self.stop_flag = True
            self.thread.join(timeout=1.0)
            reasons = [n for n, bit in self.BITS.items() if self.mask & bit]
            return {"sm_mhz": float(np.median(self.samples)) if self.samples else None, "sm_max_mhz": self.max_mhz, "reasons": reasons,
                    "samples": len(self.samples), "how": "nvml, 2 ms period, across both timed regions"}
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                pass
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 2 + i and r[2 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons, "samples": len(sm), "how": "nvidia-smi -lms 20"}


# --------------------------------------------------------------------------------------------- CPU arm
def cpu_thread_sets():
    """(label, residual-loop threads, meshing threads).  "ref4": the reference's own setting (MP_PROC_NUM = 4, CMakeLists.txt:21-24;
    meshing TBB-parallel over the cores).  "all": what is fastest on this host -- the residual loop is the only parallel part of
    localization and stops scaling near 16 threads on a 4k-20k-point loop; the voxel-parallel meshing is capped at 64 (beyond
    that the serial push dominates)."""
    n = os.cpu_count() or 1
    return [("all", min(16, n), min(64, n)), ("ref4", min(4, n), min(64, n))]


def run_cpu(wl, scans, n_warm, n_timed, t_loc, t_mesh, dump_dir=None):
    """The reference algorithm on the host cores (oracle port): returns per-scan (t_loc, t_mesh) seconds.  dump_dir: write the
    state and mesh after the last scan there (dump_outputs)."""
    from oracle_api import OracleLio, OracleMesh
    cfg = wl["lio"]
    lio = OracleLio(cfg, sum_mode=1, omp_threads=t_loc, solve_mode=1, plane_var_mode=1)   # the reference's literal formulation: serial double sums, two 18x18 inverses, per-point plane covariance loop
    mesh = OracleMesh(wl["mesh"], threads=t_mesh)
    lio.set_state(init_state_vec(scans))
    lio.voxel_map_init(scans[0]["body_full"])
    times = []
    for k in range(1, 1 + n_warm + n_timed):
        sc = scans[k]
        t0 = time.perf_counter()
        lio.predict(sc["dt"])
        iters = lio.lio_state_estimation(sc["body_ds"])
        lio.map_incremental_grow(sc["body_ds"])
        t1 = time.perf_counter()
        world = lio.transform_full(sc["body_full"])                 # transformLidar of the full scan
        mesh.push_frame(world, lio.get_state()[9:12], k)
        t2 = time.perf_counter()
        if k > n_warm:
            times.append((t1 - t0, t2 - t1))
    if dump_dir:
        verts, tris, flags = mesh.snapshot()
        dump_outputs(dump_dir, {"state": lio.get_state(), "iterations": [iters]},
                     {"mesh_vertices": verts, "mesh_triangles": tris, "mesh_triangle_flags": flags})
    return np.array(times)


def cpu_summary(tt):
    loc, mesh = tt[:, 0], tt[:, 1]
    return {"pipelined_scans_s": round(1.0 / max(float(np.mean(loc)), float(np.mean(mesh))), 3), "serial_scans_s": round(1.0 / float(np.mean(loc + mesh)), 3),
            "loc_ms": round(float(np.mean(loc)) * 1e3, 3), "mesh_ms": round(float(np.mean(mesh)) * 1e3, 3),
            "loc_ms_median_p95": [round(float(np.median(loc)) * 1e3, 3), round(float(np.percentile(loc, 95)) * 1e3, 3)],
            "mesh_ms_median_p95": [round(float(np.median(mesh)) * 1e3, 3), round(float(np.percentile(mesh, 95)) * 1e3, 3)]}


def cpu_frontend_ms(wl, scans, n):
    """The CPU arm's own front-end (what the GPU arm's e2e_raw includes): [calibration] + VoxelGrid of the raw scan, oracle port."""
    import oracle_api as oa
    ts = []
    for sc in scans[1:1 + n]:
        t0 = time.perf_counter()
        pts = oa.kitti_calib(sc["body_full"]) if wl["lio"].calib_laser else sc["body_full"]
        oa.voxel_grid(pts, wl["lio"].filter_size_surf)
        ts.append(time.perf_counter() - t0)
    return round(float(np.mean(ts)) * 1e3, 3)


def cpu_baseline_block(wl, scans, n_warm, n_timed, what):
    res = {}
    for label, tl, tm in cpu_thread_sets():
        tt = run_cpu(wl, scans, n_warm, n_timed, tl, tm)
        res[label] = dict(cpu_summary(tt), threads_loc_mesh=[tl, tm])
    best = res["all"]
    return {"value": best["pipelined_scans_s"], "unit": "scans/s", "cores": max(best["threads_loc_mesh"]), "host_cores": os.cpu_count() or 1, "kind": "port",
            "sample": f"{n_timed} scans of the same stream after {n_warm} untimed scans; {what}; value = pipelined rate 1/max(t_loc, t_mesh) at the fastest thread setting ('all')",
            "all_cores": res["all"], "reference_4_threads": res["ref4"], "frontend_ms_single_thread": cpu_frontend_ms(wl, scans, min(4, n_timed)),
            "reference_published": "Avia 24k-pt scans on i9-10900: localization 16.6 ms, meshing 25.3 ms; KITTI HDL-64: 42.2 / 31.3 ms (T-RO Table IV)"}


# --------------------------------------------------------------------------------------------- GPU arm
def algorithmic_bytes(kernel, info):
    """Compulsory bytes PER SCAN of `kernel` (DESIGN.md, SURVEY.md 8d) from the work counters of the profiled scans; the caller divides
    by the kernel's launches per scan."""
    n = info["n_ds"]
    if kernel == "k_residual":
        # per IESKF iteration (= per launch): 12 B body xyz + 16 B hash slot (key + root index) per point, 240 B per distinct matched
        # plane record, 232 B out; times the iterations run per scan
        return (28.0 * n + 240.0 * info["planes_unique"] + 232.0) * info.get("launches", {}).get("k_residual", 1.0)
    if kernel == "k_match":
        # per IESKF iteration: 12 B body xyz + 16 B hash slot per point, 240 B per distinct matched plane record, 8 B match out
        return (36.0 * n + 240.0 * info["planes_unique"]) * info.get("launches", {}).get("k_match", 1.0)
    if kernel == "k_terms":
        # per IESKF iteration: 12 B body xyz + 8 B match per point, 240 B per distinct matched plane record, 232 B of sums out
        return (20.0 * n + 240.0 * info["planes_unique"] + 232.0) * info.get("launches", {}).get("k_terms", 1.0)
    if kernel == "k_grow_voxel":
        # SURVEY 8d: 12 N + 16 N + sum over dirty nodes (96 B per stored point read by the refit + 456 B plane record written)
        return 28.0 * n + 96.0 * info["refit_points"] + 456.0 * info["refits"]
    if kernel == "k_grow_simple":
        # append-only voxels: 28 B in per point, 96 B point record + 480 B of moments read-modify-written
        return n * (28.0 + 96.0 + 2 * 480.0)
    if kernel == "k_voxel_dilate":
        # float4 per gathered kNN candidate, 27 voxel-hash probes (16 B) per voxel, smoothed position write per query, ids out
        return 16.0 * info["gathered"] + 27 * 16.0 * info["voxels_meshed"] + 24.0 * info["queries"] + 4.0 * info["dilated"]
    if kernel.startswith("k_voxel_mesh") or kernel == "k_voxel_tri_warp":
        # ids + float4 position per dilated vertex, 16 B triple-hash probe + 12 B emit per facet, incidence walk 16 B per facet pulled
        return 20.0 * info["dilated"] + 44.0 * info["faces"]
    if kernel == "k_cand_init":
        return info["candidates"] * (12.0 + 16.0 + 27 * 16.0)
    if kernel == "k_pull_vertices":
        # per dilated vertex: id + incidence-list head, 16 B per stored triangle walked (~ facets of the voxel)
        return 12.0 * info["dilated"] + 16.0 * info["faces"]
    if kernel == "k_push_add":
        return 44.0 * info["faces"]
    if kernel == "k_transform_full":
        return 24.0 * info["n_full"]
    return None


DUMP_BYTES = 64 << 20


def dump_outputs(out_dir, fixed, rows):
    """--dump-outputs: every array as out_dir/<name>.npy, float32 kept, everything else as float64 (integers up to 2^53 exactly).
    `rows` are per-row tables (vertices, facets, ...); if the whole dump would exceed DUMP_BYTES, each of them keeps the same
    fraction of its rows, chosen by a fixed seed and kept in order, so that two runs with the same arguments write the same files
    and tables of equal length keep the same rows."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {**fixed, **rows}
    arrays = {n: np.asarray(a, dtype=np.float32 if np.asarray(a).dtype == np.float32 else np.float64) for n, a in arrays.items()}
    fixed_bytes = sum(arrays[n].nbytes for n in fixed)
    row_bytes = sum(arrays[n].nbytes for n in rows)
    frac = min(1.0, (DUMP_BYTES - fixed_bytes) / row_bytes) if row_bytes else 1.0
    for name, a in arrays.items():
        if name in rows and frac < 1.0:
            a = a[np.sort(np.random.default_rng(0).choice(a.shape[0], int(a.shape[0] * frac), replace=False))]
        np.save(os.path.join(out_dir, name + ".npy"), a)


def pin(a):
    """Page-locked copy of a numpy array (the e2e inputs live in pinned host memory, the C ABI then DMAs straight from them)."""
    import torch
    t = torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
    return t.numpy(), t          # the tensor owns the pinned allocation: keep it alive next to the view


def sharded_single_stream(args, rank, world, lib, wl, scans0, dev, flush, K, W):
    """N>1 only: ONE scan stream with the VoxelMap and the mesher's per-voxel stage sharded over all ranks (north_star's
    partitioning; strong scaling).  Same timed-region rules as `value`.  Reported next to the headline replicas number."""
    import torch
    import torch.distributed as dist
    from immesh_b200 import api
    lio, mesh = api.Lio(wl["lio"], lib=lib), api.Mesh(wl["mesh"], lib=lib)
    uid = [api.comm_unique_id(lib) if rank == 0 else None, api.comm_unique_id(lib) if rank == 0 else None]
    dist.broadcast_object_list(uid, src=0)
    lio.shard(rank, world, uid[0])
    mesh.shard(rank, world, uid[1])
    lio.set_state(init_state_vec(scans0))
    lio.voxel_map_init(scans0[0]["body_full"])
    MW = wl["map_warm"]
    d_ds = [torch.from_numpy(s["body_ds"]).to(dev) for s in scans0[:2 + MW + W + K]]
    d_full = [torch.from_numpy(s["body_full"]).to(dev) for s in scans0[:2 + MW + W + K]]
    k = 1
    for _ in range(MW + W):
        lio.step_async(d_ds[k].data_ptr(), d_ds[k].shape[0], scans0[k]["dt"], on_device=True)
        mesh.push_frame_from_lio_async(lio, d_full[k].data_ptr(), d_full[k].shape[0], on_device=True)
        k += 1
    s_warm, _ = lio.wait()
    mesh.wait()
    # parity of the sharded path inside the bench run: every rank's state after the warm-up scans equals the oracle's (rank 0 runs it)
    parity = None
    if rank == 0:
        from oracle_api import OracleLio
        o = OracleLio(wl["lio"], sum_mode=0, omp_threads=8)
        o.set_state(init_state_vec(scans0))
        o.voxel_map_init(scans0[0]["body_full"])
        for j in range(1, 1 + MW + W):
            o.predict(scans0[j]["dt"])
            o.lio_state_estimation(scans0[j]["body_ds"])
            o.map_incremental_grow(scans0[j]["body_ds"])
        parity = bool(np.array_equal(o.get_state(), s_warm))
    st = torch.from_numpy(s_warm.copy()).to(dev)
    ref = st.clone()
    dist.broadcast(ref, src=0)
    same = torch.tensor([int(bool(torch.equal(st, ref)))], device=dev)
    dist.all_reduce(same, op=dist.ReduceOp.MIN)
    torch.cuda.synchronize()
    dist.barrier()
    torch.cuda.synchronize()
    api.pipeline_mark_begin(lio)
    for _ in range(K):
        lio.enqueue_memset(flush.data_ptr(), flush.numel())
        lio.step_async(d_ds[k].data_ptr(), d_ds[k].shape[0], scans0[k]["dt"], on_device=True)
        mesh.push_frame_from_lio_async(lio, d_full[k].data_ptr(), d_full[k].shape[0], on_device=True)
        k += 1
    ms = api.pipeline_mark_end(lio, mesh)
    lio.wait()
    mesh.wait()
    torch.cuda.synchronize()
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t[0])
    out = {"value": round(K / (ms * 1e-3), 3), "unit": "scans/s", "ms_per_step": round(ms / K, 4), "scaling": "strong",
           "transport": {"voxelmap": lio.shard_transport(), "mesher": mesh.shard_transport()},
           "parity": {"ranks": world, "state_equals_oracle_after_warmup_rank0": parity, "state_identical_on_all_ranks": bool(int(same.item()))},
           "what": f"one stream, VoxelMap sharded by root-voxel key and the mesher's per-voxel stage by voxel owner over {world} GPUs; "
                   "bit-identical to the single-GPU result (tests/test_parity_gpu.py::test_sharded_ranks_equal_single_gpu)"}
    lio.close()
    mesh.close()
    return out


def multi_stream_extra(S, lib, wl, scans, d_ds, d_full, flush, K, W):
    """N = 1 extra: S independent scan streams (S handle pairs, own maps and meshes) interleaved on ONE GPU.  Same timed-region
    rules as `value` (inputs resident, a 256 MB L2-flush write queued before every scan of every stream); time = max(CUDA-event
    time of the slowest session, wall clock between device-wide synchronisations)."""
    import torch
    from immesh_b200 import api
    sess = []
    for _ in range(S):
        lio, mesh = api.Lio(wl["lio"], lib=lib), api.Mesh(wl["mesh"], lib=lib)
        lio.set_state(init_state_vec(scans))
        lio.voxel_map_init(scans[0]["body_full"])
        sess.append((lio, mesh))

    def enqueue(k, with_flush):
        for lio, mesh in sess:
            if with_flush:
                lio.enqueue_memset(flush.data_ptr(), flush.numel())
            lio.step_async(d_ds[k].data_ptr(), d_ds[k].shape[0], scans[k]["dt"], on_device=True)
            mesh.push_frame_from_lio_async(lio, d_full[k].data_ptr(), d_full[k].shape[0], on_device=True)

    k = 1
    for _ in range(wl["map_warm"] + W):
        enqueue(k, False)
        k += 1
    for lio, mesh in sess:
        lio.wait()
        mesh.wait()
    torch.cuda.synchronize()
    for lio, _ in sess:
        api.pipeline_mark_begin(lio)
    t0 = time.perf_counter()
    for _ in range(K):
        enqueue(k, True)
        k += 1
    ev_ms = max(api.pipeline_mark_end(lio, mesh) for lio, mesh in sess)
    for lio, mesh in sess:
        lio.wait()
        mesh.wait()
    torch.cuda.synchronize()
    wall_ms = (time.perf_counter() - t0) * 1e3
    ms = max(ev_ms, wall_ms)
    out = {"streams": S, "value": round(S * K / (ms * 1e-3), 3), "unit": "scans/s", "ms_per_round_of_S_scans": round(ms / K, 4),
           "event_ms": round(ev_ms, 3), "wall_ms": round(wall_ms, 3), "steps_per_stream": K,
           "what": f"{S} independent streams interleaved on one GPU (own VoxelMap + mesh each); aggregate scans/s"}
    for lio, mesh in sess:
        lio.close()
        mesh.close()
    return out


def run_gpu(args, rank, world):
    import torch
    import torch.distributed as dist
    from immesh_b200 import api

    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    wl = workloads()[args.config]
    K = args.steps if args.steps is not None else wl["steps"]
    W = max(args.warmup, 3)
    MW = wl["map_warm"]
    n_prof = min(K, 10)
    n_stage = min(K, 10)
    K_raw = 0 if args.no_raw_leg else K
    n_scans = 1 + MW + W + 2 * K + K_raw + n_stage + n_prof + 1 + 6 + K + K_raw    # the last K + K_raw: a second pass of a host-buffer leg (below)
    scans = get_stream(wl, n_scans, seed=rank if args.independent_streams else 0)
    lib = api.load_library()
    dev = torch.device("cuda", local_rank)
    d_ds = [torch.from_numpy(s["body_ds"]).to(dev) for s in scans]
    d_full = [torch.from_numpy(s["body_full"]).to(dev) for s in scans]
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)   # > 126 MB L2
    torch.cuda.synchronize()

    # ---- parity gate (before anything is timed): a prefix of THIS stream through the timed path -- pipelined entry points,
    # device-resident inputs, CUDA-graph replay -- and through the oracle; no `value` unless state, map and mesh are identical
    gate = None
    if not args.no_parity_gate and (rank == 0 or args.independent_streams):
        from parity_gate import pipeline_parity
        n_gate = min(wl["gate"], len(scans) - 2)
        if not (world > 1 and not args.independent_streams):   # the sharded single-stream mode is gated by its own state check
            gate = pipeline_parity(lib, wl["lio"], wl["mesh"], scans, n_gate, dev_inputs=(d_ds, d_full), oracle_threads=(16, 32))
    if gate is not None and not gate["ok"]:
        if rank == 0:
            print(json.dumps({"metric": METRIC, "value": None, "unit": "scans/s", "n_gpus": world, "error": "parity gate failed: GPU path and oracle disagree; nothing was timed", "parity_gate": gate}))
        sys.exit(2)

    lio = api.Lio(wl["lio"], lib=lib)
    mesh = api.Mesh(wl["mesh"], lib=lib)
    if world > 1 and not args.independent_streams:
        uid = [api.comm_unique_id(lib) if rank == 0 else None, api.comm_unique_id(lib) if rank == 0 else None]
        dist.broadcast_object_list(uid, src=0)
        lio.shard(rank, world, uid[0])
        mesh.shard(rank, world, uid[1])
    lio.set_state(init_state_vec(scans))
    lio.voxel_map_init(scans[0]["body_full"])

    def step_dev(k):
        sc = scans[k]
        lio.step_dev(d_ds[k].data_ptr(), d_ds[k].shape[0], sc["dt"])
        mesh.push_frame_from_lio(lio, d_full[k].data_ptr(), d_full[k].shape[0], on_device=True)
        return lio.last_timing()[0] + mesh.last_timing()[0]

    k = 1
    for _ in range(MW):              # untimed: map densification
        step_dev(k)
        k += 1
    for _ in range(W):               # untimed warm-up steps through the timed (pipelined) path: graph capture etc.
        lio.step_async(d_ds[k].data_ptr(), d_ds[k].shape[0], scans[k]["dt"], on_device=True)
        mesh.push_frame_from_lio_async(lio, d_full[k].data_ptr(), d_full[k].shape[0], on_device=True)
        k += 1
    lio.wait()
    mesh.wait()

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    flush_bytes = flush.numel()
    # ---- timed region 1 (`value`): K scans queued back to back, inputs resident in HBM.  Localization of scan k+1
    # overlaps meshing of scan k on a second stream (the reference's own LIO || mesh-thread pipeline).  A 256 MB write is
    # queued in front of every scan as the L2 flush and is INSIDE the timed region (conservative).  Time = CUDA events
    # from the first queued operation to the completion of both streams.
    try:
        dev_uuid = str(torch.cuda.get_device_properties(local_rank).uuid)
    except Exception:
        dev_uuid = None
    sampler = ClockSampler(local_rank, dev_uuid)
    sampler.start()
    launches0 = api.launch_count(lib)
    barrier()
    api.host_wait_ms(lio, mesh)
    api.pipeline_mark_begin(lio)
    t_enq = time.perf_counter()
    for _ in range(K):
        lio.enqueue_memset(flush.data_ptr(), flush_bytes)
        lio.step_async(d_ds[k].data_ptr(), d_ds[k].shape[0], scans[k]["dt"], on_device=True)
        mesh.push_frame_from_lio_async(lio, d_full[k].data_ptr(), d_full[k].shape[0], on_device=True)
        k += 1
    enq_wall_ms = (time.perf_counter() - t_enq) * 1e3
    waits = api.host_wait_ms(lio, mesh)
    host_enqueue_ms = (enq_wall_ms - sum(waits)) / K     # host WORK to queue one scan; the waits are back-pressure from the 2-deep staging slots
    total_ms = api.pipeline_mark_end(lio, mesh)
    state, iters = lio.wait()
    mesh.wait()
    barrier()
    launches = api.launch_count(lib) - launches0
    if args.dump_outputs and rank == 0:      # what a caller of the timed path holds after its last step
        verts, tris, flags = mesh.snapshot()
        dump_outputs(args.dump_outputs, {"state": state, "iterations": [iters]},
                     {"mesh_vertices": verts, "mesh_triangles": tris, "mesh_triangle_flags": flags})
    # the flush alone, to report how much of the timed region it is
    api.pipeline_mark_begin(lio)
    for _ in range(K):
        lio.enqueue_memset(flush.data_ptr(), flush_bytes)
    flush_ms = api.pipeline_mark_end(lio, mesh) / K
    # ---- timed region 2 (`e2e`): K scans through the C ABI with HOST buffers (pinned), pipelined the same way; wall clock
    # around the calls (H2D of both clouds, D2H of state + frame counters all inside)
    for _ in range(3):     # untimed warm-up of THIS path (host-buffer entry points: their graph variant, staging buffers); the stream just continues
        lio.step_async(scans[k]["body_ds"], dt=scans[k]["dt"])
        mesh.push_frame_from_lio_async(lio, scans[k]["body_full"])
        k += 1
    lio.wait()
    mesh.wait()
    # The host-buffer legs are wall-clock measurements with the host in the loop; about one pass in fifteen on the shared boxes showed
    # a millisecond-scale stall per step (1.1-3.4 ms/step against 0.43, same code, same box, the device-timed region before it
    # unaffected: profiles/bench_history.md).  A pass slower than half the device-timed rate is measured ONCE more on the scans that
    # follow; both passes are reported (`attempts_ms_per_step`), the value is the later one.
    def slow_pass(seconds, steps):
        # slowest rank's ms/step of this pass against the slowest rank's device-timed ms/step: both reduced, so that every rank takes
        # the same decision (a second pass contains barriers)
        v = torch.tensor([seconds / steps * 1e3, total_ms / K], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(v, op=dist.ReduceOp.MAX)
        return float(v[0]) > 2.0 * float(v[1])
    e2e_attempts = []
    for attempt in range(2):
        pinned = [(pin(scans[k + j]["body_ds"]), pin(scans[k + j]["body_full"])) for j in range(K)]
        barrier()
        api.host_wait_ms(lio, mesh)
        t0 = time.perf_counter()
        h2d = d2h = 0
        for j in range(K):
            (ds, _), (full, _) = pinned[j]
            lio.step_async(ds, dt=scans[k]["dt"])
            mesh.push_frame_from_lio_async(lio, full)
            h2d += ds.nbytes + full.nbytes + 64 + 64          # scans + the two per-step parameter blocks
            d2h += 348 * 8 + 8 + 16 * 4 + 8 + 32 * 4          # LioOut block + frame counters
            k += 1
        e2e_enq_ms = (time.perf_counter() - t0) * 1e3
        e2e_waits = api.host_wait_ms(lio, mesh)
        lio.wait()
        mesh.wait()
        barrier()
        e2e_s = time.perf_counter() - t0
        del pinned
        e2e_attempts.append(round(e2e_s / K * 1e3, 4))
        if not slow_pass(e2e_s, K):
            break
    # ---- timed region 3 (`e2e_raw`): the device-resident front-end chain.  RAW full-resolution scans in pinned host memory ->
    # [KITTI laser calibration when the config sets it] -> pcl::VoxelGrid -> localization, and the (calibrated) full-resolution
    # cloud -> meshing; the down-sampled cloud and its size never leave the device.  Wall clock as for e2e.
    e2e_raw = None
    if K_raw > 0:
        vg = api.VoxelGrid(max(1 << 17, max(s["body_full"].shape[0] for s in scans) + 1024), lib=lib)
        calib = bool(wl["lio"].calib_laser)
        leaf = float(wl["lio"].filter_size_surf)
        for _ in range(3):    # untimed warm-up of THIS path: first launches of the front-end kernels, the mesher's graph variant for device-resident input
            vg.step_async_raw(lio, scans[k]["body_full"], leaf, dt=scans[k]["dt"], calib_laser=calib)
            mesh.push_frame_from_lio_async(lio, vg.input_points(), scans[k]["body_full"].shape[0], on_device=True)
            k += 1
        lio.wait()
        mesh.wait()
        raw_attempts = []
        for attempt in range(2):
            pinned = [pin(scans[k + j]["body_full"]) for j in range(K_raw)]
            barrier()
            t0 = time.perf_counter()
            raw_bytes = 0
            for j in range(K_raw):
                full, _ = pinned[j]
                vg.step_async_raw(lio, full, leaf, dt=scans[k]["dt"], calib_laser=calib)
                mesh.push_frame_from_lio_async(lio, vg.input_points(), full.shape[0], on_device=True)
                raw_bytes += full.nbytes + 128
                k += 1
            lio.wait()
            mesh.wait()
            barrier()
            raw_s = time.perf_counter() - t0
            del pinned
            raw_attempts.append(round(raw_s / K_raw * 1e3, 4))
            if not slow_pass(raw_s, K_raw):
                break
        if world > 1:
            t = torch.tensor([raw_s], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            raw_s = float(t[0])
        e2e_raw = {"value": round(K_raw * (world if args.independent_streams else 1) / raw_s, 3), "unit": "scans/s", "ms_per_step": round(raw_s / K_raw * 1e3, 4), "steps": K_raw,
                   "h2d_bytes_per_step": int(raw_bytes / K_raw), "calib_laser": calib, "attempts_ms_per_step": raw_attempts,
                   "what": "raw full-resolution scan (pinned host) -> [KITTI calibration] -> VoxelGrid down-sampling -> localization -> meshing, all on the device; only the raw scan goes up, state + counters come back"}
        vg.close()
    clocks = sampler.stop()
    # ---- blocking per-stage timing (one scan at a time, L2 flushed before each): explains where the time goes
    dev_ms, stage = [], []
    for _ in range(n_stage):
        flush.zero_()
        torch.cuda.synchronize()
        dev_ms.append(step_dev(k))
        stage.append((lio.last_timing().copy(), mesh.last_timing().copy()))
        k += 1
    # ---- profiling pass (CUDA events around every kernel; not part of any reported throughput)
    api.profile_reset(lib)
    api.profile_enable(True, lib)
    info = dict(n_ds=0, n_full=0, planes_unique=0, refits=0, refit_points=0, gathered=0, queries=0, dilated=0, faces=0, voxels_meshed=0, candidates=0)
    for _ in range(n_prof):
        flush.zero_()
        torch.cuda.synchronize()
        step_dev(k)
        nodes = lio.match_nodes()
        info["n_ds"] += d_ds[k].shape[0]
        info["n_full"] += d_full[k].shape[0]
        info["planes_unique"] += int(np.unique(nodes[nodes >= 0]).size)
        wsl = lio.work_stats()
        info["refits"] += wsl["refits"]
        info["refit_points"] += wsl["refit_points"]
        ws = mesh.work_stats()
        for key in ("gathered", "queries", "dilated", "faces", "voxels_meshed", "candidates"):
            info[key] += ws[key]
        k += 1
    api.profile_enable(False, lib)
    prof = api.profile_report(lib)
    for key in list(info):
        info[key] /= n_prof            # per scan
    kern_ms = {name: ms / n_prof for name, (ms, cnt) in prof.items()}              # per scan
    kern_launch_ms = {name: ms / cnt for name, (ms, cnt) in prof.items() if cnt}
    kern_launches_per_scan = {name: cnt / n_prof for name, (ms, cnt) in prof.items()}
    info["launches"] = kern_launches_per_scan
    dominant = max(kern_ms, key=kern_ms.get)
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak, peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    else:
        peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
    roof = None
    roof_all = {}
    for name in sorted(kern_ms, key=kern_ms.get, reverse=True)[:8]:
        bb = algorithmic_bytes(name, info)
        if bb is not None:
            gbs = bb / kern_launches_per_scan[name] / (kern_launch_ms[name] * 1e-3) / 1e9
            roof_all[name] = {"achieved_gbs": round(gbs, 3), "frac": round(gbs / peak, 6), "ms_per_launch": round(kern_launch_ms[name], 5),
                              "bytes_per_launch": round(bb / kern_launches_per_scan[name])}
    b = algorithmic_bytes(dominant, info)
    if b is None:   # never leave the headline object empty: fall back to the most expensive kernel with a byte model
        for name in sorted(kern_ms, key=kern_ms.get, reverse=True):
            if algorithmic_bytes(name, info) is not None:
                dominant, b = name, algorithmic_bytes(name, info)
                break
    if b is not None:
        per_launch_bytes = b / kern_launches_per_scan[dominant]
        achieved = per_launch_bytes / (kern_launch_ms[dominant] * 1e-3) / 1e9
        traffic = None
        tpath = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tpath) and args.config == "C100k":
            traffic = json.load(open(tpath)).get(dominant)
        roof = {"kernel": dominant, "bound": "hbm", "achieved": round(achieved, 3), "peak": peak, "unit": "GB/s", "frac": round(achieved / peak, 6),
                "traffic": traffic, "peak_source": peak_src, "bytes_per_launch": round(per_launch_bytes), "ms_per_launch": round(kern_launch_ms[dominant], 5),
                "share_of_step": round(kern_ms[dominant] / sum(kern_ms.values()), 4)}
    # whole-step roofline: algorithmic bytes of every modelled kernel of a scan / the pipelined time per scan
    step_bytes = sum(bb for bb in (algorithmic_bytes(n2, info) for n2 in kern_ms) if bb)
    # ---- max over ranks, aggregate
    per_rank_ms = None
    if world > 1:
        mine = torch.tensor([total_ms / K], dtype=torch.float64, device=dev)
        allr = [torch.zeros_like(mine) for _ in range(world)]
        dist.all_gather(allr, mine)
        per_rank_ms = [round(float(x[0]), 4) for x in allr]
        t = torch.tensor([total_ms, e2e_s], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms, e2e_s = float(t[0]), float(t[1])
    scans_done = K * (world if args.independent_streams else 1)
    cfg_block = config_block(args.config, wl, scans)
    cfg_block["parallelism"] = (f"{world} independent streams (replicas), no data-path collective" if args.independent_streams else
                                ("single GPU" if world == 1 else f"one stream, VoxelMap sharded by root-voxel key and mesher per-voxel stage by voxel owner over {world} GPUs"))
    out = {
        "metric": METRIC if args.config == "C100k" else f"scans/sec loc+mesh ({args.config})", "value": round(scans_done / (total_ms * 1e-3), 3), "unit": "scans/s",
        "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": round(total_ms / K, 4), "higher_is_better": True, "scaling": "weak" if args.independent_streams else "strong",
        "vs_baseline": None, "dtype": "f64 (f32 keys/distances, i64 fixed-point reductions)", "data": "synthetic",
        "config": cfg_block,
        "e2e": {"value": round(scans_done / e2e_s, 3), "unit": "scans/s", "h2d_bytes_per_step": int(h2d / K), "d2h_bytes_per_step": int(d2h / K),
                "ms_per_step": round(e2e_s / K * 1e3, 4), "host_buffers": "pinned (cudaHostAlloc); the C ABI copies straight from them",
                "host_work_ms_per_step": round((e2e_enq_ms - sum(e2e_waits)) / K, 4), "attempts_ms_per_step": e2e_attempts},
        "e2e_raw": e2e_raw,
        "gpu_launches": int(launches),
        "clocks": clocks,
        "parity_gate": gate,
        "timing_detail": {"l2_flush_ms_per_scan": round(flush_ms, 4),
                          "serial_ms_per_scan_blocking": round(float(np.mean(dev_ms)), 4),
                          "serial_ms_per_scan_blocking_median_p95": [round(float(np.median(dev_ms)), 4), round(float(np.percentile(dev_ms, 95)), 4)],
                          "host_enqueue_ms_per_scan": round(host_enqueue_ms, 4),
                          "ms_per_step_of_every_rank": per_rank_ms,
                          "host_enqueue_wall_ms_per_scan_incl_backpressure": round(enq_wall_ms / K, 4),
                          "cuda_graphs": api.graph_stats(lio, mesh),
                          "transport": None if world == 1 or args.independent_streams else {"voxelmap": lio.shard_transport(), "mesher": mesh.shard_transport()}},
        "stage_ms": {"lio_total": round(float(np.mean([s[0][0] for s in stage])), 4), "lio_iterations": round(float(np.mean([s[0][1] for s in stage])), 4),
                     "lio_map_update": round(float(np.mean([s[0][2] for s in stage])), 4), "mesh_total": round(float(np.mean([s[1][0] for s in stage])), 4),
                     "mesh_append": round(float(np.mean([s[1][1] for s in stage])), 4), "mesh_voxels": round(float(np.mean([s[1][2] for s in stage])), 4),
                     "mesh_push": round(float(np.mean([s[1][3] for s in stage])), 4)},
        "kernel_ms_per_scan": {k2: round(v, 5) for k2, v in sorted(kern_ms.items(), key=lambda kv: -kv[1])},
        "work_per_scan": {k2: round(v, 1) for k2, v in info.items() if k2 != "launches"},
        "roofline": roof,
        "roofline_top_kernels": roof_all,
        "roofline_whole_step": {"algorithmic_bytes_per_scan": round(step_bytes), "achieved_gbs": round(step_bytes / (total_ms / K * 1e-3) / 1e9, 3),
                                "frac": round(step_bytes / (total_ms / K * 1e-3) / 1e9 / peak, 6)},
    }
    if world == 1 and args.streams > 1:
        try:
            out["multi_stream"] = multi_stream_extra(args.streams, lib, wl, scans, d_ds, d_full, flush, K, W)
        except Exception as e:   # noqa: BLE001
            out["multi_stream"] = {"error": str(e)[:300]}
    if world > 1 and args.independent_streams and not args.no_sharded_extra:
        # The headline numbers above are complete.  The extra measurement must never cost them: a watchdog prints the line
        # without it and ends the process if the sharded pass does not finish (e.g. peer mapping unavailable on some box).
        def _bail():
            if rank == 0:
                out["sharded_single_stream"] = {"error": "did not finish within 240 s; skipped"}
                print(json.dumps(out), flush=True)
            os._exit(0)
        dog = threading.Timer(240.0, _bail)
        dog.daemon = True
        dog.start()
        try:
            scans0 = get_stream(wl, 2 + MW + W + K + 1, seed=0)
            out["sharded_single_stream"] = sharded_single_stream(args, rank, world, lib, wl, scans0, dev, flush, K, W)
        except Exception as e:   # noqa: BLE001
            out["sharded_single_stream"] = {"error": str(e)[:300]}
        dog.cancel()
    if rank == 0:
        # ---- CPU baseline on a bounded sample of the same stream (rank 0, N = 1 only)
        if world == 1 and not args.no_cpu_baseline:
            n_s = min(wl["cpu_sample"], len(scans) - 3 - min(MW, 2))
            out["cpu_baseline"] = cpu_baseline_block(wl, scans, min(MW, 2) + 2, n_s, "oracle (C++ restatement of the reference path, -O3, OpenMP residual loop + voxel-parallel meshing)")
        print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


def run_reference(args, rank, world):
    """--impl reference: the reference's CPU algorithm (oracle port; the reference itself cannot be built here) on the host cores.
    value = pipelined rate 1/max(t_loc, t_mesh), the mode the reference itself runs in and the one the GPU arm's value is."""
    if rank != 0:
        return
    wl = workloads()[args.config]
    K = args.steps if args.steps is not None else wl["steps"]
    W = max(args.warmup, 3)
    MW = wl["map_warm"]
    # without --steps: bounded so that the run ends within a few minutes
    K_eff = args.steps if args.steps is not None else min(K, 40 if args.config in ("C100k", "C1", "C2") else 8)
    scans = get_stream(wl, 1 + min(MW, 4) + W + K_eff + 1)
    label, tl, tm = cpu_thread_sets()[0]
    tt = run_cpu(wl, scans, min(MW, 4) + W, K_eff, tl, tm, dump_dir=args.dump_outputs)
    sm = cpu_summary(tt)
    v = sm["pipelined_scans_s"]
    out = {"impl": "reference", "metric": METRIC if args.config == "C100k" else f"scans/sec loc+mesh ({args.config})", "value": v, "unit": "scans/s", "n_gpus": world,
           "steps": K_eff, "warmup": W,
           "ms_per_step": round(1e3 / v, 3), "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
           "config": dict(config_block(args.config, wl, scans), parallelism="single GPU" if world == 1 else f"{world} independent streams (replicas), no data-path collective"),
           "cpu_baseline": dict(sm, value=v, unit="scans/s", cores=max(tl, tm), threads_loc_mesh=[tl, tm], host_cores=os.cpu_count() or 1, kind="port",
                                sample=f"{K_eff} scans (one per step) after {min(MW, 4) + W} untimed scans; oracle port of the reference CPU path (the reference needs ROS/Eigen/PCL/CGAL and cannot be compiled here); value = pipelined 1/max(t_loc, t_mesh)"),
           "e2e": {"value": v, "unit": "scans/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(out))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="C100k", choices=["C100k", "C1", "C2", "C3", "C4", "C5", "C5s1"],
                    help="workload: C100k = the configuration BASELINE.json's metric is quoted on (default); C1..C5 = BASELINE.json configs[0..4]")
    ap.add_argument("--mode", default=None, choices=["sharded", "replicas"],
                    help="N>1: 'replicas' (default) = every rank runs its own independent stream, weak scaling; 'sharded' = one scan stream, "
                         "VoxelMap + mesher sharded over the ranks (exchanges fused into the kernels over NVLink peer windows), strong scaling")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-raw-leg", action="store_true", help="skip the e2e_raw region (device-resident front-end chain)")
    ap.add_argument("--no-parity-gate", action="store_true", help="experiments only: skip the GPU-vs-oracle check that precedes the timed regions")
    ap.add_argument("--streams", type=int, default=None, help="N=1: also measure this many independent streams interleaved on the one GPU (reported as `multi_stream`; 1 = skip)")
    ap.add_argument("--no-sharded-extra", action="store_true", help="N>1, replicas mode: skip the additional sharded single-stream measurement")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the timed path returned after its last step (state, iteration count, mesh vertices / facets / "
                         "orientation flags) as DIR/<name>.npy, at most 64 MB in all (a seeded sample of the mesh rows beyond that)")
    args = ap.parse_args()
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    if args.mode is None:
        # default for N>1: independent scan streams per GPU (weak scaling, no data-path collective); the sharded single-stream
        # number is measured in the same run and reported next to it.
        args.mode = "replicas"
    args.independent_streams = (world > 1 and args.mode == "replicas")
    if args.streams is None:
        args.streams = 4 if args.config == "C100k" else 1
    from immesh_b200 import build
    if rank == 0:
        build.build_oracle()
    if args.impl == "reference":
        run_reference(args, rank, world)
    else:
        run_gpu(args, rank, world)


if __name__ == "__main__":
    main()
