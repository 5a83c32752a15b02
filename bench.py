#!/usr/bin/env python
"""bench.py -- ICP measurement-model throughput on B200 (BASELINE.json metric).

A "step" is ONE search pass of the hot path over one frame: body->world transform, exact 5-NN in the device
map, plane fit, point-to-plane residual, Jacobian row, HtH / Htr reduced and delivered to the host
(laserMapping.cpp:959-1080). Workloads (synthetic, lidar_imu_init_b200/scenes.py; initial pose = ground truth (+) 0.5 deg / 5 cm,
SURVEY.md 8d), selected with --config:

  C2 (default, the configuration the metric is quoted on): 240k-point Avia-shaped scan vs 5M-point map.
       N > 1: WEAK scaling -- a frame of N x 240k points; the map is replicated, every rank uploads the frame, the library
       cuts it into N slots and sums the accumulators over the ranks inside liinit_icp_iterate (NCCL, behind the C-ABI).
  C3   130k-point spinning scan (det_range 100 m) vs 10M-point map.
  C4   260k-point scans, map grown 5M -> 50M points by timed Add_Points(downsample) batches (+ a timed box delete), then the
       search pass against the grown map.
  C5   one 2M-point frame vs the 5M-point map; N > 1: STRONG scaling, slots of 2M / N points.

  value  : points*iters/s, frame resident in HBM, timed on the device (CUDA events around each step on the
           stream the kernels run on; L2 flushed between steps by a 256 MiB memset outside the events).
  e2e    : same metric through the C-ABI with HOST buffers: every step hands the pinned host frame to the library
           (N = 1: liinit_scan_attach_host, the search kernel reads it over PCIe; N > 1: liinit_scan_upload; the staged
           variant is timed next to it) and reads HtH/Htr back (liinit_icp_iterate).
  --impl reference : the reference's CPU path (verbatim ikd-Tree from oracle/_ref + the restated OpenMP loop)
           on the host cores, same metric/config, each step a bounded sample of the scan.

Prints ONE JSON line on rank 0.

  --dump-outputs DIR : after the timed steps, rank 0 writes what the last timed step returned (HtH, Htr, selected points, residual
           sum) as float64 DIR/<name>.npy. The workload comes from fixed seeds, so two builds compare output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

_REAL_STDOUT = None


def emit(obj):
    line = json.dumps(obj) + "\n"
    if _REAL_STDOUT is not None:
        os.write(_REAL_STDOUT, line.encode())
    else:
        sys.stdout.write(line)
        sys.stdout.flush()


# dram__bytes_read.sum + dram__bytes_write.sum of ONE launch of the search kernel on C2 (ncu --set full, cold cache), per index
NCU_DRAM_BYTES_KNN = {1: 124_534_016, 2: 141_602_560}   # 1: 111.01 MB read + 13.53 MB written (the kernel writes the neighbour copies)
NCU_DRAM_SOURCE = {1: "profiles/r02/ncu_full_final_metrics.txt", 2: "profiles/r01_cells/ncu_full_stream_final_metrics.txt"}
KNN_KERNEL = {1: "k_knn_scan (5-NN search on whole bricks, lockstep lane groups; dominant kernel of the pass)",
              2: "k_knn_cells_scan (5-NN search on the per-brick cell directory, one scan point per thread; dominant kernel of the pass)"}
KNN_NAME = {1: "bricks", 2: "cells"}
ALG_BYTES_PER_POINT = 132  # SURVEY.md 8(d): 16 body + 80 neighbours + 16 normal/residual + 20 ids
UNIT = "points*iters/s"

# name: (scan points per GPU-frame, map points, det_range, workload string, metric string)
CONFIGS = {
    "C2": (240_000, 5_000_000, 450.0, "C2: 240k-pt Avia-shaped scan vs 5M-pt map (BASELINE.json configs[1]), search pass",
           "ICP points*iters/s (search pass), 240k-pt scan vs 5M-pt map"),
    "C3": (130_000, 10_000_000, 100.0, "C3: 130k-pt spinning scan vs 10M-pt map (BASELINE.json configs[2]), search pass",
           "ICP points*iters/s (search pass), 130k-pt scan vs 10M-pt map"),
    "C4": (260_000, 50_000_000, 150.0, "C4: 260k-pt scans, map grown 5M -> 50M pts by Add_Points batches + box delete (BASELINE.json configs[3]), "
           "search pass against the grown map", "ICP points*iters/s (search pass), 260k-pt scan vs map grown to 50M pts"),
    "C5": (2_000_000, 5_000_000, 450.0, "C5: one 2M-pt frame vs 5M-pt map, scan points sharded over the GPUs (BASELINE.json configs[4]), search pass",
           "ICP points*iters/s (search pass), 2M-pt frame vs 5M-pt map"),
}


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler(threading.Thread):
    """Samples SM clock / throttle reasons of one GPU with NVML while the timed region runs."""

    def __init__(self, index: int, period=0.002):
        super().__init__(daemon=True)
        self.index, self.period = index, period
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._halt = threading.Event()
        self.recording = threading.Event()   # the thread polls from start() on (NVML's first queries are slow), samples count from here
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            self.ok = False

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4): "sw_power_cap",
            getattr(nv, "nvmlClocksThrottleReasonHwPowerBrakeSlowdown", 0x80): "hw_power_brake",
        }
        while not self._halt.is_set():
            try:
                mhz = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                if self.recording.is_set():
                    self.samples.append(mhz)
                    for bit, nm in names.items():
                        if r & bit:
                            self.reasons.add(nm)
            except Exception:
                pass
            time.sleep(self.period)

    def stop(self):
        self._halt.set()
        self.join(timeout=2)
        med = float(np.median(self.samples)) if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.samples)}


def make_workload(cfg: str, world: int, n_scan: int, n_map: int):
    """Scene + map + the WHOLE frame (every rank generates the same one) + poses. C2 at N > 1: N scans of n_scan points of the same
    scene and pose (different seeds) back to back -- slot r of the library's cut is scan r."""
    from lidar_imu_init_b200 import scenes
    det = CONFIGS[cfg][2]
    if cfg == "C4":
        return make_c4(n_scan, n_map)
    c = scenes.make_config("C2", seed=1, N=n_scan, M=n_map)   # ("C2" = the generic box scene generator; sizes come from the arguments)
    if det != 450.0:
        c["body_xyz"] = scenes.scan_points(c["scene"], c["pose_gt"], n_scan, seed=2, det_range=det, sigma=0.01, open_air_frac=0.01, order="voxel")
    if cfg == "C2" and world > 1:
        parts = [c["body_xyz"]]
        for r in range(1, world):
            parts.append(scenes.scan_points(c["scene"], c["pose_gt"], n_scan, seed=2 + 1000 * r, det_range=det, sigma=0.01, open_air_frac=0.01,
                                            order="voxel"))
        c["body_xyz"] = np.ascontiguousarray(np.concatenate(parts, 0))
    return c


def make_c4(n_scan: int, n_map: int):
    """C4: a long hall whose map points are ordered along x, so that Add_Points batches in that order are a sensor walking through it."""
    from lidar_imu_init_b200 import scenes
    ds = 0.15
    scene = scenes.scene_for_points(n_map, ds, aspect=(1200.0, 160.0, 20.0))
    mp = scenes.map_points(scene, ds, n_map, seed=1)
    mp = np.ascontiguousarray(mp[np.argsort(mp[:, 0], kind="stable")])
    gt = scenes.default_sensor_pose(scene)
    gt.pos_end[0] = 0.5 * scene.L
    body = scenes.scan_points(scene, gt, n_scan, seed=2, det_range=150.0, sigma=0.01, open_air_frac=0.01, order="voxel")
    return dict(scene=scene, map_xyz=mp, body_xyz=body, pose_gt=gt, pose_init=scenes.perturb_pose(gt, 3), ds=ds, imu_en=False, name="C4")


def scenes_perturb(p):
    from lidar_imu_init_b200 import scenes
    return scenes.perturb_pose(p, 77, dtheta_deg=0.05, dpos=0.01)


def config_dict(cfg: str, n_scan: int, n_map: int, ds: float):
    """The workload description BOTH arms print (same keys, same values: the driver compares them)."""
    return {"workload": CONFIGS[cfg][3], "scan_points": n_scan, "map_points": n_map, "filter_size_map": ds, "imu_en": False,
            "initial_pose": "ground truth (+) 0.5 deg / 5 cm", "open_air_frac": 0.01, "scan_order": "voxel-grid order"}


# ------------------------------------------------------------------------------------------------------
def _interleave_memory():
    """set_mempolicy(MPOL_INTERLEAVE, all nodes): the verbatim ikd-Tree is built by one thread -- without this its 0.9 GB of nodes
    land on one NUMA node and the 128-thread search arm measures that node's memory controller (1.2e6 .. 7.5e6 points*iters/s box to
    box in round 1). Best effort."""
    try:
        import ctypes
        nodes = [int(d[4:]) for d in os.listdir("/sys/devices/system/node") if d.startswith("node") and d[4:].isdigit()]
        if len(nodes) < 2:
            return "single NUMA node"
        mask = ctypes.c_ulong(sum(1 << n for n in nodes))
        libc = ctypes.CDLL(None, use_errno=True)
        rc = libc.syscall(238, 3, ctypes.byref(mask), ctypes.c_ulong(max(nodes) + 2))   # SYS_set_mempolicy, MPOL_INTERLEAVE
        return f"interleaved over {len(nodes)} NUMA nodes" if rc == 0 else f"set_mempolicy failed (errno {ctypes.get_errno()})"
    except Exception as e:
        return f"unavailable ({e!r})"


def _bind_near_gpu(torch, local_rank):
    """Run the launching thread, and allocate the pinned frame it hands to the library, on the NUMA node the GPU hangs off: the search
    kernel reads the frame over PCIe in place, and a frame on the other socket adds an inter-socket hop to every read (the e2e step
    was 0.268 .. 0.305 ms box to box without this). What a deployment does with numactl. Best effort.
    -> (affinity to restore for the CPU arm, description)"""
    try:
        pr = torch.cuda.get_device_properties(local_rank)
        bdf = f"{pr.pci_domain_id:04x}:{pr.pci_bus_id:02x}:{pr.pci_device_id:02x}.0"
        with open(f"/sys/bus/pci/devices/{bdf}/numa_node") as f:
            node = int(f.read())
        if node < 0:
            return None, f"not bound (GPU {bdf}: NUMA node unknown)"
        cpus = set()
        with open(f"/sys/devices/system/node/node{node}/cpulist") as f:
            for part in f.read().strip().split(","):
                a, _, b = part.partition("-")
                cpus.update(range(int(a), int(b or a) + 1))
        allowed = os.sched_getaffinity(0)
        use = cpus & allowed
        if not use:
            return None, f"not bound (no allowed CPU on node {node})"
        os.sched_setaffinity(0, use)
        import ctypes
        mask = ctypes.c_ulong(1 << node)
        libc = ctypes.CDLL(None, use_errno=True)
        rc = libc.syscall(238, 1, ctypes.byref(mask), ctypes.c_ulong(node + 2))   # SYS_set_mempolicy, MPOL_PREFERRED
        return allowed, f"launch thread on the {len(use)} CPUs of NUMA node {node} (GPU {bdf}), pinned frame " + \
            ("preferred on that node" if rc == 0 else f"placement left to first touch (set_mempolicy errno {ctypes.get_errno()})")
    except Exception as e:
        return None, f"not bound ({e!r})"


def _cpu_env():
    # read by libgomp when the oracle library is loaded: one thread per core, spread over the sockets, no migration
    os.environ.setdefault("OMP_PROC_BIND", "spread")
    os.environ.setdefault("OMP_PLACES", "cores")


def cpu_reference_pass(c, sample_points: int, threads: int, reps: int, warm: int, om=None):
    """Time the CPU path (oracle) on a bounded sample of the scan against the full map."""
    from oracle import oracle as orc
    kind = "reference" if orc.has_ikd() else "port"
    build_s = 0.0
    if om is None:
        om = orc.OracleMap(c["ds"], 1 if orc.has_ikd() else 0)
        t0 = time.time()
        om.build(c["map_xyz"])
        build_s = time.time() - t0
    step = max(1, len(c["body_xyz"]) // sample_points)
    body = np.ascontiguousarray(c["body_xyz"][::step][:sample_points])
    sc = orc.OracleScan(body)
    p = c["pose_init"]
    ts = []
    res = None
    for i in range(warm + reps):
        t = time.perf_counter()
        res = sc.iterate(om, p.rot_end, p.pos_end, p.R_LI, p.T_LI, c["imu_en"], True, nthreads=threads)
        dt = time.perf_counter() - t
        if i >= warm:
            ts.append(dt)
    return dict(kind=kind, n=len(body), times=ts, build_s=build_s, om=om, sc=sc, result=res)


def run_reference(args, rank, world):
    if rank != 0:
        return
    _cpu_env()
    numa = _interleave_memory()
    threads = os.cpu_count() or 1
    cfg = args.config
    c = make_workload(cfg if cfg != "C4" else "C2", 1, args.scan_points, min(args.map_points, 10_000_000))
    # size the per-step sample so that steps+warmup stay within ~2 minutes
    probe = cpu_reference_pass(c, 12000, threads, 1, 1)
    per_pt = probe["times"][0] / probe["n"]
    budget = 100.0 / max(1, args.steps + args.warmup)
    n_s = int(min(args.scan_points, max(2000, budget / per_pt)))
    om, p = probe["om"], c["pose_init"]
    from oracle import oracle as orc
    step = max(1, len(c["body_xyz"]) // n_s)
    body = np.ascontiguousarray(c["body_xyz"][::step][:n_s])
    sc = orc.OracleScan(body)
    ts = []
    for i in range(args.warmup + args.steps):
        t = time.perf_counter()
        sc.iterate(om, p.rot_end, p.pos_end, p.R_LI, p.T_LI, False, True, nthreads=threads)
        if i >= args.warmup:
            ts.append(time.perf_counter() - t)
    ms = 1e3 * float(np.median(ts))
    val = len(body) / (ms * 1e-3)
    v3 = None
    if threads > 3:
        t3 = []
        for i in range(3):
            t = time.perf_counter()
            sc.iterate(om, p.rot_end, p.pos_end, p.R_LI, p.T_LI, False, True, nthreads=3)
            t3.append(time.perf_counter() - t)
        v3 = len(body) / float(np.median(t3[1:]))
    sample = (f"{len(body)} of {args.scan_points} scan points per step vs the full {len(c['map_xyz'])}-point map, search pass, {threads} OpenMP threads "
              f"(OMP_PROC_BIND={os.environ.get('OMP_PROC_BIND')}, OMP_PLACES={os.environ.get('OMP_PLACES')}, tree memory {numa}), median of the steps")
    out = {
        "impl": "reference", "metric": CONFIGS[cfg][4], "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms, "higher_is_better": True, "scaling": "strong" if cfg == "C5" else "weak", "vs_baseline": None,
        "dtype": "f32 kNN / f64 plane+Jacobian", "data": "synthetic", "iters_per_s": val / args.scan_points,
        "config": config_dict(cfg, args.scan_points, args.map_points, c["ds"]),
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": threads, "kind": probe["kind"], "sample": sample,
                         "build_s": probe["build_s"], "value_mp_proc_num_3": v3, "ms_per_step_all": [1e3 * t for t in ts]},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(out)


# ------------------------------------------------------------------------------------------------------
def grow_map_c4(g, c, n_start: int, batch: int):
    """C4: Build(first n_start points) then Add_Points(downsample) batches to the end of the hall, each timed (wall clock incl. the H2D
    of the batch); one Delete_Point_Boxes over the first 40 m of the hall at the end."""
    import torch
    mp = c["map_xyz"]
    t0 = time.time()
    g.map_build(mp[:n_start])
    build_s = time.time() - t0
    ts, sizes = [], []
    for lo in range(n_start, len(mp), batch):
        b = mp[lo:lo + batch]
        torch.cuda.synchronize()
        t = time.perf_counter()
        g.map_add_points(b, True)
        ts.append((time.perf_counter() - t) * 1e3)
        sizes.append(len(b))
    n_before = g.map_validnum()
    sc = c["scene"]
    boxes = np.array([[-1.0, -1.0, -1.0, 40.0, sc.W + 1.0, sc.H + 1.0]], np.float32)
    torch.cuda.synchronize()
    t = time.perf_counter()
    n_del = g.map_delete_boxes(boxes)
    del_ms = (time.perf_counter() - t) * 1e3
    return {"build_points": n_start, "map_build_s": build_s, "add_batches": len(ts), "points_per_batch": batch, "add_ms_median": float(np.median(ts)) if ts else None,
            "add_ms_max": float(np.max(ts)) if ts else None, "add_points_per_s": float(np.sum(sizes) / (np.sum(ts) * 1e-3)) if ts else None,
            "map_points_after_growth": n_before, "delete_boxes_ms": del_ms, "deleted_points": int(n_del), "map_points_final": g.map_validnum(),
            "map_stats": g.map_stats(), "note": "Add_Points(downsample_on) batches of new surface, wall clock per call incl. H2D and the counters' D2H; "
                                                "one Delete_Point_Boxes over the first 40 m of the hall"}


def run_gpu(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    from lidar_imu_init_b200 import capi, sharding

    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device: the product has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    affinity0, host_binding = (None, "off (--no-bind)") if args.no_bind else _bind_near_gpu(torch, local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    cfg = args.config
    strong = cfg == "C5"
    sampler = ClockSampler(local_rank)    # polling starts now, recording at the first timed loop: NVML's first queries (milliseconds,
    sampler.start()                       # under a driver lock) stay out of the timed regions

    c = make_workload(cfg, world, args.scan_points, args.map_points)
    NF = len(c["body_xyz"])                       # points of the whole frame
    p = c["pose_init"]
    g = capi.LiInitGpu(c["ds"], max_map_points=int(args.map_points * 1.2) + 1000, max_scan_points=NF + 16, device_id=local_rank,
                       knn_group_lanes=args.group, brick_cells_log2=args.brick, knn_index=args.knn_index)
    kidx = g.knn_index()
    stream = torch.cuda.Stream(device=dev)
    g.set_stream(stream.cuda_stream)
    sharding.attach_comm(g, rank, world)          # N > 1: NCCL communicator INSIDE the library (liinit_comm_init)
    g.set_reseed(False)                           # the metric is the FIRST search pass of a scan: every timed step searches from scratch
    growth = None
    if cfg == "C4":
        growth = grow_map_c4(g, c, 5_000_000 if args.map_points >= 10_000_000 else args.map_points // 10, args.scan_points)
        build_s = growth["map_build_s"]
    else:
        t0 = time.time()
        g.map_build(c["map_xyz"])
        build_s = time.time() - t0
    # pinned host frame (packed xyz: 12 bytes per point cross PCIe, the device widens to float4) for the e2e path
    body4 = torch.from_numpy(np.ascontiguousarray(c["body_xyz"], dtype=np.float32)).pin_memory()
    SCAN_STRIDE = 3
    g.scan_upload_ptr(body4.data_ptr(), SCAN_STRIDE, NF)
    N = g.comm_info()["shard_n"]                  # points this rank processes
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def step_resident():
        """frame resident: one search pass; results (summed over the ranks inside the library when N > 1) on the host at return"""
        return g.icp_iterate(p.rot_end, p.pos_end, p.R_LI, p.T_LI, False, True)

    def step_e2e():
        # liinit_scan_attach_host -- the search kernel pulls this rank's slot of the pinned host frame over PCIe itself (N*12 bytes per
        # rank, inside the timed region); the 160-double result block comes back to the host before the call returns.
        g.scan_attach_ptr(body4.data_ptr(), SCAN_STRIDE, NF)
        return step_resident()

    def step_e2e_staged():
        # same step through liinit_scan_upload (cudaMemcpyAsync + repack in front of the search), for comparison
        g.scan_upload_ptr(body4.data_ptr(), SCAN_STRIDE, NF)
        return step_resident()

    def timed(fn, steps, warmup, do_flush):
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        knn_ms, plane_ms = [], []
        with torch.cuda.stream(stream):
            for _ in range(warmup):
                fn()
            torch.cuda.synchronize()
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize()
            l0 = g.launch_count()
            for i in range(steps):
                if do_flush:
                    flush.fill_(i & 0xff)   # > L2 (126 MB): evicts the map between timed steps; outside the events
                ev[i][0].record(stream)
                res = fn()
                ev[i][1].record(stream)
                a, b = g.last_pass_kernel_times()
                knn_ms.append(a)
                plane_ms.append(b)
            torch.cuda.synchronize()
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize()
            l1 = g.launch_count()
        ms = [a.elapsed_time(b) for a, b in ev]
        timed.last_steps = ms
        timed.last_result = res
        return float(np.sum(ms)), (l1 - l0), float(np.mean(knn_ms)), float(np.mean(plane_ms))

    sampler.recording.set()               # samples across all timed loops (each lasts only a few ms)
    tot_ms, launches, knn_ms, plane_ms = timed(step_resident, args.steps, args.warmup, True)
    step_ms = list(timed.last_steps)
    last_step = timed.last_result
    warm_ms, _, knn_warm, plane_warm = timed(step_resident, args.steps, 1, False)
    e2e_ms, _, e2e_knn_ms, e2e_plane_ms = timed(step_e2e, args.steps, args.warmup, True)
    e2e_staged_ms, _, _, _ = timed(step_e2e_staged, args.steps, args.warmup, True)
    g.scan_upload_ptr(body4.data_ptr(), SCAN_STRIDE, NF)
    clocks = sampler.stop()

    def maxr(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    tot_ms, warm_ms, e2e_ms, e2e_staged_ms = maxr(tot_ms), maxr(warm_ms), maxr(e2e_ms), maxr(e2e_staged_ms)
    ms_step = tot_ms / args.steps
    value = NF / (ms_step * 1e-3)
    e2e_val = NF / (e2e_ms / args.steps * 1e-3)
    peak, peak_src = _peaks()
    ach = ALG_BYTES_PER_POINT * N / (knn_ms * 1e-3) / 1e9
    # the result the timed steps produce (same call, same stream as the timed loops)
    with torch.cuda.stream(stream):
        H, b, m_sel, rs = step_resident()
    multi = None
    if world > 1:
        # the reduction verified on hardware, every run: sum of the ranks' OWN blocks (fetched through liinit_comm_last_local,
        # gathered over torch.distributed) against what liinit_icp_iterate returned on this rank
        loc = g.comm_last_local()
        box = [None] * world
        dist.all_gather_object(box, loc)
        tot = np.sum(np.stack(box, 0), 0)
        red = np.concatenate([H.reshape(-1), b, [rs, float(m_sel)]])
        multi = {"m_sum_of_ranks": int(round(tot[157])), "m_reduced": int(m_sel), "m_per_rank": [int(round(x[157])) for x in box],
                 "rel_err_HtH_vs_rank_sum": float(np.abs(red[:144] - tot[:144]).max() / np.abs(tot[:144]).max()),
                 "rel_err_Htr_vs_rank_sum": float(np.abs(red[144:156] - tot[144:156]).max() / np.abs(tot[144:156]).max()),
                 "collective": "sum of 160 f64 over the ranks inside liinit_icp_iterate: " + g.comm_mode()}

    conf = config_dict(cfg, args.scan_points, args.map_points, c["ds"])
    out = {
        "metric": CONFIGS[cfg][4], "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step,
        "higher_is_better": True, "scaling": "strong" if strong else "weak", "vs_baseline": None, "dtype": "f32 kNN / f64 plane+Jacobian",
        "data": "synthetic", "iters_per_s": 1e3 / ms_step, "iters_per_s_l2_warm": 1e3 / (warm_ms / args.steps),
        "config": conf,
        "details": {"frame_points": NF, "points_per_gpu": N,
                    "parallelism": "1 GPU" if world == 1 else (f"{world} GPUs, map replicated, frame of {NF} points cut into {world} slots by the library, "
                                                               "accumulators summed over the ranks inside liinit_icp_iterate (" + g.comm_mode() + ")"),
                    "l2": "flushed between timed steps (256 MiB memset outside the events)", "knn_index": KNN_NAME[kidx],
                    "knn_group_lanes": (args.group or "auto (by frame size: 4 lanes beyond 70k points per GPU)") if kidx == 1 else None, "brick_cells_log2": args.brick or 3,
                    "selected_points": int(m_sel), "map_build_s": build_s, "map_points_live": g.map_validnum(),
                    "step_ms": {"min": float(np.min(step_ms)), "median": float(np.median(step_ms)), "max": float(np.max(step_ms)),
                                "note": "this rank's device time of the timed steps; ms_per_step is their mean, max over ranks"}},
        "e2e": {"value": e2e_val, "unit": UNIT, "h2d_bytes_per_step": int(N * 12 + 192), "d2h_bytes_per_step": 160 * 8,
                "ms_per_step": e2e_ms / args.steps,
                "host_input": ("pinned packed xyz, read by the search kernel over PCIe (liinit_scan_attach_host, no staging copy)" if world == 1 else
                               "pinned packed xyz of the whole frame; every rank's search kernel reads ITS SLOT over PCIe (liinit_scan_attach_host; the "
                               "other slots would be copied when map_incremental or a download needs the whole frame)"),
                "ms_per_step_staged_copy": e2e_staged_ms / args.steps,
                "kernel_ms": e2e_knn_ms, "plane_kernel_ms": e2e_plane_ms, "host_binding": host_binding},
        "gpu_launches": int(launches),
        "clocks": clocks,
        "roofline": {"bound": "hbm", "kernel": KNN_KERNEL[kidx], "achieved": ach, "peak": peak,
                     "unit": "GB/s", "frac": ach / peak, "peak_source": peak_src, "traffic": NCU_DRAM_BYTES_KNN[kidx] if cfg == "C2" else None,
                     "algorithmic_bytes_per_launch": ALG_BYTES_PER_POINT * N, "kernel_ms": knn_ms, "plane_kernel_ms": plane_ms,
                     "kernel_ms_l2_warm": knn_warm, "plane_kernel_ms_l2_warm": plane_warm,
                     "note": "traffic = dram__bytes_read.sum + dram__bytes_write.sum of one launch of this kernel from the ncu --set full capture in "
                             + NCU_DRAM_SOURCE[kidx] + " (C2, cold cache: ncu flushes between replays), bytes per launch"},
    }
    if multi:
        out["multi_gpu_check"] = multi
    if growth:
        out["map_growth"] = growth
    # ---- extras (not part of the contract value): the other pass kinds of a real scan -----------------------
    if world == 1 and cfg != "C4":
        try:
            from lidar_imu_init_b200 import host
            rts = []
            for _ in range(10):
                g.icp_iterate(p.rot_end, p.pos_end, p.R_LI, p.T_LI, False, False)
                rts.append(g.last_pass_timing()[0])
            # a scan's LATER search passes start from the previous pass's neighbours (liinit_set_reseed, the library's default)
            g.set_reseed(True)
            p2 = scenes_perturb(p)
            sts = []
            for _ in range(6):
                g.icp_iterate(p.rot_end, p.pos_end, p.R_LI, p.T_LI, False, True)
                g.icp_iterate(p2.rot_end, p2.pos_end, p2.R_LI, p2.T_LI, False, True)      # the pose moved by 0.05 deg / 1 cm, as after an update
                sts.append(g.last_pass_kernel_times())
            seeded_knn, seeded_plane = float(np.median([a for a, _ in sts])), float(np.median([b for _, b in sts]))
            st0 = host.state_from_pose(p.rot_end, p.pos_end, p.R_LI, p.T_LI)
            sus = []
            for _ in range(5):
                g.scan_upload_ptr(body4.data_ptr(), SCAN_STRIDE, NF)
                t0 = time.perf_counter()
                _, ss = host.scan_update(g, st0, 5, False)
                sus.append((time.perf_counter() - t0) * 1e3)
            gt = c["pose_gt"]
            for rep in range(2):   # the first call pays the lazy loading of the update kernels; report the second
                g.icp_iterate(p.rot_end, p.pos_end, p.R_LI, p.T_LI, False, True)
                t0 = time.perf_counter()
                na, nn = g.map_incremental(gt.rot_end, gt.pos_end, gt.R_LI, gt.T_LI, c["ds"])
                mi_ms = (time.perf_counter() - t0) * 1e3
            out["extras"] = {"reuse_pass_kernel_ms": float(np.median(rts)), "seeded_search_pass_knn_ms": seeded_knn, "seeded_search_pass_plane_ms": seeded_plane,
                             "scan_update_ms": float(np.median(sus)),
                             "scan_update_iterations": ss["iterations"], "scan_update_search_passes": ss["search_passes"],
                             "map_incremental_ms": mi_ms, "map_incremental_added": [na, nn],
                             "note": "seeded_search_pass = a LATER search pass of the same scan (pose moved by 0.05 deg / 1 cm), started from the previous "
                                     "pass's neighbours; scan_update = liinit_scan_update (host C++ IESKF loop, max_iteration 5) on the resident scan, wall clock; "
                                     "map_incremental = classification + both inserts for the frame, wall clock"}
        except Exception as e:
            out["extras"] = {"error": repr(e)}
    if rank == 0 and world == 1 and not args.no_cpu and cfg != "C4":
        if affinity0:
            os.sched_setaffinity(0, affinity0)   # the CPU arm gets the whole machine back (its threads inherit this mask)
        _cpu_env()
        numa = _interleave_memory()
        threads = os.cpu_count() or 1
        try:
            r = cpu_reference_pass(c, min(NF, args.cpu_sample), threads, 3, 1)
            v = r["n"] / float(np.median(r["times"]))
            out["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": threads, "kind": r["kind"],
                                   "sample": f"search pass over {r['n']} of {NF} scan points vs the full {args.map_points}-pt map "
                                             f"(verbatim ikd-Tree Build {r['build_s']:.1f}s excluded; OMP_PROC_BIND={os.environ.get('OMP_PROC_BIND')}, "
                                             f"tree memory {numa}), median of 3", "iters_per_s": v / NF}
            if r["n"] == NF:
                # full-size parity for free: the oracle just evaluated the very pass the GPU was timed on
                Ho, bo, mo = r["result"]
                out["parity"] = {"checked_against": "oracle (verbatim ikd-Tree + restated loop), the whole frame, same pose",
                                 "m_gpu": int(m_sel), "m_oracle": int(mo), "m_equal": bool(int(m_sel) == int(mo)),
                                 "rel_err_HtH": float(np.abs(H - Ho).max() / np.abs(Ho).max()), "rel_err_Htr": float(np.abs(b - bo).max() / np.abs(bo).max())}
            r3 = cpu_reference_pass(c, min(NF, args.cpu_sample, 60000), min(3, threads), 2, 1, om=r["om"]) if threads > 3 else None
            if r3:
                out["cpu_baseline"]["value_mp_proc_num_3"] = r3["n"] / float(np.median(r3["times"]))
        except Exception as e:  # the oracle is test infrastructure; its absence must not hide the GPU number
            out["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": threads, "kind": "unavailable", "sample": repr(e)}
    if rank == 0 and args.dump_outputs:
        H, b, m, rs = last_step
        dump_outputs(args.dump_outputs, {"HtH": H, "Htr": b, "selected_points": m, "residual_sum": rs})
    if rank == 0:
        emit(out)
    g.close()
    if world > 1:
        dist.destroy_process_group()


def dump_outputs(out_dir, arrays):
    """--dump-outputs: what the last timed step returned, one float64 <name>.npy each. The workload is generated from fixed seeds, so
    two builds run with the same arguments can be compared output for output."""
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(a, np.float64))


def main():
    # The reference's ikd-Tree printf()s to stdout ("Multi thread started", ...): keep fd 1 clean for the one
    # JSON line by pointing it at stderr for the whole run and writing the result to the saved descriptor.
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="C2", choices=sorted(CONFIGS))
    ap.add_argument("--scan-points", type=int, default=0, help="0 = the configuration's size")
    ap.add_argument("--map-points", type=int, default=0, help="0 = the configuration's size")
    ap.add_argument("--group", type=int, default=0)
    ap.add_argument("--brick", type=int, default=0)
    ap.add_argument("--knn-index", type=int, default=0, help="0 = library default, 1 = bricks (lockstep groups), 2 = cells (cell directory)")
    ap.add_argument("--cpu-sample", type=int, default=240_000)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-bind", action="store_true", help="do not bind the launch thread / pinned frame to the GPU's NUMA node")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one returned (HtH, Htr, selected points, residual sum) to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs needs --impl ours: the reference arm sizes its scan sample by its own speed, so its outputs vary run to run")
    args.scan_points = args.scan_points or CONFIGS[args.config][0]
    args.map_points = args.map_points or CONFIGS[args.config][1]
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    run_gpu(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
