"""Device time of liinit_map_knn_search_device (csrc/knn_general.cuh) on the flagship scene, next to the k = 5 search of
liinit_map_nearest_search. Prints one JSON line (and writes it to --out when given).

Scene: C2 (scenes.make_config("C2", seed=1)), 5M map points, its 240k scan points in the world frame as queries, plus 10k far queries
(scan points moved 50 m / 1 km in random directions). For every k in {1, 5, 16, 32} x max_dist in {5, inf}: CUDA events around each
device-form call on the library's stream, L2 overwritten (256 MiB memset outside the events) before each call, median and spread over
--reps calls; the last timed output is compared with the host form's bit for bit. The k = 5 baseline is liinit_map_nearest_search in the
same process: its kernels (the 5-NN search and the gather of the neighbours) timed by torch.profiler, as is the new kernel at
k = 5 / max_dist = 5 for a like-for-like figure.

    python tools/knn_general_bench.py [--reps 20] [--out FILE]
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def device_info():
    import torch
    info = {"device": torch.cuda.get_device_name(0)}
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(0)
        info["power_limit_w"] = pynvml.nvmlDeviceGetPowerManagementLimit(h) / 1000.0
        info["sm_max_mhz"] = pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM)
    except Exception as e:   # reported, not guessed
        info["power_limit_w"] = None
        info["nvml_error"] = str(e)
    return info


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--map", type=int, default=5_000_000)
    ap.add_argument("--queries", type=int, default=240_000)
    ap.add_argument("--far", type=int, default=10_000)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    from lidar_imu_init_b200 import _build, capi, scenes
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: this benchmark measures the GPU only")
    _build.build_gpu()
    res = device_info()
    c = scenes.make_config("C2", seed=1, N=a.queries, M=a.map)
    p = c["pose_init"]
    q = np.ascontiguousarray((p.rot_end @ (p.R_LI @ c["body_xyz"].T.astype(np.float64) + p.T_LI[:, None]) + p.pos_end[:, None]).T, np.float32)
    rng = np.random.default_rng(11)
    dirs = rng.normal(size=(a.far, 3))
    dirs /= np.linalg.norm(dirs, axis=1, keepdims=True)
    dist = np.where(np.arange(a.far) < a.far // 2, 50.0, 1000.0)[:, None]
    far = (q[rng.integers(0, len(q), a.far)] + dist * dirs).astype(np.float32)
    g = capi.LiInitGpu(c["ds"], max_map_points=a.map + 1_000_000, max_scan_points=a.queries)
    t0 = time.time()
    g.map_build(c["map_xyz"])
    res.update(scene="C2 seed 1", map_points=g.map_validnum(), queries=len(q), far_queries=a.far, map_build_s=time.time() - t0,
               bricks=g.map_stats()["bricks"], reps=a.reps, l2="overwritten before every timed call (256 MiB memset outside the events)")
    dev = torch.device("cuda:0")
    stream = torch.cuda.Stream()
    g.set_stream(stream.cuda_stream)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def timed(qs, k, md):
        tq = torch.from_numpy(np.ascontiguousarray(qs)).to(dev)
        n = len(qs)
        tx = torch.empty((n, k, 3), dtype=torch.float32, device=dev)
        td = torch.empty((n, k), dtype=torch.float32, device=dev)
        tn = torch.empty(n, dtype=torch.int32, device=dev)
        ms = []
        with torch.cuda.stream(stream):
            for i in range(a.reps + 2):
                flush.fill_(i & 0xff)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream)
                g.knn_search_device(tq.data_ptr(), 3, n, k, md, tx.data_ptr(), td.data_ptr(), tn.data_ptr())
                e1.record(stream)
                e1.synchronize()
                if i >= 2:   # two warm-up calls (module load, the brick list)
                    ms.append(e0.elapsed_time(e1))
        torch.cuda.synchronize()
        hx, hd, hn = g.knn_search(qs, k, md)
        same = bool(np.array_equal(hx, tx.cpu().numpy()) and np.array_equal(hd, td.cpu().numpy()) and np.array_equal(hn, tn.cpu().numpy()))
        return {"median_ms": float(np.median(ms)), "min_ms": float(np.min(ms)), "max_ms": float(np.max(ms)),
                "found_mean": float(hn.mean()), "equals_host_form": same}

    rows = []
    for k in (1, 5, 16, 32):
        for md in (5.0, float("inf")):
            r = {"k": k, "max_dist": "inf" if md == float("inf") else md}
            r["scan"] = timed(q, k, md)
            r["far"] = timed(far, k, md)
            rows.append(r)
            print(json.dumps(r), file=sys.stderr)
    res["knn_search_device"] = rows

    # k = 5 baseline: liinit_map_nearest_search (host entry point: staging, search kernel, gather kernel, copies) -- its kernels' device time
    from torch.profiler import ProfilerActivity, profile
    with torch.cuda.stream(stream):
        g.nearest_search(q)
        n = len(q)
        tq = torch.from_numpy(q).to(dev)
        tx = torch.empty((n, 5, 3), dtype=torch.float32, device=dev)
        td = torch.empty((n, 5), dtype=torch.float32, device=dev)
        tn = torch.empty(n, dtype=torch.int32, device=dev)
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for i in range(a.reps):
                flush.fill_(i & 0xff)
                g.nearest_search(q)
                flush.fill_(i & 0xff)
                g.knn_search_device(tq.data_ptr(), 3, n, 5, 5.0, tx.data_ptr(), td.data_ptr(), tn.data_ptr())
            torch.cuda.synchronize()
    per = {}
    for ev in prof.events():
        if ev.device_type.name != "CUDA":
            continue
        for key in ("k_knn_queries", "k_gather_xyz", "k_knn_general", "k_knn_cells_queries"):
            if key in ev.name:
                per.setdefault(key, []).append(ev.device_time if hasattr(ev, "device_time") else ev.cuda_time)
    prof_ms = {k: {"median_ms": float(np.median(v)) / 1e3, "calls": len(v)} for k, v in per.items()}
    base = sum(v["median_ms"] for k, v in prof_ms.items() if k != "k_knn_general")
    new = prof_ms.get("k_knn_general", {}).get("median_ms")
    xn, dn, cn = g.nearest_search(q)
    xg, dg, cg = g.knn_search(q, 5, 5.0)
    res["k5_baseline"] = {"kernels_profiler": prof_ms, "nearest_search_kernels_ms": base, "knn_general_k5_md5_ms": new,
                          "ratio_general_over_nearest": (new / base) if (new and base) else None,
                          "same_counts_and_d2_as_nearest_search": bool(np.array_equal(cn, cg) and np.array_equal(dn, dg))}
    g.set_stream(0)
    g.close()
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
