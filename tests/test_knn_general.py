"""KD_TREE::Nearest_Search(point, k, ..., max_dist) for any 1 <= k <= 32 and any max_dist (liinit_map_knn_search / _device,
csrc/knn_general.cuh). The CPU tests run the kernels on the emulated library (tests/emul); the GPU tests run them on the device.
Arbiters: the verbatim ikd-Tree's stored answers (tests/golden/ikd_knn.npz, tools/make_golden.py ikd_knn; inputs in tests/knn_general_cases.py) and, where oracle/_ref is
built, the tree itself; the oracle's brute force (k <= 16, the size of its candidate heap) and the numpy brute force below (any k)."""
import ctypes as C
import math
import os
import shutil
import subprocess

import numpy as np
import pytest

import ikd_cases
import knn_general_cases as kc
import liinit_emul as le
from knn_general_cases import knn_search

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
INF = float("inf")
emul = pytest.mark.skipif(not le.available(), reason="needs g++ and the CUDA headers")


def bruteforce(mp, q, k, max_dist):
    """Exact k-NN with the library's rules: fp32 (dx*dx + dy*dy) + dz*dz, d2 <= max_dist compared in double, ascending (d2, x), and no
    neighbours for a query with a non-finite coordinate."""
    mp = np.ascontiguousarray(mp, np.float32)
    q = np.ascontiguousarray(q, np.float32)
    xyz = np.zeros((len(q), k, 3), np.float32)
    d2 = np.full((len(q), k), -1, np.float32)
    cnt = np.zeros(len(q), np.int32)
    for s in range(0, len(q), 64):
        qq = q[s:s + 64]
        dx, dy, dz = (qq[:, None, a] - mp[None, :, a] for a in range(3))
        d = (dx * dx + dy * dy) + dz * dz
        for i in range(len(qq)):
            if not np.isfinite(qq[i]).all():   # a non-finite query has no neighbours
                continue
            ok = np.flatnonzero(d[i].astype(np.float64) <= max_dist)
            o = ok[np.lexsort((mp[ok, 0], d[i, ok]))][:k]
            cnt[s + i] = len(o)
            xyz[s + i, :len(o)] = mp[o]
            d2[s + i, :len(o)] = d[i, o]
    return xyz, d2, cnt


def assert_same(got, want, q=None):
    """Counts and distances equal, neighbours equal. With q: which of several points tied at exactly the k-th distance is returned is
    not part of the claim (the reference's choice depends on its traversal), so a neighbour at the k-th distance of a full answer only
    has to lie at that distance from its query. Without q: bit for bit."""
    (x, d, n), (xw, dw, nw) = got, want
    assert np.array_equal(n, nw), np.flatnonzero(n != nw)[:10]
    assert np.array_equal(d, dw), np.flatnonzero((d != dw).any(1))[:10]
    if q is None:
        assert np.array_equal(x, xw), np.flatnonzero((x != xw).any((1, 2)))[:10]
        return
    k = d.shape[1]
    tied = (n == k)[:, None] & (d == d[:, -1:])
    diff = (x != xw).any(2)
    assert not (diff & ~tied).any(), np.flatnonzero((diff & ~tied).any(1))[:10]
    q = np.asarray(q, np.float32)[:, None, :]
    dx, dy, dz = (q[..., a] - x[..., a] for a in range(3))
    assert np.array_equal(((dx * dx + dy * dy) + dz * dz)[tied], d[tied])


def golden():
    c, q = kc.knn_general_case()
    G = np.load(kc.GOLD_KNN)
    assert str(G["inputs"]) == ikd_cases.digest(c["map_xyz"], q), "the inputs differ from those the stored ikd-Tree answers were computed on"
    return c, q, G


def golden_answer(G, mp, q, k, md):
    """the stored answer as (xyz, d2, cnt); d2 follows from the rows"""
    cnt = G[f"cnt_k{k}_{md}"]
    rows = G[f"nbr_k{k}_{md}"].astype(np.int32)
    xyz = ikd_cases.neighbours(rows, mp)
    dx, dy, dz = (q[:, None, a] - xyz[:, :, a] for a in range(3))
    d2 = np.where(rows >= 0, (dx * dx + dy * dy) + dz * dz, np.float32(-1))
    return xyz, d2.astype(np.float32), cnt


def ikd_live(mp, q, k, md, ds):
    """the verbatim tree itself (oracle/_ref/libikd_ref.so), or None where it is not built"""
    lib = os.path.join(ROOT, "oracle", "_ref", "libikd_ref.so")
    if not os.path.exists(lib):
        return None
    L = C.CDLL(lib)
    L.ikdref_create.restype = C.c_void_p
    L.ikdref_create.argtypes = [C.c_float]
    L.ikdref_destroy.argtypes = [C.c_void_p]
    L.ikdref_build.argtypes = [C.c_void_p, C.c_void_p, C.c_int]
    L.ikdref_nearest.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_double, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]
    mp = np.ascontiguousarray(mp, np.float32)
    q = np.ascontiguousarray(q, np.float32)
    t = L.ikdref_create(float(ds))
    L.ikdref_build(t, mp.ctypes.data, len(mp))
    xyz = np.zeros((len(q), k, 3), np.float32)
    d2 = np.zeros((len(q), k), np.float32)
    cnt = np.zeros(len(q), np.int32)
    L.ikdref_nearest(t, q.ctypes.data, len(q), k, md, xyz.ctypes.data, d2.ctypes.data, cnt.ctypes.data, 8)
    L.ikdref_destroy(t)
    return xyz, d2, cnt


def _far_queries(mp):
    rng = np.random.default_rng(5)
    base = mp[rng.choice(len(mp), 12)]
    dirs = rng.normal(size=(12, 3))
    dirs /= np.linalg.norm(dirs, axis=1, keepdims=True)
    far = (base + np.repeat([20.0, 300.0, 5e3, 2e5], 3)[:, None] * dirs).astype(np.float32)
    return np.concatenate([far, np.array([[3e5, 1, 2], [-1, -3.1e5, 0], [2, 2, 1e6]], np.float32)])


# ---- CPU: the kernels on the emulated library ------------------------------------------------------------------------------------------

@emul
@pytest.mark.parametrize("k", kc.KNN_KS)
def test_golden_grid_emul(k):
    """every (k, max_dist) of the grid on a fifth of the stored queries (all kinds: scan, open air, 50 m, 1 km, beyond the key range)"""
    c, q, G = golden()
    mp = c["map_xyz"]
    sel = np.r_[0:len(q):5, len(q) - 8:len(q)]
    g = le.EmulGpu(c["ds"], max_map_points=200_000, max_scan_points=20_000)
    g.map_build(mp)
    for md in kc.KNN_MAX_DISTS:
        got = knn_search(g, q[sel], k, md)
        want = golden_answer(G, mp, q, k, md)
        assert_same(got, tuple(a[sel] for a in want), q[sel])
        live = ikd_live(mp, q[sel], k, md, c["ds"])
        if live is not None:
            assert_same(got, live, q[sel])
    g.close()


@emul
@pytest.mark.parametrize("md", [0.0, 0.3, 0.99])
def test_small_max_dist_is_the_point_test(oracle_mod, md):
    """0 <= max_dist < 1: the point test alone (the brute-force oracle's rule; the reference's box prune is tree dependent there)"""
    c, q = ikd_cases.knn_case()
    q = np.concatenate([q[:300], c["map_xyz"][:20]])   # (map points themselves: d2 = 0 passes max_dist = 0)
    g = le.EmulGpu(c["ds"], max_map_points=200_000, max_scan_points=20_000)
    g.map_build(c["map_xyz"])
    for k in (1, 5, 16):
        xb, db, cb, _ = oracle_mod.knn_bruteforce(c["map_xyz"], q, k, md)
        assert_same(knn_search(g, q, k, md), (xb, db, cb), q)
    g.close()


@emul
def test_far_unbounded_and_nan_queries():
    c, _ = ikd_cases.knn_case()
    mp = c["map_xyz"]
    q = np.concatenate([_far_queries(mp), np.array([[np.nan, 0, 0], [0, np.inf, 0]], np.float32)])
    g = le.EmulGpu(c["ds"], max_map_points=200_000, max_scan_points=20_000)
    g.map_build(mp)
    for k, md in ((1, INF), (17, INF), (32, 1e12), (5, 5e4)):
        got = knn_search(g, q, k, md)
        assert_same(got, bruteforce(mp, q, k, md), q)
        assert got[2][-2] == 0 and got[2][-1] == 0 and np.all(got[1][-2:] == -1)
    g.close()


@emul
def test_max_dist_between_floats():
    """d2 <= max_dist with a double max_dist: a point at d2 = float(max_dist) rounded UP is out"""
    mp = np.array([[0, 0, 0], [1, 0, 0], [0, 1.5, 0], [0, 0, 2]], np.float32)
    q = np.zeros((1, 3), np.float32)
    g = le.EmulGpu(0.15, max_map_points=1000, max_scan_points=100)
    g.map_build(mp)
    d15 = float(np.float32(1.5) * np.float32(1.5))
    for md in (1.0, np.nextafter(1.0, 0), d15, np.nextafter(d15, 0), np.nextafter(d15, 9), 4.0, np.nextafter(4.0, 0)):
        assert_same(knn_search(g, q, 4, md), bruteforce(mp, q, 4, md), q)
    g.close()


@emul
def test_answers_follow_map_updates():
    """the list of bricks walked by far queries is rebuilt after every kind of map change"""
    c, q = ikd_cases.knn_case()
    mp = c["map_xyz"]
    q = np.concatenate([q[:40], _far_queries(mp)])
    g = le.EmulGpu(c["ds"], max_map_points=200_000, max_scan_points=20_000)
    g.map_build(mp[:15000])
    steps = [lambda: g.map_add_points(mp[15000:22000], True), lambda: g.map_add_points(mp[22000:] + np.float32(30), False),
             lambda: g.map_delete_boxes(np.array([[0, 0, -5, 10, 20, 5]], np.float32)), lambda: g.map_compact()]
    for step in [lambda: None] + steps:
        step()
        live = g.map_download()
        for k, md in ((8, INF), (3, 30.0)):
            assert_same(knn_search(g, q, k, md), bruteforce(live, q, k, md), q)
    g.close()


@emul
def test_k5_max_dist5_equals_nearest_search():
    c, q = ikd_cases.knn_case()
    g = le.EmulGpu(c["ds"], max_map_points=200_000, max_scan_points=20_000)
    g.map_build(c["map_xyz"])
    q = q[::6]
    assert_same(knn_search(g, q, 5, 5.0), g.nearest_search(q), q)
    g.close()


@emul
def test_argument_errors_leave_the_context_usable():
    c, q = ikd_cases.knn_case()
    g = le.EmulGpu(c["ds"], max_map_points=200_000, max_scan_points=20_000)
    g.map_build(c["map_xyz"])
    q = np.ascontiguousarray(q[:10], np.float32)
    out = np.zeros(33 * 10 * 3, np.float32)
    d2 = np.zeros(33 * 10, np.float32)
    cnt = np.zeros(10, np.int32)

    fn = g.L.liinit_map_knn_search
    fn.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_double, C.c_void_p, C.c_void_p, C.c_void_p]
    fn.restype = C.c_int

    def call(k=5, md=5.0, stride=3, n=10, qp=q.ctypes.data):
        return fn(g.h, C.c_void_p(qp), stride, n, k, md, out.ctypes.data, d2.ctypes.data, cnt.ctypes.data)
    for kw in (dict(k=0), dict(k=33), dict(md=math.nan), dict(md=-1e-9), dict(stride=5), dict(n=-1), dict(qp=0)):
        assert call(**kw) == -1, kw
        assert g.L.liinit_last_error(g.h)
    assert call(k=7, md=INF) == 0
    assert_same(knn_search(g, q, 7), bruteforce(c["map_xyz"], q, 7, INF), q)
    g.close()


@emul
def test_empty_map():
    g = le.EmulGpu(0.15, max_map_points=1000, max_scan_points=100)
    q = np.array([[0, 0, 0], [1e3, 0, 0], [3e5, 0, 0]], np.float32)
    for build in (False, True):
        if build:
            g.map_build(np.zeros((0, 3), np.float32))
        x, d, n = knn_search(g, q, 4, INF)
        assert np.all(n == 0) and np.all(d == -1) and np.all(x == 0)
    g.close()


def _build_cpp():
    from lidar_imu_init_b200 import _build
    _build.build_gpu()
    lib = os.path.join(ROOT, "lidar_imu_init_b200")
    src = os.path.join(ROOT, "tests", "cpp", "knn_general.cpp")
    exe = os.path.join(ROOT, "tests", "cpp", "knn_general")
    if os.path.exists(exe) and os.path.getmtime(exe) > max(os.path.getmtime(src), os.path.getmtime(_build.GPU_LIB)):
        return exe
    gxx = shutil.which("g++") or "/usr/bin/g++"
    subprocess.check_call([gxx, "-O1", "-std=c++14", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), "-I", os.path.join(lib, "csrc", "host"),
                           "-I", os.path.join(ROOT, "oracle", "shim"), src, "-o", exe, "-L", lib, "-lliinit_gpu", "-Wl,-rpath," + lib])
    return exe


def test_cpp_adapter_translation_unit_compiles():
    """DeviceMap::Nearest_Search(p, 10, near, d2, INFINITY) with the reference's point type: -std=c++14 -Wall -Werror"""
    assert os.path.exists(_build_cpp())


# ---- GPU ---------------------------------------------------------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("index", [1, 2])   # LIINIT_KNN_BRICKS, LIINIT_KNN_CELLS
def test_gpu_golden_grid(gpu_lib, index):
    c, q, G = golden()
    mp = c["map_xyz"]
    g = gpu_lib.LiInitGpu(c["ds"], max_map_points=200_000, max_scan_points=20_000, knn_index=index)
    g.map_build(mp)
    for k in kc.KNN_KS:
        for md in kc.KNN_MAX_DISTS:
            assert_same(knn_search(g, q, k, md), golden_answer(G, mp, q, k, md), q)
    g.close()


@pytest.mark.gpu
def test_gpu_parity_scene(gpu_lib, oracle_mod):
    """the test_gpu_parity scene (C2, N = 20k, M = 200k) against the restated oracle tree; k = 32 is beyond the oracle's candidate heap
    (16): its first 16 must be the k = 16 answer and a subset of the queries is checked against brute force"""
    from lidar_imu_init_b200 import scenes
    c = scenes.make_config("C2", N=20000, M=200000, open_air_frac=0.02)
    p = c["pose_init"]
    q = ikd_cases.world(c["body_xyz"], p)
    g = gpu_lib.LiInitGpu(c["ds"], max_map_points=400_000, max_scan_points=25_000)
    g.map_build(c["map_xyz"])
    om = oracle_mod.OracleMap(c["ds"], 0)
    om.build(c["map_xyz"])
    for md in (5.0, INF):
        for k in (1, 16):
            x, d, n, _ = om.knn(q, k, md)
            assert_same(knn_search(g, q, k, md), (x, d, n), q)
        x32, d32, n32 = knn_search(g, q, 32, md)
        x16, d16, n16 = knn_search(g, q, 16, md)
        assert np.array_equal(np.minimum(n32, 16), n16) and np.array_equal(d32[:, :16], d16)
        sub = np.r_[0:len(q):97]
        assert_same((x32[sub], d32[sub], n32[sub]), bruteforce(c["map_xyz"], q[sub], 32, md), q[sub])
    g.close()


@pytest.mark.gpu
def test_gpu_device_form_on_torch_stream(gpu_lib):
    import torch
    c, q, _ = golden()
    g = gpu_lib.LiInitGpu(c["ds"], max_map_points=200_000, max_scan_points=20_000)
    g.map_build(c["map_xyz"])
    s = torch.cuda.Stream()
    g.set_stream(s.cuda_stream)
    q4 = np.concatenate([q, np.zeros((len(q), 1), np.float32)], 1)
    for k, md in ((1, INF), (17, 5.0), (32, 30.0)):
        want = knn_search(g, q4, k, md)
        with torch.cuda.stream(s):
            tq = torch.from_numpy(q4).cuda()
            tx = torch.empty((len(q), k, 3), dtype=torch.float32, device="cuda")
            td = torch.empty((len(q), k), dtype=torch.float32, device="cuda")
            tn = torch.empty(len(q), dtype=torch.int32, device="cuda")
        g.knn_search_device(tq.data_ptr(), 4, len(q), k, md, tx.data_ptr(), td.data_ptr(), tn.data_ptr())
        s.synchronize()
        assert_same((tx.cpu().numpy(), td.cpu().numpy(), tn.cpu().numpy()), want)
    g.set_stream(0)
    g.close()


@pytest.mark.gpu
def test_gpu_more_queries_than_the_staging_capacity(gpu_lib):
    """the host form stages its queries in chunks of the staging capacity (at least 2^20 points)"""
    c, q = ikd_cases.knn_case()
    rng = np.random.default_rng(3)
    n = (1 << 20) + 5000
    qs = (q[rng.integers(0, len(q), n)] + rng.normal(0, 0.05, (n, 3))).astype(np.float32)
    g = gpu_lib.LiInitGpu(c["ds"], max_map_points=200_000, max_scan_points=1000)
    g.map_build(c["map_xyz"])
    one = knn_search(g, qs, 6, 5.0)
    h = n // 2
    a, b = knn_search(g, qs[:h], 6, 5.0), knn_search(g, qs[h:], 6, 5.0)
    assert_same(one, tuple(np.concatenate([u, v]) for u, v in zip(a, b)))
    g.close()


@pytest.mark.gpu
def test_gpu_cpp_adapter_equals_ctypes(tmp_path, gpu_lib):
    exe = _build_cpp()
    c, q, _ = golden()
    q = q[::3]
    inp, out = tmp_path / "in.bin", tmp_path / "out.bin"
    with open(inp, "wb") as f:
        f.write(np.array([len(c["map_xyz"]), len(q)], np.int32).tobytes())
        f.write(np.array([c["ds"]], np.float32).tobytes())
        f.write(np.ascontiguousarray(c["map_xyz"], np.float32).tobytes())
        f.write(np.ascontiguousarray(q, np.float32).tobytes())
    subprocess.check_call([exe, str(inp), str(out)])
    rec = np.frombuffer(open(out, "rb").read(), np.dtype([("cnt", np.int32), ("xyz", np.float32, (10, 3)), ("d2", np.float32, 10)]))
    g = gpu_lib.LiInitGpu(c["ds"], max_map_points=200_000, max_scan_points=20_000)
    g.map_build(c["map_xyz"])
    # (another context: the bricks were created in another order, so the walk of far queries may pick another of points tied at the 10th)
    assert_same((rec["xyz"], rec["d2"], rec["cnt"]), knn_search(g, q, 10, INF), q)
    g.close()
