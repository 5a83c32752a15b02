"""Inputs of the checks of KD_TREE::Nearest_Search for any k and max_dist (tests/test_knn_general.py), and how the verbatim ikd-Tree's
answers to them are stored in tests/golden/ikd_knn.npz (written by tools/make_golden.py ikd_knn with the verbatim build). Shares the scene
and the storage rules (neighbours as map rows, a digest of the inputs) of tests/ikd_cases.py."""
import ctypes as C
import os

import numpy as np

import ikd_cases

GOLD_KNN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ikd_knn.npz")
KNN_KS = (1, 5, 8, 17, 32)
KNN_MAX_DISTS = (1.0, 5.0, 30.0, float("inf"))


def knn_general_case():
    """The knn_case() scene and ~1000 queries: scan points at the perturbed pose, open-air points above the map, points 50 m and 1 km
    away, and a few beyond the range brick keys can pack at this ds (|x| / ds >= 2^20). -> (config, queries)"""
    c, w = ikd_cases.knn_case()
    rng = np.random.default_rng(31)
    mp = c["map_xyz"]
    lo, hi = mp.min(0), mp.max(0)
    scan = w[rng.choice(len(w), 700, replace=False)]
    air = rng.uniform(lo, hi + np.array([0, 0, 6], np.float32), (150, 3)).astype(np.float32)
    air[:, 2] += 2.0
    dirs = rng.normal(size=(120, 3))
    dirs /= np.linalg.norm(dirs, axis=1, keepdims=True)
    base = scan[:120].astype(np.float64)
    far = np.concatenate([base[:60] + 50.0 * dirs[:60], base[60:] + 1000.0 * dirs[60:]]).astype(np.float32)
    beyond = np.array([[3e5, 5, 1], [-3e5, 2, 0], [4, 3e5, 1], [7, -3e5, 2], [3, 4, 3e5], [1, 1, -3e5], [3e5, 3e5, 3e5], [-3e5, 1e3, -2e5]],
                      np.float32)
    return c, np.concatenate([scan, air, far, beyond])


def knn_search(g, q, k, max_dist=float("inf")):
    """liinit_map_knn_search through either binding: LiInitGpu.knn_search of the package, or the C entry point of the emulated library
    (tests/liinit_emul.EmulGpu, which the CPU tests and the LIINIT_GPU_TESTS_ON_EMUL dry run use) -> (xyz [n,k,3], d2 [n,k], cnt [n])"""
    if hasattr(g, "knn_search"):
        return g.knn_search(q, k, max_dist)
    vp = C.c_void_p
    fn = g.L.liinit_map_knn_search
    fn.argtypes = [vp, vp, C.c_int, C.c_int, C.c_int, C.c_double, vp, vp, vp]
    fn.restype = C.c_int
    q = np.ascontiguousarray(q, np.float32)
    assert q.ndim == 2 and q.shape[1] in (3, 4, 12)
    n = len(q)
    xyz = np.zeros((n, k, 3), np.float32)
    d2 = np.zeros((n, k), np.float32)
    cnt = np.zeros(n, np.int32)
    g._ck(fn(g.h, q.ctypes.data_as(vp), q.shape[1], n, int(k), float(max_dist), xyz.ctypes.data_as(vp), d2.ctypes.data_as(vp),
             cnt.ctypes.data_as(vp)))
    return xyz, d2, cnt
