"""The oracle checks against the reference's verbatim ikd-Tree (tests/test_oracle.py): their inputs, and how the tree's answers are
stored in tests/golden/ikd_tree.npz (written by tools/make_golden.py with the verbatim build). With the file the checks run on any
machine, also where oracle/_ref cannot be built."""
import hashlib
import os

import numpy as np

from lidar_imu_init_b200 import scenes

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ikd_tree.npz")


def world(body, p):
    return (p.rot_end @ (p.R_LI @ body.T.astype(np.float64) + p.T_LI[:, None]) + p.pos_end[:, None]).T.astype(np.float32)


def digest(*arrays):
    """sha256 of the inputs: tells a changed scene generator apart from a changed oracle"""
    h = hashlib.sha256()
    for a in arrays:
        h.update(np.ascontiguousarray(a).tobytes())
    return h.hexdigest()


def knn_case():
    c = scenes.make_config("C2", N=3000, M=30000, open_air_frac=0.03)
    return c, world(c["body_xyz"], c["pose_init"])


def map_rows(xyz, cnt, mp):
    """neighbours [nq, k, 3] -> their rows in the map [nq, k] (-1 past the count)"""
    row = {bytes(p): i for i, p in enumerate(np.ascontiguousarray(mp, np.float32))}
    out = np.full(xyz.shape[:2], -1, np.int32)
    for i, n in enumerate(cnt):
        out[i, :n] = [row[bytes(p)] for p in xyz[i, :n]]
    return out


def neighbours(rows, mp):
    """inverse of map_rows: the map's points, zeros past the count (as the oracle returns them)"""
    return np.where(rows[..., None] >= 0, mp[np.maximum(rows, 0)], np.float32(0))


def add_points_case():
    """-> (ds, map, [(batch, downsample_on), ...])"""
    c = scenes.make_config("C2", N=8000, M=30000, open_air_frac=0.0)
    new = world(c["body_xyz"], c["pose_gt"])
    return c["ds"], c["map_xyz"], [(new[:5000], True), (new[5000:], False), (new[3000:7000] + np.float32(0.01), True)]


def add_points_candidates(mp, batches):
    """every point the map can hold after the batches: Build's points, then each batch's"""
    return np.concatenate([mp] + [b for b, _ in batches], 0)


def delete_boxes_case():
    rng = np.random.default_rng(8)
    pts = rng.uniform(0, 20, (20000, 3)).astype(np.float32)
    pts[:50, 0] = 5.0                       # points exactly on a box face: min is inclusive, max exclusive
    pts[50:100, 0] = 9.0
    boxes = np.array([[5, 0, 0, 9, 20, 20], [0, 18, 0, 20, 20, 3]], np.float32)
    return pts, boxes


def point_set(xyz):
    return set(map(bytes, np.ascontiguousarray(xyz, np.float32)))


def live_mask(live, candidates):
    """the live set of a map as a packed bit per candidate point (every live point is one of them)"""
    s = point_set(live)
    mask = np.array([bytes(p) in s for p in np.ascontiguousarray(candidates, np.float32)])
    assert point_set(candidates[mask]) == s, "a live point is not among the candidates"
    return np.packbits(mask)


def live_set(packed, candidates):
    return point_set(candidates[np.unpackbits(packed, count=len(candidates)).astype(bool)])
