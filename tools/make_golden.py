"""Generate tests/golden/*.npz: inputs + outputs of the hot path computed with the reference's verbatim
ikd-Tree (oracle/_ref, backend 1) and the restated measurement model, plus (ikd_tree.npz) the verbatim tree's
answers to the oracle checks of tests/ikd_cases.py. Tests compare both the oracle and the CUDA path against
them, so they need no copy of the reference where they run.

Needs oracle/_ref (make -C oracle ref REF=<checkout of the reference>). Run from the repo root:  python tools/make_golden.py  (all files) or  python tools/make_golden.py ikd_tree  (that one only)
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import ikd_cases  # noqa: E402
from lidar_imu_init_b200 import scenes  # noqa: E402
from oracle import oracle as orc  # noqa: E402


def world(body, p):
    return (p.rot_end @ (p.R_LI @ body.T.astype(np.float64) + p.T_LI[:, None]) + p.pos_end[:, None]).T.astype(np.float32)


def pose_arr(p):
    return np.concatenate([p.rot_end.reshape(9), p.pos_end, p.R_LI.reshape(9), p.T_LI])


def one(name, cfg, imu_en):
    assert orc.has_ikd(), "golden vectors must come from the verbatim ikd-Tree build (make -C oracle ref)"
    c = cfg
    p = c["pose_init"]
    om = orc.OracleMap(c["ds"], 1)
    om.build(c["map_xyz"])
    sc = orc.OracleScan(c["body_xyz"])
    out = dict(map_xyz=c["map_xyz"], body_xyz=c["body_xyz"], ds=np.float64(c["ds"]), imu_en=np.int32(imu_en), pose_init=pose_arr(p),
               pose_gt=pose_arr(c["pose_gt"]))
    H, b, m = sc.iterate(om, p.rot_end, p.pos_end, p.R_LI, p.T_LI, imu_en, True)
    st = sc.get()
    out.update(s_HtH=H, s_Htr=b, s_m=np.int32(m), s_near_cnt=st["near_cnt"], s_near_xyz=st["near_xyz"], s_near_d2=st["near_d2"],
               s_selected=st["selected"], s_normvec=st["normvec"], s_world=st["world"])
    p2 = scenes.perturb_pose(p, 77, dtheta_deg=0.05, dpos=0.01)
    out["pose_2"] = pose_arr(p2)
    H2, b2, m2 = sc.iterate(om, p2.rot_end, p2.pos_end, p2.R_LI, p2.T_LI, imu_en, False)
    st2 = sc.get()
    out.update(r_HtH=H2, r_Htr=b2, r_m=np.int32(m2), r_selected=st2["selected"], r_normvec=st2["normvec"])
    gt = c["pose_gt"]
    cnt, na, nn, flags = sc.map_incremental(om, gt.rot_end, gt.pos_end, gt.R_LI, gt.T_LI, c["ds"])
    live = om.flatten()
    live = live[np.lexsort((live[:, 2], live[:, 1], live[:, 0]))]
    out.update(mi_n_add=np.int32(na), mi_n_nod=np.int32(nn), mi_flags=flags.astype(np.int8), mi_live=live)
    np.savez_compressed(os.path.join(ROOT, "tests", "golden", name + ".npz"), **out)
    print(name, "m", m, m2, "add", na, nn, "live", len(live))


def ikd_tree():
    assert orc.has_ikd(), "golden vectors must come from the verbatim ikd-Tree build (make -C oracle ref)"
    c, q = ikd_cases.knn_case()
    om = orc.OracleMap(c["ds"], 1)
    om.build(c["map_xyz"])
    x, d2, cnt, _ = om.knn(q)
    out = dict(knn_inputs=ikd_cases.digest(c["map_xyz"], q), knn_nbr=ikd_cases.map_rows(x, cnt, c["map_xyz"]), knn_d2=d2, knn_cnt=cnt)
    ds, mp, batches = ikd_cases.add_points_case()
    om = orc.OracleMap(ds, 1)
    om.build(mp)
    for b, down in batches:
        om.add_points(b, down)
    cand = ikd_cases.add_points_candidates(mp, batches)
    out.update(add_inputs=ikd_cases.digest(cand), add_validnum=np.int32(om.validnum()), add_live=ikd_cases.live_mask(om.flatten(), cand))
    pts, boxes = ikd_cases.delete_boxes_case()
    om = orc.OracleMap(0.15, 1)
    om.build(pts)
    d = om.delete_boxes(boxes)
    out.update(del_inputs=ikd_cases.digest(pts, boxes), del_deleted=np.int32(d), del_validnum=np.int32(om.validnum()),
               del_live=ikd_cases.live_mask(om.flatten(), pts))
    np.savez_compressed(ikd_cases.GOLD, **out)
    print("ikd_tree", "knn", int((cnt == 5).sum()), "add live", out["add_validnum"], "deleted", d)


if __name__ == "__main__":
    if sys.argv[1:] == ["ikd_tree"]:
        ikd_tree()
        sys.exit(0)
    one("c1_lo", scenes.make_config("C1", imu_en=False), False)
    one("c1_lio", scenes.make_config("C1", imu_en=True), True)
    one("c2small_lo", scenes.make_config("C2", N=3000, M=40000, open_air_frac=0.02, imu_en=False), False)
    one("c2small_lio", scenes.make_config("C2", N=3000, M=40000, open_air_frac=0.02, imu_en=True), True)
