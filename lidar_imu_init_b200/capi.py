"""ctypes binding of the C-ABI (include/liinit_gpu.h). Thin: one method per entry point.

The CUDA library is REQUIRED: importing a handle without the built
libliinit_gpu.so, or on a machine without a usable GPU, raises -- there is no
CPU fallback on the product path.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from . import _build

_LIB = None


class LiInitError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"liinit error {code}: {msg}")
        self.code = code


class Config(C.Structure):
    _fields_ = [("filter_size_map", C.c_float), ("max_map_points", C.c_int), ("max_scan_points", C.c_int), ("device_id", C.c_int),
                ("brick_cells_log2", C.c_int), ("hash_capacity_log2", C.c_int), ("knn_group_lanes", C.c_int), ("knn_seed_radius_cells", C.c_float), ("knn_index", C.c_int), ("reserved", C.c_int * 6)]


_f32 = np.ctypeslib.ndpointer(dtype=np.float32, flags="C_CONTIGUOUS")
_f64 = np.ctypeslib.ndpointer(dtype=np.float64, flags="C_CONTIGUOUS")
_i32 = np.ctypeslib.ndpointer(dtype=np.int32, flags="C_CONTIGUOUS")

SYMBOLS = [
    "liinit_create", "liinit_destroy", "liinit_last_error", "liinit_set_stream", "liinit_map_build", "liinit_map_add_points", "liinit_map_delete_boxes",
    "liinit_map_compact", "liinit_map_validnum", "liinit_map_size", "liinit_map_download", "liinit_map_nearest_search", "liinit_map_knn_search", "liinit_map_knn_search_device", "liinit_scan_upload", "liinit_scan_attach_host", "liinit_scan_upload_raw", "liinit_scan_download_body", "liinit_raw_upload", "liinit_raw_undistort_cv", "liinit_raw_undistort_imu",
    "liinit_raw_download", "liinit_raw_downsample",
    "liinit_icp_iterate", "liinit_icp_iterate_device", "liinit_scan_download_effect", "liinit_scan_download_state",
    "liinit_map_incremental", "liinit_last_pass_timing", "liinit_last_pass_kernel_times", "liinit_launch_count", "liinit_map_stats", "liinit_knn_index",
    "liinit_comm_unique_id", "liinit_comm_init", "liinit_comm_info", "liinit_comm_last_local", "liinit_comm_mode", "liinit_debug_esti_plane", "liinit_set_reseed",
]


def lib_path() -> str:
    # LIINIT_GPU_LIB: developer override to A/B alternative builds of the same C-ABI
    return os.environ.get("LIINIT_GPU_LIB") or _build.GPU_LIB


def load():
    """dlopen the in-tree CUDA library (no compute). Raises if it has not been built."""
    global _LIB
    if _LIB is not None:
        return _LIB
    p = lib_path()
    if not os.path.exists(p):
        raise FileNotFoundError(f"{p} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` (nvcc) first. "
                                "There is no CPU fallback.")
    L = C.CDLL(p)
    vp = C.c_void_p
    L.liinit_create.argtypes = [C.POINTER(Config), C.POINTER(vp)]
    L.liinit_destroy.argtypes = [vp]
    L.liinit_last_error.restype = C.c_char_p
    L.liinit_last_error.argtypes = [vp]
    L.liinit_set_stream.argtypes = [vp, vp]
    L.liinit_map_build.argtypes = [vp, vp, C.c_int, C.c_int]
    L.liinit_map_add_points.argtypes = [vp, vp, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int)]
    L.liinit_map_delete_boxes.argtypes = [vp, vp, C.c_int, C.POINTER(C.c_int)]
    L.liinit_map_compact.argtypes = [vp]
    L.liinit_map_validnum.argtypes = [vp, C.POINTER(C.c_int)]
    L.liinit_map_size.argtypes = [vp, C.POINTER(C.c_int)]
    L.liinit_map_download.argtypes = [vp, vp, C.c_int, C.POINTER(C.c_int)]
    L.liinit_map_nearest_search.argtypes = [vp, vp, C.c_int, C.c_int, C.c_double, vp, vp, vp]
    L.liinit_map_knn_search.argtypes = [vp, vp, C.c_int, C.c_int, C.c_int, C.c_double, vp, vp, vp]
    L.liinit_map_knn_search_device.argtypes = [vp, vp, C.c_int, C.c_int, C.c_int, C.c_double, vp, vp, vp]
    L.liinit_scan_upload.argtypes = [vp, vp, C.c_int, C.c_int]
    L.liinit_scan_attach_host.argtypes = [vp, vp, C.c_int, C.c_int]
    L.liinit_scan_upload_raw.argtypes = [vp, vp, C.c_int, C.c_int, C.c_float, C.POINTER(C.c_int)]
    L.liinit_raw_upload.argtypes = [vp, vp, C.c_int, C.c_int, C.c_int]
    L.liinit_raw_undistort_cv.argtypes = [vp, _f64, _f64, _f64]
    L.liinit_raw_undistort_imu.argtypes = [vp, _f64, C.c_int, _f64, _f64, _f64, _f64]
    L.liinit_raw_download.argtypes = [vp, vp, C.c_int, C.POINTER(C.c_int)]
    L.liinit_raw_downsample.argtypes = [vp, C.c_float, C.POINTER(C.c_int)]
    L.liinit_scan_download_body.argtypes = [vp, vp, C.c_int, C.POINTER(C.c_int)]
    L.liinit_icp_iterate.argtypes = [vp, _f64, _f64, _f64, _f64, C.c_int, C.c_int, _f64, _f64, C.POINTER(C.c_int), C.POINTER(C.c_double)]
    L.liinit_icp_iterate_device.argtypes = [vp, _f64, _f64, _f64, _f64, C.c_int, C.c_int, vp]
    L.liinit_scan_download_effect.argtypes = [vp, vp, vp, C.c_int, C.POINTER(C.c_int)]
    L.liinit_scan_download_state.argtypes = [vp, vp, vp, vp, vp, vp]
    L.liinit_map_incremental.argtypes = [vp, _f64, _f64, _f64, _f64, C.c_double, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int)]
    L.liinit_last_pass_timing.argtypes = [vp, C.POINTER(C.c_float), C.POINTER(C.c_int)]
    L.liinit_last_pass_kernel_times.argtypes = [vp, C.POINTER(C.c_float), C.POINTER(C.c_float)]
    L.liinit_launch_count.argtypes = [vp, C.POINTER(C.c_longlong)]
    L.liinit_knn_index.argtypes = [vp, C.POINTER(C.c_int)]
    L.liinit_map_stats.argtypes = [vp, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_longlong), C.POINTER(C.c_longlong)]
    L.liinit_comm_unique_id.argtypes = [vp]
    L.liinit_comm_init.argtypes = [vp, vp, C.c_int, C.c_int]
    L.liinit_debug_esti_plane.argtypes = [vp, vp, C.c_int, vp, vp]
    L.liinit_comm_last_local.argtypes = [vp, _f64]
    L.liinit_comm_mode.argtypes = [vp, C.POINTER(C.c_int)]
    L.liinit_set_reseed.argtypes = [vp, C.c_int]
    L.liinit_comm_info.argtypes = [vp, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int)]
    for s in SYMBOLS:
        getattr(L, s).restype = getattr(L, s).restype if s == "liinit_last_error" else C.c_int
    _LIB = L
    return L


def _pts(a):
    """float32 C-contiguous [n, stride] with stride in (3, 4, 12)."""
    a = np.ascontiguousarray(a, dtype=np.float32)
    if a.ndim != 2 or a.shape[1] not in (3, 4, 12):
        raise ValueError("points must be [n,3], [n,4] or [n,12] float32")
    return a


def _ptr(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


class LiInitGpu:
    """One context = one GPU + one device-resident map + one resident scan."""

    def __init__(self, filter_size_map=0.15, max_map_points=6_000_000, max_scan_points=300_000, device_id=0, brick_cells_log2=0,
                 hash_capacity_log2=0, knn_group_lanes=0, knn_seed_radius_cells=0.0, knn_index=0):
        self.L = load()
        cfg = Config(filter_size_map, max_map_points, max_scan_points, device_id, brick_cells_log2, hash_capacity_log2, knn_group_lanes, knn_seed_radius_cells,
                     knn_index)
        h = C.c_void_p()
        rc = self.L.liinit_create(C.byref(cfg), C.byref(h))
        if rc != 0:
            raise LiInitError(rc, (self.L.liinit_last_error(None) or b"").decode())
        self.h = h
        self.scan_n = 0

    def close(self):
        if getattr(self, "h", None):
            self.L.liinit_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, rc):
        if rc != 0:
            raise LiInitError(rc, (self.L.liinit_last_error(self.h) or b"").decode())

    def set_stream(self, cuda_stream: int):
        self._ck(self.L.liinit_set_stream(self.h, C.c_void_p(cuda_stream)))

    # ---- map ----
    def map_build(self, xyz):
        a = _pts(xyz)
        self._ck(self.L.liinit_map_build(self.h, _ptr(a), a.shape[1], a.shape[0]))

    def map_add_points(self, xyz, downsample_on: bool) -> int:
        a = _pts(xyz)
        added = C.c_int(0)
        if a.shape[0] == 0:
            return 0
        self._ck(self.L.liinit_map_add_points(self.h, _ptr(a), a.shape[1], a.shape[0], int(downsample_on), C.byref(added)))
        return added.value

    def map_delete_boxes(self, boxes) -> int:
        """boxes: [n, 6] float32 rows {min x,y,z, max x,y,z}; returns the number of deleted points."""
        b = np.ascontiguousarray(boxes, dtype=np.float32).reshape(-1, 6)
        d = C.c_int(0)
        self._ck(self.L.liinit_map_delete_boxes(self.h, _ptr(b), len(b), C.byref(d)))
        return d.value

    def map_compact(self):
        self._ck(self.L.liinit_map_compact(self.h))

    def map_validnum(self) -> int:
        n = C.c_int(0)
        self._ck(self.L.liinit_map_validnum(self.h, C.byref(n)))
        return n.value

    def map_size(self) -> int:
        n = C.c_int(0)
        self._ck(self.L.liinit_map_size(self.h, C.byref(n)))
        return n.value

    def map_download(self):
        n = self.map_validnum()
        out = np.zeros((max(n, 1), 3), np.float32)
        m = C.c_int(0)
        self._ck(self.L.liinit_map_download(self.h, _ptr(out), n, C.byref(m)))
        return out[:min(n, m.value)]

    def map_stats(self):
        b, s, pu, pc = C.c_int(0), C.c_int(0), C.c_longlong(0), C.c_longlong(0)
        self._ck(self.L.liinit_map_stats(self.h, C.byref(b), C.byref(s), C.byref(pu), C.byref(pc)))
        return dict(bricks=b.value, hash_slots=s.value, pool_used=pu.value, pool_cap=pc.value)

    def nearest_search(self, q, max_dist=5.0):
        a = _pts(q)
        n = a.shape[0]
        xyz = np.zeros((n, 5, 3), np.float32)
        d2 = np.zeros((n, 5), np.float32)
        cnt = np.zeros(n, np.int32)
        self._ck(self.L.liinit_map_nearest_search(self.h, _ptr(a), a.shape[1], n, max_dist, _ptr(xyz), _ptr(d2), _ptr(cnt)))
        return xyz, d2, cnt

    def knn_search(self, q, k, max_dist=float("inf")):
        """KD_TREE::Nearest_Search(q, k, ..., max_dist) for every row of q -> (xyz [n,k,3], d2 [n,k], cnt [n]); -1 / zeros past cnt"""
        a = _pts(q)
        n = a.shape[0]
        xyz = np.zeros((n, k, 3), np.float32)
        d2 = np.zeros((n, k), np.float32)
        cnt = np.zeros(n, np.int32)
        self._ck(self.L.liinit_map_knn_search(self.h, _ptr(a), a.shape[1], n, int(k), float(max_dist), _ptr(xyz), _ptr(d2), _ptr(cnt)))
        return xyz, d2, cnt

    def knn_search_device(self, q_ptr: int, stride: int, n: int, k: int, max_dist: float, out_xyz_ptr: int, out_d2_ptr: int, out_cnt_ptr: int):
        """The same search on device memory (e.g. data_ptr() of CUDA torch tensors), queued on the context's stream, no synchronisation"""
        self._ck(self.L.liinit_map_knn_search_device(self.h, C.c_void_p(q_ptr), int(stride), int(n), int(k), float(max_dist), C.c_void_p(out_xyz_ptr),
                                                     C.c_void_p(out_d2_ptr), C.c_void_p(out_cnt_ptr)))

    # ---- scan ----
    def scan_upload(self, body):
        a = _pts(body)
        self._ck(self.L.liinit_scan_upload(self.h, _ptr(a), a.shape[1], a.shape[0]))
        self.scan_n = a.shape[0]

    def scan_upload_raw(self, pts, leaf_size: float) -> int:
        """Voxel-grid downsample on the device (PCL VoxelGrid semantics), result becomes the resident scan."""
        a = _pts(pts)
        nd = C.c_int(0)
        self._ck(self.L.liinit_scan_upload_raw(self.h, _ptr(a), a.shape[1], a.shape[0], float(leaf_size), C.byref(nd)))
        self.scan_n = nd.value
        return nd.value

    # ---- raw-scan front end ----
    def raw_upload(self, pts, time_index: int = -1):
        a = np.ascontiguousarray(pts, dtype=np.float32)
        self._ck(self.L.liinit_raw_upload(self.h, _ptr(a), a.shape[1], int(time_index), a.shape[0]))
        self.raw_n = a.shape[0]

    def raw_undistort_cv(self, omega, rot_end, vel_end):
        self._ck(self.L.liinit_raw_undistort_cv(self.h, np.ascontiguousarray(omega, np.float64), np.ascontiguousarray(rot_end, np.float64).reshape(9),
                                                np.ascontiguousarray(vel_end, np.float64)))

    def raw_undistort_imu(self, poses, rot_end, pos_end, R_LI, T_LI):
        P = np.ascontiguousarray(poses, np.float64).reshape(-1, 22)
        self._ck(self.L.liinit_raw_undistort_imu(self.h, P.reshape(-1), len(P), np.ascontiguousarray(rot_end, np.float64).reshape(9),
                                                 np.ascontiguousarray(pos_end, np.float64), np.ascontiguousarray(R_LI, np.float64).reshape(9),
                                                 np.ascontiguousarray(T_LI, np.float64)))

    def raw_points(self):
        n = C.c_int(0)
        out = np.zeros((max(getattr(self, "raw_n", 0), 1), 3), np.float32)
        self._ck(self.L.liinit_raw_download(self.h, _ptr(out), len(out), C.byref(n)))
        return out[:n.value]

    def raw_downsample(self, leaf_size: float) -> int:
        nd = C.c_int(0)
        self._ck(self.L.liinit_raw_downsample(self.h, float(leaf_size), C.byref(nd)))
        self.scan_n = nd.value
        return nd.value

    def scan_body(self):
        n = C.c_int(0)
        out = np.zeros((max(self.scan_n, 1), 3), np.float32)
        self._ck(self.L.liinit_scan_download_body(self.h, _ptr(out), self.scan_n, C.byref(n)))
        return out[:n.value]

    def scan_upload_ptr(self, host_ptr: int, stride: int, n: int):
        """Upload from a raw host pointer (e.g. pinned torch tensor)."""
        self._ck(self.L.liinit_scan_upload(self.h, C.c_void_p(host_ptr), stride, n))
        self.scan_n = n

    def scan_attach_ptr(self, host_ptr: int, stride: int, n: int):
        """Zero-copy variant: `host_ptr` is page-locked memory the first search pass reads over PCIe (see the header)."""
        self._ck(self.L.liinit_scan_attach_host(self.h, C.c_void_p(host_ptr), stride, n))
        self.scan_n = n

    def icp_iterate(self, rot_end, pos_end, R_LI, T_LI, imu_en: bool, search: bool):
        HtH = np.zeros((12, 12))
        Htr = np.zeros(12)
        m = C.c_int(0)
        rs = C.c_double(0)
        self._ck(self.L.liinit_icp_iterate(self.h, np.ascontiguousarray(rot_end, np.float64).reshape(9), np.ascontiguousarray(pos_end, np.float64),
                                           np.ascontiguousarray(R_LI, np.float64).reshape(9), np.ascontiguousarray(T_LI, np.float64),
                                           int(imu_en), int(search), HtH.reshape(144), Htr, C.byref(m), C.byref(rs)))
        return HtH, Htr, m.value, rs.value

    def icp_iterate_device(self, rot_end, pos_end, R_LI, T_LI, imu_en: bool, search: bool, d_out_ptr: int):
        self._ck(self.L.liinit_icp_iterate_device(self.h, np.ascontiguousarray(rot_end, np.float64).reshape(9), np.ascontiguousarray(pos_end, np.float64),
                                                  np.ascontiguousarray(R_LI, np.float64).reshape(9), np.ascontiguousarray(T_LI, np.float64),
                                                  int(imu_en), int(search), C.c_void_p(d_out_ptr)))

    def scan_state(self):
        n = self.scan_n
        out = dict(world=np.zeros((n, 3), np.float32), near_xyz=np.zeros((n, 5, 3), np.float32), near_cnt=np.zeros(n, np.int32),
                   selected=np.zeros(n, np.uint8), normvec=np.zeros((n, 4), np.float32))
        self._ck(self.L.liinit_scan_download_state(self.h, _ptr(out["world"]), _ptr(out["near_xyz"]), _ptr(out["near_cnt"]),
                                                   _ptr(out["selected"]), _ptr(out["normvec"])))
        return out

    def scan_effect(self):
        n = self.scan_n
        ori = np.zeros((n, 3), np.float32)
        nv = np.zeros((n, 4), np.float32)
        m = C.c_int(0)
        self._ck(self.L.liinit_scan_download_effect(self.h, _ptr(ori), _ptr(nv), n, C.byref(m)))
        return ori[:m.value], nv[:m.value]

    def map_incremental(self, rot_end, pos_end, R_LI, T_LI, ds: float, flg_EKF_inited: bool = True):
        na, nn = C.c_int(0), C.c_int(0)
        self._ck(self.L.liinit_map_incremental(self.h, np.ascontiguousarray(rot_end, np.float64).reshape(9), np.ascontiguousarray(pos_end, np.float64),
                                               np.ascontiguousarray(R_LI, np.float64).reshape(9), np.ascontiguousarray(T_LI, np.float64),
                                               float(ds), int(flg_EKF_inited), C.byref(na), C.byref(nn)))
        return na.value, nn.value

    def last_pass_timing(self):
        ms, nl = C.c_float(0), C.c_int(0)
        self._ck(self.L.liinit_last_pass_timing(self.h, C.byref(ms), C.byref(nl)))
        return ms.value, nl.value

    def last_pass_kernel_times(self):
        a, b = C.c_float(0), C.c_float(0)
        self._ck(self.L.liinit_last_pass_kernel_times(self.h, C.byref(a), C.byref(b)))
        return a.value, b.value

    def debug_esti_plane(self, nb):
        """esti_plane of the device for neighbour sets nb [n, 5, 3] -> (pabcd [n, 4] f64, valid [n] bool)"""
        a = np.ascontiguousarray(nb, np.float32).reshape(-1, 15)
        out = np.zeros((len(a), 4))
        ok = np.zeros(len(a), np.uint8)
        self._ck(self.L.liinit_debug_esti_plane(self.h, _ptr(a), len(a), _ptr(out), _ptr(ok)))
        return out, ok.astype(bool)

    # ---- multi-GPU: the all-reduce of the accumulators and the gathers of per-point results live behind the C-ABI ----
    @staticmethod
    def comm_unique_id() -> bytes:
        """ncclGetUniqueId through the library (call on one rank, distribute the 128 bytes)."""
        L = load()
        buf = C.create_string_buffer(128)
        rc = L.liinit_comm_unique_id(buf)
        if rc != 0:
            raise LiInitError(rc, (L.liinit_last_error(None) or b"").decode())
        return buf.raw

    def comm_init(self, unique_id: bytes, nranks: int, rank: int):
        """Collective: attach this context to an nranks-wide communicator. From then on icp_iterate returns the sum over the
        ranks and every rank works on its slot of the uploaded frame."""
        assert len(unique_id) == 128
        buf = C.create_string_buffer(unique_id, 128)
        self._ck(self.L.liinit_comm_init(self.h, buf, int(nranks), int(rank)))

    def set_reseed(self, enabled: bool):
        """later search passes of a scan start from the previous pass's neighbours (default on); off = every search from scratch"""
        self._ck(self.L.liinit_set_reseed(self.h, int(enabled)))

    def comm_mode(self) -> str:
        v = C.c_int(0)
        self._ck(self.L.liinit_comm_mode(self.h, C.byref(v)))
        return "peer memory (fused in the plane kernel)" if v.value else "ncclAllReduce"

    def comm_last_local(self):
        out = np.zeros(160)
        self._ck(self.L.liinit_comm_last_local(self.h, out))
        return out

    def comm_info(self):
        a, b, c, d = C.c_int(), C.c_int(), C.c_int(), C.c_int()
        self._ck(self.L.liinit_comm_info(self.h, C.byref(a), C.byref(b), C.byref(c), C.byref(d)))
        return dict(nranks=a.value, rank=b.value, shard_lo=c.value, shard_n=d.value)

    def knn_index(self) -> int:
        """1 = LIINIT_KNN_BRICKS (lockstep groups over whole bricks), 2 = LIINIT_KNN_CELLS (cell directory, thread per point)."""
        v = C.c_int()
        self._ck(self.L.liinit_knn_index(self.h, C.byref(v)))
        return v.value

    def launch_count(self) -> int:
        n = C.c_longlong(0)
        self._ck(self.L.liinit_launch_count(self.h, C.byref(n)))
        return n.value
